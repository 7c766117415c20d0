// sga_kernels.cuh -- parameter block of the on-device stochastic gradient ascent (rbo_stochastic_solve_batch, sga_kernels.cu).
#pragma once
#include "rbo_device.cuh"

namespace rbo {

// Everything the per-restart step kernel reads and writes; passed by value.
struct SgaProblem {
  int B, Ms, d, maxit;          // restarts; samples per restart (trajectory m = b * Ms + sample); input dim; iteration cap
  int optimizer, use_eswavs, project;
  double eta, beta1, beta2, eps;
  double omb1, omb2;            // 1 - beta1, 1 - beta2 rounded on the host, as the host mirror's (1 - beta) is
  double lbs[RBO_MAXD], ubs[RBO_MAXD];
  const double* bias;           // [2][maxit]: 1 - beta1^t, 1 - beta2^t for t = 1..maxit (host pow)
  // rollout outputs of the current iteration
  const double* values;         // [B * Ms]
  const double* grad_x;         // [B * Ms][d]
  const int* status;            // [B * Ms]
  const int* work_counter;      // [1..8]: the rollout kernel's watchdog flags and their details
  // optimiser state
  double* x;                    // [B][d] current iterates (the x0_batch the rollout kernel reads)
  double *m, *v;                // [B][d] Adam moments
  // history, column-major as returned: x / gmean / gstd [B][maxit][d], mean / std [B][maxit]
  double *xh, *gmh, *gsh, *mh, *sh;
  // per-restart integers
  int* live;                    // [B] 1 while the restart runs
  int* n_iter;                  // [B] evaluations performed
  int* end_status;              // [B] RBO_SGA_*
  int* fail;                    // [B][2] first failing sample, its RBO_TRAJ_* status
  int* nfail;                   // [B] failed trajectories at the last evaluation
  int* sticky;                  // [16]: [0] a watchdog flag was seen in some iteration, [1..8] the work_counter entries then
};

__global__ void rbo_sga_worklist_kernel(const int* order, const int* live, int Ms, int M, int* list);
__global__ void rbo_sga_step_kernel(const __grid_constant__ SgaProblem S, int k);

}  // namespace rbo
