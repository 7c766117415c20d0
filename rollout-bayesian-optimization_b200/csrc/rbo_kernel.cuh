// rbo_kernel.cuh -- parameter block and shared-memory plan of the rollout kernel (host + device).
#pragma once
#include "rbo_device.cuh"

namespace rbo {

// Shared-memory plan (offsets in doubles from the start of dynamic shared memory).
struct SmemPlan {
  int V, Fp, G, u, Xf, yf, gyf, Xs, stage, mbar;
  int sx, sxt, sg, sH, sp;                   // per slot: x, trial x, gradient, Hessian of the merit
  int sHt, sHref, sga, sdmu, sdsig, sgh;     // per slot: trial Hessian (also the trust-region scratch), grad alpha, grad mu, grad sigma, scalars; sHref: ONE d x d reference H alpha
  int sf, slam, spred, shs, ssn;             // per slot scalars: merit f, trust-region radius, predicted decrease, alpha, |step|_2
  int ppre, ppost, phess;                    // partial sums of the row reductions
  int bestx, misc, adj;                      // [d] best candidate ; scalar/scratch area ; adjoint duals
  int sord;                                  // [3][S] uint16: evaluations of every start in the previous multistart / in the first multistart of the previous trajectory; order in which the starts are handed out
  int sbnd;                                  // [2][d] box bounds (lane-indexed reads: kernel parameters would be serialised constant loads)
  int pairs, tbl, ints;                      // int areas (in doubles)
  int total;                                 // total doubles
};

// Everything the rollout kernel needs, passed by value as a __grid_constant__ parameter.
struct DevProblem {
  // sizes
  int d, N, N8, nb8;      // input dim; base observations; N rounded up to RBO_PR; N8 / RBO_PR
  int nb32;               // number of 32-row panels of L0 (ceil(N / RBO_BR))
  int h, S, W;            // horizon; start columns; start slots evaluated together in one lock-step round
  int CS, RP, NR;         // columns per start slot (d+3); padded V row pitch (doubles); V rows (N8 + RBO_MAXFAN)
  int RSmax, NPmax;       // row splits of the reductions; capacity of the pair list
  int RSh;                // row splits of the Hessian sums (>= RSmax when shared memory allows)
  int xsm, XP;            // base locations staged in shared memory (1) or read through L1 (0); their row pitch
  int vglob;              // 1: the work matrix V does not fit shared memory and lives in Vscratch (large-n variant)
  double* Vscratch;       // [gridDim.x][NR][RP] when vglob
  double* Bscratch;       // [gridDim.x][bscratch_len]: out-of-place result of the backward pass (large-n variant)
  size_t bscratch_len;
  int M;                  // trajectories of this launch (= B * Ms)
  int Ms, B;              // sample indices owned by this handle; number of starting points evaluated in one launch (trajectory m = b * Ms + sample)
  const double* x0_batch; // [B][d] starting points when B > 1 (else x0[] below)
  int hp1;                // third dimension of the normals tensor
  int mode, flags, ntheta;
  // model
  KernelSpec kern;
  int rule_id;
  double sigma_tol, sigma_n2, k0, d2k0, ymin_base;
  double m52_c;           // sqrt(5) / length-scale (Matern-5/2 fast path)
  double fmini, theta1, htol;
  rbo_solver_opts so;
  double x0[RBO_MAXD], lbs[RBO_MAXD], ubs[RBO_MAXD];
  // resident inputs (device)
  const double* Xb;      // [d][N8] coordinate-major base locations (pad columns 0)
  const double* yb;      // [N]
  const double* c0;      // [N8] base coefficients K^-1 y (pad 0)
  const double* u0;      // [N8] L0^-1 y (pad 0)
  const double* Lf;      // forward panels of L0^-1, k-major (staged through the shared-memory ring)
  const double* Lb;      // backward (transposed) panels of L0^-1, k-major (staged through the shared-memory ring)
  const double* Lbf;     // the same panels in mma A-fragment order (read straight from L2 by the few-column backward pass)
  const double* rn;      // [M][(d+1)][hp1] column-major (sample fastest)
  const double* starts;  // [S][d]
  const double* dual_dirs;  // [M][h][d] or nullptr
  const double* x_forced;   // [M][h][d] or nullptr
  const double* gh_nodes;   // [M][gh_depth] Gauss-Hermite nodes per sample and step (RBO_FLAG_GAUSS_HERMITE)
  const double* gh_weights; // [M][gh_depth]
  int gh_depth;
  // outputs (device)
  double* values;      // [M]
  double* grad_x;      // [M][d]
  double* grad_theta;  // [M][ntheta]
  int* best_index;     // [M]
  int* grad_case;      // [M]
  int* status;         // [M]
  double* xs;          // [M][h+1][d]
  double* ys;          // [M][h+1]
  double* gys;         // [M][h+1][d]
  double* alphas;      // [M][h]
  int* n_evals;        // [M][h]
  int* start_status;   // [M][h][S]
  int* start_iters;    // [M][h][S]
  double *t_mu, *t_sigma, *t_dmu, *t_dsigma, *t_Halpha;  // extended tape (RBO_FLAG_TAPE_EX): [M][h], [M][h], [M][h][d], [M][h][d], [M][h][d*d]
  int* work_counter;   // the work counter record: scheduler and watchdog (WorkCounterIndex)
  const int* order;    // [M] trajectories in the order they are handed out (longest first, from the previous launch) or nullptr
  unsigned long long* cta_done;  // [gridDim.x] %globaltimer at the end of each CTA (tail of the persistent grid)
  double* cs_tape;     // [gridDim.x][h+2][NR] coefficient tape of the trajectory each CTA is working on
  SmemPlan pl;         // make_plan(...) evaluated on the host: the offsets are then constant-bank operands in the kernel
};

__host__ __device__ inline int ncols_adjoint(int d) { return 4 * (d + 1) + 2; }
__host__ __device__ inline int npairs_max(int d, int W) {
  int q1 = d + 1, a = W * q1 * (q1 + 1), b = 2 * q1 * q1 + 2 * q1;  // outputs of the largest column-product call
  return a > b ? a : b;
}

__host__ __device__ inline SmemPlan make_plan(int d, int N8, int h, int W, int RP, int NR, int RSmax, int NPmax, int xsm, int RSh, int vglob = 0, int S = 0) {
  SmemPlan p;
  int o = 0;
  auto take = [&](int n) { int r = o; o += (n + 1) & ~1; return r; };  // keep 16-byte alignment
  const int dd = d * d, q1 = d + 1, T2 = d * (d + 1) / 2;
  p.V = take(vglob ? 0 : NR * RP);  // large-n variant: the work matrix lives in a per-CTA global scratch (L2-resident)
  p.Fp = take((N8 + RBO_MAXFAN) * RBO_PR);
  p.G = take(RBO_MAXFAN * RBO_MAXFAN);
  p.u = take(NR);
  p.Xf = take(RBO_MAXFAN * d);
  p.yf = take(RBO_MAXFAN);
  p.gyf = take(RBO_MAXFAN * d);
  p.Xs = take(xsm ? d * (N8 + 1) : 0);
  p.stage = take(RBO_NSTAGE * RBO_CHUNK_K * RBO_LP);
  p.mbar = take(2 * RBO_NSTAGE + 2);
  p.sx = take(W * d); p.sxt = take(W * d); p.sg = take(W * d); p.sH = take(W * dd); p.sp = take(2);
  p.sHt = take(W * dd); p.sHref = take(dd); p.sga = take(W * d); p.sdmu = take(W * d); p.sdsig = take(W * d); p.sgh = take(W * 8);
  p.sf = take(W); p.slam = take(W); p.spred = take(W); p.shs = take(W); p.ssn = take(W);
  p.ppre = take(RSmax * W * q1);
  p.ppost = take(RSmax * NPmax);
  p.phess = take(RSh * W * 2 * (T2 + 1));
  p.bestx = take(d);
  p.misc = take(64 + 2 * q1 * q1 + 2 * q1);
  p.adj = take(19 * d + 32);
  p.sbnd = take(2 * d);
  p.sord = take((6 * S + 7) / 8);
  p.pairs = take((6 * (W + 2) + 1) / 2);  // product items
  p.tbl = take((T2 + 2) / 2 + 1);
  p.ints = take(64 + 10 * W + 32 * W / 2 + (ncols_adjoint(d) + W * q1 + 1) / 2);
  p.total = o;
  return p;
}

}  // namespace rbo
