// support_kernels.cuh -- declarations of the kernels of support_kernels.cu (launched by rbo_api.cu).
#pragma once
#include "rbo_device.cuh"

namespace rbo {

// rbo_stats_kernel's vector for dimension d, nth hyper-parameters, horizon h: rows (n, then n*mean, M2, n*mean^2 per output row), evaluations
// per step (max(h, 1)), case-3 histogram over t = 0..h, failures. rbo_partial_sums_* gather the rows, the failures and the watchdog flag.
struct StatsLayout {
  int rows, evals, hist, failed, len, gathered;  // the row block's length; offsets; the lengths of both vectors
  __host__ __device__ StatsLayout(int d, int nth, int h)
      : rows(1 + 3 * (1 + d + nth)), evals(rows), hist(evals + (h > 1 ? h : 1)), failed(hist + h + 1), len(failed + 1), gathered(rows + 2) {}
};

__global__ void rbo_normals_kernel(const unsigned* dirs, double* out, int M_total, int d, int H, int m_begin, int m_count);
__global__ void rbo_sobol_kernel(const unsigned* dirs, unsigned* out_u32, double* out_f64, int dim, int npoints, const double* lbs, const double* ubs);
__global__ void rbo_stats_kernel(const double* values, const double* gx, const double* gth, const int* n_evals, const int* best_index, const int* grad_case,
                                 const int* status, int M, int d, int nth, int h, double* sums);
__global__ void rbo_lpt_order_kernel(const int* n_evals, const int* grad_case, const int* best_index, int M, int hh, int* order);
__global__ void rbo_gather_sums_kernel(const double* sums, StatsLayout L, const int* work_counter, double* out);
__global__ void rbo_tr_step_kernel(const double* H, const double* g, const double* Delta, int n, int B, double* p, int* hit);
__global__ void rbo_fp64_peak_kernel(double* out, int iters);

}  // namespace rbo
