// support_kernels.cu -- the small kernels around a rollout launch: normals and Sobol points, per-handle statistics, the
// longest-first order of the next launch, the vector of the multi-GPU all-reduce, and two diagnostics (the trust-region step on
// independent subproblems, the FP64 peak). Compiled once; the rollout kernel itself is in rollout_kernel.cu.
#include "support_kernels.cuh"
#include "trust_region.cuh"

namespace rbo {

// ----------------------------------------------------------------------------------------------------
// gen_low_discrepancy_sequence (utils.jl:65-74) on the device: Sobol (utils.jl:4-13, Joe-Kuo direction numbers,
// Gray-code order, origin skipped) -> Box-Muller with log10 and pair indexing (utils.jl:23-43, Q8) -> the
// column-major reshape(N, M, D, H) and removal of the padding coordinate.
// ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned sobol_point(const unsigned* dirs, int dim, unsigned k) {
  unsigned g = k ^ (k >> 1), x = 0;
  const unsigned* v = dirs + dim * 32;
  for (int b = 0; g != 0u; ++b, g >>= 1)
    if (g & 1u) x ^= v[b];
  return x;
}

__global__ void rbo_normals_kernel(const unsigned* __restrict__ dirs, double* __restrict__ out, int M_total, int d, int H, int m_begin, int m_count) {
  const int q1 = d + 1, D = q1 + ((q1 & 1) ? 1 : 0);
  const size_t total = (size_t)m_count * q1 * H;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    int ml = (int)(idx % m_count);
    int kq = (int)((idx / m_count) % q1);
    int t = (int)(idx / ((size_t)m_count * q1));
    size_t q = (size_t)(m_begin + ml) + (size_t)M_total * kq + (size_t)M_total * D * t;  // flat index into the D x (M*H) normals
    int coord = (int)(q % D);
    unsigned pnt = (unsigned)(q / D) + 1u;  // Sobol point index (the origin is skipped)
    int c0 = coord & ~1;                    // pair (c0, c0+1)
    double u1 = (double)sobol_point(dirs, c0, pnt) * (1.0 / 4294967296.0);
    double u2 = (double)sobol_point(dirs, c0 + 1, pnt) * (1.0 / 4294967296.0);
    double rad = sqrt(-2.0 * log10(u1));
    const double two_pi = 6.283185307179586;
    out[idx] = (coord & 1) ? rad * sin(two_pi * u2) : rad * cos(two_pi * u2);
  }
}

__global__ void rbo_sobol_kernel(const unsigned* __restrict__ dirs, unsigned* __restrict__ out_u32, double* __restrict__ out_f64, int dim, int npoints,
                                 const double* __restrict__ lbs, const double* __restrict__ ubs) {
  const size_t total = (size_t)dim * npoints;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    int a = (int)(idx % dim);
    unsigned pnt = (unsigned)(idx / dim) + 1u;
    unsigned x = sobol_point(dirs, a, pnt);
    if (out_u32) out_u32[idx] = x;
    if (out_f64) {
      double uu = (double)x * (1.0 / 4294967296.0);
      out_f64[idx] = lbs ? lbs[a] + (ubs[a] - lbs[a]) * uu : uu;
    }
  }
}

// Per-handle statistics of the last rollout, laid out as StatsLayout says (the rows two-pass: mean first, then centred squares --
// rollout.jl:328-337). One CTA; M is at most a few 10^5.
__global__ void rbo_stats_kernel(const double* __restrict__ values, const double* __restrict__ gx, const double* __restrict__ gth,
                                 const int* __restrict__ n_evals, const int* __restrict__ best_index, const int* __restrict__ grad_case,
                                 const int* __restrict__ status, int M, int d, int nth, int h, double* __restrict__ sums) {
  __shared__ double red[32];
  __shared__ double s_mean;
  const int nrows = 1 + d + nth, nw = blockDim.x >> 5;
  const StatsLayout L(d, nth, h);
  auto block_sum = [&](double acc) -> double {
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    double tot = 0.0;
    for (int w = 0; w < nw; ++w) tot += red[w];
    return tot;
  };
  // trajectories that failed (status != 0: the reference would have thrown, SURVEY.md section 5) are excluded from n and from
  // every sum -- a half-factorised joint covariance yields finite garbage that must not leak into the estimate; their count is
  // reported next to the sums and travels through the same all-reduce (rbo_partial_sums_device)
  auto okay = [&](int i) { return !status || status[i] == 0; };
  double nok_acc = 0.0;
  for (int i = threadIdx.x; i < M; i += blockDim.x) nok_acc += okay(i) ? 1.0 : 0.0;
  const double nok = block_sum(nok_acc);
  for (int row = 0; row < nrows; ++row) {
    const double* base; int stride;
    if (row == 0) { base = values; stride = 1; }
    else if (row <= d) { base = gx ? gx + (row - 1) : nullptr; stride = d; }
    else { base = gth ? gth + (row - 1 - d) : nullptr; stride = nth; }
    double mean = 0.0, m2 = 0.0;
    if (base && nok > 0.0) {
      double acc = 0.0;
      for (int i = threadIdx.x; i < M; i += blockDim.x) if (okay(i)) acc += base[(size_t)i * stride];
      mean = block_sum(acc) / nok;
      if (threadIdx.x == 0) s_mean = mean;
      __syncthreads();
      mean = s_mean;
      acc = 0.0;
      for (int i = threadIdx.x; i < M; i += blockDim.x) if (okay(i)) { double v = base[(size_t)i * stride] - mean; acc += v * v; }
      m2 = block_sum(acc);
    }
    if (threadIdx.x == 0) {
      if (row == 0) sums[0] = nok;
      sums[1 + 3 * row + 0] = nok * mean;
      sums[1 + 3 * row + 1] = m2;
      sums[1 + 3 * row + 2] = nok * mean * mean;
    }
  }
  for (int j = 0; j < L.hist - L.evals; ++j) {
    double acc = 0.0;
    if (n_evals && h > 0) for (int i = threadIdx.x; i < M; i += blockDim.x) acc += n_evals[(size_t)i * h + j];
    double tot = block_sum(acc);
    if (threadIdx.x == 0) sums[L.evals + j] = tot;
  }
  for (int t = 0; t <= h + 1; ++t) {  // t = h + 1: the failed trajectories
    double acc = 0.0;
    for (int i = threadIdx.x; i < M; i += blockDim.x) {
      if (t <= h) acc += (grad_case && best_index && grad_case[i] == 3 && best_index[i] == t) ? 1.0 : 0.0;
      else acc += (status && status[i] != 0) ? 1.0 : 0.0;
    }
    double tot = block_sum(acc);
    if (threadIdx.x == 0) sums[t <= h ? L.hist + t : L.failed] = tot;
  }
}

// Longest-processing-time order for the NEXT launch on the same samples (common random numbers: the outer ascent loop and the
// bench re-evaluate the same trajectories at a nearby x0, so the evaluation counts of this launch predict the next one's costs):
// counting sort of the trajectories by descending cost. One CTA; ties in arbitrary order (scheduling only).
__global__ void rbo_lpt_order_kernel(const int* __restrict__ n_evals, const int* __restrict__ grad_case, const int* __restrict__ best_index, int M, int hh,
                                     int* __restrict__ order) {
  constexpr int NB = 2048;
  __shared__ int hist[NB];
  __shared__ int smax;
  auto cost = [&](int m) {
    int c = 1;
    for (int j = 0; j < hh; ++j) c += n_evals[(size_t)m * hh + j];
    if (grad_case[m] == 3) { const int t = best_index[m]; c += 2 * t * (t + 1); }  // the adjoint re-evaluates t policy solves with i perturbation solves each
    return c;
  };
  if (threadIdx.x == 0) smax = 1;
  for (int i = threadIdx.x; i < NB; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  int mx = 1;
  for (int m = threadIdx.x; m < M; m += blockDim.x) mx = max(mx, cost(m));
  atomicMax(&smax, mx);
  __syncthreads();
  const double scale = (double)(NB - 1) / (double)smax;
  for (int m = threadIdx.x; m < M; m += blockDim.x) atomicAdd(&hist[(int)(cost(m) * scale)], 1);
  __syncthreads();
  if (threadIdx.x == 0) {  // exclusive offsets in DESCENDING bucket order
    int run = 0;
    for (int b = NB - 1; b >= 0; --b) { const int c = hist[b]; hist[b] = run; run += c; }
  }
  __syncthreads();
  for (int m = threadIdx.x; m < M; m += blockDim.x) order[atomicAdd(&hist[(int)(cost(m) * scale)], 1)] = m;
}

// out = [the row block, number of failed trajectories, kernel watchdog flag]: the vector the multi-GPU all-reduce sums
__global__ void rbo_gather_sums_kernel(const double* __restrict__ sums, StatsLayout L, const int* __restrict__ work_counter, double* __restrict__ out) {
  for (int i = threadIdx.x; i < L.rows; i += blockDim.x) out[i] = sums[i];
  if (threadIdx.x == 0) { out[L.rows] = sums[L.failed]; out[L.rows + 1] = (work_counter[WC_STALL] || work_counter[WC_EVAL_CAP]) ? 1.0 : 0.0; }
}

// Diagnostic (rbo_tr_step_batch): the device code of the per-start trust-region step on B independent subproblems, one warp each,
// through the same dispatch as slot_logic_warp (registers for 2 <= n <= 16, shared memory otherwise). H: [B][n*n], g: [B][n],
// p: [B][n], hit: [B].
__global__ void rbo_tr_step_kernel(const double* H, const double* g, const double* Delta, int n, int B, double* p, int* hit) {
  extern __shared__ __align__(16) double trs[];
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5, w = threadIdx.x >> 5, b = blockIdx.x * wpb + w;
  if (b >= B) return;
  double* base = trs + (size_t)w * (2 * n * n + 4 * n + 32);
  double* Hs = base; double* A = Hs + n * n; double* gs = A + n * n; double* ta = gs + n; double* te = ta + n; double* yv = te + n;
  int* fr = reinterpret_cast<int*>(yv + n);
  for (int i = lane; i < n * n; i += 32) Hs[i] = H[(size_t)b * n * n + i];
  if (lane < n) { gs[lane] = g[(size_t)b * n + lane]; fr[lane] = lane; }
  __syncwarp();
  const bool h_ = (n >= 2 && n <= 16) ? tr_step16(Hs, gs, fr, n, n, Delta[b], ta, te, yv) : tr_step_warp(Hs, gs, fr, n, n, Delta[b], A, yv);
  if (lane < n) p[(size_t)b * n + lane] = yv[lane];
  if (lane == 0) hit[b] = h_ ? 1 : 0;
}

// FP64 FMA micro-benchmark: the roofline denominator for this path (MEASURED_PEAKS.json has no FP64 figure).
__global__ void rbo_fp64_peak_kernel(double* out, int iters) {
  double a[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = 1.0 + 1e-9 * (threadIdx.x + i);
  const double b = 1.0000001, c = 1e-9;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = fma(a[i], b, c);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += a[i];
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace rbo
