// sga_kernels.cu -- the per-iteration kernels of rbo_stochastic_solve_batch (include/rbo.h): stochastic_solve (utils.jl:235-265)
// from a batch of restarts with no host round trip. One iteration is
//   rbo_sga_worklist_kernel -> the rollout kernel (unchanged) -> rbo_sga_step_kernel [-> rbo_lpt_order_kernel].
// The rollout kernel hands out P.order[i] and ends a CTA at the first entry >= P.M, so the work list below (the live restarts'
// trajectories, then the sentinel M) is all it takes to stop restarts on the device.
#include "sga_kernels.cuh"

namespace rbo {

// Work list of the next rollout launch: the trajectories of the live restarts in the order of `order` (the longest-first order of
// the previous launch) or in index order, then the sentinel M up to M entries. One CTA; stable, so the list is deterministic.
__global__ void __launch_bounds__(1024) rbo_sga_worklist_kernel(const int* __restrict__ order, const int* __restrict__ live, int Ms, int M,
                                                                int* __restrict__ list) {
  __shared__ int wofs[32];
  __shared__ int s_total;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
  int base = 0;
  for (int i0 = 0; i0 < M; i0 += blockDim.x) {
    const int i = i0 + tid;
    const int m = i < M ? (order ? order[i] : i) : 0;
    const bool keep = i < M && live[m / Ms] != 0;
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) wofs[w] = __popc(bal);
    __syncthreads();
    if (tid == 0) {
      int run = 0;
      for (int j = 0; j < nw; ++j) { const int c = wofs[j]; wofs[j] = run; run += c; }
      s_total = run;
    }
    __syncthreads();
    if (keep) list[base + wofs[w] + __popc(bal & ((1u << lane) - 1u))] = m;
    base += s_total;
    __syncthreads();  // wofs / s_total are rewritten by the next chunk
  }
  for (int i = base + tid; i < M; i += blockDim.x) list[i] = M;
}

// numpy's float64 sum of n < 128 terms t(0..n-1) (pairwise_sum: sequential below 8 terms, otherwise eight interleaved partial sums
// combined pairwise, then the remainder; the reduction starts from the identity 0.0), without contractions.
template <class F>
__device__ double numpy_sum(int n, F t) {
  double res;
  if (n < 8) {
    res = 0.0;
    for (int i = 0; i < n; ++i) res = __dadd_rn(res, t(i));
  } else {
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = t(j);
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], t(i + j));
    }
    res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, t(i));
  }
  return __dadd_rn(0.0, res);
}

// One CTA per restart b, after the rollout of iteration k (0-based): the estimate over the restart's Ms trajectories (two-pass mean
// and corrected std of the values and of every grad_x row, failed trajectories excluded and counted, the first failing sample),
// the history entry, the stop tests and the optimiser step of api.update_optimizer. Stopped restarts return at once.
constexpr int SGA_THREADS = 256;
__global__ void __launch_bounds__(SGA_THREADS) rbo_sga_step_kernel(const __grid_constant__ SgaProblem S, int k) {
  __shared__ double red[SGA_THREADS / 32];
  __shared__ int ired[SGA_THREADS / 32][2];
  __shared__ double s_mean[RBO_MAXD + 1], s_std[RBO_MAXD + 1];
  __shared__ double s_bc;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int* wc = S.work_counter;
  // kernel watchdog: the memset before each rollout launch clears work_counter[1..2]; a flag seen once stops every restart
  if (S.sticky[0] != 0 || wc[1] != 0 || wc[2] != 0) {
    if (tid == 0) {
      if (b == 0 && S.sticky[0] == 0) {
        for (int i = 1; i <= 8; ++i) S.sticky[i] = wc[i];
        S.sticky[0] = 1;
      }
      S.live[b] = 0;
    }
    return;
  }
  if (!S.live[b]) return;
  const int Ms = S.Ms, d = S.d;
  const size_t t0 = (size_t)b * Ms;

  // fixed-shape reductions (lane butterfly, then the warps in order): the result does not depend on timing
  auto block_sum = [&](double acc) -> double {
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) red[w] = acc;
    __syncthreads();
    if (tid == 0) {
      double tot = 0.0;
      for (int j = 0; j < SGA_THREADS / 32; ++j) tot += red[j];
      s_bc = tot;
    }
    __syncthreads();
    const double tot = s_bc;
    __syncthreads();  // red / s_bc are reused by the next call
    return tot;
  };

  int nf = 0, first = Ms;
  for (int s = tid; s < Ms; s += SGA_THREADS)
    if (S.status[t0 + s] != 0) { ++nf; first = min(first, s); }
  for (int off = 16; off > 0; off >>= 1) {
    nf += __shfl_xor_sync(0xffffffffu, nf, off);
    first = min(first, __shfl_xor_sync(0xffffffffu, first, off));
  }
  if (lane == 0) { ired[w][0] = nf; ired[w][1] = first; }
  __syncthreads();
  nf = 0; first = Ms;
  for (int j = 0; j < SGA_THREADS / 32; ++j) { nf += ired[j][0]; first = min(first, ired[j][1]); }
  const double nok = (double)(Ms - nf);

  // rollout.jl:328-337 per restart: mean, then the centred sum of squares (two-pass), corrected std
  for (int row = 0; row <= d; ++row) {
    const double* base = row == 0 ? S.values + t0 : S.grad_x + t0 * d + (row - 1);
    const size_t stride = row == 0 ? 1 : d;
    double acc = 0.0;
    for (int s = tid; s < Ms; s += SGA_THREADS)
      if (S.status[t0 + s] == 0) acc += base[s * stride];
    const double mean = block_sum(acc) / nok;
    acc = 0.0;
    for (int s = tid; s < Ms; s += SGA_THREADS)
      if (S.status[t0 + s] == 0) { const double e = base[s * stride] - mean; acc += e * e; }
    const double m2 = block_sum(acc);
    if (tid == 0) { s_mean[row] = mean; s_std[row] = sqrt(m2 / (nok - 1.0)); }
  }
  if (tid != 0) return;

  // history, then the stop tests and the step (utils.jl:245-262)
  const size_t hk = (size_t)b * S.maxit + k;
  double* x = S.x + (size_t)b * d;
  for (int a = 0; a < d; ++a) {
    S.xh[hk * d + a] = x[a];
    S.gmh[hk * d + a] = s_mean[1 + a];
    S.gsh[hk * d + a] = s_std[1 + a];
  }
  S.mh[hk] = s_mean[0];
  S.sh[hk] = s_std[0];
  S.n_iter[b] = k + 1;
  S.nfail[b] = nf;
  int stop = -1;
  if (nf > 0) {
    // the serial reference throws at the first failing sample
    stop = RBO_SGA_FAILED;
    S.fail[2 * b] = first;
    S.fail[2 * b + 1] = S.status[t0 + first];
  } else if (S.use_eswavs) {
    // early_stopping_without_a_validation_set (utils.jl:114-123) as api.eswavs(g, std**2, M) evaluates it
    const double ratio = numpy_sum(d, [&](int a) {
      const double g = s_mean[1 + a], sd = s_std[1 + a];
      return __ddiv_rn(__dmul_rn(g, g), __dmul_rn(sd, sd));
    });
    const double lhs = __dadd_rn(1.0, -__dmul_rn(__ddiv_rn((double)Ms, (double)d), ratio));
    if (lhs > 0.0) stop = RBO_SGA_ESWAVS;
  }
  if (stop < 0) {
    // update!(optimizer; x, grad_f) (optimizers.jl:16-22, 48-75) in api.update_optimizer's operation order
    double* m = S.m + (size_t)b * d;
    double* v = S.v + (size_t)b * d;
    const double bc1 = S.bias[k], bc2 = S.bias[S.maxit + k];
    for (int a = 0; a < d; ++a) {
      const double g = s_mean[1 + a];
      double xa = x[a];
      if (S.optimizer == RBO_OPT_SGA) {
        xa = __dadd_rn(xa, __dmul_rn(S.eta, g));
      } else {
        const double ma = __dadd_rn(__dmul_rn(S.beta1, m[a]), __dmul_rn(S.omb1, g));
        const double va = __dadd_rn(__dmul_rn(S.beta2, v[a]), __dmul_rn(S.omb2, __dmul_rn(g, g)));
        m[a] = ma;
        v[a] = va;
        const double mhat = __ddiv_rn(ma, bc1), vhat = __ddiv_rn(va, bc2);
        xa = __dadd_rn(xa, __ddiv_rn(__dmul_rn(S.eta, mhat), __dadd_rn(__dsqrt_rn(vhat), S.eps)));
      }
      if (S.project) xa = xa < S.lbs[a] ? S.lbs[a] : (xa > S.ubs[a] ? S.ubs[a] : xa);  // np.clip (NaN stays NaN)
      x[a] = xa;
    }
    if (k + 1 == S.maxit) stop = RBO_SGA_MAXIT;
  }
  if (stop >= 0) {
    S.end_status[b] = stop;
    S.live[b] = 0;
  }
}

}  // namespace rbo
