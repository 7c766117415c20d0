// likelihood_kernels.cu -- the log marginal likelihood of the resident surrogate's data and its gradient in the kernel
// hyper-parameters (the objective of optimize!, rbs.jl:770-829), and the refactorisation of set_kernel! (rbs.jl:123-135), on the
// device in FP64. The O(N^3) work runs on the FP64 tensor cores (mma.sync m8n8k4, DMMA) in 64 x 64 tiles:
//
//   rbo_lik_assemble_kernel     K = [psi(|X_i - X_j|)] + sigma_n2 I from the resident sites (kern_eval: the matrix rbo_condition and the
//                               rollout kernel see), lower triangle, identity on the padding
//   rbo_lik_potrf_diag_kernel   K_kk = L_kk L_kk' in shared memory, and L_kk^-1; a non-positive pivot sets the status flag
//   rbo_lik_panel_kernel        L_ik = K_ik L_kk^-T                                  (DMMA)
//   rbo_lik_update_kernel       K_ij -= L_ik L_jk'  for the trailing lower tiles     (DMMA)
//   rbo_lik_trinv_row_kernel    block row i of W = L^-1: W_ij = -L_ii^-1 sum_{j<=k<i} L_ik W_kj   (DMMA)
//   rbo_lik_lauum_kernel        K^-1 = W'W, lower tiles                              (DMMA)
//   rbo_lik_grad_kernel         sum over j > k of (a_j a_k - K^-1_jk) dK_jk/dtheta, dK recomputed from X (no N x N dK stored)
//   rbo_lik_final_kernel        ll = -y'a/2 - sum log L_ii - N log(2 pi)/2 and the gradient, in a fixed reduction tree
//
// Every reduction runs in a fixed order and nothing is accumulated with atomics: repeated evaluations are bit for bit identical.
#include "likelihood_kernels.cuh"

namespace rbo {

namespace {
constexpr int LB = RBO_LK_B, KS = 16, SP = LB + 4;  // k-slab of the staged operands; pitch 68 = 4 (mod 16): conflict-free fragment reads
constexpr int NT = RBO_LK_THREADS;

// A GEMM operand: element (x, m) -- x = output row / column, m = summation index -- at p[m ld + x] (kmajor) or p[x ld + m].
struct Opnd {
  const double* p;
  int ld;
  bool kmajor;
};

// FP64 tensor-core tile: D(8x8) += A(8x4) * B(4x8). Lane l holds A[l >> 2][l & 3], B[l & 3][l >> 2], C[l >> 2][2 (l & 3) + {0, 1}].
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// The 64 x KS slab of an operand starting at summation index k0, four elements per thread (coalesced along the contiguous index).
__device__ __forceinline__ void load_slab(const Opnd& o, int k0, double (&r)[4]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int e = threadIdx.x + NT * q;
    r[q] = o.kmajor ? o.p[(size_t)(k0 + (e >> 6)) * o.ld + (e & 63)] : o.p[(size_t)(e >> 4) * o.ld + k0 + (e & 15)];
  }
}
// ... into shared memory, k-major with pitch SP
__device__ __forceinline__ void store_slab(bool kmajor, double* s, const double (&r)[4]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int e = threadIdx.x + NT * q;
    if (kmajor) s[(e >> 6) * SP + (e & 63)] = r[q];
    else s[(e & 15) * SP + (e >> 4)] = r[q];
  }
}

// Warp w owns rows 16 (w >> 1) + 8 rt + (lane >> 2) and columns 32 (w & 1) + 8 ct + 2 (lane & 3) + {0, 1} of the 64 x 64 tile.
using Acc = double[2][4][2];
__device__ __forceinline__ void acc_zero(Acc& acc) {
#pragma unroll
  for (int rt = 0; rt < 2; ++rt)
#pragma unroll
    for (int ct = 0; ct < 4; ++ct) acc[rt][ct][0] = acc[rt][ct][1] = 0.0;
}
// acc += sA' sB over one staged slab (sA: KS x 64 rows, sB: KS x 64 columns, both k-major)
__device__ __forceinline__ void mma_slab(Acc& acc, const double* sA, const double* sB) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, g = lane >> 2, tg = lane & 3, wr = 16 * (w >> 1), wc = 32 * (w & 1);
#pragma unroll
  for (int kk = 0; kk < KS; kk += 4) {
    double a[2], b[4];
#pragma unroll
    for (int rt = 0; rt < 2; ++rt) a[rt] = sA[(kk + tg) * SP + wr + 8 * rt + g];
#pragma unroll
    for (int ct = 0; ct < 4; ++ct) b[ct] = sB[(kk + tg) * SP + wc + 8 * ct + g];
#pragma unroll
    for (int rt = 0; rt < 2; ++rt)
#pragma unroll
      for (int ct = 0; ct < 4; ++ct) dmma(acc[rt][ct][0], acc[rt][ct][1], a[rt], b[ct]);
  }
}
// acc += sum_{m < K} A(r, m) B(c, m) (K a multiple of KS): one slab in shared memory while the next one is loaded into registers.
// Every global read of A and B has completed when this returns, so the caller may overwrite them.
__device__ void gemm_tile(Acc& acc, const Opnd& A, const Opnd& B, int K, double* sA, double* sB) {
  double ra[4], rb[4];
  load_slab(A, 0, ra);
  load_slab(B, 0, rb);
  for (int k0 = 0; k0 < K; k0 += KS) {
    __syncthreads();
    store_slab(A.kmajor, sA, ra);
    store_slab(B.kmajor, sB, rb);
    __syncthreads();
    if (k0 + KS < K) {
      load_slab(A, k0 + KS, ra);
      load_slab(B, k0 + KS, rb);
    }
    mma_slab(acc, sA, sB);
  }
}
enum Epi { EPI_SET, EPI_SUB, EPI_NEG };  // C = acc, C -= acc, C = -acc
template <Epi E>
__device__ __forceinline__ void store_tile(double* C, int ld, const Acc& acc) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, g = lane >> 2, tg = lane & 3, wr = 16 * (w >> 1), wc = 32 * (w & 1);
#pragma unroll
  for (int rt = 0; rt < 2; ++rt)
#pragma unroll
    for (int ct = 0; ct < 4; ++ct) {
      double* p = C + (size_t)(wr + 8 * rt + g) * ld + wc + 8 * ct + 2 * tg;
      for (int e = 0; e < 2; ++e) {
        if (E == EPI_SET) p[e] = acc[rt][ct][e];
        else if (E == EPI_SUB) p[e] -= acc[rt][ct][e];
        else p[e] = -acc[rt][ct][e];
      }
    }
}

// t-th tile of a lower block triangle, row by row: (i, j), j <= i
__device__ __forceinline__ void lower_tile(int t, int& i, int& j) {
  int r = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while ((r + 1) * (r + 2) / 2 <= t) ++r;
  while (r * (r + 1) / 2 > t) --r;
  i = r;
  j = t - r * (r + 1) / 2;
}
}  // namespace

// A[i][j] (i >= j, row-major, pitch NP) = psi(|X_i - X_j|), kdiag = psi(0) + sigma_n2 on the diagonal; identity on the padding
__global__ void rbo_lik_assemble_kernel(const double* __restrict__ Xpts, int d, int N, int NP, KernelSpec kern, double kdiag, double* __restrict__ A) {
  const size_t total = (size_t)NP * NP;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / NP), j = (int)(idx - (size_t)i * NP);
    if (j > i) continue;
    double v;
    if (i >= N) v = (i == j) ? 1.0 : 0.0;
    else if (i == j) v = kdiag;
    else {
      double rho2 = 0.0;
      for (int p = 0; p < d; ++p) {
        const double r = Xpts[(size_t)i * d + p] - Xpts[(size_t)j * d + p];
        rho2 = fma(r, r, rho2);
      }
      double dp, d2p;
      kern_eval(kern, sqrt(rho2), v, dp, d2p);
    }
    A[idx] = v;
  }
}

// Diagonal block kb: L_kk by a right-looking Cholesky in shared memory, then L_kk^-1 (thread c solves column c: no barrier).
// A non-positive or non-finite pivot sets status[0] = 1 (the host clears it) and continues with pivot 1 so that the rest stays finite.
__global__ void __launch_bounds__(NT) rbo_lik_potrf_diag_kernel(double* __restrict__ A, int NP, int kb, double* __restrict__ Dinv,
                                                                double* __restrict__ diagL, int* __restrict__ status) {
  extern __shared__ double sm_lk[];
  constexpr int P = LB + 1;
  double* s = sm_lk;
  double* X = sm_lk + LB * P;
  __shared__ int bad;
  const int t = threadIdx.x;
  double* Ad = A + (size_t)kb * LB * NP + (size_t)kb * LB;
  for (int e = t; e < LB * LB; e += NT) {
    const int r = e >> 6, c = e & 63;
    s[r * P + c] = c <= r ? Ad[(size_t)r * NP + c] : 0.0;
  }
  if (t == 0) bad = 0;
  __syncthreads();
  for (int j = 0; j < LB; ++j) {
    if (t == 0) {
      double p = s[j * P + j];
      if (!(p > 0.0) || !isfinite(p)) { bad = 1; p = 1.0; }
      s[j * P + j] = sqrt(p);
    }
    __syncthreads();
    if (t > j && t < LB) s[t * P + j] /= s[j * P + j];
    __syncthreads();
    for (int e = t; e < LB * LB; e += NT) {
      const int r = e >> 6, c = e & 63;
      if (c > j && r >= c) s[r * P + c] -= s[r * P + j] * s[c * P + j];
    }
    __syncthreads();
  }
  if (t < LB) {
    for (int r = t; r < LB; ++r) {
      double v = (r == t) ? 1.0 : 0.0;
      for (int m = t; m < r; ++m) v -= s[r * P + m] * X[m * P + t];
      X[r * P + t] = v / s[r * P + r];
    }
  }
  __syncthreads();
  if (t == 0 && bad) status[0] = 1;
  double* D = Dinv + (size_t)kb * LB * LB;
  for (int e = t; e < LB * LB; e += NT) {
    const int r = e >> 6, c = e & 63;
    if (c <= r) Ad[(size_t)r * NP + c] = s[r * P + c];
    D[e] = c <= r ? X[r * P + c] : 0.0;
  }
  if (t < LB) diagL[kb * LB + t] = s[t * P + t];
}

// L_ik = A_ik L_kk^-T for the block rows i > kb (in place)
__global__ void __launch_bounds__(NT) rbo_lik_panel_kernel(double* __restrict__ A, int NP, int kb, const double* __restrict__ Dinv) {
  __shared__ double sA[KS * SP], sB[KS * SP];
  double* C = A + (size_t)(kb + 1 + blockIdx.x) * LB * NP + (size_t)kb * LB;
  Acc acc;
  acc_zero(acc);
  gemm_tile(acc, {C, NP, false}, {Dinv + (size_t)kb * LB * LB, LB, false}, LB, sA, sB);
  store_tile<EPI_SET>(C, NP, acc);
}

// A_ij -= L_ik L_jk' for kb < j <= i (the diagonal tiles in full; their upper halves are never read)
__global__ void __launch_bounds__(NT) rbo_lik_update_kernel(double* __restrict__ A, int NP, int kb) {
  __shared__ double sA[KS * SP], sB[KS * SP];
  int i, j;
  lower_tile(blockIdx.x, i, j);
  i += kb + 1;
  j += kb + 1;
  Acc acc;
  acc_zero(acc);
  gemm_tile(acc, {A + (size_t)i * LB * NP + (size_t)kb * LB, NP, false}, {A + (size_t)j * LB * NP + (size_t)kb * LB, NP, false}, LB, sA, sB);
  store_tile<EPI_SUB>(A + (size_t)i * LB * NP + (size_t)j * LB, NP, acc);
}

// Block row i of W = L^-1 (plain FP64; rows < i are done): W_ii = L_ii^-1, W_ij = -L_ii^-1 (sum_{j <= k < i} L_ik W_kj) for j < i.
__global__ void __launch_bounds__(NT) rbo_lik_trinv_row_kernel(const double* __restrict__ A, int NP, int i, const double* __restrict__ Dinv,
                                                               double* __restrict__ W) {
  __shared__ double sm[(KS + LB) * SP];  // two slabs during the sum; then one slab and T (64 x 64, k-major)
  const int j = blockIdx.x;
  double* Wij = W + (size_t)i * LB * NP + (size_t)j * LB;
  const double* Di = Dinv + (size_t)i * LB * LB;
  if (j == i) {
    for (int e = threadIdx.x; e < LB * LB; e += NT) Wij[(size_t)(e >> 6) * NP + (e & 63)] = Di[e];
    return;
  }
  Acc acc;
  acc_zero(acc);
  gemm_tile(acc, {A + (size_t)i * LB * NP + (size_t)j * LB, NP, false}, {W + (size_t)j * LB * NP + (size_t)j * LB, NP, true}, (i - j) * LB,
            sm, sm + KS * SP);
  double* sT = sm + KS * SP;
  __syncthreads();
  {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, g = lane >> 2, tg = lane & 3, wr = 16 * (w >> 1), wc = 32 * (w & 1);
#pragma unroll
    for (int rt = 0; rt < 2; ++rt)
#pragma unroll
      for (int ct = 0; ct < 4; ++ct) {
        sT[(wr + 8 * rt + g) * SP + wc + 8 * ct + 2 * tg] = acc[rt][ct][0];
        sT[(wr + 8 * rt + g) * SP + wc + 8 * ct + 2 * tg + 1] = acc[rt][ct][1];
      }
  }
  acc_zero(acc);
  for (int k0 = 0; k0 < LB; k0 += KS) {
    double ra[4];
    load_slab({Di, LB, false}, k0, ra);
    __syncthreads();
    store_slab(false, sm, ra);
    __syncthreads();
    mma_slab(acc, sm, sT + k0 * SP);
  }
  store_tile<EPI_NEG>(Wij, NP, acc);
}

// Kinv_ij = sum_{k >= i} W_ki' W_kj for the lower tiles j <= i of K^-1 = W'W
__global__ void __launch_bounds__(NT) rbo_lik_lauum_kernel(const double* __restrict__ W, int NP, double* __restrict__ Kinv) {
  __shared__ double sA[KS * SP], sB[KS * SP];
  int i, j;
  lower_tile(blockIdx.x, i, j);
  Acc acc;
  acc_zero(acc);
  gemm_tile(acc, {W + (size_t)i * LB * NP + (size_t)i * LB, NP, true}, {W + (size_t)i * LB * NP + (size_t)j * LB, NP, true}, NP - i * LB, sA, sB);
  store_tile<EPI_SET>(Kinv + (size_t)i * LB * NP + (size_t)j * LB, NP, acc);
}

// One lower tile of the trace: partial[2 t + p] = sum_{j > k in the tile} (a_j a_k - Kinv_jk) d psi(|X_j - X_k|) / d theta_p. The weight 2
// of an off-diagonal pair cancels the 1/2 of the gradient; the diagonal contributes nothing (psi(0) = 1 for every family).
__global__ void __launch_bounds__(NT) rbo_lik_grad_kernel(const double* __restrict__ Xpts, int d, int N, int NP, KernelSpec kern,
                                                          const double* __restrict__ a, const double* __restrict__ Kinv, double* __restrict__ partial) {
  __shared__ double red[2][NT];
  int bi, bj;
  lower_tile(blockIdx.x, bi, bj);
  const int t = threadIdx.x;
  double g0 = 0.0, g1 = 0.0;
  for (int e = t; e < LB * LB; e += NT) {
    const int gi = bi * LB + (e >> 6), gj = bj * LB + (e & 63);
    if (gi >= N || gj >= gi) continue;
    double rho2 = 0.0;
    for (int p = 0; p < d; ++p) {
      const double r = Xpts[(size_t)gi * d + p] - Xpts[(size_t)gj * d + p];
      rho2 = fma(r, r, rho2);
    }
    double dth[2];
    kern_dtheta(kern, sqrt(rho2), dth);
    const double w = a[gi] * a[gj] - Kinv[(size_t)gi * NP + gj];
    g0 = fma(w, dth[0], g0);
    g1 = fma(w, dth[1], g1);
  }
  red[0][t] = g0;
  red[1][t] = g1;
  __syncthreads();
  for (int s = NT / 2; s > 0; s >>= 1) {
    if (t < s) {
      red[0][t] += red[0][t + s];
      red[1][t] += red[1][t + s];
    }
    __syncthreads();
  }
  if (t == 0) {
    partial[2 * (size_t)blockIdx.x] = red[0][0];
    partial[2 * (size_t)blockIdx.x + 1] = red[1][0];
  }
}

// out[0] = ll, out[1 .. nk] = d ll / d theta (one block of 1024 threads, fixed tree)
__global__ void __launch_bounds__(1024) rbo_lik_final_kernel(const double* __restrict__ y, const double* __restrict__ a, const double* __restrict__ diagL,
                                                             int N, const double* __restrict__ partial, int ntiles, int nk, double* __restrict__ out) {
  __shared__ double red[4][1024];
  const int t = threadIdx.x;
  double ya = 0.0, ld = 0.0, g0 = 0.0, g1 = 0.0;
  for (int i = t; i < N; i += 1024) {
    ya = fma(y[i], a[i], ya);
    ld += log(diagL[i]);
  }
  for (int b = t; b < ntiles; b += 1024) {
    g0 += partial[2 * (size_t)b];
    g1 += partial[2 * (size_t)b + 1];
  }
  red[0][t] = ya; red[1][t] = ld; red[2][t] = g0; red[3][t] = g1;
  __syncthreads();
  for (int s = 512; s > 0; s >>= 1) {
    if (t < s)
      for (int q = 0; q < 4; ++q) red[q][t] += red[q][t + s];
    __syncthreads();
  }
  if (t == 0) {
    const double log2pi = 1.8378770664093453;
    out[0] = -0.5 * red[0][0] - red[1][0] - 0.5 * N * log2pi;
    out[1] = red[2][0];
    if (nk > 1) out[2] = red[3][0];
  }
}

// L (N x N column-major, ld = N: what rbo_trinv_kernel reads) from the factor in A; zero above the diagonal
__global__ void rbo_lik_to_colmajor_kernel(const double* __restrict__ A, int NP, int N, double* __restrict__ L) {
  const size_t total = (size_t)N * N;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(idx / N), i = (int)(idx - (size_t)k * N);
    L[idx] = i >= k ? A[(size_t)i * NP + k] : 0.0;
  }
}

}  // namespace rbo
