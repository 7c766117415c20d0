// trust_region.cuh -- the exact trust-region step of the per-start solver (DESIGN.md section 4), one warp per subproblem. Two
// versions of one algorithm, selected by problem size: tr_step16 keeps n <= 16 free coordinates in registers, tr_step_warp takes
// any n <= 32 in shared memory. Used by the rollout kernel and by the rbo_tr_step_batch diagnostic (support_kernels.cu).
//
// TR_T / TR_ADD are cycle-counter hooks: a file that feeds them (the rollout kernel built with RBO_PHASE_TIMERS) defines both
// before the include; everywhere else they expand to nothing.
#pragma once
#include "rbo_device.cuh"

#ifndef TR_T
#define TR_T(v)
#define TR_ADD(i, t0, t1)
#endif

namespace rbo {
namespace {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(FULL, v, off);
  return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v = fmin(v, __shfl_xor_sync(FULL, v, off));
  return v;
}

// ------------------------------------------------------------------------------------------------
// Exact trust-region step by one warp for n <= 16 free coordinates (solve_tr, optim.jl:9-51; same algorithm and candidate grid
// as oracle/rbo_oracle.cpp::tr_step and as tr_step_warp below, which stays the path for n > 16). The per-start logic is a latency
// chain on one warp while the rest of the CTA waits (FP64: 8.4 cycles per dependent FMA, 118 per division, 86 per sqrt, ~45 per
// shared-memory load on B200, profiles/r3_lat_bench.txt), so this version keeps everything in REGISTERS: lane l owns row l >> 1,
// columns 8 (l & 1) .. +7 of the (zero-padded) 16 x 16 matrix and of the accumulated orthogonal factor Q; the k loop of the
// Householder tridiagonalisation is fully unrolled (static register indices), the reflector column is fetched from row k's lanes
// by shuffles (A is symmetric), the row sums are 8 local FMAs + one exchange with the partner lane, the reflector is normalised
// with rsqrt + one reciprocal instead of sqrt + division, and Q <- Q (I - beta v v') rides along off the critical path so that
// Q'g and p = Q h are single products (no serial loop over the reflectors).
//   H, g: d x d / d (shared memory); fr[0..n): free coordinates; ta, te, yv: >= n doubles each (diagonal / sub-diagonal of T,
//   Q'g then the step). Returns "hit_constraint"; the step p is left in yv[0..n).
// ------------------------------------------------------------------------------------------------
// Branch-free reciprocal / reciprocal square root for NORMAL positive arguments (no special cases; ~1 ulp). The library versions end
// in a slow-path branch that keeps the compiler from interleaving independent chains (the two candidate shifts of a lane ran one
// after the other: 310 cycles per pivot instead of ~90, profiles/r3_tr_bench.txt).
__device__ __forceinline__ double rcp_fast(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  return fma(r, e, r);
}
__device__ __forceinline__ double rsqrt_fast(double x) {
  double r;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  const double e = fma(-x, r * r, 1.0);  // 1 - x r^2
  return fma(r * e, fma(0.375, e, 0.5), r);
}
__device__ __forceinline__ double rowsum16(double v) {  // sum over the 16 rows; the two lanes of a row hold the same value
  v += __shfl_xor_sync(FULL, v, 2); v += __shfl_xor_sync(FULL, v, 4); v += __shfl_xor_sync(FULL, v, 8); v += __shfl_xor_sync(FULL, v, 16);
  return v;
}
// Two candidate shifts per lane: 0 = admissible, 1 = positive definite but |h(lam)| > Delta, 2 = not positive definite.
// Forward LDL' recurrences of T + lam I (pivots d_i, z = L^-1 b) and their lam-derivatives (d_i', z_i'), no storage:
// |h(lam)|^2 = b'(T + lam I)^-2 b = -d/dlam sum z_i^2 / d_i = sum q_i (q_i d_i' - 2 z_i'), q_i = z_i / d_i.
__device__ __forceinline__ void tri_probe2_t(const double* ta, const double* te, const double* yv, int n, double lamA, double lamB, double D2, int& outA, int& outB) {
  const double lam[2] = {lamA, lamB};
  double q[2], r[2], dd[2], zd[2], acc[2];
  bool ok[2];
  const double b0 = yv[0], a0 = ta[0];
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const double dn = a0 + lam[c];
    ok[c] = dn > 0.0; r[c] = rcp_fast(dn); dd[c] = 1.0; zd[c] = 0.0; q[c] = b0 * r[c]; acc[c] = q[c] * q[c];
  }
#pragma unroll 2
  for (int i = 1; i < n; ++i) {
    const double e = te[i - 1], a = ta[i], b = yv[i];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const double er = e * r[c], dn = fma(-e, er, a + lam[c]);
      const double ddn = fma(er * er, dd[c], 1.0), zn = fma(-e, q[c], b), zdn = er * fma(q[c], dd[c], -zd[c]);
      ok[c] = ok[c] && dn > 0.0;
      r[c] = rcp_fast(dn);
      q[c] = zn * r[c];
      acc[c] = fma(q[c], fma(q[c], ddn, -2.0 * zdn), acc[c]);
      dd[c] = ddn; zd[c] = zdn;
    }
  }
  outA = ok[0] ? (acc[0] <= D2 ? 0 : 1) : 2;
  outB = ok[1] ? (acc[1] <= D2 ? 0 : 1) : 2;
}
// lane i: component i of -(T + lam I)^-1 b, b[0..n) in shared memory; the pivots must be positive
__device__ __forceinline__ double tri_solve_dist_t(const double* ta, const double* te, const double* b, int n, double lam, int lane) {
  double myr = 0.0, myz = 0.0, r = 0.0, z = 0.0;
  for (int i = 0; i < n; ++i) {
    const double bi = b[i];
    if (i == 0) { r = rcp_fast(ta[0] + lam); z = bi; }
    else { const double e = te[i - 1], er = e * r; r = rcp_fast(fma(-e, er, ta[i] + lam)); z = fma(-er, z, bi); }
    if (lane == i) { myr = r; myz = z; }
  }
  const double e_up = (lane + 1 < n) ? te[lane] : 0.0;
  double hv = 0.0;
  for (int i = n - 1; i >= 0; --i) {
    const double hn = __shfl_sync(FULL, hv, (i + 1) & 31);
    if (lane == i) hv = (myz - ((i + 1 < n) ? e_up * hn : 0.0)) * myr;
  }
  return -hv;
}
__device__ __noinline__ bool tr_step16(const double* H, const double* g, const int* fr, int n, int d, double Delta, double* ta, double* te, double* yv) {
  // the lane id is read through a volatile asm so that nothing derived from it is hoisted out of the solver loop and kept live
  // across the tensor-core phases (the kernel sits at the 128-register cap)
  int lane;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
  const int row = lane >> 1, hf = lane & 1, c0 = 8 * hf;
  const bool rin = row < n;
  const int fi = rin ? fr[row] : 0;
  TR_T(q0_);
  double a[8], Q[8];  // my 8 columns of the matrix row and of the row of Q
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int j = c0 + c;
    a[c] = 0.0;
    if (rin && j < n) a[c] = H[fi * d + fr[j]];
    Q[c] = (row == j) ? 1.0 : 0.0;
  }
  const double gi = rin ? g[fi] : 0.0;
  const double gn = sqrt(rowsum16(gi * gi));
  TR_T(q1_); TR_ADD(4, q0_, q1_);
  // ---- Householder tridiagonalisation H_FF = Q T Q'. Step k with x = column k below the diagonal,
  // v = x - alpha e1, beta = 2 / |v|^2, p = beta A v, w = p - (beta p'v / 2) v, A <- A - v w' - w v'. A warp shuffle costs ~45 cycles
  // of latency and ~5-8 of issue on B200 (profiles/r3_shfl_bench.txt): the step is arranged for the fewest shuffles (24 doubles).
#pragma unroll
  for (int k = 0; k < 14; ++k) {
    if (k + 2 < n) {
      // column k below the diagonal = row k right of the diagonal: fetched from row k's lanes
      double v[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) { const double t = __shfl_sync(FULL, a[c], 2 * k + hf); v[c] = (c0 + c > k) ? t : 0.0; }
      double vi = __shfl_sync(FULL, a[k & 7], (lane & ~1) | (k >> 3));  // A[row][k]
      if (row <= k) vi = 0.0;
      const double x0 = __shfl_sync(FULL, a[(k + 1) & 7], 2 * k + ((k + 1) >> 3));            // A[k][k+1]
      const double aik1 = __shfl_sync(FULL, a[(k + 1) & 7], (lane & ~1) | ((k + 1) >> 3));    // A[row][k+1]
      const double qk1 = __shfl_sync(FULL, Q[(k + 1) & 7], (lane & ~1) | ((k + 1) >> 3));     // Q[row][k+1]
      double s0 = 0.0, s1 = 0.0, t0 = 0.0, t1 = 0.0, u0 = 0.0, u1 = 0.0;
#pragma unroll
      for (int c = 0; c < 8; c += 2) {
        s0 = fma(v[c], v[c], s0); s1 = fma(v[c + 1], v[c + 1], s1);
        t0 = fma(a[c], v[c], t0); t1 = fma(a[c + 1], v[c + 1], t1);
        u0 = fma(Q[c], v[c], u0); u1 = fma(Q[c + 1], v[c + 1], u1);
      }
      const double sl = s0 + s1, tl = t0 + t1, ul = u0 + u1;
      const double xn2 = sl + __shfl_xor_sync(FULL, sl, 1);
      const double traw = tl + __shfl_xor_sync(FULL, tl, 1);  // (A x)_row
      const double uraw = ul + __shfl_xor_sync(FULL, ul, 1);  // (Q x)_row
      if (!(xn2 - x0 * x0 > 0.0)) continue;                   // column already reduced (uniform)
      const double rs = rsqrt_fast(xn2), sq = xn2 * rs;        // |x|
      const double alpha = x0 > 0.0 ? -sq : sq;
      const double bk = rcp_fast(fma(fabs(x0), sq, xn2));      // beta = 2 / |x - alpha e1|^2
      const double v1 = x0 - alpha;
      if (row == k + 1) vi = v1;
      if (((k + 1) >> 3) == hf) v[(k + 1) & 7] = v1;
      const double pw = (row > k) ? bk * fma(-aik1, alpha, traw) : 0.0;  // beta (A v)_row, A v = A x - alpha A[:, k+1]
      double w[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) w[c] = __shfl_sync(FULL, pw, 2 * (c0 + c));  // p_j for my columns
      double q0 = 0.0, q1 = 0.0;
#pragma unroll
      for (int c = 0; c < 8; c += 2) { q0 = fma(w[c], v[c], q0); q1 = fma(w[c + 1], v[c + 1], q1); }
      const double ql = q0 + q1;
      const double pv = ql + __shfl_xor_sync(FULL, ql, 1);
      const double nkk = -0.5 * bk * pv, wi = fma(nkk, vi, pw);
#pragma unroll
      // The update must keep A BITWISE symmetric (the reflector column is read from row k): v_i w_j + w_i v_j is formed from two
      // rounded products and one commutative addition, never contracted into FMAs. With a merely approximately symmetric A the
      // two copies of a rounding-noise column differ by O(1) relative and the transformation stops being a similarity -- that
      // corrupted the near-zero eigenvalues of rank-deficient Hessians (tests: test_trust_region_step_matches_the_oracle_step).
      for (int c = 0; c < 8; ++c) { const double wj = fma(nkk, v[c], w[c]); a[c] = __dsub_rn(a[c], __dadd_rn(__dmul_rn(vi, wj), __dmul_rn(wi, v[c]))); }
      if (lane == 2 * (k + 1) + (k >> 3)) a[k & 7] = alpha;                       // sub-diagonal of T
      // Q <- Q (I - beta v v'): off the critical path
      const double tq = bk * fma(-qk1, alpha, uraw);
#pragma unroll
      for (int c = 0; c < 8; ++c) Q[c] = fma(-tq, v[c], Q[c]);
    }
  }
  TR_T(q2_); TR_ADD(5, q1_, q2_);
  // T and Q'g to shared memory: every lane needs all of them for the shift search
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int j = c0 + c;
    if (row == j && rin) ta[row] = a[c];
    if (row == j + 1 && rin) te[j] = a[c];
  }
  {
    // (Q'g)_j = sum over the rows of Q[row][j] g_row as a reduce-scatter: every round halves the columns a lane keeps and doubles
    // the rows they cover (8 double shuffles instead of 32); the lane ends with column c0 + 4 b4 + 2 b3 + b2 (bK = bit K of the lane)
    const bool b4 = (lane & 16) != 0, b3 = (lane & 8) != 0, b2 = (lane & 4) != 0;
    double k4[4], k2[2];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const double lo_ = Q[c] * gi, hi_ = Q[c + 4] * gi;
      k4[c] = (b4 ? hi_ : lo_) + __shfl_xor_sync(FULL, b4 ? lo_ : hi_, 16);
    }
#pragma unroll
    for (int c = 0; c < 2; ++c) k2[c] = (b3 ? k4[c + 2] : k4[c]) + __shfl_xor_sync(FULL, b3 ? k4[c] : k4[c + 2], 8);
    double k1 = (b2 ? k2[1] : k2[0]) + __shfl_xor_sync(FULL, b2 ? k2[0] : k2[1], 4);
    k1 += __shfl_xor_sync(FULL, k1, 2);
    const int j = c0 + (b4 ? 4 : 0) + (b3 ? 2 : 0) + (b2 ? 1 : 0);
    if ((lane & 2) == 0 && j < n) yv[j] = k1;
  }
  __syncwarp();
  const bool in = lane < n;
  double glo = INFINITY;
  if (in) glo = ta[lane] - (lane > 0 ? fabs(te[lane - 1]) : 0.0) - (lane + 1 < n ? fabs(te[lane]) : 0.0);
  glo = warp_min(glo);  // Gershgorin lower bound of lambda_min(T)
  const double D2 = Delta * Delta;
  double lo = 0.0, hi = fmax(0.0, -glo) + gn / Delta;
  bool hit = true, lo_notpd = false;
  TR_T(q3_); TR_ADD(6, q2_, q3_);
  for (int round = 0; round < RBO_TR_ROUNDS; ++round) {
    // 64 candidates per round, two per lane (c = lane, lane + 32); the last one is hi, known to be admissible
    const double base = lo, wd = hi - lo;
    const double lamA = (round == 0) ? wd * (double)lane / 63.0 : base + wd * (double)(lane + 1) / 64.0;
    const double lamB = (round == 0) ? wd * (double)(lane + 32) / 63.0 : base + wd * (double)(lane + 33) / 64.0;
    int oa, ob;
    tri_probe2_t(ta, te, yv, n, lamA, lamB, D2, oa, ob);
    const unsigned long long adm = ((unsigned long long)__ballot_sync(FULL, ob == 0) << 32) | __ballot_sync(FULL, oa == 0) | (1ull << 63);
    const unsigned long long pdm = ((unsigned long long)__ballot_sync(FULL, ob != 2) << 32) | __ballot_sync(FULL, oa != 2);
    const int cf = __ffsll((long long)adm) - 1;
    if (round == 0) {
      if (cf == 0) { hi = 0.0; hit = false; break; }
      lo_notpd = ((pdm >> (cf - 1)) & 1ull) == 0ull;
      hi = (cf == 63) ? hi : wd * (double)cf / 63.0;
      lo = wd * (double)(cf - 1) / 63.0;
    } else {
      if (cf > 0) lo_notpd = ((pdm >> (cf - 1)) & 1ull) == 0ull;
      hi = (cf == 63) ? hi : base + wd * (double)(cf + 1) / 64.0;
      lo = (cf == 0) ? base : base + wd * (double)cf / 64.0;
    }
  }
  TR_T(q4_); TR_ADD(7, q3_, q4_);
  double h = tri_solve_dist_t(ta, te, yv, n, hi, lane);
  if (hit && lo_notpd) {
    const double hn2 = warp_sum(in ? h * h : 0.0);
    if (hn2 < D2) {  // hard case (to the resolution of the search): complete along the lowest eigenvector of T
      __syncwarp();
      if (in) yv[lane] = 1.0;
      __syncwarp();
      double z = 0.0;
      for (int itn = 0; itn < 2; ++itn) {
        const double z2 = tri_solve_dist_t(ta, te, yv, n, hi, lane);
        const double zn = 1.0 / sqrt(warp_sum(in ? z2 * z2 : 0.0));
        z = in ? z2 * zn : 0.0;
        __syncwarp();
        if (in) yv[lane] = z;
        __syncwarp();
      }
      const double hz = warp_sum(in ? h * z : 0.0);
      const double tau = -hz + sqrt(fmax(hz * hz + (D2 - hn2), 0.0));
      h += tau * z;
    }
  }
  TR_T(q5_); TR_ADD(8, q4_, q5_);
  // ---- p = Q h, row layout again
  __syncwarp();
  if (in) yv[lane] = h;
  __syncwarp();
  double p0 = 0.0, p1 = 0.0;
#pragma unroll
  for (int c = 0; c < 8; c += 2) {
    const double h0 = (c0 + c < n) ? yv[c0 + c] : 0.0, h1 = (c0 + c + 1 < n) ? yv[c0 + c + 1] : 0.0;
    p0 = fma(Q[c], h0, p0); p1 = fma(Q[c + 1], h1, p1);
  }
  const double pl_ = p0 + p1;
  const double pr = pl_ + __shfl_xor_sync(FULL, pl_, 1);
  __syncwarp();
  if (hf == 0 && rin) yv[row] = pr;
  __syncwarp();
  TR_T(q6_); TR_ADD(9, q5_, q6_);
  return hit;
}

// ------------------------------------------------------------------------------------------------
// Exact trust-region step by one warp (solve_tr, optim.jl:9-51): minimise g'p + p'Hp/2, |p|_2 <= Delta over the free
// coordinates fr[0..n). Lane i < n owns row i / component i of the reduced system; the step p is left in yv[0..n). General n <= 32; tr_step16 is the fast path. A: n x n scratch.
// Householder tridiagonalisation H_FF = Q T Q' (reflectors kept in A below the sub-diagonal), then the admissible shifts
// S = {lam >= 0: T + lam I positive definite, |h(lam)| <= Delta} = [lam*, inf) are searched by RBO_TR_ROUNDS rounds of 32-way
// multisection -- lane j tests one candidate with the forward LDL' recurrences and their lam-derivatives (no storage) --;
// lam* = 0 is the interior Newton step, the hard case is completed along the lowest eigenvector (optim.jl:39-46).
// Same algorithm, candidate grid included, as oracle/rbo_oracle.cpp::tr_step.
// ------------------------------------------------------------------------------------------------
// Two candidate shifts per lane: 0 = admissible, 1 = positive definite but |h(lam)| > Delta, 2 = not positive definite.
// yv[i] = component i of Q'g (shared memory). Forward LDL' recurrences of T + lam I and their lam-derivatives:
// |h(lam)|^2 = b'(T + lam I)^-2 b = -d/dlam sum z_i^2 / d_i, no storage, no backward pass.
__device__ __forceinline__ void tri_probe2(const double* A, const double* yv, int n, double lamA, double lamB, double D2, int& outA, int& outB) {
  const double lam[2] = {lamA, lamB};
  double z[2], r[2], dd[2], zd[2], acc[2];
  bool ok[2];
  const double b0 = yv[0], a0 = A[0];
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const double dn = a0 + lam[c];
    ok[c] = dn > 0.0; r[c] = 1.0 / dn; dd[c] = 1.0; zd[c] = 0.0; z[c] = b0; acc[c] = (b0 * b0) * r[c] * r[c];
  }
  for (int i = 1; i < n; ++i) {
    const double e = A[i * n + i - 1], a = A[i * n + i], b = yv[i];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const double er = e * r[c], dn = a + lam[c] - e * er;
      const double ddn = fma(er * er, dd[c], 1.0), zn = b - er * z[c], zdn = er * (r[c] * dd[c] * z[c] - zd[c]);
      ok[c] = ok[c] && dn > 0.0;
      r[c] = 1.0 / dn;
      acc[c] += (zn * zn * ddn - 2.0 * zn * zdn * dn) * r[c] * r[c];
      dd[c] = ddn; z[c] = zn; zd[c] = zdn;
    }
  }
  outA = ok[0] ? (acc[0] <= D2 ? 0 : 1) : 2;
  outB = ok[1] ? (acc[1] <= D2 ? 0 : 1) : 2;
}
// lane i: component i of -(T + lam I)^-1 b, b[0..n) in shared memory; the pivots must be positive
__device__ __forceinline__ double tri_solve_dist(const double* A, const double* b, int n, double lam, int lane) {
  double myr = 0.0, myz = 0.0, r = 0.0, z = 0.0;
  for (int i = 0; i < n; ++i) {
    const double bi = b[i];
    if (i == 0) { r = 1.0 / (A[0] + lam); z = bi; }
    else { const double e = A[i * n + i - 1], er = e * r; r = 1.0 / (A[i * n + i] + lam - e * er); z = bi - er * z; }
    if (lane == i) { myr = r; myz = z; }
  }
  const double te = (lane + 1 < n) ? A[(lane + 1) * n + lane] : 0.0;
  double hv = 0.0;
  for (int i = n - 1; i >= 0; --i) {
    const double hn = __shfl_sync(FULL, hv, (i + 1) & 31);
    if (lane == i) hv = (myz - ((i + 1 < n) ? te * hn : 0.0)) * myr;
  }
  return -hv;
}
// A: n x n scratch; yv: n-vector scratch (shared memory, per slot)
__device__ __noinline__ bool tr_step_warp(const double* H, const double* g, const int* fr, int n, int d, double Delta, double* A, double* yv) {
  const int lane = threadIdx.x & 31;
  const bool in = lane < n;
  const int myc = in ? fr[lane] : 0;
  const double gF = in ? g[myc] : 0.0;
  if (n == 1) {
    const double hh = H[fr[0] * d + fr[0]], g0 = g[fr[0]];
    const bool inside = hh > 0.0 && fabs(g0 / hh) <= Delta;
    __syncwarp();
    if (lane == 0) yv[0] = inside ? -g0 / hh : (g0 > 0.0 ? -Delta : Delta);
    __syncwarp();
    return !inside;
  }
  for (int e = lane; e < n * n; e += 32) { const int i = e / n, j = e - i * n; A[e] = H[fr[i] * d + fr[j]]; }
  if (in) yv[lane] = gF;
  double gn = 0.0;
  for (int i = 0; i < n; ++i) { const double t = g[fr[i]]; gn = fma(t, t, gn); }
  gn = sqrt(gn);
  __syncwarp();
  // ---- Householder tridiagonalisation H_FF = Q T Q' with y <- Q'y fused in. Every lane evaluates the short dot products
  // itself from shared memory (cheaper than FP64 shuffle reductions at these sizes). After step k: column k below the
  // sub-diagonal keeps v_k (rows k+2..), A[k][k+1] its first component and A[k][k+2] beta_k.
  for (int k = 0; k + 2 < n; ++k) {
    double xa = 0.0, xb = 0.0;
    for (int i = k + 1; i + 1 < n; i += 2) { const double u0 = A[i * n + k], u1 = A[(i + 1) * n + k]; xa = fma(u0, u0, xa); xb = fma(u1, u1, xb); }
    if (((n - k - 1) & 1) != 0) { const double u0 = A[(n - 1) * n + k]; xa = fma(u0, u0, xa); }
    const double xn2 = xa + xb, x0 = A[(k + 1) * n + k];
    const double alpha = (x0 > 0.0 ? -1.0 : 1.0) * sqrt(xn2);
    const double vtv = xn2 - 2.0 * alpha * x0 + alpha * alpha;
    if (!(vtv > 0.0) || !(xn2 - x0 * x0 > 0.0)) {  // column already reduced (uniform)
      __syncwarp();
      if (lane == 0) { A[k * n + k + 2] = 0.0; }
      __syncwarp();
      continue;
    }
    const double bk = 2.0 / vtv, v1 = x0 - alpha;
    const bool mine = lane > k && in;
    const double vi = (lane == k + 1) ? v1 : (mine ? A[lane * n + k] : 0.0);
    double t = 0.0;
    if (mine) {
      t = A[lane * n + k + 1] * v1;
      for (int j = k + 2; j < n; ++j) t = fma(A[lane * n + j], A[j * n + k], t);
    }
    const double pw = bk * t;
    if (mine) A[k * n + lane] = pw;  // row k beyond the diagonal is free: scratch for p
    __syncwarp();
    double pv = A[k * n + k + 1] * v1, vy = v1 * yv[k + 1];
    for (int j = k + 2; j < n; ++j) { const double vj = A[j * n + k]; pv = fma(A[k * n + j], vj, pv); vy = fma(vj, yv[j], vy); }
    const double kk = 0.5 * bk * pv, wi = pw - kk * vi;
    __syncwarp();
    if (mine) {
      yv[lane] -= bk * vy * vi;
      A[lane * n + k + 1] -= vi * (A[k * n + k + 1] - kk * v1) + wi * v1;
      for (int j = k + 2; j < n; ++j) { const double vj = A[j * n + k]; A[lane * n + j] -= vi * (A[k * n + j] - kk * vj) + wi * vj; }
    }
    __syncwarp();
    if (lane == k + 1) A[lane * n + k] = alpha;                                 // sub-diagonal of T
    if (lane == k) { A[k * n + k + 1] = v1; A[k * n + k + 2] = bk; }            // first component of v_k, beta_k
    __syncwarp();
  }
  double glo = INFINITY;
  if (in) glo = A[lane * n + lane] - (lane > 0 ? fabs(A[lane * n + lane - 1]) : 0.0) - (lane + 1 < n ? fabs(A[(lane + 1) * n + lane]) : 0.0);
  glo = warp_min(glo);  // Gershgorin lower bound of lambda_min(T)
  const double D2 = Delta * Delta;
  double lo = 0.0, hi = fmax(0.0, -glo) + gn / Delta;
  bool hit = true, lo_notpd = false;
  for (int round = 0; round < RBO_TR_ROUNDS; ++round) {
    // 64 candidates per round, two per lane (c = lane, lane + 32); the last one is hi, known to be admissible
    const double base = lo, wd = hi - lo;
    const double lamA = (round == 0) ? wd * (double)lane / 63.0 : base + wd * (double)(lane + 1) / 64.0;
    const double lamB = (round == 0) ? wd * (double)(lane + 32) / 63.0 : base + wd * (double)(lane + 33) / 64.0;
    int oa, ob;
    tri_probe2(A, yv, n, lamA, lamB, D2, oa, ob);
    const unsigned long long adm = ((unsigned long long)__ballot_sync(FULL, ob == 0) << 32) | __ballot_sync(FULL, oa == 0) | (1ull << 63);
    const unsigned long long pdm = ((unsigned long long)__ballot_sync(FULL, ob != 2) << 32) | __ballot_sync(FULL, oa != 2);
    const int cf = __ffsll((long long)adm) - 1;
    if (round == 0) {
      if (cf == 0) { hi = 0.0; hit = false; break; }
      lo_notpd = ((pdm >> (cf - 1)) & 1ull) == 0ull;
      hi = (cf == 63) ? hi : wd * (double)cf / 63.0;
      lo = wd * (double)(cf - 1) / 63.0;
    } else {
      if (cf > 0) lo_notpd = ((pdm >> (cf - 1)) & 1ull) == 0ull;
      hi = (cf == 63) ? hi : base + wd * (double)(cf + 1) / 64.0;
      lo = (cf == 0) ? base : base + wd * (double)cf / 64.0;
    }
  }
  double h = tri_solve_dist(A, yv, n, hi, lane);
  if (hit && lo_notpd) {
    const double hn2 = warp_sum(in ? h * h : 0.0);
    if (hn2 < D2) {  // hard case (to the resolution of the search): complete along the lowest eigenvector of T
      __syncwarp();
      if (in) yv[lane] = 1.0;
      __syncwarp();
      double z = 0.0;
      for (int itn = 0; itn < 2; ++itn) {
        const double z2 = tri_solve_dist(A, yv, n, hi, lane);
        const double zn = 1.0 / sqrt(warp_sum(in ? z2 * z2 : 0.0));
        z = in ? z2 * zn : 0.0;
        __syncwarp();
        if (in) yv[lane] = z;
        __syncwarp();
      }
      const double hz = warp_sum(in ? h * z : 0.0);
      const double tau = -hz + sqrt(fmax(hz * hz + (D2 - hn2), 0.0));
      h += tau * z;
    }
  }
  // ---- p = Q h: reflectors in descending order
  __syncwarp();
  if (in) yv[lane] = h;
  __syncwarp();
  for (int k = n - 3; k >= 0; --k) {
    const double bk = A[k * n + k + 2], v1 = A[k * n + k + 1];
    if (bk == 0.0) continue;
    double dot = v1 * yv[k + 1];
    for (int j = k + 2; j < n; ++j) dot = fma(A[j * n + k], yv[j], dot);
    const double vi = (lane == k + 1) ? v1 : ((lane > k + 1 && in) ? A[lane * n + k] : 0.0);
    __syncwarp();
    if (lane > k && in) yv[lane] -= bk * dot * vi;
    __syncwarp();
  }
  return hit;
}

}  // namespace
}  // namespace rbo
