// rollout_kernel.cu -- the hot path of librbo.so: one CTA per (quasi-)Monte-Carlo trajectory, persistent grid
// with a dynamic trajectory counter, FP64 throughout, written for sm_100a.
//
// What one CTA does for one sample index m (reference: rollout.jl:279-340 -> rollout! :39-74, resolve :108-111,
// gradient :233-277):
//   * keeps the trajectory's state in shared memory: the (<= 8) fantasy rows of the Cholesky factor as one
//     8-row panel, the coefficient tape cs[0..h+1], u = L^-1 y, fantasy locations / draws;
//   * every surrogate evaluation is expressed as column operations on a shared-memory matrix V (rows =
//     observations, columns = right-hand sides): build kernel columns, "triangular solves" as panel products with the
//     EXPLICIT inverse of the base factor (32-row panels streamed once per pass by a TMA producer warp through a
//     3-stage shared-memory ring, FP64 tensor-core MMA by the consumer warps) followed by the <= 8 fantasy rows,
//     then row reductions (A'B products of column blocks on the tensor cores, fixed-order row splits);
//   * the multi-start inner solve (replacing rbf_optim.jl:68-101 / Optim.IPNewton) keeps W start slots busy in
//     lock-step rounds: each round evaluates (alpha, grad alpha, Hess alpha) at one trial point per active slot,
//     one warp per slot then runs one step of the exact trust-region Newton method (DESIGN.md section 4; the n <= 16
//     subproblem entirely in registers, tr_step16), finished slots are refilled from the start queue;
//   * the adjoint (rollout.jl:233-277) replays the tape: each policy solve i = t..1 is re-evaluated ONCE and its
//     perturbation columns (rbs.jl:633-764) are pushed into the right-hand sides of the earlier duals.
//
// This file is compiled twice (see the Makefile): RBO_VGLOB = 0 is the kernel whose work matrix V lives in shared memory
// (rbo_rollout_kernel; the compiler then addresses V with shared-memory instructions), RBO_VGLOB = 1 the large-n variant
// whose V is a per-CTA scratch in global memory that stays L2-resident (rbo_rollout_kernel_largen; north_star: "L0 ... read
// through L2 when n is large", BASELINE config C5 with n = 1000, d = 20). Everything else is the same code. The trust-region
// step is in trust_region.cuh, the small kernels around a launch in support_kernels.cu.
#include "rbo_kernel.cuh"

#ifndef RBO_VGLOB
#define RBO_VGLOB 0
#endif
// The large-n build walks the work matrix (and the base locations) in global memory: its row loops are unrolled deeper so that
// more L2 loads are in flight per warp; the shared-memory build sits at the register cap and keeps the shallow unroll.
#if RBO_VGLOB
#define RBO_ROW_UNROLL _Pragma("unroll 4")
#else
#define RBO_ROW_UNROLL _Pragma("unroll 2")
#endif
#if RBO_VGLOB
#define RBO_KERNEL_NAME rbo_rollout_kernel_largen
#define g_phase_cycles g_phase_cycles_largen
#define g_aux_cycles g_aux_cycles_largen
#define g_tr_cycles g_tr_cycles_largen
#else
#define RBO_KERNEL_NAME rbo_rollout_kernel
#endif

#ifdef RBO_PHASE_TIMERS
namespace rbo {
__device__ unsigned long long g_phase_cycles[16];
__device__ unsigned long long g_aux_cycles[16];  // histogram of the per-start solver-step durations (slot_logic_warp), bins of 4000 cycles, the last one open
__device__ unsigned long long g_tr_cycles[16];   // per-start logic, summed over all logic warps: [calls, pre, tr step, post, tr: load, householder, write-out, probes, solve, back-transform]
}  // namespace rbo
#define TR_T(v) long long v = clock64()
#define TR_ADD(i, t0, t1) do { if ((threadIdx.x & 31) == 0) atomicAdd(&g_tr_cycles[i], (unsigned long long)((t1) - (t0))); } while (0)
#define PT_DECL long long pt_t0 = clock64()
#define PT_MARK(i) do { if (threadIdx.x == 0) { long long t1_ = clock64(); atomicAdd(&g_phase_cycles[i], (unsigned long long)(t1_ - pt_t0)); pt_t0 = t1_; } } while (0)
#else
#define PT_DECL
#define PT_MARK(i)
#endif
#include "trust_region.cuh"

namespace rbo {

namespace {

// int-area layout
enum { I_M = 0, I_NACT = 1, I_TSTATUS = 2, I_BEST = 3, I_EVALS = 4, I_T = 5, I_CASE = 6, I_NEXT = 7, I_ARR = 64 };
#ifndef RBO_SPIN_CAP
#define RBO_SPIN_CAP (1u << 28)  // polls of an mbarrier before the wait is declared dead (seconds; a healthy wait takes microseconds)
#endif

// max over the warp of a value that is >= 0 in every lane: the IEEE bit pattern of non-negative doubles is monotone, so two integer
// REDUX instructions replace five shuffle rounds (a shuffle costs ~45 cycles of latency on B200)
__device__ __forceinline__ double warp_max_nonneg(double v) {
  const unsigned hi = (unsigned)__double2hiint(v), lo = (unsigned)__double2loint(v);
  const unsigned mh = __reduce_max_sync(FULL, hi);
  const unsigned ml = __reduce_max_sync(FULL, hi == mh ? lo : 0u);
  return __hiloint2double((int)mh, (int)ml);
}
// index of (p, q), p <= q, in the row-major upper triangle of an n x n matrix
__device__ __forceinline__ int tri_idx(int p, int q, int n) { return p * n - (p * (p - 1)) / 2 + (q - p); }
// sum of the RS row-split partial sums part[r * stride + e] of a reduction, in a fixed order from 0.0: results do not depend
// on which warp computed which split
__device__ __forceinline__ double split_sum(const double* part, int RS, int stride, int e) {
  double s = 0.0;
  for (int r = 0; r < RS; ++r) s += part[(size_t)r * stride + e];
  return s;
}

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
  // ---- fantasy rows on the tensor cores -------------------------------------------------------------------
  // Fp: rows 0..N8-1 hold F (Fp[i*8 + r] = F[r][i]), rows N8..N8+7 hold Ginv = G^-1 (Fp[(N8+kk)*8 + r] = Ginv[r][kk]).
  // C-fragment (row g, columns 2 tg, 2 tg + 1) -> B-fragment (k = tg / tg + 4, column g) of the same 8x8 tile.
__device__ __forceinline__ void c_to_b(double c0, double c1, int g, int tg, double& b0, double& b1) {
    const int s0 = tg * 4 + (g >> 1), s1 = s0 + 16;
    const double a0 = __shfl_sync(FULL, c0, s0), a1 = __shfl_sync(FULL, c1, s0);
    const double e0 = __shfl_sync(FULL, c0, s1), e1 = __shfl_sync(FULL, c1, s1);
    b0 = (g & 1) ? a1 : a0; b1 = (g & 1) ? e1 : e0;
  }
  // w_bot = Ginv^T t of one column group (t = fantasy rows of V, rows >= nfan masked): C-fragment of w_bot.
__device__ __forceinline__ void fan_wbot(const double* V, const double* Fp, int RP, int N8, int cB, int nfan, int g, int tg, double& w0, double& w1) {
    const double t0 = (tg < nfan) ? V[(size_t)(N8 + tg) * RP + cB] : 0.0;
    const double t1 = (tg + 4 < nfan) ? V[(size_t)(N8 + tg + 4) * RP + cB] : 0.0;
    w0 = 0.0; w1 = 0.0;
    dmma(w0, w1, Fp[(size_t)(N8 + g) * 8 + tg], t0);       // A[r = g][kk = tg] = Ginv[kk][r]
    dmma(w0, w1, Fp[(size_t)(N8 + g) * 8 + 4 + tg], t1);
    if (g >= nfan) { w0 = 0.0; w1 = 0.0; }
  }

  // V <- L^-T V (N <= 256), every warp of the CTA working: the backward pass of the inner
  // solve has <= 8 columns, far too few to keep a staged panel stream busy, so here the panels of L0^-1 (A-fragment order,
  // Lbf) are read straight from L2, prefetched one tile ahead in place. Task = (column group, pair of block rows {c, nb-1-c}
  // -- equal work --, row quarter). Results stay in registers until every warp has finished reading the right-hand sides.
__device__ __noinline__ void bwd_direct(double* V, const double* Fp, const int* colidx, const double* Lbf, int RP, int N8, int nb, int ncols, int nfan, int warp, int lane, double* scratch = nullptr) {
    const unsigned FULL = 0xffffffffu;
    const int g = lane >> 2, tg = lane & 3;
    const int ngroups = (ncols + 7) >> 3, ncls = (nb + 1) >> 1, tpg = ncls * 4;
    auto cols = [&](int group, int& cB, int& c0, int& c1, bool& v0, bool& v1) {
      const int i0 = 8 * group, first = colidx[i0];
      cB = (i0 + g < ncols) ? colidx[i0 + g] : first;
      v0 = i0 + 2 * tg < ncols; v1 = i0 + 2 * tg + 1 < ncols;
      c0 = v0 ? colidx[i0 + 2 * tg] : first; c1 = v1 ? colidx[i0 + 2 * tg + 1] : first;
    };
    if (nfan > 0) {
      // top rows: v_i -= sum_r F[r][i] w_bot[r], one 8-row tile per warp-task
      const int ntile = N8 >> 3;
      for (int task = warp; task < ngroups * ntile; task += RBO_NWARPS) {
        const int group = task / ntile, i0 = 8 * (task - group * ntile);
        int cB, c0, c1; bool v0, v1;
        cols(group, cB, c0, c1, v0, v1);
        double w0, w1, b0, b1;
        fan_wbot(V, Fp, RP, N8, cB, nfan, g, tg, w0, w1);
        c_to_b(w0, w1, g, tg, b0, b1);
        double* vr = V + (size_t)(i0 + g) * RP;
        double x0 = vr[c0], x1 = vr[c1];
        dmma(x0, x1, Fp[(size_t)(i0 + g) * 8 + tg], -b0);  // A[i][r = tg] = F[r][i]
        dmma(x0, x1, Fp[(size_t)(i0 + g) * 8 + 4 + tg], -b1);
        __syncwarp();
        if (v0) vr[c0] = x0;
        if (v1) vr[c1] = x1;
      }
      __syncthreads();
      // fantasy rows: t -> w_bot (the products below see them only through zero coefficients)
      for (int group = warp; group < ngroups; group += RBO_NWARPS) {
        int cB, c0, c1; bool v0, v1;
        cols(group, cB, c0, c1, v0, v1);
        double w0, w1;
        fan_wbot(V, Fp, RP, N8, cB, nfan, g, tg, w0, w1);
        __syncwarp();
        if (v0) V[(size_t)(N8 + g) * RP + c0] = w0;
        if (v1) V[(size_t)(N8 + g) * RP + c1] = w1;
      }
    }
#if RBO_VGLOB
    {
      // ---- large-n variant: task = (column group, pair of block rows {c, nb-1-c} -- equal work --); a warp takes all four row
      // quarters of its block rows, so every right-hand-side fragment read from the (global, L2-resident) work matrix feeds four
      // tensor-core tiles. The panels stream straight from L2 in A-fragment order. Results go to a per-CTA scratch (out of place:
      // other tasks still read the right-hand sides) and are copied back, 8 columns per group.
      const int ntask = ngroups * ncls;
      __syncthreads();  // fantasy-row update of the top rows stored
      for (int task = warp; task < ntask; task += RBO_NWARPS) {
        const int group = task / ncls, cls = task - group * ncls;
        int cB, c0, c1; bool v0, v1;
        cols(group, cB, c0, c1, v0, v1);
        const int rp4 = 4 * RP, rp8 = 8 * RP;
        for (int hh = 0; hh < 2; ++hh) {
          const int ib = hh ? nb - 1 - cls : cls, rb = RBO_BR * ib;
          if (hh && ib == cls) continue;
          const int nc = nb - ib, chunk0 = nb * ib - ib * (ib - 1) / 2;
          const int nq = min(4, (N8 - rb + 7) >> 3);  // row quarters of this block row that lie below N8 (uniform)
          const double2* ap = reinterpret_cast<const double2*>(Lbf) + (size_t)chunk0 * 512 + lane;  // 128 double2 per tile, 4 tiles per chunk
          const double* vd = V + (size_t)(rb + tg) * RP + cB;
          double acc[4][4];
#pragma unroll
          for (int q = 0; q < 4; ++q) { acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.0; }
          for (int cc = 0; cc < nc; ++cc) {
            const double* v = (cc < nc - 1) ? vd + (size_t)(RBO_BR + RBO_CHUNK_K * cc) * RP : vd;
            double bv[8];
#pragma unroll
            for (int pp = 0; pp < 4; ++pp) { bv[2 * pp] = v[pp * rp8]; bv[2 * pp + 1] = v[pp * rp8 + rp4]; }
            const double2* ac = ap + (size_t)512 * cc;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              if (q < nq) {
                double2 A[4];
#pragma unroll
                for (int pp = 0; pp < 4; ++pp) A[pp] = __ldg(ac + 128 * q + 32 * pp);
#pragma unroll
                for (int pp = 0; pp < 4; ++pp) {
                  dmma(acc[q][0], acc[q][1], A[pp].x, bv[2 * pp]);
                  dmma(acc[q][2], acc[q][3], A[pp].y, bv[2 * pp + 1]);
                }
              }
            }
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int row = rb + 8 * q + g;
            if (q < nq && row < N8) {
              double* o = scratch + ((size_t)group * N8 + row) * 8 + 2 * tg;
              o[0] = acc[q][0] + acc[q][2]; o[1] = acc[q][1] + acc[q][3];
            }
          }
        }
      }
      __syncthreads();
      for (int idx = threadIdx.x; idx < ngroups * N8 * 8; idx += RBO_THREADS) {
        const int group = idx / (N8 * 8), r2 = idx - group * N8 * 8, row = r2 >> 3, cc = r2 & 7;
        if (8 * group + cc < ncols) V[(size_t)row * RP + colidx[8 * group + cc]] = scratch[idx];
      }
    }
#else  // the shared-memory build never takes the scratch path and the large-n build always does: each compiles only its own
    // ---- base rows: w_I = sum_{J >= I} Linv[J][I]^T b_J ; one task per warp and batch, a batch = whole column groups
    const int gpb = RBO_NWARPS / tpg;  // column groups per batch (tpg <= RBO_NWARPS is the caller's condition)
    for (int gb = 0; gb < ngroups; gb += gpb) {
      const int group = gb + warp / tpg, rem = warp % tpg, cls = rem >> 2, rq = rem & 3;
      const bool wact = warp < gpb * tpg && group < ngroups;
      int cB = 0, c0 = 0, c1 = 0; bool v0 = false, v1 = false;
      if (wact) cols(group, cB, c0, c1, v0, v1);
      double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
      const int rp4 = 4 * RP, rp8 = 8 * RP;
      __syncthreads();  // fantasy-row update of the top rows / previous batch stored
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int ib = hh ? nb - 1 - cls : cls, rb = RBO_BR * ib;
        // warp-uniform: the block row exists, is not visited twice, and this row quarter lies (partly) below N8
        if (!wact || (hh && ib == cls) || rb + 8 * rq >= N8) continue;
        const int nc = nb - ib, chunk0 = nb * ib - ib * (ib - 1) / 2;
        const double2* ap = reinterpret_cast<const double2*>(Lbf) + (size_t)(chunk0 * 4 + rq) * 128 + lane;  // 128 double2 per tile, 512 per chunk
        const double* vd = V + (rb + tg) * RP + cB;  // right-hand-side rows of block ib (used by the last, diagonal tile)
        double e0 = 0.0, e1 = 0.0, o0 = 0.0, o1 = 0.0;  // two accumulator chains over the whole block row
        // the A fragments of the next tile are loaded into the registers of the fragment that has just been issued (no second buffer:
        // the function has to live with the registers the caller leaves it, and a spilled prefetch buffer is worse than a shorter distance)
        double2 A[4];
#pragma unroll
        for (int pp = 0; pp < 4; ++pp) A[pp] = __ldg(ap + 32 * pp);
        for (int cc = 0; cc < nc; ++cc) {
          const double* v = (cc < nc - 1) ? vd + (RBO_BR + RBO_CHUNK_K * cc) * RP : vd;
          const double2* an = ap + 512 * (cc + 1 < nc ? cc + 1 : cc);
#pragma unroll
          for (int pp = 0; pp < 4; ++pp) {
            dmma(e0, e1, A[pp].x, v[pp * rp8]);
            dmma(o0, o1, A[pp].y, v[pp * rp8 + rp4]);
            A[pp] = __ldg(an + 32 * pp);
          }
        }
        acc[hh][0] = e0 + o0; acc[hh][1] = e1 + o1;
      }
      __syncthreads();  // all right-hand-side rows of this batch have been read
      if (wact) {
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int ib = hh ? nb - 1 - cls : cls;
          if (hh && ib == cls) continue;
          const int row = RBO_BR * ib + 8 * rq + g;
          if (row < N8) {
            if (v0) V[(size_t)row * RP + c0] = acc[hh][0];
            if (v1) V[(size_t)row * RP + c1] = acc[hh][1];
          }
        }
      }
    }
#endif
  }

struct K {
  const DevProblem& P;
  const SmemPlan& pl;
  double* sm;
  int* si;
  int tid, lane, warp;
  int nf;  // number of fantasy rows that are active for the current operation (uniform over the CTA)
  int CCOL, UCOL;  // columns of V that hold the current coefficients c and u = L^-1 y
  double *V, *Fp, *G, *u, *Xf, *yf, *gyf, *misc, *adj, *bestx, *Xs, *stage;
  double* cst;     // this CTA's coefficient tape in global memory: cst[k * NR + j] = cs[k][j] (rbs.jl:326)
  unsigned long long* mbar;
  unsigned qglob;  // running count of staged panel chunks (ring position and mbarrier parity)
  int *alist, *phase, *sstat, *siter, *stry, *sstart, *sevals, *sflag, *sfr, *colidx, *items, *tbld;
  unsigned short *evprev, *evfirst, *sorder;  // [S] evaluations of every start in the previous multistart of this CTA / in the first multistart of its previous trajectory; hand-out order of the starts

  __device__ K(const DevProblem& P_, double* sm_) : P(P_), pl(P_.pl), sm(sm_) {
    tid = threadIdx.x; lane = tid & 31; warp = tid >> 5;
    nf = 0;
    CCOL = P.RP - 1; UCOL = P.RP - 2;
#if RBO_VGLOB
    V = P.Vscratch + (size_t)blockIdx.x * P.NR * P.RP;
#else
    V = sm + pl.V;
#endif
    Fp = sm + pl.Fp; G = sm + pl.G; u = sm + pl.u; Xs = sm + pl.Xs; stage = sm + pl.stage;
    mbar = reinterpret_cast<unsigned long long*>(sm + pl.mbar); qglob = 0;
    cst = P.cs_tape + (size_t)blockIdx.x * (P.h + 2) * P.NR;
    Xf = sm + pl.Xf; yf = sm + pl.yf; gyf = sm + pl.gyf; misc = sm + pl.misc; adj = sm + pl.adj; bestx = sm + pl.bestx;
    si = reinterpret_cast<int*>(sm + pl.ints);
    items = reinterpret_cast<int*>(sm + pl.pairs);
    tbld = reinterpret_cast<int*>(sm + pl.tbl);
    evprev = reinterpret_cast<unsigned short*>(sm + pl.sord); evfirst = evprev + P.S; sorder = evfirst + P.S;
    const int W = P.W;
    alist = si + I_ARR; phase = alist + W; sstat = phase + W; siter = sstat + W; stry = siter + W;
    sstart = stry + W; sevals = sstart + W; sflag = sevals + W; sfr = sflag + W; colidx = sfr + 32 * W;
  }

  __device__ __forceinline__ double xcoord(int j, int p) const {
    return j < P.N8 ? (P.xsm ? Xs[p * P.XP + j] : __ldg(P.Xb + (size_t)p * P.N8 + j)) : Xf[(j - P.N8) * P.d + p];
  }
  __device__ __forceinline__ bool row_active(int j) const { return j < P.N || (j >= P.N8 && j < P.N8 + nf); }

  // (p, q) table of the upper triangle of size d, packed p | q << 8
  __device__ void build_tables() {
    const int d = P.d;
    for (int e = tid; e < d * (d + 1) / 2; e += RBO_THREADS) {
      int p = 0, t = e;
      while (t >= d - p) { t -= d - p; ++p; }
      tbld[e] = p | ((p + t) << 8);
    }
  }

  // column `col` of V <- vector v (length NR)
  __device__ void set_column(int col, const double* v) {
    for (int j = tid; j < P.NR; j += RBO_THREADS) V[(size_t)j * P.RP + col] = v[j];
  }

  // ------------------------------------------------------------------------------------------------
  // Kernel columns for `np` points: column block at cb(s) gets [kx | b*r (d columns) | a | b] for every row
  // (rbf.jl:180-208 eval_KxX / eval_gradKxX and the eval_Hk coefficients of rbf.jl:141-150). Inactive rows get 0.
  // ------------------------------------------------------------------------------------------------
  template <class PT, class CB>
  __device__ void fill_columns(int np, PT pt, CB cb) {
    const int d = P.d, NR = P.NR, RP = P.RP;
    for (int idx = tid; idx < np * NR; idx += RBO_THREADS) {
      int s = idx / NR, j = idx - s * NR;
      double* row = V + (size_t)j * RP + cb(s);
      if (!row_active(j)) {
        for (int q = 0; q < d + 3; ++q) row[q] = 0.0;
        continue;
      }
      const double* x = pt(s);
      // coordinates of row j: base rows are coordinate-major (stride XP in shared memory / N8 in global), fantasy rows point-major
      const bool base = j < P.N8;
      const double* xc = base ? (P.xsm ? Xs + j : P.Xb + j) : Xf + (j - P.N8) * d;
      const int xst = base ? (P.xsm ? P.XP : P.N8) : 1;
      double rho2 = 0.0;
#if RBO_VGLOB
#pragma unroll 4
#endif
      for (int p = 0; p < d; ++p) { double r = x[p] - xc[p * xst]; rho2 = fma(r, r, rho2); }
      double psi, a, b, gb;
      if (P.kern.id == RBO_KERNEL_MATERN52) {
        // closed forms without divisions: b = psi'/rho = -(c^2/3)(1+s)e^-s, a = (psi'' - b)/rho^2 = (c^4/3) e^-s; at rho = 0 they
        // reduce to psi''(0) and a finite value that only ever multiplies r = 0 (rbf.jl:141-150)
        const double cc = P.m52_c, c2 = cc * cc, s_ = cc * sqrt(rho2), e = exp(-s_);
        psi = (1.0 + s_ * (1.0 + s_ * (1.0 / 3.0))) * e;
        b = -(c2 * (1.0 / 3.0)) * (1.0 + s_) * e;
        a = (c2 * c2 * (1.0 / 3.0)) * e;
      } else {
        kern_radial(P.kern, rho2, psi, a, b, gb);
      }
      row[0] = psi;
#if RBO_VGLOB
#pragma unroll 4
#endif
      for (int p = 0; p < d; ++p) row[1 + p] = b * (x[p] - xc[p * xst]);
      row[d + 1] = a;
      row[d + 2] = b;
    }
  }

  // ------------------------------------------------------------------------------------------------
  // Row reductions on the FP64 tensor cores.
  //   colprod: for every product item {colA, na, colB, nb, out}: out[rs][p * nb + q] = sum over the rows of split rs of
  //            V[j][colA + p] * V[j][colB + q]   (A' * B down the rows; 16 x 16 output blocks, 4 rows per DMMA step).
  //   hess_sums: HC = sum_j c_j Hk(x - X_j), HW = sum_j w_j Hk(x - X_j) for np points, r = x - X_j built on the fly.
  // A warp-task = (item, output block, row split); the RS partial sums are added in a fixed order by the consumer, so
  // results do not depend on scheduling.
  // ------------------------------------------------------------------------------------------------
  __device__ int choose_rs(int nblocks, int nw = RBO_NWARPS) const {
    int rs = nw / (nblocks > 0 ? nblocks : 1);
    return rs < 1 ? 1 : (rs > P.RSmax ? P.RSmax : rs);
  }
  // xcol >= 0: the LAST of the nb B-columns is column xcol of V instead of colB + nb - 1
  __device__ __forceinline__ void set_item(int i, int colA, int na, int colB, int nb, int out, int xcol = -1) {
    int* it = items + 6 * i;
    it[0] = colA; it[1] = na; it[2] = colB; it[3] = nb; it[4] = out; it[5] = xcol;
  }
  __device__ static __forceinline__ int nblk16(int n) { return (n + 15) >> 4; }

  // dst[rs * nout + item.out + p * nb + q]; nout = total number of outputs of this call (stride between row splits)
  __device__ void colprod(int nitems, int nout, double* dst, int RS, int wbase = 0, int nw = RBO_NWARPS) {
    const int RP = P.RP, nrows = P.N8 + nf, g = lane >> 2, tg = lane & 3;
    int ntask = 0;
    for (int i = 0; i < nitems; ++i) ntask += nblk16(items[6 * i + 1]) * nblk16(items[6 * i + 3]);
    if (warp < wbase || warp >= wbase + nw) return;
    for (int task = warp - wbase; task < ntask * RS; task += nw) {
      int t = task / RS;
      const int rs = task - t * RS;
      int i = 0, nbA, nbB;
      for (;; ++i) { nbA = nblk16(items[6 * i + 1]); nbB = nblk16(items[6 * i + 3]); if (t < nbA * nbB) break; t -= nbA * nbB; }
      const int* it = items + 6 * i;
      const int colA = it[0], na = it[1], colB = it[2], nb = it[3], mb = t / nbB, nk = t - mb * nbB;
      const int ca0 = colA + min(16 * mb + g, na - 1), ca1 = colA + min(16 * mb + 8 + g, na - 1);
      const int xcol = it[5], ib0 = min(16 * nk + g, nb - 1), ib1 = min(16 * nk + 8 + g, nb - 1);
      const int cb0 = (xcol >= 0 && ib0 == nb - 1) ? xcol : colB + ib0, cb1 = (xcol >= 0 && ib1 == nb - 1) ? xcol : colB + ib1;
      double c00[2] = {0.0, 0.0}, c01[2] = {0.0, 0.0}, c10[2] = {0.0, 0.0}, c11[2] = {0.0, 0.0};
      const bool hiA = na - 16 * mb > 8, hiB = nb - 16 * nk > 8;  // second 8-row / 8-column tile in use (warp-uniform)
      // full 4-row steps without predicates, then at most one ragged step
      const int step = 4 * RS * RP, nfull = nrows & ~3;
      const double* row = V + (4 * rs + tg) * RP;
      int j0 = 4 * rs;
RBO_ROW_UNROLL
      for (; j0 < nfull; j0 += 4 * RS, row += step) {
        const double a0 = row[ca0], b0 = row[cb0];
        dmma(c00[0], c00[1], a0, b0);
        if (hiB) dmma(c01[0], c01[1], a0, row[cb1]);
        if (hiA) {
          const double a1 = row[ca1];
          dmma(c10[0], c10[1], a1, b0);
          if (hiB) dmma(c11[0], c11[1], a1, row[cb1]);
        }
      }
      if (j0 < nrows) {
        const bool in = j0 + tg < nrows;
        const double* rw = in ? row : V;
        const double a0 = in ? rw[ca0] : 0.0, b0 = in ? rw[cb0] : 0.0;
        dmma(c00[0], c00[1], a0, b0);
        if (hiB) { const double b1 = in ? rw[cb1] : 0.0; dmma(c01[0], c01[1], a0, b1); }
        if (hiA) {
          const double a1 = in ? rw[ca1] : 0.0;
          dmma(c10[0], c10[1], a1, b0);
          if (hiB) { const double b1 = in ? rw[cb1] : 0.0; dmma(c11[0], c11[1], a1, b1); }
        }
      }
      double* o = dst + (size_t)rs * nout + it[4];
      const int p0 = 16 * mb + g, p1 = p0 + 8, q0 = 16 * nk + 2 * tg, q1_ = q0 + 8;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        if (p0 < na && q0 + e < nb) o[p0 * nb + q0 + e] = c00[e];
        if (p0 < na && q1_ + e < nb) o[p0 * nb + q1_ + e] = c01[e];
        if (p1 < na && q0 + e < nb) o[p1 * nb + q0 + e] = c10[e];
        if (p1 < na && q1_ + e < nb) o[p1 * nb + q1_ + e] = c11[e];
      }
    }
  }

  // Hk = a r r' + b I (rbf.jl:141-150): entries (p <= q) accumulate a r_p r_q, the b-weighted sums go to the extra entry T2.
  // phess[((rs * np + s) * 2 + which) * (T2 + 1) + e], which = 0 (c-weighted, rbs.jl:516-523) / 1 (w-weighted, rbs.jl:542-545).
  // Columns: (a, b) at cab(s) + d+1, d+2 ; w at cw(s) ; c in CCOL.
  template <int MASK, class PT, class CAB, class CW>  // MASK bit 0: c-weighted sums (HC), bit 1: w-weighted sums (HW)
  __device__ void hess_sums(int np, PT pt, CAB cab, CW cw, int RS, int wbase = 0, int nw = RBO_NWARPS) {
    const int d = P.d, RP = P.RP, T2 = d * (d + 1) / 2, nrows = P.N8 + nf, g = lane >> 2, tg = lane & 3;
    const int nbd = nblk16(d), nblk = nbd * (nbd + 1) / 2;  // upper-triangular 16 x 16 blocks
    double* out = sm + pl.phess;
    if (warp < wbase || warp >= wbase + nw) return;
    for (int task = warp - wbase; task < np * nblk * RS; task += nw) {
      const int s = task / (nblk * RS), rem = task - s * nblk * RS, blk = rem / RS, rs = rem - blk * RS;
      int mb = 0, t = blk;
      while (t >= nbd - mb) { t -= nbd - mb; ++mb; }
      const int nk = mb + t;
      const double* x = pt(s);
      const int colab = cab(s) + d + 1, colw = cw(s);
      const int p0 = min(16 * mb + g, d - 1), p1 = min(16 * mb + 8 + g, d - 1), q0 = min(16 * nk + g, d - 1), q1_ = min(16 * nk + 8 + g, d - 1);
      const double xp0 = x[p0], xp1 = x[p1], xq0 = x[q0], xq1 = x[q1_];
      const bool diag = mb == nk;                                       // diagonal block: q == p, and the (p1, q0) tile lies below the diagonal
      const bool hiP = d - 16 * mb > 8, hiQ = d - 16 * nk > 8;        // second 8-wide tile in use (warp-uniform)
      double cC[4][2], cW[4][2], bC = 0.0, bW = 0.0;
#pragma unroll
      for (int i = 0; i < 4; ++i) { cC[i][0] = cC[i][1] = 0.0; cW[i][0] = cW[i][1] = 0.0; }
      // base rows: coordinates straight from the coordinate-major table (shared or global), no per-element branching
      const int xst = P.xsm ? P.XP : P.N8;
      const int op0 = p0 * xst, op1 = p1 * xst, oq0 = q0 * xst, oq1 = q1_ * xst;
      const int nbase4 = P.N8 & ~3;
      auto body = [&](const double* row, bool in, double rp0, double rp1, double rq0, double rq1) {
        const double aj = in ? row[colab] : 0.0, bj = in ? row[colab + 1] : 0.0;
        const double wj = (MASK & 2) ? row[colw] : 0.0, cj = (MASK & 1) ? row[CCOL] : 0.0;
        const double ca = cj * aj, wa = wj * aj;
        if (g == 0) { bC = fma(cj, bj, bC); bW = fma(wj, bj, bW); }
        if (MASK & 1) {
          dmma(cC[0][0], cC[0][1], ca * rp0, rq0);
          if (hiQ) dmma(cC[1][0], cC[1][1], ca * rp0, rq1);
          if (hiP) {
            if (!diag) dmma(cC[2][0], cC[2][1], ca * rp1, rq0);
            if (hiQ) dmma(cC[3][0], cC[3][1], ca * rp1, rq1);
          }
        }
        if (MASK & 2) {
          dmma(cW[0][0], cW[0][1], wa * rp0, rq0);
          if (hiQ) dmma(cW[1][0], cW[1][1], wa * rp0, rq1);
          if (hiP) {
            if (!diag) dmma(cW[2][0], cW[2][1], wa * rp1, rq0);
            if (hiQ) dmma(cW[3][0], cW[3][1], wa * rp1, rq1);
          }
        }
      };
      int j0 = 4 * rs;
      const int jstep = 4 * RS;
      const double* row = V + (j0 + tg) * RP;
      if (P.xsm) {
        const double* xs = Xs + j0 + tg;
RBO_ROW_UNROLL
        for (; j0 < nbase4; j0 += jstep, row += jstep * RP, xs += jstep) {
          const double rp0 = xp0 - xs[op0], rp1 = xp1 - xs[op1];
          const double rq0 = diag ? rp0 : xq0 - xs[oq0], rq1 = diag ? rp1 : xq1 - xs[oq1];
          body(row, true, rp0, rp1, rq0, rq1);
        }
      } else {
        const double* xs = P.Xb + j0 + tg;
RBO_ROW_UNROLL
        for (; j0 < nbase4; j0 += jstep, row += jstep * RP, xs += jstep) {
          const double rp0 = xp0 - __ldg(xs + op0), rp1 = xp1 - __ldg(xs + op1);
          const double rq0 = diag ? rp0 : xq0 - __ldg(xs + oq0), rq1 = diag ? rp1 : xq1 - __ldg(xs + oq1);
          body(row, true, rp0, rp1, rq0, rq1);
        }
      }
      for (; j0 < nrows; j0 += jstep) {  // the fantasy rows
        const int j = j0 + tg;
        const bool in = j < nrows;
        const int jj = in ? j : 0;
        body(V + (size_t)jj * RP, in, xp0 - xcoord(jj, p0), xp1 - xcoord(jj, p1), xq0 - xcoord(jj, q0), xq1 - xcoord(jj, q1_));
      }
      bC += __shfl_xor_sync(FULL, bC, 1); bC += __shfl_xor_sync(FULL, bC, 2);
      bW += __shfl_xor_sync(FULL, bW, 1); bW += __shfl_xor_sync(FULL, bW, 2);
      double* oC = out + ((size_t)(rs * np + s) * 2 + 0) * (T2 + 1);
      double* oW = out + ((size_t)(rs * np + s) * 2 + 1) * (T2 + 1);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int p = 16 * mb + 8 * (i >> 1) + g;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int q = 16 * nk + 8 * (i & 1) + 2 * tg + e;
          if (p <= q && q < d) {
            const int idx = tri_idx(p, q, d);
            if (MASK & 1) oC[idx] = cC[i][e];
            if (MASK & 2) oW[idx] = cW[i][e];
          }
        }
      }
      if (blk == 0 && lane == 0) { if (MASK & 1) oC[T2] = bC; if (MASK & 2) oW[T2] = bW; }
    }
  }

  // ------------------------------------------------------------------------------------------------
  // Panel pipeline: TMA bulk copies of the packed L0^-1 chunks into a shared-memory ring (see tri_solve below).
  // ------------------------------------------------------------------------------------------------
  __device__ __forceinline__ unsigned smem_u32(const void* p) const { return (unsigned)__cvta_generic_to_shared(p); }

  // Initialises the panel pipeline ONCE per kernel: full barriers expect the producer's arrive (+ the copy's bytes), empty
  // barriers expect one arrive from EVERY consumer warp (RBO_NCONS) for every chunk, whether or not the warp has columns to
  // work on in that pass. The barriers are never re-initialised, so there is no invalidate / init window to get wrong and the
  // running chunk count qglob is identical in all threads by construction. Call from all threads before the first pass.
  __device__ void pipe_init() {
    if (tid == 0) {
      for (int i = 0; i < RBO_NSTAGE; ++i) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar[i])) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(&mbar[RBO_NSTAGE + i])), "r"(RBO_NCONS) : "memory");
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    qglob = 0;
    __syncthreads();
  }
  __device__ void pipe_fini() {  // all passes done: release the barrier objects
    __syncthreads();
    if (tid == 0)
      for (int i = 0; i < 2 * RBO_NSTAGE; ++i) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(&mbar[i])) : "memory");
  }
  __device__ __forceinline__ void chunk_issue(unsigned q, const double* src, int ndoubles) {  // one thread
    const unsigned st = q % RBO_NSTAGE, mb = smem_u32(&mbar[st]), dst = smem_u32(stage + (size_t)st * RBO_CHUNK_K * RBO_LP);
    const unsigned bytes = (unsigned)ndoubles * 8u;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(mb) : "memory");
  }
  // consumer side: plain spin on the full barrier (hot path)
  __device__ __forceinline__ void full_wait(unsigned q) {
    const unsigned mb = smem_u32(&mbar[q % RBO_NSTAGE]), parity = (q / RBO_NSTAGE) & 1u;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(mb), "r"(parity) : "memory");
  }
  // producer side: stage of chunk q was released by all consumers of chunk q - NSTAGE. Bounded spin: a release that never
  // comes is a protocol bug; it is recorded (the host reports the launch as failed) and the producer carries on, so the
  // consumers still receive every chunk and the kernel terminates instead of hanging the GPU.
  __device__ __forceinline__ void empty_wait(unsigned q) {
    const unsigned mb = smem_u32(&mbar[RBO_NSTAGE + q % RBO_NSTAGE]), parity = ((q / RBO_NSTAGE) - 1u) & 1u;
    for (unsigned spins = 0; spins < RBO_SPIN_CAP; ++spins) {
      unsigned ok;
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(mb), "r"(parity) : "memory");
      if (ok) return;
    }
    if (atomicExch(P.work_counter + WC_STALL, 1) == 0) {
      P.work_counter[WC_WAIT_KIND] = 2; P.work_counter[WC_WAIT_CHUNK] = (int)q; P.work_counter[WC_WAIT_WARP] = warp;
      P.work_counter[WC_WAIT_CONSUMERS] = RBO_NCONS; P.work_counter[WC_WAIT_BLOCK] = blockIdx.x;
    }
  }
  __device__ __forceinline__ void empty_arrive(unsigned q) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&mbar[RBO_NSTAGE + q % RBO_NSTAGE])) : "memory");
  }

  // FP64 tensor-core tile: D(8x8) += A(8x4) * B(4x8). Lane l holds A[l >> 2][l & 3], B[l & 3][l >> 2], C[l >> 2][2 (l & 3) + {0, 1}].
  __device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) const {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
  }

  // One 32-k chunk of a 32-row panel against the 8 columns of this warp's group: C[MTW row tiles][8x8] += L[rows x 32k] * V[32k x 8].
  // buf: staged chunk, k-major with pitch RBO_LP, already offset to the warp's first row tile; vrow0: V row of chunk-relative
  // k = 0; cB: this lane's B-fragment column offset.
  template <int MTW>
  __device__ __forceinline__ void mma_chunk(const double* buf, const double* vrow0, int cB, int g, int tg, double (*c)[2], int nt) const {
    const int RP = P.RP;
    const double* vp = vrow0 + (size_t)tg * RP + cB;
    const double* ap = buf + (size_t)tg * RBO_LP + g;
    if (nt >= MTW) {
#pragma unroll
      for (int kt = 0; kt < RBO_CHUNK_K / 4; ++kt) {
        const double b = vp[(size_t)(4 * kt) * RP];
#pragma unroll
        for (int mt = 0; mt < MTW; ++mt) dmma(c[mt][0], c[mt][1], ap[4 * kt * RBO_LP + 8 * mt], b);
      }
    } else {  // last block row: only the row tiles below N8 exist (the fantasy rows have their own panel); nt is warp-uniform
#pragma unroll
      for (int kt = 0; kt < RBO_CHUNK_K / 4; ++kt) {
        const double b = vp[(size_t)(4 * kt) * RP];
#pragma unroll
        for (int mt = 0; mt < MTW; ++mt)
          if (mt < nt) dmma(c[mt][0], c[mt][1], ap[4 * kt * RBO_LP + 8 * mt], b);
      }
    }
  }
  __device__ __forceinline__ void group_sync(int NRQ, int group) const {  // the NRQ warps that share a column group
    if (NRQ == 1) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(1 + group), "r"(32 * NRQ) : "memory");
  }

  template <bool FWD>
  __device__ __forceinline__ const double* pan_ptr(int ib) const {  // global address of panel ib (see rbo_set_surrogate)
    const size_t chunk = (size_t)RBO_LP * RBO_BR;
    return FWD ? P.Lf + chunk * ((size_t)ib * (ib + 1) / 2) : P.Lb + chunk * ((size_t)P.nb32 * ib - (size_t)ib * (ib - 1) / 2);
  }

  // C-fragment (row g, columns 2 tg, 2 tg + 1) -> B-fragment (k = tg / tg + 4, column g) of the same 8x8 tile.
  __device__ __forceinline__ void c_to_b(double c0, double c1, int g, int tg, double& b0, double& b1) const { rbo::c_to_b(c0, c1, g, tg, b0, b1); }
  __device__ void bwd_direct(int ncols, int nfan) {
#if RBO_VGLOB
    rbo::bwd_direct(V, Fp, colidx, P.Lbf, P.RP, P.N8, P.nb32, ncols, nfan, warp, lane, P.Bscratch + (size_t)blockIdx.x * P.bscratch_len);
#else
    rbo::bwd_direct(V, Fp, colidx, P.Lbf, P.RP, P.N8, P.nb32, ncols, nfan, warp, lane);
#endif
  }

  // "Triangular solves" of `ncols` columns of V (indices in colidx[]) against L = [L0 0; F G]: FWD: V <- L^-1 V, else V <- L^-T V.
  //  * The host stores the EXPLICIT inverse of L0 as 32-row panels, k-major (pitch RBO_LP), cut into uniform 32-k chunks, so
  //    a block row of the result is a plain product with right-hand-side rows: v_I = sum_{J<=I} Linv[I][J] b_J. The block rows
  //    are visited in the order that overwrites a block only after its last use as input (descending for FWD).
  //  * Warp RBO_NCONS is the producer: it streams the chunks ONCE per pass into a 3-stage shared-memory ring with TMA bulk
  //    copies (cp.async.bulk + mbarrier complete_tx), throttled by "empty" mbarriers that every consumer warp releases.
  //  * A column group = 8 columns; NRQ = 1, 2 or 4 warps share a group (32 / NRQ rows each) and accumulate with FP64
  //    tensor-core tiles (mma.sync m8n8k4); they meet at a named barrier before the block row is overwritten.
  //  * The fantasy rows (<= 8, per trajectory) are one more panel that already sits in shared memory (DMMA as well).
  //  * The backward direction with few columns (the inner solve: one per start) takes bwd_direct() instead.
  template <bool FWD>
  __device__ void tri_solve(int ncols, int nfan) {
    if (ncols <= 0) return;
    const int ngroups = (ncols + 7) >> 3;  // a column group = 8 consecutive entries of colidx[]
    if (!FWD && (RBO_VGLOB || ((P.nb32 + 1) >> 1) * 4 <= RBO_NWARPS)) { bwd_direct(ncols, nfan); return; }
    if (ngroups * 4 <= RBO_NCONS) tri_solve_impl<FWD, 4>(ncols, nfan);
    else if (ngroups * 2 <= RBO_NCONS) tri_solve_impl<FWD, 2>(ncols, nfan);
    else tri_solve_impl<FWD, 1>(ncols, nfan);
  }

  // NRQ warps share one column group: each owns 32 / NRQ rows (MTW = 4 / NRQ row tiles) of every panel and they meet at a
  // named barrier around the diagonal step.
  template <bool FWD, int NRQ>
  __device__ void tri_solve_impl(int ncols, int nfan) {
    constexpr int MTW = 4 / NRQ, GPB = RBO_NCONS / NRQ;  // row tiles per warp; column groups per batch
    const int RP = P.RP, N8 = P.N8, nb = P.nb32;
    const int ngroups = (ncols + 7) >> 3;
    const int nbatch = (ngroups + GPB - 1) / GPB;
    const unsigned chunks_per_pass = (unsigned)(nb * (nb + 1) / 2);
    const int ncons = min(ngroups, GPB) * NRQ;  // consumer warps of this pass: warps 0 .. ncons-1
    if (warp == RBO_NCONS) {
      // ---------------- producer warp ----------------
      if (lane == 0) {
        unsigned q = qglob;
        for (int bt = 0; bt < nbatch; ++bt)
          for (int i = 0; i < nb; ++i) {
            const int ib = FWD ? nb - 1 - i : i, nc = FWD ? ib + 1 : nb - ib;
            const double* src = pan_ptr<FWD>(ib);
            for (int c = 0; c < nc; ++c, ++q) {
              if (q >= RBO_NSTAGE) empty_wait(q);
              chunk_issue(q, src + (size_t)c * RBO_CHUNK_K * RBO_LP, RBO_CHUNK_K * RBO_LP);
            }
          }
      }
      qglob += (unsigned)nbatch * chunks_per_pass;
      __syncwarp();
      return;
    }
    const bool part = warp < ncons;  // warps beyond take no columns in this pass but still consume (wait + release) every chunk
    // ---------------- consumer warps ----------------
    const int g = lane >> 2, tg = lane & 3;
    const int gl = warp / NRQ, rq = warp - gl * NRQ;  // group slot within the batch, row quarter
    unsigned q = qglob;
    for (int bt = 0; bt < nbatch; ++bt) {
      const int group = bt * GPB + gl;
      const bool wact = part && group < ngroups;  // warp-uniform
      // column offsets: cB for the B fragment (column g), c0/c1 for the C fragment (columns 2 tg, 2 tg + 1)
      const int i0 = 8 * group;
      const bool vB = wact && i0 + g < ncols, v0 = wact && i0 + 2 * tg < ncols, v1 = wact && i0 + 2 * tg + 1 < ncols;
      const int first = colidx[wact ? i0 : 0];
      const int cB = vB ? colidx[i0 + g] : first, c0 = v0 ? colidx[i0 + 2 * tg] : first, c1 = v1 ? colidx[i0 + 2 * tg + 1] : first;
      // fantasy-row helpers (done by the rq == 0 warp of the group): column = g, k-part fp = tg
      double* fv = V + cB;
      const int fp = tg;

      if (!FWD && nfan > 0 && wact) {
        if (rq == 0) {
          // w_bot = Ginv^T t restricted to the active rows: w_r = sum_kk Ginv[kk][r] t[kk], Ginv[kk][r] = Fp[(N8 + r)*8 + kk]
          double t[8], wb[8];
#pragma unroll
          for (int r = 0; r < 8; ++r) t[r] = (r < nfan) ? fv[(size_t)(N8 + r) * RP] : 0.0;
          __syncwarp();
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            double s = 0.0;
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) s = fma(Fp[(size_t)(N8 + r) * 8 + kk], t[kk], s);
            wb[r] = (r < nfan) ? s : 0.0;
          }
          if (vB && fp == 0) {
#pragma unroll
            for (int r = 0; r < 8; ++r) fv[(size_t)(N8 + r) * RP] = wb[r];
          }
          for (int i = fp; i < N8; i += 4) {  // top rows: v_i -= sum_r F[r][i] w_bot[r]
            const double* f = Fp + (size_t)i * 8;
            double s = 0.0;
#pragma unroll
            for (int r = 0; r < 8; ++r) s = fma(f[r], wb[r], s);
            if (vB) fv[(size_t)i * RP] -= s;
          }
        }
        group_sync(NRQ, gl);
      }

      double c[MTW][2];
#pragma unroll
      for (int mt = 0; mt < MTW; ++mt) { c[mt][0] = 0.0; c[mt][1] = 0.0; }
      const int rofs = 8 * MTW * rq;  // first row (within a panel) owned by this warp
      for (int i = 0; i < nb; ++i) {
        // explicit-inverse panels: block row ib of the result only needs RIGHT-HAND-SIDE rows (blocks <= ib forward, >= ib
        // backward), so the block rows are visited in the order that overwrites a block only after its last use as input
        const int ib = FWD ? nb - 1 - i : i, nc = FWD ? ib + 1 : nb - ib, rb = RBO_BR * ib;
        for (int cc = 0; cc < nc; ++cc, ++q) {
#ifdef RBO_PHASE_TIMERS
          long long tw0 = clock64();
#endif
          full_wait(q);
#ifdef RBO_PHASE_TIMERS
          if (tid == 0) atomicAdd(&g_phase_cycles[FWD ? 12 : 13], (unsigned long long)(clock64() - tw0));
#endif
          const double* buf = stage + (size_t)(q % RBO_NSTAGE) * RBO_CHUNK_K * RBO_LP + rofs;
          if (wact) {
            const int nt = (N8 - rb - rofs + 7) >> 3;  // row tiles of this warp that lie below N8 (<= 0: none)
            if (cc < nc - 1) {
              const int krow0 = (FWD ? 0 : rb + RBO_BR) + cc * RBO_CHUNK_K;  // V row of the first k of this chunk
              mma_chunk<MTW>(buf, V + (size_t)krow0 * RP, cB, g, tg, c, nt);
            } else {
              // last chunk of the panel = diagonal block of the inverse applied to the panel's own right-hand-side rows
              mma_chunk<MTW>(buf, V + (size_t)rb * RP, cB, g, tg, c, nt);
              group_sync(NRQ, gl);  // every warp of the group has read the right-hand-side rows
#pragma unroll
              for (int mt = 0; mt < MTW; ++mt) {
                const int row = rb + rofs + 8 * mt + g;
                if (row < N8) {
                  if (v0) V[(size_t)row * RP + c0] = c[mt][0];
                  if (v1) V[(size_t)row * RP + c1] = c[mt][1];
                }
                c[mt][0] = 0.0; c[mt][1] = 0.0;
              }
              asm volatile("" ::: "memory");  // keeps the stores of this panel ahead of the next panel's loads in program order (and the register allocation compact)
            }
          }
          __syncwarp();
          if (lane == 0) empty_arrive(q);
        }
      }

      // the fantasy-row product below reads ALL top rows of the group's columns: the other warps of the group must have stored
      // their rows of the last block row first
      if (FWD && nfan > 0 && wact && NRQ > 1) group_sync(NRQ, gl);
      if (FWD && nfan > 0 && wact && rq == 0) {
        // a = F v_top on the tensor cores (four interleaved accumulator chains), t = b_bot - a, v_bot = Ginv t
        double a0[2] = {0.0, 0.0}, a1[2] = {0.0, 0.0};
        const double* fa = Fp + (size_t)tg * 8 + g;          // A[r = g][k = i] = F[r][i] = Fp[i*8 + r]
        const double* vb = V + (size_t)tg * RP + cB;
        const int nkt = N8 >> 2;  // even (N8 is a multiple of 8)
#pragma unroll 2
        for (int kt = 0; kt < nkt; kt += 2) {
          dmma(a0[0], a1[0], fa[(size_t)(4 * kt) * 8], vb[(size_t)(4 * kt) * RP]);
          dmma(a0[1], a1[1], fa[(size_t)(4 * kt + 4) * 8], vb[(size_t)(4 * kt + 4) * RP]);
        }
        const double s0 = a0[0] + a0[1], s1 = a1[0] + a1[1];
        double* vr = V + (size_t)(N8 + g) * RP;
        const double t0 = (g < nfan) ? vr[c0] - s0 : 0.0, t1 = (g < nfan) ? vr[c1] - s1 : 0.0;
        double b0, b1, r0 = 0.0, r1 = 0.0;
        c_to_b(t0, t1, g, tg, b0, b1);
        dmma(r0, r1, Fp[(size_t)(N8 + tg) * 8 + g], b0);       // A[r = g][kk = tg] = Ginv[r][kk]
        dmma(r0, r1, Fp[(size_t)(N8 + tg + 4) * 8 + g], b1);
        if (g >= nfan) { r0 = 0.0; r1 = 0.0; }
        __syncwarp();
        if (v0) vr[c0] = r0;
        if (v1) vr[c1] = r1;
        __syncwarp();
      }
    }
    qglob = q;
  }

  // ------------------------------------------------------------------------------------------------
  // One warp assembles the surrogate evaluation of slot `sl` from the partial sums (rbs.jl:513-577).
  //   aidx / np: position of the slot in the reduction outputs; RS*: row splits used by each reduction.
  // Writes sdmu, sdsig (grad sigma), sga (grad alpha), sHt (-(H alpha + mu-sigma cross term)), sHref (H alpha as the
  // reference computes it, Q1) and sgh = [alpha, g_mu, g_sig, g_muth, g_sigth, sigma, mu, finite].
  // ------------------------------------------------------------------------------------------------
  // s2/tq come from `p1` (q1 outputs per point: |v0|^2, V_p.v0), the Gram V_p.V_q from `pg` (d x d per point).
  __device__ void assemble_warp(int sl, int aidx, int np, int RSpre, const double* p1, int nout1, int RS1, const double* pg, int noutg, int goff, int gld,
                                int RSg, int RShc, int RShw, double fstar, double* Href /* d x d or nullptr: the reference's H alpha is only kept for the adjoint / extended tape */) {
    const int d = P.d, dd = d * d, q1 = d + 1, T2 = d * (d + 1) / 2;
    const double* ppre = sm + pl.ppre; const double* phess = sm + pl.phess;
    const int nout_pre = np * q1;
    double* dmu = sm + pl.sdmu + sl * d; double* dsig = sm + pl.sdsig + sl * d; double* ga = sm + pl.sga + sl * d;
    double* Ht = sm + pl.sHt + sl * dd; double* gh = sm + pl.sgh + sl * 8;
    auto pre = [&](int e) {
      if (RSpre < 0) return split_sum(p1, RS1, nout1, e * (-RSpre) + q1);  // V_e . u from the fused product
      return split_sum(ppre, RSpre, nout_pre, aidx * q1 + e);
    };
    auto one = [&](int e) { return split_sum(p1, RS1, nout1, e); };
    auto gramf = [&](int p, int q) { return split_sum(pg, RSg, noutg, goff + p * gld + q); };
    auto hes = [&](int which, int e) { return split_sum(phess, which ? RShw : RShc, np * 2 * (T2 + 1), (aidx * 2 + which) * (T2 + 1) + e); };
    const double mu = pre(0);
    const double var = P.k0 - one(0);  // rbs.jl:528 (kx.w == |L^-1 kx|^2)
    const double sigma = sqrt(var), isg = 1.0 / sigma;
    const GPart g = rule_eval(P.rule_id, P.sigma_tol, mu, sigma, P.theta1, fstar);
    bool fin = isfinite(g.g);
    for (int p = lane; p < d; p += 32) {
      double m = pre(1 + p), sg = -one(1 + p) * isg;  // rbs.jl:514, 529
      double a = g.g_mu * m + g.g_sig * sg;            // rbs.jl:567
      dmu[p] = m; dsig[p] = sg; ga[p] = a;
      fin = fin && isfinite(a);
    }
    __syncwarp();
    const double bC = hes(0, T2), bW = hes(1, T2);
    for (int e = lane; e < T2; e += 32) {
      const int pq = tbld[e], p = pq & 0xff, q = pq >> 8;
      double gram = gramf(p, q), hc = hes(0, e), hw = hes(1, e);
      if (p == q) { hc += bC; hw += bW; }
      double hs = (-dsig[p] * dsig[q] - gram - hw) * isg;                                                            // rbs.jl:541-546
      double href = g.g_mumu * dmu[p] * dmu[q] + g.g_mu * hc + g.g_sigsig * dsig[p] * dsig[q] + g.g_sig * hs;        // rbs.jl:568
      double htrue = href + g.g_musig * (dmu[p] * dsig[q] + dsig[p] * dmu[q]);
      if (Href) { Href[p * d + q] = href; Href[q * d + p] = href; }
      Ht[p * d + q] = -htrue; Ht[q * d + p] = -htrue;
      fin = fin && isfinite(htrue);
    }
    fin = __all_sync(FULL, fin);
    if (lane == 0) {
      gh[0] = g.g; gh[1] = g.g_mu; gh[2] = g.g_sig; gh[3] = g.g_muth; gh[4] = g.g_sigth; gh[5] = sigma; gh[6] = mu;
      gh[7] = fin ? 1.0 : 0.0;
    }
    __syncwarp();
  }

  // ------------------------------------------------------------------------------------------------
  // One step of the per-start state machine (trust-region Newton on the merit -log(alpha) / -alpha, specified in DESIGN.md
  // section 4; modelled on tr_newton, optim.jl:68-114), run by ONE WARP for slot `sl` right after assemble_warp(). Returns
  // true (uniformly) if the slot has a new trial point in sxt and stays active.
  // ------------------------------------------------------------------------------------------------
  __device__ bool slot_logic_warp(int sl, bool single = false) {
    const int d = P.d, dd = d * d;
    const rbo_solver_opts& o = P.so;
    double* x = sm + pl.sx + sl * d; double* xt = sm + pl.sxt + sl * d; double* g = sm + pl.sg + sl * d;
    double* H = sm + pl.sH + sl * dd;
    double* Ht = sm + pl.sHt + sl * dd;  // trial Hessian from the evaluation; dead after the accept decision, then the scratch of the trust-region step
    double* A = Ht;
    const double* ga = sm + pl.sga + sl * d; const double* gh = sm + pl.sgh + sl * 8;
    int* fr = sfr + 32 * sl;
    TR_T(l0_);
    // per-slot scalars: merit f, trust-region radius, predicted decrease of the pending trial, alpha at x
    double f = (sm + pl.sf)[sl], Delta = (sm + pl.slam)[sl], pred = (sm + pl.spred)[sl], alpha = (sm + pl.shs)[sl];
    int iters = siter[sl], tries = stry[sl], flg = sflag[sl];  // flg bit 0: log merit, bit 1: the pending trial hit the trust-region boundary
    double sn = (sm + pl.ssn)[sl];
    const double at = gh[0];
    bool fin = gh[7] != 0.0;
    const int ph = phase[sl];
    __syncwarp();
    auto store = [&](int status, bool keep) {
      if (lane == 0) {
        (sm + pl.sf)[sl] = f; (sm + pl.slam)[sl] = Delta; (sm + pl.spred)[sl] = pred; (sm + pl.shs)[sl] = alpha; (sm + pl.ssn)[sl] = sn;
        siter[sl] = iters; stry[sl] = tries; sflag[sl] = flg;
        if (!keep) sstat[sl] = status;
        phase[sl] = keep ? 1 : 2;
      }
      __syncwarp();
      return keep;
    };
    const double* lb = sm + pl.sbnd; const double* ub = lb + d;
    const int T2 = d * (d + 1) / 2;
    auto accept_state = [&](double fnew) {  // (x, alpha, f, g, H) <- trial evaluation, in the merit's variables; fnew = merit at the trial point
      alpha = at;
      f = fnew;
      if (flg & 1) {
        const double ia = 1.0 / at;
        for (int a = lane; a < d; a += 32) { x[a] = xt[a]; g[a] = -ga[a] * ia; }
        __syncwarp();
        for (int e = lane; e < T2; e += 32) {  // H = Ht / alpha + (ga / alpha)(ga / alpha)', both triangles
          const int pq = tbld[e], p = pq & 0xff, q = pq >> 8;
          const double hv = Ht[p * d + q] * ia + g[p] * g[q];
          H[p * d + q] = hv; H[q * d + p] = hv;
        }
      } else {
        for (int a = lane; a < d; a += 32) { x[a] = xt[a]; g[a] = -ga[a]; }
        for (int i = lane; i < dd; i += 32) H[i] = Ht[i];
      }
      __syncwarp();
    };
    if (lane == 0) sevals[sl] += 1;
    bool fresh;
    if (ph == 0) {
      if (!fin) {
        for (int a = lane; a < d; a += 32) x[a] = xt[a];
        alpha = nan("");
        return store(RBO_SOLVE_NAN, false);
      }
      flg = (P.rule_id != RBO_RULE_LCB && at > 0.0) ? 1 : 0;
      accept_state((flg & 1) ? -log(at) : -at);
      if (single) return store(RBO_SOLVE_CONVERGED, false);  // one evaluation at a given point (extended tape): no iteration
      double wmax = 0.0;
      for (int a = 0; a < d; ++a) wmax = fmax(wmax, P.ubs[a] - P.lbs[a]);
      Delta = fmin(o.delta0_box * wmax, o.delta0_ell * P.kern.th[0]);
      iters = 0; tries = 0;
      fresh = true;
    } else {
      fin = fin && (!(flg & 1) || at > 0.0);
      const double ft = fin ? ((flg & 1) ? -log(at) : -at) : 0.0;
      const double rho = fin ? (f - ft) / pred : -1.0;
      if (fin && rho >= o.eta) {  // optim.jl:99
        accept_state(ft);
        if (rho > 0.75 && (flg & 2) && sn >= 0.8 * Delta) {  // optim.jl:95-96
          double dm2 = 0.0;
          for (int a = 0; a < d; ++a) { const double wd = P.ubs[a] - P.lbs[a]; dm2 = fma(wd, wd, dm2); }
          Delta = fmin(2.0 * Delta, sqrt(dm2));
        } else if (rho < 0.25) Delta = 0.25 * sn;  // optim.jl:93-94
        tries = 0;
        iters += 1;
        if (iters >= o.maxit) return store(RBO_SOLVE_MAXIT, false);
        fresh = true;
      } else {
        Delta = 0.25 * fmin(Delta, sn);
        tries += 1;
        if (tries >= o.maxtry) return store(RBO_SOLVE_STALLED, false);
        fresh = false;
      }
    }
    // active set (lane a <-> coordinate a) and projected gradient of alpha
    const bool in = lane < d;
    const double xa = in ? x[lane] : 0.0, gg = in ? g[lane] : 0.0;
    const double lba = in ? lb[lane] : 0.0, uba = in ? ub[lane] : 0.0;
    const bool act = in && ((xa <= lba && gg > 0.0) || (xa >= uba && gg < 0.0));
    const bool isfree = in && !act;
    const unsigned fmask = __ballot_sync(FULL, isfree);
    const int nfree = __popc(fmask);
    if (isfree) fr[__popc(fmask & ((1u << lane) - 1u))] = lane;  // free coordinates in ascending order
    double pg = warp_max_nonneg(isfree ? fabs(gg) : 0.0);
    if (flg & 1) pg *= alpha;
    __syncwarp();
    if (fresh && pg <= o.gtol * fmax(1.0, fabs(alpha))) return store(RBO_SOLVE_CONVERGED, false);
    const int myc = lane < nfree ? fr[lane] : 0;  // coordinate owned by this lane in the reduced system
    const double xmax = warp_max_nonneg(fabs(xa));
    for (;;) {
      double* yv = sm + pl.sdmu + sl * d;  // grad mu / grad sigma / grad alpha of the evaluation are not needed any more: scratch
      TR_T(l1_); TR_ADD(1, l0_, l1_); TR_ADD(0, 0, 1);
      const bool hit = (nfree >= 2 && nfree <= 16) ? tr_step16(H, g, fr, nfree, d, Delta, sm + pl.sdsig + sl * d, sm + pl.sga + sl * d, yv)
                                                  : tr_step_warp(H, g, fr, nfree, d, Delta, A, yv);
      const double t = lane < nfree ? yv[lane] : 0.0;
      TR_T(l2_); TR_ADD(2, l1_, l2_);
      if (in) xt[lane] = xa;
      __syncwarp();
      if (lane < nfree) xt[myc] = fmin(fmax(x[myc] + t, lb[myc]), ub[myc]);
      __syncwarp();
      const double sa = in ? xt[lane] - xa : 0.0;
      const double smax = warp_max_nonneg(fabs(sa));
      if (smax <= o.xtol * fmax(1.0, xmax)) { sn = sqrt(warp_sum(sa * sa)); return store(RBO_SOLVE_STEP_TINY, false); }
      // H s: the step goes to shared memory (the scratch is free again), then lane a walks row a of H
      if (in) yv[lane] = sa;
      __syncwarp();
      double hsv = 0.0;
      if (in) {
        const double* Hr = H + lane * d;
        if ((d & 1) == 0) {  // rows and the scratch are 16-byte aligned: two entries per load
          double h1 = 0.0;
          for (int b = 0; b < d; b += 2) {
            const double2 hh = *reinterpret_cast<const double2*>(Hr + b), ss = *reinterpret_cast<const double2*>(yv + b);
            hsv = fma(hh.x, ss.x, hsv); h1 = fma(hh.y, ss.y, h1);
          }
          hsv += h1;
        } else for (int b = 0; b < d; ++b) hsv = fma(Hr[b], yv[b], hsv);
      }
      // |s|^2, g's, s'Hs in the same shuffle rounds
      double r0 = sa * sa, r1 = gg * sa, r2 = sa * hsv;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        r0 += __shfl_xor_sync(FULL, r0, off); r1 += __shfl_xor_sync(FULL, r1, off); r2 += __shfl_xor_sync(FULL, r2, off);
      }
      sn = sqrt(r0);
      const double gs = r1, sHs = r2;
      const double pr = -(gs + 0.5 * sHs);  // mu_diff of optim.jl:88 for the projected step
      if (!(pr > 0.0)) {
        Delta = 0.25 * fmin(Delta, sn);
        tries += 1;
        if (tries >= o.maxtry) return store(RBO_SOLVE_STALLED, false);
        continue;
      }
      const bool pred_tiny = pr <= o.pred_tol * fmax(1.0, fabs(f));
      if (!hit && (pred_tiny || smax <= o.stol * fmax(1.0, xmax))) {
        // final interior Newton step, taken without another evaluation; alpha follows the model
        for (int a = lane; a < d; a += 32) x[a] = xt[a];
        alpha = (flg & 1) ? alpha * exp(pr) : alpha + pr;
        return store(RBO_SOLVE_FINAL_STEP, false);
      }
      if (pred_tiny) return store(RBO_SOLVE_PRED_TINY, false);
      pred = pr;
      flg = (flg & 1) | (hit ? 2 : 0);
      TR_T(l3_); TR_ADD(3, l2_, l3_);
      return store(0, true);
    }
  }

  // loads start `sid` into slot `sl`
  __device__ void load_start(int sl, int sid) {
    const int d = P.d;
    phase[sl] = 0; sstat[sl] = RBO_SOLVE_MAXIT; siter[sl] = 0; stry[sl] = 0; sevals[sl] = 0; sstart[sl] = sid; sflag[sl] = 0;
    for (int a = 0; a < d; ++a) {
      double v = __ldg(P.starts + (size_t)sid * d + a);
      (sm + pl.sxt)[sl * d + a] = fmin(fmax(v, P.lbs[a]), P.ubs[a]);
    }
  }

  // ------------------------------------------------------------------------------------------------
  // multistart_base_solve! (rbf_optim.jl:68-101 / :103-134): all S starts through W slots in lock-step rounds.
  // The coefficients of the active surrogate must be in column CCOL. Result: bestx (argmax), misc[0] = -alpha
  // there, si[I_BEST] (or -1), si[I_EVALS]. Ties resolve to the lowest start index (findmin: first minimum).
  // ------------------------------------------------------------------------------------------------
  // single = true: ONE evaluation at `bestx` through slot 0 (no clamping, no start list): afterwards slot 0 holds mu, sigma, alpha,
  // grad mu, grad sigma and the reference's H alpha there (the extended tape of the step-level parity tests).
  __device__ void multistart(size_t tape_off, bool single = false, bool first = false) {
    const int d = P.d, W = P.W, q1 = d + 1;
    __syncthreads();
    // Longest first: the starts are handed out in descending order of the evaluations they needed in the previous multistart of
    // this CTA (the same start points, a surrogate that differs by one fantasy observation) -- for the first step of a trajectory:
    // in the first step of the CTA's previous trajectory (ties and the very first multistart: start order). With 8+2 starts on
    // 5 slots the lock-step rounds end when the slowest start ends; one start of C3 systematically needs 15 evaluations against a
    // mean of 8 -- begun in the first wave instead of the second it no longer sets the tail (rounds per trajectory 124 -> 105).
    // The result does not depend on the order: the argmin compares (value, start index).
    const unsigned short* evsrc = first ? evfirst : evprev;
    for (int i = tid; i < P.S; i += RBO_THREADS) {
      const unsigned e = evsrc[i];
      int r = 0;
      for (int j = 0; j < P.S; ++j) { const unsigned ej = evsrc[j]; r += (ej > e || (ej == e && j < i)) ? 1 : 0; }
      sorder[r] = (unsigned short)i;
    }
    __syncthreads();
    if (tid == 0) {
      si[I_BEST] = -1; si[I_EVALS] = 0; misc[0] = 0.0;
      const int n0 = single ? 1 : min(W, P.S);
      for (int i = 0; i < n0; ++i) { alist[i] = i; load_start(i, single ? i : (int)sorder[i]); }
      if (single) for (int a = 0; a < d; ++a) (sm + pl.sxt)[a] = bestx[a];
      si[I_NACT] = n0; si[I_NEXT] = single ? P.S : n0;
    }
    __syncthreads();
    int nact = si[I_NACT];
    PT_DECL;
    const long long round_cap = (long long)P.S * (P.so.maxit + 2) * (P.so.maxtry + 2);  // no start can use more evaluations than that
    long long rounds_ = 0;
    while (nact > 0) {
      if (++rounds_ > round_cap) { if (tid == 0) P.work_counter[WC_EVAL_CAP] = 1; break; }
      auto pt = [&](int s) { return (const double*)(sm + pl.sxt + alist[s] * d); };
      auto cb = [&](int s) { return alist[s] * P.CS; };
      PT_MARK(9);
      fill_columns(nact, pt, cb);
      for (int i = tid; i < nact * q1; i += RBO_THREADS) { int s = i / q1; colidx[i] = alist[s] * P.CS + (i - s * q1); }
      // mu = kx.c = (L^-1 kx).(L^-1 y) = v0.u and grad mu = V_g' u (rbs.jl:513-514) ride along with the Gram product after the solve
      const int nbq = nblk16(q1);
      __syncthreads();
      PT_MARK(0);
      tri_solve<true>(nact * q1, nf);
      const int q2 = q1 + 1;  // B columns: the slot's q1 solved columns and u
      for (int s = tid; s < nact; s += RBO_THREADS) set_item(s, alist[s] * P.CS, q1, alist[s] * P.CS, q2, s * q1 * q2, UCOL);  // |v0|^2, V_p.v0, V_p.V_q | V_p.u
      __syncthreads();
      PT_MARK(2);
      const int RS1 = choose_rs(nact * nbq * nblk16(q2)), RSg = RS1;
      colprod(nact, nact * q1 * q2, sm + pl.ppost, RS1);
      for (int i = tid; i < nact; i += RBO_THREADS) colidx[i] = alist[i] * P.CS;
      __syncthreads();
      PT_MARK(3);
      tri_solve<false>(nact, nf);  // w = L^-T v0 (rbs.jl:525)
      __syncthreads();
      PT_MARK(4);
      const int nbd = nblk16(d);
      const int RShw = max(1, min(P.RSh, RBO_NWARPS / (nact * (nbd * (nbd + 1) / 2)))), RShc = RShw;  // row splits: enough to occupy every warp
      hess_sums<3>(nact, pt, cb, cb, RShw);
      __syncthreads();
      PT_MARK(5);
      // the row-split partial sums are added (fixed order) by all threads, in place: the per-start warps then read one value per
      // entry instead of RS -- their time is what the other eleven warps wait for
      {
        const int n1 = nact * q1 * q2, nh = nact * 2 * (d * (d + 1) / 2 + 1);
        double* pp = sm + pl.ppost; double* ph = sm + pl.phess;
        if (RS1 > 1) for (int i = tid; i < n1; i += RBO_THREADS) { double a_ = pp[i]; for (int r = 1; r < RS1; ++r) a_ += pp[(size_t)r * n1 + i]; pp[i] = a_; }
        if (RShw > 1) for (int i = tid; i < nh; i += RBO_THREADS) { double a_ = ph[i]; for (int r = 1; r < RShw; ++r) a_ += ph[(size_t)r * nh + i]; ph[i] = a_; }
        __syncthreads();
      }
      // per-start logic: one warp per active slot
      for (int s = warp; s < nact; s += RBO_NWARPS) {
        const int sl = alist[s];
        assemble_warp(sl, s, nact, -q2, sm + pl.ppost + s * q1 * q2, nact * q1 * q2, 1, sm + pl.ppost, nact * q1 * q2, s * q1 * q2 + q2 + 1, q2, 1, 1, 1, misc[1], single ? sm + pl.sHref : nullptr);
#ifdef RBO_PHASE_TIMERS
        long long ta_ = clock64();
        if (tid == 0) atomicAdd(&g_phase_cycles[8], (unsigned long long)(ta_ - pt_t0));
#endif
        slot_logic_warp(sl, single);
#ifdef RBO_PHASE_TIMERS
        if (tid == 0) atomicAdd(&g_phase_cycles[14], (unsigned long long)(clock64() - ta_));
        if (lane == 0) { long long dt_ = clock64() - ta_; int b_ = (int)(dt_ / 4000); atomicAdd(&g_aux_cycles[b_ > 15 ? 15 : b_], 1ull); }  // duration histogram of the solver step
#endif
      }
      __syncthreads();
      PT_MARK(6);
      if (tid == 0) {
        int na2 = 0;
        for (int i = 0; i < nact; ++i) {
          const int sl = alist[i];
          if (phase[sl] == 1) { alist[na2++] = sl; continue; }
          // finished start: candidate (discard NaN, rbf_optim.jl:96), first minimum wins (rbf_optim.jl:97)
          const int sid = sstart[sl];
          const double f = -(sm + pl.shs)[sl];  // -alpha at the start's final point
          const double* x = sm + pl.sx + sl * d;
          bool bad = !isfinite(f);
          for (int a = 0; a < d; ++a) bad = bad || isnan(x[a]);
          si[I_EVALS] += sevals[sl];
          if (!single) { evprev[sid] = (unsigned short)min(sevals[sl], 65535); if (first) evfirst[sid] = evprev[sid]; }
          if (P.start_status && !single) P.start_status[tape_off + sid] = sstat[sl];
          if (P.start_iters && !single) P.start_iters[tape_off + sid] = siter[sl];
          if (!bad && (si[I_BEST] < 0 || f < misc[0] || (f == misc[0] && sid < si[I_BEST]))) {
            si[I_BEST] = sid; misc[0] = f;
            for (int a = 0; a < d; ++a) bestx[a] = x[a];
          }
          if (si[I_NEXT] < P.S) { load_start(sl, (int)sorder[si[I_NEXT]]); si[I_NEXT] += 1; alist[na2++] = sl; }
        }
        si[I_NACT] = na2;
      }
      __syncthreads();
      PT_MARK(7);
#ifdef RBO_PHASE_TIMERS
      if (tid == 0) atomicAdd(&g_phase_cycles[15], 1ull);
#endif
      nact = si[I_NACT];
    }
    if (tid == 0 && si[I_BEST] < 0) {
      if (si[I_TSTATUS] == RBO_TRAJ_OK) si[I_TSTATUS] = RBO_TRAJ_ALL_STARTS_NAN;
      for (int a = 0; a < d; ++a) bestx[a] = nan("");
    }
    __syncthreads();
  }

  // ================================================================================================
  // Phases of one trajectory m, each called from exactly one place in the kernel. The joint draw + condition! and the adjoint
  // stay in the kernel body: as member functions they moved ptxas's spills into the multistart loop (268 B of spill stores
  // instead of 104 in the shared-memory build).
  // ================================================================================================
  // Sample index (normals, dual directions, forced locations, nodes) and starting point of trajectory m: recomputed at the few
  // places they are needed instead of being kept live across the whole trajectory.
  __device__ __forceinline__ int sample(int m) const { return m % P.Ms; }
  __device__ __forceinline__ int start_point(int m) const { return m / P.Ms; }

  // trajectory init: reset!(fs) (rbs.jl:476-480)
  __device__ __forceinline__ void begin_trajectory() {
    const int N8 = P.N8, NR = P.NR, RP = P.RP;
    for (int i = tid; i < (N8 + RBO_MAXFAN) * 8; i += RBO_THREADS) Fp[i] = 0.0;
    for (int i = tid; i < 64; i += RBO_THREADS) G[i] = ((i >> 3) == (i & 7)) ? 1.0 : 0.0;
    for (int i = tid; i < NR; i += RBO_THREADS) { double c = (i < N8) ? __ldg(P.c0 + i) : 0.0; cst[i] = c; V[(size_t)i * RP + CCOL] = c; }
    for (int i = tid; i < NR; i += RBO_THREADS) { double u0 = (i < N8) ? __ldg(P.u0 + i) : 0.0; u[i] = u0; V[(size_t)i * RP + UCOL] = u0; }
    __syncthreads();
    if (tid < 8) Fp[(size_t)(N8 + tid) * 8 + tid] = 1.0;  // inverse of the identity fantasy block
    if (tid == 0) { misc[1] = P.ymin_base; si[I_TSTATUS] = RBO_TRAJ_OK; }
    nf = 0;
    __syncthreads();
  }

  // Chooses the location x_step into bestx: x0 at step 0, else the policy solve (or the caller's x-path when teacher-forced),
  // followed by the extended tape's single evaluation at the chosen point. Holds the one call of multistart().
  __device__ __forceinline__ void choose_location(int m, int step) {
    const int d = P.d, h = P.h;
    const bool myopic = (P.flags & RBO_FLAG_MYOPIC_INTERNAL) != 0;
    if (step == 0) {
      if (tid < d) bestx[tid] = P.x0_batch ? __ldg(P.x0_batch + (size_t)start_point(m) * d + tid) : P.x0[tid];  // rollout.jl:46
      __syncthreads();
    } else {
      for (int pass = 0; pass < 2; ++pass) {
        const bool single = pass == 1;  // pass 1: the extended tape's evaluation at the chosen point
        if (single && (myopic || !(P.flags & RBO_FLAG_TAPE_EX))) break;
        if (!single && !myopic && (P.flags & RBO_FLAG_TEACHER_FORCED)) {
          // teacher forcing: the caller's x-path, or (RBO_FLAG_REPLAY_TAPE) the x-path the previous rollout left on the device
          if (tid < d) bestx[tid] = (P.flags & RBO_FLAG_REPLAY_TAPE) ? P.xs[((size_t)m * (h + 1) + step) * d + tid] : P.x_forced[((size_t)sample(m) * h + (step - 1)) * d + tid];
          if (tid == 0) { si[I_EVALS] = 0; misc[0] = nan(""); }
        } else {
          // multistart_base_solve!(fs, xnext; fantasy_index = step-1) (rollout.jl:58-66, rbf_optim.jl:68-101) -- column CCOL holds
          // cs[fantasy_index + 2] (1-based) = the coefficients after `step` fantasies -- or, myopic,
          // multistart_base_solve!(::Surrogate, ...) (rbf_optim.jl:103-134): the base surrogate, no fantasies
          if (single) __syncthreads();
          multistart(single ? 0 : (myopic ? (size_t)m * P.S : ((size_t)m * h + (step - 1)) * P.S), single, !single && step == 1);
        }
        __syncthreads();
        if (!single) {
          if (!myopic && tid == 0) {
            if (P.n_evals) P.n_evals[(size_t)m * h + step - 1] = si[I_EVALS];
            if (P.alphas) P.alphas[(size_t)m * h + step - 1] = -misc[0];
          }
        } else {
          // extended tape (SURVEY.md section 7.4): sx = fs(x_step, theta; fantasy_index = step - 1), the surrogate evaluation the
          // policy solve of this step maximised (rbs.jl:482-581); slot 0 holds it after the single evaluation
          const size_t o = (size_t)m * h + step - 1;
          const double* gh = sm + pl.sgh;
          if (tid == 0) { P.t_mu[o] = gh[6]; P.t_sigma[o] = gh[5]; if (P.alphas) P.alphas[o] = gh[0]; }
          for (int i = tid; i < d; i += RBO_THREADS) { P.t_dmu[o * d + i] = (sm + pl.sdmu)[i]; P.t_dsigma[o * d + i] = (sm + pl.sdsig)[i]; }
          for (int i = tid; i < d * d; i += RBO_THREADS) P.t_Halpha[o * d * d + i] = (sm + pl.sHref)[i];
          __syncthreads();
        }
      }
    }
  }

  // the result of the myopic solve (rbf_optim.jl:103-134): the maximiser and its value
  __device__ __forceinline__ void store_myopic(int m) {
    const int d = P.d;
    if (tid < d) P.xs[(size_t)m * d + tid] = bestx[tid];
    if (tid == 0) {
      P.values[m] = -misc[0];
      if (P.n_evals) P.n_evals[m] = si[I_EVALS];
      if (P.status) P.status[m] = si[I_TSTATUS];
      if (P.best_index) P.best_index[m] = si[I_BEST];
      if (P.grad_case) P.grad_case[m] = 0;
    }
  }

  // resolve (rollout.jl:108-111): the value, the index t of the best observation, the gradient case, and the trajectory's tape
  __device__ __forceinline__ void resolve(int m) {
    const int d = P.d, h = P.h;
    if (tid == 0) {
      double best = yf[0];
      int t = 0;
      for (int j = 1; j <= h; ++j) if (yf[j] < best) { best = yf[j]; t = j; }  // findmin: first minimum (rollout.jl:77-82)
      double val = fmax(P.fmini - best, 0.0);
      if (P.flags & RBO_FLAG_GAUSS_HERMITE) {
        // resolve(gho; fmini) (observables.jl:66-72); get_gradient(gho; at) = weights[at] * gradients[:, at] (observables.jl:157)
        const double* wq = P.gh_weights + (size_t)sample(m) * P.gh_depth;
        val = __ldg(wq + t) * val / 1.7724538509055159;
        for (int j = 0; j <= h; ++j)
          for (int a = 0; a < d; ++a) gyf[j * d + a] *= __ldg(wq + j);
      }
      P.values[m] = val;
      si[I_T] = t;
      int tc = 0;
      if (P.mode == RBO_MODE_VALUE_GRAD) tc = (P.fmini <= best) ? 1 : (t == 0 ? 2 : 3);  // rollout.jl:241-251
      si[I_CASE] = tc;
      if (P.best_index) P.best_index[m] = t;
      if (P.grad_case) P.grad_case[m] = tc;
    }
    __syncthreads();
    if (P.xs) for (int i = tid; i < (h + 1) * d; i += RBO_THREADS) P.xs[(size_t)m * (h + 1) * d + i] = Xf[i];
    if (P.gys) for (int i = tid; i < (h + 1) * d; i += RBO_THREADS) P.gys[(size_t)m * (h + 1) * d + i] = gyf[i];
    if (P.ys) for (int i = tid; i <= h; i += RBO_THREADS) P.ys[(size_t)m * (h + 1) + i] = yf[i];
    __syncthreads();
  }
};

}  // namespace

__global__ void __launch_bounds__(RBO_THREADS, 1) RBO_KERNEL_NAME(const __grid_constant__ DevProblem P) {
  extern __shared__ __align__(128) double smem[];
  K k(P, smem);
  const int tid = k.tid, d = P.d, N8 = P.N8, NR = P.NR, RP = P.RP, h = P.h, q1 = d + 1;
  double* bestx = k.bestx;
  double* misc = k.misc;  // misc[0] best f, misc[1] fstar, misc[2..7] scalars, misc[8..] scratch
  int* si = k.si;
  k.build_tables();
  for (int i = tid; i < 2 * d; i += RBO_THREADS) smem[P.pl.sbnd + i] = i < d ? P.lbs[i] : P.ubs[i - d];
  for (int i = tid; i < P.S; i += RBO_THREADS) { k.evprev[i] = 0; k.evfirst[i] = 0; }
  k.pipe_init();
  for (int i = tid; i < NR * RP; i += RBO_THREADS) k.V[i] = 0.0;  // rows beyond the fantasy block are read (times exact zeros of L0's padding) but never written
  if (P.xsm) for (int i = tid; i < d * N8; i += RBO_THREADS) k.Xs[(i / N8) * P.XP + (i % N8)] = __ldg(P.Xb + i);
  __syncthreads();

  for (;;) {
    __syncthreads();
    if (tid == 0) {
      // dynamic scheduler; with an order from the previous launch the trajectories are handed out longest-first (LPT), which
      // shortens the tail of the persistent grid -- the per-trajectory results do not depend on the order
      const int i = atomicAdd(P.work_counter + WC_SCHED, 1);
      si[I_M] = (i < P.M) ? (P.order ? P.order[i] : i) : P.M;
    }
    __syncthreads();
    const int m = si[I_M];
    if (m >= P.M) break;

    k.begin_trajectory();
    // multistart() is inlined at exactly ONE call site, in choose_location() (a second or third copy pushes the kernel over its
    // register budget): the myopic solve, the policy solves of the rollout and the single evaluation of the extended tape all go
    // through it.
    const bool myopic = (P.flags & RBO_FLAG_MYOPIC_INTERNAL) != 0;
    for (int step = myopic ? 1 : 0; step <= (myopic ? 1 : h); ++step) {
      k.choose_location(m, step);
      if (myopic) {
        k.store_myopic(m);
        break;
      }

      // ============ joint draw at x_step (observables.jl:106-121, rbs.jl:588-611) and condition! (rbs.jl:431-441) ============
      {
        PT_DECL;
        auto pt = [&](int) { return (const double*)bestx; };
        auto cb0 = [&](int) { return 0; };
        k.fill_columns(1, pt, cb0);
        k.set_column(k.UCOL, k.u);
        for (int i = tid; i < q1; i += RBO_THREADS) k.colidx[i] = i;
        if (tid == 0) k.set_item(0, 0, q1, k.CCOL, 1, 0);  // mu, grad mu
        __syncthreads();
        const int nbq = K::nblk16(q1);
        const int RSpre = k.choose_rs(nbq);
        k.colprod(1, q1, smem + k.pl.ppre, RSpre);
        __syncthreads();
        k.tri_solve<true>(q1, k.nf);
        if (tid == 0) { k.set_item(0, 0, q1, 0, q1, 0); k.set_item(1, 0, 1, k.UCOL, 1, q1 * q1); }  // V'V and l . u
        __syncthreads();
        const int nsg = q1 * q1 + 1;
        const int RSpost = k.choose_rs(nbq * nbq + 1);
        k.colprod(2, nsg, smem + k.pl.ppost, RSpost);
        __syncthreads();
        // Sigma = Dk(0) - A K^-1 A' = Dk(0) - V'V (rbs.jl:531-536)
        double* Sg = misc + 8;  // (d+1) x (d+1)
        for (int e = tid; e < nsg; e += RBO_THREADS) {
          const double acc = split_sum(smem + k.pl.ppost, RSpost, nsg, e);
          if (e < q1 * q1) {
            const int p = e / q1, q = e - p * q1;
            const double dk = (p == q) ? (p == 0 ? P.k0 : -P.d2k0) : 0.0;  // eval_Dk(kernel, 0) rbf.jl:152-159
            if (p <= q) { Sg[p * q1 + q] = dk - acc; Sg[q * q1 + p] = dk - acc; }  // Symmetric(...) takes the upper triangle
            if (p == 0) misc[8 + q1 * q1 + q1 + q] = acc;  // [|v0|^2, V_q.v0]: sigma and grad sigma of the Gauss-Hermite observable
            if (e == 0) misc[4] = acc;  // |l|^2
          } else misc[5] = acc;         // l . u
        }
        if (tid < q1) misc[8 + q1 * q1 + tid] = split_sum(smem + k.pl.ppre, RSpre, q1, tid);  // [mu, grad mu]
        __syncthreads();
        if (tid == 0) {
          const int r = k.nf;  // index of the new fantasy row
          const double* dmu = misc + 8 + q1 * q1;
          double yv;
          if (P.flags & RBO_FLAG_GAUSS_HERMITE) {
            // GaussHermiteObservable functor (observables.jl:54-64): y = mu + sqrt(2) sigma node, grad y = grad mu + sqrt(2) grad sigma node
            const double* raw = misc + 8 + q1 * q1 + q1;
            const double var = P.k0 - raw[0];  // rbs.jl:528
            if (!(var >= 0.0) && si[I_TSTATUS] == RBO_TRAJ_OK) si[I_TSTATUS] = RBO_TRAJ_NEG_VARIANCE;
            const double sigma = sqrt(var), node = __ldg(P.gh_nodes + (size_t)k.sample(m) * P.gh_depth + step), s2n = 1.4142135623730951 * node;
            yv = dmu[0] + s2n * sigma;
            for (int a = 0; a < d; ++a) k.gyf[r * d + a] = dmu[1 + a] + s2n * (-raw[1 + a] / sigma);  // rbs.jl:529
          } else {
            bool pd = chol_inplace(Sg, q1, q1);
            if (!pd && si[I_TSTATUS] == RBO_TRAJ_OK) si[I_TSTATUS] = RBO_TRAJ_NOT_PD_JOINT;
            const double* rnm = P.rn + (size_t)k.sample(m) + (size_t)P.Ms * q1 * step;
            yv = dmu[0] + Sg[0] * __ldg(rnm);
            for (int a = 0; a < d; ++a) {
              double v = dmu[1 + a];
              for (int j = 0; j <= a + 1; ++j) v += Sg[(a + 1) * q1 + j] * __ldg(rnm + (size_t)P.Ms * j);
              k.gyf[r * d + a] = v;
            }
          }
          k.yf[r] = yv;
          for (int a = 0; a < d; ++a) k.Xf[r * d + a] = bestx[a];
          misc[1] = fmin(misc[1], yv);
          // new Cholesky row (rbs.jl:403-420): l = L^-1 k (already in column 0), l_rr = sqrt(k0 + sigma_n2 - l.l)
          double s = (P.k0 + P.sigma_n2) - misc[4];
          if (!(s > 0.0) && si[I_TSTATUS] == RBO_TRAJ_OK) si[I_TSTATUS] = RBO_TRAJ_NOT_PD_ROW;
          double lrr = sqrt(s);
          for (int j = 0; j < r; ++j) k.G[r * 8 + j] = k.V[(size_t)(N8 + j) * RP];
          k.G[r * 8 + r] = lrr;
          // inverse of the lower-triangular 8x8 fantasy block, stored k-major: Fp[(N8 + kk)*8 + rr] = Ginv[rr][kk]
          for (int cc = 0; cc < 8; ++cc) {
            double col[8];
            for (int rr = 0; rr < 8; ++rr) {
              double t = (rr == cc) ? 1.0 : 0.0;
              for (int j = cc; j < rr; ++j) t -= k.G[rr * 8 + j] * col[j];
              col[rr] = (rr < cc) ? 0.0 : t / k.G[rr * 8 + rr];
            }
            for (int rr = 0; rr < 8; ++rr) k.Fp[(size_t)(N8 + cc) * 8 + rr] = col[rr];
          }
          k.u[N8 + r] = (yv - misc[5]) / lrr;
          k.V[(size_t)(N8 + r) * RP + k.UCOL] = k.u[N8 + r];  // the inner solves read u from its column
        }
        __syncthreads();
        {
          const int r = k.nf;
          for (int j = tid; j < N8; j += RBO_THREADS) k.Fp[(size_t)j * 8 + r] = k.V[(size_t)j * RP];
          for (int j = tid; j < NR; j += RBO_THREADS) k.V[(size_t)j * RP + k.CCOL] = k.u[j];
          if (tid == 0) k.colidx[0] = k.CCOL;
        }
        k.nf += 1;
        __syncthreads();
        // coefficients: c = L^-T (L^-1 y) (rbs.jl:422-429); L^-1 y is maintained incrementally in u
        k.tri_solve<false>(1, k.nf);
        __syncthreads();
        for (int j = tid; j < NR; j += RBO_THREADS) k.cst[(size_t)(step + 1) * NR + j] = k.V[(size_t)j * RP + k.CCOL];
        __syncthreads();
        PT_MARK(10);
      }
    }

    if (myopic) continue;
    k.resolve(m);
    // ============ gradient(T) (rollout.jl:233-277) ============
    PT_DECL;
    if (P.mode == RBO_MODE_VALUE_GRAD) {
      const int tc = si[I_CASE], t = si[I_T], nth = P.ntheta;
      if (tc == 1) {
        for (int i = tid; i < d; i += RBO_THREADS) P.grad_x[(size_t)m * d + i] = 0.0;
        for (int i = tid; i < nth; i += RBO_THREADS) P.grad_theta[(size_t)m * nth + i] = 0.0;
      } else if (tc == 2) {
        for (int i = tid; i < d; i += RBO_THREADS) P.grad_x[(size_t)m * d + i] = -k.gyf[i];  // -get_gradient(at = 1)
        for (int i = tid; i < nth; i += RBO_THREADS) P.grad_theta[(size_t)m * nth + i] = 0.0;
      } else {
        // adjoint work area: xbars[(j)*d], acc[(j)*d] for j = 0..8 ; ybars[0..11] ; gx[d] ; gth
        double* xbars = k.adj; double* accr = k.adj + 9 * d; double* ybars = k.adj + 18 * d; double* gxa = ybars + 12; double* gtha = gxa + d;
        for (int i = tid; i < 19 * d + 16; i += RBO_THREADS) k.adj[i] = 0.0;
        __syncthreads();
        if (tid == 0) ybars[t + 1] = 1.0;  // rollout.jl:256
        const int CB_RAW = 0, CB_SOL = d + 3, CB_U = 2 * d + 4, CB_Q = 3 * d + 5;
        const double* dd_m = P.dual_dirs ? P.dual_dirs + (size_t)k.sample(m) * h * d : nullptr;
        for (int i = t; i >= 1; --i) {
          // ---- re-evaluate policy solve i: fs(x_i, theta; fantasy_index = i-1) (rollout.jl:114-124) ----
          k.nf = i;
          const double* c = k.cst + (size_t)i * NR;
          const double* xi = k.Xf + (size_t)i * d;
          auto pt = [&](int) { return xi; };
          auto cbr = [&](int) { return CB_RAW; };
          auto cbs = [&](int) { return CB_SOL; };
          __syncthreads();
          k.fill_columns(1, pt, cbr);
          k.set_column(k.CCOL, c);
          __syncthreads();
          for (int idx = tid; idx < NR * q1; idx += RBO_THREADS) {
            int j = idx / q1, q = idx - j * q1;
            k.V[(size_t)j * RP + CB_SOL + q] = k.V[(size_t)j * RP + CB_RAW + q];
          }
          for (int q = tid; q < q1; q += RBO_THREADS) k.colidx[q] = CB_SOL + q;
          if (tid == 0) k.set_item(0, CB_RAW, q1, k.CCOL, 1, 0);
          __syncthreads();
          const int nbq = K::nblk16(q1), nbd = K::nblk16(d);
          const int RSpre = k.choose_rs(nbq);
          k.colprod(1, q1, smem + k.pl.ppre, RSpre);
          k.tri_solve<true>(q1, k.nf);
          __syncthreads();
          if (tid == 0) k.set_item(0, CB_SOL, q1, CB_SOL, q1, 0);
          __syncthreads();
          const int RSpost = k.choose_rs(nbq * nbq);
          k.colprod(1, q1 * q1, smem + k.pl.ppost, RSpost);
          __syncthreads();
          k.tri_solve<false>(q1, k.nf);  // w = SOL[:,0], Dw = SOL[:,1..d] (rbs.jl:525-526)
          __syncthreads();
          const int RShess = k.choose_rs(nbd * (nbd + 1) / 2);
          k.hess_sums<3>(1, pt, cbr, cbs, RShess);
          __syncthreads();
          if (k.warp == 0) {
            double fst = P.ymin_base;  // f* over the active slice y[1:N+i]
            for (int j = 0; j < i; ++j) fst = fmin(fst, k.yf[j]);
            k.assemble_warp(0, 0, 1, RSpre, smem + k.pl.ppost, q1 * q1, RSpost, smem + k.pl.ppost, q1 * q1, q1 + 1, q1, RSpost, RShess, RShess, fst, smem + k.pl.sHref);
            if (tid == 0) {
              misc[2] = fst;
              // ---- solve_dual_x for j = i (rollout.jl:150-191) with the contributions of later solves already pushed ----
              double* Hlu = smem + k.pl.sHt;  // slot-0 scratch (d x d): the trial Hessian is not needed here
              const double* Href = smem + k.pl.sHref;
              int piv[RBO_MAXD];
              double det;
              for (int a = 0; a < d; ++a) for (int b = 0; b < d; ++b) Hlu[a * d + b] = Href[a * d + b];
              lu_factor(Hlu, d, piv, &det);
              double* xb = xbars + (size_t)i * d;
              if (det < P.htol) {  // rollout.jl:159-161 (Q3)
                for (int a = 0; a < d; ++a) xb[a] = 0.0;
                misc[3] = 0.0;
              } else {
                for (int a = 0; a < d; ++a) xb[a] = -k.gyf[(size_t)(i - 1) * d + a] * ybars[i + 1] - accr[(size_t)i * d + a];  // rollout.jl:164-165 (Q4)
                for (int a = 0; a < d; ++a) for (int b = 0; b < d; ++b) Hlu[a * d + b] = Href[b * d + a];  // hessian(sx)' (rollout.jl:188)
                double det2;
                if (!lu_factor(Hlu, d, piv, &det2) && si[I_TSTATUS] == RBO_TRAJ_OK) si[I_TSTATUS] = RBO_TRAJ_SINGULAR_HESSIAN;
                lu_solve(Hlu, d, piv, xb);
                misc[3] = 1.0;
                // gather_q (rollout.jl:220-231): d2alpha/dx dtheta = grad_mu g_mu_theta + grad_sigma g_sigma_theta (rbs.jl:575-577)
                const double* gh = smem + k.pl.sgh; const double* dmu = smem + k.pl.sdmu; const double* dsg = smem + k.pl.sdsig;
                double s = 0.0;
                for (int a = 0; a < d; ++a) s += (dmu[a] * gh[3] + dsg[a] * gh[4]) * xb[a];
                gtha[0] += s;
              }
            }
          }
          __syncthreads();
          if (misc[3] == 0.0) continue;  // xbar_i = 0: every term it feeds vanishes
          const double* xb = xbars + (size_t)i * d;
          const double sigma = (smem + k.pl.sgh)[5];
          for (int p = 0; p < i; ++p) {
            // perturbation of fantasy location x_p inside policy solve i: d unit directions (spatial, rbs.jl:652-694)
            // and one direction dual_dirs[:, p] (data perturbation surrogate, rbs.jl:711-760)
            const int rowp = N8 + p;
            const double* xp = k.Xf + (size_t)p * d;
            // phase A: u_a = grad_k(X_a - X_p) . (-dx) per row (rbf.jl:210-228 restricted to the moved column)
            for (int j = tid; j < NR; j += RBO_THREADS) {
              double* rowU = k.V + (size_t)j * RP + CB_U; double* rowQ = k.V + (size_t)j * RP + CB_Q;
              if (!k.row_active(j) || j == rowp) { for (int q = 0; q < q1; ++q) { rowU[q] = 0.0; rowQ[q] = 0.0; } continue; }
              double rho2 = 0.0;
              for (int a = 0; a < d; ++a) { double r = k.xcoord(j, a) - xp[a]; rho2 = fma(r, r, rho2); }
              double psi, a_, b_, gb_;
              kern_radial(P.kern, rho2, psi, a_, b_, gb_);
              if (!(rho2 > 0.0)) b_ = 0.0;
              double cp = k.V[(size_t)rowp * RP + k.CCOL], rd = 0.0;
              for (int a = 0; a < d; ++a) {
                double r = k.xcoord(j, a) - xp[a];
                double uu = -b_ * r;
                rowU[a] = uu; rowQ[a] = uu * cp;
                if (dd_m) rd += r * dd_m[(size_t)p * d + a];
              }
              double ud = -b_ * rd;
              rowU[d] = ud; rowQ[d] = ud * cp;
            }
            if (tid == 0) { k.set_item(0, CB_U, q1, k.CCOL, 1, 0); k.set_item(1, CB_U, q1, CB_SOL, 1, q1); }  // u.c ; u.w
            __syncthreads();
            // phase B: (dK c)_p = u.c ; u.w
            const int RSb = k.choose_rs(2 * nbq);
            k.colprod(2, 2 * q1, smem + k.pl.ppost, RSb);
            __syncthreads();
            double* uw = misc + 8;  // [q1]
            for (int e = tid; e < 2 * q1; e += RBO_THREADS) {
              const double acc = split_sum(smem + k.pl.ppost, RSb, 2 * q1, e);
              if (e >= q1) uw[e - q1] = acc; else k.V[(size_t)rowp * RP + CB_Q + e] = acc;
            }
            for (int q = tid; q < q1; q += RBO_THREADS) k.colidx[q] = CB_Q + q;
            __syncthreads();
            // phase C: dc = -K^-1 (dK c) (rbs.jl:675)
            k.tri_solve<true>(q1, k.nf);
            __syncthreads();
            k.tri_solve<false>(q1, k.nf);
            // phase D: dots [kx, grad_kx]'.Q (w = 0..d) and Dw'.U (w = d+1..2d) per direction q
            if (tid == 0) { k.set_item(0, CB_RAW, q1, CB_Q, q1, 0); k.set_item(1, CB_SOL + 1, d, CB_U, q1, q1 * q1); }
            __syncthreads();
            const int nD = q1 * q1 + d * q1;
            const int RSd = k.choose_rs(nbq * nbq + nbd * nbq);
            k.colprod(2, nD, smem + k.pl.ppost, RSd);
            __syncthreads();
            // phase E: assemble delta grad alpha per direction and push it into the earlier duals
            if (tid < q1) {
              const int q = tid;
              const double* gh = smem + k.pl.sgh; const double* dmu = smem + k.pl.sdmu; const double* dsg = smem + k.pl.sdsig;
              const double* rowp_v = k.V + (size_t)rowp * RP;
              auto dq = [&](int w) { return split_sum(smem + k.pl.ppost, RSd, nD, w * q1 + q); };
              const double cp = rowp_v[k.CCOL], wp = rowp_v[CB_SOL];
              double dxv[RBO_MAXD];
              for (int a = 0; a < d; ++a) dxv[a] = (q < d) ? (a == q ? 1.0 : 0.0) : (dd_m ? dd_m[(size_t)p * d + a] : 0.0);
              // dkx_p = grad_k(x - X_p).(-dx) (rbf.jl:230-245); dgkx_p = Hk(x - X_p)(-dx) (rbf.jl:247-262)
              double dkx = 0.0, rdx = 0.0;
              for (int a = 0; a < d; ++a) { dkx -= rowp_v[CB_RAW + 1 + a] * dxv[a]; rdx += (xi[a] - xp[a]) * dxv[a]; }
              const double a_ = rowp_v[CB_RAW + d + 1], b_ = rowp_v[CB_RAW + d + 2];
              double dmu_v = dkx * cp - dq(0);                                        // rbs.jl:680 (dc = -Q)
              double dsig_v = (-2.0 * dkx * wp + 2.0 * wp * uw[q]) / (2.0 * sigma);   // rbs.jl:683, w'dK w = 2 w_p (u.w)
              GPart ghat = rule_eval(P.rule_id, P.sigma_tol, dmu_v, dsig_v, P.theta1, misc[2]);  // rbs.jl:687-688 (Q6)
              double push = 0.0;
              for (int a = 0; a < d; ++a) {
                double dgkx = -(a_ * rdx * (xi[a] - xp[a]) + b_ * dxv[a]);
                double dgmu = dgkx * cp - dq(1 + a);                                  // rbs.jl:681
                double val = gh[1] * dgmu + ghat.g_mu * dmu[a] + ghat.g_sig * dsg[a];
                if (q < d) {                                                          // spatial: + g_sigma * delta grad sigma (rbs.jl:684,690)
                  double dwdkw = wp * dq(d + 1 + a) + rowp_v[CB_SOL + 1 + a] * uw[q];
                  double dgsig = (dwdkw - dgkx * wp - rowp_v[CB_SOL + 1 + a] * dkx - dsig_v * dsg[a]) / sigma;
                  val += gh[2] * dgsig;
                }
                push += val * xb[a];
              }
              if (q < d) {
                if (p == 0) gxa[q] += push;               // gather_g: g[i+1]' * xbars[i] (rollout.jl:199-215, 271)
                else accr[(size_t)p * d + q] += push;     // solve_dual_x(p): x_dual -= dri' * xbars[i] (rollout.jl:185)
              } else {
                ybars[p + 1] += push;                     // solve_dual_y(solve_index = p) (rollout.jl:144)
              }
            }
            __syncthreads();
          }
        }
        // g[1] = grad mu(x_0) under the base GP (rollout.jl:194-196), final assembly rollout.jl:267-276
        k.nf = 0;
        {
          const double* x0p = k.Xf;
          auto pt = [&](int) { return x0p; };
          auto cb0 = [&](int) { return 0; };
          __syncthreads();
          k.fill_columns(1, pt, cb0);
          k.set_column(k.CCOL, k.cst);
          if (tid == 0) k.set_item(0, 0, q1, k.CCOL, 1, 0);
          __syncthreads();
          const int RSpre = k.choose_rs(K::nblk16(q1));
          k.colprod(1, q1, smem + k.pl.ppre, RSpre);
          __syncthreads();
          for (int a = tid; a < d; a += RBO_THREADS) P.grad_x[(size_t)m * d + a] = -(split_sum(smem + k.pl.ppre, RSpre, q1, 1 + a) * ybars[1] + gxa[a]);
          for (int a = tid; a < nth; a += RBO_THREADS) P.grad_theta[(size_t)m * nth + a] = (a == 0) ? -gtha[0] : 0.0;
        }
        k.nf = h + 1;
      }
    }
    __syncthreads();
    PT_MARK(11);
    if (tid == 0 && P.status) P.status[m] = si[I_TSTATUS];
  }
  k.pipe_fini();
  if (tid == 0 && P.cta_done) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); P.cta_done[blockIdx.x] = t; }
}

}  // namespace rbo

#ifdef RBO_PHASE_TIMERS
// development aid (not part of include/rbo.h): per-phase cycle counters of the rollout kernel
#if RBO_VGLOB
#define rbo_debug_phase_cycles rbo_debug_phase_cycles_largen
#define rbo_debug_aux_cycles rbo_debug_aux_cycles_largen
#define rbo_debug_tr_cycles rbo_debug_tr_cycles_largen
#endif
extern "C" int rbo_debug_tr_cycles(void*, unsigned long long* out16, int reset) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out16, rbo::g_tr_cycles, sizeof(unsigned long long) * 16);
  if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(rbo::g_tr_cycles, z, sizeof(z)); }
  return 0;
}
extern "C" int rbo_debug_phase_cycles(void*, unsigned long long* out16, int reset) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out16, rbo::g_phase_cycles, sizeof(unsigned long long) * 16);
  if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(rbo::g_phase_cycles, z, sizeof(z)); }
  return 0;
}
extern "C" int rbo_debug_aux_cycles(void*, unsigned long long* out16, int reset) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out16, rbo::g_aux_cycles, sizeof(unsigned long long) * 16);
  if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(rbo::g_aux_cycles, z, sizeof(z)); }
  return 0;
}
#endif
