// rbo_device.cuh -- scalar device helpers shared by the kernels of librbo.so (sm_100a, FP64).
// Each function cites the reference code whose arithmetic it reproduces.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/rbo.h"

#define RBO_MAXD 32      // max input dimension d
#define RBO_THREADS 512  // threads per CTA of the rollout kernel
#define RBO_NWARPS (RBO_THREADS / 32)
#define RBO_NCONS (RBO_NWARPS - 1)  // consumer warps of the panel pipeline; warp RBO_NCONS is the TMA producer
#define RBO_PR 8         // rows per factor panel
#define RBO_MAXFAN 8     // fantasy rows per trajectory (h + 1 <= 8)
#define RBO_BR 32        // rows per packed L0 panel (block row of the blocked triangular solve)
#define RBO_LP 36        // doubles per k in a packed L0 panel: 32 rows + 4 pad (288-byte pitch)
#define RBO_CHUNK_K 32   // k-values per staged panel chunk (32 * 288 B = 9216 B per bulk copy); == RBO_BR
#define RBO_NSTAGE 3     // stages of the panel ring buffer
#define RBO_TR_ROUNDS 3  // rounds of 64-way multisection for the trust-region shift (oracle: TR_ROUNDS, TR_CAND)
#define RBO_FLAG_MYOPIC_INTERNAL (1 << 16)  // kernel-internal: myopic multistart against the base surrogate

namespace rbo {

// DevProblem::work_counter, cleared before every rollout launch; the SGA loop's sticky record keeps the same indices.
enum WorkCounterIndex : int {
  WC_SCHED = 0,                  // next entry of the hand-out order
  WC_STALL = 1, WC_EVAL_CAP = 2,  // flags: a panel pipeline wait never completed; an inner solve exceeded its evaluation bound
  WC_WAIT_KIND = 4, WC_WAIT_CHUNK, WC_WAIT_WARP, WC_WAIT_CONSUMERS, WC_WAIT_BLOCK,  // the stalled wait
  WC_STICKY_SEEN = 0, WC_STICKY_HANDLE = 9,  // sticky record: a flag was seen in some iteration; the index of the flagging handle
  WC_LEN = 16
};

struct KernelSpec {
  int id;
  double th[4];
};

// psi, psi', psi'' of the radial kernels (rbf.jl:60-103; derivatives are what ForwardDiff yields at rbf.jl:41-46,
// written in closed form).
__host__ __device__ inline void kern_eval(const KernelSpec& k, double rho, double& psi, double& dpsi, double& d2psi) {
  switch (k.id) {
    case RBO_KERNEL_MATERN52: {
      double c = sqrt(5.0) / k.th[0], s = c * rho, e = exp(-s);
      psi = (1.0 + s * (1.0 + s / 3.0)) * e;
      dpsi = -(c * c * rho / 3.0) * (1.0 + s) * e;
      d2psi = (c * c / 3.0) * (s * s - s - 1.0) * e;
      break;
    }
    case RBO_KERNEL_MATERN32: {
      double c = sqrt(3.0) / k.th[0], s = c * rho, e = exp(-s);
      psi = (1.0 + s) * e;
      dpsi = -c * c * rho * e;
      d2psi = c * c * (s - 1.0) * e;
      break;
    }
    case RBO_KERNEL_MATERN12: {
      double l = k.th[0], e = exp(-rho / l);
      psi = e;
      dpsi = -e / l;
      d2psi = e / (l * l);
      break;
    }
    case RBO_KERNEL_SE: {
      double l2 = k.th[0] * k.th[0];
      psi = exp(-rho * rho / (2.0 * l2));
      dpsi = -rho / l2 * psi;
      d2psi = (rho * rho / (l2 * l2) - 1.0 / l2) * psi;
      break;
    }
    default: {  // RBO_KERNEL_PERIODIC
      const double pi = 3.141592653589793;
      double l = k.th[0], p = k.th[1], u = pi * rho / p, sn = sin(u);
      psi = exp(-2.0 * sn * sn / (l * l));
      double q = -(2.0 * pi / (p * l * l));
      dpsi = q * sin(2.0 * u) * psi;
      d2psi = q * (cos(2.0 * u) * (2.0 * pi / p) * psi + sin(2.0 * u) * dpsi);
      break;
    }
  }
}

// Derivatives of psi(rho) with respect to the kernel hyper-parameters: dth[0] = d psi / d l (every family), dth[1] = d psi / d p
// (Periodic only). The objective of the maximum-likelihood fit (rbs.jl:770-829) needs them; psi(0) = 1 does not depend on them.
__host__ __device__ inline void kern_dtheta(const KernelSpec& k, double rho, double* dth) {
  dth[1] = 0.0;
  switch (k.id) {
    case RBO_KERNEL_MATERN52: {
      const double l = k.th[0], s = sqrt(5.0) / l * rho;
      dth[0] = s * s * (1.0 + s) / (3.0 * l) * exp(-s);
      break;
    }
    case RBO_KERNEL_MATERN32: {
      const double l = k.th[0], s = sqrt(3.0) / l * rho;
      dth[0] = s * s / l * exp(-s);
      break;
    }
    case RBO_KERNEL_MATERN12: {
      const double l = k.th[0];
      dth[0] = rho / (l * l) * exp(-rho / l);
      break;
    }
    case RBO_KERNEL_SE: {
      const double l = k.th[0], l2 = l * l;
      dth[0] = rho * rho / (l2 * l) * exp(-rho * rho / (2.0 * l2));
      break;
    }
    default: {  // RBO_KERNEL_PERIODIC
      const double pi = 3.141592653589793;
      const double l = k.th[0], p = k.th[1], u = pi * rho / p, sn = sin(u);
      const double psi = exp(-2.0 * sn * sn / (l * l));
      dth[0] = 4.0 * sn * sn / (l * l * l) * psi;
      dth[1] = 2.0 * u * sin(2.0 * u) / (l * l * p) * psi;
      break;
    }
  }
}

// Radial quantities at distance rho: psi, b = psi'/rho, a = (psi'' - psi'/rho)/rho^2, so that
// grad k = b r (rbf.jl:127-134, 0 at rho = 0) and Hk = a r r' + b I (rbf.jl:141-150, psi''(0) I at rho = 0).
__host__ __device__ inline void kern_radial(const KernelSpec& k, double rho2, double& psi, double& a, double& b, double& gb) {
  double rho = sqrt(rho2), dpsi, d2psi;
  kern_eval(k, rho, psi, dpsi, d2psi);
  if (rho > 0.0) {
    b = dpsi / rho;
    a = (d2psi - b) / rho2;
    gb = b;
  } else {
    b = d2psi;  // Hessian coefficient at coincident points
    a = 0.0;
    gb = 0.0;   // gradient coefficient: eval_grad_k returns 0 (rbf.jl:129-131)
  }
}

// Decision-rule value and partials (decision_rules.jl:84-127; partials = closed forms of the nested ForwardDiff
// derivatives of decision_rules.jl:23-34).
struct GPart {
  double g, g_mu, g_sig, g_mumu, g_sigsig, g_muth, g_sigth, g_musig;
};

__host__ __device__ inline GPart rule_eval(int rule, double sigma_tol, double mu, double sigma, double th1, double fstar) {
  GPart r;
  r.g = r.g_mu = r.g_sig = r.g_mumu = r.g_sigsig = r.g_muth = r.g_sigth = r.g_musig = 0.0;
  if (rule == RBO_RULE_LCB) {
    r.g = th1 * sigma - mu;
    r.g_mu = -1.0;
    r.g_sig = th1;
    r.g_sigth = 1.0;
    return r;
  }
  if (sigma < sigma_tol) return r;  // decision_rules.jl:87-89: the constant 0 and therefore zero partials
  const double inv_sqrt2 = 0.70710678118654752440, inv_sqrt2pi = 0.39894228040143267794;
  double imp = fstar - mu - th1, z = imp / sigma;
  double Phi = 0.5 * erfc(-z * inv_sqrt2), phi = exp(-0.5 * z * z) * inv_sqrt2pi;
  if (rule == RBO_RULE_EI) {
    r.g = imp * Phi + sigma * phi;
    r.g_mu = -Phi;
    r.g_sig = phi;
    r.g_mumu = phi / sigma;
    r.g_sigsig = z * z * phi / sigma;
    r.g_muth = phi / sigma;
    r.g_sigth = z * phi / sigma;
    r.g_musig = z * phi / sigma;
  } else {  // POI
    double s2 = sigma * sigma;
    r.g = Phi;
    r.g_mu = -phi / sigma;
    r.g_sig = -z * phi / sigma;
    r.g_mumu = -z * phi / s2;
    r.g_sigsig = (2.0 * z - z * z * z) * phi / s2;
    r.g_muth = r.g_mumu;
    r.g_sigth = (1.0 - z * z) * phi / s2;
    r.g_musig = (1.0 - z * z) * phi / s2;
  }
  return r;
}

// In-place lower Cholesky of an n x n row-major matrix with leading dimension ld. Returns false if not PD.
__device__ inline bool chol_inplace(double* A, int n, int ld) {
  for (int j = 0; j < n; ++j) {
    double s = A[j * ld + j];
    for (int k = 0; k < j; ++k) s -= A[j * ld + k] * A[j * ld + k];
    if (!(s > 0.0) || !isfinite(s)) return false;
    double ljj = sqrt(s);
    A[j * ld + j] = ljj;
    for (int i = j + 1; i < n; ++i) {
      double t = A[i * ld + j];
      for (int k = 0; k < j; ++k) t -= A[i * ld + k] * A[j * ld + k];
      A[i * ld + j] = t / ljj;
    }
  }
  return true;
}

// LU with partial pivoting, row-major n x n (ld = n). det as Julia's det(::Matrix) (rollout.jl:159).
__device__ inline bool lu_factor(double* A, int n, int* piv, double* det) {
  double dt = 1.0;
  bool ok = true;
  for (int k = 0; k < n; ++k) {
    int p = k;
    double mx = fabs(A[k * n + k]);
    for (int i = k + 1; i < n; ++i)
      if (fabs(A[i * n + k]) > mx) { mx = fabs(A[i * n + k]); p = i; }
    piv[k] = p;
    if (p != k) {
      for (int j = 0; j < n; ++j) { double t = A[k * n + j]; A[k * n + j] = A[p * n + j]; A[p * n + j] = t; }
      dt = -dt;
    }
    double akk = A[k * n + k];
    dt *= akk;
    if (akk == 0.0) { ok = false; continue; }
    for (int i = k + 1; i < n; ++i) {
      double lik = A[i * n + k] / akk;
      A[i * n + k] = lik;
      for (int j = k + 1; j < n; ++j) A[i * n + j] -= lik * A[k * n + j];
    }
  }
  *det = dt;
  return ok;
}
__device__ inline void lu_solve(const double* A, int n, const int* piv, double* b) {
  for (int k = 0; k < n; ++k) { double t = b[k]; b[k] = b[piv[k]]; b[piv[k]] = t; }
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < i; ++j) b[i] -= A[i * n + j] * b[j];
  for (int i = n - 1; i >= 0; --i) {
    for (int j = i + 1; j < n; ++j) b[i] -= A[i * n + j] * b[j];
    b[i] /= A[i * n + i];
  }
}

}  // namespace rbo
