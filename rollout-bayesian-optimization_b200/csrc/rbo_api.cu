// rbo_api.cu -- the C ABI of librbo.so (include/rbo.h): handle, device-resident inputs, launches.
// No CPU fallback anywhere: every entry point that computes does so with the sm_100a kernels of rollout_kernel.cu.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "rbo_kernel.cuh"
#include "sga_kernels.cuh"
#include "sobol_dirs.h"

namespace rbo {
__global__ void rbo_rollout_kernel(const __grid_constant__ DevProblem P);
__global__ void rbo_rollout_kernel_largen(const __grid_constant__ DevProblem P);  // same source, work matrix in global memory
__global__ void rbo_normals_kernel(const unsigned* dirs, double* out, int M_total, int d, int H, int m_begin, int m_count);
__global__ void rbo_sobol_kernel(const unsigned* dirs, unsigned* out_u32, double* out_f64, int dim, int npoints, const double* lbs, const double* ubs);
__global__ void rbo_stats_kernel(const double* values, const double* gx, const double* gth, const int* n_evals, const int* best_index, const int* grad_case,
                                 const int* status, int M, int d, int nth, int h, double* sums);
__global__ void rbo_fp64_peak_kernel(double* out, int iters);
__global__ void rbo_tr_step_kernel(const double* H, const double* g, const double* Delta, int n, int B, double* p, int* hit);
__global__ void rbo_gather_sums_kernel(const double* sums, int need, int idx_failed, const int* work_counter, double* out);
__global__ void rbo_lpt_order_kernel(const int* n_evals, const int* grad_case, const int* best_index, int M, int hh, int* order);
// surrogate_kernels.cu
__global__ void rbo_trinv_kernel(const double* L, int N, int N32, double* Linv, int ldi);
__global__ void rbo_pack_fwd_kernel(const double* Linv, int ldi, int nb32, double* Lf);
__global__ void rbo_pack_bwd_kernel(const double* Linv, int ldi, int nb32, double* Lb, double* Lbf);
__global__ void rbo_matvec_lower_kernel(const double* Linv, int ldi, int n, const double* v, double* out);
__global__ void rbo_matvec_lower_t_kernel(const double* Linv, int ldi, int n, const double* v, double scale, double* out);
__global__ void rbo_layout_x_kernel(const double* Xpts, int d, int N, int N8, double* Xb);
__global__ void rbo_kvec_kernel(const double* Xpts, int d, int N, const double* x, KernelSpec kern, double* out);
__global__ void rbo_dots_kernel(const double* l, const double* u, int n, double* scal);
__global__ void rbo_append_row_kernel(double* Linv, int ldi, int n, const double* tmp, const double* scal, double kdiag, double ynew, double* u, int* status);
}  // namespace rbo

using namespace rbo;

static thread_local std::string g_create_error;

// A move-only owned device allocation of `cap` elements of T that only grows: cudaFree / cudaMalloc synchronise the device and
// cost ~0.1 s on a busy context, so a long-lived handle keeps its largest buffers. Converts to T* for kernel arguments and copies.
template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;

  DevBuf() = default;
  DevBuf(DevBuf&& o) noexcept { swap(o); }
  DevBuf& operator=(DevBuf&& o) noexcept {
    swap(o);
    return *this;
  }
  ~DevBuf() { reset(); }
  void swap(DevBuf& o) noexcept {
    std::swap(p, o.p);
    std::swap(cap, o.cap);
  }

  // Holds at least n elements afterwards; the contents do not survive a reallocation. Empty after a failure.
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    reset();
    cudaError_t e = cudaMalloc((void**)&p, n * sizeof(T));
    if (e == cudaSuccess) cap = n;
    else p = nullptr;
    return e;
  }
  void reset() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  operator T*() const { return p; }
};

struct rbo_handle {
  int device = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int num_sms = 0, max_smem = 0;
  std::string err;
  rbo_solver_opts so;
  // surrogate
  bool have_sur = false;
  int d = 0, N = 0, N8 = 0, nb8 = 0, nb32 = 0;
  KernelSpec kern;
  int rule_id = 0;
  double sigma_tol = 1e-8, sigma_n2 = 1e-6, k0 = 1, d2k0 = 0, ymin_base = 0;
  DevBuf<double> Xb, yb, c0, u0, Lf, Lb, Lbf, x0_batch;
  // normals / starts
  int M = 0, hp1 = 0;
  DevBuf<double> rn;
  int S = 0;
  DevBuf<double> starts;
  DevBuf<unsigned> sobol_dirs;
  // outputs, and the shape of the last launch they hold (what the read-back calls and RBO_FLAG_REPLAY_TAPE go by)
  int outM = 0, outh = -1, outS = 0, outd = 0, outnth = 0;
  DevBuf<double> values, grad_x, grad_theta, xs, ys, gys, alphas;
  DevBuf<int> best_index, grad_case, status, n_evals, start_status, start_iters;
  DevBuf<int> work_counter;
  DevBuf<double> sums;
  int sums_len = 0;
  DevBuf<double> dual_dirs, x_forced, cs_tape, gh_nodes, gh_weights;
  int gh_depth = 0, gh_M = 0;
  int last_mode = 0;
  double htol = 1e-4;
  int rs_cap = 0;           // development knob: cap on the row splits of the Gram reductions (0 = default)
  int vglob_wmax = 0;       // development knob: cap on the start slots of the large-n variant (0 = default)
  int force_vglob = 0;      // development / test knob: use the large-n variant even when shared memory would do
  DevBuf<double> Vscratch, Bscratch;
  DevBuf<double> t_mu, t_sigma, t_dmu, t_dsigma, t_Halpha;
  bool tex_valid = false;
  bool xs_valid = false;    // the x-path of the last rollout is on the device (RBO_FLAG_REPLAY_TAPE)
  DevBuf<int> order;        // longest-first order of the trajectories of the last launch (scheduling hint for the next one)
  int order_M = 0;          // 0: no valid order
  int lpt = 1;              // RBO_TUNE_LPT
  DevBuf<unsigned long long> cta_done;  // per-CTA finish time of the last launch (device %globaltimer)
  // resident surrogate in its canonical device form (rbo_set_surrogate / rbo_condition): L0^-1 row-major with pitch ldi,
  // the observation sites point-major, work vectors
  DevBuf<double> Ld, Linv, Xpts, wk;
  DevBuf<int> dstat;
  int ldi = 0, cap_rows = 0;
  // rbo_stochastic_solve_batch: optimiser state, bias corrections and history (doubles); per-restart integers; the work list
  DevBuf<double> sga_dbl;
  DevBuf<int> sga_int, worklist;

  ~rbo_handle() {
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (own_stream) cudaStreamDestroy(own_stream);
  }
};

static int fail(rbo_handle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else g_create_error = buf;
  return code;
}

#define CK(h, call)                                                                                       \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess) return fail(h, RBO_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// D2H of the first n elements of src into dst unless dst is NULL (stream-ordered: the caller synchronises).
template <class T>
static cudaError_t copy_out(T* dst, const DevBuf<T>& src, size_t n, cudaStream_t stream) {
  return dst ? cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToHost, stream) : cudaSuccess;
}

extern "C" {

int rbo_abi_version(void) { return RBO_ABI_VERSION; }

void rbo_default_solver_opts(rbo_solver_opts* o) {
  o->maxit = 100;
  o->maxtry = 30;
  o->gtol = 1e-10;
  o->xtol = 1e-15;
  o->pred_tol = 1e-13;
  o->eta = 0.1;
  o->delta0_box = 0.5;
  o->delta0_ell = 1.0;
  o->stol = 1e-5;
}

const char* rbo_last_error(const rbo_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int rbo_create(rbo_handle** out, int device_id) {
  if (!out) return fail(nullptr, RBO_ERR_ARG, "rbo_create: out is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, RBO_ERR_CUDA, "rbo_create: no CUDA device (%s); librbo has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  if (device_id < 0 || device_id >= ndev) return fail(nullptr, RBO_ERR_ARG, "rbo_create: device %d out of range (have %d)", device_id, ndev);
  auto h = std::make_unique<rbo_handle>();  // released by every failure below
  h->device = device_id;
  rbo_default_solver_opts(&h->so);
  if (const char* e = getenv("RBO_FORCE_LARGE_N")) h->force_vglob = atoi(e) != 0;  // test knob: whole suites under the large-n variant
  CK(nullptr, cudaSetDevice(device_id));
  cudaDeviceProp prop;
  CK(nullptr, cudaGetDeviceProperties(&prop, device_id));
  if (prop.major < 10) return fail(nullptr, RBO_ERR_UNSUPPORTED, "rbo_create: device sm_%d%d is not Blackwell (sm_100a required)", prop.major, prop.minor);
  h->num_sms = prop.multiProcessorCount;
  h->max_smem = (int)prop.sharedMemPerBlockOptin;
  CK(nullptr, cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  h->stream = h->own_stream;
  CK(nullptr, cudaEventCreate(&h->ev0));
  CK(nullptr, cudaEventCreate(&h->ev1));
  CK(nullptr, h->work_counter.reserve(16));  // [0] trajectory scheduler, [1..2] kernel watchdog flags
  CK(nullptr, h->cta_done.reserve(1024));
  CK(nullptr, h->sobol_dirs.reserve(sizeof(rbo_sobol_dirs_host) / sizeof(unsigned)));
  CK(nullptr, cudaMemcpyAsync(h->sobol_dirs, rbo_sobol_dirs_host, sizeof(rbo_sobol_dirs_host), cudaMemcpyHostToDevice, h->stream));
  CK(nullptr, cudaStreamSynchronize(h->stream));
  CK(nullptr, cudaFuncSetAttribute(rbo_rollout_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem));
  CK(nullptr, cudaFuncSetAttribute(rbo_rollout_kernel_largen, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem));
  *out = h.release();
  return RBO_SUCCESS;
}

int rbo_destroy(rbo_handle* h) {
  if (!h) return RBO_SUCCESS;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  delete h;
  return RBO_SUCCESS;
}

int rbo_set_stream(rbo_handle* h, void* cuda_stream) {
  if (!h) return RBO_ERR_ARG;
  h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
  return RBO_SUCCESS;
}

int rbo_set_solver_opts(rbo_handle* h, const rbo_solver_opts* o) {
  if (!h || !o) return RBO_ERR_ARG;
  if (o->maxit < 1 || o->maxtry < 1 || !(o->delta0_box > 0.0) || !(o->delta0_ell > 0.0) || !(o->eta > 0.0 && o->eta < 0.25) || !(o->stol >= 0.0))
    return fail(h, RBO_ERR_ARG, "rbo_set_solver_opts: invalid options");
  h->so = *o;
  return RBO_SUCCESS;
}

int rbo_set_tuning(rbo_handle* h, int key, int value) {
  if (!h) return RBO_ERR_ARG;
  switch (key) {
    case RBO_TUNE_LARGE_N: h->force_vglob = value != 0; return RBO_SUCCESS;
    case RBO_TUNE_LARGE_N_SLOTS: if (value < 0 || value > RBO_NCONS) break; h->vglob_wmax = value; return RBO_SUCCESS;
    case RBO_TUNE_LPT: h->lpt = value != 0; h->order_M = 0; return RBO_SUCCESS;
    case RBO_TUNE_ROW_SPLITS: if (value < 0 || value > 4) break; h->rs_cap = value; return RBO_SUCCESS;
    default: break;
  }
  return fail(h, RBO_ERR_ARG, "rbo_set_tuning: unknown key %d or value %d out of range", key, value);
}

int rbo_set_htol(rbo_handle* h, double htol) {
  if (!h) return RBO_ERR_ARG;
  h->htol = htol;
  return RBO_SUCCESS;
}

// (Re)packs everything the rollout kernel streams from the canonical device form (Linv, Xpts): Xb, Lf, Lb, Lbf. Stream-ordered.
static int repack_surrogate(rbo_handle* h) {
  const int N = h->N, d = h->d, BR = RBO_BR, LP = RBO_LP;
  const int N8 = (N + RBO_PR - 1) / RBO_PR * RBO_PR, nb32 = (N + BR - 1) / BR;
  h->N8 = N8; h->nb8 = N8 / RBO_PR; h->nb32 = nb32;
  const size_t nchunks = (size_t)nb32 * (nb32 + 1) / 2, nLf = (size_t)LP * BR * nchunks, nLbf = (size_t)1024 * nchunks;
  CK(h, h->Xb.reserve((size_t)d * N8));
  CK(h, h->Lf.reserve(nLf));
  CK(h, h->Lb.reserve(nLf));
  CK(h, h->Lbf.reserve(nLbf));
  CK(h, cudaMemsetAsync(h->Lf, 0, nLf * 8, h->stream));  // the 4 pad doubles per k
  CK(h, cudaMemsetAsync(h->Lb, 0, nLf * 8, h->stream));
  rbo_layout_x_kernel<<<(d * N8 + 255) / 256, 256, 0, h->stream>>>(h->Xpts, d, N, N8, h->Xb);
  dim3 grid(8, nb32);
  rbo_pack_fwd_kernel<<<grid, 256, 0, h->stream>>>(h->Linv, h->ldi, nb32, h->Lf);
  rbo_pack_bwd_kernel<<<grid, 256, 0, h->stream>>>(h->Linv, h->ldi, nb32, h->Lb, h->Lbf);
  CK(h, cudaGetLastError());
  return RBO_SUCCESS;
}

// Capacity of the canonical form: rows_needed rows of L0^-1 (pitch = capacity, so that rbo_condition appends rows in place).
// Grows into new buffers (keep: with the current rows copied over) that replace the old ones only once every step succeeded,
// so that a failure leaves the handle as it was.
static int reserve_surrogate(rbo_handle* h, int d, int rows_needed, bool keep) {
  const int N32 = (rows_needed + RBO_BR - 1) / RBO_BR * RBO_BR;
  if (N32 <= h->cap_rows && h->Linv && (size_t)rows_needed * d <= h->Xpts.cap) return RBO_SUCCESS;
  const int cap = (rows_needed + 64 + RBO_BR - 1) / RBO_BR * RBO_BR;
  CK(h, h->dstat.reserve(4));
  DevBuf<double> Linv, Xpts, yb, c0, u0, wk;
  CK(h, Linv.reserve((size_t)cap * cap));
  CK(h, Xpts.reserve((size_t)cap * d));
  // vectors that grow with the observation count
  CK(h, yb.reserve(cap));
  CK(h, c0.reserve(cap));
  CK(h, u0.reserve(cap));
  CK(h, wk.reserve((size_t)4 * cap + 64));
  CK(h, cudaMemsetAsync(Linv, 0, (size_t)cap * cap * 8, h->stream));
  if (keep && h->Linv) {
    const int rows = (h->N + RBO_BR - 1) / RBO_BR * RBO_BR;
    CK(h, cudaMemcpy2DAsync(Linv, (size_t)cap * 8, h->Linv, (size_t)h->ldi * 8, (size_t)rows * 8, rows, cudaMemcpyDeviceToDevice, h->stream));
    CK(h, cudaMemcpyAsync(Xpts, h->Xpts, (size_t)h->N * d * 8, cudaMemcpyDeviceToDevice, h->stream));
  }
  CK(h, cudaMemsetAsync(c0, 0, (size_t)cap * 8, h->stream));
  CK(h, cudaMemsetAsync(u0, 0, (size_t)cap * 8, h->stream));
  CK(h, cudaMemsetAsync(yb, 0, (size_t)cap * 8, h->stream));
  if (keep && h->yb) {
    CK(h, cudaMemcpyAsync(yb, h->yb, (size_t)h->N * 8, cudaMemcpyDeviceToDevice, h->stream));
    CK(h, cudaMemcpyAsync(c0, h->c0, (size_t)h->N * 8, cudaMemcpyDeviceToDevice, h->stream));
    CK(h, cudaMemcpyAsync(u0, h->u0, (size_t)h->N * 8, cudaMemcpyDeviceToDevice, h->stream));
  }
  CK(h, cudaStreamSynchronize(h->stream));  // the old buffers are freed when the locals they are swapped into go out of scope
  h->Linv.swap(Linv);
  h->Xpts.swap(Xpts);
  h->yb.swap(yb);
  h->c0.swap(c0);
  h->u0.swap(u0);
  h->wk.swap(wk);
  h->ldi = cap;
  h->cap_rows = cap;
  return RBO_SUCCESS;
}

int rbo_set_surrogate(rbo_handle* h, int d, int N, const double* X, int ldX, const double* L, int ldL, const double* y, const double* c,
                      double sigma_n2, int kernel_id, const double* ktheta, int nktheta, int rule_id, double sigma_tol) {
  if (!h) return RBO_ERR_ARG;
  if (d < 1 || d > RBO_MAXD) return fail(h, RBO_ERR_UNSUPPORTED, "rbo_set_surrogate: d = %d outside [1, %d]", d, RBO_MAXD);
  if (N < 1 || !X || !L || !y || !c || ldX < d || ldL < N) return fail(h, RBO_ERR_ARG, "rbo_set_surrogate: bad arguments");
  if (kernel_id < RBO_KERNEL_MATERN12 || kernel_id > RBO_KERNEL_PERIODIC) return fail(h, RBO_ERR_ARG, "rbo_set_surrogate: unknown kernel id %d", kernel_id);
  if (rule_id < RBO_RULE_EI || rule_id > RBO_RULE_LCB) return fail(h, RBO_ERR_ARG, "rbo_set_surrogate: unknown decision rule id %d", rule_id);
  if (nktheta < 1 || nktheta > 4 || !ktheta) return fail(h, RBO_ERR_ARG, "rbo_set_surrogate: kernel hyper-parameters missing");
  if ((size_t)N * 16 > 200 * 1024) return fail(h, RBO_ERR_UNSUPPORTED, "rbo_set_surrogate: N = %d observations exceed the inversion kernel's shared-memory column (12800)", N);
  CK(h, cudaSetDevice(h->device));
  if (d != h->d) {
    // buffers laid out for another input dimension are no longer valid (normals are M x (d+1) x hp1, starts d x S, ...)
    h->M = 0; h->hp1 = 0; h->S = 0; h->gh_M = 0; h->gh_depth = 0;
    h->rn.reset();
    h->starts.reset();
    h->gh_nodes.reset();
    h->gh_weights.reset();
    h->cap_rows = 0;  // Xpts is sized with d
  }
  h->have_sur = false;
  int rc = reserve_surrogate(h, d, N, false);
  if (rc) return rc;
  h->d = d; h->N = N;
  h->kern.id = kernel_id;
  for (int i = 0; i < 4; ++i) h->kern.th[i] = i < nktheta ? ktheta[i] : 0.0;
  h->rule_id = rule_id; h->sigma_tol = sigma_tol; h->sigma_n2 = sigma_n2;
  double a, b;
  kern_eval(h->kern, 0.0, h->k0, a, b);
  h->d2k0 = b;
  double ymin = y[0];
  for (int j = 0; j < N; ++j) ymin = std::min(ymin, y[j]);
  h->ymin_base = ymin;
  const int N32 = (N + RBO_BR - 1) / RBO_BR * RBO_BR;
  // H2D of what FantasySurrogate(s, h) copies (rbs.jl:345-381): X (d x N), the lower factor, y, c
  CK(h, h->Ld.reserve((size_t)N * N));
  CK(h, cudaMemcpy2DAsync(h->Xpts, (size_t)d * 8, X, (size_t)ldX * 8, (size_t)d * 8, N, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemcpy2DAsync(h->Ld, (size_t)N * 8, L, (size_t)ldL * 8, (size_t)N * 8, N, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemsetAsync(h->c0, 0, h->c0.cap * 8, h->stream));
  CK(h, cudaMemsetAsync(h->u0, 0, h->u0.cap * 8, h->stream));
  CK(h, cudaMemcpyAsync(h->yb, y, (size_t)N * 8, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemcpyAsync(h->c0, c, (size_t)N * 8, cudaMemcpyHostToDevice, h->stream));
  // Explicit inverse of the base factor on the device in double-double arithmetic (one rounding per stored entry): every later
  // "triangular solve" against L0 is then a dependency-free panel product on the FP64 tensor cores.
  CK(h, cudaMemsetAsync(h->Linv, 0, (size_t)N32 * h->ldi * 8, h->stream));
  {
    const int wpc = std::max(1, std::min(4, (int)((200 * 1024) / ((size_t)N * 16))));
    const size_t smem = (size_t)wpc * 2 * N * 8;
    CK(h, cudaFuncSetAttribute(rbo_trinv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 48 * 1024)));
    rbo_trinv_kernel<<<(N32 + wpc - 1) / wpc, 32 * wpc, smem, h->stream>>>(h->Ld, N, N32, h->Linv, h->ldi);
    CK(h, cudaGetLastError());
  }
  // u0 = L^-1 y (kept so that the coefficient re-solve of rbs.jl:422-429 only needs the backward half)
  rbo_matvec_lower_kernel<<<(N + 7) / 8, 256, 0, h->stream>>>(h->Linv, h->ldi, N, h->yb, h->u0);
  CK(h, cudaGetLastError());
  rc = repack_surrogate(h);
  if (rc) return rc;
  CK(h, cudaStreamSynchronize(h->stream));  // the caller's buffers may change after return
  h->have_sur = true;
  return RBO_SUCCESS;
}

int rbo_condition(rbo_handle* h, const double* x, double y) {
  if (!h || !x) return RBO_ERR_ARG;
  if (!h->have_sur) return fail(h, RBO_ERR_STATE, "rbo_condition: no surrogate (rbo_set_surrogate)");
  CK(h, cudaSetDevice(h->device));
  const int n = h->N, d = h->d;
  if ((size_t)(n + 1) * 16 > 200 * 1024) return fail(h, RBO_ERR_UNSUPPORTED, "rbo_condition: too many observations");
  int rc = reserve_surrogate(h, d, n + 1, true);
  if (rc) return rc;
  double* kv = h->wk; double* lv = kv + h->cap_rows; double* tmp = lv + h->cap_rows; double* scal = tmp + h->cap_rows; double* xd = scal + 8;
  CK(h, cudaMemcpyAsync(xd, x, (size_t)d * 8, cudaMemcpyHostToDevice, h->stream));
  if (n % RBO_BR == 0) {
    // the factor grows by a panel: its padding rows are the identity
    std::vector<double> one(1, 1.0);
    CK(h, cudaMemsetAsync(h->Linv + (size_t)n * h->ldi, 0, (size_t)RBO_BR * h->ldi * 8, h->stream));
    for (int r = n + 1; r < n + RBO_BR; ++r) CK(h, cudaMemcpyAsync(h->Linv + (size_t)r * h->ldi + r, one.data(), 8, cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
  }
  // update_covariance! (rbs.jl:166-183): k = psi(|x - X_j|); update_cholesky! (rbs.jl:185-203): l = L^-1 k, l_nn = sqrt(k0 + sigma_n2 - l.l)
  rbo_kvec_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(h->Xpts, d, n, xd, h->kern, kv);
  rbo_matvec_lower_kernel<<<(n + 7) / 8, 256, 0, h->stream>>>(h->Linv, h->ldi, n, kv, lv);
  rbo_dots_kernel<<<1, 32, 0, h->stream>>>(lv, h->u0, n, scal);
  rbo_matvec_lower_t_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(h->Linv, h->ldi, n, lv, 1.0, tmp);
  rbo_append_row_kernel<<<(n + 256) / 256, 256, 0, h->stream>>>(h->Linv, h->ldi, n, tmp, scal, h->k0 + h->sigma_n2, y, h->u0, h->dstat);
  CK(h, cudaGetLastError());
  int st = 0;
  CK(h, cudaMemcpyAsync(&st, h->dstat, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  if (st != 0) return fail(h, RBO_ERR_NUMERIC, "rbo_condition: PosDefException -- the extended kernel matrix is not positive definite (rbs.jl:196)");
  CK(h, cudaMemcpyAsync(h->Xpts + (size_t)n * d, xd, (size_t)d * 8, cudaMemcpyDeviceToDevice, h->stream));
  CK(h, cudaMemcpyAsync(h->yb + n, &y, 8, cudaMemcpyHostToDevice, h->stream));
  h->N = n + 1;
  h->ymin_base = std::min(h->ymin_base, y);
  // update_coefficients! (rbs.jl:205-212): c = L^-T (L^-1 y), a full re-solve in the reference as well
  rbo_matvec_lower_t_kernel<<<(n + 1 + 127) / 128, 128, 0, h->stream>>>(h->Linv, h->ldi, n + 1, h->u0, 1.0, h->c0);
  CK(h, cudaGetLastError());
  rc = repack_surrogate(h);
  if (rc) return rc;
  CK(h, cudaStreamSynchronize(h->stream));
  return RBO_SUCCESS;
}

int rbo_get_surrogate(rbo_handle* h, int* N_out, double* X, int ldX, double* y, double* c) {
  if (!h) return RBO_ERR_ARG;
  if (!h->have_sur) return fail(h, RBO_ERR_STATE, "rbo_get_surrogate: no surrogate");
  CK(h, cudaSetDevice(h->device));
  if (N_out) *N_out = h->N;
  if (X) { if (ldX < h->d) return fail(h, RBO_ERR_ARG, "rbo_get_surrogate: ldX < d"); CK(h, cudaMemcpy2DAsync(X, (size_t)ldX * 8, h->Xpts, (size_t)h->d * 8, (size_t)h->d * 8, h->N, cudaMemcpyDeviceToHost, h->stream)); }
  if (y) CK(h, cudaMemcpyAsync(y, h->yb, (size_t)h->N * 8, cudaMemcpyDeviceToHost, h->stream));
  if (c) CK(h, cudaMemcpyAsync(c, h->c0, (size_t)h->N * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return RBO_SUCCESS;
}

int rbo_set_normals(rbo_handle* h, const double* rn, int M_total, int hp1, int m_begin, int m_count) {
  if (!h) return RBO_ERR_ARG;
  if (!h->have_sur) return fail(h, RBO_ERR_STATE, "rbo_set_normals: call rbo_set_surrogate first");
  if (!rn || M_total < 1 || hp1 < 1 || m_begin < 0 || m_count < 1 || m_begin + m_count > M_total) return fail(h, RBO_ERR_ARG, "rbo_set_normals: bad arguments");
  CK(h, cudaSetDevice(h->device));
  const int q1 = h->d + 1;
  CK(h, h->rn.reserve((size_t)m_count * q1 * hp1));
  // strided slice [m_begin, m_begin+m_count) of the sample-fastest tensor
  CK(h, cudaMemcpy2DAsync(h->rn, (size_t)m_count * 8, rn + m_begin, (size_t)M_total * 8, (size_t)m_count * 8, (size_t)q1 * hp1, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  h->M = m_count; h->hp1 = hp1; h->order_M = 0;
  return RBO_SUCCESS;
}

int rbo_generate_normals(rbo_handle* h, int M_total, int hp1, int m_begin, int m_count) {
  if (!h) return RBO_ERR_ARG;
  if (!h->have_sur) return fail(h, RBO_ERR_STATE, "rbo_generate_normals: call rbo_set_surrogate first");
  if (M_total < 1 || hp1 < 1 || m_begin < 0 || m_count < 1 || m_begin + m_count > M_total) return fail(h, RBO_ERR_ARG, "rbo_generate_normals: bad arguments");
  const int q1 = h->d + 1, D = q1 + (q1 & 1);
  if (D > RBO_SOBOL_MAXDIM) return fail(h, RBO_ERR_UNSUPPORTED, "rbo_generate_normals: %d Sobol dimensions > %d", D, RBO_SOBOL_MAXDIM);
  if ((double)M_total * hp1 >= 4294967295.0) return fail(h, RBO_ERR_UNSUPPORTED, "rbo_generate_normals: more than 2^32 Sobol points");
  CK(h, cudaSetDevice(h->device));
  CK(h, h->rn.reserve((size_t)m_count * q1 * hp1));
  size_t total = (size_t)m_count * q1 * hp1;
  int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)h->num_sms * 8);
  rbo_normals_kernel<<<blocks, 256, 0, h->stream>>>(h->sobol_dirs, h->rn, M_total, h->d, hp1, m_begin, m_count);
  CK(h, cudaGetLastError());
  h->M = m_count; h->hp1 = hp1; h->order_M = 0;
  return RBO_SUCCESS;
}

int rbo_get_normals(rbo_handle* h, double* out) {
  if (!h || !out) return RBO_ERR_ARG;
  if (!h->rn) return fail(h, RBO_ERR_STATE, "rbo_get_normals: no normals resident");
  CK(h, cudaSetDevice(h->device));
  CK(h, cudaMemcpyAsync(out, h->rn, (size_t)h->M * (h->d + 1) * h->hp1 * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return RBO_SUCCESS;
}

int rbo_set_quadrature(rbo_handle* h, const double* nodes, const double* weights, int depth, int m_count) {
  if (!h) return RBO_ERR_ARG;
  if (!nodes || !weights || depth < 1 || m_count < 1) return fail(h, RBO_ERR_ARG, "rbo_set_quadrature: bad arguments");
  CK(h, cudaSetDevice(h->device));
  const size_t n = (size_t)depth * m_count;
  CK(h, h->gh_nodes.reserve(n));
  CK(h, h->gh_weights.reserve(n));
  CK(h, cudaMemcpyAsync(h->gh_nodes, nodes, n * 8, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemcpyAsync(h->gh_weights, weights, n * 8, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  h->gh_depth = depth; h->gh_M = m_count;
  return RBO_SUCCESS;
}

int rbo_set_starts(rbo_handle* h, const double* starts, int S) {
  if (!h) return RBO_ERR_ARG;
  if (!h->have_sur) return fail(h, RBO_ERR_STATE, "rbo_set_starts: call rbo_set_surrogate first");
  if (!starts || S < 1) return fail(h, RBO_ERR_ARG, "rbo_set_starts: bad arguments");
  if (S > 65535) return fail(h, RBO_ERR_UNSUPPORTED, "rbo_set_starts: %d starts (the kernel keeps per-start counters and the hand-out order as 16-bit values: at most 65535)", S);
  CK(h, cudaSetDevice(h->device));
  CK(h, h->starts.reserve((size_t)S * h->d));
  CK(h, cudaMemcpyAsync(h->starts, starts, (size_t)S * h->d * 8, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  h->S = S;
  return RBO_SUCCESS;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// Makes the output buffers hold a launch of M trajectories (horizon hor, S starts) and records that shape.
static int ensure_outputs(rbo_handle* h, int M, int hor, int S, int d, int nth) {
  if (h->outM == M && h->outh == hor && h->outS == S && h->outd == d && h->outnth == nth) return RBO_SUCCESS;
  const int hh = std::max(hor, 1);
  h->outM = 0; h->outh = -1; h->xs_valid = false;  // the record is only valid once every buffer below holds its shape
  CK(h, h->values.reserve((size_t)M));
  CK(h, h->grad_x.reserve((size_t)M * d));
  CK(h, h->grad_theta.reserve((size_t)M * nth));
  CK(h, h->best_index.reserve((size_t)M));
  CK(h, h->grad_case.reserve((size_t)M));
  CK(h, h->status.reserve((size_t)M));
  CK(h, h->xs.reserve((size_t)M * (hor + 1) * d));
  CK(h, h->ys.reserve((size_t)M * (hor + 1)));
  CK(h, h->gys.reserve((size_t)M * (hor + 1) * d));
  CK(h, h->alphas.reserve((size_t)M * hh));
  CK(h, h->n_evals.reserve((size_t)M * hh));
  CK(h, h->start_status.reserve((size_t)M * hh * S));
  CK(h, h->start_iters.reserve((size_t)M * hh * S));
  h->sums_len = 1 + 3 * (1 + d + nth) + hh + (hor + 2) + 2;
  CK(h, h->sums.reserve((size_t)h->sums_len + 1 + 3 * (1 + d + nth) + 2));  // + the gathered partial-sums vector (rbo_partial_sums_host)
  h->outM = M; h->outh = hor; h->outS = S; h->outd = d; h->outnth = nth;
  return RBO_SUCCESS;
}

// Chooses the number of start slots W (starts evaluated in lock-step) so that the shared-memory plan fits.
struct PlanChoice { int W, RP, NR, RSmax, NPmax, xsm; size_t bytes; int RSh; int vglob; };
static bool choose_plan(const rbo_handle* h, int hor, int S, int mode, PlanChoice* pc) {
  const int d = h->d, N8 = h->N8, CS = d + 3, NR = std::max(N8 + RBO_MAXFAN, h->nb32 * RBO_BR);
  const int nadj = (mode == RBO_MODE_VALUE_GRAD) ? ncols_adjoint(d) : 0;  // the adjoint's column plan is only needed with gradients
  // Preference: (i) row splits >= 2 and the base locations in shared memory, with the largest W that still allows it
  // (provided that W covers at least half of the start list); (ii) otherwise the largest W with whatever fits.
  auto try_plan = [&](int W, int RSmax, int xsm, int vglob = 0) {
    int RP = std::max(W * CS, nadj) + 2;
    if ((RP & 1) == 0) RP += 1;  // odd pitch: conflict-free column walks
    int NPmax = npairs_max(d, W);
    SmemPlan pl = make_plan(d, N8, hor, W, RP, NR, RSmax, NPmax, xsm, RSmax, vglob, S);
    size_t bytes = (size_t)pl.total * 8;
    if (bytes > (size_t)h->max_smem) return false;
    *pc = {W, RP, NR, RSmax, NPmax, xsm, bytes, RSmax, vglob};
    // the Hessian sums are tensor-pipe bound per scheduler: give them enough row splits to occupy every warp if that still fits
    const int want = std::min(4, std::max(RSmax, RBO_NWARPS / W));
    for (int rsh = want; rsh > RSmax; --rsh) {
      SmemPlan p2 = make_plan(d, N8, hor, W, RP, NR, RSmax, NPmax, xsm, rsh, vglob, S);
      if ((size_t)p2.total * 8 <= (size_t)h->max_smem) { pc->RSh = rsh; pc->bytes = (size_t)p2.total * 8; break; }
    }
    return true;
  };
  const int Wmax = std::min(S, RBO_NCONS);
  for (int W = Wmax; !h->force_vglob && W >= std::max(1, std::min(Wmax, (S + 1) / 2)); --W) {
    int rs = std::min(h->rs_cap > 0 ? h->rs_cap : 4, std::min(4, std::max(2, RBO_NWARPS / W)));
    if (try_plan(W, rs, 1)) return true;
    if (rs > 2 && try_plan(W, 2, 1)) return true;
  }
  for (int W = Wmax; !h->force_vglob && W >= 1; --W) {
    const int tries[4][2] = {{2, 1}, {1, 1}, {2, 0}, {1, 0}};
    for (auto& t : tries) if (try_plan(W, t[0], t[1])) return true;
  }
  // Large-n variant (north_star: "L0 ... read through L2 when n is large"; BASELINE config C5): the work matrix moves to a
  // per-CTA scratch in global memory (it stays L2-resident), everything else keeps its place in shared memory. The base
  // locations are then read through L1 as well. More start slots per round amortise the stream of L0^-1 over more columns.
  // measured at the C5 shape (n = 1000, d = 20): 4-5 slots are best; more slots enlarge the scratch (148 CTAs x NR x RP doubles)
  // beyond what stays L2-resident and leave fewer row splits for the reductions
  const int Wg = std::min(Wmax, h->vglob_wmax > 0 ? h->vglob_wmax : 5);
  for (int W = Wg; W >= 1; --W)
    for (int rs = std::min(4, std::max(2, RBO_NWARPS / W)); rs >= 1; --rs)
      if (try_plan(W, rs, 0, 1)) return true;
  return false;
}

static double f_eval(double n, double d) { return 2 * n * n * (d + 1) + n * (4 * d * d + 11 * d + 31); }
static double f_step(double n, double d) { return 2 * n * n * (d + 1) + 2 * n * (d + 1) * (d + 1) + 3 * n * n + (d + 1) * (d + 1) * (d + 1) / 3.0; }
// what this implementation executes per evaluation: (d+1) forward + 1 backward substitutions, Gram + two Hessian sums
static double f_eval_exec(double n, double d) { return n * n * (d + 2) + n * (3 * d * (d + 1) + 4 * d + 40); }

// Validates a launch, chooses its plan, makes the output and scratch buffers hold it and fills the rollout kernel's parameter block
// P (P.order: the longest-first order of the previous launch when it applies) and its grid. Enqueues no kernel.
static int prepare_launch(rbo_handle* h, const double* x0, const double* theta, int ntheta, const double* lbs, const double* ubs, int horizon,
                          double fmini, int mode, int flags, const double* dual_dirs_dev, const double* x_forced_dev,
                          const double* x0_batch_dev, int B, DevProblem& P, PlanChoice& pc, int& grid) {
  const bool myopic = (flags & RBO_FLAG_MYOPIC_INTERNAL) != 0, ghq = (flags & RBO_FLAG_GAUSS_HERMITE) != 0;
  if (!h->have_sur) return fail(h, RBO_ERR_STATE, "rbo_rollout: no surrogate (rbo_set_surrogate)");
  if (ghq && !h->gh_nodes) return fail(h, RBO_ERR_STATE, "rbo_rollout: no quadrature data (rbo_set_quadrature)");
  if (!h->rn && !myopic && !ghq) return fail(h, RBO_ERR_STATE, "rbo_rollout: no normals (rbo_set_normals / rbo_generate_normals)");
  if (!h->starts && !(flags & RBO_FLAG_TEACHER_FORCED)) return fail(h, RBO_ERR_STATE, "rbo_rollout: no starts (rbo_set_starts)");
  if (!x0 || !theta || !lbs || !ubs || ntheta < 1) return fail(h, RBO_ERR_ARG, "rbo_rollout: bad arguments");
  if (horizon < 0 || horizon + 1 > RBO_MAXFAN) return fail(h, RBO_ERR_UNSUPPORTED, "rbo_rollout: horizon %d not in [0, %d]", horizon, RBO_MAXFAN - 1);
  if (!myopic && !ghq && horizon + 1 > h->hp1) return fail(h, RBO_ERR_ARG, "rbo_rollout: normals hold %d steps, horizon + 1 = %d needed", h->hp1, horizon + 1);
  if (ghq && horizon + 1 > h->gh_depth) return fail(h, RBO_ERR_ARG, "rbo_rollout: quadrature depth %d < horizon + 1 = %d", h->gh_depth, horizon + 1);
  const int Ms = myopic ? 1 : (ghq ? h->gh_M : h->M);  // sample indices
  const int M = Ms * std::max(B, 1);                    // trajectories of this launch
  if (flags & RBO_FLAG_REPLAY_TAPE) {
    // second phase of the two-phase call: replay the x-path of the previous rollout of this handle (still on the device)
    if (myopic || h->outh != horizon || h->outM != M || !h->xs_valid) return fail(h, RBO_ERR_STATE, "rbo_rollout: RBO_FLAG_REPLAY_TAPE needs a preceding rollout with the same samples and horizon on this handle");
    flags |= RBO_FLAG_TEACHER_FORCED;
  } else if ((flags & RBO_FLAG_TEACHER_FORCED) && !x_forced_dev) return fail(h, RBO_ERR_ARG, "rbo_rollout: teacher forcing without x_forced");
  if (mode != RBO_MODE_VALUE && mode != RBO_MODE_VALUE_GRAD) return fail(h, RBO_ERR_ARG, "rbo_rollout: bad mode");
  for (int a = 0; a < h->d; ++a)
    if (!(lbs[a] <= ubs[a])) return fail(h, RBO_ERR_ARG, "rbo_rollout: lower bound above upper bound in dimension %d", a);
  CK(h, cudaSetDevice(h->device));
  const int S = std::max(h->S, 1);
  if (!choose_plan(h, horizon, S, mode, &pc))
    return fail(h, RBO_ERR_UNSUPPORTED, "rbo_rollout: problem (d=%d, N=%d, h=%d) needs more than %d bytes of shared memory per CTA", h->d, h->N, horizon, h->max_smem);
  if (getenv("RBO_DEBUG")) fprintf(stderr, "[rbo] plan: W=%d RP=%d NR=%d RSmax=%d NPmax=%d xsm=%d smem=%zu B (limit %d)\n", pc.W, pc.RP, pc.NR, pc.RSmax, pc.NPmax, pc.xsm, pc.bytes, h->max_smem);
  if (getenv("RBO_DEBUG")) fprintf(stderr, "[rbo] plan: RSh=%d vglob=%d\n", pc.RSh, pc.vglob);
  int rc = ensure_outputs(h, M, horizon, S, h->d, ntheta);
  if (rc) return rc;
  memset(&P, 0, sizeof(P));
  P.d = h->d; P.N = h->N; P.N8 = h->N8; P.nb8 = h->nb8; P.nb32 = h->nb32; P.h = horizon; P.S = S; P.W = pc.W; P.RSmax = pc.RSmax; P.NPmax = pc.NPmax; P.xsm = pc.xsm; P.XP = h->N8 + 1;
  P.RSh = pc.RSh;
  P.pl = make_plan(P.d, P.N8, horizon, pc.W, pc.RP, pc.NR, pc.RSmax, pc.NPmax, pc.xsm, pc.RSh, pc.vglob, S);
  P.vglob = pc.vglob;
  P.CS = h->d + 3; P.RP = pc.RP; P.NR = pc.NR; P.M = M; P.Ms = Ms; P.B = std::max(B, 1); P.x0_batch = (B > 1 || x0_batch_dev) ? x0_batch_dev : nullptr; P.hp1 = h->hp1; P.mode = mode; P.flags = flags; P.ntheta = ntheta;
  P.kern = h->kern; P.rule_id = h->rule_id; P.sigma_tol = h->sigma_tol; P.sigma_n2 = h->sigma_n2; P.k0 = h->k0; P.d2k0 = h->d2k0;
  P.ymin_base = h->ymin_base; P.m52_c = std::sqrt(5.0) / h->kern.th[0]; P.fmini = fmini; P.theta1 = theta[0]; P.htol = h->htol; P.so = h->so;
  for (int a = 0; a < h->d; ++a) { P.x0[a] = x0[a]; P.lbs[a] = lbs[a]; P.ubs[a] = ubs[a]; }
  P.Xb = h->Xb; P.yb = h->yb; P.c0 = h->c0; P.u0 = h->u0; P.Lf = h->Lf; P.Lb = h->Lb; P.Lbf = h->Lbf; P.rn = h->rn; P.starts = h->starts;
  P.dual_dirs = dual_dirs_dev; P.x_forced = x_forced_dev;
  P.gh_nodes = h->gh_nodes; P.gh_weights = h->gh_weights; P.gh_depth = h->gh_depth;
  P.values = h->values; P.grad_x = h->grad_x; P.grad_theta = h->grad_theta; P.best_index = h->best_index; P.grad_case = h->grad_case;
  P.status = h->status; P.xs = h->xs; P.ys = h->ys; P.gys = h->gys; P.alphas = h->alphas; P.n_evals = h->n_evals;
  P.start_status = h->start_status; P.start_iters = h->start_iters;
  P.work_counter = h->work_counter;
  h->tex_valid = false;
  if (flags & RBO_FLAG_TAPE_EX) {
    if (myopic) return fail(h, RBO_ERR_ARG, "rbo_rollout: RBO_FLAG_TAPE_EX does not apply to the myopic solve");
    const size_t n = (size_t)M * std::max(horizon, 1), d = h->d;
    CK(h, h->t_mu.reserve(n));
    CK(h, h->t_sigma.reserve(n));
    CK(h, h->t_dmu.reserve(n * d));
    CK(h, h->t_dsigma.reserve(n * d));
    CK(h, h->t_Halpha.reserve(n * d * d));
    P.t_mu = h->t_mu; P.t_sigma = h->t_sigma; P.t_dmu = h->t_dmu; P.t_dsigma = h->t_dsigma; P.t_Halpha = h->t_Halpha;
    h->tex_valid = true;
  }
  grid = std::min(M, h->num_sms);
  // longest-first hand-out when the previous launch ran the same trajectories (same normals, nearby x0): only worth it beyond two waves
  P.order = (h->lpt && !myopic && h->order_M == M && M > 2 * grid && !(flags & RBO_FLAG_TEACHER_FORCED)) ? h->order.p : nullptr;
  P.cta_done = grid <= 1024 ? h->cta_done.p : nullptr;
  CK(h, h->cs_tape.reserve((size_t)grid * (horizon + 2) * pc.NR));
  P.cs_tape = h->cs_tape;
  if (pc.vglob) {
    CK(h, h->Vscratch.reserve((size_t)grid * pc.NR * pc.RP));
    P.Vscratch = h->Vscratch;
    P.bscratch_len = (size_t)h->N8 * 8 * ((std::max(h->d + 1, pc.W) + 7) / 8);  // widest backward pass: q1 columns (adjoint) or W (inner solve)
    CK(h, h->Bscratch.reserve((size_t)grid * P.bscratch_len));
    P.Bscratch = h->Bscratch;
  }
  return RBO_SUCCESS;
}

// The rollout kernel of a prepared problem (the caller has cleared work_counter: the scheduler counter and the watchdog flags).
static cudaError_t enqueue_rollout(const rbo_handle* h, const DevProblem& P, const PlanChoice& pc, int grid) {
  if (pc.vglob) rbo_rollout_kernel_largen<<<grid, RBO_THREADS, pc.bytes, h->stream>>>(P);
  else rbo_rollout_kernel<<<grid, RBO_THREADS, pc.bytes, h->stream>>>(P);
  return cudaGetLastError();
}

// wd: the work_counter entries the rollout kernel's watchdog writes ([1], [2] flags; [4..8] where it waited)
static int watchdog_fail(rbo_handle* h, const int* wd) {
  return fail(h, RBO_ERR_CUDA, "rollout kernel watchdog: %s%s (wait kind %d, chunk %d, warp %d, consumers %d, block %d)", wd[1] ? "[panel pipeline wait never completed] " : "",
              wd[2] ? "[inner solve exceeded its evaluation bound]" : "", wd[4], wd[5], wd[6], wd[7], wd[8]);
}

static int launch_rollout(rbo_handle* h, const double* x0, const double* theta, int ntheta, const double* lbs, const double* ubs, int horizon,
                          double fmini, int mode, int flags, const double* dual_dirs_dev, const double* x_forced_dev, bool want_summary,
                          rbo_summary* summary, const double* x0_batch_dev = nullptr, int B = 1) {
  DevProblem P;
  PlanChoice pc;
  int grid = 0;
  int rc = prepare_launch(h, x0, theta, ntheta, lbs, ubs, horizon, fmini, mode, flags, dual_dirs_dev, x_forced_dev, x0_batch_dev, B, P, pc, grid);
  if (rc) return rc;
  flags = P.flags;
  const bool myopic = (flags & RBO_FLAG_MYOPIC_INTERNAL) != 0;
  const int M = P.M;
  CK(h, cudaMemsetAsync(h->work_counter, 0, 16 * sizeof(int), h->stream));
  CK(h, cudaEventRecord(h->ev0, h->stream));
  CK(h, enqueue_rollout(h, P, pc, grid));
  rbo_stats_kernel<<<1, 1024, 0, h->stream>>>(h->values, mode == RBO_MODE_VALUE_GRAD ? h->grad_x.p : nullptr, mode == RBO_MODE_VALUE_GRAD ? h->grad_theta.p : nullptr,
                                              h->n_evals, h->best_index, h->grad_case, h->status, M, h->d, ntheta, horizon, h->sums);
  CK(h, cudaGetLastError());
  CK(h, cudaEventRecord(h->ev1, h->stream));
  if (h->lpt && !myopic && horizon > 0 && M > 2 * grid && !(flags & RBO_FLAG_TEACHER_FORCED)) {
    CK(h, h->order.reserve(M));
    rbo_lpt_order_kernel<<<1, 1024, 0, h->stream>>>(h->n_evals, h->grad_case, h->best_index, M, std::max(horizon, 1), h->order);
    CK(h, cudaGetLastError());
    h->order_M = M;
  } else if (!(flags & RBO_FLAG_TEACHER_FORCED)) h->order_M = 0;
  h->last_mode = mode;
  h->xs_valid = !myopic;
  if (want_summary && summary) {
    std::vector<double> sums(h->sums_len);
    int wd[16] = {0};
    std::vector<unsigned long long> td(grid);
    CK(h, cudaMemcpyAsync(sums.data(), h->sums, (size_t)h->sums_len * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaMemcpyAsync(wd, h->work_counter, sizeof(wd), cudaMemcpyDeviceToHost, h->stream));
    if (P.cta_done) CK(h, cudaMemcpyAsync(td.data(), h->cta_done, (size_t)grid * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    if (wd[1] || wd[2]) return watchdog_fail(h, wd);
    float ms = 0;
    CK(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    const int d = h->d, hh = std::max(horizon, 1), nrows = 1 + d + ntheta;
    const double n = sums[0];
    summary->n_traj = M;
    summary->mean = n > 0 ? sums[1] / n : NAN;
    summary->std = n > 1 ? std::sqrt(sums[2] / (n - 1)) : NAN;
    summary->kernel_ms = ms;
    summary->gpu_launches = 2 + (h->order_M == M ? 1 : 0);
    summary->tail_ms = 0.0;
    if (P.cta_done) {
      std::sort(td.begin(), td.end());
      summary->tail_ms = (double)(td.back() - td[grid / 2]) * 1e-6;  // last CTA to finish minus the median CTA
    }
    const double* ev = sums.data() + 1 + 3 * nrows;
    const double* hist = ev + hh;
    summary->n_failed = (int)hist[horizon + 2];
    double fl = 0, fx = 0;
    long long ne = 0;
    if (myopic) {
      ne = (long long)ev[0];
      fl = ev[0] * f_eval(h->N, d);
      fx = ev[0] * f_eval_exec(h->N, d);
    } else {
      fl = M * f_step(h->N, d); fx = M * f_step(h->N, d) * 0.5;
      for (int j = 1; j <= horizon; ++j) {
        double nj = h->N + j, e = ev[j - 1];
        ne += (long long)e;
        fl += e * f_eval(nj, d) + M * f_step(nj, d);
        fx += e * f_eval_exec(nj, d) + M * f_step(nj, d) * 0.5;
      }
    }
    if (mode == RBO_MODE_VALUE_GRAD)
      for (int t = 1; t <= horizon; ++t) {  // F_adj(t) for the hist[t] trajectories whose best step is t (case 3)
        double fa = t * (2.0 / 3.0) * d * d * d;
        for (int i = 1; i <= t; ++i) { double ni = h->N + i; fa += f_eval(ni, d) + i * (d + 1) * (2 * ni * ni + 6 * ni * d); }
        fl += hist[t] * fa;
        fx += hist[t] * fa;
      }
    summary->flops = fl;
    summary->flops_executed = fx;
    summary->n_evals = ne;
  }
  return RBO_SUCCESS;
}

// rbo_rollout and rbo_rollout_batch: the launch on host inputs -- the dual directions (VALUE_GRAD), the forced x-path and, for a
// batch, the B starting points x0_batch (d x B) are uploaded first -- and the per-trajectory results back to the host.
static int rollout_host(rbo_handle* h, const double* x0, const double* x0_batch, int B, const double* theta, int ntheta, const double* lbs,
                        const double* ubs, int horizon, double fmini, int mode, int flags, const double* dual_dirs, const double* x_forced,
                        double* values, double* grad_x, double* grad_theta, int32_t* best_index, int32_t* grad_case, int32_t* status,
                        rbo_summary* summary) {
  const bool grad = mode == RBO_MODE_VALUE_GRAD;
  const bool forced = (flags & RBO_FLAG_TEACHER_FORCED) && !(flags & RBO_FLAG_REPLAY_TAPE);
  CK(h, cudaSetDevice(h->device));
  const size_t Ms = (flags & RBO_FLAG_GAUSS_HERMITE) ? (size_t)h->gh_M : (size_t)h->M;
  const size_t nd = Ms * std::max(horizon, 0) * h->d;
  if (grad && dual_dirs) {
    CK(h, h->dual_dirs.reserve(nd));
    CK(h, cudaMemcpyAsync(h->dual_dirs, dual_dirs, nd * 8, cudaMemcpyHostToDevice, h->stream));
  }
  if (forced && x_forced) {
    CK(h, h->x_forced.reserve(nd));
    CK(h, cudaMemcpyAsync(h->x_forced, x_forced, nd * 8, cudaMemcpyHostToDevice, h->stream));
  }
  if (x0_batch) {
    CK(h, h->x0_batch.reserve((size_t)B * h->d));
    CK(h, cudaMemcpyAsync(h->x0_batch, x0_batch, (size_t)B * h->d * 8, cudaMemcpyHostToDevice, h->stream));
  }
  rbo_summary local;
  int rc = launch_rollout(h, x0, theta, ntheta, lbs, ubs, horizon, fmini, mode, flags, (grad && dual_dirs) ? h->dual_dirs.p : nullptr,
                          forced ? h->x_forced.p : nullptr, true, summary ? summary : &local, x0_batch ? h->x0_batch.p : nullptr, B);
  if (rc) return rc;
  return rbo_get_results(h, values, grad ? grad_x : nullptr, grad ? grad_theta : nullptr, best_index, grad_case, status);
}

extern "C" {

int rbo_rollout(rbo_handle* h, const double* x0, const double* theta, int ntheta, const double* lbs, const double* ubs, int horizon, double fmini,
                int mode, int flags, const double* dual_dirs, const double* x_forced, double* values, double* grad_x, double* grad_theta,
                int32_t* best_index, int32_t* grad_case, int32_t* status, rbo_summary* summary) {
  if (!h) return RBO_ERR_ARG;
  if (!values) return fail(h, RBO_ERR_ARG, "rbo_rollout: values is NULL");
  if (mode == RBO_MODE_VALUE_GRAD && (!grad_x || !grad_theta)) return fail(h, RBO_ERR_ARG, "rbo_rollout: gradient containers missing in VALUE_GRAD mode");
  return rollout_host(h, x0, nullptr, 1, theta, ntheta, lbs, ubs, horizon, fmini, mode, flags, dual_dirs, x_forced, values, grad_x, grad_theta,
                      best_index, grad_case, status, summary);
}

int rbo_rollout_device(rbo_handle* h, const double* x0, const double* theta, int ntheta, const double* lbs, const double* ubs, int horizon,
                       double fmini, int mode, int flags, const double* dual_dirs_device, const double* x_forced_device, rbo_summary* summary) {
  if (!h) return RBO_ERR_ARG;
  return launch_rollout(h, x0, theta, ntheta, lbs, ubs, horizon, fmini, mode, flags, dual_dirs_device, x_forced_device, summary != nullptr, summary);
}

int rbo_rollout_batch(rbo_handle* h, const double* x0s, int n_x0, const double* theta, int ntheta, const double* lbs, const double* ubs, int horizon,
                      double fmini, int mode, const double* dual_dirs, double* values, double* grad_x, double* grad_theta, int32_t* status,
                      rbo_summary* summary) {
  if (!h) return RBO_ERR_ARG;
  if (!x0s || n_x0 < 1 || !values) return fail(h, RBO_ERR_ARG, "rbo_rollout_batch: bad arguments");
  if (mode == RBO_MODE_VALUE_GRAD && (!grad_x || !grad_theta)) return fail(h, RBO_ERR_ARG, "rbo_rollout_batch: gradient containers missing in VALUE_GRAD mode");
  if (!h->rn) return fail(h, RBO_ERR_STATE, "rbo_rollout_batch: no normals (rbo_set_normals / rbo_generate_normals)");
  return rollout_host(h, x0s, x0s, n_x0, theta, ntheta, lbs, ubs, horizon, fmini, mode, 0, dual_dirs, nullptr, values, grad_x, grad_theta,
                      nullptr, nullptr, status, summary);
}

void rbo_default_sga_opts(rbo_sga_opts* o) {
  if (!o) return;
  o->optimizer = RBO_OPT_ADAM;
  o->max_iterations = 50;  // utils.jl:244
  o->use_eswavs = 1;
  o->project = 0;
  o->eta = 1e-3;  // optimizers.jl:35-40
  o->beta1 = 0.9;
  o->beta2 = 0.999;
  o->eps = 1e-8;
}

int rbo_stochastic_solve_batch(rbo_handle* h, const rbo_sga_opts* o, const double* x0s, int n_x0, const double* theta, int ntheta,
                               const double* lbs, const double* ubs, int horizon, double fmini, const double* dual_dirs,
                               double* x_final, int32_t* n_iter, int32_t* end_status, int32_t* fail_out, double* x_hist,
                               double* mean_hist, double* std_hist, double* gmean_hist, double* gstd_hist, rbo_summary* summary) {
  if (!h) return RBO_ERR_ARG;
  const char* me = "rbo_stochastic_solve_batch";
  if (!o || !x0s || !x_final || !n_iter || !end_status) return fail(h, RBO_ERR_ARG, "%s: o, x0s, x_final, n_iter and end_status are required", me);
  if (n_x0 < 1) return fail(h, RBO_ERR_ARG, "%s: n_x0 = %d < 1", me, n_x0);
  if (o->max_iterations < 1) return fail(h, RBO_ERR_ARG, "%s: max_iterations = %d < 1", me, o->max_iterations);
  if (o->optimizer != RBO_OPT_SGA && o->optimizer != RBO_OPT_ADAM) return fail(h, RBO_ERR_ARG, "%s: unknown optimizer %d", me, o->optimizer);
  if (!(o->eta > 0.0)) return fail(h, RBO_ERR_ARG, "%s: eta = %g must be > 0", me, o->eta);
  if (!h->have_sur) return fail(h, RBO_ERR_STATE, "%s: no surrogate (rbo_set_surrogate)", me);
  if (!h->rn) return fail(h, RBO_ERR_STATE, "%s: no normals (rbo_set_normals / rbo_generate_normals)", me);
  if (!h->starts) return fail(h, RBO_ERR_STATE, "%s: no starts (rbo_set_starts)", me);
  CK(h, cudaSetDevice(h->device));
  const int B = n_x0, d = h->d, Ms = h->M, maxit = o->max_iterations;
  CK(h, h->x0_batch.reserve((size_t)B * d));
  CK(h, cudaMemcpyAsync(h->x0_batch, x0s, (size_t)B * d * 8, cudaMemcpyHostToDevice, h->stream));
  if (dual_dirs) {
    const size_t nd = (size_t)Ms * std::max(horizon, 0) * d;
    CK(h, h->dual_dirs.reserve(nd));
    CK(h, cudaMemcpyAsync(h->dual_dirs, dual_dirs, nd * 8, cudaMemcpyHostToDevice, h->stream));
  }
  DevProblem P;
  PlanChoice pc;
  int grid = 0;
  int rc = prepare_launch(h, x0s, theta, ntheta, lbs, ubs, horizon, fmini, RBO_MODE_VALUE_GRAD, 0, dual_dirs ? h->dual_dirs.p : nullptr, nullptr,
                          h->x0_batch.p, B, P, pc, grid);
  if (rc) return rc;
  const int M = P.M;
  // the conditions under which launch_rollout hands out longest-first; the order then follows the previous iteration's costs
  const bool lpt = h->lpt && horizon > 0 && M > 2 * grid;
  if (lpt) CK(h, h->order.reserve(M));
  const int* order = P.order;

  // device state: doubles [m | v | bias | x_hist | gmean_hist | gstd_hist | mean_hist | std_hist], ints [live | n_iter | end_status |
  // fail (2 per restart) | nfail | sticky watchdog record (16)]
  const size_t nx = (size_t)d * B, nh = (size_t)maxit * B;
  const size_t o_bias = 2 * nx, o_xh = o_bias + 2 * (size_t)maxit, o_gmh = o_xh + nh * d, o_gsh = o_gmh + nh * d, o_mh = o_gsh + nh * d,
               o_sh = o_mh + nh, n_dbl = o_sh + nh;
  const size_t i_iter = B, i_end = 2 * (size_t)B, i_fail = 3 * (size_t)B, i_nfail = 5 * (size_t)B, i_sticky = 6 * (size_t)B, n_int = i_sticky + 16;
  CK(h, h->sga_dbl.reserve(n_dbl));
  CK(h, h->sga_int.reserve(n_int));
  CK(h, h->worklist.reserve(M));
  double* D = h->sga_dbl;
  int* I = h->sga_int;
  std::vector<double> bias(2 * (size_t)maxit);
  for (int t = 1; t <= maxit; ++t) {  // the host mirror's 1 - beta**t: Python's float ** int is the C library's pow
    bias[t - 1] = 1.0 - std::pow(o->beta1, (double)t);
    bias[maxit + t - 1] = 1.0 - std::pow(o->beta2, (double)t);
  }
  std::vector<int> ist(n_int, 0);
  for (int b = 0; b < B; ++b) { ist[b] = 1; ist[i_end + b] = -1; ist[i_fail + 2 * b] = -1; ist[i_fail + 2 * b + 1] = 0; }
  CK(h, cudaMemsetAsync(D, 0, 2 * nx * 8, h->stream));
  CK(h, cudaMemcpyAsync(D + o_bias, bias.data(), bias.size() * 8, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemsetAsync(D + o_xh, 0xff, (n_dbl - o_xh) * 8, h->stream));  // all-ones bytes: NaN past n_iter
  CK(h, cudaMemcpyAsync(I, ist.data(), n_int * sizeof(int), cudaMemcpyHostToDevice, h->stream));

  SgaProblem S;
  memset(&S, 0, sizeof(S));
  S.B = B; S.Ms = Ms; S.d = d; S.maxit = maxit;
  S.optimizer = o->optimizer; S.use_eswavs = o->use_eswavs != 0; S.project = o->project != 0;
  S.eta = o->eta; S.beta1 = o->beta1; S.beta2 = o->beta2; S.eps = o->eps;
  S.omb1 = 1.0 - o->beta1; S.omb2 = 1.0 - o->beta2;
  for (int a = 0; a < d; ++a) { S.lbs[a] = lbs[a]; S.ubs[a] = ubs[a]; }
  S.bias = D + o_bias;
  S.values = h->values; S.grad_x = h->grad_x; S.status = h->status; S.work_counter = h->work_counter;
  S.x = h->x0_batch; S.m = D; S.v = D + nx;
  S.xh = D + o_xh; S.gmh = D + o_gmh; S.gsh = D + o_gsh; S.mh = D + o_mh; S.sh = D + o_sh;
  S.live = I; S.n_iter = I + i_iter; S.end_status = I + i_end; S.fail = I + i_fail; S.nfail = I + i_nfail; S.sticky = I + i_sticky;

  // every iteration enqueued at once: a launch after the last restart stopped hands out nothing
  P.order = h->worklist;
  int launches = 0;
  CK(h, cudaEventRecord(h->ev0, h->stream));
  for (int k = 0; k < maxit; ++k) {
    rbo_sga_worklist_kernel<<<1, 1024, 0, h->stream>>>(order, S.live, Ms, M, h->worklist);
    CK(h, cudaGetLastError());
    CK(h, cudaMemsetAsync(h->work_counter, 0, 16 * sizeof(int), h->stream));
    CK(h, enqueue_rollout(h, P, pc, grid));
    rbo_sga_step_kernel<<<B, 256, 0, h->stream>>>(S, k);
    CK(h, cudaGetLastError());
    launches += 3;
    if (lpt) {
      rbo_lpt_order_kernel<<<1, 1024, 0, h->stream>>>(h->n_evals, h->grad_case, h->best_index, M, horizon, h->order);
      CK(h, cudaGetLastError());
      order = h->order;
      ++launches;
    }
  }
  CK(h, cudaEventRecord(h->ev1, h->stream));
  h->order_M = lpt ? M : 0;
  h->last_mode = RBO_MODE_VALUE_GRAD;
  // the per-trajectory buffers now hold each restart's last iteration: no read-back and no replay until the next rollout
  h->outM = 0; h->outh = -1; h->xs_valid = false;

  std::vector<int> ires(n_int);
  CK(h, cudaMemcpyAsync(x_final, h->x0_batch, nx * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(ires.data(), I, n_int * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  if (x_hist) CK(h, cudaMemcpyAsync(x_hist, D + o_xh, nh * d * 8, cudaMemcpyDeviceToHost, h->stream));
  if (gmean_hist) CK(h, cudaMemcpyAsync(gmean_hist, D + o_gmh, nh * d * 8, cudaMemcpyDeviceToHost, h->stream));
  if (gstd_hist) CK(h, cudaMemcpyAsync(gstd_hist, D + o_gsh, nh * d * 8, cudaMemcpyDeviceToHost, h->stream));
  if (mean_hist) CK(h, cudaMemcpyAsync(mean_hist, D + o_mh, nh * 8, cudaMemcpyDeviceToHost, h->stream));
  if (std_hist) CK(h, cudaMemcpyAsync(std_hist, D + o_sh, nh * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  std::memcpy(n_iter, ires.data() + i_iter, (size_t)B * sizeof(int));
  std::memcpy(end_status, ires.data() + i_end, (size_t)B * sizeof(int));
  if (fail_out) std::memcpy(fail_out, ires.data() + i_fail, 2 * (size_t)B * sizeof(int));
  if (ires[i_sticky]) return watchdog_fail(h, ires.data() + i_sticky);
  if (summary) {
    float ms = 0;
    CK(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    memset(summary, 0, sizeof(*summary));
    summary->mean = NAN;
    summary->std = NAN;
    summary->kernel_ms = ms;
    summary->gpu_launches = launches;
    long long ntraj = 0, nfailed = 0;
    for (int b = 0; b < B; ++b) { ntraj += (long long)ires[i_iter + b] * Ms; nfailed += ires[i_nfail + b]; }
    summary->n_traj = (int)ntraj;
    summary->n_failed = (int)nfailed;
  }
  return RBO_SUCCESS;
}

int rbo_partial_sums_device(rbo_handle* h, double* sums_device, int len) {
  if (!h || !sums_device) return RBO_ERR_ARG;
  const int need = 1 + 3 * (1 + h->outd + h->outnth);
  if (!h->sums || len < need + 2) return fail(h, RBO_ERR_ARG, "rbo_partial_sums_device: need %d doubles (1 + 3 (1 + d + ntheta) + 2)", need + 2);
  CK(h, cudaSetDevice(h->device));
  const int hh = std::max(h->outh, 1);
  const int idx_failed = need + hh + (h->outh + 2);  // sums layout of rbo_stats_kernel: rows, evaluations per step, case-3 histogram, failures
  rbo_gather_sums_kernel<<<1, 64, 0, h->stream>>>(h->sums, need, idx_failed, h->work_counter, sums_device);
  CK(h, cudaGetLastError());
  return RBO_SUCCESS;
}

int rbo_partial_sums_host(rbo_handle* h, double* sums, int len) {
  if (!h || !sums) return RBO_ERR_ARG;
  const int need = 1 + 3 * (1 + h->outd + h->outnth) + 2;
  if (!h->sums || len < need) return fail(h, RBO_ERR_ARG, "rbo_partial_sums_host: need %d doubles (1 + 3 (1 + d + ntheta) + 2)", need);
  CK(h, cudaSetDevice(h->device));
  double* tmp = h->sums + h->sums_len;  // the sums buffer is allocated with room for the gathered vector
  int rc = rbo_partial_sums_device(h, tmp, need);
  if (rc) return rc;
  CK(h, cudaMemcpyAsync(sums, tmp, (size_t)need * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));  // this is the call that waits for the (asynchronous) rbo_rollout_device of this handle
  return RBO_SUCCESS;
}

int rbo_get_results(rbo_handle* h, double* values, double* grad_x, double* grad_theta, int32_t* best_index, int32_t* grad_case, int32_t* status) {
  if (!h) return RBO_ERR_ARG;
  if (h->outh < 0 || h->outM <= 0) return fail(h, RBO_ERR_STATE, "rbo_get_results: no rollout has run");
  if ((grad_x || grad_theta) && h->last_mode != RBO_MODE_VALUE_GRAD) return fail(h, RBO_ERR_STATE, "rbo_get_results: the last rollout computed no gradients");
  CK(h, cudaSetDevice(h->device));
  const size_t M = h->outM;
  CK(h, copy_out(values, h->values, M, h->stream));
  CK(h, copy_out(grad_x, h->grad_x, M * h->outd, h->stream));
  CK(h, copy_out(grad_theta, h->grad_theta, M * h->outnth, h->stream));
  CK(h, copy_out(best_index, h->best_index, M, h->stream));
  CK(h, copy_out(grad_case, h->grad_case, M, h->stream));
  CK(h, copy_out(status, h->status, M, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return RBO_SUCCESS;
}

int rbo_finalize_sums(const double* sums, int d, int ntheta, double* mean, double* std_, double* gx_mean, double* gx_std, double* gth_mean, double* gth_std) {
  if (!sums) return RBO_ERR_ARG;
  const double n = sums[0];
  const int need = 1 + 3 * (1 + d + ntheta);
  // a failed trajectory (where the reference would have thrown) or a kernel watchdog flag on ANY rank poisons the estimate
  if (sums[need] > 0.0 || sums[need + 1] > 0.0) return RBO_ERR_NUMERIC;
  if (!(n > 0)) return RBO_ERR_ARG;
  for (int row = 0; row < 1 + d + ntheta; ++row) {
    const double sm = sums[1 + 3 * row], m2 = sums[2 + 3 * row], smm = sums[3 + 3 * row];
    const double mu = sm / n;
    // sum over groups of [M2_g + n_g (mean_g - mean)^2] = sum M2_g + sum n_g mean_g^2 - n mean^2
    const double tot = std::max(m2 + smm - n * mu * mu, 0.0);
    const double sd = n > 1 ? std::sqrt(tot / (n - 1)) : NAN;
    if (row == 0) { if (mean) *mean = mu; if (std_) *std_ = sd; }
    else if (row <= d) { if (gx_mean) gx_mean[row - 1] = mu; if (gx_std) gx_std[row - 1] = sd; }
    else { if (gth_mean) gth_mean[row - 1 - d] = mu; if (gth_std) gth_std[row - 1 - d] = sd; }
  }
  return RBO_SUCCESS;
}

int rbo_get_tape(rbo_handle* h, double* xs, double* ys, double* gys, double* alphas, int32_t* n_evals, int32_t* start_status, int32_t* start_iters) {
  if (!h) return RBO_ERR_ARG;
  if (h->outh < 0) return fail(h, RBO_ERR_STATE, "rbo_get_tape: no rollout has run");
  CK(h, cudaSetDevice(h->device));
  const size_t M = h->outM, hor = h->outh, hh = std::max(h->outh, 1), d = h->outd, S = h->outS;
  CK(h, copy_out(xs, h->xs, M * (hor + 1) * d, h->stream));
  CK(h, copy_out(ys, h->ys, M * (hor + 1), h->stream));
  CK(h, copy_out(gys, h->gys, M * (hor + 1) * d, h->stream));
  CK(h, copy_out(alphas, h->alphas, M * hh, h->stream));
  CK(h, copy_out(n_evals, h->n_evals, M * hh, h->stream));
  CK(h, copy_out(start_status, h->start_status, M * hh * S, h->stream));
  CK(h, copy_out(start_iters, h->start_iters, M * hh * S, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return RBO_SUCCESS;
}

extern "C" int rbo_get_tape_ex(rbo_handle* h, double* mu, double* sigma, double* dmu, double* dsigma, double* Halpha) {
  if (!h) return RBO_ERR_ARG;
  if (!h->tex_valid) return fail(h, RBO_ERR_STATE, "rbo_get_tape_ex: the last rollout did not run with RBO_FLAG_TAPE_EX");
  CK(h, cudaSetDevice(h->device));
  const size_t n = (size_t)h->outM * std::max(h->outh, 0), d = h->outd;
  CK(h, copy_out(mu, h->t_mu, n, h->stream));
  CK(h, copy_out(sigma, h->t_sigma, n, h->stream));
  CK(h, copy_out(dmu, h->t_dmu, n * d, h->stream));
  CK(h, copy_out(dsigma, h->t_dsigma, n * d, h->stream));
  CK(h, copy_out(Halpha, h->t_Halpha, n * d * d, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return RBO_SUCCESS;
}

static int sobol_common(rbo_handle* h, int dim, int npoints, uint32_t* out_u32, double* out_f64, const double* lbs, const double* ubs) {
  if (!h) return RBO_ERR_ARG;
  if (dim < 1 || dim > RBO_SOBOL_MAXDIM || npoints < 1) return fail(h, RBO_ERR_ARG, "sobol: dim %d / npoints %d out of range", dim, npoints);
  CK(h, cudaSetDevice(h->device));
  const size_t total = (size_t)dim * npoints;
  DevBuf<unsigned> du;
  DevBuf<double> df, db;
  if (out_u32) CK(h, du.reserve(total));
  if (out_f64) CK(h, df.reserve(total));
  if (lbs) {
    CK(h, db.reserve((size_t)2 * dim));
    CK(h, cudaMemcpyAsync(db, lbs, (size_t)dim * 8, cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaMemcpyAsync(db + dim, ubs, (size_t)dim * 8, cudaMemcpyHostToDevice, h->stream));
  }
  int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)h->num_sms * 8);
  rbo_sobol_kernel<<<blocks, 256, 0, h->stream>>>(h->sobol_dirs, du, df, dim, npoints, db, db ? db + dim : nullptr);
  CK(h, cudaGetLastError());
  CK(h, copy_out(out_u32, du, total, h->stream));
  CK(h, copy_out(out_f64, df, total, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return RBO_SUCCESS;
}

int rbo_sobol_uniform(rbo_handle* h, int dim, int npoints, double* out) { return sobol_common(h, dim, npoints, nullptr, out, nullptr, nullptr); }
int rbo_sobol_uint32(rbo_handle* h, int dim, int npoints, uint32_t* out) { return sobol_common(h, dim, npoints, out, nullptr, nullptr, nullptr); }

int rbo_generate_initial_guesses(rbo_handle* h, int S, int d, const double* lbs, const double* ubs, double* out) {
  if (!h || !lbs || !ubs || !out || S < 0 || d < 1) return RBO_ERR_ARG;
  if (S > 0) {
    int rc = sobol_common(h, d, S, nullptr, out, lbs, ubs);
    if (rc) return rc;
  }
  const double eps = 1e-6;  // utils.jl:146
  for (int a = 0; a < d; ++a) { out[(size_t)S * d + a] = lbs[a] + eps; out[(size_t)(S + 1) * d + a] = ubs[a] - eps; }
  return RBO_SUCCESS;
}

int rbo_multistart_base_solve(rbo_handle* h, const double* theta, int ntheta, const double* lbs, const double* ubs, double* xfinal, double* alpha,
                              rbo_summary* summary) {
  if (!h) return RBO_ERR_ARG;
  if (!xfinal) return fail(h, RBO_ERR_ARG, "rbo_multistart_base_solve: xfinal is NULL");
  if (!h->have_sur) return fail(h, RBO_ERR_STATE, "rbo_multistart_base_solve: no surrogate");
  double x0[RBO_MAXD] = {0};
  rbo_summary local;
  int rc = launch_rollout(h, x0, theta, ntheta, lbs, ubs, 0, 0.0, RBO_MODE_VALUE, RBO_FLAG_MYOPIC_INTERNAL, nullptr, nullptr, true, summary ? summary : &local);
  if (rc) return rc;
  double a = 0;
  int st = 0;
  CK(h, cudaMemcpyAsync(xfinal, h->xs, (size_t)h->d * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(&a, h->values, 8, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(&st, h->status, 4, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  if (alpha) *alpha = a;
  if (st != RBO_TRAJ_OK) return fail(h, RBO_ERR_NUMERIC, "rbo_multistart_base_solve: every start produced NaN (rbf_optim.jl:129-130 would throw)");
  return RBO_SUCCESS;
}

int rbo_num_sms(const rbo_handle* h) { return h ? h->num_sms : 0; }



int rbo_fp64_peak(rbo_handle* h, double* tflops) {
  if (!h || !tflops) return RBO_ERR_ARG;
  CK(h, cudaSetDevice(h->device));
  const int blocks = h->num_sms * 4, threads = 512, iters = 4096;
  DevBuf<double> out;
  CK(h, out.reserve((size_t)blocks * threads));
  double best = 0;
  for (int rep = 0; rep < 5; ++rep) {
    CK(h, cudaEventRecord(h->ev0, h->stream));
    rbo_fp64_peak_kernel<<<blocks, threads, 0, h->stream>>>(out, iters);
    CK(h, cudaEventRecord(h->ev1, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    float ms;
    CK(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    double fl = (double)blocks * threads * iters * 16.0 * 2.0;
    if (rep > 0) best = std::max(best, fl / (ms * 1e-3) / 1e12);
  }
  *tflops = best;
  return RBO_SUCCESS;
}

int rbo_tr_step_batch(rbo_handle* h, int n, int B, const double* H, const double* g, const double* Delta, double* p, int* hit) {
  if (!h || !H || !g || !Delta || !p || !hit || B < 1) return RBO_ERR_ARG;
  if (n < 1 || n > RBO_MAXD) return fail(h, RBO_ERR_UNSUPPORTED, "rbo_tr_step_batch: n = %d outside [1, %d]", n, RBO_MAXD);
  CK(h, cudaSetDevice(h->device));
  DevBuf<double> dH, dg, dD, dp;
  DevBuf<int> dh;
  CK(h, dH.reserve((size_t)B * n * n));
  CK(h, dg.reserve((size_t)B * n));
  CK(h, dD.reserve(B));
  CK(h, dp.reserve((size_t)B * n));
  CK(h, dh.reserve(B));
  CK(h, cudaMemcpyAsync(dH, H, (size_t)B * n * n * 8, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemcpyAsync(dg, g, (size_t)B * n * 8, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemcpyAsync(dD, Delta, (size_t)B * 8, cudaMemcpyHostToDevice, h->stream));
  const int wpb = n > 16 ? 2 : 4;  // <= 48 KB of dynamic shared memory
  const size_t smem = (size_t)wpb * (2 * n * n + 4 * n + 32) * 8;
  rbo_tr_step_kernel<<<(B + wpb - 1) / wpb, 32 * wpb, smem, h->stream>>>(dH, dg, dD, n, B, dp, dh);
  CK(h, cudaGetLastError());
  CK(h, copy_out(p, dp, (size_t)B * n, h->stream));
  CK(h, copy_out(hit, dh, B, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return RBO_SUCCESS;
}

}  // extern "C"
