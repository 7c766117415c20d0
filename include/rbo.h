/*
 * rbo.h -- C ABI of librbo.so: the B200-native (sm_100a, FP64 CUDA) implementation of the Monte-Carlo
 * rollout acquisition estimator and its adjoint gradient.
 *
 * The reference (DarianNwankwo/Rollout-Bayesian-Optimization) is pure Julia with no FFI; the seam this
 * library plugs into is the Julia call
 *     simulate_trajectory_mc(T::Trajectory, tp::TrajectoryParameters; inner_solve_xstarts, resolutions,
 *                            spatial_gradients_container, hyperparameter_gradients_container)
 * (rollout.jl:279-340). A Julia shim re-defines that method as marshalling + `ccall` into the entry points
 * below (see INTEGRATION.md and rollout-bayesian-optimization_b200/julia/). Each entry point cites the
 * reference code it replaces.
 *
 * Conventions: all arrays FP64, column-major (Julia layout), caller-owned, host memory unless the name
 * says "device"; every function returns 0 (RBO_SUCCESS) or a negative error code and records a message
 * retrievable with rbo_last_error(). A handle is bound to one CUDA device and one stream; it is
 * thread-compatible (one thread at a time per handle). There is NO CPU fallback: without a CUDA device
 * rbo_create() fails with RBO_ERR_CUDA.
 */
#ifndef RBO_H
#define RBO_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RBO_ABI_VERSION 2

typedef struct rbo_handle rbo_handle;

enum { RBO_SUCCESS = 0, RBO_ERR_ARG = -1, RBO_ERR_CUDA = -2, RBO_ERR_STATE = -3, RBO_ERR_UNSUPPORTED = -4, RBO_ERR_NUMERIC = -5 };

/* rbf.jl:60-103 : RadialBasisFunction constructors (kernel_id is derived from rbf.constructor) */
enum { RBO_KERNEL_MATERN12 = 0, RBO_KERNEL_MATERN32 = 1, RBO_KERNEL_MATERN52 = 2, RBO_KERNEL_SE = 3, RBO_KERNEL_PERIODIC = 4 };
/* decision_rules.jl:84-127 : DecisionRule.name */
enum { RBO_RULE_EI = 0, RBO_RULE_POI = 1, RBO_RULE_LCB = 2 };
/* which outputs rbo_rollout computes: resolutions only, or resolutions + gradient(T) (rollout.jl:318-323) */
enum { RBO_MODE_VALUE = 0, RBO_MODE_VALUE_GRAD = 1 };
/* flags */
enum {
  RBO_FLAG_TEACHER_FORCED = 1, /* x_1..x_h supplied by the caller (step-level parity tests) */
  RBO_FLAG_TAPE_EX = 4,        /* also record mu, sigma, grad mu, grad sigma, H alpha, alpha of the policy solve's surrogate evaluation at
                                  every chosen x_j (one extra evaluation per step): rbo_get_tape_ex */
  RBO_FLAG_REPLAY_TAPE = 8,    /* teacher-force the x-path the PREVIOUS rollout of this handle left on the device (same samples, same horizon):
                                  second phase of the two-phase call that reproduces the reference's rand(dim) consumption (rollout.jl:133):
                                  phase 1 = RBO_MODE_VALUE (values, best_index), host draws the dual directions for the case-3 samples
                                  in the reference's order, phase 2 = RBO_MODE_VALUE_GRAD | this flag (no inner solves, bitwise replay) */
  RBO_FLAG_GAUSS_HERMITE = 2   /* simulate_trajectory_ghq (rollout.jl:409-467): GaussHermiteObservable draws (observables.jl:32-81,157)
                                  from the nodes / weights of rbo_set_quadrature instead of the normals */
};

/* per-trajectory status: what the reference would have thrown for that sample (SURVEY.md section 5) */
enum {
  RBO_TRAJ_OK = 0,
  RBO_TRAJ_NOT_PD_ROW = 1,      /* rbs.jl:412  PosDefException in update_cholesky! */
  RBO_TRAJ_NEG_VARIANCE = 2,    /* rbs.jl:528  DomainError in sqrt */
  RBO_TRAJ_NOT_PD_JOINT = 3,    /* rbs.jl:537  PosDefException in the joint value/gradient covariance */
  RBO_TRAJ_ALL_STARTS_NAN = 4,  /* rbf_optim.jl:96-97 findmin over an empty collection */
  RBO_TRAJ_SINGULAR_HESSIAN = 5 /* rollout.jl:188 SingularException */
};

/* per-start inner-solve status */
enum { RBO_SOLVE_CONVERGED = 0, RBO_SOLVE_MAXIT = 1, RBO_SOLVE_STEP_TINY = 2, RBO_SOLVE_PRED_TINY = 3, RBO_SOLVE_STALLED = 4, RBO_SOLVE_NAN = 5,
       RBO_SOLVE_FINAL_STEP = 6 /* ended with an interior Newton step below stol, taken without re-evaluation */ };

/* Inner box-constrained maximiser (replaces Optim.IPNewton, rbf_optim.jl:24-30): projected trust-region Newton with the
 * exact subproblem solution, modelled on the reference's own tr_newton / solve_tr (optim.jl:9-114), on the merit
 * -log(alpha) (EI, POI) or -alpha (LCB). Radius update and acceptance as optim.jl:93-99. */
typedef struct {
  int32_t maxit;     /* accepted steps per start */
  int32_t maxtry;    /* consecutive rejected / non-descent steps before a start is declared stalled */
  double gtol;       /* stop: max |projected gradient of alpha| <= gtol * max(1, |alpha|) */
  double xtol;       /* stop: max |step| <= xtol * max(1, max |x|) */
  double pred_tol;   /* stop: predicted decrease of the merit <= pred_tol * max(1, |merit|) */
  double eta;        /* acceptance ratio rho >= eta (optim.jl:99: 0.1) */
  double delta0_box; /* initial radius = min(delta0_box * widest box side, */
  double delta0_ell; /*                      delta0_ell * kernel hyper-parameter ktheta[0] (the length-scale)) */
  double stol;       /* an interior Newton step with max |s| <= stol * max(1, max |x|) is taken without re-evaluation and ends the start */
} rbo_solver_opts;

/* Summary of one estimator evaluation: ExpectedTrajectoryOutput (trajectory.jl:112-134) computed as
 * rollout.jl:328-337 over the trajectories this handle processed, plus accounting for bench.py. */
typedef struct {
  double mean, std;             /* mu_x_theta, sigma_mu_x_theta (corrected sample std) */
  int32_t n_traj, n_failed;     /* trajectories processed / with status != RBO_TRAJ_OK */
  double kernel_ms;             /* device time of the rollout kernel(s), CUDA events on the handle's stream */
  double flops;                 /* algorithmic FP64 flops (SURVEY.md 8d formula with the solver's measured evaluation counts) */
  double flops_executed;        /* FP64 flops this implementation executes for the same work (fewer: forward-only solves) */
  int64_t n_evals;              /* acquisition evaluations performed by the inner solves */
  int32_t gpu_launches;         /* kernels launched by this call */
  double tail_ms;               /* tail of the persistent grid: last CTA to finish minus the median CTA (device %globaltimer) */
} rbo_summary;

/* ---- life cycle ------------------------------------------------------------------------------ */
int rbo_abi_version(void);
/* Creates a handle on CUDA device `device_id` with its own non-blocking stream. */
int rbo_create(rbo_handle** out, int device_id);
int rbo_destroy(rbo_handle* h);
/* Message of the last failing call on this handle (or of rbo_create when h == NULL). */
const char* rbo_last_error(const rbo_handle* h);
/* Use an externally owned cudaStream_t (e.g. torch's current stream); NULL restores the handle's own stream. */
int rbo_set_stream(rbo_handle* h, void* cuda_stream);
void rbo_default_solver_opts(rbo_solver_opts* o);
int rbo_set_solver_opts(rbo_handle* h, const rbo_solver_opts* o);
/* htol of solve_dual_x (rollout.jl:156; the reference never overrides its default 1e-4): a policy solve whose
 * det(H alpha) < htol contributes a zero dual (Q3). Exposed so tests can exercise the full adjoint. */
int rbo_set_htol(rbo_handle* h, double htol);

/* Execution knobs (results do not depend on them beyond rounding): RBO_TUNE_LARGE_N != 0 forces the large-n variant of the
 * kernel -- work matrix in an L2-resident global scratch instead of shared memory; chosen automatically when a problem does
 * not fit 227 KB (e.g. n = 1000, d = 20) -- and RBO_TUNE_LARGE_N_SLOTS caps its start slots per round (0 = default). */
enum { RBO_TUNE_LARGE_N = 1, RBO_TUNE_LARGE_N_SLOTS = 2,
       RBO_TUNE_LPT = 3 /* default 1: hand the trajectories out longest-first, using the evaluation counts of the previous launch on the
                           same samples as the cost estimate (scheduling only: per-trajectory results do not depend on it) */,
       RBO_TUNE_ROW_SPLITS = 4 /* cap (1..4, 0 = default) on the row splits of the Gram reductions: plan experiments */ };
int rbo_set_tuning(rbo_handle* h, int key, int value);

/* ---- inputs (resident on the device until replaced) ------------------------------------------ */
/* The base surrogate the fantasy surrogate is built from: FantasySurrogate(s, h) (rbs.jl:345-381) reads
 * fs.X[:,1:N], fs.L[1:N,1:N], fs.y[1:N], fs.cs[1], fs.sigma_n2, fs.psi, fs.g.
 * X: d x N (ldX >= d).  L: N x N lower triangle of a column-major buffer with leading dimension ldL
 * (Julia's LowerTriangular .data).  c = K^-1 y.
 * N <= 12800 bounds only the inversion into the device form; the rollout admits fewer observations (see rbo_rollout). */
int rbo_set_surrogate(rbo_handle* h, int d, int N, const double* X, int ldX, const double* L, int ldL,
                      const double* y, const double* c, double sigma_n2, int kernel_id, const double* ktheta,
                      int nktheta, int rule_id, double sigma_tol);

/* condition!(s::Surrogate, x, y) (rbs.jl:214-222) on the RESIDENT surrogate: appends the observation (x[d], y), extends the
 * kernel-matrix row (update_covariance!, rbs.jl:166-183), the factor by one row (update_cholesky!, rbs.jl:185-203: here the
 * matching row of L0^-1) and re-solves the coefficients (update_coefficients!, rbs.jl:205-212), all on the device: the factor
 * never returns to the host between Bayesian-optimisation iterations. RBO_ERR_NUMERIC where the reference would throw
 * PosDefException; the resident surrogate is then unchanged. Normals, starts and quadrature data stay valid. */
int rbo_condition(rbo_handle* h, const double* x, double y);
/* Reads the resident surrogate back (any pointer may be NULL): N, X (d x N, ldX >= d), y[N], c[N] = K^-1 y. */
int rbo_get_surrogate(rbo_handle* h, int* N, double* X, int ldX, double* y, double* c);

/* tp.rnstream_sequence (trajectory.jl:47): M_total x (d+1) x hp1, column-major, sample index fastest.
 * This handle keeps samples [m_begin, m_begin + m_count). */
int rbo_set_normals(rbo_handle* h, const double* rn, int M_total, int hp1, int m_begin, int m_count);
/* gen_low_discrepancy_sequence(M_total, d, hp1) (utils.jl:65-74: Sobol -> log10 Box-Muller -> reshape)
 * generated on the device for samples [m_begin, m_begin + m_count). Requires rbo_set_surrogate (for d). */
int rbo_generate_normals(rbo_handle* h, int M_total, int hp1, int m_begin, int m_count);
/* Copies the handle's normals back: out is m_count x (d+1) x hp1 column-major. */
int rbo_get_normals(rbo_handle* h, double* out);
/* Quadrature data of simulate_trajectory_ghq (rollout.jl:409-467): for sample i the reference sets the observable's
 * nodes / weights to nodes[indices[i]], weights[indices[i]] (rollout.jl:431-432). nodes, weights: depth x m_count,
 * column-major (step fastest), depth >= horizon + 1. Used by rbo_rollout with RBO_FLAG_GAUSS_HERMITE. */
int rbo_set_quadrature(rbo_handle* h, const double* nodes, const double* weights, int depth, int m_count);
/* inner_solve_xstarts (rollout.jl:282): d x S, S = number of columns (the reference passes S+2). S <= 65535. */
int rbo_set_starts(rbo_handle* h, const double* starts, int S);

/* ---- the hot path ---------------------------------------------------------------------------- */
/* simulate_trajectory_mc (rollout.jl:279-340) for the handle's samples.
 *   x0[d], lbs[d], ubs[d]   : tp.x0, tp.spatial_lbs/ubs      theta[ntheta] : tp.theta (decision-rule hypers)
 *   horizon                 : tp.horizon (hp1 of the normals must be >= horizon + 1)
 *   fmini                   : minimum(get_observations(base surrogate)) as the reference computes it
 *                             (rollout.jl:109,234: over the zero-padded capacity-length vector)
 *   dual_dirs               : d x horizon x m_count, the rand(dim) draws of solve_dual_y (rollout.jl:133),
 *                             indexed [k, solve_index, m]; NULL = zeros. Only read in VALUE_GRAD mode.
 *   x_forced                : d x horizon x m_count, only with RBO_FLAG_TEACHER_FORCED
 *   values[m_count]         : resolutions (rollout.jl:318)
 *   grad_x[d x m_count], grad_theta[ntheta x m_count] : the gradient containers (rollout.jl:321-322); both required in
 *                             RBO_MODE_VALUE_GRAD (RBO_ERR_ARG otherwise), ignored in RBO_MODE_VALUE
 *   best_index, grad_case, status : int32[m_count], may be NULL (t of rollout.jl:235; case 1/2/3 of :239-251)
 *   summary                 : may be NULL
 * Largest N: the fantasy factor block and its pitch stay in shared memory even in the large-n variant, so the largest N a
 * rollout admits depends on d, the horizon, the number of start columns and the mode: e.g. 2640 at d = 10, h = 5 and 2296 at
 * d = 20, h = 2 (10 start columns, with gradients, 227 KB of shared memory per block on the B200). Beyond it RBO_ERR_UNSUPPORTED;
 * the handle stays usable (a smaller surrogate can be set).
 */
int rbo_rollout(rbo_handle* h, const double* x0, const double* theta, int ntheta, const double* lbs, const double* ubs,
                int horizon, double fmini, int mode, int flags, const double* dual_dirs, const double* x_forced,
                double* values, double* grad_x, double* grad_theta, int32_t* best_index, int32_t* grad_case,
                int32_t* status, rbo_summary* summary);

/* The estimator at n_x0 starting points in ONE launch (SURVEY.md section 8 f.1: the batch of stochastic-ascent restarts of
 * the reference's outer loop, utils.jl:235-265 / the old driver's --batch-size): trajectory (b, m) starts at x0s[:, b] and uses
 * sample m of the resident normals (common random numbers across the batch, as a serial loop over simulate_trajectory_mc
 * with the same TrajectoryParameters would). x0s: d x n_x0; dual_dirs: d x h x m_count (shared by the batch) or NULL;
 * values: m_count x n_x0, grad_x: d x m_count x n_x0, grad_theta: ntheta x m_count x n_x0, status: m_count x n_x0
 * (column-major, sample index fastest within a starting point). Identical, bit for bit, to n_x0 calls of rbo_rollout. */
int rbo_rollout_batch(rbo_handle* h, const double* x0s, int n_x0, const double* theta, int ntheta, const double* lbs, const double* ubs, int horizon,
                      double fmini, int mode, const double* dual_dirs, double* values, double* grad_x, double* grad_theta, int32_t* status,
                      rbo_summary* summary);
/* Same computation, results left on the device (no per-trajectory D2H): only x0 (d doubles) goes in and the
 * partial sums come out through rbo_partial_sums_device. Used by the SGA loop and by bench.py's device-resident
 * timing. dual_dirs_device / x_forced_device are device pointers or NULL. */
int rbo_rollout_device(rbo_handle* h, const double* x0, const double* theta, int ntheta, const double* lbs,
                       const double* ubs, int horizon, double fmini, int mode, int flags,
                       const double* dual_dirs_device, const double* x_forced_device, rbo_summary* summary);

/* ---- stochastic gradient ascent of the estimator over x0 (utils.jl:235-265), all on the device --- */
enum { RBO_OPT_SGA = 0, RBO_OPT_ADAM = 1 };                         /* StandardSGA (optimizers.jl:6-22) / Adam (optimizers.jl:25-75) */
enum { RBO_SGA_MAXIT = 0, RBO_SGA_ESWAVS = 1, RBO_SGA_FAILED = 2 };  /* why a restart ended */
typedef struct {
  int32_t optimizer;      /* RBO_OPT_* */
  int32_t max_iterations; /* estimator evaluations per restart (utils.jl:244: 50) */
  int32_t use_eswavs;     /* stop a restart when the ESWAVS test of utils.jl:114-123 holds */
  int32_t project;        /* 0: no projection (the reference); 1: clamp x to [lbs, ubs] after every step */
  double eta, beta1, beta2, eps; /* step size; Adam's moment decays and denominator guard (unused by RBO_OPT_SGA) */
} rbo_sga_opts;
/* Adam, eta 1e-3, beta1 0.9, beta2 0.999, eps 1e-8 (optimizers.jl:35-40), 50 iterations, ESWAVS on, no projection. */
void rbo_default_sga_opts(rbo_sga_opts* o);
/* stochastic_solve (utils.jl:235-265) from n_x0 = B restarts at once: each restart b starts at x0s[:, b] with a fresh optimiser
 * state and evaluates the estimator on all of this handle's samples (common random numbers across restarts and iterations, as
 * rbo_rollout_batch). The host enqueues every iteration and synchronises once at the end. For restart b and k = 1..max_iterations:
 *   1. the VALUE_GRAD rollout of every sample at x_k;
 *   2. record x_k, the mean and corrected std of the values, the mean and corrected std of every grad_x row (two-pass, in a fixed
 *      reduction order: deterministic; failed trajectories are excluded);
 *   3. a failed trajectory ends the restart with RBO_SGA_FAILED at x_k; fail[:, b] = (first failing sample index in sample order,
 *      as the serial reference throws there; its RBO_TRAJ_* status);
 *   4. with use_eswavs, (1 - (M/d) * sum(g^2 / var)) > 0 (var = std^2 of the rounded std, the sum in numpy's order) ends the
 *      restart with RBO_SGA_ESWAVS at x_k;
 *   5. otherwise the optimiser step of api.update_optimizer / update! (optimizers.jl:16-22, 48-75), then the clamp if project.
 * A restart that performs max_iterations evaluations ends with RBO_SGA_MAXIT and x_final is the iterate after its last step.
 * Numerics: the step is evaluated in the reference's operation order without contractions, m = b1 m + (1-b1) g,
 * v = b2 v + (1-b2) g g, x += (eta mhat) / (sqrt(vhat) + eps), with the bias corrections 1 - b^t computed on the host by the C
 * library's pow: the iterates equal, bit for bit, the host mirror's update fed the recorded gradient means.
 *   dual_dirs : d x h x m_count, shared by all restarts and iterations, or NULL = zeros
 *   x_final   : d x B;  n_iter, end_status : B each (evaluations performed, RBO_SGA_*);  fail : 2 x B or NULL
 *   x_hist, mean_hist, std_hist, gmean_hist, gstd_hist : NULL or d x maxit x B, maxit x B, maxit x B, d x maxit x B,
 *               d x maxit x B (column-major); NaN past n_iter[b]
 *   summary   : may be NULL; kernel_ms of the whole loop, gpu_launches, n_traj = trajectories run, n_failed
 * Errors: RBO_ERR_ARG for n_x0 < 1, max_iterations < 1, an unknown optimiser or eta <= 0; RBO_ERR_STATE without surrogate,
 * normals or starts; the plan limits of rbo_rollout (RBO_ERR_UNSUPPORTED); RBO_ERR_CUDA with the watchdog message if the rollout
 * kernel reported a stuck pipeline (every restart stops then). Afterwards the handle keeps its surrogate, normals and starts;
 * RBO_FLAG_REPLAY_TAPE and the per-trajectory read-backs are refused until the next rollout, because the last launch did not
 * run every restart. One GPU only: the per-iteration statistics of several would need an all-reduce inside the loop. */
int rbo_stochastic_solve_batch(rbo_handle* h, const rbo_sga_opts* o, const double* x0s, int n_x0, const double* theta, int ntheta,
                               const double* lbs, const double* ubs, int horizon, double fmini, const double* dual_dirs,
                               double* x_final, int32_t* n_iter, int32_t* end_status, int32_t* fail, double* x_hist,
                               double* mean_hist, double* std_hist, double* gmean_hist, double* gstd_hist, rbo_summary* summary);

/* Per-handle partial statistics of the last rollout, for the multi-GPU all-reduce:
 * sums = [n, n*mean_v, M2_v, n*mean_v^2, (n*mean, M2, n*mean^2) per grad_x row..., per grad_theta row..., n_failed, watchdog]
 * length 1 + 3*(1 + d + ntheta) + 2. Written to a DEVICE buffer (e.g. a torch tensor handed to NCCL), stream-ordered.
 * n counts the trajectories with status RBO_TRAJ_OK only -- failed ones are excluded from every sum and counted in n_failed;
 * watchdog != 0 if the kernel reported a stuck pipeline or an inner solve beyond its evaluation bound.
 * M2 is the centred sum of squares around this handle's own mean (two-pass, as rollout.jl:328-337). */
int rbo_partial_sums_device(rbo_handle* h, double* sums_device, int len);
/* The same vector on the HOST, for a single-process multi-GPU host (e.g. Julia: one handle per device, rbo_rollout_device on each --
 * the launches are asynchronous --, then this call per handle, an element-wise sum, rbo_finalize_sums): waits for this handle's launch. */
int rbo_partial_sums_host(rbo_handle* h, double* sums, int len);
/* Per-trajectory results of the last rollout of this handle (its shard of the containers): any pointer may be NULL. */
int rbo_get_results(rbo_handle* h, double* values, double* grad_x, double* grad_theta, int32_t* best_index, int32_t* grad_case, int32_t* status);
/* Host-side merge of all-reduced sums into means / corrected sample stds (Chan's pairwise update). Returns RBO_ERR_NUMERIC
 * when any rank reported a failed trajectory or a watchdog flag (the reference would have thrown): no silent estimates. */
int rbo_finalize_sums(const double* sums, int d, int ntheta, double* mean, double* std, double* gx_mean,
                      double* gx_std, double* gth_mean, double* gth_std);

/* Tape of the last rollout (single-trajectory inspection, sample(T)/best(T) of rollout.jl:85-105, and the
 * step-level parity tests). Any pointer may be NULL.
 *   xs[d x (h+1) x m_count], ys[(h+1) x m_count], gys[d x (h+1) x m_count], alphas[h x m_count],
 *   n_evals[h x m_count] (int32), start_status / start_iters [S x h x m_count] (int32) */
int rbo_get_tape(rbo_handle* h, double* xs, double* ys, double* gys, double* alphas, int32_t* n_evals,
                 int32_t* start_status, int32_t* start_iters);

/* Extended tape of the last rollout run with RBO_FLAG_TAPE_EX: sx_j = fs(x_j, theta; fantasy_index = j-1) (rbs.jl:482-581), the
 * surrogate evaluation policy solve j maximised, at the chosen x_j, j = 1..h:
 *   mu[h x m_count], sigma[h x m_count], dmu[d x h x m_count], dsigma[d x h x m_count], Halpha[d x d x h x m_count] (the
 *   reference's H alpha, rbs.jl:568, i.e. without the mu-sigma cross term). alphas of rbo_get_tape then holds alpha(x_j) in
 *   teacher-forced mode as well. Any pointer may be NULL. */
int rbo_get_tape_ex(rbo_handle* h, double* mu, double* sigma, double* dmu, double* dsigma, double* Halpha);

/* ---- generators the reference's host code provides (utils.jl), same arithmetic on the device -- */
/* gen_uniform (utils.jl:4-13): dim x npoints Sobol points (Joe-Kuo, Gray code, origin skipped). */
int rbo_sobol_uniform(rbo_handle* h, int dim, int npoints, double* out);
int rbo_sobol_uint32(rbo_handle* h, int dim, int npoints, uint32_t* out);
/* generate_initial_guesses (utils.jl:145-153): out is d x (S+2). */
int rbo_generate_initial_guesses(rbo_handle* h, int S, int d, const double* lbs, const double* ubs, double* out);

/* ---- myopic solve (what experiments/*_bayesopt.jl time) --------------------------------------- */
/* multistart_base_solve!(::Surrogate, xfinal; ...) (rbf_optim.jl:103-134) against the resident base
 * surrogate and starts: xfinal[d], and optionally the acquisition value there. */
int rbo_multistart_base_solve(rbo_handle* h, const double* theta, int ntheta, const double* lbs, const double* ubs,
                              double* xfinal, double* alpha, rbo_summary* summary);

/* ---- measurement support ---------------------------------------------------------------------- */
/* Dense FP64 FMA micro-benchmark on this handle's device (TFLOP/s): the roofline denominator of this path,
 * because MEASURED_PEAKS.json carries no FP64 figure. */
int rbo_fp64_peak(rbo_handle* h, double* tflops);
/* Diagnostic: the device code of the inner solver's exact trust-region step (DESIGN.md section 4; replaces the subproblem solves
 * inside Optim.IPNewton, rbf_optim.jl:24-30, and follows solve_tr, optim.jl:9-51) on B independent subproblems
 * min g'p + p'Hp/2, |p|_2 <= Delta: H[B][n*n] (symmetric, row-major), g[B][n], Delta[B] -> p[B][n], hit[B] (1: constraint
 * active). 2 <= n <= 16 takes the register-resident path of the rollout kernel, other n the general one. For step-level parity
 * tests against the oracle's orc_tr_step. */
int rbo_tr_step_batch(rbo_handle* h, int n, int B, const double* H, const double* g, const double* Delta, double* p, int* hit);
/* Number of SMs of the handle's device. */
int rbo_num_sms(const rbo_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* RBO_H */
