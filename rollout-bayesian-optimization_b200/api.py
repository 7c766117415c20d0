"""Host-side mirror of the reference's Julia interface for the rollout path, over the C ABI of librbo.so.

The reference's host language (Julia) is not installed in this image, so the host side that tests and bench.py
drive is this Python mirror: same type and function names, argument meaning and error behaviour as the
reference (file:line cited per item), marshalling into exactly the C entry points a Julia `ccall` shim binds
(see julia/rollout_bayesian_optimization.jl and INTEGRATION.md). Julia's `f!` names drop the `!`.

Arrays follow Julia's layout: X is d x N (columns are points), containers are d x M, all column-major.
Nothing here computes the hot path on the CPU: simulate_trajectory_mc / multistart_base_solve call the CUDA
library and raise if it is missing.
"""
import ctypes as C

import numpy as np
from scipy.linalg import cholesky, solve_triangular

from . import _lib
from ._lib import Handle, RboError, Summary, dptr, iptr

DEFAULT_CAPACITY = 100  # constants.jl:12
GROUND_TRUTH_OBSERVATIONS = -1  # constants.jl:7

KERNEL_IDS = {"Matern12": 0, "Matern32": 1, "Matern52": 2, "SquaredExponential": 3, "Periodic": 4}
RULE_IDS = {"EI": 0, "POI": 1, "LCB": 2}


# ----------------------------------------------------------------------------------------------------
# rbf.jl:7-103  RadialBasisFunction and its constructors
# ----------------------------------------------------------------------------------------------------
class RadialBasisFunction:
    """rbf.jl:7-14. `constructor` names the kernel (rbf.jl:13) and selects the device kernel id."""

    def __init__(self, theta, constructor):
        self.θ = np.asarray(theta, dtype=np.float64).copy()
        self.constructor = constructor
        self.kernel_id = KERNEL_IDS[constructor]

    def __call__(self, rho):  # rbf.jl:20 with the kernels of rbf.jl:60-103
        rho = np.asarray(rho, dtype=np.float64)
        t = self.θ
        if self.constructor == "Matern52":
            s = np.sqrt(5.0) / t[0] * rho
            return (1 + s * (1 + s / 3.0)) * np.exp(-s)
        if self.constructor == "Matern32":
            s = np.sqrt(3.0) / t[0] * rho
            return (1 + s) * np.exp(-s)
        if self.constructor == "Matern12":
            return np.exp(-rho / t[0])
        if self.constructor == "SquaredExponential":
            return np.exp(-rho**2 / (2 * t[0] ** 2))
        return np.exp(-2 * np.sin(np.pi * rho / t[1]) ** 2 / t[0] ** 2)

    def __repr__(self):
        return f"RadialBasisFunction{{{self.constructor}}}"


def Matern52(theta=(1.0,)):
    return RadialBasisFunction(theta, "Matern52")


def Matern32(theta=(1.0,)):
    return RadialBasisFunction(theta, "Matern32")


def Matern12(theta=(1.0,)):
    return RadialBasisFunction(theta, "Matern12")


def SquaredExponential(theta=(1.0,)):
    return RadialBasisFunction(theta, "SquaredExponential")


def Periodic(theta=(1.0, 1.0)):
    return RadialBasisFunction(theta, "Periodic")


def eval_KXX(rbf, X, sigma_n2=1e-6):  # rbf.jl:161-178
    diff = X[:, :, None] - X[:, None, :]
    K = rbf(np.sqrt(np.sum(diff * diff, axis=0)))
    np.fill_diagonal(K, rbf(0.0))
    return K + sigma_n2 * np.eye(X.shape[1])


def eval_KxX(rbf, x, X):  # rbf.jl:180-191
    return rbf(np.sqrt(np.sum((x[:, None] - X) ** 2, axis=0)))


# ----------------------------------------------------------------------------------------------------
# decision_rules.jl:4-135
# ----------------------------------------------------------------------------------------------------
class DecisionRule:
    """decision_rules.jl:4-15. The partials the reference builds with ForwardDiff (l.23-34) live on the device."""

    def __init__(self, name, sigma_tol=1e-8):
        if name == "Random":
            raise NotImplementedError("RandomAcquisition (decision_rules.jl:129-135) draws from the host RNG and is outside the CUDA path")
        self.name = name
        self.rule_id = RULE_IDS[name]
        self.σtol = sigma_tol

    def __repr__(self):
        return f"DecisionRule{{{self.name}}}"


def EI(σtol=1e-8):  # decision_rules.jl:84-99
    return DecisionRule("EI", σtol)


def POI(σtol=1e-8):  # decision_rules.jl:101-115
    return DecisionRule("POI", σtol)


def LCB():  # decision_rules.jl:117-127
    return DecisionRule("LCB", 0.0)


def get_name(dr):
    return dr.name


# ----------------------------------------------------------------------------------------------------
# rbs.jl:30-222  Surrogate (host-side producer of the path's inputs)
# ----------------------------------------------------------------------------------------------------
class Surrogate:
    """rbs.jl:30-118: pre-allocated X, K, L, y, c with `observed` valid entries."""

    def __init__(self, ψ, X, y, capacity=DEFAULT_CAPACITY, decision_rule=None, σn2=1e-6):
        X = np.asarray(X, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64)
        assert len(y) <= capacity, "Capacity must be >= number of observations."  # rbs.jl:84
        d, N = X.shape
        self.ψ, self.σn2, self.g = ψ, σn2, decision_rule if decision_rule is not None else EI()
        self.capacity, self.observed = capacity, len(y)
        self.X = np.zeros((d, capacity), order="F")
        self.K = np.zeros((capacity, capacity), order="F")
        self.L = np.zeros((capacity, capacity), order="F")
        self.y = np.zeros(capacity)
        self.c = np.zeros(capacity)
        self.X[:, :N] = X
        self.y[:N] = y
        self._refactor()

    def _refactor(self):  # rbs.jl:90-101, 123-135
        N = self.observed
        self.K[:N, :N] = eval_KXX(self.ψ, self.X[:, :N], self.σn2)
        self.L[:N, :N] = cholesky(self.K[:N, :N], lower=True)
        L = self.L[:N, :N]
        self.c[:N] = solve_triangular(L.T, solve_triangular(L, self.y[:N], lower=True), lower=False)


def get_observed(s):
    return s.observed


def get_active_covariates(s):
    return s.X[:, : s.observed]


def get_active_observations(s):
    return s.y[: s.observed]


def get_observations(s):
    return s.y  # rbs.jl:22: the whole capacity-length, zero-padded vector (Q2)


def set_decision_rule(s, g):  # rbs.jl:75
    s.g = g


def set_kernel(s, kernel):  # rbs.jl:123-135
    s.ψ = kernel
    s._refactor()


def reset(s, X=None, y=None):
    """reset!(s::Surrogate, X, y) (rbs.jl:147-164) or reset!(fs::FantasySurrogate) (rbs.jl:476-480)."""
    if isinstance(s, FantasySurrogate):
        s.fantasies_observed = 0
        return
    X = np.asarray(X, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    N = X.shape[1]
    s.X[:, :N] = X
    s.y[:N] = y
    s.observed = len(y)
    s._refactor()


def condition(s, xnew, ynew):
    """condition!(s::Surrogate, x, y) (rbs.jl:214-222): rank-1 extension of K, L and a full coefficient re-solve."""
    if s.observed == s.capacity:
        raise RboError("surrogate is full (the reference's resize, rbs.jl:137-145, is not reproduced)")
    n = s.observed + 1
    s.X[:, n - 1] = xnew
    s.y[n - 1] = ynew
    s.observed = n
    kx = eval_KxX(s.ψ, np.asarray(xnew, dtype=np.float64), s.X[:, : n - 1])
    s.K[n - 1, n - 1] = s.ψ(0.0) + s.σn2
    s.K[n - 1, : n - 1] = kx
    s.K[: n - 1, n - 1] = kx
    L21 = solve_triangular(s.L[: n - 1, : n - 1], kx, lower=True) if n > 1 else kx
    s.L[n - 1, : n - 1] = L21
    rem = s.K[n - 1, n - 1] - L21 @ L21
    if not rem > 0:
        raise np.linalg.LinAlgError("PosDefException: update_cholesky! (rbs.jl:196)")
    s.L[n - 1, n - 1] = np.sqrt(rem)
    L = s.L[:n, :n]
    s.c[:n] = solve_triangular(L.T, solve_triangular(L, s.y[:n], lower=True), lower=False)
    return s


class FantasySurrogate:
    """rbs.jl:320-381. On the CUDA path only the base part (first `observed` rows/columns) is read; the fantasy
    rows are per-trajectory scratch that lives in shared memory on the device."""

    def __init__(self, s, horizon):
        self.h = horizon
        self.update(s)

    def update(self, s):  # rbs.jl:345-381 / 453-473 (update!)
        N, cap, h = s.observed, s.capacity, self.h
        self.ψ, self.σn2, self.g, self.capacity, self.observed = s.ψ, s.σn2, s.g, cap, N
        d = s.X.shape[0]
        self.X = np.zeros((d, cap + h + 1), order="F")
        self.X[:, :N] = s.X[:, :N]
        self.L = np.zeros((cap + h + 1, cap + h + 1), order="F")
        self.L[:N, :N] = s.L[:N, :N]
        self.y = np.zeros(cap + h + 1)
        self.y[:N] = s.y[:N]
        self.cs = [s.c[:N].copy()]
        self.fantasies_observed = 0


def update(fs, s):
    fs.update(s)


# ----------------------------------------------------------------------------------------------------
# trajectory.jl:17-134
# ----------------------------------------------------------------------------------------------------
class Trajectory:
    """trajectory.jl:17-37."""

    def __init__(self, base_surrogate, fantasy_surrogate, start, hypers, horizon):
        self.s, self.fs = base_surrogate, fantasy_surrogate
        self.x0 = np.asarray(start, dtype=np.float64).copy()
        self.θ = np.asarray(hypers, dtype=np.float64).copy()
        self.horizon = horizon
        self.observable = None
        self._engine = None


class TrajectoryParameters:
    """trajectory.jl:43-106, including the shape checks of l.58-62 (raised as AssertionError like Julia's @assert)."""

    def __init__(self, start, hypers, horizon, mc_iterations, use_low_discrepancy_sequence, spatial_lowerbounds,
                 spatial_upperbounds, rnstream_sequence=None, device=0):
        self.x0 = np.asarray(start, dtype=np.float64).copy()
        self.θ = np.asarray(hypers, dtype=np.float64).copy()
        self.horizon, self.mc_iters = int(horizon), int(mc_iterations)
        self.spatial_lbs = np.asarray(spatial_lowerbounds, dtype=np.float64).copy()
        self.spatial_ubs = np.asarray(spatial_upperbounds, dtype=np.float64).copy()
        n = len(self.x0)
        assert len(self.spatial_lbs) == n and len(self.spatial_ubs) == n, \
            "Lower and upper bounds must be the same length as the initial point"
        if rnstream_sequence is None:
            if use_low_discrepancy_sequence:
                rnstream_sequence = gen_low_discrepancy_sequence(self.mc_iters, n, self.horizon + 1, device=device)
            else:
                rnstream_sequence = np.asfortranarray(np.random.randn(self.mc_iters, n + 1, self.horizon + 1))
        rn = np.asfortranarray(rnstream_sequence, dtype=np.float64)
        assert rn.shape[1] == n + 1 and rn.shape[2] <= self.horizon + 1, \
            "Random number stream must have d + 1 rows and h + 1 columns for each sample"
        assert rn.shape[0] == self.mc_iters, f"Random number stream must have at least mc_iters ({self.mc_iters}) samples"
        self.rnstream_sequence = rn


def get_spatial_bounds(tp):
    return tp.spatial_lbs, tp.spatial_ubs


def get_starting_point(tp):
    return tp.x0.copy()


def set_starting_point(tp, x):
    tp.x0[:] = x


def get_hyperparameters(tp):
    return tp.θ.copy()


class ExpectedTrajectoryOutput:
    """trajectory.jl:112-134."""

    def __init__(self, μxθ, σ_μxθ, grad_μx=None, σ_grad_μx=None, grad_μθ=None, σ_grad_μθ=None, summary=None):
        self.μxθ, self.σ_μxθ = μxθ, σ_μxθ
        self.grad_μx, self.σ_grad_μx, self.grad_μθ, self.σ_grad_μθ = grad_μx, σ_grad_μx, grad_μθ, σ_grad_μθ
        self.summary = summary


def mean(eto):
    return eto.μxθ


def std(eto):
    return eto.σ_μxθ


def gradient(eto, wrt_hypers=False):
    return eto.grad_μθ if wrt_hypers else eto.grad_μx


def std_gradient(eto, wrt_hypers=False):
    return eto.σ_grad_μθ if wrt_hypers else eto.σ_grad_μx


# ----------------------------------------------------------------------------------------------------
# utils.jl generators (device implementations behind the ABI)
# ----------------------------------------------------------------------------------------------------
_shared_handles = {}


def _handle(device=0):
    if device not in _shared_handles:
        _shared_handles[device] = Handle(device)
    return _shared_handles[device]


def gen_uniform(samples, dim=1, device=0):  # utils.jl:4-13
    h = _handle(device)
    out = np.zeros((dim, samples), order="F")
    h.check(h.lib.rbo_sobol_uniform(h.h, dim, samples, dptr(out)))
    return out


def gen_low_discrepancy_sequence(samples, dim, horizon, device=0):
    """utils.jl:65-74, generated on the device: returns samples x (dim+1) x horizon (column-major)."""
    h = Handle(device)
    try:
        # the generator needs d; a one-point dummy surrogate provides it without touching the path's state
        X = np.zeros((dim, 1), order="F"); L = np.ones((1, 1), order="F"); y = np.zeros(1); c = np.zeros(1); kt = np.ones(1)
        h.check(h.lib.rbo_set_surrogate(h.h, dim, 1, dptr(X), dim, dptr(L), 1, dptr(y), dptr(c), 1e-6, 2, dptr(kt), 1, 0, 1e-8))
        h.check(h.lib.rbo_generate_normals(h.h, samples, horizon, 0, samples))
        out = np.zeros((samples, dim + 1, horizon), order="F")
        h.check(h.lib.rbo_get_normals(h.h, dptr(out)))
        return out
    finally:
        h.close()


def generate_initial_guesses(N, lbs, ubs, device=0):  # utils.jl:145-153
    lbs = np.asarray(lbs, dtype=np.float64); ubs = np.asarray(ubs, dtype=np.float64)
    d = len(lbs)
    h = _handle(device)
    out = np.zeros((d, N + 2), order="F")
    h.check(h.lib.rbo_generate_initial_guesses(h.h, N, d, dptr(lbs), dptr(ubs), dptr(out)))
    return out


class ExperimentSetup:
    """utils.jl:174-194."""

    def __init__(self, tp, number_of_starts, device=0):
        lbs, ubs = get_spatial_bounds(tp)
        self.tp = tp
        self.inner_solve_xstarts = generate_initial_guesses(number_of_starts, lbs, ubs, device=device)
        self.resolutions = np.zeros(tp.mc_iters)
        self.spatial_gradients_container = np.zeros((len(tp.x0), tp.mc_iters), order="F")
        self.hyperparameter_gradients_container = np.zeros((len(tp.θ), tp.mc_iters), order="F")


def get_container(es, symbol):  # utils.jl:196-206
    if symbol == "f":
        return es.resolutions
    if symbol == "grad_f":
        return es.spatial_gradients_container
    if symbol == "grad_hypers":
        return es.hyperparameter_gradients_container
    raise ValueError("Unknown symbol. Use either :f, :grad_f, or :grad_hypers")


def get_starts(es):
    return es.inner_solve_xstarts


# ----------------------------------------------------------------------------------------------------
# The engine: one handle per device with the inputs it currently holds
# ----------------------------------------------------------------------------------------------------
class RolloutEngine:
    """Marshals (Surrogate/FantasySurrogate, normals, starts) into a librbo handle; keeps them resident."""

    def __init__(self, device=0, stream=None):
        self.handle = Handle(device)
        self.lib = self.handle.lib
        if stream is not None:
            self.handle.check(self.lib.rbo_set_stream(self.handle.h, C.c_void_p(stream)))
        self.d = None
        self.m_count = 0

    def close(self):
        self.handle.close()

    def set_solver_opts(self, **kw):
        o = _lib.SolverOpts()
        self.lib.rbo_default_solver_opts(C.byref(o))
        for k, v in kw.items():
            setattr(o, k, v)
        self.handle.check(self.lib.rbo_set_solver_opts(self.handle.h, C.byref(o)))

    def set_tuning(self, large_n=None, large_n_slots=None, lpt=None, row_splits=None):
        """Execution knobs of rbo_set_tuning: force the large-n kernel variant / cap its start slots, longest-first hand-out,
        cap the row splits of the Gram reductions (1..4, 0 = default)."""
        if large_n is not None:
            self.handle.check(self.lib.rbo_set_tuning(self.handle.h, 1, int(bool(large_n))))
        if large_n_slots is not None:
            self.handle.check(self.lib.rbo_set_tuning(self.handle.h, 2, int(large_n_slots)))
        if lpt is not None:
            self.handle.check(self.lib.rbo_set_tuning(self.handle.h, 3, int(bool(lpt))))
        if row_splits is not None:
            self.handle.check(self.lib.rbo_set_tuning(self.handle.h, 4, int(row_splits)))

    def set_htol(self, htol):
        self.handle.check(self.lib.rbo_set_htol(self.handle.h, float(htol)))

    def set_surrogate(self, fs):
        """fs: FantasySurrogate or Surrogate. Reads X[:,1:N], L[1:N,1:N], y[1:N], coefficients (rbs.jl:345-381)."""
        N = fs.observed
        d = fs.X.shape[0]
        c = fs.cs[0] if isinstance(fs, FantasySurrogate) else fs.c[:N]
        X = np.asfortranarray(fs.X)
        L = np.asfortranarray(fs.L)
        y = np.ascontiguousarray(fs.y[:N])
        c = np.ascontiguousarray(c, dtype=np.float64)
        kt = np.ascontiguousarray(fs.ψ.θ, dtype=np.float64)
        self.handle.check(self.lib.rbo_set_surrogate(self.handle.h, d, N, dptr(X), X.shape[0], dptr(L), L.shape[0], dptr(y), dptr(c),
                                                     fs.σn2, fs.ψ.kernel_id, dptr(kt), len(kt), fs.g.rule_id, fs.g.σtol))
        self.d = d

    def condition(self, xnew, ynew):
        """condition!(s::Surrogate, x, y) (rbs.jl:214-222) on the device-resident surrogate (rbo_condition)."""
        x = np.ascontiguousarray(xnew, dtype=np.float64)
        self.handle.check(self.lib.rbo_condition(self.handle.h, dptr(x), float(ynew)))

    def get_surrogate(self):
        """The resident surrogate: X (d x N), y, c = K^-1 y."""
        n = C.c_int()
        self.handle.check(self.lib.rbo_get_surrogate(self.handle.h, C.byref(n), None, 0, None, None))
        X = np.zeros((self.d, n.value), order="F"); y = np.zeros(n.value); c = np.zeros(n.value)
        self.handle.check(self.lib.rbo_get_surrogate(self.handle.h, C.byref(n), dptr(X), self.d, dptr(y), dptr(c)))
        return X, y, c

    def set_normals(self, rn, m_begin=0, m_count=None):
        rn = np.asfortranarray(rn, dtype=np.float64)
        M = rn.shape[0]
        m_count = M - m_begin if m_count is None else m_count
        self.handle.check(self.lib.rbo_set_normals(self.handle.h, dptr(rn), M, rn.shape[2], m_begin, m_count))
        self.m_count = m_count

    def generate_normals(self, M_total, hp1, m_begin=0, m_count=None):
        m_count = M_total - m_begin if m_count is None else m_count
        self.handle.check(self.lib.rbo_generate_normals(self.handle.h, M_total, hp1, m_begin, m_count))
        self.m_count = m_count

    def get_normals(self, hp1):
        out = np.zeros((self.m_count, self.d + 1, hp1), order="F")
        self.handle.check(self.lib.rbo_get_normals(self.handle.h, dptr(out)))
        return out

    def set_quadrature(self, nodes, weights):
        """nodes, weights: depth x M (column m = nodes[indices[m]] of rollout.jl:431-432)."""
        nodes = np.asfortranarray(nodes, dtype=np.float64); weights = np.asfortranarray(weights, dtype=np.float64)
        if nodes.shape != weights.shape or nodes.ndim != 2:
            raise ValueError("nodes and weights must both be depth x M")
        self.handle.check(self.lib.rbo_set_quadrature(self.handle.h, dptr(nodes), dptr(weights), nodes.shape[0], nodes.shape[1]))
        self.m_count = nodes.shape[1]

    def set_starts(self, starts):
        starts = np.asfortranarray(starts, dtype=np.float64)
        self.handle.check(self.lib.rbo_set_starts(self.handle.h, dptr(starts), starts.shape[1]))
        self.S = starts.shape[1]

    def rollout(self, x0, theta, lbs, ubs, horizon, fmini, values, grad_x=None, grad_theta=None, dual_dirs=None,
                x_forced=None, best_index=None, grad_case=None, status=None, gauss_hermite=False, tape_ex=False, replay=False,
                want_grad=None):
        x0 = np.ascontiguousarray(x0, dtype=np.float64); theta = np.ascontiguousarray(theta, dtype=np.float64)
        lbs = np.ascontiguousarray(lbs, dtype=np.float64); ubs = np.ascontiguousarray(ubs, dtype=np.float64)
        mode = 1 if (grad_x is not None and grad_theta is not None) else 0  # rollout.jl:319
        if want_grad is not None:
            mode = 1 if want_grad else 0
        flags = (1 if x_forced is not None else 0) | (2 if gauss_hermite else 0) | (4 if tape_ex else 0) | (8 if replay else 0)
        if dual_dirs is not None:
            dual_dirs = np.asfortranarray(dual_dirs, dtype=np.float64)
        if x_forced is not None:
            x_forced = np.asfortranarray(x_forced, dtype=np.float64)
        s = Summary()
        self.handle.check(self.lib.rbo_rollout(self.handle.h, dptr(x0), dptr(theta), len(theta), dptr(lbs), dptr(ubs), horizon, float(fmini),
                                               mode, flags, dptr(dual_dirs), dptr(x_forced), dptr(values), dptr(grad_x), dptr(grad_theta),
                                               iptr(best_index), iptr(grad_case), iptr(status), C.byref(s)))
        return s

    def rollout_batch(self, x0s, theta, lbs, ubs, horizon, fmini, values, grad_x=None, grad_theta=None, dual_dirs=None, status=None):
        """x0s: d x B; values: M x B; grad_x: d x M x B; grad_theta: ntheta x M x B (column-major)."""
        x0s = np.asfortranarray(x0s, dtype=np.float64); theta = np.ascontiguousarray(theta, dtype=np.float64)
        lbs = np.ascontiguousarray(lbs, dtype=np.float64); ubs = np.ascontiguousarray(ubs, dtype=np.float64)
        mode = 1 if (grad_x is not None and grad_theta is not None) else 0
        if dual_dirs is not None:
            dual_dirs = np.asfortranarray(dual_dirs, dtype=np.float64)
        s = Summary()
        self.handle.check(self.lib.rbo_rollout_batch(self.handle.h, dptr(x0s), x0s.shape[1], dptr(theta), len(theta), dptr(lbs), dptr(ubs), horizon,
                                                     float(fmini), mode, dptr(dual_dirs), dptr(values), dptr(grad_x), dptr(grad_theta), iptr(status),
                                                     C.byref(s)))
        return s

    def rollout_device(self, x0, theta, lbs, ubs, horizon, fmini, mode, dual_dirs_ptr=None, want_summary=False):
        x0 = np.ascontiguousarray(x0, dtype=np.float64); theta = np.ascontiguousarray(theta, dtype=np.float64)
        lbs = np.ascontiguousarray(lbs, dtype=np.float64); ubs = np.ascontiguousarray(ubs, dtype=np.float64)
        s = Summary() if want_summary else None
        self.handle.check(self.lib.rbo_rollout_device(self.handle.h, dptr(x0), dptr(theta), len(theta), dptr(lbs), dptr(ubs), horizon, float(fmini),
                                                      mode, 0, C.c_void_p(dual_dirs_ptr) if dual_dirs_ptr else None, None,
                                                      C.byref(s) if want_summary else None))
        return s

    def stochastic_solve_batch(self, x0s, theta, lbs, ubs, horizon, fmini, dual_dirs=None, optimizer=None, max_iterations=50,
                               use_eswavs=True, project=False):
        """rbo_stochastic_solve_batch: stochastic_solve (utils.jl:235-265) from every column of x0s (d x B) in one library call, all
        iterations on the device. `optimizer` (StandardSGA or an unused Adam; default Adam()) supplies the hyper-parameters only.
        project=True clamps x to [lbs, ubs] after every step. Returns a dict: x_final (d x B), n_iter, end_status (B each: SGA_MAXIT,
        SGA_ESWAVS, SGA_FAILED), fail (2 x B: first failing sample, its status), x_hist (d x max_iterations x B), mean_hist, std_hist
        (max_iterations x B), gmean_hist, gstd_hist (d x max_iterations x B; NaN past n_iter) and summary."""
        o = _sga_opts(Adam() if optimizer is None else optimizer, max_iterations, use_eswavs, project)
        x0s, theta, lbs, ubs, dual_dirs = _sga_arrays(x0s, theta, lbs, ubs, horizon, dual_dirs, self.d, self.m_count or None)
        d, B, T = x0s.shape[0], x0s.shape[1], int(max_iterations)
        r = dict(x_final=np.zeros((d, B), order="F"), n_iter=np.zeros(B, np.int32), end_status=np.zeros(B, np.int32),
                 fail=np.zeros((2, B), np.int32, order="F"), x_hist=np.zeros((d, T, B), order="F"), mean_hist=np.zeros((T, B), order="F"),
                 std_hist=np.zeros((T, B), order="F"), gmean_hist=np.zeros((d, T, B), order="F"), gstd_hist=np.zeros((d, T, B), order="F"))
        s = Summary()
        self.handle.check(self.lib.rbo_stochastic_solve_batch(
            self.handle.h, C.byref(o), dptr(x0s), B, dptr(theta), len(theta), dptr(lbs), dptr(ubs), int(horizon), float(fmini), dptr(dual_dirs),
            dptr(r["x_final"]), iptr(r["n_iter"]), iptr(r["end_status"]), iptr(r["fail"]), dptr(r["x_hist"]), dptr(r["mean_hist"]),
            dptr(r["std_hist"]), dptr(r["gmean_hist"]), dptr(r["gstd_hist"]), C.byref(s)))
        r["summary"] = s
        return r

    def tape(self, horizon, ntheta=1):
        M, d, S, hh = self.m_count, self.d, getattr(self, "S", 1), max(horizon, 1)
        r = dict(xs=np.zeros((d, horizon + 1, M), order="F"), ys=np.zeros((horizon + 1, M), order="F"),
                 gys=np.zeros((d, horizon + 1, M), order="F"), alphas=np.zeros((hh, M), order="F"),
                 n_evals=np.zeros((hh, M), np.int32, order="F"), start_status=np.zeros((S, hh, M), np.int32, order="F"),
                 start_iters=np.zeros((S, hh, M), np.int32, order="F"))
        self.handle.check(self.lib.rbo_get_tape(self.handle.h, dptr(r["xs"]), dptr(r["ys"]), dptr(r["gys"]), dptr(r["alphas"]),
                                                iptr(r["n_evals"]), iptr(r["start_status"]), iptr(r["start_iters"])))
        return r

    def tape_ex(self, horizon):
        """Extended tape (rbo_get_tape_ex) of the last rollout run with tape_ex=True."""
        M, d, hh = self.m_count, self.d, max(horizon, 1)
        r = dict(mu=np.zeros((hh, M), order="F"), sigma=np.zeros((hh, M), order="F"), dmu=np.zeros((d, hh, M), order="F"),
                 dsigma=np.zeros((d, hh, M), order="F"), Halpha=np.zeros((d, d, hh, M), order="F"))
        self.handle.check(self.lib.rbo_get_tape_ex(self.handle.h, dptr(r["mu"]), dptr(r["sigma"]), dptr(r["dmu"]), dptr(r["dsigma"]), dptr(r["Halpha"])))
        return r

    def multistart_base_solve(self, theta, lbs, ubs):
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        lbs = np.ascontiguousarray(lbs, dtype=np.float64); ubs = np.ascontiguousarray(ubs, dtype=np.float64)
        x = np.zeros(self.d)
        a = C.c_double()
        s = Summary()
        self.handle.check(self.lib.rbo_multistart_base_solve(self.handle.h, dptr(theta), len(theta), dptr(lbs), dptr(ubs), dptr(x), C.byref(a), C.byref(s)))
        return x, a.value, s

    def fp64_peak(self):
        t = C.c_double()
        self.handle.check(self.lib.rbo_fp64_peak(self.handle.h, C.byref(t)))
        return t.value

    def num_sms(self):
        return self.lib.rbo_num_sms(self.handle.h)

    def tr_step_batch(self, H, g, Delta):
        """Diagnostic: the kernel's exact trust-region step (DESIGN.md section 4) on B subproblems: H [B, n, n], g [B, n], Delta [B]
        -> (p [B, n], hit [B]); the counterpart of the oracle's tr_step."""
        H = np.ascontiguousarray(H, dtype=np.float64); g = np.ascontiguousarray(g, dtype=np.float64)
        Delta = np.ascontiguousarray(Delta, dtype=np.float64)
        B, n = g.shape
        if H.shape != (B, n, n) or Delta.shape != (B,):
            raise ValueError("tr_step_batch: H must be [B, n, n], g [B, n], Delta [B]")
        p = np.zeros((B, n)); hit = np.zeros(B, np.int32)
        self.handle.check(self.lib.rbo_tr_step_batch(self.handle.h, n, B, dptr(H), dptr(g), dptr(Delta), dptr(p), iptr(hit)))
        return p, hit.astype(bool)


def _mean_std_rows(A):
    """rollout.jl:328-337: Distributions.mean / std(..., mean=) -- corrected sample std per row."""
    A = np.atleast_2d(A)
    mu = A.mean(axis=1)
    sd = np.sqrt(((A - mu[:, None]) ** 2).sum(axis=1) / (A.shape[1] - 1)) if A.shape[1] > 1 else np.full(A.shape[0], np.nan)
    return mu, sd


def draw_dual_directions(values, best_index, d, h, rand=np.random.rand):
    """The rand(dim) draws of solve_dual_y (rollout.jl:133) in the reference's consumption order: samples in ascending order; only
    those whose gradient is the back-substitution of rollout.jl:253-276 (payoff > 0 and best step t >= 1); for each, j = t, t-1,
    .., 1 fills the direction of solve_index j-1. Returns d x h x M (zeros where the reference draws nothing)."""
    M = len(values)
    dd = np.zeros((d, max(h, 1), M), order="F")
    for m in range(M):
        t = int(best_index[m])
        if values[m] > 0.0 and t >= 1:       # case 3: fmini > best observation and the best step is a fantasy step
            for j in range(t, 0, -1):
                dd[:, j - 1, m] = rand(d)
    return dd


# what the reference throws where a trajectory ends with RBO_TRAJ_* status k (SURVEY.md section 5)
_TRAJ_ERRORS = {1: "PosDefException (rbs.jl:412)", 2: "DomainError (rbs.jl:528)", 3: "PosDefException (rbs.jl:537)",
                4: "ArgumentError: reducing over an empty collection (rbf_optim.jl:97)", 5: "SingularException (rollout.jl:188)"}


def simulate_trajectory_mc(T, tp, *, inner_solve_xstarts, resolutions, spatial_gradients_container=None,
                           hyperparameter_gradients_container=None, dual_directions=None, device=0, keep_resident=False, rng_rand=None):
    """simulate_trajectory_mc (rollout.jl:279-340) on the GPU.

    Fills `resolutions[m]` and the gradient containers in place and returns ExpectedTrajectoryOutput, exactly
    like the reference. `dual_directions` (d x h x M) stands for the `rand(dim)` draws of rollout.jl:133 (Q5); by
    default they are drawn from the host RNG (`rng_rand`, default numpy's global one) in the reference's own
    data-dependent consumption order through a two-phase call (see draw_dual_directions).
    Raises RboError if a trajectory failed where the reference would have thrown (first failing sample).
    """
    d, h, M = len(tp.x0), tp.horizon, tp.mc_iters
    T.x0[:] = tp.x0  # set_start! (rollout.jl:287)
    eng = T._engine if (keep_resident and T._engine is not None) else RolloutEngine(device)
    try:
        if not (keep_resident and T._engine is not None):
            eng.set_surrogate(T.fs)
            eng.set_normals(tp.rnstream_sequence)
            eng.set_starts(inner_solve_xstarts)
        want_grad = spatial_gradients_container is not None and hyperparameter_gradients_container is not None
        fmini = float(np.min(get_observations(T.s)))  # rollout.jl:109 (zero-padded capacity vector, Q2)
        status = np.zeros(M, np.int32)
        if want_grad and dual_directions is None and h > 0:
            # Two-phase call (rollout.jl:133, Q5): the reference draws rand(dim) inside solve_dual_y, i.e. only for the trajectories
            # whose gradient takes the back-substitution (case 3), t draws each (j = t, t-1, .., 1 -> solve_index j-1), in sample
            # order. Phase 1 computes values and best indices, the host replays exactly that consumption of its global RNG,
            # phase 2 replays the device-resident x-path (bitwise, no inner solves) with the gradient.
            best = np.zeros(M, np.int32)
            eng.rollout(tp.x0, tp.θ, tp.spatial_lbs, tp.spatial_ubs, h, fmini, resolutions, best_index=best, status=status, want_grad=False)
            dual_directions = draw_dual_directions(resolutions, best, d, h, rand=rng_rand if rng_rand is not None else np.random.rand)
            summary = eng.rollout(tp.x0, tp.θ, tp.spatial_lbs, tp.spatial_ubs, h, fmini, resolutions, spatial_gradients_container,
                                  hyperparameter_gradients_container, dual_dirs=dual_directions, status=status, replay=True)
        else:
            summary = eng.rollout(tp.x0, tp.θ, tp.spatial_lbs, tp.spatial_ubs, h, fmini, resolutions,
                                  spatial_gradients_container if want_grad else None,
                                  hyperparameter_gradients_container if want_grad else None,
                                  dual_dirs=dual_directions if want_grad else None, status=status)
    finally:
        if keep_resident:
            T._engine = eng
        else:
            eng.close()
    bad = np.nonzero(status)[0]
    if len(bad):
        raise RboError(f"sample {bad[0] + 1}: {_TRAJ_ERRORS.get(int(status[bad[0]]), 'error')}")
    μ, σ = _mean_std_rows(resolutions)
    if not want_grad:
        return ExpectedTrajectoryOutput(float(μ[0]), float(σ[0]), summary=summary)
    gx, sgx = _mean_std_rows(spatial_gradients_container)
    gt, sgt = _mean_std_rows(hyperparameter_gradients_container)
    return ExpectedTrajectoryOutput(float(μ[0]), float(σ[0]), gx, sgx, gt, sgt, summary=summary)


def generate_indices(num_nodes, max_depth):
    """generate_indices (utils.jl:217-221): all num_nodes^max_depth index vectors (1-based), first position fastest."""
    grids = np.meshgrid(*([np.arange(1, num_nodes + 1)] * max_depth), indexing="ij")
    return [list(map(int, v)) for v in np.stack([g.ravel(order="F") for g in grids], axis=1)]


def gausshermite(n):
    """Nodes and weights of the n-point Gauss-Hermite rule (weight exp(-x^2)), what the reference's callers pass as
    `nodes`, `weights` (observables.jl:54-72 uses the sqrt(2) / sqrt(pi) change of variables of that rule)."""
    return np.polynomial.hermite.hermgauss(n)


def simulate_trajectory_ghq(T, tp, *, inner_solve_xstarts, resolutions, nodes, weights, indices,
                            spatial_gradients_container=None, hyperparameter_gradients_container=None,
                            dual_directions=None, device=0):
    """simulate_trajectory_ghq (rollout.jl:409-467) on the GPU: one trajectory per entry of `indices` (1-based index
    vectors of length depth >= horizon + 1), driven by the GaussHermiteObservable (observables.jl:32-81,157)."""
    d, h, M = len(tp.x0), tp.horizon, len(indices)
    T.x0[:] = tp.x0  # set_start! (rollout.jl:422)
    nodes = np.asarray(nodes, dtype=np.float64); weights = np.asarray(weights, dtype=np.float64)
    idx = np.asarray(indices, dtype=np.int64) - 1  # M x depth
    if idx.ndim != 2 or idx.min() < 0 or idx.max() >= len(nodes):
        raise RboError("BoundsError: indices must be equal-length vectors of 1-based node indices")  # nodes[indices[i]]
    if idx.shape[1] < h + 1:
        raise RboError("AssertionError: Maximum invocations have been used")  # observables.jl:55
    if len(resolutions) < M:
        raise RboError("BoundsError: resolutions shorter than indices")
    want_grad = spatial_gradients_container is not None and hyperparameter_gradients_container is not None
    vals = np.zeros(M)
    gx = np.zeros((d, M), order="F") if want_grad else None
    gt = np.zeros((len(tp.θ), M), order="F") if want_grad else None
    status = np.zeros(M, np.int32)
    eng = RolloutEngine(device)
    try:
        eng.set_surrogate(T.fs)
        eng.set_quadrature(nodes[idx].T, weights[idx].T)
        eng.set_starts(inner_solve_xstarts)
        if want_grad and dual_directions is None and h > 0:
            dual_directions = np.asfortranarray(np.random.rand(d, h, M))
        fmini = float(np.min(get_observations(T.s)))  # rollout.jl:109
        summary = eng.rollout(tp.x0, tp.θ, tp.spatial_lbs, tp.spatial_ubs, h, fmini, vals, gx, gt,
                              dual_dirs=dual_directions if want_grad else None, status=status, gauss_hermite=True)
    finally:
        eng.close()
    bad = np.nonzero(status)[0]
    if len(bad):
        names = {1: "PosDefException (rbs.jl:412)", 2: "DomainError (rbs.jl:528)",
                 4: "ArgumentError: reducing over an empty collection (rbf_optim.jl:97)", 5: "SingularException (rollout.jl:188)"}
        raise RboError(f"sample {bad[0] + 1}: {names.get(int(status[bad[0]]), 'error')}")
    resolutions[:M] = vals  # rollout.jl:444; entries past length(indices) are left as they were
    μ, σ = _mean_std_rows(resolutions)  # rollout.jl:455-456 take the whole vector
    if not want_grad:
        return ExpectedTrajectoryOutput(float(μ[0]), float(σ[0]), summary=summary)
    spatial_gradients_container[:, :M] = gx
    hyperparameter_gradients_container[:, :M] = gt
    mgx, sgx = _mean_std_rows(spatial_gradients_container)
    mgt, sgt = _mean_std_rows(hyperparameter_gradients_container)
    return ExpectedTrajectoryOutput(float(μ[0]), float(σ[0]), mgx, sgx, mgt, sgt, summary=summary)


def simulate_trajectory_mc_batch(T, tp, x0s, *, inner_solve_xstarts, dual_directions=None, want_gradients=True, device=0):
    """simulate_trajectory_mc (rollout.jl:279-340) at every column of x0s (d x B) in ONE launch: what a serial loop
    `for x0 in eachcol(x0s); set_starting_point!(tp, x0); simulate_trajectory_mc(T, tp; ...)` computes (same normals for every
    starting point, as the shared TrajectoryParameters imply). Returns a list of ExpectedTrajectoryOutput, one per column."""
    x0s = np.asfortranarray(x0s, dtype=np.float64)
    d, h, M, B = len(tp.x0), tp.horizon, tp.mc_iters, x0s.shape[1]
    nth = len(tp.θ)
    vals = np.zeros((M, B), order="F")
    gx = np.zeros((d, M, B), order="F") if want_gradients else None
    gt = np.zeros((nth, M, B), order="F") if want_gradients else None
    status = np.zeros((M, B), np.int32, order="F")
    if want_gradients and dual_directions is None and h > 0:
        dual_directions = np.asfortranarray(np.random.rand(d, h, M))
    eng = RolloutEngine(device)
    try:
        eng.set_surrogate(T.fs)
        eng.set_normals(tp.rnstream_sequence)
        eng.set_starts(inner_solve_xstarts)
        fmini = float(np.min(get_observations(T.s)))
        summary = eng.rollout_batch(x0s, tp.θ, tp.spatial_lbs, tp.spatial_ubs, h, fmini, vals, gx, gt,
                                    dual_dirs=dual_directions if want_gradients else None, status=status)
    finally:
        eng.close()
    if np.any(status):
        b, m = np.argwhere(status.T != 0)[0]
        raise RboError(f"starting point {b + 1}, sample {m + 1}: trajectory failed with status {int(status[m, b])}")
    out = []
    for b in range(B):
        μ, σ = _mean_std_rows(vals[:, b])
        if not want_gradients:
            out.append(ExpectedTrajectoryOutput(float(μ[0]), float(σ[0]), summary=summary))
            continue
        mgx, sgx = _mean_std_rows(gx[:, :, b])
        mgt, sgt = _mean_std_rows(gt[:, :, b])
        out.append(ExpectedTrajectoryOutput(float(μ[0]), float(σ[0]), mgx, sgx, mgt, sgt, summary=summary))
    return out


def multistart_base_solve(surrogate, xfinal, *, spatial_lbs, spatial_ubs, guesses, θfixed, device=0):
    """multistart_base_solve!(::Surrogate, xfinal; ...) (rbf_optim.jl:103-134): writes the argmax into xfinal."""
    eng = RolloutEngine(device)
    try:
        eng.set_surrogate(surrogate)
        eng.set_starts(guesses)
        x, alpha, summary = eng.multistart_base_solve(θfixed, spatial_lbs, spatial_ubs)
    finally:
        eng.close()
    xfinal[:] = x
    return alpha, summary


# ----------------------------------------------------------------------------------------------------
# optimizers.jl:6-75 and the SGA loop of utils.jl:235-265
# ----------------------------------------------------------------------------------------------------
class StandardSGA:
    def __init__(self, η=0.01):
        self.η = η


class Adam:
    def __init__(self, η=0.001, β1=0.9, β2=0.999, ε=1e-8, t=0):
        self.η, self.β1, self.β2, self.ε, self.t = η, β1, β2, ε, t
        self.m, self.v = [], []  # the reference keeps the whole history (optimizers.jl:30-31, 60-63)


def update_optimizer(optimizer, x, grad_f):
    """update!(optimizer; x, grad_f) (optimizers.jl:16-22, 48-75): ascent step, in place on x."""
    grad_f = np.asarray(grad_f, dtype=np.float64)
    if isinstance(optimizer, StandardSGA):
        x += optimizer.η * grad_f
        return x
    if len(optimizer.m) == 0 and len(optimizer.v) == 0:
        optimizer.m.append(np.zeros(len(grad_f)))
        optimizer.v.append(np.zeros(len(grad_f)))
    optimizer.t += 1
    optimizer.m.append(optimizer.β1 * optimizer.m[-1] + (1 - optimizer.β1) * grad_f)
    optimizer.v.append(optimizer.β2 * optimizer.v[-1] + (1 - optimizer.β2) * grad_f**2)
    mhat = optimizer.m[-1] / (1 - optimizer.β1**optimizer.t)
    vhat = optimizer.v[-1] / (1 - optimizer.β2**optimizer.t)
    x += optimizer.η * mhat / (np.sqrt(vhat) + optimizer.ε)
    return x


def early_stopping_without_a_validation_set(grad_f, var_grad_f, sample_size):  # utils.jl:114-123
    dim = len(grad_f)
    ratio = np.sum(grad_f**2 / var_grad_f)
    return (1.0 - (sample_size / dim) * ratio) > 0.0


eswavs = early_stopping_without_a_validation_set


def stochastic_solve(optimizer, T, tp, es, start, max_iterations=50, use_eswavs=True, dual_directions=None, device=0):
    """utils.jl:235-265 with the undefined `simulate_adjoint_trajectory` replaced by simulate_trajectory_mc
    (the only live estimator at HEAD). The surrogate, normals and starts stay resident on the device across
    iterations; only x0 changes (common random numbers, SURVEY.md 3.5). Returns (x, history)."""
    tpc = TrajectoryParameters(np.array(start, dtype=np.float64), tp.θ, tp.horizon, tp.mc_iters, False, tp.spatial_lbs,
                               tp.spatial_ubs, rnstream_sequence=tp.rnstream_sequence)
    history = []
    T._engine = None
    try:
        for _ in range(max_iterations):
            eto = simulate_trajectory_mc(T, tpc, inner_solve_xstarts=get_starts(es), resolutions=get_container(es, "f"),
                                         spatial_gradients_container=get_container(es, "grad_f"),
                                         hyperparameter_gradients_container=get_container(es, "grad_hypers"),
                                         dual_directions=dual_directions, device=device, keep_resident=True)
            history.append((tpc.x0.copy(), mean(eto), gradient(eto).copy()))
            if use_eswavs and eswavs(gradient(eto), std_gradient(eto) ** 2, tp.mc_iters):
                break
            update_optimizer(optimizer, tpc.x0, gradient(eto))
    finally:
        if T._engine is not None:
            T._engine.close()
            T._engine = None
    return tpc.x0.copy(), history


# ----------------------------------------------------------------------------------------------------
# The SGA loop from a batch of restarts on the device (rbo_stochastic_solve_batch)
# ----------------------------------------------------------------------------------------------------
SGA_MAXIT, SGA_ESWAVS, SGA_FAILED = 0, 1, 2  # RBO_SGA_*: why a restart ended


def _sga_opts(optimizer, max_iterations, use_eswavs, project):
    """rbo_sga_opts from a StandardSGA or Adam that supplies the hyper-parameters only: every restart starts from a fresh optimiser
    state, so an Adam that has already stepped (t > 0) is rejected rather than silently reset."""
    o = _lib.SgaOpts()
    o.max_iterations, o.use_eswavs, o.project = int(max_iterations), int(bool(use_eswavs)), int(bool(project))
    if isinstance(optimizer, Adam):
        if optimizer.t != 0 or len(optimizer.m) or len(optimizer.v):
            raise ValueError(f"stochastic_solve_batch: the Adam optimiser has already taken {optimizer.t} steps; every restart starts "
                             "from a fresh state, so pass an unused Adam")
        o.optimizer, o.eta, o.beta1, o.beta2, o.eps = 1, optimizer.η, optimizer.β1, optimizer.β2, optimizer.ε
    elif isinstance(optimizer, StandardSGA):
        o.optimizer, o.eta, o.beta1, o.beta2, o.eps = 0, optimizer.η, 0.0, 0.0, 0.0
    else:
        raise TypeError(f"stochastic_solve_batch: optimizer must be StandardSGA or Adam, not {type(optimizer).__name__}")
    if o.max_iterations < 1:
        raise ValueError(f"stochastic_solve_batch: max_iterations = {o.max_iterations} < 1")
    if not o.eta > 0:
        raise ValueError(f"stochastic_solve_batch: step size η = {o.eta} must be > 0")
    return o


def _sga_arrays(x0s, theta, lbs, ubs, horizon, dual_dirs, d=None, M=None):
    """Shape checks of rbo_stochastic_solve_batch's host arrays (d, M: the engine's input dimension and samples, when known)."""
    x0s = np.asfortranarray(x0s, dtype=np.float64)
    if x0s.ndim != 2 or x0s.shape[1] < 1:
        raise ValueError(f"stochastic_solve_batch: the starting points must be a d x B matrix with B >= 1, got shape {x0s.shape}")
    if d is not None and x0s.shape[0] != d:
        raise ValueError(f"stochastic_solve_batch: starting points of dimension {x0s.shape[0]}, the surrogate has d = {d}")
    d = x0s.shape[0]
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    lbs = np.ascontiguousarray(lbs, dtype=np.float64); ubs = np.ascontiguousarray(ubs, dtype=np.float64)
    if lbs.shape != (d,) or ubs.shape != (d,):
        raise ValueError(f"stochastic_solve_batch: bounds of shapes {lbs.shape}, {ubs.shape}; expected ({d},)")
    if theta.ndim != 1 or len(theta) < 1:
        raise ValueError("stochastic_solve_batch: theta must be a non-empty vector")
    if dual_dirs is not None:
        dual_dirs = np.asfortranarray(dual_dirs, dtype=np.float64)
        if dual_dirs.ndim != 3 or dual_dirs.shape[:2] != (d, horizon) or (M is not None and dual_dirs.shape[2] != M):
            raise ValueError(f"stochastic_solve_batch: dual directions of shape {dual_dirs.shape}; expected ({d}, {horizon}, M = {M})")
    return x0s, theta, lbs, ubs, dual_dirs


def stochastic_solve_batch(optimizer, T, tp, es, starts, max_iterations=50, use_eswavs=True, dual_directions=None, device=0):
    """stochastic_solve (utils.jl:235-265) from every column of `starts` (d x B) at once, on the device: one library call, one
    synchronisation. Each restart runs the loop of `stochastic_solve` with its own optimiser state (from `optimizer`'s
    hyper-parameters; an Adam with t > 0 is rejected) and its own ESWAVS stop, on the same normals (common random numbers).

    `dual_directions` (d x h x M) is shared by every restart and iteration. When None, ONE rand(d, h, M) buffer is drawn from numpy's
    global RNG and reused, as simulate_trajectory_mc_batch does: this is not the reference's per-iteration rand(dim) consumption (Q5),
    which `stochastic_solve` reproduces through its two-phase call.

    Returns (X_final, histories): X_final is d x B (each restart's iterate after its last step, or the x at which it stopped);
    histories[b] lists the (x, mean, grad) tuples of `stochastic_solve` for restart b. Raises RboError naming the restart and the
    sample when a trajectory failed where the reference would have thrown."""
    d, h, M = len(tp.x0), tp.horizon, tp.mc_iters
    _sga_opts(optimizer, max_iterations, use_eswavs, False)
    starts = _sga_arrays(starts, tp.θ, tp.spatial_lbs, tp.spatial_ubs, h, dual_directions, d, M)[0]
    if dual_directions is None and h > 0:
        dual_directions = np.asfortranarray(np.random.rand(d, h, M))
    eng = RolloutEngine(device)
    try:
        eng.set_surrogate(T.fs)
        eng.set_normals(tp.rnstream_sequence)
        eng.set_starts(get_starts(es))
        fmini = float(np.min(get_observations(T.s)))  # rollout.jl:109
        r = eng.stochastic_solve_batch(starts, tp.θ, tp.spatial_lbs, tp.spatial_ubs, h, fmini, dual_dirs=dual_directions, optimizer=optimizer,
                                       max_iterations=max_iterations, use_eswavs=use_eswavs)
    finally:
        eng.close()
    failed = np.nonzero(r["end_status"] == SGA_FAILED)[0]
    if len(failed):
        b = int(failed[0])
        m, code = int(r["fail"][0, b]), int(r["fail"][1, b])
        raise RboError(f"restart {b + 1}, sample {m + 1}: {_TRAJ_ERRORS.get(code, 'error')}")
    histories = [[(r["x_hist"][:, k, b].copy(), float(r["mean_hist"][k, b]), r["gmean_hist"][:, k, b].copy()) for k in range(int(r["n_iter"][b]))]
                 for b in range(starts.shape[1])]
    return r["x_final"], histories
