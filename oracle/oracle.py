"""ctypes binding of oracle/librbo_oracle.so -- the CPU restatement of the reference path.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs. The product package never imports this module.
PARITY UNPINNED (see rbo_oracle.h): no Julia, no reference golden vectors.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

KERNEL_IDS = {"matern12": 0, "matern32": 1, "matern52": 2, "se": 3, "periodic": 4}
RULE_IDS = {"EI": 0, "POI": 1, "LCB": 2}
FLAG_TEACHER_FORCED, FLAG_FAST_PERTURB, FLAG_FACTORED, FLAG_GAUSS_HERMITE = 1, 2, 4, 8


class SolverOpts(C.Structure):
    _fields_ = [("maxit", C.c_int), ("maxtry", C.c_int), ("gtol", C.c_double), ("xtol", C.c_double),
                ("pred_tol", C.c_double), ("eta", C.c_double), ("delta0_box", C.c_double),
                ("delta0_ell", C.c_double), ("stol", C.c_double)]


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class Problem(C.Structure):
    _fields_ = [("d", C.c_int), ("N", C.c_int), ("h", C.c_int), ("M", C.c_int), ("S", C.c_int),
                ("kernel_id", C.c_int), ("nktheta", C.c_int), ("ktheta", C.c_double * 4),
                ("rule_id", C.c_int), ("sigma_tol", C.c_double), ("sigma_n2", C.c_double),
                ("X", _dp), ("ldX", C.c_int), ("L", _dp), ("ldL", C.c_int), ("y", _dp), ("c", _dp),
                ("x0", _dp), ("theta", _dp), ("ntheta", C.c_int), ("lbs", _dp), ("ubs", _dp),
                ("fmini", C.c_double), ("rn", _dp), ("rn_hp1", C.c_int), ("starts", _dp),
                ("dual_dirs", _dp), ("x_forced", _dp), ("mode", C.c_int), ("flags", C.c_int),
                ("htol", C.c_double), ("solver", SolverOpts), ("nthreads", C.c_int), ("gh_nodes", _dp), ("gh_weights", _dp)]


class Outputs(C.Structure):
    _fields_ = [("values", _dp), ("grad_x", _dp), ("grad_theta", _dp), ("best_index", _ip), ("grad_case", _ip),
                ("status", _ip), ("xs", _dp), ("ys", _dp), ("gys", _dp), ("alphas", _dp), ("n_evals", _ip),
                ("start_status", _ip), ("start_iters", _ip), ("t_mu", _dp), ("t_sigma", _dp), ("t_dmu", _dp), ("t_dsigma", _dp),
                ("t_Halpha", _dp)]


def build(force=False):
    so = os.path.join(_HERE, "librbo_oracle.so")
    src = [os.path.join(_HERE, f) for f in ("rbo_oracle.cpp", "rbo_oracle.h", "sobol_joe_kuo.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.orc_rollout.argtypes = [C.POINTER(Problem), C.POINTER(Outputs)]
        _LIB.orc_rollout.restype = C.c_int
        _LIB.orc_default_solver_opts.argtypes = [C.POINTER(SolverOpts)]
        _LIB.orc_eval_point.argtypes = [C.POINTER(Problem), C.c_int, _dp, _dp, _dp, _dp]
        _LIB.orc_multistart_solve.argtypes = [C.POINTER(Problem), C.c_int, _dp, _dp, _dp, _dp, _ip, _ip, _dp, _dp]
        _LIB.orc_fit_surrogate.argtypes = [C.c_int, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp, C.c_double, _dp, _dp, _dp]
        _LIB.orc_sobol_uniform.argtypes = [C.c_int, C.c_int, _dp]
        _LIB.orc_sobol_uint32.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_uint)]
        _LIB.orc_gen_low_discrepancy_sequence.argtypes = [C.c_int, C.c_int, C.c_int, _dp]
        _LIB.orc_generate_initial_guesses.argtypes = [C.c_int, C.c_int, _dp, _dp, _dp]
        _LIB.orc_kernel_scalars.argtypes = [C.c_int, _dp, C.c_double, _dp]
        _LIB.orc_mean_std.argtypes = [_dp, C.c_int, C.c_int, _dp, _dp]
        _LIB.orc_rule_partials.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _dp]
        _LIB.orc_tr_step.argtypes = [C.c_int, _dp, _dp, C.c_double, _dp]
        _LIB.orc_tr_step.restype = C.c_int
    return _LIB


def _f(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def default_solver_opts():
    o = SolverOpts()
    lib().orc_default_solver_opts(C.byref(o))
    return o


def fit_surrogate(X, y, kernel="matern52", ktheta=(1.0,), sigma_n2=1e-6):
    """rbs.jl:77-118. X is d x N (columns are points). Returns K, L (N x N numpy, L lower), c."""
    X = np.asfortranarray(X, dtype=np.float64)
    d, N = X.shape
    y = _f(y)
    kt = _f(list(ktheta) + [0.0] * (4 - len(ktheta)))
    K = np.zeros((N, N), order="F")
    L = np.zeros((N, N), order="F")
    c = np.zeros(N)
    rc = lib().orc_fit_surrogate(d, N, _ptr(X), d, _ptr(y), KERNEL_IDS[kernel], _ptr(kt), sigma_n2, _ptr(K), _ptr(L), _ptr(c))
    if rc:
        raise np.linalg.LinAlgError("kernel matrix not positive definite")
    return K, L, c


class OracleProblem:
    """Keeps the numpy buffers alive next to the C struct."""

    def __init__(self, X, L, y, c, x0, lbs, ubs, rn, starts, *, h, kernel="matern52", ktheta=(1.0,), rule="EI",
                 theta=(0.0,), sigma_n2=1e-6, sigma_tol=1e-8, fmini=None, mode=1, flags=0, dual_dirs=None,
                 x_forced=None, htol=1e-4, nthreads=0, solver=None, gh_nodes=None, gh_weights=None):
        self.X = np.asfortranarray(X, dtype=np.float64)
        self.d, self.N = self.X.shape
        self.L = np.asfortranarray(L, dtype=np.float64)
        self.y, self.c, self.x0 = _f(y), _f(c), _f(x0)
        self.lbs, self.ubs, self.theta = _f(lbs), _f(ubs), _f(theta)
        self.rn = np.asfortranarray(rn, dtype=np.float64)  # M x (d+1) x hp1
        self.M = self.rn.shape[0]
        assert self.rn.shape[1] == self.d + 1 and self.rn.shape[2] >= h + 1
        self.starts = np.asfortranarray(starts, dtype=np.float64)  # d x S
        self.S = self.starts.shape[1]
        self.h = h
        self.dual_dirs = None if dual_dirs is None else np.asfortranarray(dual_dirs, dtype=np.float64)  # d x h x M
        self.x_forced = None if x_forced is None else np.asfortranarray(x_forced, dtype=np.float64)  # d x h x M
        p = Problem()
        p.d, p.N, p.h, p.M, p.S = self.d, self.N, h, self.M, self.S
        p.kernel_id = KERNEL_IDS[kernel]
        p.nktheta = len(ktheta)
        for i, t in enumerate(ktheta):
            p.ktheta[i] = t
        p.rule_id = RULE_IDS[rule]
        p.sigma_tol, p.sigma_n2 = sigma_tol, sigma_n2
        p.X, p.ldX, p.L, p.ldL = _ptr(self.X), self.d, _ptr(self.L), self.L.shape[0]
        p.y, p.c, p.x0 = _ptr(self.y), _ptr(self.c), _ptr(self.x0)
        p.theta, p.ntheta, p.lbs, p.ubs = _ptr(self.theta), len(self.theta), _ptr(self.lbs), _ptr(self.ubs)
        p.fmini = float(np.min(self.y)) if fmini is None else fmini
        p.rn, p.rn_hp1, p.starts = _ptr(self.rn), self.rn.shape[2], _ptr(self.starts)
        p.dual_dirs, p.x_forced = _ptr(self.dual_dirs), _ptr(self.x_forced)
        p.mode, p.flags, p.htol, p.nthreads = mode, flags, htol, nthreads
        if self.x_forced is not None:  # a given x-path is followed: no inner solve runs
            p.flags |= FLAG_TEACHER_FORCED
            assert self.x_forced.shape == (self.d, h, self.M)
        self.gh_nodes = None if gh_nodes is None else np.asfortranarray(gh_nodes, dtype=np.float64)      # (h+1) x M
        self.gh_weights = None if gh_weights is None else np.asfortranarray(gh_weights, dtype=np.float64)
        p.gh_nodes, p.gh_weights = _ptr(self.gh_nodes), _ptr(self.gh_weights)
        if self.gh_nodes is not None:
            p.flags |= FLAG_GAUSS_HERMITE
            assert self.gh_nodes.shape == (h + 1, self.M)
        p.solver = solver if solver is not None else default_solver_opts()
        self.p = p

    def rollout(self, tape=True):
        d, h, M, S, nth = self.d, self.h, self.M, self.S, len(self.theta)
        r = {
            "values": np.zeros(M), "grad_x": np.zeros((d, M), order="F"), "grad_theta": np.zeros((nth, M), order="F"),
            "best_index": np.zeros(M, np.int32), "grad_case": np.zeros(M, np.int32), "status": np.zeros(M, np.int32),
        }
        if tape:
            r.update(xs=np.zeros((d, h + 1, M), order="F"), ys=np.zeros((h + 1, M), order="F"),
                     gys=np.zeros((d, h + 1, M), order="F"), alphas=np.zeros((max(h, 1), M), order="F"),
                     n_evals=np.zeros((max(h, 1), M), np.int32, order="F"),
                     start_status=np.zeros((S, max(h, 1), M), np.int32, order="F"),
                     start_iters=np.zeros((S, max(h, 1), M), np.int32, order="F"),
                     t_mu=np.zeros((max(h, 1), M), order="F"), t_sigma=np.zeros((max(h, 1), M), order="F"),
                     t_dmu=np.zeros((d, max(h, 1), M), order="F"), t_dsigma=np.zeros((d, max(h, 1), M), order="F"),
                     t_Halpha=np.zeros((d, d, max(h, 1), M), order="F"))
        o = Outputs()
        for k, v in r.items():
            setattr(o, k, v.ctypes.data_as(_ip if v.dtype == np.int32 else _dp))
        rc = lib().orc_rollout(C.byref(self.p), C.byref(o))
        assert rc == 0
        return r

    def eval_point(self, x, Xf=None, yf=None):
        d = self.d
        nf = 0 if Xf is None else np.asarray(Xf).shape[1]
        Xf_ = np.asfortranarray(Xf if nf else np.zeros((d, 1)), dtype=np.float64)
        yf_ = _f(yf if nf else [0.0])
        out = np.zeros(12 + 4 * d + 4 * d * d)
        x = _f(x)
        st = lib().orc_eval_point(C.byref(self.p), nf, _ptr(Xf_), _ptr(yf_), _ptr(x), _ptr(out))
        names = ["mu", "sigma", "alpha", "fstar", "g_mu", "g_sig", "g_mumu", "g_sigsig", "g_th", "g_thth", "g_muth", "g_sigth"]
        r = {n: out[i] for i, n in enumerate(names)}
        o = 12
        for n in ("dmu", "dsigma", "dalpha"):
            r[n] = out[o:o + d].copy(); o += d
        for n in ("Hmu", "Hsigma", "Halpha_ref", "Halpha_true"):
            r[n] = out[o:o + d * d].reshape(d, d).copy(); o += d * d
        r["d2alpha_dxdtheta"] = out[o:o + d].copy()
        r["status"] = st
        return r

    def multistart(self, Xf=None, yf=None):
        d, S = self.d, self.S
        nf = 0 if Xf is None else np.asarray(Xf).shape[1]
        Xf_ = np.asfortranarray(Xf if nf else np.zeros((d, 1)), dtype=np.float64)
        yf_ = _f(yf if nf else [0.0])
        xb, fb = np.zeros(d), C.c_double()
        sst, sit = np.zeros(S, np.int32), np.zeros(S, np.int32)
        sx, sf = np.zeros((d, S), order="F"), np.zeros(S)
        rc = lib().orc_multistart_solve(C.byref(self.p), nf, _ptr(Xf_), _ptr(yf_), _ptr(xb), C.byref(fb),
                                        sst.ctypes.data_as(_ip), sit.ctypes.data_as(_ip), _ptr(sx), _ptr(sf))
        return {"x": xb, "f": fb.value, "rc": rc, "start_status": sst, "start_iters": sit, "start_x": sx, "start_f": sf}


def sobol_uniform(dim, n):
    out = np.zeros((dim, n), order="F")
    lib().orc_sobol_uniform(dim, n, _ptr(out))
    return out


def sobol_uint32(dim, n):
    out = np.zeros((dim, n), dtype=np.uint32, order="F")
    lib().orc_sobol_uint32(dim, n, out.ctypes.data_as(C.POINTER(C.c_uint)))
    return out


def gen_low_discrepancy_sequence(M, d, H):
    out = np.zeros((M, d + 1, H), order="F")
    lib().orc_gen_low_discrepancy_sequence(M, d, H, _ptr(out))
    return out


def generate_initial_guesses(S, lbs, ubs):
    lbs, ubs = _f(lbs), _f(ubs)
    d = len(lbs)
    out = np.zeros((d, S + 2), order="F")
    lib().orc_generate_initial_guesses(S, d, _ptr(lbs), _ptr(ubs), _ptr(out))
    return out


def kernel_scalars(kernel, ktheta, rho):
    kt = _f(list(ktheta) + [0.0] * (4 - len(ktheta)))
    out = np.zeros(3)
    lib().orc_kernel_scalars(KERNEL_IDS[kernel], _ptr(kt), float(rho), _ptr(out))
    return out


def mean_std(v):
    v = _f(v)
    m, s = C.c_double(), C.c_double()
    lib().orc_mean_std(_ptr(v), len(v), 1, C.byref(m), C.byref(s))
    return m.value, s.value


def rule_partials(rule, mu, sigma, theta1, fstar, sigma_tol=1e-8):
    """[g, g_mu, g_sig, g_mumu, g_sigsig, g_muth, g_sigth, g_musig] of the C++ oracle's decision rule."""
    out = np.zeros(8)
    lib().orc_rule_partials(RULE_IDS[rule], sigma_tol, float(mu), float(sigma), float(theta1), float(fstar), _ptr(out))
    return out


def tr_step(H, g, Delta):
    """Exact trust-region step of the oracle's inner solve: returns (p, hit_constraint)."""
    H = np.ascontiguousarray(H, dtype=np.float64); g = _f(g)
    p = np.zeros(len(g))
    hit = lib().orc_tr_step(len(g), _ptr(H), _ptr(g), float(Delta), _ptr(p))
    return p, bool(hit)
