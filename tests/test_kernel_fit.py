"""Kernel hyper-parameters fitted on the device: rbo_log_marginal_likelihood, rbo_set_kernel and rbo_fit_kernel (optimize!,
rbs.jl:770-829; set_kernel!, rbs.jl:123-135) against an independent numpy/scipy restatement (dense K, LAPACK Cholesky, explicit
K^-1 and the trace formula), a host refit of the surrogate, and themselves (determinism, failure paths, shards).

Tolerances (FP64):
  * ll: 1e-10 relative;
  * gradient: |g_device - g_numpy| <= 16 kappa(K) eps (||a||^2 + ||K^-1||_F) ||dK/dtheta||_F, with kappa(K) the 2-norm condition number
    computed here: the first-order bound of the trace tr((a a' - K^-1) dK) / 2 when both sides carry a normwise relative error kappa eps;
  * set_kernel: c within 1e-9 relative to max |c| (the floor of test_condition_on_device_matches_host_refit), and a teacher-forced
    rollout within that test's tolerances (values 1e-9 relative, gradients 1e-6 relative to each trajectory's largest component).
"""
import ctypes as C

import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve
from scipy.optimize import minimize
from scipy.spatial.distance import cdist

from conftest import relerr

EPS = np.finfo(np.float64).eps
KERNEL_ID = {"Matern12": 0, "Matern32": 1, "Matern52": 2, "SquaredExponential": 3, "Periodic": 4}


# ---- numpy restatement (test infrastructure: the product never imports it) ---------------------------------------------------------
def psi_family(kernel, rho, theta):
    """psi(rho; theta) of rbf.jl:60-103; theta = (l,) or, for Periodic, (l, p)."""
    l = theta[0]
    if kernel == "Matern52":
        s = np.sqrt(5.0) * rho / l
        return (1 + s + s * s / 3.0) * np.exp(-s)
    if kernel == "Matern32":
        s = np.sqrt(3.0) * rho / l
        return (1 + s) * np.exp(-s)
    if kernel == "Matern12":
        return np.exp(-rho / l)
    if kernel == "SquaredExponential":
        return np.exp(-0.5 * (rho / l) ** 2)
    return np.exp(-2.0 * np.sin(np.pi * rho / theta[1]) ** 2 / l**2)


def dpsi_dtheta(kernel, rho, theta):
    """[d psi / d theta_i] in closed form, one array per hyper-parameter."""
    l = theta[0]
    if kernel == "Matern52":
        s = np.sqrt(5.0) * rho / l
        return [(s * s / l) * (1 + s) / 3.0 * np.exp(-s)]
    if kernel == "Matern32":
        s = np.sqrt(3.0) * rho / l
        return [(s * s / l) * np.exp(-s)]
    if kernel == "Matern12":
        return [(rho / l**2) * np.exp(-rho / l)]
    if kernel == "SquaredExponential":
        return [(rho**2 / l**3) * np.exp(-0.5 * (rho / l) ** 2)]
    u = np.pi * rho / theta[1]
    psi = psi_family(kernel, rho, theta)
    return [psi * 4.0 * np.sin(u) ** 2 / l**3, psi * (2.0 / l**2) * np.sin(2 * u) * u / theta[1]]


def kmat(X, kernel, theta, sn2):
    R = cdist(X.T, X.T)
    K = psi_family(kernel, R, theta)
    np.fill_diagonal(K, 1.0)
    return K + sn2 * np.eye(X.shape[1]), R


def lml(X, y, kernel, theta, sn2, full=False):
    """ll = -y'K^-1 y/2 - log det K/2 - N log(2 pi)/2 and grad_i = tr((a a' - K^-1) dK/dtheta_i) / 2, a = K^-1 y."""
    K, R = kmat(X, kernel, theta, sn2)
    cf = cho_factor(K, lower=True)
    a = cho_solve(cf, y)
    N = len(y)
    ll = -0.5 * float(y @ a) - float(np.sum(np.log(np.diag(cf[0])))) - 0.5 * N * np.log(2 * np.pi)
    Kinv = cho_solve(cf, np.eye(N))
    dKs = []
    for dK in dpsi_dtheta(kernel, R, theta):
        dK = np.array(dK, dtype=np.float64)
        np.fill_diagonal(dK, 0.0)
        dKs.append(dK)
    g = np.array([0.5 * float(np.sum((np.outer(a, a) - Kinv) * dK)) for dK in dKs])
    if full:
        return ll, g, dict(K=K, a=a, Kinv=Kinv, dKs=dKs)
    return ll, g


def gp_draw(kernel, theta, d, N, seed, sn2=1e-6):
    rng = np.random.default_rng(seed)
    X = np.asfortranarray(rng.random((d, N)))
    K, _ = kmat(X, kernel, theta, sn2)
    return X, np.linalg.cholesky(K) @ rng.standard_normal(N)


def make_sur(pkg, kernel, theta, X, y, sn2=1e-6, extra=8):
    return pkg.Surrogate(getattr(pkg, kernel)(list(theta)), X, y, capacity=X.shape[1] + extra, decision_rule=pkg.EI(), σn2=sn2)


FAMILIES = [("Matern12", (0.5,)), ("Matern32", (0.4,)), ("Matern52", (0.3,)), ("SquaredExponential", (0.25,)), ("Periodic", (0.3, 1.3))]


# ---- CPU -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel,theta", FAMILIES)
def test_numpy_gradient_matches_central_differences(kernel, theta):
    """The reference's own fd_check idiom (runtests.jl:11-20) on the restatement, every hyper-parameter of every family."""
    # psi(|x - x'|) of the periodic kernel is positive definite on the line only, and ill-conditioned there unless sigma_n2 is larger
    d, sn2 = (1, 1e-3) if kernel == "Periodic" else (3, 1e-6)
    X, y = gp_draw(kernel, theta, d, 25, 11, sn2)
    _, g = lml(X, y, kernel, theta, sn2)
    for i in range(len(theta)):
        h = 1e-5 * theta[i]
        tp, tm = list(theta), list(theta)
        tp[i] += h
        tm[i] -= h
        fd = (lml(X, y, kernel, tp, sn2)[0] - lml(X, y, kernel, tm, sn2)[0]) / (2 * h)
        assert abs(g[i] - fd) <= 1e-7 * max(abs(fd), 1.0), (i, g[i], fd)


def test_default_fit_options(pkg):
    lib = pkg._lib.load()
    o = pkg._lib.FitOpts()
    lib.rbo_default_fit_opts(C.byref(o))
    assert (o.max_iterations, o.max_evals, o.gtol, o.ftol) == (30, 200, 1e-6, 1e-12)


# ---- GPU: evaluation parity ------------------------------------------------------------------------------------------------------
# (kernel, theta, N, d, sigma_n2): every family, N across the 64-row blocks and the DMMA tiles, d in {1, 6, 20, 32}. The periodic kernel
# is positive definite on the line only (d = 1), where dense sites make it as ill-conditioned as 1 / sigma_n2: 1e-3 keeps kappa near 1e4.
PARITY = [("Matern52", (0.3,), 1, 1, 1e-6), ("Matern12", (0.3,), 7, 1, 1e-6), ("Periodic", (0.3, 1.3), 7, 1, 1e-6),
          ("SquaredExponential", (0.15,), 31, 6, 1e-6), ("Periodic", (0.3, 1.3), 32, 1, 1e-3), ("Matern32", (0.4,), 33, 20, 1e-6),
          ("Matern52", (0.5,), 64, 32, 1e-6), ("Matern12", (0.3,), 65, 6, 1e-6), ("Periodic", (0.5, 0.8), 65, 1, 1e-3),
          ("Matern12", (0.05,), 200, 1, 1e-6), ("SquaredExponential", (0.5,), 200, 20, 1e-6), ("Periodic", (0.2, 1.7), 200, 1, 1e-3),
          ("Matern52", (0.5,), 1000, 6, 1e-6), ("SquaredExponential", (0.9,), 1000, 32, 1e-6), ("Matern32", (0.7,), 2640, 20, 1e-6)]


def engine_for(pkg, sur, h=1):
    eng = pkg.RolloutEngine(0)
    eng.set_surrogate(pkg.FantasySurrogate(sur, h))
    return eng


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,theta,N,d,sn2", PARITY)
def test_log_marginal_likelihood_matches_numpy(pkg, kernel, theta, N, d, sn2):
    X, y = gp_draw(kernel, theta, d, N, 100 + N + d, sn2)
    sur = make_sur(pkg, kernel, theta, X, y, sn2)
    # evaluate at a point other than the resident one: the resident factor must not be what is used
    th = tuple(t * 1.1 for t in theta)
    ll, g, aux = lml(X, y, kernel, th, sn2, full=True)
    eng = engine_for(pkg, sur)
    try:
        lld, gd = eng.log_marginal_likelihood(th)
        lld2, gd2 = eng.log_marginal_likelihood(th)
        assert lld == lld2 and np.array_equal(gd, gd2)  # bit for bit
        assert abs(lld - ll) <= 1e-10 * abs(ll), (lld, ll)
        ev = np.linalg.eigvalsh(aux["K"])
        kappa = ev[-1] / ev[0]
        for i, dK in enumerate(aux["dKs"]):
            tol = 16 * kappa * EPS * (aux["a"] @ aux["a"] + np.linalg.norm(aux["Kinv"])) * np.linalg.norm(dK)
            assert abs(gd[i] - g[i]) <= tol, (i, gd[i], g[i], tol, kappa)
        if N <= 200:  # the device gradient against centred differences of the device ll
            for i in range(len(th)):
                hh = 1e-5 * th[i]
                tp, tm = list(th), list(th)
                tp[i] += hh
                tm[i] -= hh
                fd = (eng.log_marginal_likelihood(tp, grad=False)[0] - eng.log_marginal_likelihood(tm, grad=False)[0]) / (2 * hh)
                assert abs(gd[i] - fd) <= 1e-6 * max(abs(fd), 1.0), (i, gd[i], fd)
        # the resident surrogate is untouched
        _, _, c = eng.get_surrogate()
        assert np.array_equal(c, sur.c[:N])
    finally:
        eng.close()


# ---- GPU: set_kernel -------------------------------------------------------------------------------------------------------------
def rollout_case(orc, d, M, h, S):
    lbs, ubs, x0 = np.zeros(d), np.ones(d), np.full(d, 0.5)
    rn = orc.gen_low_discrepancy_sequence(M, d, h + 1)
    starts = orc.generate_initial_guesses(S, lbs, ubs)
    dd = np.asfortranarray(np.random.default_rng(3).random((d, h, M)))
    return lbs, ubs, x0, rn, starts, dd


def do_rollout(eng, d, M, h, x0, lbs, ubs, fmini, dd, x_forced=None):
    v, gx, gt, st = np.zeros(M), np.zeros((d, M), order="F"), np.zeros((1, M), order="F"), np.zeros(M, np.int32)
    eng.rollout(x0, np.zeros(1), lbs, ubs, h, fmini, v, gx, gt, dual_dirs=dd, x_forced=x_forced, status=st)
    return v, gx, st


@pytest.mark.gpu
@pytest.mark.parametrize("grow", [0, 5])
def test_set_kernel_matches_host_refit(pkg, orc, grow):
    """rbo_set_kernel after rbo_set_surrogate (grow = 0) and after rbo_condition has grown the surrogate across a 32-row panel boundary
    (62 -> 67: the uploaded factor is stale) against a host set_kernel! of the same data: c, and a teacher-forced rollout."""
    d, N, h, M, S = 4, 62, 2, 24, 3
    X, y = gp_draw("Matern52", (0.5,), d, N, 21)
    sur = make_sur(pkg, "Matern52", (0.5,), X, y)
    lbs, ubs, x0, rn, starts, dd = rollout_case(orc, d, M, h, S)
    rng = np.random.default_rng(9)
    newx, newy = rng.random((d, grow)), rng.standard_normal(grow) * 0.3
    eng = pkg.RolloutEngine(0)
    try:
        eng.set_surrogate(pkg.FantasySurrogate(sur, h)); eng.set_normals(rn); eng.set_starts(starts)
        for j in range(grow):
            eng.condition(newx[:, j], newy[j])
        Xh, yh = np.concatenate([X, newx], axis=1), np.concatenate([y, newy])
        eng.set_kernel(pkg.Matern52([0.35]))
        Xd, yd, cd = eng.get_surrogate()
        assert np.array_equal(Xd, Xh) and np.array_equal(yd, yh)
        ref = make_sur(pkg, "Matern52", (0.35,), Xh, yh)
        n = N + grow
        assert relerr(cd, ref.c[:n], floor=np.abs(ref.c[:n]).max()) < 1e-9
        fmini = float(np.min(yh))
        v, gx, st = do_rollout(eng, d, M, h, x0, lbs, ubs, fmini, dd)
        xs = eng.tape(h)["xs"]
        eng2 = pkg.RolloutEngine(0)
        try:
            eng2.set_surrogate(pkg.FantasySurrogate(ref, h)); eng2.set_normals(rn); eng2.set_starts(starts)
            v2, g2, s2 = do_rollout(eng2, d, M, h, x0, lbs, ubs, fmini, dd, x_forced=np.asfortranarray(xs[:, 1:, :]))
        finally:
            eng2.close()
        assert np.all(st == 0) and np.all(s2 == 0) and relerr(v, v2) < 1e-9
        gscale = np.maximum(np.abs(g2).max(axis=0, keepdims=True), 1e-6)
        assert np.max(np.abs(gx - g2) / gscale) < 1e-6
        # rbo_condition keeps working after the refit, across the next panel boundary as well
        Xc, yc = Xh, yh
        for j in range(34 - grow):
            xn, yn = rng.random(d), 0.3 * rng.standard_normal()
            eng.condition(xn, yn)
            Xc, yc = np.concatenate([Xc, xn[:, None]], axis=1), np.append(yc, yn)
        ref2 = make_sur(pkg, "Matern52", (0.35,), Xc, yc, extra=2)
        _, _, cc = eng.get_surrogate()
        assert len(cc) == len(yc) and relerr(cc, ref2.c[:len(yc)], floor=np.abs(ref2.c[:len(yc)]).max()) < 1e-9
    finally:
        eng.close()


# ---- GPU: the fit ----------------------------------------------------------------------------------------------------------------
def scipy_fit(X, y, kernel, theta0, lb, ub, sn2=1e-6):
    """scipy L-BFGS-B on the numpy objective in log theta from the same start."""
    def f(t):
        ll, g = lml(X, y, kernel, np.exp(t), sn2)
        return -ll, -g * np.exp(t)
    r = minimize(f, np.log(theta0), jac=True, method="L-BFGS-B", bounds=list(zip(np.log(lb), np.log(ub))),
                 options=dict(ftol=1e-15, gtol=1e-10, maxiter=200))
    return np.exp(r.x), -r.fun


def proj_grad_log(kt, g, lb, ub):
    gl = g * kt
    return np.where(((kt <= lb) & (gl < 0)) | ((kt >= ub) & (gl > 0)), 0.0, gl)


@pytest.mark.gpu
def test_fit_matches_scipy_on_gp_prior_data(pkg):
    """C3 shape (d = 10, N = 200), Matern-5/2 prior draw with l = 0.7, start l = 0.2, box [0.05, 5]."""
    X, y = gp_draw("Matern52", (0.7,), 10, 200, 1906)
    sur = make_sur(pkg, "Matern52", (0.2,), X, y)
    lb, ub = np.array([0.05]), np.array([5.0])
    ks, lls = scipy_fit(X, y, "Matern52", [0.2], lb, ub)
    eng = engine_for(pkg, sur)
    try:
        r = eng.fit_kernel(lb, ub)
        assert r["status"] in (pkg.FIT_GTOL, pkg.FIT_FTOL) and r["n_iter"] <= 30
        assert r["ll"] >= lls - 1e-8 * abs(lls), (r["ll"], lls)
        assert abs(r["ktheta"][0] - ks[0]) <= 1e-4 * ks[0], (r["ktheta"], ks)
        assert np.max(np.abs(proj_grad_log(r["ktheta"], r["grad"], lb, ub))) <= 1e-6 * max(1.0, abs(r["ll"]))
        assert r["ll"] == eng.log_marginal_likelihood(r["ktheta"])[0]
        # the resident surrogate is the refit at the optimum
        _, _, c = eng.get_surrogate()
        ref = make_sur(pkg, "Matern52", tuple(r["ktheta"]), X, y)
        assert relerr(c, ref.c[:200], floor=np.abs(ref.c[:200]).max()) < 1e-9
        # a repeated fit from the same start is bit for bit the same
        eng.set_kernel(pkg.Matern52([0.2]))
        r2 = eng.fit_kernel(lb, ub)
        assert all(np.array_equal(r[k], r2[k]) for k in r)
    finally:
        eng.close()
    # the host-mirror entry point
    s2 = make_sur(pkg, "Matern52", (0.2,), X, y)
    r3 = pkg.optimize(s2, lb, ub)
    assert np.array_equal(s2.ψ.θ, r3["ktheta"]) and np.array_equal(r3["ktheta"], r["ktheta"])
    assert relerr(s2.c[:200], ref.c[:200], floor=np.abs(ref.c[:200]).max()) < 1e-12


@pytest.mark.gpu
def test_fit_periodic_two_parameters(pkg):
    X, y = gp_draw("Periodic", (0.5, 1.2), 1, 60, 5, 1e-3)
    sur = make_sur(pkg, "Periodic", (0.6, 1.1), X, y, 1e-3)
    lb, ub = np.array([0.1, 0.5]), np.array([3.0, 3.0])
    eng = engine_for(pkg, sur)
    try:
        ll0 = eng.log_marginal_likelihood([0.6, 1.1])[0]
        r = eng.fit_kernel(lb, ub)
        assert r["ktheta"].shape == (2,) and r["status"] in (pkg.FIT_GTOL, pkg.FIT_FTOL)
        assert r["ll"] > ll0 and not np.array_equal(r["ktheta"], [0.6, 1.1])
        assert np.all(r["ktheta"] != [0.6, 1.1])  # both parameters moved
        if r["status"] == pkg.FIT_GTOL:
            assert np.max(np.abs(proj_grad_log(r["ktheta"], r["grad"], lb, ub))) <= 1e-6 * max(1.0, abs(r["ll"]))
        ks, lls = scipy_fit(X, y, "Periodic", [0.6, 1.1], lb, ub, 1e-3)
        assert r["ll"] >= lls - 1e-6 * abs(lls), (r, ks, lls)
    finally:
        eng.close()


@pytest.mark.gpu
def test_fit_on_the_upper_bound_returns_it_exactly(pkg):
    X, y = gp_draw("Matern52", (0.7,), 10, 200, 1906)
    eng = engine_for(pkg, make_sur(pkg, "Matern52", (0.2,), X, y))
    try:
        r = eng.fit_kernel([0.05], [0.4])
        assert r["ktheta"][0] == 0.4 and r["status"] == pkg.FIT_GTOL and r["grad"][0] > 0
    finally:
        eng.close()


@pytest.mark.gpu
def test_fit_then_rollout_equals_set_kernel_on_a_fresh_handle(pkg, orc):
    """One start slot per start (3 + 2 starts): the rollout does not depend on the handle's history."""
    d, N, h, M, S = 4, 40, 2, 32, 3
    X, y = gp_draw("Matern52", (0.5,), d, N, 33)
    sur = make_sur(pkg, "Matern52", (0.2,), X, y)
    lbs, ubs, x0, rn, starts, dd = rollout_case(orc, d, M, h, S)
    fmini = float(np.min(y))
    a, b = pkg.RolloutEngine(0), pkg.RolloutEngine(0)
    try:
        a.set_surrogate(pkg.FantasySurrogate(sur, h)); a.set_normals(rn); a.set_starts(starts)
        r = a.fit_kernel([0.05], [5.0])
        b.set_surrogate(pkg.FantasySurrogate(sur, h)); b.set_normals(rn); b.set_starts(starts)
        b.set_kernel(pkg.Matern52(list(r["ktheta"])))
        assert all(np.array_equal(p, q) for p, q in zip(a.get_surrogate(), b.get_surrogate()))
        ra, rb = do_rollout(a, d, M, h, x0, lbs, ubs, fmini, dd), do_rollout(b, d, M, h, x0, lbs, ubs, fmini, dd)
        assert all(np.array_equal(p, q) for p, q in zip(ra, rb))
    finally:
        a.close(); b.close()


# ---- GPU: failure paths ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_failures_leave_the_handle_unchanged(pkg, orc):
    """sigma_n2 = 0, Periodic, sites 0 and 0.5: at p = 0.5, sin(pi) rounds so that psi = 1 exactly and K has two equal rows; at p = 1
    it is positive definite."""
    d, h, M, S = 1, 1, 16, 2
    X = np.asfortranarray([[0.0, 0.5]])
    y = np.array([0.3, -0.2])
    sur = pkg.Surrogate(pkg.Periodic([1.0, 1.0]), X, y, capacity=4, decision_rule=pkg.EI(), σn2=0.0)
    lbs, ubs, x0, rn, starts, dd = rollout_case(orc, d, M, h, S)
    eng = pkg.RolloutEngine(0)
    try:
        eng.set_surrogate(pkg.FantasySurrogate(sur, h)); eng.set_normals(rn); eng.set_starts(starts)
        before = eng.get_surrogate()
        r0 = do_rollout(eng, d, M, h, x0, lbs, ubs, -0.2, dd)
        lib, hd = eng.lib, eng.handle.h
        kt = np.array([1.0, 0.5])
        ll = C.c_double()
        assert lib.rbo_log_marginal_likelihood(hd, pkg._lib.dptr(kt), 2, C.byref(ll), None) == -5
        assert lib.rbo_set_kernel(hd, 4, pkg._lib.dptr(kt), 2) == -5
        o = pkg._lib.FitOpts()
        lib.rbo_default_fit_opts(C.byref(o))
        lb, ub = np.array([1.0, 0.25]), np.array([1.0, 0.5])
        assert lib.rbo_fit_kernel(hd, C.byref(o), pkg._lib.dptr(lb), pkg._lib.dptr(ub), None, None, None, None, None, None) == -5
        after = eng.get_surrogate()
        assert all(p.tobytes() == q.tobytes() for p, q in zip(before, after))
        r1 = do_rollout(eng, d, M, h, x0, lbs, ubs, -0.2, dd)
        assert all(p.tobytes() == q.tobytes() for p, q in zip(r0, r1))
        # argument errors
        one, two = np.array([1.0]), np.array([1.0, 1.0])
        assert lib.rbo_log_marginal_likelihood(hd, pkg._lib.dptr(one), 1, C.byref(ll), None) == -1  # Periodic takes 2
        assert lib.rbo_log_marginal_likelihood(hd, pkg._lib.dptr(np.array([1.0, -1.0])), 2, C.byref(ll), None) == -1
        assert lib.rbo_set_kernel(hd, 2, pkg._lib.dptr(two), 2) == -1
        assert lib.rbo_set_kernel(hd, 7, pkg._lib.dptr(one), 1) == -1
        assert lib.rbo_set_kernel(None, 2, pkg._lib.dptr(one), 1) == -1
        assert lib.rbo_fit_kernel(hd, C.byref(o), pkg._lib.dptr(np.array([2.0, 1.0])), pkg._lib.dptr(two), None, None, None, None, None, None) == -1
        assert lib.rbo_fit_kernel(hd, C.byref(o), pkg._lib.dptr(np.array([0.0, 1.0])), pkg._lib.dptr(two), None, None, None, None, None, None) == -1
        assert lib.rbo_fit_kernel(hd, None, pkg._lib.dptr(two), pkg._lib.dptr(two), None, None, None, None, None, None) == -1
        assert lib.rbo_fit_kernel(None, C.byref(o), pkg._lib.dptr(two), pkg._lib.dptr(two), None, None, None, None, None, None) == -1
        assert all(p.tobytes() == q.tobytes() for p, q in zip(before, eng.get_surrogate()))
    finally:
        eng.close()


# ---- GPU: shards -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fit_on_one_shard_and_set_kernel_on_the_other(pkg, orc):
    """Two handles on one device, each with half of the samples: fit on one, rbo_set_kernel(theta*) on the other. The resident surrogates
    agree bit for bit, and the sharded ascent equals the one-handle call (5 + 2 starts: one start slot per start)."""
    d, N, h, M, S = 6, 30, 2, 64, 5
    X, y = gp_draw("Matern52", (0.6,), d, N, 77)
    sur = make_sur(pkg, "Matern52", (0.3,), X, y)
    lbs, ubs, x0, rn, starts, dd = rollout_case(orc, d, M, h, S)
    fmini = float(np.min(y))
    engs = [pkg.RolloutEngine(0) for _ in range(3)]
    try:
        for e, (m0, mc) in zip(engs, [(0, M // 2), (M // 2, M - M // 2), (0, M)]):
            e.set_surrogate(pkg.FantasySurrogate(sur, h)); e.set_normals(rn, m0, mc); e.set_starts(starts)
        r = engs[0].fit_kernel([0.05], [5.0])
        for e in engs[1:]:
            e.set_kernel(pkg.Matern52(list(r["ktheta"])))
        s0 = engs[0].get_surrogate()
        for e in engs[1:]:
            assert all(np.array_equal(p, q) for p, q in zip(s0, e.get_surrogate()))
        x0s = np.asfortranarray(0.2 + 0.6 * np.random.default_rng(4).random((d, 3)))
        kw = dict(optimizer=pkg.Adam(η=0.02), max_iterations=6, use_eswavs=False)
        a = pkg.stochastic_solve_batch_sharded(engs[:2], x0s, np.zeros(1), lbs, ubs, h, fmini, dual_dirs=dd, **kw)
        b = engs[2].stochastic_solve_batch(x0s, np.zeros(1), lbs, ubs, h, fmini, dual_dirs=dd, **kw)
        for k in ("x_final", "n_iter", "end_status", "x_hist", "mean_hist", "gmean_hist"):
            assert np.array_equal(a[k], b[k], equal_nan=True), k
    finally:
        for e in engs:
            e.close()


@pytest.mark.gpu
def test_fit_box_must_match_the_resident_family(pkg):
    """rbo_fit_kernel reads the box and writes its outputs for the resident family's count of hyper-parameters: the Python wrapper
    refuses a box of another length before the library reads past it."""
    X, y = gp_draw("Periodic", (0.5, 1.2), 1, 20, 5, 1e-3)
    eng = engine_for(pkg, make_sur(pkg, "Periodic", (0.6, 1.1), X, y, 1e-3))
    try:
        with pytest.raises(ValueError):
            eng.fit_kernel([0.1], [3.0])
        eng.set_kernel(pkg.Matern52([0.3]))  # the family changes with set_kernel
        with pytest.raises(ValueError):
            eng.fit_kernel([0.1, 0.5], [3.0, 3.0])
        assert eng.fit_kernel([0.05], [5.0])["ktheta"].shape == (1,)
    finally:
        eng.close()


@pytest.mark.gpu
def test_rejected_trials_leave_no_error_text_after_a_successful_fit(pkg):
    """sigma_n2 = 0, Periodic, sites 0 and 0.5, equal targets: ll grows as p falls towards 0.5, where K is singular, so the line search
    meets trials at which K is not positive definite and rejects them. The fit succeeds and rbo_last_error stays empty."""
    sur = pkg.Surrogate(pkg.Periodic([1.0, 0.9]), np.asfortranarray([[0.0, 0.5]]), np.array([0.3, 0.3]), capacity=4,
                        decision_rule=pkg.EI(), σn2=0.0)
    eng = engine_for(pkg, sur)
    try:
        r = eng.fit_kernel([1.0, 0.5], [1.0, 0.9])
        assert 0.5 < r["ktheta"][1] < 0.9 and r["ktheta"][0] == 1.0
        assert r["n_evals"] > r["n_iter"] + 1  # some trials were rejected
        assert eng.lib.rbo_last_error(eng.handle.h) == b""
    finally:
        eng.close()
