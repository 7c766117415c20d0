"""CPU tests that pin the oracle (oracle/rbo_oracle.cpp) as far as it can be pinned without Julia:
closed forms and finite differences (the reference's own test idiom, runtests.jl:11-20), scipy's Sobol,
and an independent numpy restatement (oracle/py_restatement.py)."""
import numpy as np
import pytest
from scipy.stats import qmc

from conftest import oracle_problem, relerr
from oracle import py_restatement as pr


def small_problem(pkg, orc, name="C2", M=6, N=14, h=2, S=4, mode=1, seed=3, **kw):
    wl = pkg.problems.make_workload(name, M=M, N=N, h=h, S=S, seed=seed)
    sur = wl.surrogate()
    rn = orc.gen_low_discrepancy_sequence(M, wl.d, h + 1)
    starts = orc.generate_initial_guesses(S, wl.lbs, wl.ubs)
    dd = np.asfortranarray(np.random.default_rng(seed).random((wl.d, max(h, 1), M)))
    return wl, sur, rn, starts, dd, oracle_problem(orc, wl, sur, rn, starts, mode, dual_dirs=dd, **kw)


@pytest.mark.parametrize("kernel,theta", [("matern52", (0.456,)), ("matern32", (0.456,)), ("matern12", (0.456,)), ("se", (0.456,)), ("periodic", (0.8, 1.3))])
def test_kernel_derivatives_fd(orc, kernel, theta):
    # runtests.jl:23-54: rho = 0.123, theta = 0.456, h = 1e-6, rtol 1e-8 (second derivative via the first)
    rho, h = 0.123, 1e-6
    p, dp, d2p = orc.kernel_scalars(kernel, theta, rho)
    fp = (orc.kernel_scalars(kernel, theta, rho + h)[0] - orc.kernel_scalars(kernel, theta, rho - h)[0]) / (2 * h)
    fdp = (orc.kernel_scalars(kernel, theta, rho + h)[1] - orc.kernel_scalars(kernel, theta, rho - h)[1]) / (2 * h)
    assert abs(fp - dp) <= 1e-8 * max(1, abs(dp))
    assert abs(fdp - d2p) <= 1e-7 * max(1, abs(d2p))


def test_matern52_closed_forms(orc):
    # SURVEY.md section 4: psi' = -(5 rho / 3 l^2)(1+s) e^-s, psi'' = (5 / 3 l^2)(s^2 - s - 1) e^-s
    for rho in (0.0, 1e-3, 0.3, 2.0):
        l = 0.7
        s = np.sqrt(5) * rho / l
        p, dp, d2p = orc.kernel_scalars("matern52", (l,), rho)
        assert np.isclose(p, (1 + s + s * s / 3) * np.exp(-s), rtol=1e-14)
        assert np.isclose(dp, -(5 * rho / (3 * l * l)) * (1 + s) * np.exp(-s), rtol=1e-13, atol=1e-300)
        assert np.isclose(d2p, (5 / (3 * l * l)) * (s * s - s - 1) * np.exp(-s), rtol=1e-13)
        assert np.isclose(p, pr.psi52(rho, l), rtol=1e-14) and np.isclose(d2p, pr.d2psi52(rho, l), rtol=1e-13)


def test_surrogate_eval_fd_ladder(pkg, orc):
    # runtests.jl:83-118: mu, sigma, alpha and their gradient / Hessian against centred differences
    wl, sur, rn, starts, dd, P = small_problem(pkg, orc, N=20)
    rng = np.random.default_rng(0)
    Xf = np.asfortranarray(rng.random((wl.d, 2)))
    yf = np.array([-0.3, 0.1])
    x = rng.random(wl.d)
    e = P.eval_point(x, Xf, yf)
    hstep = 1e-5
    for key, gkey, Hkey in (("mu", "dmu", "Hmu"), ("sigma", "dsigma", "Hsigma"), ("alpha", "dalpha", "Halpha_true")):
        g_fd = np.zeros(wl.d)
        H_fd = np.zeros((wl.d, wl.d))
        for a in range(wl.d):
            dx = np.zeros(wl.d); dx[a] = hstep
            ep, em = P.eval_point(x + dx, Xf, yf), P.eval_point(x - dx, Xf, yf)
            g_fd[a] = (ep[key] - em[key]) / (2 * hstep)
            H_fd[:, a] = (ep[gkey] - em[gkey]) / (2 * hstep)
        assert relerr(e[gkey], g_fd, floor=np.abs(g_fd).max()) < 1e-7, key
        assert relerr(e[Hkey], H_fd, floor=np.abs(H_fd).max()) < 1e-6, key
    # Q1: the reference's H alpha omits the mu-sigma cross term and therefore does NOT match finite differences
    assert relerr(e["Halpha_ref"], H_fd, floor=np.abs(H_fd).max()) > 1e-3


def test_ei_partials_fd(pkg, orc):
    # decision_rules.jl:23-34 partials against differences of g in (mu, sigma, theta)
    from scipy.special import erfc
    def g(mu, s, th, fs):
        z = (fs - mu - th) / s
        return (fs - mu - th) * 0.5 * erfc(-z / np.sqrt(2)) + s * np.exp(-0.5 * z * z) / np.sqrt(2 * np.pi)
    mu, s, th, fs, h = 0.3, 0.7, 0.05, 0.1, 1e-5
    e = pr.ei_partials(mu, s, th, fs)
    assert np.isclose(e["g"], g(mu, s, th, fs), rtol=1e-14)
    assert np.isclose(e["g_mu"], (g(mu + h, s, th, fs) - g(mu - h, s, th, fs)) / (2 * h), rtol=1e-8)
    assert np.isclose(e["g_sig"], (g(mu, s + h, th, fs) - g(mu, s - h, th, fs)) / (2 * h), rtol=1e-8)
    assert np.isclose(e["g_mumu"], (g(mu + h, s, th, fs) - 2 * g(mu, s, th, fs) + g(mu - h, s, th, fs)) / h**2, rtol=1e-5)
    assert np.isclose(e["g_sigsig"], (g(mu, s + h, th, fs) - 2 * g(mu, s, th, fs) + g(mu, s - h, th, fs)) / h**2, rtol=1e-5)


def test_sobol_matches_scipy_joe_kuo(orc):
    for dim in (1, 2, 3, 7, 12, 22):
        n = 300
        ref = qmc.Sobol(dim, scramble=False).random_base2(9)[1:n + 1]  # scipy's first point is the origin
        got = orc.sobol_uniform(dim, n)
        assert np.array_equal(got.T, ref)
    # Sobol.jl's documented 2-D prefix (SURVEY.md A.8)
    assert np.array_equal(orc.sobol_uniform(2, 5).T, np.array([[.5, .5], [.75, .25], [.25, .75], [.375, .375], [.875, .875]]))


def test_low_discrepancy_sequence_known_answer(orc):
    # SURVEY.md Appendix C (derived, not reference truth): gen_low_discrepancy_sequence(4, 2, 2)
    R = orc.gen_low_discrepancy_sequence(4, 2, 2)
    assert R.shape == (4, 3, 2)
    assert np.allclose(R[0], [[-0.77592524854393186, 0.24081517181790421], [3.06e-17, 0.45179639513383107], [-2.02e-16, -0.95031046873742475]], rtol=1e-12, atol=1e-15)
    assert np.isclose(R[1, 1, 0], 0.49987745820010715, rtol=1e-13) and np.isclose(R[1, 2, 0], -1.0973240098785431, rtol=1e-13)
    # independent emulation of utils.jl:23-43, 65-74 with scipy
    M, d, H = 5, 3, 3
    D = d + 1
    S = qmc.Sobol(D, scramble=False).random_base2(5)[1:M * H + 1].T
    Nn = np.zeros_like(S)
    for i in range(D):
        if i % 2 == 0:
            Nn[i] = np.sqrt(-2 * np.log10(S[i])) * np.cos(2 * np.pi * S[i + 1])
        else:
            Nn[i] = np.sqrt(-2 * np.log10(S[i - 1])) * np.sin(2 * np.pi * S[i])
    ref = Nn.reshape(-1, order="F").reshape((M, D, H), order="F")
    assert np.allclose(orc.gen_low_discrepancy_sequence(M, d, H), ref, rtol=1e-13, atol=1e-16)


def test_initial_guesses(orc):
    lbs, ubs = np.array([-5.0, 0.0]), np.array([10.0, 15.0])
    G = orc.generate_initial_guesses(3, lbs, ubs)
    assert G.shape == (2, 5)
    assert np.allclose(G[:, 0], lbs + 0.5 * (ubs - lbs))
    assert np.allclose(G[:, 3], lbs + 1e-6) and np.allclose(G[:, 4], ubs - 1e-6)


def test_fit_surrogate_matches_scipy(pkg, orc):
    wl = pkg.problems.make_workload("C2", N=30)
    K, L, c = orc.fit_surrogate(wl.X, wl.y, "matern52", (wl.ell,), 1e-6)
    sur = wl.surrogate()
    assert relerr(K, sur.K[:30, :30]) < 1e-14 and relerr(L, sur.L[:30, :30]) < 1e-12 and relerr(c, sur.c[:30]) < 1e-9


def test_oracle_vs_numpy_restatement_teacher_forced(pkg, orc):
    """Forward draws, conditioning and the three-case adjoint gradient of the C++ oracle against the independent
    numpy transcription, on the x-path the oracle's own inner solve produced."""
    wl, sur, rn, starts, dd, P = small_problem(pkg, orc, M=8, N=12, h=3, S=4)
    r = P.rollout()
    assert np.all(r["status"] == 0)
    cases = set()
    for m in range(wl.M):
        z = rn[m, :, :]
        fs, obs, grads = pr.rollout_teacher_forced(wl.X, wl.y, wl.ell, wl.sigma_n2, wl.h, wl.x0, wl.theta, z, r["xs"][:, 1:, m])
        assert relerr(obs, r["ys"][:, m]) < 1e-9
        assert relerr(grads, r["gys"][:, :, m]) < 1e-8
        gx, gth, case, t = pr.trajectory_gradient(fs, obs, grads, wl.theta, float(np.min(sur.y)), dd[:, :, m])
        assert case == r["grad_case"][m] and t == r["best_index"][m]
        cases.add(case)
        assert relerr(gx, r["grad_x"][:, m], floor=max(1e-6, np.abs(gx).max())) < 1e-6, (m, case, gx, r["grad_x"][:, m])
        assert relerr(gth, r["grad_theta"][:, m], floor=max(1e-6, np.abs(gth).max())) < 1e-6
        assert np.isclose(r["values"][m], max(float(np.min(sur.y)) - obs.min(), 0.0), rtol=1e-10, atol=1e-12)
    assert 3 in cases


def test_oracle_follows_a_forced_x_path(pkg, orc):
    """x_forced teacher-forces the oracle on a path that is not its own (what the parity tests feed back from the CUDA kernel): no
    inner solve runs, the tape holds the given path, and draws and gradients are those of the numpy restatement on that path."""
    wl, sur, rn, starts, dd, P = small_problem(pkg, orc, M=6, N=12, h=3, S=4)
    free = P.rollout()
    xf = np.asfortranarray(0.5 * free["xs"][:, 1:, :] + 0.25)  # inside the unit box, away from the oracle's maximisers
    r = oracle_problem(orc, wl, sur, rn, starts, 1, dual_dirs=dd, x_forced=xf).rollout()
    assert np.all(r["n_evals"] == 0) and np.array_equal(r["xs"][:, 1:, :], xf) and np.all(r["status"] == 0)
    for m in range(wl.M):
        fs, obs, grads = pr.rollout_teacher_forced(wl.X, wl.y, wl.ell, wl.sigma_n2, wl.h, wl.x0, wl.theta, rn[m], xf[:, :, m])
        assert relerr(obs, r["ys"][:, m]) < 1e-9 and relerr(grads, r["gys"][:, :, m]) < 1e-8
        gx, gth, case, t = pr.trajectory_gradient(fs, obs, grads, wl.theta, float(np.min(sur.y)), dd[:, :, m])
        assert case == r["grad_case"][m] and t == r["best_index"][m]
        assert relerr(gx, r["grad_x"][:, m], floor=max(1e-6, np.abs(gx).max())) < 1e-6


def test_case3_gradients_are_exercised(pkg, orc):
    """With htol = 1e-4 (rollout.jl:156) and an even dimension some case-3 duals survive the det test (Q3)."""
    wl, sur, rn, starts, dd, P = small_problem(pkg, orc, name="GP:2:0.25", M=64, N=12, h=3, S=4)
    r = P.rollout()
    c3 = r["grad_case"] == 3
    assert c3.sum() > 0
    nz = np.abs(r["grad_x"][:, c3]).max(axis=0) > 0
    assert nz.sum() > 0
    # and the numpy restatement agrees on those trajectories
    for m in np.nonzero(c3)[0][nz][:6]:
        fs, obs, grads = pr.rollout_teacher_forced(wl.X, wl.y, wl.ell, wl.sigma_n2, wl.h, wl.x0, wl.theta, rn[m], r["xs"][:, 1:, m])
        gx, gth, case, t = pr.trajectory_gradient(fs, obs, grads, wl.theta, float(np.min(sur.y)), dd[:, :, m])
        assert case == 3 and relerr(gx, r["grad_x"][:, m], floor=np.abs(gx).max()) < 1e-6
        assert relerr(gth, r["grad_theta"][:, m], floor=max(np.abs(gth).max(), 1e-9)) < 1e-6


def test_fast_perturbation_equals_dense(pkg, orc):
    wl, sur, rn, starts, dd, P = small_problem(pkg, orc, name="GP:2:0.25", M=32, N=12, h=3, S=4)
    r = P.rollout(tape=False)
    wl2, sur2, rn2, st2, dd2, P2 = small_problem(pkg, orc, name="GP:2:0.25", M=32, N=12, h=3, S=4, flags=orc.FLAG_FAST_PERTURB)
    r2 = P2.rollout(tape=False)
    assert relerr(r2["grad_x"], r["grad_x"], floor=1e-3) < 1e-9
    assert relerr(r2["values"], r["values"]) < 1e-12


def test_factored_formulation_close(pkg, orc):
    """sigma^2 = k0 - |L^-1 kx|^2 (what the CUDA path evaluates) against the reference's k0 - kx.(K^-1 kx)."""
    wl, sur, rn, starts, dd, P = small_problem(pkg, orc, M=4, N=30, h=1, S=3)
    wl2, sur2, rn2, st2, dd2, P2 = small_problem(pkg, orc, M=4, N=30, h=1, S=3, flags=orc.FLAG_FACTORED)
    x = np.random.default_rng(5).random(wl.d)
    e1, e2 = P.eval_point(x), P2.eval_point(x)
    for k in ("mu", "sigma", "alpha"):
        assert np.isclose(e1[k], e2[k], rtol=1e-10)
    assert relerr(e1["Halpha_true"], e2["Halpha_true"], floor=np.abs(e1["Halpha_true"]).max()) < 1e-9


def test_inner_solve_converges_and_is_deterministic(pkg, orc):
    wl, sur, rn, starts, dd, P = small_problem(pkg, orc, M=1, N=20, h=1, S=6)
    a, b = P.multistart(), P.multistart()
    assert np.array_equal(a["x"], b["x"]) and a["f"] == b["f"]
    assert a["rc"] == 0 and np.all(a["x"] >= wl.lbs) and np.all(a["x"] <= wl.ubs)
    # at the reported maximiser the projected gradient is tiny
    e = P.eval_point(a["x"])
    g = -e["dalpha"]
    free = ~(((a["x"] <= wl.lbs) & (g > 0)) | ((a["x"] >= wl.ubs) & (g < 0)))
    assert np.abs(g[free]).max(initial=0.0) < 1e-7
    # first minimum wins (rbf_optim.jl:97)
    k = int(np.nanargmin(a["start_f"]))
    assert np.allclose(a["x"], a["start_x"][:, k])


def test_mean_std_matches_numpy(orc):
    v = np.random.default_rng(1).random(1000)
    m, s = orc.mean_std(v)
    assert np.isclose(m, v.mean(), rtol=1e-14) and np.isclose(s, v.std(ddof=1), rtol=1e-12)


def gh_inputs(pkg, n_nodes, depth):
    """nodes[indices[m]] / weights[indices[m]] of rollout.jl:431-432 as (depth x M) arrays."""
    nodes, weights = pkg.gausshermite(n_nodes)
    idx = np.asarray(pkg.generate_indices(n_nodes, depth)) - 1
    return np.asfortranarray(nodes[idx].T), np.asfortranarray(weights[idx].T)


def test_generate_indices_order(pkg):
    # utils.jl:217-221: collect(product(1:n, 1:n, ...)) runs the FIRST position fastest
    idx = pkg.generate_indices(3, 2)
    assert idx[:4] == [[1, 1], [2, 1], [3, 1], [1, 2]] and len(idx) == 9 and idx[-1] == [3, 3]


def test_gauss_hermite_horizon0_is_expected_improvement(pkg, orc):
    """h = 0: sum_m w_m max(fmini - (mu + sqrt2 sigma z_m), 0) / sqrt(pi) is the n-point Gauss-Hermite estimate of
    E[max(fmini - y, 0)], y ~ N(mu, sigma^2) = EI with xi = 0 (observables.jl:54-72); the sample gradients
    (observables.jl:157, no 1/sqrt(pi) -- the later definition wins) sum to sqrt(pi) grad EI."""
    n = 96
    wl = pkg.problems.make_workload("C2", M=n, N=14, h=0, S=4, seed=3)
    sur = wl.surrogate()
    nodes, weights = gh_inputs(pkg, n, 1)
    rn = np.zeros((n, wl.d + 1, 1), order="F")
    starts = orc.generate_initial_guesses(4, wl.lbs, wl.ubs)
    P = oracle_problem(orc, wl, sur, rn, starts, 1, gh_nodes=nodes, gh_weights=weights)
    r = P.rollout()
    e = P.eval_point(wl.x0, np.zeros((wl.d, 0), order="F"), np.zeros(0))
    assert np.all(r["status"] == 0)
    # the kink of max(., 0) limits Gauss-Hermite to ~1/n accuracy
    assert abs(r["values"].sum() - e["alpha"]) <= 2e-2 * abs(e["alpha"])
    assert set(np.unique(r["grad_case"])) <= {1, 2}
    # the sample gradients are the exact derivative of the finite quadrature sum (away from its kinks)
    x0, step, fd = wl.x0.copy(), 1e-6, np.zeros(wl.d)
    for a in range(wl.d):
        vals = []
        for sgn in (1, -1):
            wl.x0 = x0.copy(); wl.x0[a] += sgn * step
            vals.append(oracle_problem(orc, wl, sur, rn, starts, 0, gh_nodes=nodes, gh_weights=weights).rollout()["values"].sum())
        fd[a] = (vals[0] - vals[1]) / (2 * step)
    wl.x0 = x0
    assert np.allclose(r["grad_x"].sum(axis=1) / np.sqrt(np.pi), fd, rtol=1e-6, atol=1e-9)


def test_gauss_hermite_observable_formula(pkg, orc):
    """Teacher-forced GH rollout: y_k = mu_k(x_k) + sqrt(2) sigma_k(x_k) node_k re-derived with eval_point on the
    surrogate extended by the earlier fantasy points; value = w[t] max(fmini - min y, 0) / sqrt(pi)."""
    wl = pkg.problems.make_workload("C2", M=9, N=14, h=1, S=4, seed=3)
    sur = wl.surrogate()
    nodes, weights = gh_inputs(pkg, 3, 2)
    rn = np.zeros((9, wl.d + 1, 2), order="F")
    starts = orc.generate_initial_guesses(4, wl.lbs, wl.ubs)
    P = oracle_problem(orc, wl, sur, rn, starts, 1, gh_nodes=nodes, gh_weights=weights)
    r = P.rollout()
    fmini = float(np.min(sur.y))
    for m in range(9):
        ys = []
        for k in range(2):
            e = P.eval_point(r["xs"][:, k, m], np.asfortranarray(r["xs"][:, :k, m]), np.asarray(ys))
            ys.append(e["mu"] + np.sqrt(2) * e["sigma"] * nodes[k, m])
            assert np.isclose(ys[-1], r["ys"][k, m], rtol=1e-10, atol=1e-12)
            gy = (e["dmu"] + np.sqrt(2) * e["dsigma"] * nodes[k, m]) * weights[k, m]
            assert np.allclose(gy, r["gys"][:, k, m], rtol=1e-9, atol=1e-12)
        t = int(np.argmin(ys))
        assert np.isclose(r["values"][m], weights[t, m] * max(fmini - min(ys), 0.0) / np.sqrt(np.pi), rtol=1e-12, atol=1e-15)


@pytest.mark.parametrize("name", ["mc_hartmann6", "mc_gp2d", "ghq_hartmann6"])
def test_oracle_reproduces_golden(orc, name):
    """The committed fixtures (tests/golden/gen_golden.py: oracle output cross-checked with the numpy restatement) pin the
    oracle against silent drift: free-running rollout from the stored inputs must reproduce every stored output."""
    import os
    f = np.load(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))
    kw = {}
    if "gh_nodes" in f.files:
        kw = dict(gh_nodes=f["gh_nodes"], gh_weights=f["gh_weights"])
    P = orc.OracleProblem(f["X"], f["L"], f["y"], f["c"], f["x0"], f["lbs"], f["ubs"], f["rn"], f["starts"], h=int(f["h"]), kernel="matern52",
                          ktheta=(float(f["ell"]),), rule="EI", theta=f["theta"], sigma_n2=float(f["sigma_n2"]), fmini=float(f["fmini"]), mode=1,
                          dual_dirs=f["dual_dirs"], **kw)
    r = P.rollout()
    assert np.all(r["status"] == 0)
    assert np.array_equal(r["best_index"], f["best_index"]) and np.array_equal(r["grad_case"], f["grad_case"])
    for key, tol in (("xs", 1e-10), ("ys", 1e-10), ("gys", 1e-9), ("values", 1e-10), ("alphas", 1e-10)):
        assert relerr(r[key], f[key]) < tol, key
    gscale = np.maximum(np.abs(f["grad_x"]).max(axis=0, keepdims=True), 1e-9)
    assert np.max(np.abs(r["grad_x"] - f["grad_x"]) / gscale) < 1e-7


# ---------------------------------------------------------------------------------------------------
# Decision-rule partials of BOTH compiled implementations (the oracle's C++ and the product's rbo_device.cuh, the latter
# built for the host) by centred finite differences -- the runtests.jl:11-20 idiom. Covers EI, POI, LCB including the
# mixed partials g_mu_theta, g_sigma_theta, g_mu_sigma that only the adjoint / the solver's true Hessian consume.
# ---------------------------------------------------------------------------------------------------
def _device_scalars_lib():
    import ctypes as C, os, shutil, subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    src = os.path.join(here, "helpers", "device_scalars.cu")
    so = os.path.join(here, "helpers", "libdevice_scalars.so")
    hdr = os.path.join(os.path.dirname(here), "rollout-bayesian-optimization_b200", "csrc", "rbo_device.cuh")
    if not os.path.exists(so) or max(os.path.getmtime(src), os.path.getmtime(hdr)) > os.path.getmtime(so):
        # $NVCC, else nvcc on PATH, else the toolkit location csrc/Makefile builds with: the build needs no PATH entry, nor does this
        nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        subprocess.check_call([nvcc, "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets", "-Xcompiler", "-fPIC", "-shared", "-o", so, src])
    lib = C.CDLL(so)
    dp = C.POINTER(C.c_double)
    lib.dev_rule_partials.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, dp]
    lib.dev_kernel_scalars.argtypes = [C.c_int, dp, C.c_double, dp]
    return lib


def _rule_fn(which, orc):
    if which == "oracle":
        return lambda rule, mu, sg, th, fs: orc.rule_partials(rule, mu, sg, th, fs)
    lib = _device_scalars_lib()
    ids = {"EI": 0, "POI": 1, "LCB": 2}

    def f(rule, mu, sg, th, fs):
        out = np.zeros(8)
        lib.dev_rule_partials(ids[rule], 1e-8, mu, sg, th, fs, out.ctypes.data_as(__import__("ctypes").POINTER(__import__("ctypes").c_double)))
        return out
    return f


@pytest.mark.parametrize("which", ["oracle", "product"])
@pytest.mark.parametrize("rule", ["EI", "POI", "LCB"])
def test_rule_partials_by_finite_differences(orc, which, rule):
    f = _rule_fn(which, orc)
    rng = np.random.default_rng(4)
    for _ in range(12):
        mu, sg, th, fs = rng.normal(0.2, 0.8), rng.uniform(0.05, 1.5), rng.uniform(0.0, 2.5) if rule == "LCB" else rng.uniform(0.0, 0.3), rng.normal(0.0, 0.6)
        g, g_mu, g_sig, g_mumu, g_sigsig, g_muth, g_sigth, g_musig = f(rule, mu, sg, th, fs)
        e = 1e-5
        d = lambda i, k, dm=0.0, ds=0.0, dt=0.0: (f(rule, mu + dm, sg + ds, th + dt, fs)[i] - f(rule, mu - dm, sg - ds, th - dt, fs)[i]) / (2 * k)
        sc = lambda v: max(1e-6, abs(v))
        assert abs(d(0, e, dm=e) - g_mu) < 1e-7 * sc(g_mu) + 1e-9
        assert abs(d(0, e, ds=e) - g_sig) < 1e-7 * sc(g_sig) + 1e-9
        assert abs(d(1, e, dm=e) - g_mumu) < 1e-6 * sc(g_mumu) + 1e-8
        assert abs(d(2, e, ds=e) - g_sigsig) < 1e-6 * sc(g_sigsig) + 1e-8
        assert abs(d(1, e, ds=e) - g_musig) < 1e-6 * sc(g_musig) + 1e-8 and abs(d(2, e, dm=e) - g_musig) < 1e-6 * sc(g_musig) + 1e-8
        assert abs(d(1, e, dt=e) - g_muth) < 1e-6 * sc(g_muth) + 1e-8
        assert abs(d(2, e, dt=e) - g_sigth) < 1e-6 * sc(g_sigth) + 1e-8
    # below sigma_tol EI and POI are the constant 0 with zero partials (decision_rules.jl:87-89, 104-106)
    if rule != "LCB":
        assert np.all(f(rule, 0.1, 1e-9, 0.0, 0.0) == 0.0)


def test_product_kernel_scalars_by_finite_differences():
    """psi', psi'' and the radial coefficients a = (psi'' - psi'/rho)/rho^2, b = psi'/rho of rbo_device.cuh (host build)."""
    import ctypes as C
    lib = _device_scalars_lib()
    dp = C.POINTER(C.c_double)
    for kid, th in ((0, [0.6, 0, 0, 0]), (1, [0.45, 0, 0, 0]), (2, [0.7, 0, 0, 0]), (3, [0.35, 0, 0, 0]), (4, [0.9, 1.7, 0, 0])):
        kt = np.array(th, dtype=np.float64)
        def ev(rho):
            out = np.zeros(6)
            lib.dev_kernel_scalars(kid, kt.ctypes.data_as(dp), rho, out.ctypes.data_as(dp))
            return out
        for rho in (0.123, 0.456, 1.3):
            o, hh = ev(rho), 1e-6
            assert abs((ev(rho + hh)[0] - ev(rho - hh)[0]) / (2 * hh) - o[1]) < 1e-7 * max(1.0, abs(o[1]))
            assert abs((ev(rho + hh)[1] - ev(rho - hh)[1]) / (2 * hh) - o[2]) < 1e-6 * max(1.0, abs(o[2]))
            assert np.isclose(o[4], o[1] / rho, rtol=1e-13) and np.isclose(o[3], (o[2] - o[1] / rho) / rho**2, rtol=1e-12) and o[5] == o[4]
        o0 = ev(0.0)
        assert o0[3] == 0.0 and o0[4] == o0[2] and o0[5] == 0.0  # rbf.jl:129-131, 149: grad k = 0, Hk = psi''(0) I at coincident points


def _tr_exact(H, g, Delta):
    w, Q = np.linalg.eigh(H)
    gt = Q.T @ g
    if w[0] > 0:
        p = -Q @ (gt / w)
        if np.linalg.norm(p) <= Delta:
            return p
    lo = max(0.0, -w[0])
    f = lambda lam: np.linalg.norm(gt / (w + lam)) - Delta
    hi = lo + np.linalg.norm(g) / Delta + 1.0
    a, b = lo + 1e-14 * max(1.0, abs(lo)), hi
    if f(a) < 0:  # hard case
        y = np.where(w + lo > 1e-12 * max(abs(w).max(), 1e-300), -gt / np.where(w + lo > 1e-12, w + lo, 1.0), 0.0)
        y[0] = np.sqrt(max(Delta**2 - y @ y + y[0] ** 2, 0.0))
        return Q @ y
    for _ in range(200):
        m = 0.5 * (a + b)
        if f(m) > 0: a = m
        else: b = m
    return -Q @ (gt / (w + b))


def test_oracle_trust_region_step_is_exact(orc):
    """orc_tr_step (Householder tridiagonalisation + 64-way multisection, the algorithm the CUDA warp runs as well) against a
    dense eigendecomposition: feasibility, the model value of the exact minimiser, interior Newton steps, and the hard case."""
    rng = np.random.default_rng(12)
    model = lambda H, g, p: g @ p + 0.5 * p @ H @ p
    for n in (1, 2, 3, 6, 10, 20, 31):
        for trial in range(12):
            A = rng.standard_normal((n, n)); H = 0.5 * (A + A.T)
            if trial % 3 == 0:
                H = A @ A.T + 0.1 * np.eye(n)      # positive definite
            g = rng.standard_normal(n)
            Delta = float(rng.choice([1e-3, 0.1, 1.0, 30.0]))
            p, hit = orc.tr_step(H, g, Delta)
            pe = _tr_exact(H, g, Delta)
            assert np.linalg.norm(p) <= Delta * (1 + 1e-9)
            scale = abs(model(H, g, pe)) + 1e-300
            # the shift is located to 4e-6 of its initial bracket (3 rounds of 64-way multisection; a 4th round costs 2 % of the
            # throughput and saves no evaluation): |p| may fall short of Delta by up to ~1 % when the shift sits just above
            # -lambda_min and the bracket is much wider than the shift -- immaterial for a trust-region method
            assert model(H, g, p) <= model(H, g, pe) + 2e-2 * scale, (n, trial, model(H, g, p), model(H, g, pe))
            if hit and n > 1:
                assert np.linalg.norm(p) >= Delta * (1 - 2e-2)
            if not hit:
                assert np.allclose(H @ p, -g, rtol=1e-8, atol=1e-10) and np.all(np.linalg.eigvalsh(H) > 0)
    # hard case: the gradient has no component along the eigenvector of the most negative eigenvalue
    Q, _ = np.linalg.qr(rng.standard_normal((6, 6)))
    w = np.array([-2.0, 0.5, 1.0, 1.5, 2.0, 3.0])
    H = Q @ np.diag(w) @ Q.T; H = 0.5 * (H + H.T)
    g = Q[:, 1:] @ rng.standard_normal(5) * 0.1
    p, hit = orc.tr_step(H, g, 2.0)
    pe = _tr_exact(H, g, 2.0)
    assert hit and abs(np.linalg.norm(p) - 2.0) < 1e-6 and model(H, g, p) <= model(H, g, pe) + 1e-3 * abs(model(H, g, pe))
