"""Every execution plan of the rollout kernel held to the oracle.

Before each launch the library chooses a plan (choose_plan in csrc/rbo_api.cu): W, the start slots solved in lock-step; RSmax
and RSh, the row splits of the Gram reductions and of the Hessian sums; xsm, the base locations staged in shared memory (1) or
read through L1 (0); vglob, the work matrix in shared memory (0) or in the global scratch of the large-n variant (1). Each choice
is a different code path of rollout_kernel.cu, and results must not depend on it beyond rounding.

The shapes and knobs below give each case a plan that no other test runs, on a device with the B200's 232448 B of opt-in shared
memory per block. Every case reads the plan the library printed (RBO_DEBUG) and fails when it drifted from its target, so a
change to choose_plan cannot silently take the coverage away. Run with -s to see the plans.
"""
import re

import numpy as np
import pytest

from conftest import oracle_problem, relerr
from test_gpu_parity import custom_case, custom_oracle, frac_within, run_custom

pytestmark = pytest.mark.gpu

B200_SMEM_OPTIN = 232448
PLAN_RE = re.compile(r"\[rbo\] plan: W=(\d+) RP=\d+ NR=\d+ RSmax=(\d+) NPmax=\d+ xsm=(\d+) smem=\d+ B \(limit (\d+)\)\n"
                     r"\[rbo\] plan: RSh=(\d+) vglob=(\d+)")
KEYS = ("W", "RSmax", "RSh", "xsm", "vglob")


def plans_since_last_call(capfd):
    """The plans of the launches since the last call, as the library prints them with RBO_DEBUG set."""
    return [dict(W=int(m[0]), RSmax=int(m[1]), xsm=int(m[2]), limit=int(m[3]), RSh=int(m[4]), vglob=int(m[5]))
            for m in PLAN_RE.findall(capfd.readouterr().err)]


def assert_plan(capfd, label, want, launches=1):
    """Every launch since the last call ran the plan `want` (a dict over KEYS); returns that plan."""
    got = plans_since_last_call(capfd)
    assert len(got) == launches, (label, got)
    for p in got:
        assert p["limit"] == B200_SMEM_OPTIN, (f"{label}: the device offers {p['limit']} B of shared memory per block, not the "
                                               f"{B200_SMEM_OPTIN} B of the B200 these shapes were chosen for: choose them again")
        assert {k: p[k] for k in KEYS} == want, f"{label}: ran the plan {p}, not the target {want}"
    with capfd.disabled():
        print(f"\n[plan] {label}: " + " ".join(f"{k}={got[0][k]}" for k in KEYS))
    return got[0]


def plan(W, RSmax, RSh, xsm, vglob):
    return dict(W=W, RSmax=RSmax, RSh=RSh, xsm=xsm, vglob=vglob)


# name: d, N, h, S (Sobol starts; + 2 corner columns), ncols (keep only the first ncols start columns), M, knobs of the case,
# target plan, knobs of another plan the free run is compared with
CASES = {
    "shared, base locations through L1, with gradients": (12, 200, 2, 8, None, 16, {}, plan(5, 1, 2, 0, 0), {"large_n": True}),
    "shared, base locations through L1, RSh > RSmax": (8, 296, 2, 8, None, 16, {}, plan(5, 2, 3, 0, 0), {"large_n": True}),
    "row splits capped at 1": (3, 18, 3, 2, None, 24, {"row_splits": 1}, plan(4, 1, 4, 1, 0), {}),
    "row splits capped at 2": (3, 18, 3, 2, None, 24, {"row_splits": 2}, plan(4, 2, 4, 1, 0), {}),
    "row splits capped at 3": (3, 18, 3, 2, None, 24, {"row_splits": 3}, plan(4, 3, 4, 1, 0), {}),
    "large-n, one start slot": (20, 260, 2, 1, None, 16, {"large_n_slots": 1}, plan(1, 4, 4, 0, 1), {}),
    "large-n, two start columns": (20, 260, 2, 1, 2, 16, {}, plan(2, 4, 4, 0, 1), {"large_n_slots": 1}),
    "large-n, three start columns": (20, 260, 2, 1, None, 16, {}, plan(3, 4, 4, 0, 1), {"large_n_slots": 2}),
    "large-n, 8 start slots": (20, 260, 2, 8, None, 16, {"large_n_slots": 8}, plan(8, 1, 2, 0, 1), {}),
    "large-n, start slots capped at 15 (10 columns)": (20, 260, 2, 8, None, 16, {"large_n_slots": 15}, plan(10, 1, 1, 0, 1), {}),
    "large-n at d = 31": (31, 100, 1, 2, None, 16, {}, plan(4, 1, 1, 0, 1), {"large_n_slots": 2}),
}
# the extended tape (H alpha at every chosen x_j) for one plan of each kernel that reads the base locations through L1
TAPE_EX = {"shared, base locations through L1, with gradients", "large-n, one start slot"}


def ell(d):
    return (0.6 * np.sqrt(d),)


@pytest.mark.parametrize("name", list(CASES))
def test_plan_against_oracle_and_another_plan(pkg, orc, monkeypatch, capfd, name):
    """Matern-5/2 + EI on GP-prior data, value + gradient. (1) Teacher-forced on the oracle's x-path, under the case's plan, to the
    tolerances of test_teacher_forced_step_parity (the kernel matrices here have kappa <= 1e6: kappa * eps ~ 1e-10); with the
    extended tape to the 1e-10 of test_extended_tape_step_level_parity. (2) Free-running under the case's plan against another
    plan on the same inputs, to the thresholds of test_large_n_variant_equals_shared_memory_variant."""
    d, N, h, S, ncols, M, knobs, want, other = CASES[name]
    monkeypatch.setenv("RBO_DEBUG", "1")
    sur, P, rn, starts, dd, lbs, ubs, x0 = custom_case(pkg, orc, d, N, h, M, S, "Matern52", ell(d), "EI", (0.0,), ncols=ncols)
    theta = np.zeros(1)
    ref = P.rollout()
    assert np.all(ref["status"] == 0)
    tex = name in TAPE_EX
    got = run_custom(pkg, sur, rn, starts, dd, lbs, ubs, x0, theta, h, x_forced=np.asfortranarray(ref["xs"][:, 1:, :]), tuning=knobs,
                     tape_ex=tex)
    assert_plan(capfd, name + " (teacher-forced)", want)
    assert np.array_equal(got["status"], ref["status"])
    assert np.array_equal(got["best_index"], ref["best_index"]) and np.array_equal(got["grad_case"], ref["grad_case"])
    assert relerr(got["ys"], ref["ys"]) < 1e-9
    assert relerr(got["gys"], ref["gys"]) < 1e-8
    assert relerr(got["values"], ref["values"]) < 1e-9
    gscale = np.maximum(np.abs(ref["grad_x"]).max(axis=0, keepdims=True), 1e-6)
    assert np.max(np.abs(got["grad_x"] - ref["grad_x"]) / gscale) < 1e-6
    assert np.max(np.abs(got["grad_theta"] - ref["grad_theta"]) / np.maximum(np.abs(ref["grad_theta"]), 1e-6)) < 1e-6
    if tex:
        for key, mine in (("t_mu", "mu"), ("t_sigma", "sigma"), ("t_dmu", "dmu"), ("t_dsigma", "dsigma"), ("t_Halpha", "Halpha")):
            err = np.abs(got["tape_ex"][mine] - ref[key]).max() / max(np.abs(ref[key]).max(), 1e-300)
            assert err < 1e-10, (key, err)
        assert np.abs(got["alphas"] - ref["alphas"]).max() / max(np.abs(ref["alphas"]).max(), 1e-300) < 1e-10
    # free-running, the case's plan against another plan
    free = run_custom(pkg, sur, rn, starts, dd, lbs, ubs, x0, theta, h, tuning=knobs)
    assert_plan(capfd, name + " (free-running)", want)
    assert np.all(free["status"] == 0)
    base = run_custom(pkg, sur, rn, starts, dd, lbs, ubs, x0, theta, h, tuning=other)
    p = plans_since_last_call(capfd)
    assert len(p) == 1 and {k: p[0][k] for k in KEYS} != want, (name, p)
    assert np.all(base["status"] == 0)
    fv, ev = frac_within(free["values"], base["values"], 1e-9, 1.0)
    fx, ex = frac_within(free["xs"], base["xs"], 1e-8, 1.0)
    assert fv >= 0.98 and fx >= 0.98, (ev, ex, p[0])
    gscale = np.maximum(np.abs(base["grad_x"]).max(axis=0, keepdims=True), 1e-6)
    assert np.mean(np.max(np.abs(free["grad_x"] - base["grad_x"]) / gscale, axis=0) < 1e-6) >= 0.97


@pytest.mark.parametrize("d,N,h,Mfull", [(10, 2640, 5, 16384), (20, 2296, 2, 65536)])
def test_largest_n_the_plan_admits(pkg, orc, monkeypatch, capfd, d, N, h, Mfull):
    """The largest N with a rollout plan at d = 10, h = 5 (C3 grown) and at d = 20, h = 2 (C5 grown), 8 + 2 starts: the
    large-n variant with one start slot and one row split, within 32 B / 208 B of the B200's 232448 B. Even there the fantasy
    factor block and its pitch stay in shared memory, so N + 8 has no plan.
    (1) Free-running on 8 sample indices of the full normal stream, then the oracle teacher-forced on the kernel's x-path (it runs
    no inner solves), to the rule of test_c5_shape_parity: 5e-8 on draws and values. With sigma_n^2 = 1e-6 the kernel matrices have
    kappa ~ 9e6 (d = 10) and ~ 7e5 (d = 20), printed below; sigma^2 = k0 - |L^-1 kx|^2 carries kappa * eps ~ 2e-9 relative.
    (2) On the same handle a surrogate 8 observations larger is refused with RBO_ERR_UNSUPPORTED; (3) with the first surrogate set
    back, the handle reproduces the first rollout bitwise."""
    monkeypatch.setenv("RBO_DEBUG", "1")
    want = plan(1, 1, 1, 0, 1)
    sur, _, _, starts, _, lbs, ubs, x0 = custom_case(pkg, orc, d, N, h, 1, 8, "Matern52", ell(d), "EI", (0.0,))
    big = custom_case(pkg, orc, d, N + 8, h, 1, 8, "Matern52", ell(d), "EI", (0.0,), seed=6)[0]
    w = np.linalg.eigvalsh(sur.K[:N, :N])
    kappa = w[-1] / w[0]
    pick = np.sort(np.random.default_rng(3).choice(Mfull, 8, replace=False))
    rn = np.asfortranarray(orc.gen_low_discrepancy_sequence(Mfull, d, h + 1)[pick])
    dd = np.asfortranarray(np.random.default_rng(7).random((d, h, 8)))
    theta, fmini = np.zeros(1), float(np.min(sur.y))
    eng = pkg.RolloutEngine(0)

    def rollout():
        out = dict(values=np.zeros(8), grad_x=np.zeros((d, 8), order="F"), grad_theta=np.zeros((1, 8), order="F"),
                   best_index=np.zeros(8, np.int32), grad_case=np.zeros(8, np.int32), status=np.zeros(8, np.int32))
        eng.rollout(x0, theta, lbs, ubs, h, fmini, out["values"], out["grad_x"], out["grad_theta"], dual_dirs=dd,
                    best_index=out["best_index"], grad_case=out["grad_case"], status=out["status"])
        out.update(eng.tape(h))
        return out

    try:
        eng.set_surrogate(pkg.FantasySurrogate(sur, h))
        eng.set_normals(rn)
        eng.set_starts(starts)
        a = rollout()
        assert_plan(capfd, f"d={d} N={N} h={h}", want)
        eng.set_surrogate(pkg.FantasySurrogate(big, h))
        with pytest.raises(pkg.RboError, match="librbo error -4"):  # RBO_ERR_UNSUPPORTED
            rollout()
        eng.set_surrogate(pkg.FantasySurrogate(sur, h))
        b = rollout()
        assert_plan(capfd, f"d={d} N={N} h={h}, after the refusal", want)
    finally:
        eng.close()
    for key in ("values", "grad_x", "grad_theta", "best_index", "grad_case", "status", "xs", "ys", "gys"):
        assert np.array_equal(a[key], b[key]), key
    assert np.all(a["status"] == 0)
    tf = custom_oracle(orc, sur, x0, lbs, ubs, rn, starts, h, "Matern52", ell(d), "EI", (0.0,), dual_dirs=dd,
                       x_forced=np.asfortranarray(a["xs"][:, 1:, :])).rollout()
    assert np.all(tf["n_evals"] == 0)
    with capfd.disabled():
        print(f"\n[kappa] d={d} N={N}: kernel matrix kappa = {kappa:.2e}, draws max rel err {relerr(a['ys'], tf['ys']):.1e}")
    assert relerr(a["ys"], tf["ys"]) < 5e-8 and relerr(a["gys"], tf["gys"], floor=np.abs(tf["gys"]).max()) < 5e-8
    assert relerr(a["values"], tf["values"]) < 5e-8
    assert np.array_equal(a["grad_case"], tf["grad_case"]) and np.array_equal(a["best_index"], tf["best_index"])
    gscale = np.maximum(np.abs(tf["grad_x"]).max(axis=0, keepdims=True), 1e-6)
    assert np.max(np.abs(a["grad_x"] - tf["grad_x"]) / gscale) < 1e-5


# ---------------------------------------------------------------------------------------------------
# The other entry points on the large-n variant (d = 20, N = 260 with gradients does not fit shared memory)
# ---------------------------------------------------------------------------------------------------
def test_gauss_hermite_on_the_large_n_variant(pkg, orc, monkeypatch, capfd):
    """RBO_FLAG_GAUSS_HERMITE, 3 nodes, h = 2 (M = 27), teacher-forced against the oracle: the assertions of
    test_gauss_hermite_teacher_forced_parity."""
    monkeypatch.setenv("RBO_DEBUG", "1")
    d, N, h, n_nodes = 20, 260, 2, 3
    M = n_nodes ** (h + 1)
    sur, _, _, starts, dd, lbs, ubs, x0 = custom_case(pkg, orc, d, N, h, M, 2, "Matern52", ell(d), "EI", (0.0,))
    nodes, weights = pkg.gausshermite(n_nodes)
    idx = np.asarray(pkg.generate_indices(n_nodes, h + 1)) - 1
    gn, gw = np.asfortranarray(nodes[idx].T), np.asfortranarray(weights[idx].T)
    rn0 = np.zeros((M, d + 1, h + 1), order="F")
    ref = custom_oracle(orc, sur, x0, lbs, ubs, rn0, starts, h, "Matern52", ell(d), "EI", (0.0,), dual_dirs=dd, gh_nodes=gn,
                        gh_weights=gw).rollout()
    eng = pkg.RolloutEngine(0)
    try:
        eng.set_surrogate(pkg.FantasySurrogate(sur, h))
        eng.set_quadrature(gn, gw)
        eng.set_starts(starts)
        vals, gx, gt = np.zeros(M), np.zeros((d, M), order="F"), np.zeros((1, M), order="F")
        bi, gc, st = np.zeros(M, np.int32), np.zeros(M, np.int32), np.zeros(M, np.int32)
        eng.rollout(x0, np.zeros(1), lbs, ubs, h, float(np.min(sur.y)), vals, gx, gt, dual_dirs=dd,
                    x_forced=np.asfortranarray(ref["xs"][:, 1:, :]), best_index=bi, grad_case=gc, status=st, gauss_hermite=True)
        tape = eng.tape(h)
    finally:
        eng.close()
    assert_plan(capfd, "Gauss-Hermite", plan(4, 4, 4, 0, 1))
    assert np.array_equal(st, ref["status"]) and np.array_equal(bi, ref["best_index"]) and np.array_equal(gc, ref["grad_case"])
    assert relerr(tape["ys"], ref["ys"]) < 1e-9 and relerr(tape["gys"], ref["gys"]) < 1e-8
    assert relerr(vals, ref["values"], floor=np.abs(ref["values"]).max()) < 1e-9
    gscale = np.maximum(np.abs(ref["grad_x"]).max(axis=0, keepdims=True), 1e-9)
    assert np.max(np.abs(gx - ref["grad_x"]) / gscale) < 1e-6
    assert np.max(np.abs(gt - ref["grad_theta"]) / np.maximum(np.abs(ref["grad_theta"]), 1e-9)) < 1e-6
    assert (ref["grad_case"] == 3).sum() > 0


def test_batch_on_the_large_n_variant(pkg, orc, monkeypatch, capfd):
    """rbo_rollout_batch, 3 starting points x M = 100: 300 trajectories, more than twice the 148-CTA grid, so that the next launch
    on the same samples hands them out longest-first. The batch equals three rbo_rollout calls bitwise; the longest-first launch
    at moved starting points equals a fresh handle's launch there bitwise (moving them makes a skipped or repeated trajectory
    visible: stale outputs of the first launch would differ)."""
    monkeypatch.setenv("RBO_DEBUG", "1")
    d, N, h, M, B = 20, 260, 2, 100, 3
    want = plan(4, 4, 4, 0, 1)
    sur, _, rn, starts, dd, lbs, ubs, x0 = custom_case(pkg, orc, d, N, h, M, 2, "Matern52", ell(d), "EI", (0.0,))
    rng = np.random.default_rng(3)
    x0s = np.asfortranarray(rng.random((d, B)))
    moved = np.asfortranarray(rng.random((d, B)))
    theta, fmini = np.zeros(1), float(np.min(sur.y))

    def batch(eng, at):
        v, gx, gt, st = np.zeros((M, B), order="F"), np.zeros((d, M, B), order="F"), np.zeros((1, M, B), order="F"), np.zeros((M, B), np.int32, order="F")
        s = eng.rollout_batch(at, theta, lbs, ubs, h, fmini, v, gx, gt, dual_dirs=dd, status=st)
        assert np.all(st == 0)
        return (v, gx, gt), s

    def engine():
        eng = pkg.RolloutEngine(0)
        eng.set_surrogate(pkg.FantasySurrogate(sur, h))
        eng.set_normals(rn)
        eng.set_starts(starts)
        return eng

    eng = engine()
    try:
        eng.set_tuning(lpt=True)
        assert M * B > 2 * min(M * B, eng.num_sms()), "the batch must exceed two waves of the grid for the longest-first order"
        first, s = batch(eng, x0s)
        assert s.gpu_launches == 3  # rollout, statistics, longest-first order for the next launch
        ordered, _ = batch(eng, moved)
        assert_plan(capfd, "batch", want, launches=2)
        for b in range(B):
            v, gx, gt = np.zeros(M), np.zeros((d, M), order="F"), np.zeros((1, M), order="F")
            eng.rollout(x0s[:, b], theta, lbs, ubs, h, fmini, v, gx, gt, dual_dirs=dd)
            assert np.array_equal(v, first[0][:, b]) and np.array_equal(gx, first[1][:, :, b]) and np.array_equal(gt, first[2][:, :, b])
        assert_plan(capfd, "rollout at one starting point", want, launches=B)
    finally:
        eng.close()
    fresh_eng = engine()
    try:
        fresh, _ = batch(fresh_eng, moved)
    finally:
        fresh_eng.close()
    for a, b in zip(ordered, fresh):
        assert np.array_equal(a, b)
    assert not np.array_equal(ordered[0], first[0])


@pytest.mark.parametrize("name,large_n,want", [("C5", False, plan(5, 2, 2, 0, 1)), ("N=260", False, plan(2, 2, 3, 0, 0)),
                                               ("N=260", True, plan(5, 3, 3, 0, 1))])
def test_myopic_solve_plans(pkg, orc, monkeypatch, capfd, name, large_n, want):
    """multistart_base_solve (horizon 0, values only) against the oracle's multistart, 8 + 2 starts, d = 20: at the C5 shape
    (N = 1000, the large-n variant) and at N = 260 on the shared-memory kernel and forced onto the large-n variant. Tolerances of
    test_myopic_multistart_base_solve."""
    monkeypatch.setenv("RBO_DEBUG", "1")
    if name == "C5":
        wl = pkg.problems.make_workload("C5", M=1)
        assert wl.d == 20 and wl.N == 1000 and wl.S == 8
        sur = wl.surrogate()
        starts = orc.generate_initial_guesses(wl.S, wl.lbs, wl.ubs)
        P = oracle_problem(orc, wl, sur, orc.gen_low_discrepancy_sequence(1, wl.d, wl.h + 1), starts, 0)
        lbs, ubs, theta = wl.lbs, wl.ubs, wl.theta
    else:
        sur, P, _, starts, _, lbs, ubs, _ = custom_case(pkg, orc, 20, 260, 0, 1, 8, "Matern52", ell(20), "EI", (0.0,))
        theta = np.zeros(1)
    ref = P.multistart()
    eng = pkg.RolloutEngine(0)
    try:
        eng.set_tuning(large_n=large_n)
        eng.set_surrogate(sur)
        eng.set_starts(starts)
        x, alpha, _ = eng.multistart_base_solve(theta, lbs, ubs)
    finally:
        eng.close()
    assert_plan(capfd, f"myopic {name}" + (", large-n forced" if large_n else ""), want)
    assert relerr(x, ref["x"]) < 1e-7 and np.isclose(alpha, -ref["f"], rtol=1e-8), (x, ref["x"], alpha, -ref["f"])
