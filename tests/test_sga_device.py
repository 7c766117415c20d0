"""rbo_stochastic_solve_batch: stochastic gradient ascent of the rollout acquisition (utils.jl:235-265) from a batch of restarts, every
iteration on the device.

The device loop is held to the host: each recorded iterate is re-evaluated with rbo_rollout (per-trajectory results are bitwise those
of the batched launch, so the statistics differ only in summation order: 1e-13 relative to the summands), and the host mirror's
optimiser step, fed the recorded gradient means, must reproduce the next iterate bit for bit, as must the ESWAVS decisions."""
import ctypes as C

import numpy as np
import pytest

from conftest import relerr


def c2_case(pkg, orc, M=64, N=24, S=5, seed=7):
    """C2-like shape (d = 6, Hartmann-6 data, h = 2)."""
    wl = pkg.problems.make_workload("C2", M=M, N=N, h=2, S=S)
    sur = wl.surrogate()
    rn = orc.gen_low_discrepancy_sequence(wl.M, wl.d, wl.h + 1)
    starts = orc.generate_initial_guesses(wl.S, wl.lbs, wl.ubs)
    dd = np.asfortranarray(np.random.default_rng(seed).random((wl.d, wl.h, wl.M)))
    return wl, sur, rn, starts, dd


def engine(pkg, h, sur, rn, starts, tuning=None):
    eng = pkg.RolloutEngine(0)
    if tuning:
        eng.set_tuning(**tuning)
    eng.set_surrogate(pkg.FantasySurrogate(sur, h))
    eng.set_normals(rn)
    eng.set_starts(starts)
    return eng


def random_starts(wl, B, seed):
    u = np.random.default_rng(seed).random((wl.d, B))
    return np.asfortranarray(wl.lbs[:, None] + (wl.ubs - wl.lbs)[:, None] * (0.15 + 0.7 * u))


def solve(eng, wl, sur, x0s, dd, **kw):
    return eng.stochastic_solve_batch(x0s, wl.theta, wl.lbs, wl.ubs, wl.h, float(np.min(sur.y)), dual_dirs=dd, **kw)


def assert_same(r1, r2):
    for key in ("x_final", "n_iter", "end_status", "fail", "x_hist", "mean_hist", "std_hist", "gmean_hist", "gstd_hist"):
        assert np.array_equal(r1[key], r2[key], equal_nan=r1[key].dtype.kind == "f"), key


def eswavs_lhs(g, sd, M):
    """1 - (M/d) sum(g^2 / var) as api.eswavs evaluates it (> 0: stop)."""
    return 1.0 - (M / len(g)) * np.sum(g**2 / sd**2)


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("opt,project", [("adam", False), ("sga", False), ("adam", True)])
def test_device_loop_replays_on_the_host(pkg, orc, opt, project):
    wl, sur, rn, starts, dd = c2_case(pkg, orc)
    B, iters, M = 4, 8, wl.M
    x0s = random_starts(wl, B, 1)
    if project:
        x0s[:, 0] = wl.lbs + 1e-3  # a restart that starts at the boundary, so that the clamp acts
    make = (lambda: pkg.Adam(η=0.02)) if opt == "adam" else (lambda: pkg.StandardSGA(η=0.02))
    fmini = float(np.min(sur.y))
    eng = engine(pkg, wl.h, sur, rn, starts)
    try:
        r = solve(eng, wl, sur, x0s, dd, optimizer=make(), max_iterations=iters, use_eswavs=False, project=project)
        assert np.all(r["n_iter"] == iters) and np.all(r["end_status"] == pkg.SGA_MAXIT)
        assert r["summary"].n_traj == B * M * iters and r["summary"].n_failed == 0 and r["summary"].kernel_ms > 0
        v, gx, gt, st = np.zeros(M), np.zeros((wl.d, M), order="F"), np.zeros((1, M), order="F"), np.zeros(M, np.int32)
        clamped = False
        for b in range(B):
            o = make()
            x = x0s[:, b].copy()
            for k in range(iters):
                assert np.array_equal(r["x_hist"][:, k, b], x), (b, k)
                eng.rollout(x, wl.theta, wl.lbs, wl.ubs, wl.h, fmini, v, gx, gt, dual_dirs=dd, status=st)
                assert not st.any()
                # summation order only: 1e-13 relative to the magnitude of the summands
                assert abs(r["mean_hist"][k, b] - v.mean()) <= 1e-13 * np.abs(v).mean()
                assert abs(r["std_hist"][k, b] - v.std(ddof=1)) <= 1e-13 * v.std(ddof=1)
                assert np.all(np.abs(r["gmean_hist"][:, k, b] - gx.mean(axis=1)) <= 1e-13 * np.abs(gx).mean(axis=1))
                assert np.all(np.abs(r["gstd_hist"][:, k, b] - gx.std(axis=1, ddof=1)) <= 1e-13 * gx.std(axis=1, ddof=1))
                pkg.update_optimizer(o, x, r["gmean_hist"][:, k, b])
                if project:
                    clamped |= bool(np.any((x < wl.lbs) | (x > wl.ubs)))
                    np.clip(x, wl.lbs, wl.ubs, out=x)
            assert np.array_equal(r["x_final"][:, b], x), b
        assert clamped == project
    finally:
        eng.close()


@pytest.mark.gpu
def test_eswavs_stops_restarts_independently(pkg, orc):
    """Restarts that stop early next to restarts that run to the cap, each decision bitwise api.eswavs's. The starting points are picked
    from a probe run without ESWAVS: where a first ascent ended (the gradient estimate vanishes there) and far from it. M = 1024 makes
    the test sharp enough to keep going where the gradient is large; B * M > 148 SMs, so the persistent grid hands out several
    trajectories per CTA while restarts stop."""
    wl, sur, rn, starts, dd = c2_case(pkg, orc, M=1024)
    M, d, maxit = wl.M, wl.d, 6
    eng = engine(pkg, wl.h, sur, rn, starts)
    try:
        first = solve(eng, wl, sur, random_starts(wl, 1, 2), dd, optimizer=pkg.Adam(η=0.02), max_iterations=40, use_eswavs=False)
        cand = np.asfortranarray(np.concatenate([first["x_final"], random_starts(wl, 12, 3)], axis=1))
        probe = solve(eng, wl, sur, cand, dd, optimizer=pkg.Adam(η=0.02), max_iterations=maxit, use_eswavs=False)
        q = (M / d) * np.sum(probe["gmean_hist"] ** 2 / probe["gstd_hist"] ** 2, axis=0)  # maxit x candidates; < 1: ESWAVS stops
        print("(M/d) sum(g^2/var) per iteration and candidate:\n", np.round(q, 3))
        # the stop test precedes the step, so a restart can also stop at its last evaluation: "early" means before the last one
        early_c = (q[:-1] < 1).any(axis=0)
        capped_c = (q >= 1).all(axis=0)
        assert early_c.any() and capped_c.any(), "the candidates must contain both kinds of restart"
        pick = list(np.nonzero(early_c)[0][:3]) + list(np.nonzero(capped_c)[0][:3])
        x0s = np.asfortranarray(cand[:, sorted(pick)])
        B = x0s.shape[1]
        r = solve(eng, wl, sur, x0s, dd, optimizer=pkg.Adam(η=0.02), max_iterations=maxit, use_eswavs=True)
        for b in range(B):
            decisions = []
            for k in range(int(r["n_iter"][b])):
                g, sd = r["gmean_hist"][:, k, b], r["gstd_hist"][:, k, b]
                assert abs(eswavs_lhs(g, sd, M)) > 1e-12, "a decision within 1e-12 of the threshold: choose other data"
                decisions.append(bool(pkg.eswavs(g, sd**2, M)))
            stop = decisions.index(True) + 1 if True in decisions else None
            if stop is not None:
                assert r["n_iter"][b] == stop and r["end_status"][b] == pkg.SGA_ESWAVS
                assert np.array_equal(r["x_final"][:, b], r["x_hist"][:, stop - 1, b])  # keeps the x at which it stopped
                assert np.all(np.isnan(r["x_hist"][:, stop:, b])) and np.all(np.isnan(r["mean_hist"][stop:, b]))
            else:
                assert r["n_iter"][b] == maxit and r["end_status"][b] == pkg.SGA_MAXIT
        early = r["end_status"] == pkg.SGA_ESWAVS
        print("n_iter", r["n_iter"], "end_status", r["end_status"])
        assert np.array_equal(early, early_c[sorted(pick)]) and np.all(r["n_iter"][early] < maxit)
        assert np.array_equal(r["end_status"] == pkg.SGA_MAXIT, capped_c[sorted(pick)])
        # the restarts that keep going do not depend on the others
        keep = np.nonzero(~early)[0]
        r2 = solve(eng, wl, sur, np.asfortranarray(x0s[:, keep]), dd, optimizer=pkg.Adam(η=0.02), max_iterations=maxit, use_eswavs=True)
        sub = {k: (v[..., keep] if isinstance(v, np.ndarray) else v) for k, v in r.items()}
        assert_same(sub, r2)
    finally:
        eng.close()


@pytest.mark.gpu
def test_agrees_with_the_host_loop(pkg, orc):
    """Each restart matches api.stochastic_solve (one host round trip per iteration, tied to the oracle by
    test_sga_loop_matches_oracle_driven_loop) with the same dual directions, in every iterate."""
    wl, sur, rn, starts, dd = c2_case(pkg, orc)
    iters = 6
    fs = pkg.FantasySurrogate(sur, wl.h)
    T = pkg.Trajectory(sur, fs, start=wl.x0, hypers=wl.theta, horizon=wl.h)
    tp = pkg.TrajectoryParameters(wl.x0, wl.theta, wl.h, wl.M, False, wl.lbs, wl.ubs, rnstream_sequence=rn)
    es = pkg.ExperimentSetup(tp, wl.S)
    x0s = random_starts(wl, 2, 4)
    X, hists = pkg.stochastic_solve_batch(pkg.Adam(η=0.02), T, tp, es, x0s, max_iterations=iters, use_eswavs=False, dual_directions=dd)
    for b in range(2):
        xb, hist = pkg.stochastic_solve(pkg.Adam(η=0.02), T, tp, es, x0s[:, b], max_iterations=iters, use_eswavs=False, dual_directions=dd)
        assert len(hists[b]) == len(hist) == iters
        for (x1, m1, g1), (x2, m2, g2) in zip(hists[b], hist):
            assert relerr(x1, x2) < 1e-9 and abs(m1 - m2) < 1e-9 and relerr(g1, g2) < 1e-9
        assert relerr(X[:, b], xb) < 1e-9


@pytest.mark.gpu
def test_failure_is_reported_never_averaged(pkg, orc):
    """Matern-1/2 makes the joint value/gradient covariance indefinite on every sample (rbs.jl:537): every restart ends at its first
    evaluation, names sample 0 with the status rbo_rollout reports there, and the handle then runs a healthy surrogate correctly."""
    from test_gpu_parity import custom_case
    d, N, h, M, S = 3, 18, 2, 16, 3
    sur, _, rn, starts, dd, lbs, ubs, x0 = custom_case(pkg, orc, d, N, h, M, S, "Matern12", (0.6,), "EI", (0.01,))
    theta, fmini = np.array([0.01]), float(np.min(sur.y))
    x0s = np.asfortranarray(np.stack([x0, np.full(d, 0.3)], axis=1))
    eng = engine(pkg, h, sur, rn, starts)
    try:
        r = eng.stochastic_solve_batch(x0s, theta, lbs, ubs, h, fmini, dual_dirs=dd, max_iterations=5)
        assert np.all(r["end_status"] == pkg.SGA_FAILED) and np.all(r["n_iter"] == 1)
        assert np.array_equal(r["x_final"], x0s)
        assert r["summary"].n_failed == r["summary"].n_traj == 2 * M
        for b in range(2):
            v, gx, gt, st = np.zeros(M), np.zeros((d, M), order="F"), np.zeros((1, M), order="F"), np.zeros(M, np.int32)
            eng.rollout(x0s[:, b], theta, lbs, ubs, h, fmini, v, gx, gt, dual_dirs=dd, status=st)
            assert st[0] != 0 and r["fail"][0, b] == 0 and r["fail"][1, b] == st[0]
        # the same handle, a healthy surrogate of the same dimension: equal to a fresh handle
        good, _, rn2, starts2, dd2, lbs, ubs, x0 = custom_case(pkg, orc, d, N, h, M, S, "Matern52", (0.5,), "EI", (0.0,))
        eng.set_surrogate(pkg.FantasySurrogate(good, h)); eng.set_normals(rn2); eng.set_starts(starts2)
        kw = dict(dual_dirs=dd2, max_iterations=4, use_eswavs=False)
        a = eng.stochastic_solve_batch(x0s, np.zeros(1), lbs, ubs, h, float(np.min(good.y)), **kw)
        assert np.all(a["end_status"] == pkg.SGA_MAXIT)
        fresh = engine(pkg, h, good, rn2, starts2)
        try:
            assert_same(a, fresh.stochastic_solve_batch(x0s, np.zeros(1), lbs, ubs, h, float(np.min(good.y)), **kw))
        finally:
            fresh.close()
    finally:
        eng.close()
    fs = pkg.FantasySurrogate(sur, h)
    T = pkg.Trajectory(sur, fs, start=x0, hypers=theta, horizon=h)
    tp = pkg.TrajectoryParameters(x0, theta, h, M, False, lbs, ubs, rnstream_sequence=rn)
    es = pkg.ExperimentSetup(tp, S)
    with pytest.raises(pkg.RboError, match=r"restart 1, sample 1: PosDefException"):
        pkg.stochastic_solve_batch(pkg.Adam(), T, tp, es, x0s, max_iterations=3, dual_directions=dd)


@pytest.mark.gpu
def test_handle_state_after_the_loop(pkg, orc):
    """Afterwards rollout / rollout_batch equal a fresh handle bitwise; RBO_FLAG_REPLAY_TAPE and the partial sums are refused (the last
    launch did not run every restart, and no statistics ran over it); the large-n variant agrees with the shared-memory one."""
    import torch
    wl, sur, rn, starts, dd = c2_case(pkg, orc)
    M, d, fmini = wl.M, wl.d, float(np.min(sur.y))
    nsum = 1 + 3 * (1 + d + 1) + 2

    def partial_sums(e):
        host, dev = np.zeros(nsum), torch.zeros(nsum, dtype=torch.float64, device="cuda:0")
        rc = (e.lib.rbo_partial_sums_host(e.handle.h, pkg._lib.dptr(host), nsum), e.lib.rbo_partial_sums_device(e.handle.h, C.c_void_p(dev.data_ptr()), nsum))
        torch.cuda.synchronize()
        return rc, host, dev.cpu().numpy()

    x0s = random_starts(wl, 3, 5)
    eng = engine(pkg, wl.h, sur, rn, starts)
    fresh = engine(pkg, wl.h, sur, rn, starts)
    big = engine(pkg, wl.h, sur, rn, starts, tuning=dict(large_n=True))
    try:
        r = solve(eng, wl, sur, x0s, dd, max_iterations=6, use_eswavs=False)
        assert partial_sums(eng)[0] == (-3, -3)  # RBO_ERR_STATE
        with pytest.raises(pkg.RboError, match=r"librbo error -3"):  # RBO_ERR_STATE
            eng.rollout(wl.x0, wl.theta, wl.lbs, wl.ubs, wl.h, fmini, np.zeros(M), np.zeros((d, M), order="F"), np.zeros((1, M), order="F"),
                        dual_dirs=dd, replay=True)
        for e in (eng, fresh):
            out = dict(v=np.zeros(M), gx=np.zeros((d, M), order="F"), gt=np.zeros((1, M), order="F"), st=np.zeros(M, np.int32),
                       bi=np.zeros(M, np.int32), vb=np.zeros((M, 3), order="F"), gxb=np.zeros((d, M, 3), order="F"),
                       gtb=np.zeros((1, M, 3), order="F"), stb=np.zeros((M, 3), np.int32, order="F"))
            e.rollout(wl.x0, wl.theta, wl.lbs, wl.ubs, wl.h, fmini, out["v"], out["gx"], out["gt"], dual_dirs=dd, status=out["st"],
                      best_index=out["bi"])
            out.update(e.tape(wl.h))
            rc, out["sums_host"], out["sums_device"] = partial_sums(e)
            assert rc == (0, 0)
            e.rollout_batch(r["x_final"], wl.theta, wl.lbs, wl.ubs, wl.h, fmini, out["vb"], out["gxb"], out["gtb"], dual_dirs=dd, status=out["stb"])
            if e is eng:
                got = out
        for k, v in out.items():
            assert np.array_equal(got[k], v), k
        rb = solve(big, wl, sur, x0s, dd, max_iterations=3, use_eswavs=False)
        ra = solve(fresh, wl, sur, x0s, dd, max_iterations=3, use_eswavs=False)
        for k in ("x_final", "x_hist", "mean_hist", "gmean_hist"):
            assert relerr(rb[k], ra[k]) < 1e-8, k
        assert np.array_equal(rb["n_iter"], ra["n_iter"])
    finally:
        eng.close(); fresh.close(); big.close()


@pytest.mark.gpu
def test_argument_and_state_errors(pkg, orc):
    from test_gpu_parity import custom_case
    wl, sur, rn, starts, dd = c2_case(pkg, orc, M=8)
    lib = pkg._lib.load()
    d, B, T = wl.d, 2, 4
    x0s = random_starts(wl, B, 6)
    xf, ni, es_, fl = np.zeros((d, B), order="F"), np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros((2, B), np.int32, order="F")
    p = pkg._lib.dptr
    i = pkg._lib.iptr

    def call(eng, nx0=B, **opts):
        o = pkg._lib.SgaOpts()
        lib.rbo_default_sga_opts(C.byref(o))
        o.max_iterations = T
        for k, v in opts.items():
            setattr(o, k, v)
        rc = lib.rbo_stochastic_solve_batch(eng.handle.h, C.byref(o), p(x0s), nx0, p(wl.theta), 1, p(wl.lbs), p(wl.ubs), wl.h,
                                            float(np.min(sur.y)), p(dd), p(xf), i(ni), i(es_), i(fl), None, None, None, None, None, None)
        return rc, lib.rbo_last_error(eng.handle.h).decode()

    eng = pkg.RolloutEngine(0)
    try:
        rc, msg = call(eng)
        assert rc == -3 and "rbo_stochastic_solve_batch" in msg and "surrogate" in msg
        eng.set_surrogate(pkg.FantasySurrogate(sur, wl.h))
        rc, msg = call(eng)
        assert rc == -3 and "normals" in msg
        eng.set_normals(rn)
        rc, msg = call(eng)
        assert rc == -3 and "starts" in msg
        eng.set_starts(starts)
        assert call(eng)[0] == 0
        for kw, word in ((dict(nx0=0), "n_x0"), (dict(max_iterations=0), "max_iterations"), (dict(optimizer=2), "optimizer"),
                         (dict(eta=0.0), "eta"), (dict(eta=-1e-3), "eta"), (dict(eta=float("nan")), "eta")):
            rc, msg = call(eng, **kw)
            assert rc == -1 and word in msg, (kw, msg)
        # the plan limits of rbo_rollout: d = 10, h = 5 admits N = 2640 with 8 + 2 starts, not N = 2648
        dd10 = np.asfortranarray(np.random.default_rng(1).random((10, 5, 2)))
        big, _, rn10, starts10, _, lbs, ubs, _ = custom_case(pkg, orc, 10, 2648, 5, 2, 8, "Matern52", (1.2,), "EI", (0.0,))
        eng.set_surrogate(pkg.FantasySurrogate(big, 5)); eng.set_normals(rn10); eng.set_starts(starts10)
        with pytest.raises(pkg.RboError, match=r"librbo error -4"):  # RBO_ERR_UNSUPPORTED
            eng.stochastic_solve_batch(np.full((10, 2), 0.5), np.zeros(1), lbs, ubs, 5, float(np.min(big.y)), dual_dirs=dd10, max_iterations=2)
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------------------------------------------
def test_default_sga_opts_are_the_reference_defaults(pkg):
    o = pkg._lib.SgaOpts()
    pkg._lib.load().rbo_default_sga_opts(C.byref(o))
    assert (o.optimizer, o.max_iterations, o.use_eswavs, o.project) == (1, 50, 1, 0)  # RBO_OPT_ADAM, utils.jl:244
    assert (o.eta, o.beta1, o.beta2, o.eps) == (1e-3, 0.9, 0.999, 1e-8)  # optimizers.jl:35-40
    a = pkg.Adam()
    assert (a.η, a.β1, a.β2, a.ε) == (o.eta, o.beta1, o.beta2, o.eps)


def test_wrapper_rejects_bad_input_before_any_library_call(pkg, monkeypatch):
    def no_library(*a, **k):
        raise AssertionError("the library was called")

    monkeypatch.setattr(pkg.api, "RolloutEngine", no_library)
    d, h, M = 3, 2, 8
    rn = np.zeros((M, d + 1, h + 1), order="F")
    tp = pkg.TrajectoryParameters(np.full(d, 0.5), np.zeros(1), h, M, False, np.zeros(d), np.ones(d), rnstream_sequence=rn)
    starts = np.full((d, 2), 0.5)
    used = pkg.Adam()
    pkg.update_optimizer(used, np.zeros(d), np.ones(d))
    with pytest.raises(ValueError, match="already taken 1 steps"):
        pkg.stochastic_solve_batch(used, None, tp, None, starts)
    bad = [dict(optimizer=pkg.Adam(), starts=np.full(d, 0.5)),               # a vector, not d x B
           dict(optimizer=pkg.Adam(), starts=np.full((d + 1, 2), 0.5)),      # wrong dimension
           dict(optimizer=pkg.Adam(), starts=np.zeros((d, 0))),              # no restart
           dict(optimizer=pkg.Adam(), starts=starts, dual_directions=np.zeros((d, h, M + 1))),
           dict(optimizer=pkg.Adam(), starts=starts, max_iterations=0),
           dict(optimizer=pkg.StandardSGA(η=0.0), starts=starts)]
    for kw in bad:
        with pytest.raises(ValueError):
            pkg.stochastic_solve_batch(kw.pop("optimizer"), None, tp, None, kw.pop("starts"), **kw)
    with pytest.raises(TypeError):
        pkg.stochastic_solve_batch("adam", None, tp, None, starts)
