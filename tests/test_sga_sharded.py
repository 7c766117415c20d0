"""rbo_stochastic_solve_batch_sharded: the on-device stochastic gradient ascent over the samples of several handles, each holding one shard
of the normals. Every result must equal, bit for bit, rbo_stochastic_solve_batch on one handle that holds all samples, whatever the split,
the order of the handles and the devices. The cases use 5 + 2 starts, so that every start has a start slot of its own: only then are the
rollout kernel's per-trajectory results independent of the order it hands trajectories out (include/rbo.h)."""
import ctypes as C

import numpy as np
import pytest

from test_sga_device import assert_same, c2_case, engine, random_starts, solve


def shard_engines(pkg, h, sur, rn, starts, shards, devices=None, tuning=None):
    """One engine per (m_begin, m_count) of `shards`, in that order (engine 0 leads)."""
    engs = []
    try:
        for i, (m0, mc) in enumerate(shards):
            e = pkg.RolloutEngine(devices[i] if devices else 0)
            engs.append(e)
            if tuning:
                e.set_tuning(**tuning)
            e.set_surrogate(pkg.FantasySurrogate(sur, h))
            e.set_normals(rn, m0, mc)
            e.set_starts(starts)
    except BaseException:
        close(engs)
        raise
    return engs


def close(engs):
    for e in engs:
        e.close()


def solve_sharded(pkg, engs, wl, sur, x0s, dd, **kw):
    return pkg.stochastic_solve_batch_sharded(engs, x0s, wl.theta, wl.lbs, wl.ubs, wl.h, float(np.min(sur.y)), dual_dirs=dd, **kw)


def rollout_outputs(eng, wl, sur, dd, x0):
    """A VALUE_GRAD rollout of the engine's shard at x0 with the matching slice of the dual directions."""
    M, d = eng.m_count, wl.d
    out = dict(v=np.zeros(M), gx=np.zeros((d, M), order="F"), gt=np.zeros((1, M), order="F"), st=np.zeros(M, np.int32), bi=np.zeros(M, np.int32))
    dds = np.asfortranarray(dd[:, :, eng.m_begin:eng.m_begin + M])
    eng.rollout(x0, wl.theta, wl.lbs, wl.ubs, wl.h, float(np.min(sur.y)), out["v"], out["gx"], out["gt"], dual_dirs=dds, status=out["st"],
                best_index=out["bi"])
    return out


def assert_rollouts_like_fresh(pkg, engs, wl, sur, rn, starts, dd):
    """Each engine's next rollout equals, bitwise, a fresh engine's on the same shard."""
    for e in engs:
        fresh = shard_engines(pkg, wl.h, sur, rn, starts, [(e.m_begin, e.m_count)])
        try:
            a, b = rollout_outputs(e, wl, sur, dd, wl.x0), rollout_outputs(fresh[0], wl, sur, dd, wl.x0)
            for k in a:
                assert np.array_equal(a[k], b[k]), k
        finally:
            close(fresh)


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("opt,project", [("adam", False), ("sga", False), ("adam", True)])
def test_one_handle_is_the_single_handle_call(pkg, orc, opt, project):
    wl, sur, rn, starts, dd = c2_case(pkg, orc)
    x0s = random_starts(wl, 4, 1)
    if project:
        x0s[:, 0] = wl.lbs + 1e-3
    make = (lambda: pkg.Adam(η=0.02)) if opt == "adam" else (lambda: pkg.StandardSGA(η=0.02))
    eng = engine(pkg, wl.h, sur, rn, starts)
    try:
        kw = dict(max_iterations=8, use_eswavs=False, project=project)
        a = solve(eng, wl, sur, x0s, dd, optimizer=make(), **kw)
        b = solve_sharded(pkg, [eng], wl, sur, x0s, dd, optimizer=make(), **kw)
        assert_same(a, b)
        for f in ("n_traj", "n_failed", "gpu_launches"):
            assert getattr(a["summary"], f) == getattr(b["summary"], f), f
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("lpt", [True, False])
def test_three_handles_equal_one_with_eswavs(pkg, orc, lpt):
    """Uneven shards handed to the call out of shard order (the leader holds the middle one), restarts picked as in
    test_eswavs_stops_restarts_independently so that some stop early and some reach the cap. B * M_shard > 2 * 148 on every handle:
    the persistent grid wraps and, with lpt, every handle hands out longest-first from its own previous iteration."""
    wl, sur, rn, starts, dd = c2_case(pkg, orc, M=1024)
    M, d, maxit = wl.M, wl.d, 6
    full = engine(pkg, wl.h, sur, rn, starts, tuning=dict(lpt=lpt))
    engs = shard_engines(pkg, wl.h, sur, rn, starts, [(301, 512), (813, 211), (0, 301)], tuning=dict(lpt=lpt))
    try:
        first = solve(full, wl, sur, random_starts(wl, 1, 2), dd, optimizer=pkg.Adam(η=0.02), max_iterations=40, use_eswavs=False)
        cand = np.asfortranarray(np.concatenate([first["x_final"], random_starts(wl, 12, 3)], axis=1))
        probe = solve(full, wl, sur, cand, dd, optimizer=pkg.Adam(η=0.02), max_iterations=maxit, use_eswavs=False)
        q = (M / d) * np.sum(probe["gmean_hist"] ** 2 / probe["gstd_hist"] ** 2, axis=0)
        early_c, capped_c = (q[:-1] < 1).any(axis=0), (q >= 1).all(axis=0)
        assert early_c.any() and capped_c.any(), "the candidates must contain both kinds of restart"
        pick = sorted(list(np.nonzero(early_c)[0][:3]) + list(np.nonzero(capped_c)[0][:3]))
        x0s = np.asfortranarray(cand[:, pick])
        ref = solve(full, wl, sur, x0s, dd, optimizer=pkg.Adam(η=0.02), max_iterations=maxit, use_eswavs=True)
        assert np.any(ref["end_status"] == pkg.SGA_ESWAVS) and np.any(ref["end_status"] == pkg.SGA_MAXIT)
        r = solve_sharded(pkg, engs, wl, sur, x0s, dd, optimizer=pkg.Adam(η=0.02), max_iterations=maxit, use_eswavs=True)
        assert_same(r, ref)
        assert r["summary"].n_traj == ref["summary"].n_traj == int(np.sum(ref["n_iter"])) * M
        assert r["summary"].n_failed == 0
    finally:
        full.close()
        close(engs)


@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["adam", "sga"])
def test_three_handles_uneven_small_shards(pkg, orc, opt):
    """M = 90 split 17 / 43 / 30, given out of shard order; B * M = 360 > 148, so the leader's gathered grid is wider than any one
    handle's launch."""
    wl, sur, rn, starts, dd = c2_case(pkg, orc, M=90)
    x0s = random_starts(wl, 4, 8)
    make = (lambda: pkg.Adam(η=0.02)) if opt == "adam" else (lambda: pkg.StandardSGA(η=0.02))
    full = engine(pkg, wl.h, sur, rn, starts)
    engs = shard_engines(pkg, wl.h, sur, rn, starts, [(60, 30), (0, 17), (17, 43)])
    try:
        for eswavs in (False, True):
            ref = solve(full, wl, sur, x0s, dd, optimizer=make(), max_iterations=7, use_eswavs=eswavs)
            assert_same(solve_sharded(pkg, engs, wl, sur, x0s, dd, optimizer=make(), max_iterations=7, use_eswavs=eswavs), ref)
    finally:
        full.close()
        close(engs)


@pytest.mark.gpu
def test_failure_in_another_handles_shard(pkg, orc):
    """The Matern-1/2 case of test_failure_is_reported_never_averaged with the leader holding the last shard: global sample 0 fails on
    another handle, every restart ends SGA_FAILED naming it, with the status of the single-handle call."""
    from test_gpu_parity import custom_case
    d, N, h, M, S = 3, 18, 2, 16, 3
    sur, _, rn, starts, dd, lbs, ubs, x0 = custom_case(pkg, orc, d, N, h, M, S, "Matern12", (0.6,), "EI", (0.01,))
    theta, fmini = np.array([0.01]), float(np.min(sur.y))
    x0s = np.asfortranarray(np.stack([x0, np.full(d, 0.3)], axis=1))
    full = engine(pkg, h, sur, rn, starts)
    engs = shard_engines(pkg, h, sur, rn, starts, [(11, 5), (0, 6), (6, 5)])
    try:
        ref = full.stochastic_solve_batch(x0s, theta, lbs, ubs, h, fmini, dual_dirs=dd, max_iterations=5)
        r = pkg.stochastic_solve_batch_sharded(engs, x0s, theta, lbs, ubs, h, fmini, dual_dirs=dd, max_iterations=5)
        assert np.all(r["end_status"] == pkg.SGA_FAILED) and np.all(r["fail"][0] == 0)
        assert np.all(r["fail"][1] != 0) and np.array_equal(r["fail"], ref["fail"])
        assert_same(r, ref)
        assert r["summary"].n_failed == r["summary"].n_traj == 2 * M
    finally:
        full.close()
        close(engs)


@pytest.mark.gpu
def test_several_devices(pkg, orc):
    import torch
    ndev = min(torch.cuda.device_count(), 4)
    if ndev < 2:
        pytest.skip(f"{torch.cuda.device_count()} CUDA device(s): the several-device case needs at least 2")
    wl, sur, rn, starts, dd = c2_case(pkg, orc, M=1024)
    x0s = random_starts(wl, 8, 9)
    bounds = [wl.M * i // ndev for i in range(ndev + 1)]
    full = engine(pkg, wl.h, sur, rn, starts)
    engs = shard_engines(pkg, wl.h, sur, rn, starts, [(bounds[i], bounds[i + 1] - bounds[i]) for i in range(ndev)], devices=list(range(ndev)))
    try:
        ref = solve(full, wl, sur, x0s, dd, optimizer=pkg.Adam(η=0.02), max_iterations=6)
        assert_same(solve_sharded(pkg, engs, wl, sur, x0s, dd, optimizer=pkg.Adam(η=0.02), max_iterations=6), ref)
        # the leader on another device, the shards in reverse
        assert_same(solve_sharded(pkg, engs[::-1], wl, sur, x0s, dd, optimizer=pkg.Adam(η=0.02), max_iterations=6), ref)
    finally:
        full.close()
        close(engs)


@pytest.mark.gpu
def test_handle_state_after_the_loop(pkg, orc):
    """Every handle refuses the per-trajectory read-backs, the partial sums and RBO_FLAG_REPLAY_TAPE; its next rollout equals a fresh
    handle's, and so do the partial sums of a non-leader handle after it."""
    import torch
    wl, sur, rn, starts, dd = c2_case(pkg, orc, M=40)
    lib = pkg._lib.load()
    nsum = 1 + 3 * (1 + wl.d + 1) + 2
    dev = torch.zeros(nsum, dtype=torch.float64, device="cuda:0")
    engs = shard_engines(pkg, wl.h, sur, rn, starts, [(25, 15), (0, 25)])
    try:
        solve_sharded(pkg, engs, wl, sur, random_starts(wl, 3, 5), dd, max_iterations=4, use_eswavs=False)
        for e in engs:
            assert lib.rbo_get_results(e.handle.h, pkg._lib.dptr(np.zeros(e.m_count)), None, None, None, None, None) == -3
            assert lib.rbo_partial_sums_host(e.handle.h, pkg._lib.dptr(np.zeros(nsum)), nsum) == -3
            assert lib.rbo_partial_sums_device(e.handle.h, C.c_void_p(dev.data_ptr()), nsum) == -3
            M = e.m_count
            with pytest.raises(pkg.RboError, match=r"librbo error -3"):  # RBO_ERR_STATE
                e.rollout(wl.x0, wl.theta, wl.lbs, wl.ubs, wl.h, float(np.min(sur.y)), np.zeros(M), np.zeros((wl.d, M), order="F"),
                          np.zeros((1, M), order="F"), dual_dirs=np.asfortranarray(dd[:, :, e.m_begin:e.m_begin + M]), replay=True)
        assert_rollouts_like_fresh(pkg, engs, wl, sur, rn, starts, dd)
        # the non-leader handle's partial sums after that rollout are a fresh handle's after the same rollout
        fresh = shard_engines(pkg, wl.h, sur, rn, starts, [(engs[1].m_begin, engs[1].m_count)])
        try:
            sums = []
            for e in (engs[1], fresh[0]):
                rollout_outputs(e, wl, sur, dd, wl.x0)
                sums.append(np.zeros(nsum))
                assert lib.rbo_partial_sums_host(e.handle.h, pkg._lib.dptr(sums[-1]), nsum) == 0
            assert np.array_equal(sums[0], sums[1]) and sums[0][0] > 0
        finally:
            close(fresh)
    finally:
        close(engs)


@pytest.mark.gpu
def test_argument_and_state_errors(pkg, orc):
    """Every check of the sharded call, made before anything is enqueued; afterwards every handle still runs a rollout equal to a fresh
    handle's."""
    wl, sur, rn, starts, dd = c2_case(pkg, orc, M=12)
    lib = pkg._lib.load()
    d, B = wl.d, 2
    x0s = random_starts(wl, B, 6)
    xf, ni, es_, fl = np.zeros((d, B), order="F"), np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros((2, B), np.int32, order="F")
    p, i = pkg._lib.dptr, pkg._lib.iptr

    def call(handles, n=None):
        o = pkg._lib.SgaOpts()
        lib.rbo_default_sga_opts(C.byref(o))
        o.max_iterations = 3
        hs = (C.c_void_p * max(len(handles), 1))(*[h for h in handles])
        rc = lib.rbo_stochastic_solve_batch_sharded(hs, len(handles) if n is None else n, C.byref(o), p(x0s), B, p(wl.theta), 1, p(wl.lbs),
                                                    p(wl.ubs), wl.h, float(np.min(sur.y)), p(dd), p(xf), i(ni), i(es_), i(fl), None, None,
                                                    None, None, None, None)
        return rc, lib.rbo_last_error(handles[0] if handles and handles[0] and n != 0 else None).decode()

    def hv(e):
        return e.handle.h.value

    good = shard_engines(pkg, wl.h, sur, rn, starts, [(0, 5), (5, 7)])
    others = []
    try:
        a, b = good
        assert call([hv(a), hv(b)])[0] == 0
        rc, msg = call([hv(a), hv(b)], n=0)
        assert rc == -1 and "n_handles" in msg
        rc, msg = call([hv(a), None])
        assert rc == -1 and "NULL" in msg
        rc, msg = call([hv(a), hv(a)])
        assert rc == -1 and "same handle" in msg
        # shards that do not tile: a gap, an overlap, an incomplete cover
        gap = shard_engines(pkg, wl.h, sur, rn, starts, [(6, 6)])
        over = shard_engines(pkg, wl.h, sur, rn, starts, [(4, 8)])
        part = shard_engines(pkg, wl.h, sur, rn, starts, [(5, 5)])
        others += gap + over + part
        for extra in (gap[0], over[0], part[0]):
            rc, msg = call([hv(a), hv(extra)])
            assert rc == -1 and "tile" in msg, msg
        # handles that disagree: N, the number of starts, hp1, M_total, d
        wl20, sur20, _, _, _ = c2_case(pkg, orc, M=12, N=20)
        n20 = shard_engines(pkg, wl.h, sur20, rn, starts, [(5, 7)])
        s4 = shard_engines(pkg, wl.h, sur, rn, starts[:, :4], [(5, 7)])
        rn4 = orc.gen_low_discrepancy_sequence(wl.M, wl.d, wl.h + 2)
        hp4 = shard_engines(pkg, wl.h, sur, rn4, starts, [(5, 7)])
        _, _, rn13, _, _ = c2_case(pkg, orc, M=13)
        m13 = shard_engines(pkg, wl.h, sur, rn13, starts, [(5, 8)])
        from test_gpu_parity import custom_case
        sur3, _, rn3, starts3, _, _, _, _ = custom_case(pkg, orc, 3, 24, wl.h, 12, 5, "Matern52", (0.5,), "EI", (0.0,))
        d3 = shard_engines(pkg, wl.h, sur3, rn3, starts3, [(5, 7)])
        others += n20 + s4 + hp4 + m13 + d3
        for extra in (n20[0], s4[0], hp4[0], m13[0], d3[0]):
            rc, msg = call([hv(a), hv(extra)])
            assert rc == -1 and "handle 1 holds" in msg, msg
        # a handle without surrogate, normals or starts
        bare = pkg.RolloutEngine(0)
        others.append(bare)
        rc, msg = call([hv(a), hv(bare)])
        assert rc == -3 and "handle 1 has no surrogate" in msg, msg
        bare.set_surrogate(pkg.FantasySurrogate(sur, wl.h))
        rc, msg = call([hv(a), hv(bare)])
        assert rc == -3 and "handle 1 has no normals" in msg, msg
        bare.set_normals(rn, 5, 7)
        rc, msg = call([hv(a), hv(bare)])
        assert rc == -3 and "handle 1 has no starts" in msg, msg
        # the checks of rbo_stochastic_solve_batch
        with pytest.raises(pkg.RboError, match=r"librbo error -1: rbo_stochastic_solve_batch_sharded: max_iterations"):
            o = pkg._lib.SgaOpts()
            lib.rbo_default_sga_opts(C.byref(o))
            o.max_iterations = 0
            hs = (C.c_void_p * 2)(hv(a), hv(b))
            a.handle.check(lib.rbo_stochastic_solve_batch_sharded(hs, 2, C.byref(o), p(x0s), B, p(wl.theta), 1, p(wl.lbs), p(wl.ubs), wl.h,
                                                                  0.0, p(dd), p(xf), i(ni), i(es_), i(fl), None, None, None, None, None, None))
        assert_rollouts_like_fresh(pkg, good + gap + over + part, wl, sur, rn, starts, dd)
        r = solve_sharded(pkg, good, wl, sur, x0s, dd, max_iterations=3)
        full = engine(pkg, wl.h, sur, rn, starts)
        try:
            assert_same(r, solve(full, wl, sur, x0s, dd, max_iterations=3))
        finally:
            full.close()
    finally:
        close(good)
        close(others)


# ---------------------------------------------------------------------------------------------------------------------------------
def test_symbol_and_argtypes(pkg):
    fn = pkg._lib.load().rbo_stochastic_solve_batch_sharded
    assert fn.restype is C.c_int and len(fn.argtypes) == 22
    assert fn.argtypes[0] is C.POINTER(C.c_void_p) and fn.argtypes[2] is C.POINTER(pkg._lib.SgaOpts)


class _FakeEngine:
    """An engine's shard record only: any other attribute (the handle, the library) fails the test."""

    def __init__(self, m_begin, m_count, M_total, d=3):
        self.m_begin, self.m_count, self.M_total, self.d = m_begin, m_count, M_total, d

    def __getattr__(self, name):
        raise AssertionError(f"the library was reached through engine.{name}")


def test_wrapper_rejects_bad_shards_before_any_library_call(pkg, monkeypatch):
    x0s, th, lb, ub = np.full((3, 2), 0.5), np.zeros(1), np.zeros(3), np.ones(3)
    with pytest.raises(ValueError, match="no engine"):
        pkg.stochastic_solve_batch_sharded([], x0s, th, lb, ub, 2, 0.0)
    for shards in ([(0, 5, 12), (6, 6, 12)],      # gap
                   [(0, 5, 12), (4, 8, 12)],      # overlap
                   [(0, 5, 12), (5, 5, 12)],      # short of M_total
                   [(0, 5, 12), (5, 7, 13)],      # different M_total
                   [(5, 7, 12), (5, 7, 12)]):     # no shard at 0
        with pytest.raises(ValueError, match="do not tile"):
            pkg.stochastic_solve_batch_sharded([_FakeEngine(*s) for s in shards], x0s, th, lb, ub, 2, 0.0)

    def no_library(*a, **k):
        raise AssertionError("the library was called")

    monkeypatch.setattr(pkg.api, "RolloutEngine", no_library)
    d, h, M = 3, 2, 8
    rn = np.zeros((M, d + 1, h + 1), order="F")
    tp = pkg.TrajectoryParameters(np.full(d, 0.5), np.zeros(1), h, M, False, np.zeros(d), np.ones(d), rnstream_sequence=rn)
    for devices in ([], list(range(M + 1))):
        with pytest.raises(ValueError, match="devices"):
            pkg.stochastic_solve_batch(pkg.Adam(), None, tp, None, np.full((d, 2), 0.5), devices=devices)
