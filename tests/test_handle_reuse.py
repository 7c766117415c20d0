"""One long-lived handle against fresh ones.

A caller such as the Julia shim keeps one handle per process and only re-uploads what changed, so one handle sees surrogates
of different d and N and launches of different M, horizon and start counts; its device buffers only grow. After every step
below, its results must be bitwise those of the same calls on a fresh handle: the kernel is deterministic, and the
longest-first hand-out does not change results (test_longest_first_schedule_does_not_change_results)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


class Problem:
    """Seeded inputs of one workload: surrogate, normals, starts, dual directions."""

    def __init__(self, pkg, name, seed=0, **kw):
        self.pkg = pkg
        self.wl = wl = pkg.problems.make_workload(name, **kw)
        self.sur = wl.surrogate()
        rng = np.random.default_rng(seed)
        self.rn = np.asfortranarray(rng.standard_normal((wl.M, wl.d + 1, wl.h + 1)))
        self.starts = np.asfortranarray(wl.lbs[:, None] + (wl.ubs - wl.lbs)[:, None] * rng.random((wl.d, wl.S)))
        self.dd = np.asfortranarray(rng.random((wl.d, wl.h, wl.M)))
        self.fmini = float(np.min(self.sur.y))

    def set_surrogate(self, eng):
        eng.set_surrogate(self.pkg.FantasySurrogate(self.sur, self.wl.h))

    def load(self, eng):
        self.set_surrogate(eng)
        eng.set_normals(self.rn)
        eng.set_starts(self.starts)

    def rollout(self, eng, grad=True, M=None, dd=None, **flags):
        """rbo_rollout on eng's resident inputs: every per-trajectory output, the tape and, with tape_ex, the extended tape."""
        wl = self.wl
        M = wl.M if M is None else M
        out = dict(values=np.zeros(M), best_index=np.zeros(M, np.int32), grad_case=np.zeros(M, np.int32), status=np.zeros(M, np.int32))
        if grad:
            out.update(grad_x=np.zeros((wl.d, M), order="F"), grad_theta=np.zeros((1, M), order="F"))
        eng.rollout(wl.x0, wl.theta, wl.lbs, wl.ubs, wl.h, self.fmini, out["values"], out.get("grad_x"), out.get("grad_theta"),
                    dual_dirs=(self.dd if dd is None else dd) if grad else None, best_index=out["best_index"],
                    grad_case=out["grad_case"], status=out["status"], **flags)
        eng.m_count = M  # the wrapper sizes the tape by the samples it uploaded last, normals or quadrature
        tape = eng.tape(wl.h)
        out.update((k, tape[k]) for k in ("xs", "ys", "n_evals", "start_status"))
        if flags.get("tape_ex"):
            out.update(("ex_" + k, v) for k, v in eng.tape_ex(wl.h).items())
        return out


def fresh(pkg, *calls):
    """The calls, in order, on a new handle: the result of each."""
    eng = pkg.RolloutEngine(0)
    try:
        return [call(eng) for call in calls]
    finally:
        eng.close()


def assert_bitwise(got, want, step):
    if isinstance(want, dict):
        assert got.keys() == want.keys(), step
        got, want = [got[k] for k in want], [want[k] for k in want]
    for i, (a, b) in enumerate(zip(got, want)):
        assert a.shape == b.shape and a.tobytes() == b.tobytes(), (step, i)


def test_reused_handle_equals_fresh_handles(pkg):
    eng = pkg.RolloutEngine(0)
    try:
        # 1-2. d = 6 then d = 2 with more trajectories: the extended tape holds M max(h, 1) entries per quantity for the new shape
        p1 = Problem(pkg, "C2", M=64, h=3, S=10)
        p1.load(eng)
        got = p1.rollout(eng, tape_ex=True)
        assert_bitwise(got, fresh(pkg, p1.load, lambda e: p1.rollout(e, tape_ex=True))[1], "C2 d=6")
        p2 = Problem(pkg, "GP:2:0.25", N=12, M=128, h=3)
        p2.load(eng)
        got = p2.rollout(eng, tape_ex=True)
        assert_bitwise(got, fresh(pkg, p2.load, lambda e: p2.rollout(e, tape_ex=True))[1], "GP:2 M=128")

        # 3. horizon and start count change
        p3 = Problem(pkg, "GP:3:0.4", N=37, h=7, M=48, S=3)
        p3.load(eng)
        got = p3.rollout(eng)
        assert_bitwise(got, fresh(pkg, p3.load, p3.rollout)[1], "GP:3 h=7")

        # 4. Gauss-Hermite on the same handle, then Monte Carlo again
        nodes, weights = pkg.gausshermite(2)
        idx = np.asarray(pkg.generate_indices(2, p3.wl.h + 1)) - 1
        Mgh = idx.shape[0]
        dd_gh = np.asfortranarray(np.random.default_rng(1).random((p3.wl.d, p3.wl.h, Mgh)))

        def quadrature(e):
            e.set_quadrature(nodes[idx].T, weights[idx].T)

        def ghq(e):
            return p3.rollout(e, M=Mgh, dd=dd_gh, gauss_hermite=True)

        quadrature(eng)
        got = [ghq(eng), p3.rollout(eng)]
        want = fresh(pkg, p3.load, quadrature, ghq, p3.rollout)[2:]
        assert_bitwise(got[0], want[0], "Gauss-Hermite")
        assert_bitwise(got[1], want[1], "Monte Carlo after Gauss-Hermite")

        # 5. smaller outputs; replaying the x-path of a launch of another shape is a state error; the two-phase call
        p5 = Problem(pkg, "C2", M=32)
        p5.load(eng)
        with pytest.raises(pkg.RboError, match="error -3"):
            p5.rollout(eng, replay=True)
        got = [p5.rollout(eng, grad=False), p5.rollout(eng, replay=True)]
        want = fresh(pkg, p5.load, lambda e: p5.rollout(e, grad=False), lambda e: p5.rollout(e, replay=True))[1:]
        assert_bitwise(got[0], want[0], "value phase")
        assert_bitwise(got[1], want[1], "replay phase")

        # 6. the large-n variant for one launch (its scratch buffers stay reserved), then the shared-memory variant
        for large in (True, False):
            eng.set_tuning(large_n=large)
            got = p5.rollout(eng)
            assert_bitwise(got, fresh(pkg, p5.load, lambda e: e.set_tuning(large_n=large), p5.rollout)[2], f"large_n={large}")

        # 7. another surrogate, then one of smaller d and N conditioned on the device across the 32-row panel boundary (30 -> 34)
        # and, on both handles, on to 100 rows: beyond the capacity of 96 rows, so the canonical form grows with its rows kept
        p5.set_surrogate(eng)
        p7 = Problem(pkg, "GP:2:0.25", N=30, M=32, h=2)
        rng = np.random.default_rng(3)
        newx, newy = rng.random((2, 70)), 0.3 * rng.standard_normal(70)

        def condition(first, last):
            def call(e):
                for j in range(first, last):
                    e.condition(newx[:, j], newy[j])
                return e.get_surrogate()
            return call

        def normals_and_starts(e):
            e.set_normals(p7.rn)
            e.set_starts(p7.starts)

        p7.set_surrogate(eng)
        got = [condition(0, 4)(eng)]
        normals_and_starts(eng)
        got += [p7.rollout(eng), condition(4, 70)(eng)]
        want = fresh(pkg, p7.set_surrogate, condition(0, 4), normals_and_starts, p7.rollout, condition(4, 70))
        assert_bitwise(got[0], want[1], "conditioned to 34 rows")
        assert_bitwise(got[1], want[3], "rollout on the conditioned surrogate")
        assert_bitwise(got[2], want[4], "conditioned to 100 rows")
        N = p7.wl.N
        Xh = np.concatenate([p7.sur.X[:, :N], newx], axis=1)
        yh = np.concatenate([p7.sur.y[:N], newy])
        X, y, c = got[2]
        assert np.array_equal(X, Xh) and np.array_equal(y, yh)
        ref = pkg.Surrogate(pkg.Matern52([p7.wl.ell]), Xh, yh, capacity=N + 75, decision_rule=pkg.EI(), σn2=p7.wl.sigma_n2)
        assert np.max(np.abs(c - ref.c[:N + 70])) < 1e-7 * np.abs(ref.c[:N + 70]).max()
    finally:
        eng.close()
