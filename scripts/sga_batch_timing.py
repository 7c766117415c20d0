"""The stochastic-gradient ascent (Adam, ESWAVS off, same dual directions) from B restarts, three ways on one GPU:
  (a) B sequential api.stochastic_solve calls (one host round trip per iteration and restart);
  (b) a host loop over rbo_rollout_batch, one launch per iteration for all restarts (the best a caller could do before
      rbo_stochastic_solve_batch): the containers come back, numpy takes the means, api.update_optimizer steps each restart;
  (c) rbo_stochastic_solve_batch: every iteration enqueued on the device, one synchronisation.
Then the cost of an iteration enqueued after every restart has stopped: a Matern-1/2 surrogate on the same sites fails every trajectory
(rbs.jl:537), so every restart stops at its first evaluation and the remaining iterations hand out nothing.
Usage: python scripts/sga_batch_timing.py [shape ...]   (shapes: C2, C3, C4; default all three)"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import __graft_entry__ as g  # noqa: E402

# name: (workload, overrides, restarts, iterations)
SHAPES = {"C2": ("C2", dict(M=64), 8, 50), "C3": ("C3", dict(M=50), 8, 20), "C4": ("C4", dict(M=4096), 8, 10)}


def setup(pkg, wl):
    sur = wl.surrogate()
    fs = pkg.FantasySurrogate(sur, wl.h)
    T = pkg.Trajectory(sur, fs, start=wl.x0, hypers=wl.theta, horizon=wl.h)
    tp = pkg.TrajectoryParameters(wl.x0, wl.theta, wl.h, wl.M, True, wl.lbs, wl.ubs)
    es = pkg.ExperimentSetup(tp, wl.S)
    return sur, T, tp, es


def engine(pkg, wl, T, tp, es):
    eng = pkg.RolloutEngine(0)
    eng.set_surrogate(T.fs)
    eng.set_normals(tp.rnstream_sequence)
    eng.set_starts(es.inner_solve_xstarts)
    return eng


def host_batch_loop(pkg, eng, wl, sur, x0s, dd, iters, eta):
    """(b): one rbo_rollout_batch per iteration, statistics and Adam steps on the host."""
    d, M, B = wl.d, wl.M, x0s.shape[1]
    X = x0s.copy(order="F")
    opts = [pkg.Adam(η=eta) for _ in range(B)]
    vb, gxb, gtb = np.zeros((M, B), order="F"), np.zeros((d, M, B), order="F"), np.zeros((1, M, B), order="F")
    st = np.zeros((M, B), np.int32, order="F")
    fmini = float(np.min(sur.y))
    for _ in range(iters):
        eng.rollout_batch(X, wl.theta, wl.lbs, wl.ubs, wl.h, fmini, vb, gxb, gtb, dual_dirs=dd, status=st)
        if st.any():
            raise pkg.RboError("a trajectory failed")
        for b in range(B):
            pkg.update_optimizer(opts[b], X[:, b], gxb[:, :, b].mean(axis=1))
    return X


def run(pkg, name):
    wname, kw, B, iters = SHAPES[name]
    wl = pkg.problems.make_workload(wname, **kw)
    sur, T, tp, es = setup(pkg, wl)
    dd = np.asfortranarray(np.random.default_rng(7).random((wl.d, wl.h, wl.M)))
    x0s = np.asfortranarray(wl.lbs[:, None] + (wl.ubs - wl.lbs)[:, None] * (0.15 + 0.7 * np.random.default_rng(1).random((wl.d, B))))
    eta, fmini = 0.01, float(np.min(sur.y))
    print(f"{name}: d={wl.d} N={wl.N} h={wl.h} M={wl.M} starts={wl.S}+2, B={B} restarts, {iters} Adam iterations (eta {eta}), ESWAVS off", flush=True)

    # (a) sequential api.stochastic_solve (each call sets up its own handle, as a caller of that API does)
    pkg.stochastic_solve(pkg.Adam(η=eta), T, tp, es, x0s[:, 0], max_iterations=1, use_eswavs=False, dual_directions=dd)  # warm-up
    t0 = time.perf_counter()
    xa = np.stack([pkg.stochastic_solve(pkg.Adam(η=eta), T, tp, es, x0s[:, b], max_iterations=iters, use_eswavs=False,
                                        dual_directions=dd)[0] for b in range(B)], axis=1)
    ta = time.perf_counter() - t0

    eng = engine(pkg, wl, T, tp, es)
    try:
        # (b) host loop over rbo_rollout_batch
        host_batch_loop(pkg, eng, wl, sur, x0s, dd, 1, eta)  # warm-up
        t0 = time.perf_counter()
        xb = host_batch_loop(pkg, eng, wl, sur, x0s, dd, iters, eta)
        tb = time.perf_counter() - t0
        # (c) rbo_stochastic_solve_batch
        eng.stochastic_solve_batch(x0s, wl.theta, wl.lbs, wl.ubs, wl.h, fmini, dual_dirs=dd, optimizer=pkg.Adam(η=eta), max_iterations=1,
                                   use_eswavs=False)  # warm-up
        t0 = time.perf_counter()
        r = eng.stochastic_solve_batch(x0s, wl.theta, wl.lbs, wl.ubs, wl.h, fmini, dual_dirs=dd, optimizer=pkg.Adam(η=eta), max_iterations=iters,
                                       use_eswavs=False)
        tc = time.perf_counter() - t0
    finally:
        eng.close()
    xc = r["x_final"]
    dev_ab = float(np.max(np.abs(xa - xc))); dev_bb = float(np.max(np.abs(xb - xc)))
    print(f"  (a) {B} x api.stochastic_solve      {ta * 1e3:9.1f} ms  ({ta / iters * 1e3:8.2f} ms per iteration of all restarts)")
    print(f"  (b) host loop over rollout_batch  {tb * 1e3:9.1f} ms  ({tb / iters * 1e3:8.2f} ms per iteration)")
    print(f"  (c) rbo_stochastic_solve_batch    {tc * 1e3:9.1f} ms  ({tc / iters * 1e3:8.2f} ms per iteration; device {r['summary'].kernel_ms:.1f} ms, "
          f"{r['summary'].gpu_launches} kernels)   (a)/(c) {ta / tc:.2f}x   (b)/(c) {tb / tc:.2f}x")
    print(f"  max |x_final| difference vs (c): (a) {dev_ab:.2e}  (b) {dev_bb:.2e}", flush=True)

    # empty iterations: every restart stops at its first evaluation (Matern-1/2: every trajectory fails), the rest hand out nothing
    sur12 = pkg.Surrogate(pkg.Matern12([wl.ell]), wl.X, wl.y, capacity=wl.N + wl.capacity_extra, σn2=wl.sigma_n2)
    T12 = pkg.Trajectory(sur12, pkg.FantasySurrogate(sur12, wl.h), start=wl.x0, hypers=wl.theta, horizon=wl.h)
    eng = engine(pkg, wl, T12, tp, es)
    try:
        def failing(n):
            t0 = time.perf_counter()
            rr = eng.stochastic_solve_batch(x0s, wl.theta, wl.lbs, wl.ubs, wl.h, fmini, dual_dirs=dd, max_iterations=n, use_eswavs=False)
            dt = time.perf_counter() - t0
            if not (np.all(rr["end_status"] == pkg.SGA_FAILED) and np.all(rr["n_iter"] == 1)):
                raise RuntimeError(f"not every restart stopped at its first evaluation: {rr['end_status']} {rr['n_iter']}")
            return dt, rr["summary"].kernel_ms
        failing(1)
        K = 50
        w1, k1 = failing(1)
        wK, kK = failing(1 + K)
        print(f"  empty iteration (after every restart stopped): {(kK - k1) / K * 1e3:.1f} us device, {(wK - w1) / K * 1e3:.1f} us wall "
              f"(vs {tc / iters * 1e3:.2f} ms per live iteration)", flush=True)
    finally:
        eng.close()


def main():
    pkg = g.load_package()
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
        gpu = q.stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        gpu = torch.cuda.get_device_name(0)
    print(f"GPU: {gpu}", flush=True)
    for name in sys.argv[1:] or list(SHAPES):
        run(pkg, name)


if __name__ == "__main__":
    main()
