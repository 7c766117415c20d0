"""The on-device stochastic-gradient ascent (Adam, ESWAVS off, same dual directions) from B = 8 restarts with the samples split evenly
over 1, 2, 4 and 8 GPUs (as many as the machine has) in one process: rbo_stochastic_solve_batch_sharded, one handle per GPU. Where the
machine has fewer than 2 or 4 GPUs, 2 and 4 handles share GPU 0 instead: that measures what the gather and broadcast cost, not scaling.

For every GPU count: the wall clock of one call after a warm-up call, the speed-up over one GPU, and the per-iteration cost of the
gather and broadcast (from a separate, profiled call: on the leader, the end of the step kernel minus the end of the last rollout
kernel of the same iteration on any GPU; with one GPU that is the step kernel alone).

Every split must give the final iterates and histories of one handle bit for bit wherever one handle's own result does not depend on
the order in which trajectories are handed out. The script checks that first (one handle, longest-first hand-out on and off). With
more starts than the rollout kernel's start slots it does depend on it: a CTA hands out the starts of a trajectory longest-first by
the evaluation counts of its previous trajectory, and the row splits of the sums follow the number of active slots, so the rounding
of a trajectory follows the CTA's history. Then the script reports the largest difference of the final iterates instead.
Usage: python scripts/sga_sharded_timing.py [shape ...]   (shapes: C4, C2, C2-S5; default all three)"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import __graft_entry__ as g  # noqa: E402

# name: (workload, overrides, restarts, iterations)
# C2-S5: 5 + 2 starts, every start in a slot of its own, so that one handle's result is independent of the hand-out order
SHAPES = {"C4": ("C4", dict(M=4096), 8, 10), "C2": ("C2", dict(M=1024), 8, 10), "C2-S5": ("C2", dict(M=1024, S=5), 8, 10)}
KEYS = ("x_final", "n_iter", "end_status", "fail", "x_hist", "mean_hist", "std_hist", "gmean_hist", "gstd_hist")


def engines(pkg, wl, T, tp, es, n, ndev, lpt=True):
    engs = []
    for i in range(n):
        m0, m1 = wl.M * i // n, wl.M * (i + 1) // n
        e = pkg.RolloutEngine(i if n <= ndev else 0)
        engs.append(e)
        e.set_tuning(lpt=lpt)
        e.set_surrogate(T.fs)
        e.set_normals(tp.rnstream_sequence, m0, m1 - m0)
        e.set_starts(es.inner_solve_xstarts)
    return engs


def gather_gap_ms(prof, iters):
    """Mean over iterations of (end of the step kernel) - (latest end of that iteration's rollout kernels), in ms, from the trace. The
    rollouts of iteration k wait for step k - 1, so they are the ones that end between the two steps."""
    step, roll = [], []
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        if "rbo_sga_step_kernel" in ev.name:
            step.append(ev.time_range.end)
        elif "rbo_rollout_kernel" in ev.name:
            roll.append(ev.time_range.end)
    if len(step) != iters or not roll:
        return float("nan")
    step.sort()
    gaps = []
    for k in range(iters):
        ends = [t for t in roll if (k == 0 or t > step[k - 1]) and t <= step[k]]
        if not ends:
            return float("nan")
        gaps.append(step[k] - max(ends))
    return float(np.mean(gaps)) * 1e-3


def run(pkg, name, counts, ndev):
    import torch
    wname, kw, B, iters = SHAPES[name]
    wl = pkg.problems.make_workload(wname, **kw)
    sur = wl.surrogate()
    T = pkg.Trajectory(sur, pkg.FantasySurrogate(sur, wl.h), start=wl.x0, hypers=wl.theta, horizon=wl.h)
    tp = pkg.TrajectoryParameters(wl.x0, wl.theta, wl.h, wl.M, True, wl.lbs, wl.ubs)
    es = pkg.ExperimentSetup(tp, wl.S)
    dd = np.asfortranarray(np.random.default_rng(7).random((wl.d, wl.h, wl.M)))
    x0s = np.asfortranarray(wl.lbs[:, None] + (wl.ubs - wl.lbs)[:, None] * (0.15 + 0.7 * np.random.default_rng(1).random((wl.d, B))))
    eta, fmini = 0.01, float(np.min(sur.y))
    print(f"{name}: d={wl.d} N={wl.N} h={wl.h} M={wl.M} starts={wl.S}+2, B={B} restarts, {iters} Adam iterations (eta {eta}), ESWAVS off",
          flush=True)

    def call(engs, n_iter):
        return pkg.stochastic_solve_batch_sharded(engs, x0s, wl.theta, wl.lbs, wl.ubs, wl.h, fmini, dual_dirs=dd, optimizer=pkg.Adam(η=eta),
                                                  max_iterations=n_iter, use_eswavs=False)

    rows, results = [], {}
    for n in counts:
        engs = engines(pkg, wl, T, tp, es, n, ndev)
        try:
            call(engs, 1)  # warm-up: module loads, buffers, peer access
            t0 = time.perf_counter()
            r = call(engs, iters)
            wall = time.perf_counter() - t0
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                call(engs, iters)
            gap = gather_gap_ms(prof, iters)
        finally:
            for e in engs:
                e.close()
        results[n] = r
        rows.append((n, n if n <= ndev else 1, wall, r["summary"].kernel_ms, r["summary"].gpu_launches, gap))
    engs = engines(pkg, wl, T, tp, es, 1, ndev, lpt=False)
    try:
        no_lpt = call(engs, iters)
    finally:
        engs[0].close()

    def same(a, b):
        return all(np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f") for k in KEYS)

    order_free = same(no_lpt, results[1])
    t1 = rows[0][2]
    print(f"  {'handles':>7}  {'GPUs':>4}  {'wall ms':>9}  {'per iter ms':>11}  {'leader device ms':>16}  {'launches':>8}  {'speed-up':>8}  "
          f"{'gather+step per iter ms':>23}")
    for n, ng, wall, kms, nl, gap in rows:
        print(f"  {n:7d}  {ng:4d}  {wall * 1e3:9.1f}  {wall / iters * 1e3:11.2f}  {kms:16.1f}  {nl:8d}  {t1 / wall:7.2f}x  {gap:23.3f}")
    if order_free:
        for n in counts:
            assert same(results[n], results[1]), (name, n)
        print(f"  x_final and every history bit-identical over {', '.join(map(str, counts))} handle(s)", flush=True)
    else:
        dx = {n: float(np.max(np.abs(results[n]["x_final"] - results[1]["x_final"]))) for n in counts}
        print(f"  one handle depends on the hand-out order here: longest-first off vs on, max |x_final difference| "
              f"{float(np.max(np.abs(no_lpt['x_final'] - results[1]['x_final']))):.2e}; handles vs 1: "
              + ", ".join(f"{n}: {v:.2e}" for n, v in dx.items()), flush=True)


def main():
    pkg = g.load_package()
    import torch
    ndev = torch.cuda.device_count()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
        gpus = q.stdout.strip().splitlines()
    except OSError:
        gpus = [torch.cuda.get_device_name(i) for i in range(ndev)]
    print(f"{ndev} GPU(s): " + "; ".join(sorted(set(gpus))), flush=True)
    counts = [n for n in (1, 2, 4, 8) if n <= max(ndev, 4)]
    for name in sys.argv[1:] or list(SHAPES):
        run(pkg, name, counts, ndev)


if __name__ == "__main__":
    main()
