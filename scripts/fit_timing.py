"""Timing of the kernel hyper-parameter fit on the device (rbo_log_marginal_likelihood, rbo_fit_kernel) against the host path, on one GPU.

Data: a Matern-5/2 GP-prior draw (l = 0.7, sigma_n2 = 1e-6) at the sites of C2 (d = 6), C3 (d = 10) and C5 (d = 20)-like shapes, for
N = 50, 200, 1000, 2640, 5000 and 12800 (d = 20 from N = 1000 on).
  * Per likelihood evaluation (value + gradient, warmed-up calls): the call's time (CUDA events on the handle's stream around the call,
    which synchronises once), the time the device spends in kernels (a separate torch.profiler run: the sum of the kernels' durations),
    the share of the call outside kernels (1 - kernel / call: launches, the gaps between them, the read-back and the host's wait), the
    achieved FP64 rate on the count N^3/3 (Cholesky) + N^3/3 (L^-1) + N^3/3 (L^-T L^-1) + O(N^2 d) over the call's time, against
    rbo_fp64_peak measured in the same run, and the share of the kernel time in each phase (kernels grouped by name).
  * Per fit (start l = 0.2, box [0.05, 5]): evaluations and wall time of rbo_fit_kernel, against the host path -- numpy Cholesky and
    gradient driven by scipy L-BFGS-B, then rbo_set_surrogate -- up to N = 2640 (beyond it the host path takes minutes per fit).
  * One BO iteration at C3 (N = 200, d = 10) and C5 (N = 1000, d = 20): (a) host condition + host fit + rbo_set_surrogate against
    (b) rbo_condition + rbo_fit_kernel.
Usage: python scripts/fit_timing.py [N ...]   (writes the report to stdout)"""
import os
import subprocess
import sys
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
from scipy.linalg import cho_factor, cho_solve  # noqa: E402
from scipy.optimize import minimize  # noqa: E402
from scipy.spatial.distance import cdist  # noqa: E402

import __graft_entry__ as g  # noqa: E402

SN2, ELL, START, BOX = 1e-6, 0.7, 0.2, (0.05, 5.0)
HOST_MAX_N = 2640


def matern52(R, l):
    s = np.sqrt(5.0) * R / l
    return (1 + s + s * s / 3.0) * np.exp(-s)


def host_lml(X, y, l):
    """numpy / LAPACK: ll and d ll / d l (the host path the device replaces)."""
    R = cdist(X.T, X.T)
    K = matern52(R, l)
    np.fill_diagonal(K, 1.0)
    K[np.diag_indices_from(K)] += SN2
    cf = cho_factor(K, lower=True)
    a = cho_solve(cf, y)
    ll = -0.5 * y @ a - np.sum(np.log(np.diag(cf[0]))) - 0.5 * len(y) * np.log(2 * np.pi)
    s = np.sqrt(5.0) * R / l
    dK = (s * s / l) * (1 + s) / 3.0 * np.exp(-s)
    g_ = 0.5 * (a @ dK @ a - np.sum(cho_solve(cf, np.eye(len(y))) * dK))
    return ll, g_, cf


def host_fit(X, y, l0):
    nev = [0]

    def f(t):
        nev[0] += 1
        ll, g_, _ = host_lml(X, y, np.exp(t[0]))
        return -ll, np.array([-g_ * np.exp(t[0])])
    r = minimize(f, [np.log(l0)], jac=True, method="L-BFGS-B", bounds=[(np.log(BOX[0]), np.log(BOX[1]))], options=dict(maxiter=30))
    return float(np.exp(r.x[0])), nev[0]


def surrogate_inputs(pkg, X, y, l):
    """What rbo_set_surrogate reads, built without the host Surrogate's dense N x N x d distance tensor."""
    K = matern52(cdist(X.T, X.T), l)
    np.fill_diagonal(K, 1.0 + SN2)
    L = np.linalg.cholesky(K)
    c = cho_solve((L, True), y)
    return SimpleNamespace(observed=len(y), X=np.asfortranarray(X), L=np.asfortranarray(L), y=y, c=c, ψ=pkg.Matern52([l]), σn2=SN2, g=pkg.EI())


def data(N, seed=1906):
    d = 6 if N < 200 else (10 if N < 1000 else 20)
    rng = np.random.default_rng(seed)
    X = rng.random((d, N))
    K = matern52(cdist(X.T, X.T), ELL)
    np.fill_diagonal(K, 1.0 + SN2)
    y = np.linalg.cholesky(K) @ rng.standard_normal(N)
    return d, X, y


def main():
    import torch
    pkg = g.load_package()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print(f"GPU: {q.stdout.strip().splitlines()[0] if q.stdout.strip() else torch.cuda.get_device_name(0)}")
    Ns = [int(a) for a in sys.argv[1:]] or [50, 200, 1000, 2640, 5000, 12800]
    eng = pkg.RolloutEngine(0)
    stream = torch.cuda.Stream()
    eng.lib.rbo_set_stream(eng.handle.h, stream.cuda_stream)  # events on the handle's stream
    peak = eng.fp64_peak()
    print(f"rbo_fp64_peak: {peak:.1f} TFLOP/s (FP64 FMA micro-benchmark, same run)\n")
    print("per likelihood evaluation (value + gradient, Matern-5/2):")
    print(f"{'N':>6} {'d':>3} {'call ms':>9} {'kernel ms':>9} {'outside kernels':>15} {'TFLOP/s':>8} {'of peak':>7}   phases (share of kernel time)")
    fits = []
    for N in Ns:
        d, X, y = data(N)
        start = surrogate_inputs(pkg, X, y, START)
        eng.set_surrogate(start)
        reps = 20 if N <= 1000 else (5 if N <= 5000 else 3)
        for _ in range(2):
            eng.log_marginal_likelihood([ELL])
        dev = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            eng.log_marginal_likelihood([ELL])
            e1.record(stream)
            e1.synchronize()
            dev.append(e0.elapsed_time(e1))
        dm = float(np.median(dev))
        flops = float(N) ** 3 + 2.0 * N * N * d
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA], acc_events=True) as prof:
            eng.log_marginal_likelihood([ELL])
            torch.cuda.synchronize()
        ph = {}
        for ev in prof.events():
            if ev.device_type.name != "CUDA" or "rbo_" not in ev.name:
                continue
            n = ev.name
            key = ("assemble" if "assemble" in n else "cholesky" if ("potrf" in n or "panel" in n or "update" in n) else "L^-1" if "trinv" in n
                   else "K^-1" if "lauum" in n else "gradient pass" if ("grad_kernel" in n or "final" in n) else "a = K^-1 y")
            ph[key] = ph.get(key, 0.0) + ev.time_range.elapsed_us()
        tot = sum(ph.values()) or 1.0
        phs = ", ".join(f"{k} {v / tot:.2f}" for k, v in ph.items())
        km = tot * 1e-3
        print(f"{N:>6} {d:>3} {dm:>9.3f} {km:>9.3f} {1 - km / dm:>15.2f} {flops / dm * 1e-9:>8.2f} {flops / dm * 1e-9 / peak:>7.2f}   {phs}", flush=True)
        # the fit, from the start point
        eng.fit_kernel([BOX[0]], [BOX[1]])  # warm-up
        eng.set_surrogate(start)
        t0 = time.perf_counter()
        r = eng.fit_kernel([BOX[0]], [BOX[1]])
        tf = time.perf_counter() - t0
        host = None
        if N <= HOST_MAX_N:
            t0 = time.perf_counter()
            lh, nh = host_fit(X, y, START)
            eng.set_surrogate(surrogate_inputs(pkg, X, y, lh))
            host = (time.perf_counter() - t0, nh, lh)
        fits.append((N, d, r, tf, host))
    print("\nper fit (start l = 0.2, box [0.05, 5]):")
    print(f"{'N':>6} {'device evals':>12} {'device s':>9} {'l*':>10}   host path (scipy L-BFGS-B + numpy + rbo_set_surrogate)")
    for N, d, r, tf, host in fits:
        hs = f"{host[0]:.3f} s, {host[1]} evals, l* = {host[2]:.6f}, speed-up {host[0] / tf:.1f}x" if host else f"not run (N > {HOST_MAX_N})"
        print(f"{N:>6} {r['n_evals']:>12} {tf:>9.3f} {r['ktheta'][0]:>10.6f}   {hs}")
    print("\none BO iteration: condition on one new observation, refit, make the refit resident")
    for name in ("C3", "C5"):
        N, d = (200, 10) if name == "C3" else (1000, 20)
        _, X, y = data(N + 1)
        x_new, y_new = X[:, N], y[N]
        X, y = X[:, :N], y[:N]
        s = pkg.Surrogate(pkg.Matern52([START]), X, y, capacity=N + 2, σn2=SN2)
        eng.set_surrogate(s)
        t0 = time.perf_counter()
        pkg.condition(s, x_new, y_new)
        lh, _ = host_fit(s.X[:, :N + 1], s.y[:N + 1], START)
        pkg.set_kernel(s, pkg.Matern52([lh]))
        eng.set_surrogate(s)
        ta = time.perf_counter() - t0
        s = pkg.Surrogate(pkg.Matern52([START]), X, y, capacity=N + 2, σn2=SN2)
        eng.set_surrogate(s)
        t0 = time.perf_counter()
        eng.condition(x_new, y_new)
        r = eng.fit_kernel([BOX[0]], [BOX[1]])
        tb = time.perf_counter() - t0
        print(f"  {name} (N = {N} -> {N + 1}, d = {d}): (a) host {ta * 1e3:.1f} ms (l* = {lh:.6f});  (b) device {tb * 1e3:.1f} ms "
              f"(l* = {r['ktheta'][0]:.6f}, {r['n_evals']} evaluations);  {ta / tb:.1f}x")
    eng.close()


if __name__ == "__main__":
    main()
