"""CPU tests of the host-side mirror and of the C-ABI library's surface (no compute calls without a GPU)."""
import ctypes as C
import os
import re

import numpy as np
import pytest


def test_library_exports_every_declared_symbol(pkg):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "rbo.h")).read()
    declared = set(re.findall(r"\b(rbo_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"rbo_handle"}
    lib = C.CDLL(pkg.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(pkg._lib.SYMBOLS), declared ^ set(pkg._lib.SYMBOLS)
    assert pkg._lib.load().rbo_abi_version() == 2


def test_no_cpu_fallback_without_gpu(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(pkg.RboError, match="no CUDA device"):
        pkg.Handle(0)


def test_product_never_imports_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pdir = os.path.join(root, "rollout-bayesian-optimization_b200")
    for dp, _, files in os.walk(pdir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".jl")):
                txt = open(os.path.join(dp, f)).read()
                for pat in (r"import\s+oracle", r"from\s+oracle", r"#include\s+\"[^\"]*oracle", r"librbo_oracle", r"orc_[a-z_]+\("):
                    assert not re.search(pat, txt), (pat, os.path.join(dp, f))


def test_surrogate_condition_matches_refit(pkg):
    # rbs.jl:214-222: rank-1 extension == fresh factorisation
    rng = np.random.default_rng(0)
    X, y = rng.random((3, 9)), rng.standard_normal(9)
    s = pkg.Surrogate(pkg.Matern52([0.6]), X[:, :6], y[:6], capacity=12)
    for j in range(6, 9):
        pkg.condition(s, X[:, j], y[j])
    t = pkg.Surrogate(pkg.Matern52([0.6]), X, y, capacity=12)
    assert s.observed == 9
    assert np.allclose(s.L[:9, :9], t.L[:9, :9], rtol=1e-10) and np.allclose(s.c[:9], t.c[:9], rtol=1e-8)
    assert pkg.get_observations(s).shape == (12,) and pkg.get_observations(s)[9:].max() == 0.0  # zero padded (Q2)
    fs = pkg.FantasySurrogate(s, 3)
    assert fs.L.shape == (12 + 4, 12 + 4) and np.array_equal(fs.cs[0], s.c[:9])


def test_trajectory_parameters_validation(pkg):
    rn = np.zeros((4, 3, 2))
    tp = pkg.TrajectoryParameters(np.zeros(2), np.zeros(1), 1, 4, False, np.zeros(2), np.ones(2), rnstream_sequence=rn)
    assert tp.rnstream_sequence.flags["F_CONTIGUOUS"]
    with pytest.raises(AssertionError):
        pkg.TrajectoryParameters(np.zeros(2), np.zeros(1), 1, 5, False, np.zeros(2), np.ones(2), rnstream_sequence=rn)
    with pytest.raises(AssertionError):
        pkg.TrajectoryParameters(np.zeros(2), np.zeros(1), 1, 4, False, np.zeros(3), np.ones(2), rnstream_sequence=rn)


def test_adam_and_sga_updates(pkg):
    # optimizers.jl:16-22, 48-75
    x = np.zeros(2)
    pkg.update_optimizer(pkg.StandardSGA(η=0.1), x, np.array([1.0, -2.0]))
    assert np.allclose(x, [0.1, -0.2])
    opt, x = pkg.Adam(), np.zeros(2)
    g = np.array([0.5, -0.25])
    pkg.update_optimizer(opt, x, g)
    assert np.allclose(x, 1e-3 * g / (np.abs(g) + 1e-8)) and opt.t == 1 and len(opt.m) == 2
    assert pkg.eswavs(np.array([1e-3, 1e-3]), np.array([1.0, 1.0]), 10)
    assert not pkg.eswavs(np.array([1.0, 1.0]), np.array([1.0, 1.0]), 10)


def test_finalize_sums_merges_shards(pkg):
    """rbo_finalize_sums (host arithmetic only): merging per-shard [n, n*mean, M2, n*mean^2] blocks reproduces the
    global mean / corrected std -- the algebra behind the multi-GPU all-reduce."""
    lib = pkg._lib.load()
    rng = np.random.default_rng(3)
    d, nth = 3, 1
    shards = [rng.standard_normal((1 + d + nth, n)) + 2.0 for n in (5, 11, 8)]
    tot = np.zeros(1 + 3 * (1 + d + nth) + 2)  # ..., n_failed, watchdog
    for A in shards:
        n = A.shape[1]
        tot[0] += n
        for r in range(A.shape[0]):
            mu = A[r].mean()
            tot[1 + 3 * r] += n * mu
            tot[2 + 3 * r] += ((A[r] - mu) ** 2).sum()
            tot[3 + 3 * r] += n * mu * mu
    allA = np.concatenate(shards, axis=1)
    m, s = C.c_double(), C.c_double()
    gm, gs, tm, ts = np.zeros(d), np.zeros(d), np.zeros(nth), np.zeros(nth)
    p = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    assert lib.rbo_finalize_sums(p(tot), d, nth, C.byref(m), C.byref(s), p(gm), p(gs), p(tm), p(ts)) == 0
    assert np.isclose(m.value, allA[0].mean()) and np.isclose(s.value, allA[0].std(ddof=1))
    assert np.allclose(gm, allA[1:1 + d].mean(axis=1)) and np.allclose(gs, allA[1:1 + d].std(axis=1, ddof=1))
    assert np.allclose(tm, allA[1 + d:].mean(axis=1)) and np.allclose(ts, allA[1 + d:].std(axis=1, ddof=1))
    # a failed trajectory or a watchdog flag on any rank poisons the merged estimate: RBO_ERR_NUMERIC (-5), never a silent number
    for idx in (-2, -1):
        bad = tot.copy(); bad[idx] = 1.0
        assert lib.rbo_finalize_sums(p(bad), d, nth, C.byref(m), C.byref(s), p(gm), p(gs), p(tm), p(ts)) == -5


def test_bench_reference_arm_runs_on_cpu(pkg, orc, tmp_path):
    """`bench.py --impl reference` (the CPU restatement on host cores) needs no GPU and prints the contract's JSON line; its
    --dump-outputs holds the first 16 trajectories of the C3 workload, re-run here through the oracle from the workload's inputs."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample", "16",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "trajectories/s" and line["value"] > 0
    for key in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    v, gx = np.load(tmp_path / "values.npy"), np.load(tmp_path / "grad_x.npy")
    assert v.shape == (16,) and gx.shape == (10, 16) and np.all(np.load(tmp_path / "status.npy") == 0)
    from conftest import oracle_problem, relerr
    wl = pkg.problems.make_workload("C3")
    rn = np.asfortranarray(orc.gen_low_discrepancy_sequence(wl.M, wl.d, wl.h + 1)[:16])
    dd = np.asfortranarray(np.random.default_rng(7).random((wl.d, wl.h, wl.M))[:, :, :16])
    ref = oracle_problem(orc, wl, wl.surrogate(), rn, orc.generate_initial_guesses(wl.S, wl.lbs, wl.ubs), 1, dual_dirs=dd).rollout(tape=False)
    assert relerr(v, ref["values"]) < 1e-12 and relerr(gx, ref["grad_x"], floor=np.abs(ref["grad_x"]).max()) < 1e-12
    assert np.isclose(np.load(tmp_path / "mean.npy")[0], ref["values"].mean(), rtol=1e-12)
    assert np.allclose(np.load(tmp_path / "grad_x_mean.npy"), ref["grad_x"].mean(axis=1), rtol=1e-12, atol=1e-14)


def test_bench_dump_outputs_stays_under_its_size_limit(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float64 .npy files; above the size limit a fixed seeded subset of the sample indices is kept."""
    import bench
    rng = np.random.default_rng(0)
    M, d = 5000, 1  # one gradient row: sample_index is a third of what a kept sample costs, well above the header slack
    per_traj = {"values": rng.random(M), "grad_x": rng.random((d, M)), "status": np.zeros(M, np.int32)}
    estimate = {"mean": np.array([per_traj["values"].mean()])}
    bench.dump_outputs(str(tmp_path / "all"), per_traj, estimate)
    assert np.array_equal(np.load(tmp_path / "all" / "grad_x.npy"), per_traj["grad_x"])
    assert not (tmp_path / "all" / "sample_index.npy").exists()
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 100_000)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), per_traj, estimate)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["grad_x.npy", "mean.npy", "sample_index.npy", "status.npy", "values.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 100_000
    keep = np.load(tmp_path / "a" / "sample_index.npy").astype(np.int64)
    assert len(keep) > M // 4 and np.all(np.diff(keep) > 0)
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "grad_x.npy"), per_traj["grad_x"][:, keep])
