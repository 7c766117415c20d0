#!/usr/bin/env python3
"""bench.py -- rollout trajectories/sec (value + adjoint gradient) of the CUDA path, with the CPU restatement beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C3] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE evaluation of the Monte-Carlo rollout estimator (rollout.jl:279-340): all M trajectories of the
workload (forward rollout + adjoint gradient), sharded over the N GPUs by sample index (strong scaling: M is fixed),
followed by the only collective of the path, one NCCL all-reduce of the partial statistics.
Workload = BASELINE.json configs[2] ("C3": d=10, n=200, h=5, M=16384, 8+2 starts, FP64) -- the configuration the
metric "trajectories/sec (value+grad) at 1/2/4/8 B200" is quoted on.

  value : inputs already resident in HBM, results left on the device (rbo_rollout_device), CUDA events, max over ranks.
  e2e   : the reference-facing call (rbo_set_surrogate + rbo_set_normals + rbo_set_starts + rbo_rollout) with HOST
          buffers in pinned memory: every step re-uploads its inputs and reads the per-trajectory containers back.
  roofline : algorithmic FP64 flops (SURVEY.md 8d formula, with the solver's own evaluation counts) / kernel time,
          against an FP64 FMA micro-benchmark run in this process (MEASURED_PEAKS.json carries no FP64 figure).
  cpu_baseline : oracle/ (C++/OpenMP restatement of the reference -- NOT Julia, which is not installed) on a bounded
          sample of the same workload, all host threads.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as graft  # noqa: E402

METRIC = "rollout trajectories/sec (value+grad)"
UNIT = "trajectories/s"
# dram__bytes_read.sum + dram__bytes_write.sum of one launch of the rollout kernel (ncu --set full, 1 GPU, default M): (bytes, capture)
TRAFFIC_NCU = {"C3": (120366848, "profiles/r3_dram_c3_fullM.csv")}  # algorithmic: 15.7 MB (normals + dual directions); the rest is local-memory (stack / spill) lines written back from L2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps: of the device-resident and the e2e arm, or of --impl reference (the CPU baseline legs beside the "
                         "b200 arm run once; C4's full loop follows --sga-iters)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="C3")
    ap.add_argument("--M", type=int, default=None, help="override the number of trajectories")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--normals", default="reference", choices=["reference", "iid"],
                    help="reference = gen_low_discrepancy_sequence (utils.jl:65-74) on the device; iid = seeded N(0,1)")
    ap.add_argument("--cpu-sample", type=int, default=None, help="trajectories in the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sga-iters", type=int, default=100, help="C4: Adam iterations of the full stochastic-gradient-ascent loop")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (per-trajectory results and the merged estimate) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir, per_traj, estimate):
    """Writes the arrays to out_dir/<name>.npy as float64. per_traj: name -> array whose LAST axis is the sample index (all M of
    them). If these exceed DUMP_LIMIT_BYTES, a fixed seeded subset of the sample indices is kept, listed in sample_index.npy;
    all files together, npy headers included, stay within DUMP_LIMIT_BYTES."""
    os.makedirs(out_dir, exist_ok=True)
    M = next(iter(per_traj.values())).shape[-1]
    per_sample = 8 * sum(a.size // M for a in per_traj.values())
    budget = DUMP_LIMIT_BYTES - 8 * sum(np.size(a) for a in estimate.values()) - 4096 * (len(per_traj) + len(estimate) + 1)
    if per_sample * M > budget:
        # each kept sample also costs its 8-byte entry in sample_index
        keep = np.sort(np.random.default_rng(0).choice(M, budget // (per_sample + 8), replace=False))
        per_traj = {k: a[..., keep] for k, a in per_traj.items()}
        per_traj["sample_index"] = keep
    for name, a in list(per_traj.items()) + list(estimate.items()):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def workload_config(wl, normals, n_gpus):
    return {"workload": f"{wl.name}: d={wl.d} n={wl.N} h={wl.h} M={wl.M} starts={wl.S}+2 Matern52(l={wl.ell}) EI {'value+adjoint-gradient' if wl.with_grad else 'value only'} FP64"
                        + (" -- a step is ONE Adam iteration of the stochastic-gradient-ascent loop (utils.jl:235-265), inputs resident" if wl.name == "C4" else ""),
            "normals": "gen_low_discrepancy_sequence (Sobol + log10 Box-Muller, generated on device)" if normals == "reference" else "iid N(0,1), numpy seed 1906",
            "sharding": f"samples split contiguously over {n_gpus} GPU(s); one all-reduce of 1+3(1+d+ntheta) doubles per step",
            "l2": "L2 flushed between timed steps (256 MiB write)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_oracle_problem(orc, wl, sur, rn, starts, dd, nthreads=0, mode=1):
    return graft._oracle_problem(orc, wl, sur, rn, starts, mode, dual_dirs=dd, nthreads=nthreads)


# trajectories per host core in the CPU sample: about 5-15 s of oracle time on the GPU box's cores
CPU_SAMPLE_PER_CORE = {"C1": 512, "C2": 96, "C3": 48, "C4": 16, "C5": 2}


def workload_inputs(pkg, orc_or_none, wl, normals, M):
    """Full-M normals / dual directions of the workload on the host (the CPU legs slice their sample from these)."""
    if normals == "reference":
        from oracle import oracle as orc
        rn = orc.gen_low_discrepancy_sequence(M, wl.d, wl.h + 1)
    else:
        rn = np.asfortranarray(np.random.default_rng(1906).standard_normal((M, wl.d + 1, wl.h + 1)))
    dd = np.asfortranarray(np.random.default_rng(7).random((wl.d, max(wl.h, 1), M)))
    return rn, dd


def cpu_leg(wl_name, M, sample, nthreads, normals, rn_full=None, dd_full=None):
    """The oracle (CPU restatement of the reference) on the FIRST `sample` sample indices of the workload's own M-trajectory
    normals tensor (so its per-trajectory results are comparable with the GPU arm's), `nthreads` host threads."""
    from oracle import oracle as orc
    pkg = graft.load_package()
    wl = pkg.problems.make_workload(wl_name, M=M)
    sur = wl.surrogate()
    if rn_full is None:
        rn_full, dd_full = workload_inputs(pkg, orc, wl, normals, M)
    rn = np.asfortranarray(rn_full[:sample]); dd = np.asfortranarray(dd_full[:, :, :sample])
    starts = orc.generate_initial_guesses(wl.S, wl.lbs, wl.ubs)
    P = build_oracle_problem(orc, wl, sur, rn, starts, dd, nthreads, mode=1 if wl.with_grad else 0)
    t0 = time.perf_counter()
    r = P.rollout(tape=False)
    dt = time.perf_counter() - t0
    return sample / dt, dt, r


def run_reference(args):
    """--impl reference: the reference's CPU path. Julia is not installed on this image, so this is the C++/OpenMP
    restatement under oracle/ (kind = "port"), all host threads, each step a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pkg = graft.load_package()
    wl_full = pkg.problems.make_workload(args.workload, M=args.M)
    cores = os.cpu_count() or 1
    sample = min(wl_full.M, args.cpu_sample or max(cores * CPU_SAMPLE_PER_CORE.get(args.workload, 16), 16))
    rn_full, dd_full = workload_inputs(pkg, None, wl_full, args.normals, wl_full.M)
    times = []
    for i in range(args.warmup + args.steps):
        tput, dt, r = cpu_leg(args.workload, wl_full.M, sample, cores, args.normals, rn_full, dd_full)
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:  # the last timed step: the first `sample` trajectories of the workload
        keys = ("values", "status") + (("grad_x", "grad_theta") if wl_full.with_grad else ())
        estimate = {"mean": np.array([r["values"].mean()]), "std": np.array([r["values"].std(ddof=1)])}
        if wl_full.with_grad:
            estimate.update(grad_x_mean=r["grad_x"].mean(axis=1), grad_x_std=r["grad_x"].std(axis=1, ddof=1))
        dump_outputs(args.dump_outputs, {k: r[k] for k in keys}, estimate)
    ms = 1e3 * float(np.mean(times))
    value = sample / (ms * 1e-3)
    s1 = max(2, min(sample, sample // cores))
    t1, dt1, _ = cpu_leg(args.workload, wl_full.M, s1, 1, args.normals, rn_full, dd_full)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(wl_full, args.normals, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"first {sample} of {wl_full.M} sample indices per step (oracle/rbo_oracle.cpp, OpenMP dynamic schedule; Julia reference not runnable here)",
                             "single_thread": {"value": t1, "unit": UNIT, "sample": f"first {s1} sample indices, 1 thread (the reference itself is serial, rollout.jl:293)"}},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", local_rank if world > 1 else 0)
    pkg = graft.load_package()

    wl = pkg.problems.make_workload(args.workload, M=args.M)
    M, d, h = wl.M, wl.d, wl.h
    want_grad = bool(wl.with_grad)
    mode = 1 if want_grad else 0
    sga = args.workload == "C4"  # BASELINE config 4: the stochastic-gradient-ascent loop; a step = one optimizer iteration
    m_begin = (M * rank) // world
    m_count = (M * (rank + 1)) // world - m_begin
    sur = wl.surrogate()
    fs = pkg.FantasySurrogate(sur, h)
    fmini = float(np.min(pkg.get_observations(sur)))
    stream = torch.cuda.Stream(dev)  # a real (non-legacy) stream shared by torch's events and the library's launches
    torch.cuda.set_stream(stream)
    eng = pkg.RolloutEngine(dev.index, stream=stream.cuda_stream)
    starts = pkg.generate_initial_guesses(wl.S, wl.lbs, wl.ubs, device=dev.index)
    rng = np.random.default_rng(7)
    dd_full = np.asfortranarray(rng.random((d, max(h, 1), M)))
    dd_host = np.ascontiguousarray(dd_full[:, :, m_begin:m_begin + m_count].transpose(2, 1, 0))  # [m][h][d] == column-major d x h x m
    dd_dev = torch.from_numpy(dd_host).to(dev)

    # ---- resident inputs for the device-timed arm
    eng.set_surrogate(fs)
    if args.normals == "reference":
        eng.generate_normals(M, h + 1, m_begin, m_count)
    else:
        rn_full = np.asfortranarray(np.random.default_rng(1906).standard_normal((M, d + 1, h + 1)))
        eng.set_normals(rn_full, m_begin, m_count)
    eng.set_starts(starts)
    rn_shard = eng.get_normals(h + 1)  # host copy of this rank's normals for the e2e arm (m_count x (d+1) x (h+1))

    nsum = 1 + 3 * (1 + d + 1) + 2  # rows, then [n_failed, watchdog]: they travel through the same all-reduce
    sums = torch.zeros(nsum, dtype=torch.float64, device=dev)
    sums_pin = torch.empty(nsum, dtype=torch.float64, pin_memory=True)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    p = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    x_cur = wl.x0.copy()
    adam = pkg.Adam()  # optimizers.jl:35-40 defaults: eta 1e-3, beta1 .9, beta2 .999, eps 1e-8

    def finalize(fin):
        mean_v, std_v = ctypes.c_double(), ctypes.c_double()
        gm, gs, tm, ts = np.zeros(d), np.zeros(d), np.zeros(1), np.zeros(1)
        eng.lib.rbo_finalize_sums(p(fin), d, 1, ctypes.byref(mean_v), ctypes.byref(std_v), p(gm), p(gs), p(tm), p(ts))
        return mean_v.value, std_v.value, gm, gs

    def device_step():
        eng.rollout_device(x_cur, wl.theta, wl.lbs, wl.ubs, h, fmini, mode, dual_dirs_ptr=dd_dev.data_ptr() if want_grad else None)
        eng.handle.check(eng.lib.rbo_partial_sums_device(eng.handle.h, ctypes.c_void_p(sums.data_ptr()), nsum))
        if world > 1:
            dist.all_reduce(sums)
        if sga:
            # stochastic_solve (utils.jl:235-265): the ascent step needs the gradient estimate on the host -- 37 doubles D2H,
            # then update!(optimizer; x, grad) (optimizers.jl:48-75); inputs stay resident, only x0 changes (common random numbers)
            sums_pin.copy_(sums, non_blocking=True)
            stream.synchronize()
            _, _, gm, _ = finalize(sums_pin.numpy())
            pkg.update_optimizer(adam, x_cur, gm)
            np.clip(x_cur, wl.lbs, wl.ubs, out=x_cur)

    def timed(step_fn, steps, warmup):
        for _ in range(warmup):
            step_fn()
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in ev:
            flush.fill_(1)  # L2 flush between timed steps (not timed)
            a.record(stream)
            step_fn()
            b.record(stream)
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in ev)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(dev.index)
    if rank == 0:
        sampler.start()
    total_ms = timed(device_step, args.steps, max(args.warmup, 3))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # what a caller of the timed path receives from its last step: the per-trajectory containers of this rank's shard
        # (rbo_get_results) and the estimate merged from the all-reduced partial sums; the later arms overwrite both
        res = {"values": np.zeros(m_count), "status": np.zeros(m_count, np.int32)}
        if want_grad:
            res.update(grad_x=np.zeros((d, m_count), order="F"), grad_theta=np.zeros((len(wl.theta), m_count), order="F"))
        eng.handle.check(eng.lib.rbo_get_results(eng.handle.h, pkg._lib.dptr(res["values"]), pkg._lib.dptr(res.get("grad_x")),
                                                 pkg._lib.dptr(res.get("grad_theta")), None, None, pkg._lib.iptr(res["status"])))
        shards = [res]
        if world > 1:
            shards = [None] * world
            dist.all_gather_object(shards, res)
        if rank == 0:
            est_mean, est_std, est_gm, est_gs = finalize(sums.cpu().numpy())
            estimate = {"mean": np.array([est_mean]), "std": np.array([est_std])}
            if want_grad:
                estimate.update(grad_x_mean=est_gm, grad_x_std=est_gs)
            if sga:
                estimate["x"] = x_cur.copy()  # the iterate the last Adam step produced
            dump_outputs(args.dump_outputs, {k: np.concatenate([s[k] for s in shards], axis=-1) for k in res}, estimate)
    ms_per_step = total_ms / args.steps
    value = M / (ms_per_step * 1e-3)

    sga_info = None
    if sga:
        # the whole loop of BASELINE config 4: args.sga_iters Adam iterations from the box centre, ESWAVS stop disabled
        x_cur[:] = wl.x0
        adam = pkg.Adam()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.sga_iters):
            device_step()
        e1.record(stream)
        barrier()
        tl = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tl, op=dist.ReduceOp.MAX)
        sga_info = {"iterations": args.sga_iters, "total_ms": float(tl.item()), "ms_per_iteration": float(tl.item()) / args.sga_iters,
                    "x_final": x_cur.tolist(), "optimizer": "Adam(eta=1e-3, beta1=0.9, beta2=0.999, eps=1e-8), ESWAVS off (utils.jl:235-265, optimizers.jl:35-75)"}
        x_cur[:] = wl.x0

    # statistics of one more step at the workload's x0 (checks the all-reduce path) and accounting from one summarised launch
    sga_saved, sga = sga, False
    device_step()
    sga = sga_saved
    stream.synchronize()
    mean_v, std_v, gm, gs = finalize(sums.cpu().numpy())
    summ = eng.rollout_device(wl.x0, wl.theta, wl.lbs, wl.ubs, h, fmini, mode, dual_dirs_ptr=dd_dev.data_ptr() if want_grad else None, want_summary=True)
    acct = torch.tensor([summ.flops, summ.flops_executed, float(summ.n_evals), float(summ.n_failed), summ.kernel_ms], dtype=torch.float64, device=dev)
    kmax = torch.tensor([summ.kernel_ms, summ.tail_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(acct)
        dist.all_reduce(kmax, op=dist.ReduceOp.MAX)
    acct = acct.cpu().numpy()

    # ---- e2e arm: reference-facing call with host buffers (pinned), H2D + D2H inside the timed region
    def pinned(shape, dtype=np.float64, order="F"):
        n = int(np.prod(shape))
        t = torch.empty(n, dtype=torch.float64 if dtype == np.float64 else torch.int32, pin_memory=True)
        return t.numpy().reshape(shape, order=order), t

    rn_pin, _k1 = pinned(rn_shard.shape); rn_pin[...] = rn_shard
    dd_pin, _k2 = pinned((d, max(h, 1), m_count)); dd_pin[...] = dd_full[:, :, m_begin:m_begin + m_count]
    res_pin, _k3 = pinned((m_count,)); gx_pin, _k4 = pinned((d, m_count)); gt_pin, _k5 = pinned((1, m_count))
    st_pin, _k6 = pinned((m_count,), np.int32)
    starts_pin, _k7 = pinned(starts.shape); starts_pin[...] = starts
    N = sur.observed
    h2d = 8 * (d * N + N * N + 2 * N) + rn_pin.nbytes + starts_pin.nbytes + (dd_pin.nbytes if want_grad else 0)  # X, L, y, c as the caller holds them + normals, starts, dual directions
    d2h = res_pin.nbytes + ((gx_pin.nbytes + gt_pin.nbytes) if want_grad else 0) + st_pin.nbytes + (nsum + 32) * 8

    def e2e_step():
        eng.set_surrogate(fs)                       # fs.X, fs.L, fs.y, fs.cs[1] -> device (inverted and packed on the device)
        eng.set_normals(rn_pin)                     # tp.rnstream_sequence shard
        eng.set_starts(starts_pin)                  # inner_solve_xstarts
        eng.rollout(wl.x0, wl.theta, wl.lbs, wl.ubs, h, fmini, res_pin, gx_pin if want_grad else None, gt_pin if want_grad else None,
                    dual_dirs=dd_pin if want_grad else None, status=st_pin)
        if world > 1:
            eng.handle.check(eng.lib.rbo_partial_sums_device(eng.handle.h, ctypes.c_void_p(sums.data_ptr()), nsum))
            dist.all_reduce(sums)

    e2e_steps = args.steps
    e2e_ms = timed(e2e_step, e2e_steps, 1) / e2e_steps
    e2e_value = M / (e2e_ms * 1e-3)
    ok_e2e = int(st_pin.max()) == 0
    # host wall-clock breakdown of one more e2e step (not part of any reported number)
    brk = {}
    def _t(name, fn):
        t0 = time.perf_counter(); fn(); torch.cuda.synchronize(dev); brk[name] = round(1e3 * (time.perf_counter() - t0), 3)
    _t("set_surrogate", lambda: eng.set_surrogate(fs))
    _t("set_normals", lambda: eng.set_normals(rn_pin))
    _t("set_starts", lambda: eng.set_starts(starts_pin))
    _t("rollout+d2h", lambda: eng.rollout(wl.x0, wl.theta, wl.lbs, wl.ubs, h, fmini, res_pin, gx_pin if want_grad else None, gt_pin if want_grad else None,
                                          dual_dirs=dd_pin if want_grad else None, status=st_pin))
    peak_tf = eng.fp64_peak() if rank == 0 else 0.0
    gpu_vals, gpu_gx = res_pin.copy(), gx_pin.copy()
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()  # the CPU legs below run on rank 0 alone: no idle rank spins on the host cores
    if rank != 0:
        return

    kernel_ms, tail_ms = float(kmax[0].item()), float(kmax[1].item())
    achieved_tf = acct[0] / (kernel_ms * 1e-3) / 1e12  # whole-job flops / slowest rank's kernel time
    achieved_per_gpu = achieved_tf / world
    cpu, parity = None, None
    if not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        sample = min(m_count, args.cpu_sample or max(cores * CPU_SAMPLE_PER_CORE.get(args.workload, 16), 16))
        # the CPU arm runs the FIRST `sample` sample indices of the same normals tensor / dual directions as rank 0's shard,
        # so its per-trajectory results double as a parity check of the benchmarked run
        rn_cpu = np.asfortranarray(rn_shard[:sample]) if m_begin == 0 else None
        tput, dt, r = cpu_leg(args.workload, M, sample, cores, args.normals, rn_cpu if rn_cpu is not None else None, dd_full)
        s1 = max(2, min(sample, sample // cores))
        t1, dt1, _ = cpu_leg(args.workload, M, s1, 1, args.normals, rn_cpu, dd_full)
        cpu = {"value": tput, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"first {sample} of {M} sample indices in {dt:.1f} s (oracle/rbo_oracle.cpp = C++/OpenMP restatement of the reference; Julia not installed)",
               "single_thread": {"value": t1, "unit": UNIT, "sample": f"first {s1} sample indices in {dt1:.1f} s, 1 thread (the reference itself is serial, rollout.jl:293)"}}
        ev = np.abs(gpu_vals[:sample] - r["values"]) / np.maximum(1.0, np.abs(r["values"]))
        parity = {"n": int(sample), "max_rel_err_values": float(ev.max()), "frac_values_within_1e-8": float(np.mean(ev <= 1e-8))}
        if want_grad:
            gsc = np.maximum(np.abs(r["grad_x"]).max(axis=0), 1e-6)
            eg = np.abs(gpu_gx[:, :sample] - r["grad_x"]).max(axis=0) / gsc
            parity.update({"frac_grad_within_1e-5": float(np.mean(eg <= 1e-5)), "max_rel_err_grad": float(eg.max())})
        parity["ok"] = bool(parity["frac_values_within_1e-8"] >= 0.98 and parity.get("frac_grad_within_1e-5", 1.0) >= 0.97)
    traffic = TRAFFIC_NCU.get(args.workload) if (args.M is None and world == 1) else None
    line = {
        "metric": METRIC if want_grad else "rollout trajectories/sec (value only)", "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(wl, args.normals, world),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms,
                "steps": e2e_steps, "all_trajectories_ok": ok_e2e, "host_breakdown_ms": brk},
        "gpu_launches": 4 * args.steps,  # per step: rollout kernel + statistics + longest-first order for the next launch + partial-sums gather
        "roofline": {"bound": "tensor", "pipe": "FP64 (mma.sync.m8n8k4.f64 and DFMA share the same 64 FMA/clk/SM)", "achieved": achieved_per_gpu, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_per_gpu / peak_tf,
                     # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of this kernel on this workload (1 GPU), from the ncu
                     # capture named in traffic_source
                     "traffic": traffic[0] if traffic else None,
                     "traffic_unit": "bytes per launch", "traffic_source": traffic[1] if traffic else None,
                     "kernel": "rbo_rollout_kernel_largen" if args.workload == "C5" else "rbo_rollout_kernel", "kernel_ms": kernel_ms,
                     "flops_per_launch": acct[0] / world, "flops_executed_per_launch": acct[1] / world,
                     "frac_executed": acct[1] / world / (kernel_ms * 1e-3) / 1e12 / peak_tf,
                     "peak_source": "rbo_fp64_peak: dense FP64 FMA micro-benchmark in this process (MEASURED_PEAKS.json has no FP64 figure)",
                     "kernel_share_of_step": kernel_ms / ms_per_step,
                     # tail of the persistent grid on the slowest rank: last CTA to finish minus the median CTA (device globaltimer)
                     "tail_ms": tail_ms, "tail_share_of_kernel": tail_ms / kernel_ms},
        "cpu_baseline": cpu,
        "parity_in_bench": parity,
        "estimate": {"mean": mean_v, "std": std_v, "grad_x_mean": gm.tolist(), "n_failed": int(acct[3]),
                     "acquisition_evals_per_trajectory": acct[2] / M},
    }
    if sga_info:
        line["sga_loop"] = sga_info
    print(json.dumps(line), flush=True)
    if parity is not None and not parity["ok"]:
        print("bench.py: parity_in_bench FAILED: " + json.dumps(parity), file=sys.stderr)
        sys.exit(3)


if __name__ == "__main__":
    main()
