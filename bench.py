#!/usr/bin/env python
"""bench.py -- headline benchmark: Pallas MSM points/s over resident generators (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--log-n L] [--impl ours|reference]
  torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU)

A "step" is one MSM  sum_i s_i * G_i  over n = 2^L points per GPU (default 2^24, the size the metric is quoted on;
1 GiB of affine bases + 512 MiB of scalars per GPU, so every step streams inputs far larger than the 126 MB L2).
With N > 1 the MSM is sharded by point slice behind the C ABI (halo_comm_*, csrc/comm.cu: every rank holds its own
2^L-point slice of an N * 2^L-point MSM -- weak scaling -- and the ranks' partials meet in one ncclAllGather on the
library's stream).

`value`       points/s, inputs resident in HBM, CUDA events on the library's stream, max over ranks; two steps in flight
              (submit / collect over device-resident scalars); the strictly sequential figure is `sequential_calls`.
`e2e`         same metric through the C ABI with HOST scalars: H2D of the step's scalars and D2H of the partials inside
              the timed region.  Pipelined from pinned memory (`value`), the blocking drop-in call from pinned memory
              (`blocking_call`) and from PAGEABLE memory (`blocking_call_pageable`: what a Rust Vec<Fr> is).
`variable_base` the same MSM without the precomputed multiples of the generators (the path of point_dot / IPA rounds).
`roofline`    integer pipe (IMAD) for the dominant phase, the bucket accumulation; peak measured in-run by the library's
              IMAD microbenchmark (MEASURED_PEAKS.json carries no integer figure).  `frac` uses SURVEY 8(d)'s canonical
              accounting (c = 16: 16 windows x 10 modmul per point); `executed` restates it with the multiplications the
              kernels actually issue.
`strong_scaling` ONE MSM of 2^16 .. 2^24 points sharded over the N GPUs (BASELINE config 5), ms / points/s / fraction of
              the N-GPU integer roofline per size, each result checked against the oracle.
`oracle_match` the timed result equals the CPU oracle's (N = 1: its arkworks-shaped Pippenger at the same 2^24 size -- the
              same run is the `cpu_baseline` -- and the discrete-log property; N > 1: the discrete-log property per slice).
`cpu_baseline` / `--impl reference`: the reference's arkworks algorithm restated in C (oracle/), timed on the host cores at
              the SAME size (one 2^24-point MSM per step).  The reference itself is Rust and cannot run here.

`--dump-outputs DIR` writes the result of the last timed step (rank 0; either arm) to DIR/msm_result.npy, so that two builds
run with the same arguments (same derived generators, same seeded scalars) can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CURVE = os.environ.get("HALO_B200_CURVE", "pallas")  # "vesta": the other half of the cycle, same kernels (DESIGN section 7)
METRIC = f"{CURVE}_msm_points_per_s"
UNIT = "points/s"
IMAD_PER_MODMUL = 136  # SURVEY.md section 8(d): 2 N^2 + N for N = 8 limbs
CANON_W = 16           # canonical c = 16 -> 16 windows x 10 modmul per point in the bucket accumulation
SCALAR_SEED = 4        # SURVEY 8(d) config 5


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def make_config(log_n, world):
    """The workload, identical for both arms (`--impl ours` and `--impl reference`)."""
    n = 1 << log_n
    return {"workload": f"{CURVE}_msm_2^{log_n}_per_gpu", "points_per_gpu": n, "total_points": n * world,
            "bases": "derived generators G_i (main.rs:18-45 rule)", "scalars": f"uniform 254-bit, numpy PCG64 seed {SCALAR_SEED} + rank",
            "parallelism": f"point-slice x{world}, one all-gather per MSM" if world > 1 else "single GPU",
            "l2": "inputs_exceed_l2 (>= 1.5 GiB streamed per step)"}


def bench_scalars(n, seed_offset):
    """Seeded synthetic scalars as Montgomery limbs: any 4-limb value below 2^254 < r is the Montgomery form of some scalar."""
    rng = np.random.Generator(np.random.PCG64(SCALAR_SEED + seed_offset))
    a = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)
    return a


def dump_outputs(out_dir, point_jac):
    """Writes an MSM result as DIR/msm_result.npy: float64 [2, 8], the affine x and y as canonical integers in eight
    little-endian 32-bit words each (exact in float64).  Affine, because two builds may return different Jacobian
    representatives of the same point; (0, 0) is not on y^2 = x^3 + 5 and stands for the point at infinity."""
    from oracle import oracle as O

    xy = O.pt_to_affine_ints(point_jac) or (0, 0)
    words = np.array([[(v >> (32 * i)) & 0xFFFFFFFF for i in range(8)] for v in xy], dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "msm_result.npy"), words)


class ClockSampler(threading.Thread):
    """Samples SM clock, power and clock-event reasons of one GPU during a timed region (B200_PROFILING.md recipe): in-process
    NVML every 10 ms when the bindings load (a 0.6 s timed region gets ~60 samples), else `nvidia-smi` every 200 ms."""

    def __init__(self, index, uuid=None):
        super().__init__(daemon=True)
        self.index, self.uuid, self.rows, self.stop_flag = index, uuid, [], threading.Event()
        self.source = "nvidia-smi"

    def _nvml_handle(self):
        import pynvml as nv

        nv.nvmlInit()
        if self.uuid:
            try:
                return nv, nv.nvmlDeviceGetHandleByUUID(("GPU-" + str(self.uuid)).encode())
            except Exception:
                pass
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        phys = self.index
        if vis and all(v.strip().isdigit() for v in vis.split(",")):
            phys = int(vis.split(",")[self.index])
        return nv, nv.nvmlDeviceGetHandleByIndex(phys)

    def _run_nvml(self):
        nv, h = self._nvml_handle()
        names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap))
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)  # any failure lands in the fallback before the first row
        self.source = "nvml"
        while not self.stop_flag.is_set():
            try:
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                self.rows.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), mx, nv.nvmlDeviceGetPowerUsage(h) / 1000.0,
                                  [name for name, bit in names if mask & bit]))
            except Exception:
                pass
            self.stop_flag.wait(0.01)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                r = [c.strip() for c in out.split(",")]
                if len(r) >= 7 and r[0].isdigit():
                    why = [name for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7])
                           if v.lower().startswith("active")]
                    self.rows.append((int(r[0]), int(r[1]) if r[1].isdigit() else 0, float(r[2]) if r[2].replace(".", "").isdigit() else 0.0, why))
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            self.source = "nvidia-smi"
            self._run_smi()

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        rows = list(self.rows)
        sm = sorted(r[0] for r in rows)
        pw = sorted(r[2] for r in rows)
        reasons = sorted({w for r in rows for w in r[3]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_mhz_min": sm[0] if sm else None,
                "sm_max_mhz": max((r[1] for r in rows), default=None), "power_w_median": pw[len(pw) // 2] if pw else None,
                "power_w_max": pw[-1] if pw else None, "reasons": reasons, "samples": len(rows), "source": self.source}


def host_threads():
    """All host cores this process may use.  torchrun exports OMP_NUM_THREADS=1; the CPU arm must not inherit that."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(n)  # read by libgomp when the oracle library is loaded
    return n


def run_reference(args):
    """The reference's CPU path (arkworks-shaped Pippenger restated in oracle/halo_oracle.c) on the SAME workload: one MSM of
    2^log_n derived generators x seeded scalars per step, all host threads (windows x point chunks)."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    threads = host_threads()
    from oracle import oracle as O

    n = 1 << args.log_n
    t0 = time.perf_counter()
    bases = O.derive_points_fast(2, n)  # setup, untimed
    setup_s = time.perf_counter() - t0
    scalars = bench_scalars(n, 0)
    for _ in range(min(args.warmup, 1)):
        O.msm_affine(bases, scalars, threads=threads)
    t = time.perf_counter()
    for _ in range(args.steps):
        res = O.msm_affine(bases, scalars, threads=threads)
    dt = (time.perf_counter() - t) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    ok = bool(O.pt_eq(res, O.msm_derived_by_dlog(0, scalars, threads=threads)))
    val = n / dt
    sample = (f"one MSM of 2^{args.log_n} points per step = the full per-GPU workload, {args.steps} timed steps after "
              f"{min(args.warmup, 1)} warm-up; field core in MULX / ADC assembly, windows x point chunks over {threads} host threads"
              + (f"; with {world} GPUs the other arm runs {world} such slices at once, this arm times one slice" if world > 1 else ""))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32x8 (255-bit Montgomery)", "data": "synthetic",
        "config": make_config(args.log_n, world),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "self_check": ok, "setup_s": setup_s,
        "note": "reference is Rust/arkworks (no toolchain here): timed arm is its algorithm restated in C (oracle/), kind=port",
    }), flush=True)


def run_ours(args):
    import torch
    import torch.distributed as dist

    import halo_accumulation_b200 as H
    from halo_accumulation_b200 import parallel

    rank, world, local = dist_env()
    if not os.path.exists(os.path.join(ROOT, "halo-accumulation_b200", "lib", "libhalo_b200.so")) and rank == 0:
        H.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL's own log lines (NCCL_DEBUG, if the launcher sets it) are left alone: the one JSON line is printed last
        dist.init_process_group("nccl", device_id=dev)
    n = 1 << args.log_n
    ctx = H.Context(local, n)
    comm = parallel.make_comm(ctx, None, dev) if world > 1 else None
    n_global = n * world
    first = rank * n
    t0 = time.perf_counter()
    if comm:
        comm.derive_generators(n_global)  # this rank's point slice of the N * n point MSM
    else:
        ctx.derive_generators(n)
    derive_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    if not args.no_precompute:  # FIXED-base tables: multiples 2^(off_w) G_i of the resident generators (setup)
        comm.precompute_generators(0) if comm else ctx.precompute_generators(0)
    precompute_s = time.perf_counter() - t0
    h_page = bench_scalars(n, rank)                    # pageable host memory (numpy)
    h_scalars = torch.empty((n, 4), dtype=torch.int64, pin_memory=True)
    h_scalars.copy_(torch.from_numpy(h_page.view(np.int64)))
    d_scalars = h_scalars.to(dev)
    torch.cuda.synchronize()
    h_np = h_scalars.numpy().view(np.uint64)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxr(*vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def step_resident():
        if comm:
            return comm.msm_gens_sharded_resident(d_scalars.data_ptr(), n, n_global)
        return ctx.msm_gens_resident(d_scalars.data_ptr(), n)

    def step_e2e(h):
        if comm:
            return comm.msm_gens_sharded(h, n_global)
        return ctx.msm_gens(h)

    def finish(part):
        return comm.allgather_sum(part) if comm else part

    # ---- resident, strictly sequential blocking calls ----
    for _ in range(args.warmup):
        res_seq = step_resident()
    barrier()
    ctx.timer_start()
    for _ in range(args.steps):
        res_seq = step_resident()
    seq_ms = max(ctx.timer_stop(), 0.0) / args.steps

    # ---- resident (`value`): K MSM steps over scalars resident in HBM, two steps in flight (halo_msm_gens_submit_resident /
    # _collect): the counting sort of step k+1 (L2-atomic bound) runs beside the bucket accumulation of step k ----
    def run_pipelined(k_steps, submit):
        t = submit()
        out = None
        for k in range(k_steps):
            nxt = submit() if k + 1 < k_steps else None
            out = finish(ctx.msm_gens_collect(t))
            t = nxt
        return out

    run_pipelined(max(args.warmup, 2), lambda: ctx.msm_gens_submit_resident(d_scalars.data_ptr(), n))
    barrier()
    dev_uuid = getattr(torch.cuda.get_device_properties(local), "uuid", None)
    sampler = ClockSampler(local, dev_uuid)
    sampler.start()
    l0 = ctx.kernel_launches()
    ctx.timer_start()
    w0 = time.perf_counter()
    res = run_pipelined(args.steps, lambda: ctx.msm_gens_submit_resident(d_scalars.data_ptr(), n))
    ev_ms = ctx.timer_stop()
    barrier()
    wall_ms = (time.perf_counter() - w0) * 1e3
    launches = ctx.kernel_launches() - l0
    clocks = sampler.summary()
    ms_step = max(ev_ms, 0.0) / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res)  # `res` is the collected (and, with N > 1, all-gathered) result of the last step

    # ---- e2e (host buffers through the C ABI) ----
    def timed_host(f, steps, warm):
        for _ in range(warm):
            out = f()
        barrier()
        w = time.perf_counter()
        for _ in range(steps):
            out = f()
        barrier()
        return out, (time.perf_counter() - w) * 1e3 / steps

    res_e, e2e_sync_ms = timed_host(lambda: step_e2e(h_np), args.steps, max(args.warmup, 1))        # blocking call, pinned
    res_pg, e2e_page_ms = timed_host(lambda: step_e2e(h_page), max(3, args.steps // 2), 1)          # blocking call, pageable
    run_pipelined(max(args.warmup, 2), lambda: ctx.msm_gens_submit(h_np))                           # both slots allocate on first use
    barrier()
    w0 = time.perf_counter()
    res_p = run_pipelined(args.steps, lambda: ctx.msm_gens_submit(h_np))
    barrier()
    e2e_ms = (time.perf_counter() - w0) * 1e3 / args.steps

    # ---- per-phase profile of the FIXED-base path (dominant phase: bucket accumulation), CUDA events on the library's stream ----
    ctx.set_profiling(True)
    acc_ms = []
    phase_sampler = ClockSampler(local, dev_uuid)
    phase_sampler.start()
    for _ in range(max(3, min(args.steps, 5))):
        ctx.msm_gens_resident(d_scalars.data_ptr(), n)
        acc_ms.append(ctx.last_msm_timings())
    phase_clocks = phase_sampler.summary()
    ctx.set_profiling(False)
    phases = {k: float(np.mean([t[k] for t in acc_ms])) for k in acc_ms[0]}

    # ---- variable base: the same MSM without the tables of precomputed multiples ----
    ctx.set_fixed_base(False)
    var_steps = max(3, args.steps // 2)
    res_var = step_resident()
    barrier()
    ctx.timer_start()
    for _ in range(var_steps):
        res_var = step_resident()
    var_ms = max(ctx.timer_stop(), 0.0) / var_steps
    ctx.set_fixed_base(True)

    ms_step, e2e_ms, wall_step, phases["accumulate"], e2e_sync_ms, seq_ms, var_ms, e2e_page_ms = maxr(
        ms_step, e2e_ms, wall_ms / args.steps, phases["accumulate"], e2e_sync_ms, seq_ms, var_ms, e2e_page_ms)
    same = all(H.points_equal(res, x) for x in (res_e, res_p, res_seq, res_var, res_pg))

    # ---- the oracle's verdict on the timed result (untimed; the oracle is the checker, never the thing measured) ----
    from oracle import oracle as O

    threads_cpu = host_threads()
    cpu = None
    th = max(1, threads_cpu // world)
    dl_local = O.msm_derived_by_dlog(first, h_page, threads=th)   # (sum_i a_i s_i) * (-1, 2) over this rank's slice
    dl_total = comm.allgather_sum(dl_local) if comm else dl_local
    oracle_match = {"dlog_property": bool(O.pt_eq(res, dl_total))}
    if world == 1 and not args.no_cpu_baseline:
        gs = ctx.get_generators(0, n)                              # the very bases the GPU used, read back
        t = time.perf_counter()
        exp = O.msm_affine(gs, h_page, threads=threads_cpu)         # arkworks-shaped Pippenger at the SAME size
        dt = time.perf_counter() - t
        del gs
        oracle_match["pippenger_same_size"] = bool(O.pt_eq(res, exp))
        cpu = {"value": n / dt, "unit": UNIT, "cores": threads_cpu, "kind": "port",
               "sample": f"1 MSM of 2^{args.log_n} points = the full workload, same bases and scalars as the GPU arm ({dt:.1f} s); "
                         f"arkworks-shaped Pippenger restated in C (field core in MULX / ADC assembly), windows x point chunks over {threads_cpu} threads"}
    ok_all = all(oracle_match.values())
    if world > 1:
        t = torch.tensor([1.0 if ok_all else 0.0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        ok_all = bool(t.item() > 0.5)

    # ---- integer-pipe peak, measured here: independent IMAD chains on every SM ----
    sms = torch.cuda.get_device_properties(local).multi_processor_count
    blocks, threads, iters = sms * 8, 256, 4096
    imad_ms = min(ctx.test_imad_throughput(0, blocks, threads, iters) for _ in range(3))
    imad_peak = blocks * threads * iters * 16 / imad_ms / 1e9  # T IMAD32/s: dependent-multiplicand mad.lo.u32 chains (1 ms burst)
    # the same microbenchmark back to back for ~2 s: the integer pipe's rate at the clocks the power cap allows under
    # sustained load (MEASURED_PEAKS.json makes the same burst / sustained distinction for bf16)
    imad_sust, imad_sust_clocks = None, None
    if rank == 0 or world > 1:
        it8 = iters * 8
        smp = ClockSampler(local, dev_uuid)
        smp.start()
        t_end, runs = time.perf_counter() + 2.0, []
        while time.perf_counter() < t_end:
            runs.append(ctx.test_imad_throughput(0, blocks, threads, it8))
        imad_sust_clocks = smp.summary()
        tail = sorted(runs[len(runs) // 2:])
        imad_sust = blocks * threads * it8 * 16 / tail[len(tail) // 2] / 1e9

    def whole_msm_frac(points, ms, gpus=1):
        return (points * 160 + 14.68e6) * IMAD_PER_MODMUL / (ms * 1e-3) / 1e12 / (imad_peak * gpus)

    # ---- strong scaling (BASELINE config 5): ONE MSM of 2^lg points over the N GPUs ----
    strong = None
    if not args.no_strong:
        strong = strong_scaling_sweep(args, ctx, comm, world, rank, dev, barrier, maxr, whole_msm_frac, O, th)

    out = None
    if rank == 0:
        total_points = n * world
        alg_imad = n * CANON_W * 10 * IMAD_PER_MODMUL  # algorithmic IMAD32 of the accumulation phase (canonical c = 16)
        achieved = alg_imad / (phases["accumulate"] * 1e-3) / 1e12
        traffic = None  # dram__bytes_read + dram__bytes_write of the accumulation phase, from the committed ncu capture
        traffic_file = None
        for fn in ("r02_traffic.json", "r01_traffic.json"):
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", fn)))["accumulate_phase_pair_tree"]
                if tj["workload"] == f"{CURVE}_msm_2^{args.log_n}_per_gpu" and tj["fixed_base_tables"] == (not args.no_precompute):
                    traffic, traffic_file = tj["dram_bytes_read"] + tj["dram_bytes_write"], fn
                    break
            except Exception:
                pass
        # executed work: W windows x (6.2 modmul per affine pair-tree addition for the first P levels, 10 for the XYZZ tail)
        secondary = None
        if world == 1 and not args.no_secondary:
            secondary = secondary_metrics(ctx, args)
        out = {
            "metric": METRIC, "value": total_points / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32x8 (255-bit Montgomery)", "data": "synthetic",
            "config": make_config(args.log_n, world),
            "impl_config": {"window_c": "auto", "fixed_base_tables": (not args.no_precompute),
                            "steps_in_flight": "2 (halo_msm_gens_submit_resident / _collect: the counting sort of step k+1 overlaps the accumulation of step k)",
                            "collective": f"ncclAllGather inside libhalo_b200.so (halo_comm_*), NCCL {H._capi.load().halo_nccl_version()}" if world > 1 else None},
            "oracle_match": ok_all, "oracle_checks": oracle_match, "paths_agree": same,
            "wall_ms_per_step": wall_step,
            "sequential_calls": {"api": ("halo_msm_gens_sharded_resident" if world > 1 else "halo_msm_gens_resident") + " (one blocking call per step, nothing overlaps)",
                                 "ms_per_step": seq_ms, "value": total_points / (seq_ms * 1e-3)},
            "variable_base": {"api": "same call without halo_precompute_generators tables (W bucket sets, Horner on the host): the path of point_dot / the IPA rounds",
                              "ms_per_step": var_ms, "value": total_points / (var_ms * 1e-3), "whole_msm_frac": whole_msm_frac(n, var_ms)},
            "e2e": {"value": total_points / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                    "api": "halo_msm_gens_submit / halo_msm_gens_collect (pinned host scalars, two steps in flight)",
                    "h2d_bytes_per_step": n * 32, "d2h_bytes_per_step": 3 * 128, "result_matches_resident": same,
                    "blocking_call": {"api": ("halo_msm_gens_sharded" if world > 1 else "halo_msm_gens") + " from pinned host memory (one call per step)",
                                      "value": total_points / (e2e_sync_ms * 1e-3), "ms_per_step": e2e_sync_ms},
                    "blocking_call_pageable": {"api": "the same call from PAGEABLE host memory (a plain Vec<Fr> / numpy array), staged through pinned chunks inside the library",
                                               "value": total_points / (e2e_page_ms * 1e-3), "ms_per_step": e2e_page_ms}},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "imad", "bound_note": "integer pipe (IMAD32 issue rate): the path is big-integer arithmetic, neither HBM nor tensor bound; BASELINE.json's north_star asks for the fraction of the integer-pipe roofline", "kernel": "bucket accumulation phase: k_pair_fwd / k_pair_bwd x 4 tree passes (affine, batched inversion) + k_accumulate (XYZZ tail)", "achieved": achieved, "peak": imad_peak, "unit": "TIMAD32/s",
                         "frac": achieved / imad_peak, "traffic": traffic, "traffic_unit": f"DRAM bytes of the phase per MSM (ncu, profiles/{traffic_file})",
                         "hbm_gbs_phase": (traffic / (phases["accumulate"] * 1e-3) / 1e9) if traffic else None,
                         "peak_source": "measured in this run (libhalo_b200 mad.lo.u32 microbenchmark, 16 independent chains per thread, all SMs); MEASURED_PEAKS.json has no integer-pipe figure. IMAD.WIDE / IMAD.HI issue at half this rate (profiles/r01_imad_pipe_rates.jsonl)",
                         "algorithmic": f"{n} pts x {CANON_W} windows x 10 modmul x {IMAD_PER_MODMUL} IMAD32 per launch (SURVEY 8d canonical accounting, c = 16)",
                         "launch_ms": phases["accumulate"], "phases_ms": phases, "clocks_phase": phase_clocks,
                         "peak_sustained": imad_sust, "frac_of_sustained_peak": (achieved / imad_sust) if imad_sust else None,
                         "peak_sustained_note": "the same IMAD microbenchmark back to back for 2 s (median of the second half): `peak` is a 1 ms burst at boost clocks, "
                                                "the phase is timed inside back-to-back MSMs under the board's power cap; `frac` stays against the burst figure",
                         "clocks_peak_sustained": imad_sust_clocks,
                         "whole_msm_frac": whole_msm_frac(n, ms_step),
                         "executed": {"note": "what the kernels issue: 13 windows (c = 20), 15/16 of the additions affine in the pair tree (6.2 modmul each: 5M + 1S + shared inversion), the rest XYZZ (10)",
                                      "modmul_per_point": 13 * (15 / 16 * 6.2 + 1 / 16 * 10),
                                      "frac": n * 13 * (15 / 16 * 6.2 + 1 / 16 * 10) * IMAD_PER_MODMUL / (phases["accumulate"] * 1e-3) / 1e12 / imad_peak}},
            "strong_scaling": strong,
            "cpu_baseline": cpu,
            "secondary": secondary,
            "derive_generators_s": derive_s, "precompute_tables_s": precompute_s,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
    if comm:
        comm.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return out


def strong_scaling_sweep(args, ctx, comm, world, rank, dev, barrier, maxr, whole_msm_frac, O, oracle_threads):
    """ONE MSM of 2^lg points, lg = 16 .. log_n, sharded by point slice over the `world` GPUs (strong scaling): FIXED-base
    tables per slice, device-resident scalars, the library's all-gather inside the timed region, CUDA events on the
    library's stream, max over ranks.  Every size is checked against the oracle (discrete-log property of the derived
    generators on every rank's slice; the arkworks-shaped Pippenger as well up to 2^20)."""
    import torch

    import halo_accumulation_b200 as H

    rows = {}
    for lg in [l for l in (16, 18, 20, 22, 24) if l <= args.log_n]:
        nt = 1 << lg
        if nt < world:
            continue
        first, count = H.comm_slice(nt, rank, world)
        if comm:
            comm.derive_generators(nt)
            comm.precompute_generators(0)
        else:
            ctx.derive_generators(nt)
            ctx.precompute_generators(0)
        h = bench_scalars(nt, 100 + lg)[first:first + count]
        d = torch.from_numpy(h.view(np.int64).copy()).to(dev)
        torch.cuda.synchronize()
        call = (lambda: comm.msm_gens_sharded_resident(d.data_ptr(), count, nt)) if comm else (lambda: ctx.msm_gens_resident(d.data_ptr(), count))
        reps = 20 if lg <= 20 else (8 if lg <= 22 else 4)
        for _ in range(3):
            out = call()
        best = 1e30
        for _ in range(3):
            barrier()
            ctx.timer_start()
            for _ in range(reps):
                out = call()
            best = min(best, maxr(ctx.timer_stop() / reps)[0])
        dl = O.msm_derived_by_dlog(first, h, threads=oracle_threads)
        exp = comm.allgather_sum(dl) if comm else dl
        ok = bool(O.pt_eq(out, exp))
        if lg <= 20 and rank == 0:
            ok = ok and bool(O.pt_eq(out, O.msm_affine(O.derive_points_fast(2, nt), bench_scalars(nt, 100 + lg), threads=oracle_threads)))
        rows[f"2^{lg}"] = {"ms": best, "points_per_s": nt / (best * 1e-3), "frac_of_imad_roofline": whole_msm_frac(nt, best, world),
                           "points_per_gpu": count, "oracle_match": ok}
        del d
    return {"gpus": world, "what": "one MSM of 2^lg points sharded by point slice over the GPUs; FIXED-base tables; scalars resident; "
                                   "all-gather and finish inside the timed call; fraction = SURVEY 8(d) whole-MSM work / time / (gpus x measured IMAD peak)",
            "sizes": rows}


def secondary_metrics(ctx, args):
    """ASDL decider and PCDL open at n = 2^20 (BASELINE.json metric, second half; configs 3-4), device timings."""
    from halo_accumulation_b200 import acc, pcdl

    lg = args.secondary_log_n
    n, d = 1 << lg, (1 << lg) - 1
    ctx.derive_generators_range(0, n)
    if not args.no_precompute:
        ctx.precompute_generators(0)
    rng = np.random.Generator(np.random.PCG64(5))

    def rs(k):
        a = rng.integers(0, 1 << 64, size=(k, 4), dtype=np.uint64)
        a[:, 3] &= np.uint64((1 << 62) - 1)
        return a

    p, z = rs(n), rs(1)[0]
    w, wb, q = rs(1)[0], rs(1)[0], rs(n - 1)
    def timed(f, reps=2):  # one warm-up call (first use allocates the context's device buffers), then the best of `reps`
        out = f()
        best = 1e18
        for _ in range(reps):
            t = time.perf_counter()
            out = f()
            best = min(best, (time.perf_counter() - t) * 1e3)
        return out, best

    Cm, commit_ms = timed(lambda: pcdl.commit(ctx, p, d, w))
    pi, open_ms = timed(lambda: pcdl.open(ctx, p, Cm, d, z, w, q, wb))
    _, open_plain_ms = timed(lambda: pcdl.open(ctx, p, pcdl.commit(ctx, p, d), d, z))
    from halo_accumulation_b200 import group

    v = group.scalar_dot(ctx, p, group.construct_powers(ctx, z, n))
    pcdl.check(ctx, Cm, d, z, v, pi)
    best = 1e9
    for _ in range(3):
        t = time.perf_counter()
        pcdl.check(ctx, Cm, d, z, v, pi)
        best = min(best, (time.perf_counter() - t) * 1e3)
    # one accumulation step + decider
    q0 = acc.new_instance(Cm, d, z, v, pi)
    h0r, wr, qr, wbr = rs(2), rs(1)[0], rs(n - 1), rs(1)[0]
    a, prover_ms = timed(lambda: acc.prover(ctx, d, [q0], h0r, wr, qr, wbr))
    acc.verifier(ctx, d, [q0], a)
    dec = 1e9
    for _ in range(3):
        t = time.perf_counter()
        acc.decider(ctx, a)
        dec = min(dec, (time.perf_counter() - t) * 1e3)
    # the oracle's decision on the accumulator just timed (its decider = succinct check + one 2^20 MSM on the host cores)
    from oracle import oracle as O

    S, Hh = ctx.get_SH()
    O.set_params(S, Hh, ctx.get_generators(0, n))
    t = time.perf_counter()
    orc = O.acc_decider(O.Accumulator.from_buffer_copy(bytes(a)), threads=host_threads())
    orc_ms = (time.perf_counter() - t) * 1e3
    return {f"asdl_decider_ms_2^{lg}": dec, f"pcdl_check_ms_2^{lg}": best, f"pcdl_open_hiding_ms_2^{lg}": open_ms, f"pcdl_open_ms_2^{lg}": open_plain_ms,
            f"pcdl_commit_ms_2^{lg}": commit_ms, f"asdl_prover_ms_2^{lg}": prover_ms,
            "oracle_decider_accepts": orc == 0, f"oracle_decider_cpu_ms_2^{lg}": orc_ms,
            "timing": "host wall clock around the synchronous call, best of 2 after one warm-up (open_ms includes a commit)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--log-n", type=int, default=24, help="log2 of the points per GPU")
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--secondary-log-n", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling sweep (one MSM of 2^16 .. 2^log_n points over the GPUs)")
    ap.add_argument("--no-precompute", action="store_true", help="variable-base path only (no tables of precomputed multiples)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of the last timed step to DIR/msm_result.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # the tree may be read-only and is never written: no bytecode caches next to the modules imported below
    sys.dont_write_bytecode = True
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
