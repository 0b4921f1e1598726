"""Transform probe (DESIGN.md K8), one B200.

1. Device time of the batched transform (forward, inverse, coset forward) at 2^12, 2^16, 2^20, 2^22 and 2^24 with k = 1, and
   at 2^20 with k = 8 (256 MiB, larger than the 126 MB L2; 2^20 with k = 1 is 32 MiB and stays in L2 between passes and calls).
   Context.ntt_resident on a torch CUDA tensor, warm-up first; torch.profiler over `reps` calls gives the kernel time of
   k_ntt_pass (and k_ntt_pows, the per-call coset table), and CUDA events on the context stream the time of a whole call.
   Multiplications from the shapes: (n / 2) lg n butterflies, 2 n per pass after the first (the two-level twiddle and its
   product), 2 n for coset factors, n for the n^-1 of a plain inverse.  The timed output is compared with Context.ntt (host
   in, host out) on the same input.
2. pcdl.commit_evals against pcdl.commit_batch of the already-interpolated coefficients at 2^16 and 2^20, k = 1 and 8
   (FIXED-base tables for 2^20 generators): the transform's added cost.  Both take one (k, n, 4) array, so neither packs a
   copy on the host.  Host clock around the synchronising calls, warm-up,
   best of 5; the commitments are compared projectively.
3. pcdl.open_multi_evals against pcdl.open_multi at (k, T, m) = (8, 3, 12) at 2^20, without hiding; every output compared.
Appends one JSON line per row, each with the card's name and power limit read in the same run, to the file named by the first
argument (default profiles/r09_ntt.jsonl)."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
import halo_accumulation_b200 as H  # noqa: E402
from halo_accumulation_b200 import pcdl  # noqa: E402

path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r09_ntt.jsonl")
os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
out = open(path, "a")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]


def emit(d):
    d["gpu"] = gpu
    line = json.dumps(d)
    print(line, flush=True)
    out.write(line + "\n")


rng = np.random.Generator(np.random.PCG64(2033))


def rs(*shape):
    a = rng.integers(0, 1 << 64, size=(*shape, 4), dtype=np.uint64)
    a[..., 3] &= np.uint64((1 << 62) - 1)  # below 2^254 < r: canonical
    return a


def passes(lg):
    return 1 if lg <= 11 else -(-lg // 11)


def mults(k, lg, inverse, coset):
    n = 1 << lg
    return k * ((n // 2) * lg + 2 * n * (passes(lg) - 1) + (2 * n if coset else n if inverse else 0))


def best(f, reps=5):
    f()
    b = 1e30
    for _ in range(reps):
        t = time.perf_counter()
        f()
        b = min(b, (time.perf_counter() - t) * 1e3)
    return b


import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

ctx = H.Context(0, 1 << 24)
try:
    # ---- 1. the transform ----
    for lg, k in ((12, 1), (16, 1), (20, 1), (20, 8), (22, 1), (24, 1)):
        n = 1 << lg
        x = rs(k, n)
        g = rs(1)[0]
        for mode in ("forward", "inverse", "coset_forward"):
            inv, sh = mode == "inverse", g if mode == "coset_forward" else None
            want = ctx.ntt(x, lg, inv, sh)
            t = torch.from_numpy(x.view(np.int64).copy()).cuda()
            torch.cuda.synchronize()
            ctx.ntt_resident(t.data_ptr(), k, lg, inv, sh)
            ok = bool(np.array_equal(t.cpu().numpy().view(np.uint64), want))
            reps = max(5, min(200, (1 << 26) // (k * n)))
            for _ in range(3):
                ctx.ntt_resident(t.data_ptr(), k, lg, inv, sh)
            ctx.timer_start()
            for _ in range(reps):
                ctx.ntt_resident(t.data_ptr(), k, lg, inv, sh)
            call_ms = ctx.timer_stop() / reps
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    ctx.ntt_resident(t.data_ptr(), k, lg, inv, sh)
                torch.cuda.synchronize()
            pass_us = pows_us = 0.0
            for e in prof.key_averages():
                if "k_ntt_pass" in e.key:
                    pass_us += e.device_time_total
                elif "k_ntt_pows" in e.key:
                    pows_us += e.device_time_total
            kern_ms = (pass_us + pows_us) / 1e3 / reps
            m = mults(k, lg, inv, sh is not None)
            emit(dict(probe="ntt", lg=lg, k=k, mode=mode, passes=passes(lg), reps=reps, equal_to_host_path=ok,
                      kernel_ms=round(kern_ms, 4), pass_kernels_ms=round(pass_us / 1e3 / reps, 4),
                      coset_table_ms=round(pows_us / 1e3 / reps, 4), call_ms=round(call_ms, 4), mults=m,
                      gmults_per_s=round(m / kern_ms / 1e6, 2), hbm_bytes_min=2 * 32 * k * n * passes(lg),
                      hbm_gb_per_s=round(2 * 32 * k * n * passes(lg) / kern_ms / 1e6, 1),
                      fits_l2=bool(32 * k * n <= 126e6 // 2)))
            del t
    # ---- 2. commit_evals vs commit_batch ----
    ctx.derive_generators(1 << 20)
    ctx.precompute_generators(0)
    for lg in (16, 20):
        d = (1 << lg) - 1
        for k in (1, 8):
            E = rs(k, 1 << lg)
            ps = ctx.ntt(E, lg, True)  # (k, n, 4): packed in place, as E is
            a = pcdl.commit_evals(ctx, E, d)
            b = pcdl.commit_batch(ctx, ps, d)
            ok = all(H.points_equal(a[j], b[j]) for j in range(k))
            te = best(lambda: pcdl.commit_evals(ctx, E, d))
            tb = best(lambda: pcdl.commit_batch(ctx, ps, d))
            emit(dict(probe="commit_evals", lg=lg, k=k, commit_evals_ms=round(te, 3), commit_batch_ms=round(tb, 3),
                      added_ms=round(te - tb, 3), equal=ok))
    # ---- 3. open_multi_evals vs open_multi ----
    lg, k = 20, 8
    d = (1 << lg) - 1
    E = rs(k, 1 << lg)
    ps = ctx.ntt(E, lg, True)
    Cs = pcdl.commit_evals(ctx, E, d)
    # z, omega z, omega^-1 z (Montgomery limbs are linear: multiply the residue zR by the canonical omega^+-1)
    from oracle.oracle import R_MOD as r_mod
    w = int.from_bytes(H.domain_root(lg).tobytes(), "little") * pow(1 << 256, -1, r_mod) % r_mod
    z = int.from_bytes(rs(1)[0].tobytes(), "little") % r_mod
    zs = np.stack([np.frombuffer((z * f % r_mod).to_bytes(32, "little"), np.uint64) for f in (1, w, pow(w, -1, r_mod))])
    qs = [(0, 0), (0, 1), (0, 2), (1, 0), (2, 1), (3, 2), (4, 0), (4, 2), (5, 1), (6, 0), (7, 2), (6, 1)]
    r1 = pcdl.open_multi_evals(ctx, E, Cs, d, zs, qs)
    r2 = pcdl.open_multi(ctx, ps, Cs, d, zs, qs)
    ok = all(np.array_equal(r1[i], r2[i]) for i in (0, 2, 4, 5)) and H.points_equal(r1[1], r2[1]) and H.points_equal(r1[3], r2[3])
    pcdl.check(ctx, r1[3], d, r1[4], r1[5], r1[6])
    te = best(lambda: pcdl.open_multi_evals(ctx, E, Cs, d, zs, qs), 3)
    tm = best(lambda: pcdl.open_multi(ctx, ps, Cs, d, zs, qs), 3)
    emit(dict(probe="open_multi_evals", lg=lg, k=k, T=3, m=12, open_multi_evals_ms=round(te, 3), open_multi_ms=round(tm, 3),
              added_ms=round(te - tm, 3), equal=bool(ok), check="accepted"))
finally:
    ctx.close()
