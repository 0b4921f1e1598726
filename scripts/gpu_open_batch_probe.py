"""Batch opening probe (DESIGN.md K3b), one B200, FIXED-base tables precomputed for 2^20 generators.

1. k sequential pcdl.open calls against ONE pcdl.open_batch, n = 2^16 and 2^20 coefficients (degree bound 2^20 - 1 for both:
   the opening's cost follows d, the upload and the two linear passes follow n), k = 1, 8, 64, with and without hiding.  Host
   clock around the synchronising calls, a warm-up first, best of 3.  In every row the combined claim passes pcdl.check, and at
   k = 1 the batch's proof equals open's.
2. Phases of one batch, by host clock around the synchronising entry points: halo_poly_eval_many (upload + z powers +
   evaluation), halo_poly_combine_resident (combination + degree scan) and the rest of open_batch (alpha, C = sum alpha^j C_j,
   the opening).  In a separate pass torch.profiler gives the device time of the evaluation kernels (k_powers is counted with
   the opening, which builds its own powers), of k_poly_combine and of the host-to-device copies.
Appends one JSON line per row, each with the card's name and power limit read in the same run, to the file named by the first
argument (default profiles/r07_open_batch.jsonl)."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
import halo_accumulation_b200 as H  # noqa: E402
from halo_accumulation_b200 import _capi, pcdl  # noqa: E402

path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r07_open_batch.jsonl")
os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
out = open(path, "a")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]


def emit(d):
    d["gpu"] = gpu
    line = json.dumps(d)
    print(line, flush=True)
    out.write(line + "\n")


rng = np.random.Generator(np.random.PCG64(2031))


def rs(k, n=None):
    a = rng.integers(0, 1 << 64, size=(k, 4) if n is None else (k, n, 4), dtype=np.uint64)
    a[..., 3] &= np.uint64((1 << 62) - 1)
    return a


def best(f, reps=3):
    f()
    b = 1e30
    for _ in range(reps):
        t = time.perf_counter()
        f()
        b = min(b, (time.perf_counter() - t) * 1e3)
    return b


def clock(f):
    t = time.perf_counter()
    r = f()
    return r, (time.perf_counter() - t) * 1e3


N = 1 << 20
D = N - 1
ctx = H.Context(0, N)
ctx.derive_generators(N)
ctx.precompute_generators(0)
lib = _capi.load()
p64 = _capi.p64
cases = []

for lg in (16, 20):
    n = 1 << lg
    for k in (1, 8, 64):
        polys = rs(k, n)  # one array: the batch reads the packed coefficients without a copy
        ps = list(polys)
        z = rs(1)[0]
        for hiding in (False, True):
            ws = rs(k) if hiding else None
            q = rs(n - 1) if hiding else None
            wb = rs(1)[0] if hiding else None
            Cs = pcdl.commit_batch(ctx, polys, D, ws)

            def loop():
                return [pcdl.open(ctx, p, Cs[j], D, z, None if ws is None else ws[j], q, wb) for j, p in enumerate(ps)]

            def batch():
                return pcdl.open_batch(ctx, polys, Cs, D, z, ws, q, wb)

            vs, Cm, v, pi = batch()
            pcdl.check(ctx, Cm, D, z, v, pi)
            if k == 1:
                ref = loop()[0]
                assert all(H.points_equal(np.array(pi.Ls[i]), np.array(ref.Ls[i])) for i in range(pi.lg_n))
                assert H.points_equal(np.array(pi.U), np.array(ref.U)) and list(pi.c) == list(ref.c)
            t_loop, t_batch = best(loop), best(batch)
            row = dict(probe="open_batch", n=n, d=D, k=k, hiding=hiding, loop_ms=round(t_loop, 3), batch_ms=round(t_batch, 3),
                       speedup=round(t_loop / t_batch, 2), check="accepted")
            if k > 1:  # phases of one batch: the device entry points open_batch calls, timed one by one
                lens = np.full(k, n, dtype=np.uint64)
                vs_out = np.zeros((k, 4), dtype=np.uint64)
                alpha, deg = rs(1)[0], C.c_uint64()
                packed = polys.reshape(-1, 4)
                for _ in range(2):
                    rc, t_eval = clock(lambda: lib.halo_poly_eval_many(ctx._h, p64(packed), p64(lens), C.c_uint64(k), C.c_uint64(N),
                                                                       p64(z), p64(vs_out)))
                    assert rc == 0
                    rc, t_comb = clock(lambda: lib.halo_poly_combine_resident(ctx._h, p64(alpha), C.byref(deg)))
                    assert rc == 0
                row.update(upload_eval_ms=round(t_eval, 3), combine_ms=round(t_comb, 3),
                           open_and_claim_ms=round(t_batch - t_eval - t_comb, 3), upload_bytes=k * n * 32)
                cases.append((n, k, hiding, polys, Cs, z, ws, q, wb))
            emit(row)
        del ps

# device time of the new kernels and the copies, one profiled batch per case (profiler on: not used for the timings above)
try:
    from torch.profiler import ProfilerActivity, profile

    for n, k, hiding, polys, Cs, z, ws, q, wb in cases:
        pcdl.open_batch(ctx, polys, Cs, D, z, ws, q, wb)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            pcdl.open_batch(ctx, polys, Cs, D, z, ws, q, wb)
        dev = {}
        for e in prof.key_averages():
            us = getattr(e, "device_time_total", None)
            if us is None:
                us = e.cuda_time_total
            for key, pat in (("eval_kernels_ms", "k_poly_eval"), ("combine_kernel_ms", "k_poly_combine"), ("h2d_copy_ms", "HtoD")):
                if pat in e.key:
                    dev[key] = dev.get(key, 0.0) + us / 1e3
        emit(dict(probe="open_batch_device", n=n, k=k, hiding=hiding, **{a: round(b, 3) for a, b in dev.items()}))
except Exception as ex:  # the timings above stand without the profile
    emit(dict(probe="open_batch_device", error=repr(ex)))
ctx.close()
