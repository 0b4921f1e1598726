"""Batch commit probe (DESIGN.md K2c), one B200, FIXED-base tables precomputed for 2^20 generators.

1. Main comparison: k sequential pcdl.commit calls against ONE pcdl.commit_batch, n = 2^12, 2^16, 2^20 coefficients,
   k = 1, 8, 64, with and without hiding.  The two paths' points are asserted equal in the same run.
2. Window sweep: commit_batch (no hiding) with halo_set_msm_window forced (variable base: 2^12 and 2^16), and with the FIXED
   tables rebuilt at other windows (2^20); k = 8 and 64.  This sweep sets the group policy of halo_msm_gens_many.
Host clock around the synchronising calls, a warm-up first, best of 3.

Appends one JSON line per measurement, each with the card's name and power limit read in the same run, to the file named by
the first argument (default profiles/r06_commit_batch.jsonl)."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
import halo_accumulation_b200 as H  # noqa: E402
from halo_accumulation_b200 import pcdl  # noqa: E402

path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r06_commit_batch.jsonl")
os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
out = open(path, "a")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]


def emit(d):
    d["gpu"] = gpu
    line = json.dumps(d)
    print(line, flush=True)
    out.write(line + "\n")


rng = np.random.Generator(np.random.PCG64(2029))


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


N = 1 << 20
ctx = H.Context(0, N)
ctx.derive_generators(N)
ctx.precompute_generators(0)
S, _ = ctx.get_SH()

for lg in (12, 16, 20):
    n, d = 1 << lg, N - 1
    for k in (1, 8, 64):
        polys = rs(k, n)  # one array: the batch reads the packed coefficients without a copy
        ps = list(polys)
        for hiding in (False, True):
            ws = rs(k) if hiding else None

            def loop():
                return [pcdl.commit(ctx, p, d, None if ws is None else ws[j]) for j, p in enumerate(ps)]

            def batch():
                return pcdl.commit_batch(ctx, polys, d, ws)

            a, b = loop(), batch()
            assert all(H.points_equal(a[j], b[j]) for j in range(k)), (lg, k, hiding)
            t_loop, t_batch = best(loop), best(batch)
            emit(dict(probe="commit_batch", n=n, k=k, hiding=hiding, loop_ms=round(t_loop, 3), batch_ms=round(t_batch, 3),
                      speedup=round(t_loop / t_batch, 2)))
        del polys, ps

# window sweep (no hiding): variable base by halo_set_msm_window, FIXED base by the window of the precomputed tables
for lg, windows in ((12, (7, 8, 9, 10, 11, 12, 13)), (16, (9, 10, 11, 12, 13, 14))):
    n = 1 << lg
    for k in (8, 64):
        ps = rs(k, n)
        ref = pcdl.commit_batch(ctx, ps, N - 1)
        for c in windows:
            ctx.set_msm_window(c)
            got = pcdl.commit_batch(ctx, ps, N - 1)
            assert all(H.points_equal(ref[j], got[j]) for j in range(k)), (lg, k, c)
            emit(dict(probe="commit_batch_window", n=n, k=k, fixed=False, c=c, batch_ms=round(best(lambda: pcdl.commit_batch(ctx, ps, N - 1)), 3),
                      route=ctx.test_msm_route(0)))
        ctx.set_msm_window(0)
for k in (8, 64):
    ps = rs(k, N)
    ctx.precompute_generators(0)
    ref = pcdl.commit_batch(ctx, ps, N - 1)
    for c in (16, 18, 19, 20):
        ctx.precompute_generators(c)
        got = pcdl.commit_batch(ctx, ps, N - 1)
        assert all(H.points_equal(ref[j], got[j]) for j in range(k)), (k, c)
        emit(dict(probe="commit_batch_window", n=N, k=k, fixed=True, c=c, batch_ms=round(best(lambda: pcdl.commit_batch(ctx, ps, N - 1)), 3),
                  loop_ms=round(best(lambda: [pcdl.commit(ctx, p, N - 1) for p in ps]), 3), route=ctx.test_msm_route(0)))
    del ps
ctx.close()
