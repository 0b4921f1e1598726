"""Batch decider probe (DESIGN.md K5b), one B200, FIXED-base tables (precompute_generators(0)).

1. End to end: k sequential pcdl.check against ONE pcdl.check_batch over the same k hiding claims, lg n in {16, 20},
   k in {1, 2, 8, 64}; host clock around the synchronising calls, warm-up first, best of 5; the decisions are asserted
   identical (accept on the honest claims; the same (index, code) with one corrupted claim).
2. k_h_lincomb alone (CUDA events, best of 5 after a warm-up): ns per coefficient and claim at n in {2^20, 2^24}.

Appends one JSON line per measurement, each with the card's name and power limit read in the same run, to the file named
by the first argument (default profiles/r03_batch_check.jsonl, whose earlier lines -- the A/B against the removed per-claim
k_h_expand loop -- are kept)."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
import halo_accumulation_b200 as H  # noqa: E402
from halo_accumulation_b200 import acc, group, pcdl  # noqa: E402

path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r03_batch_check.jsonl")
os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
out = open(path, "a")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]


def emit(d):
    d["gpu"] = gpu
    line = json.dumps(d)
    print(line, flush=True)
    out.write(line + "\n")


rng = np.random.Generator(np.random.PCG64(2026))


def rs(k):
    a = rng.integers(0, 1 << 64, size=(k, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)
    return a


def best(f, reps=5):
    f()
    b = 1e30
    for _ in range(reps):
        t = time.perf_counter()
        f()
        b = min(b, (time.perf_counter() - t) * 1e3)
    return b


def decision(f):
    try:
        f()
        return None
    except pcdl.Rejected as e:
        return e.code


ctx = H.Context(0, 1 << 24)
for lg in (16, 20):
    n, d = 1 << lg, (1 << lg) - 1
    ctx.derive_generators(n)
    ctx.precompute_generators(0)
    claims = []
    for j in range(64):  # hiding claims of degree < d
        p, (z, w, wb) = rs(n - 1 - j), rs(3)
        q = rs(p.shape[0] - 1)
        Cm = pcdl.commit(ctx, p, d, w)
        v = group.scalar_dot(ctx, p, group.construct_powers(ctx, z, p.shape[0]))
        claims.append(acc.new_instance(Cm, d, z, v, pcdl.open(ctx, p, Cm, d, z, w, q, wb)))
    rho = rs(1)[0]
    for k in (1, 2, 8, 64):
        qs = claims[:k]
        seq = lambda: [pcdl.check(ctx, np.array(q.C), q.d, np.array(q.z), np.array(q.v), q.pi) for q in qs]  # noqa: E731
        bat = lambda: pcdl.check_batch(ctx, qs, rho)  # noqa: E731
        assert decision(seq) is None and decision(bat) is None
        t_seq, t_bat = best(seq), best(bat)
        emit({"end_to_end": "pcdl.check x k vs pcdl.check_batch", "n": f"2^{lg}", "k": k, "hiding": True, "fixed_base": True,
              "sequential_ms": round(t_seq, 3), "batch_ms": round(t_bat, 3), "speedup": round(t_seq / t_bat, 2),
              "batch_ms_per_claim": round(t_bat / k, 4)})
    bad = type(claims[5]).from_buffer_copy(bytes(claims[5]))
    bad.v[0] ^= 1
    qs = claims[:5] + [bad] + claims[6:8]
    first = None
    for j, q in enumerate(qs):
        c = decision(lambda: pcdl.check(ctx, np.array(q.C), q.d, np.array(q.z), np.array(q.v), q.pi))
        if c is not None:
            first = (j, c)
            break
    try:
        pcdl.check_batch(ctx, qs, rho)
        got = None
    except pcdl.Rejected as e:
        got = (e.index, e.code)
    assert got == first == (5, -10), (got, first)
    emit({"reject_equivalence": f"2^{lg}", "k": len(qs), "batch": list(got), "sequential_first_reject": list(first)})

lib = ctx._lib
lib.halo_test_h_lincomb_bench.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.POINTER(C.c_float)]
for lg in (20, 24):
    for k in (1, 2, 16, 64):
        ms = C.c_float()
        ctx._chk(lib.halo_test_h_lincomb_bench(ctx._h, lg, k, C.byref(ms)))
        emit({"kernel": "k_h_lincomb", "n": f"2^{lg}", "k": k, "ms": round(ms.value, 4),
              "ns_per_coeff_claim": round(ms.value * 1e6 / ((1 << lg) * k), 4)})
ctx.close()
