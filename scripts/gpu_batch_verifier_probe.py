"""Batch verifier probe (DESIGN.md K5c), one B200, FIXED-base tables (precompute_generators(0)).

1. End to end: k sequential acc.verifier against ONE acc.verifier_batch over the same k steps of an IVC chain (m = 1 for the
   first step, 2 after; hiding instances), lg n in {16, 20}, k in {1, 8, 64}, and k = 1000 at 2^16 (the 64 distinct steps
   repeated); host clock around the synchronising calls, warm-up first, best of 3.  The fast path of many accumulators
   (benches/acc.rs acc_compare): k verifiers + decider against verifier_batch + decider at k = 64.
2. The C' / C* path inside the batches: verifier_batch and pcdl.check_batch at k = 64 with "combine_min_outputs" 0 (device)
   and -1 (host threads).
3. halo_test_point_combine alone, device (k_point_combine) against host GLV on up to 16 threads, N = 1 .. 4096 outputs,
   best of 5 after a warm-up: the crossover that sets the default of "combine_min_outputs".
Decisions are asserted identical in the same run (accept on the honest steps; the same (index, code) with one corrupted step).

Appends one JSON line per measurement, each with the card's name and power limit read in the same run, to the file named by
the first argument (default profiles/r04_batch_verifier.jsonl)."""
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

path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r04_batch_verifier.jsonl")
os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
out = open(path, "a")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]


def emit(d):
    d["gpu"] = gpu
    line = json.dumps(d)
    print(line, flush=True)
    out.write(line + "\n")


rng = np.random.Generator(np.random.PCG64(2027))


def rs(k):
    a = rng.integers(0, 1 << 64, size=(k, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)
    return a


def best(f, reps=3):
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
    except acc.Rejected as e:
        return (e.index, e.code)


def seq_first_reject(d, steps):
    for i, (qs, a) in enumerate(steps):
        r = decision(lambda: acc.verifier(ctx, d, qs, a))
        if r is not None:
            return (i, r[1])
    return None


for lg in (16, 20):
    n, d = 1 << lg, (1 << lg) - 1
    ctx = H.Context(0, 1 << 20)  # a fresh context per size: the end-to-end lines run with the default "combine_min_outputs"
    ctx.derive_generators(n)
    ctx.precompute_generators(0)
    steps, a, claims = [], None, []
    for s in range(64):
        p, (z, w, wb) = rs(n - 1 - s), rs(3)
        q = rs(p.shape[0] - 1)
        Cm = pcdl.commit(ctx, p, d, w)
        v = group.scalar_dot(ctx, p, group.construct_powers(ctx, z, p.shape[0]))
        inst = acc.new_instance(Cm, d, z, v, pcdl.open(ctx, p, Cm, d, z, w, q, wb))
        claims.append(inst)
        qs = [acc.to_instance(a), inst] if a is not None else [inst]
        a = acc.prover(ctx, d, qs, rs(2), rs(1)[0], rs(n - 1), rs(1)[0])
        steps.append((qs, a))
    rho = rs(1)[0]
    for k in (1, 8, 64) + ((1000,) if lg == 16 else ()):
        st = [steps[i % len(steps)] for i in range(k)]
        seq = lambda: [acc.verifier(ctx, d, qs, ac) for qs, ac in st]  # noqa: E731
        bat = lambda: acc.verifier_batch(ctx, d, st, rho)  # noqa: E731
        assert decision(seq) is None and decision(bat) is None
        t_seq, t_bat = best(seq), best(bat)
        emit({"end_to_end": "acc.verifier x k vs acc.verifier_batch", "n": f"2^{lg}", "k": k, "m": "1 then 2", "hiding": True,
              "fixed_base": True, "sequential_ms": round(t_seq, 3), "batch_ms": round(t_bat, 3), "speedup": round(t_seq / t_bat, 2),
              "batch_ms_per_step": round(t_bat / k, 4)})
    fast_seq = lambda: ([acc.verifier(ctx, d, qs, ac) for qs, ac in steps], acc.decider(ctx, steps[-1][1]))  # noqa: E731
    fast_bat = lambda: (acc.verifier_batch(ctx, d, steps, rho), acc.decider(ctx, steps[-1][1]))  # noqa: E731
    t_fs, t_fb = best(fast_seq), best(fast_bat)
    emit({"fast_path": "k verifiers + decider vs verifier_batch + decider", "n": f"2^{lg}", "k": 64, "sequential_ms": round(t_fs, 3),
          "batch_ms": round(t_fb, 3), "speedup": round(t_fs / t_fb, 2)})
    for kind in ("v", "pi_c"):
        bad = list(steps[:16])
        qs, ac = bad[9]
        ac = type(ac).from_buffer_copy(bytes(ac))
        qs = [type(q).from_buffer_copy(bytes(q)) for q in qs]
        if kind == "v":
            ac.v[0] ^= 1
        else:
            qs[-1].pi.c[0] ^= 1
        bad[9] = (qs, ac)
        first = seq_first_reject(d, bad)
        got = decision(lambda: acc.verifier_batch(ctx, d, bad, rho))
        assert got == first and first[0] == 9, (got, first)
        emit({"reject_equivalence": f"2^{lg}", "corrupted": kind, "k": len(bad), "batch": list(got), "sequential_first_reject": list(first)})
    for label, thr in (("device", 0), ("host", -1)):
        ctx.set_tuning("combine_min_outputs", thr)
        t_v = best(lambda: acc.verifier_batch(ctx, d, steps, rho))
        t_c = best(lambda: pcdl.check_batch(ctx, claims, rho))
        emit({"c_prime_path": label, "combine_min_outputs": thr, "n": f"2^{lg}", "k": 64, "verifier_batch_ms": round(t_v, 3),
              "verifier_batch_outputs": 64 + sum(1 for qs, _ in steps for q in qs if q.pi.hiding),
              "check_batch_ms": round(t_c, 3), "check_batch_outputs": 64})
    ctx.close()

ctx = H.Context(0, 1 << 20)
ctx.derive_generators(1 << 16)
lib = ctx._lib
u64 = lambda x: x.ctypes.data_as(C.POINTER(C.c_uint64))  # noqa: E731
from oracle import oracle as O  # noqa: E402

jac = np.ascontiguousarray(O.affine_to_jac(ctx.get_generators(0, 8192)))
for N in (1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 4096):
    P, Q = np.ascontiguousarray(jac[:N]), np.ascontiguousarray(jac[4096:4096 + N])
    a, b = rs(N), rs(N)
    res = {}
    for path_id, label in ((1, "device"), (0, "host16")):
        o = np.zeros((N, 8), dtype=np.uint64)
        res[label] = best(lambda: ctx._chk(lib.halo_test_point_combine(ctx._h, path_id, u64(P), u64(Q), u64(a), u64(b), N, u64(o))), 5)
        res[label + "_out"] = o.copy()
    assert np.array_equal(res["device_out"], res["host16_out"])
    emit({"kernel": "k_point_combine (halo_test_point_combine)", "outputs": N, "device_ms": round(res["device"], 4),
          "host_glv_16_threads_ms": round(res["host16"], 4), "host_threads": min(16, os.cpu_count() or 1),
          "device_faster": res["device"] < res["host16"]})
ctx.close()
