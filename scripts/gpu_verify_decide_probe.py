"""Batch verify-and-decide probe (DESIGN.md K5d), one B200, FIXED-base tables (precompute_generators(0)), hiding instances.

For lg n in {16, 20}, over the steps of one IVC chain (m = 1 for the first step, 2 after) and their accumulators:
1. The fast path of one chain (k_dec = 1, the last step's accumulator), k = 1, 8, 64: acc.verifier_batch + acc.decider_batch
   (the pair the fused call stands for), acc.verifier_batch + acc.decider (benches/acc.rs acc_compare) and ONE
   acc.verify_decide_batch.
2. k IVC proofs (k = k_dec = 8, 64): acc.verifier_batch over the k steps + acc.decider_batch over their k accumulators
   against ONE acc.verify_decide_batch.
Each line also has verifier_batch and decider_batch alone: the fused call's ceiling is about the larger of the two when the
generator part hides behind the steps' transcripts.  Host clock around the synchronising calls, a warm-up first, best of 3.
Decisions are asserted identical in the same run: accept on the honest input, and the same (index, code) with one corrupted
step and with one corrupted decided accumulator.

Appends one JSON line per measurement, each with the card's name and power limit read in the same run, to the file named by
the first argument (default profiles/r05_verify_decide.jsonl)."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
import halo_accumulation_b200 as H  # noqa: E402
from halo_accumulation_b200 import acc, group, pcdl  # noqa: E402

path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r05_verify_decide.jsonl")
os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
out = open(path, "a")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]


def emit(d):
    d["gpu"] = gpu
    line = json.dumps(d)
    print(line, flush=True)
    out.write(line + "\n")


rng = np.random.Generator(np.random.PCG64(2028))


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


for lg in (16, 20):
    n, d = 1 << lg, (1 << lg) - 1
    ctx = H.Context(0, 1 << 20)
    ctx.derive_generators(n)
    ctx.precompute_generators(0)
    steps, a = [], None
    for s in range(64):
        p, (z, w, wb) = rs(n - 1 - s), rs(3)
        q = rs(p.shape[0] - 1)
        Cm = pcdl.commit(ctx, p, d, w)
        v = group.scalar_dot(ctx, p, group.construct_powers(ctx, z, p.shape[0]))
        inst = acc.new_instance(Cm, d, z, v, pcdl.open(ctx, p, Cm, d, z, w, q, wb))
        qs = [acc.to_instance(a), inst] if a is not None else [inst]
        a = acc.prover(ctx, d, qs, rs(2), rs(1)[0], rs(n - 1), rs(1)[0])
        steps.append((qs, a))
    rho = rs(1)[0]
    cases = [(k, 1, "fast path of one chain") for k in (1, 8, 64)] + [(k, k, "k IVC proofs") for k in (8, 64)]
    for k, k_dec, label in cases:
        st = steps[:k]
        dec = [ac for _, ac in st[k - k_dec:]]
        vb = lambda: acc.verifier_batch(ctx, d, st, rho)  # noqa: E731
        db = lambda: acc.decider_batch(ctx, dec, rho)  # noqa: E731
        pair = lambda: (vb(), db())  # noqa: E731
        fused = lambda: acc.verify_decide_batch(ctx, d, st, dec, rho)  # noqa: E731
        assert decision(pair) is None and decision(fused) is None
        t_vb, t_db, t_pair, t_fused = best(vb), best(db), best(pair), best(fused)
        line = {"end_to_end": "verifier_batch + decider_batch vs verify_decide_batch", "case": label, "n": f"2^{lg}", "k": k,
                "k_dec": k_dec, "m": "1 then 2", "hiding": True, "fixed_base": True, "verifier_batch_ms": round(t_vb, 3),
                "decider_batch_ms": round(t_db, 3), "two_calls_ms": round(t_pair, 3), "fused_ms": round(t_fused, 3),
                "speedup": round(t_pair / t_fused, 3)}
        if k_dec == 1:
            single = lambda: (vb(), acc.decider(ctx, dec[0]))  # noqa: E731
            line["verifier_batch_plus_decider_ms"] = round(best(single), 3)
        emit(line)
    # the same decisions with one corrupted step and one corrupted decided accumulator (k = k_dec = 16)
    st = steps[:16]
    dec = [ac for _, ac in st]
    for kind in ("step_v", "step_pi_c", "acc_pi_c", "acc_v"):
        bad_st, bad_dec = list(st), list(dec)
        if kind.startswith("step"):
            qs, ac = bad_st[9]
            ac = type(ac).from_buffer_copy(bytes(ac))
            qs = [type(q).from_buffer_copy(bytes(q)) for q in qs]
            if kind == "step_v":
                ac.v[0] ^= 1
            else:
                qs[-1].pi.c[0] ^= 1
            bad_st[9] = (qs, ac)
        else:
            ac = type(dec[5]).from_buffer_copy(bytes(dec[5]))
            if kind == "acc_pi_c":
                ac.pi.c[0] ^= 1
            else:
                ac.v[0] ^= 1
            bad_dec[5] = ac
        r_v = decision(lambda: acc.verifier_batch(ctx, d, bad_st, rho))
        r_d = decision(lambda: acc.decider_batch(ctx, bad_dec, rho))
        pair = r_v if r_v is not None else (None if r_d is None else (len(bad_st) + r_d[0], r_d[1]))
        got = decision(lambda: acc.verify_decide_batch(ctx, d, bad_st, bad_dec, rho))
        assert got == pair and pair is not None, (kind, got, pair)
        emit({"reject_equivalence": f"2^{lg}", "corrupted": kind, "k": len(bad_st), "k_dec": len(bad_dec), "fused": list(got),
              "two_calls": list(pair)})
    ctx.close()
