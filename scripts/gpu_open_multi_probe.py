"""Multi-point opening probe (DESIGN.md K3c), one B200, FIXED-base tables precomputed for 2^20 generators.

1. The same claims opened three ways: (a) m single pcdl.open calls, (b) T pcdl.open_batch calls, one per point, (c) ONE
   pcdl.open_multi.  n = 2^16 and 2^20 coefficients per polynomial, degree bound 2^20 - 1 for both, (k, T, m) = (8, 2, 16)
   (every polynomial at both points), (8, 3, 12) (ragged: one, two or three points per polynomial) and (64, 2, 128), with and
   without hiding.  Host clock around the synchronising calls, a warm-up first, best of 3.  Every claim of every method passes
   pcdl.check in the same run.
2. Phases of one open_multi by host clock around the device entry points it calls: upload (halo_poly_upload), query
   evaluation (halo_poly_eval_queries), quotient + Q's MSM (halo_poly_quotient), u_t (halo_poly_eval_queries at x3),
   combination (halo_poly_lincomb_resident); the rest (challenges, C, the opening) is open_multi's total minus these.
3. torch.profiler, in passes of its own: the device time of the quotient kernels (k_quot_chunks, k_quot_carry, k_quot_write)
   in one halo_poly_quotient call, and their field-multiplication rate; the A/B of the one-point kernels of K3b
   (k_powers + k_poly_eval_many + k_poly_eval_final; k_poly_combine) against the K3c kernels on the same inputs (k_quot_chunks +
   k_quot_carry as k one-point queries; k_poly_lincomb with weights alpha^j) on r07's shapes.
Appends one JSON line per row, each with the card's name and power limit read in the same run, to the file named by the first
argument (default profiles/r08_open_multi.jsonl)."""
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

path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r08_open_multi.jsonl")
os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
out = open(path, "a")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]


def emit(d):
    d["gpu"] = gpu
    line = json.dumps(d)
    print(line, flush=True)
    out.write(line + "\n")


rng = np.random.Generator(np.random.PCG64(2032))


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
    assert r == 0, r
    return (time.perf_counter() - t) * 1e3


def shape(k, T, ragged):
    if not ragged:
        return [(j, t) for t in range(T) for j in range(k)]
    return [(0, 0), (0, 1), (0, 2), (1, 0), (2, 1), (3, 2), (4, 0), (4, 2), (5, 1), (6, 0), (7, 2), (6, 1)]


def dev_ms(prof, pats):
    r = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = e.cuda_time_total
        for key, pat in pats:
            if pat in e.key:
                r[key] = r.get(key, 0.0) + us / 1e3
    return {a: round(b, 4) for a, b in r.items()}


N = 1 << 20
D = N - 1
ctx = H.Context(0, N)
ctx.derive_generators(N)
ctx.precompute_generators(0)
lib = _capi.load()
p64 = _capi.p64
profiled = []

for lg in (16, 20):
    n = 1 << lg
    for k, T, m, ragged in ((8, 2, 16, False), (8, 3, 12, True), (64, 2, 128, False)):
        polys = rs(k, n)
        ps = list(polys)
        zs = rs(T)
        qs = shape(k, T, ragged)
        assert len(qs) == m
        for hiding in (False, True):
            ws = rs(k) if hiding else None
            q = rs(n - 1) if hiding else None
            wQ = rs(1)[0] if hiding else None
            wb = rs(1)[0] if hiding else None
            Cs = pcdl.commit_batch(ctx, polys, D, ws)
            at = [[j for j, t in qs if t == tt] for tt in range(T)]

            def single():
                return [(j, t, pcdl.open(ctx, ps[j], Cs[j], D, zs[t], None if ws is None else ws[j], q, wb)) for j, t in qs]

            def batches():
                return [(t, pcdl.open_batch(ctx, polys[at[t]], Cs[at[t]], D, zs[t], None if ws is None else ws[at[t]], q, wb))
                        for t in range(T)]

            def multi():
                return pcdl.open_multi(ctx, polys, Cs, D, zs, qs, ws, wQ, q, wb)

            # every claim checked: the single opens at their own v = p_j(z_t) (from the multi opening's vs)
            vs, Q, us, Cm, x, v, pi = multi()
            pcdl.check(ctx, Cm, D, x, v, pi)
            for (j, t, pij), vi in zip(single(), vs):
                pcdl.check(ctx, Cs[j], D, zs[t], vi, pij)
            for t, (bvs, bC, bv, bpi) in batches():
                pcdl.check(ctx, bC, D, zs[t], bv, bpi)
            t_single, t_batch, t_multi = best(single), best(batches), best(multi)
            row = dict(probe="open_multi", n=n, d=D, k=k, T=T, m=m, ragged=ragged, hiding=hiding, single_ms=round(t_single, 3),
                       per_point_batch_ms=round(t_batch, 3), multi_ms=round(t_multi, 3),
                       multi_vs_batch=round(t_batch / t_multi, 2), check="accepted")
            # phases: the device entry points of open_multi, one by one, on the same inputs
            lens = np.full(k, n, dtype=np.uint64)
            packed = polys.reshape(-1, 4)
            qp = np.array([j for j, _ in qs], dtype=np.uint64)
            qt = np.array([t for _, t in qs], dtype=np.uint64)
            wts, scl = rs(m), rs(T)
            vs_o, rems, Qo = np.zeros((m, 4), dtype=np.uint64), np.zeros((T, 4), dtype=np.uint64), np.zeros(12, dtype=np.uint64)
            ev, allj, zero = np.zeros((k, 4), dtype=np.uint64), np.arange(k, dtype=np.uint64), np.zeros(k, dtype=np.uint64)
            x3, cs, one, deg = rs(1), rs(k), np.array([1, 0, 0, 0], dtype=np.uint64), C.c_uint64()
            for _ in range(2):
                t_up = clock(lambda: lib.halo_poly_upload(ctx._h, p64(packed), p64(lens), C.c_uint64(k), C.c_uint64(N)))
                t_ev = clock(lambda: lib.halo_poly_eval_queries(ctx._h, p64(zs), C.c_uint64(T), p64(qp), p64(qt), C.c_uint64(m),
                                                                p64(vs_o)))
                t_q = clock(lambda: lib.halo_poly_quotient(ctx._h, p64(zs), p64(scl), C.c_uint64(T), p64(qp), p64(qt), p64(wts),
                                                           C.c_uint64(m), p64(rems), p64(Qo)))
                t_u = clock(lambda: lib.halo_poly_eval_queries(ctx._h, p64(x3), C.c_uint64(1), p64(allj), p64(zero), C.c_uint64(k),
                                                               p64(ev)))
                t_c = clock(lambda: lib.halo_poly_lincomb_resident(ctx._h, p64(cs), p64(one), C.byref(deg)))
            row.update(upload_ms=round(t_up, 3), query_eval_ms=round(t_ev, 3), quotient_and_Q_msm_ms=round(t_q, 3),
                       u_eval_ms=round(t_u, 3), lincomb_ms=round(t_c, 3),
                       challenges_C_and_opening_ms=round(t_multi - t_up - t_ev - t_q - t_u - t_c, 3), upload_bytes=k * n * 32)
            emit(row)
            if not hiding:
                profiled.append((n, k, T, m, packed, lens, zs, scl, qp, qt, wts))
        del ps, polys

try:
    from torch.profiler import ProfilerActivity, profile

    # the quotient kernels of one halo_poly_quotient, and their multiplication rate: per coefficient and point t with m_t
    # terms, k_quot_chunks does m_t + 1 multiplications and k_quot_write m_t + 2 (the scans add about 3 per 16 coefficients)
    for n, k, T, m, packed, lens, zs, scl, qp, qt, wts in profiled:
        rems, Qo = np.zeros((T, 4), dtype=np.uint64), np.zeros(12, dtype=np.uint64)
        assert lib.halo_poly_upload(ctx._h, p64(packed), p64(lens), C.c_uint64(k), C.c_uint64(N)) == 0

        def quotient():
            return lib.halo_poly_quotient(ctx._h, p64(zs), p64(scl), C.c_uint64(T), p64(qp), p64(qt), p64(wts), C.c_uint64(m),
                                          p64(rems), p64(Qo))

        assert quotient() == 0
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                assert quotient() == 0
        d = dev_ms(prof, (("chunks_ms", "k_quot_chunks"), ("carry_ms", "k_quot_carry"), ("write_ms", "k_quot_write")))
        d = {a: round(b / 3, 4) for a, b in d.items()}
        tot = sum(d.values())
        mults = n * (2 * m + 3 * T) + 3 * T * (n // 16)
        emit(dict(probe="open_multi_quotient_kernels", n=n, k=k, T=T, m=m, **d, quotient_kernels_ms=round(tot, 4),
                  field_mults=mults, gmul_per_s=round(mults / (tot * 1e-3) / 1e9, 1)))

    # A/B on r07's one-point shapes: the K3b kernels against the K3c kernels, same inputs, alternating, 5 calls each
    for lg in (16, 20):
        n = 1 << lg
        for k in (8, 64):
            polys = rs(k, n)
            packed, lens = polys.reshape(-1, 4), np.full(k, n, dtype=np.uint64)
            z, alpha = rs(1), rs(1)[0]
            pw = np.zeros((k, 4), dtype=np.uint64)
            assert lib.halo_construct_powers(ctx._h, p64(alpha), C.c_uint64(k), p64(pw)) == 0
            allj, zero = np.arange(k, dtype=np.uint64), np.zeros(k, dtype=np.uint64)
            v_old, v_new = np.zeros((k, 4), dtype=np.uint64), np.zeros((k, 4), dtype=np.uint64)
            deg_o, deg_n = C.c_uint64(), C.c_uint64()
            zq = np.zeros(4, dtype=np.uint64)
            rems, Qo = np.zeros((1, 4), dtype=np.uint64), np.zeros(12, dtype=np.uint64)
            w1 = np.zeros((k, 4), dtype=np.uint64)
            one = pw[0].copy()

            def old():
                assert lib.halo_poly_eval_many(ctx._h, p64(packed), p64(lens), C.c_uint64(k), C.c_uint64(N), p64(z[0]), p64(v_old)) == 0
                assert lib.halo_poly_combine_resident(ctx._h, p64(alpha), C.byref(deg_o)) == 0

            def new():
                assert lib.halo_poly_eval_queries(ctx._h, p64(z), C.c_uint64(1), p64(allj), p64(zero), C.c_uint64(k), p64(v_new)) == 0
                assert lib.halo_poly_lincomb_resident(ctx._h, p64(pw), p64(zq), C.byref(deg_n)) == 0

            old()
            # the quotient call makes the upload's q resident for k_poly_lincomb (weight 0 in the A/B)
            assert lib.halo_poly_quotient(ctx._h, p64(z), p64(one), C.c_uint64(1), p64(allj[:1]), p64(zero[:1]), p64(w1[:1]),
                                          C.c_uint64(1), p64(rems), p64(Qo)) == 0
            new()
            assert np.array_equal(v_old, v_new) and deg_o.value == deg_n.value
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    new()
            dn = dev_ms(prof, (("eval_ms", "k_quot_"), ("combine_ms", "k_poly_lincomb")))
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    old()
            do = dev_ms(prof, (("eval_ms", "k_poly_eval"), ("powers_ms", "k_powers"), ("combine_ms", "k_poly_combine")))
            do["eval_ms"] = do.get("eval_ms", 0) + do.pop("powers_ms", 0)
            emit(dict(probe="open_multi_ab_one_point", n=n, k=k, outputs_equal=True,
                      old_eval_ms=round(do["eval_ms"] / 5, 4), new_eval_ms=round(dn["eval_ms"] / 5, 4),
                      old_combine_ms=round(do["combine_ms"] / 5, 4), new_combine_ms=round(dn["combine_ms"] / 5, 4)))
            del polys
except Exception as ex:  # the timings above stand without the profile
    emit(dict(probe="open_multi_device", error=repr(ex)))
ctx.close()
