"""Every MSM and opening variant that halo_set_tuning can select, against the oracle and against each other.

The knobs choose alternative CUDA kernels and launch geometries (the quad accumulation with 2 or 4 lanes per bucket and 4 or 6
CTAs per SM, thread-per-bucket and lane-claiming accumulation, the one-lane and quad bucket reductions, both pass-0 kernels of
the pair tree, the window of the frozen IPA tail, one or two lanes for batches).  Each row below first asserts, through
halo_test_msm_route, that the kernel it means to test actually ran -- a knob the policy overrides fails the row instead of
passing it silently -- and then compares the point with the oracle.  Expected points are computed once per input and shared by
every row; generator MSMs use the discrete logs of the derived generators (oracle.msm_derived_by_dlog), caller-base MSMs the
oracle's Pippenger.

test_every_tuning_key_is_documented_and_covered runs without a GPU: it keeps the keys halo_set_tuning accepts, the list in
include/halo_b200.h and the coverage of this file (or of the test named for a key in ELSEWHERE) in step."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from oracle.oracle import R_MOD

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

# 2^17 + 4096 generators: the FIXED-base path needs n >= 2^17 points (msm_gens_device), and the extra 4096 give it a ragged
# length at an offset
N_GENS = (1 << 17) + 4096
N_FIXED, OFF_FIXED = (1 << 17) + 1234, 777

# the values halo_ctx starts with (csrc/common.cuh); every row restores them in `finally`
DEFAULTS = {"acc_static": 0, "acc_blocks_per_sm": 0, "acc_quad": 1, "acc_quad_max_buckets": 1 << 15, "acc_quad_lanes": 0,
            "acc_quad_blocks": 0, "pair_passes": -1, "pair_bwd_async": 1, "reduce_quad": 1, "ipa_two_lanes": 1,
            "ipa_freeze_len": 0, "ipa_frozen_c": 9, "sort_ahead": 1}

# keys whose variants are compared with the oracle in another module (host buffers, sorts, deferred stages, batch checks):
# key -> test file that sets it
ELSEWHERE = {
    "split_blocking": "test_gpu_core.py", "split_first_16ths": "test_gpu_core.py", "split_second_16ths": "test_gpu_core.py",
    "stage_pageable": "test_gpu_core.py", "stage_threads": "test_gpu_core.py", "sort2": "test_gpu_core.py",
    "sort2_min_lg": "test_gpu_core.py", "ipa_defer_rounds": "test_gpu_pcdl.py", "ipa_defer2_rounds": "test_gpu_pcdl.py",
    "ipa_fold_call_min_lg": "test_gpu_pcdl.py", "combine_min_outputs": "test_gpu_batch_verifier.py",
}


def _plan_nb(c, fixed=False):
    """Bucket count of a plan of window c (csrc/msm.cu plan_fill)."""
    return (1 << (c - 1)) * (1 if fixed else 255 // c + 1)


def _auto_c(n):
    """Window of msm_make_plan for n points."""
    lg = max(0, (n - 1).bit_length())
    return 4 if lg <= 6 else 7 if lg <= 8 else 8 if lg <= 10 else 11 if lg <= 12 else 10 if lg <= 15 else 11 if lg <= 16 else 13 if lg <= 19 else 16


def _restore(ctx):
    for k, v in DEFAULTS.items():
        ctx.set_tuning(k, v)
    ctx.set_msm_window(0)
    ctx.set_profiling(False)
    ctx.set_fixed_base(True)


def _route(ctx, lane=0, **want):
    r = ctx.test_msm_route(lane)
    bad = {k: (r[k], v) for k, v in want.items() if r[k] != v}
    assert not bad, f"route {bad} (got, wanted); full record {r}"
    return r


@pytest.fixture(scope="module")
def tv(ctx, oracle):
    """The session context with N_GENS derived generators, the oracle holding the same parameters, and the expected point
    of every input set.  Generator cases: name -> (scalars, offset, expected); caller-base cases: name -> (bases, scalars,
    infinity flags, expected)."""
    import torch

    O = oracle
    ctx.derive_generators(N_GENS)
    S, H = ctx.get_SH()
    O.set_params(S, H, ctx.get_generators(0, N_GENS))
    _restore(ctx)
    big = O.random_scalars(1, 5)[0]

    def g(sc, off):
        sc = np.ascontiguousarray(sc, dtype=np.uint64)
        return sc, off, O.msm_derived_by_dlog(off, sc, threads=8)

    small = {"uniform": g(O.random_scalars(5000, 1), 100)}
    for n in (1, 2, 33, 1023, 5000, (1 << 16) - 4321):  # ragged, at an offset
        small[f"ragged_{n}"] = g(O.random_scalars(n, 10 + n), 777)
    small["zeros"] = g(np.zeros((4096, 4), dtype=np.uint64), 3)
    small["r_minus_1"] = g(np.tile(O.to_mont([R_MOD - 1])[0], (4096, 1)), 5)
    small["two_254_plus_i"] = g(O.to_mont([(1 << 254) + i for i in range(4096)]), 9)
    small["all_equal"] = g(np.tile(big, (5000, 1)), 11)  # one bucket per window holds every entry: the split hand-off

    # deep at window 4 (n W >= 256 NB) and below the 2^21 entries from which the policy adds pair passes
    deep = {"uniform": g(O.random_scalars(20000, 20), 777), "all_equal": g(np.tile(big, (5000, 1)), 0)}
    fixed = {"uniform": g(O.random_scalars(N_FIXED, 30), OFF_FIXED), "all_equal": g(np.tile(big, (1 << 17, 1)), 0),
             "two_254_plus_i": g(O.to_mont([(1 << 254) + i for i in range(1 << 17)]), N_GENS - (1 << 17))}

    # caller bases (halo_msm): duplicates, s and -s on one base, infinity flags (test_gpu_core's pair-tree edge inputs)
    n = 2048
    gs = ctx.get_generators(100, n).copy()
    sc = O.random_scalars(n, 33)
    gs[1::2] = gs[0::2]
    sc[1:1024:2] = sc[0:1024:2]
    sc[1025::2] = ctx.test_fp_op(1, 5, sc[1024::2])
    inf = np.zeros(n, dtype=np.uint8)
    inf[[5, 6, 77, 1500, 2047]] = 1
    same_g, same_s = np.tile(gs[3], (n, 1)), np.tile(sc[3], (n, 1))
    g2 = np.concatenate([gs[:n // 2], gs[:n // 2]])
    s2 = np.concatenate([sc[:n // 2], ctx.test_fp_op(1, 5, sc[:n // 2])])
    bases = {"dup_cancel_inf": (gs, sc, inf, O.msm_affine(gs, sc, inf=inf, threads=8)),
             "one_base_one_scalar": (same_g, same_s, None, O.msm_affine(same_g, same_s, threads=8)),
             "all_cancel": (g2, s2, None, O.pt_from_affine_ints(None))}
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    yield dict(ctx=ctx, O=O, small=small, deep=deep, fixed=fixed, bases=bases, sm=sm)
    _restore(ctx)
    ctx.derive_generators(1 << 16)
    S, H = ctx.get_SH()
    O.set_params(S, H, ctx.get_generators(0, 1 << 16))


def _gens(tv, cases, want, names=None, **route):
    """Runs the generator cases, asserts the route of each (want(c) -> dict, or route kwargs) and the oracle's point."""
    ctx, O = tv["ctx"], tv["O"]
    got = {}
    for name in names or cases:
        sc, off, exp = cases[name]
        p = ctx.msm_gens(sc, off=off)
        r = ctx.test_msm_route(0)
        w = dict(route, **(want(r) if want else {}))
        bad = {k: (r[k], v) for k, v in w.items() if r[k] != v}
        assert not bad, f"{name}: route {bad} (got, wanted); full record {r}"
        assert O.pt_eq(p, exp), (name, r)
        got[name] = p
    return got


def _bases(tv, windows=(0,), want=None, **route):
    ctx, O = tv["ctx"], tv["O"]
    for c in windows:
        ctx.set_msm_window(c)
        for name, (b, s, inf, exp) in tv["bases"].items():
            p = ctx.msm(b, s, inf)
            r = ctx.test_msm_route(0)
            w = dict(route, **(want(r) if want else {}))
            bad = {k: (r[k], v) for k, v in w.items() if r[k] != v}
            assert not bad, f"{name} c={c}: route {bad} (got, wanted); full record {r}"
            assert O.pt_eq(p, exp), (name, c)
    ctx.set_msm_window(0)


# ---- accumulation ---------------------------------------------------------------------------------------------------------
@gpu
def test_default_policy_routes(tv):
    """Without knobs: small MSMs take the quad kernel (4 lanes, 4 CTAs per SM, quad reduction), deep variable-base ones the
    thread-per-bucket kernel, FIXED-base ones the automatic pair passes.  The matrix below departs from these."""
    ctx = tv["ctx"]
    try:
        _gens(tv, tv["small"], None, acc=2, quad_lanes=4, quad_blocks=4, P=0, reduce_quad=1, two_lanes=0, fixed=0)
        _bases(tv, acc=2, quad_lanes=4, quad_blocks=4)
        ctx.set_msm_window(4)
        _gens(tv, tv["deep"], None, acc=1, P=0, c=4)
        ctx.set_msm_window(0)
        ctx.precompute_generators(11)
        _gens(tv, tv["fixed"], None, fixed=1, c=11, pass0_async=1)
        assert ctx.test_msm_route(0)["c"] == 0  # the read cleared the record
    finally:
        _restore(ctx)


@gpu
@pytest.mark.parametrize("lanes,blocks", [(2, 4), (2, 6), (4, 4), (4, 6)])
def test_accumulate_quad_lanes_and_blocks(tv, lanes, blocks):
    """k_accumulate_quad in each of its four builds: ragged sizes, edge scalars, oversized buckets (split hand-off), caller
    bases with duplicates / cancellations / infinity, forced windows 4, 7 and 11, and the bucket count just at
    acc_quad_max_buckets."""
    ctx = tv["ctx"]
    want = dict(acc=2, quad_lanes=lanes, quad_blocks=blocks, P=0)
    try:
        ctx.set_tuning("acc_quad_lanes", lanes)
        ctx.set_tuning("acc_quad_blocks", blocks)
        _gens(tv, tv["small"], None, **want)
        _bases(tv, windows=(0, 7, 11), **want)
        for c, names in ((4, ["ragged_33", "ragged_1023"]), (7, ["ragged_1023", "all_equal", "r_minus_1"]),
                         (11, ["ragged_1023", "all_equal", "r_minus_1"])):  # (from 2048 points window 4 is deep: static)
            ctx.set_msm_window(c)
            _gens(tv, tv["small"], None, names=names, c=c, **want)
        ctx.set_msm_window(0)
        nb = _plan_nb(_auto_c(5000))
        ctx.set_tuning("acc_quad_max_buckets", nb)  # NB == the limit: still quad
        _gens(tv, tv["small"], None, names=["uniform", "ragged_5000", "all_equal"], **want)
    finally:
        _restore(ctx)


@gpu
def test_accumulate_quad_off_and_limit(tv):
    """acc_quad = 0, and acc_quad_max_buckets one below the plan's bucket count (and 0): the small MSMs fall to the
    lane-claiming k_accumulate, with its grid of min(NB / 128, 4 CTAs per SM)."""
    ctx, sm = tv["ctx"], tv["sm"]
    grid = lambda r: dict(acc_grid=min(math.ceil(_plan_nb(r["c"]) / 128), sm * 4))  # noqa: E731
    try:
        ctx.set_tuning("acc_quad", 0)
        _gens(tv, tv["small"], grid, acc=0, quad_lanes=0, P=0)
        _bases(tv, windows=(0, 7), want=grid, acc=0)
        ctx.set_tuning("acc_quad", 1)
        ctx.set_tuning("acc_quad_max_buckets", _plan_nb(_auto_c(5000)) - 1)
        _gens(tv, tv["small"], grid, names=["uniform", "ragged_5000", "all_equal"], acc=0)
        _gens(tv, tv["small"], None, names=["ragged_33"], acc=2)  # fewer buckets: still quad
        ctx.set_tuning("acc_quad_max_buckets", 0)
        _gens(tv, tv["small"], grid, acc=0)
    finally:
        _restore(ctx)


@gpu
@pytest.mark.parametrize("P", [0, 2, 4])
@pytest.mark.parametrize("static", [1, 2])
def test_accumulate_static_and_claiming(tv, static, P):
    """acc_static = 1 (k_accumulate_static, both template copies) and 2 (lane claiming forced on deep buckets), with and
    without pair passes, at a deep variable-base shape (c = 4, 20 000 points) and at shallow ones."""
    ctx = tv["ctx"]
    kind = 1 if static == 1 else 0
    try:
        ctx.set_tuning("acc_static", static)
        ctx.set_tuning("pair_passes", P)
        ctx.set_msm_window(4)
        _gens(tv, tv["deep"], None, acc=kind, P=P, c=4)
        ctx.set_msm_window(0)
        _gens(tv, tv["small"], None, names=["uniform", "ragged_1", "ragged_1023", "ragged_61215", "all_equal", "two_254_plus_i"],
              acc=kind, P=P)
        _bases(tv, windows=(0,), acc=kind, P=P)
    finally:
        _restore(ctx)


@gpu
@pytest.mark.parametrize("bps", [1, 2, 8])
def test_accumulate_blocks_per_sm(tv, bps):
    """acc_blocks_per_sm: few persistent CTAs of k_accumulate, each looping over many buckets (forced window 16: 2^19
    buckets, far more than the grid), deep buckets (acc_static = 2) and a small MSM (acc_quad = 0)."""
    ctx, sm = tv["ctx"], tv["sm"]
    try:
        ctx.set_tuning("acc_blocks_per_sm", bps)
        ctx.set_msm_window(16)
        _gens(tv, tv["deep"], None, acc=0, acc_grid=sm * bps, c=16)
        ctx.set_tuning("acc_static", 2)
        ctx.set_msm_window(4)
        _gens(tv, tv["deep"], None, acc=0, acc_grid=min(_plan_nb(4) // 128, sm * bps), c=4)
        ctx.set_tuning("acc_static", 0)
        ctx.set_msm_window(13)
        ctx.set_tuning("acc_quad", 0)
        _gens(tv, tv["small"], None, names=["uniform", "ragged_33", "all_equal"], acc=0, acc_grid=min(_plan_nb(13) // 128, sm * bps))
    finally:
        _restore(ctx)


# ---- FIXED base ------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("c", [8, 11, 13, 16])
def test_fixed_base_variants(tv, c):
    """FIXED-base tables at window c: the automatic route, then without pair passes through each accumulation kernel (the
    quad builds, thread per bucket, lane claiming with 2 CTAs per SM) and the one-lane reduction."""
    ctx, sm = tv["ctx"], tv["sm"]
    nb = _plan_nb(c, fixed=True)
    rows = [({}, dict()),
            ({"pair_passes": 0}, dict(P=0, acc=2, quad_lanes=4, quad_blocks=4)),
            ({"pair_passes": 0, "acc_quad_lanes": 2, "acc_quad_blocks": 6}, dict(P=0, acc=2, quad_lanes=2, quad_blocks=6)),
            ({"pair_passes": 0, "acc_static": 1}, dict(P=0, acc=1)),
            ({"pair_passes": 0, "acc_static": 2, "acc_blocks_per_sm": 2}, dict(P=0, acc=0, acc_grid=min(math.ceil(nb / 128), 2 * sm))),
            ({"pair_passes": 0, "acc_quad": 0, "reduce_quad": 0}, dict(P=0, acc=0, reduce_quad=0))]
    try:
        ctx.precompute_generators(c)
        first = None
        for knobs, want in rows:
            _restore(ctx)
            for k, v in knobs.items():
                ctx.set_tuning(k, v)
            got = _gens(tv, tv["fixed"], None, fixed=1, c=c, **want)
            first = first or got
            assert all(tv["O"].pt_eq(got[k], first[k]) for k in got), knobs
    finally:
        _restore(ctx)


# ---- bucket reduction ------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("quad", [0, 1])
def test_reduce_variants(tv, quad):
    """reduce_quad on single-slab (variable c = 7, FIXED c = 8) and multi-slab plans (variable c = 13, FIXED c = 16).  The
    quad reduction is refused above its size limit: variable base at c = 16 (2^19 buckets) reduces with one lane either way."""
    ctx = tv["ctx"]
    try:
        ctx.set_tuning("reduce_quad", quad)
        for c in (7, 13):
            ctx.set_msm_window(c)
            _gens(tv, tv["small"], None, names=["uniform", "ragged_33", "all_equal", "two_254_plus_i"], c=c, reduce_quad=quad)
        _bases(tv, windows=(7, 13), reduce_quad=quad)
        ctx.set_msm_window(16)
        _gens(tv, tv["deep"], None, c=16, reduce_quad=0)
        ctx.set_msm_window(0)
        for c in (8, 16):
            ctx.precompute_generators(c)
            _gens(tv, tv["fixed"], None, fixed=1, c=c, reduce_quad=quad)
    finally:
        _restore(ctx)


# ---- pair tree -------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("async_,P", [(0, 1), (0, 3), (0, 5), (0, 8), (1, 1), (1, 3), (1, 5), (1, 7), (1, 8)])
def test_pair_tree_pass0_kernels(tv, async_, P):
    """Both pass-0 kernels of the pair tree (k_pair_bwd0 with cp.async staging, k_pair_bwd<true> with per-lane gathers) at P =
    1 .. 8 passes, variable and FIXED base: the tangent (P + P), cancellation (P - P) and infinity operands of caller bases at
    windows 4, 8 and 12, ragged and oversized-bucket generator inputs."""
    ctx = tv["ctx"]
    want = dict(P=P, pass0_async=async_)
    try:
        ctx.set_tuning("pair_bwd_async", async_)
        ctx.set_tuning("pair_passes", P)
        _bases(tv, windows=(4, 8, 12), **want)
        _gens(tv, tv["small"], None, names=["uniform", "ragged_1", "ragged_2", "ragged_33", "ragged_1023", "all_equal", "zeros",
                                            "r_minus_1"], fixed=0, **want)
        ctx.precompute_generators(11)
        _gens(tv, tv["fixed"], None, fixed=1, **want)
    finally:
        _restore(ctx)


# ---- batches on two lanes, profiling ---------------------------------------------------------------------------------------
def _h_msm_with(ctx, xis, bases, sc, inf):
    from halo_accumulation_b200._capi import p64

    out_h, out_s = np.zeros(12, dtype=np.uint64), np.zeros(12, dtype=np.uint64)
    ctx._chk(ctx._lib.halo_h_msm_with(ctx._h, p64(xis), xis.shape[0] - 1, p64(bases), inf.ctypes.data_as(C.POINTER(C.c_uint8)),
                                      p64(sc), C.c_uint64(sc.shape[0]), p64(out_h), p64(out_s)))
    return out_h, out_s


def _h_msm_batch(ctx, xis_list, w, bases, sc, inf):
    u64 = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint64))  # noqa: E731
    lgs = np.array([x.shape[0] - 1 for x in xis_list], dtype=np.uint32)
    xis = np.ascontiguousarray(np.concatenate(xis_list))
    out = np.zeros(12, dtype=np.uint64)
    ctx._chk(ctx._lib.halo_h_msm_batch(ctx._h, u64(xis), lgs.ctypes.data_as(C.POINTER(C.c_uint32)), u64(w), len(xis_list), u64(bases),
                                       inf.ctypes.data_as(C.POINTER(C.c_uint8)), u64(sc), sc.shape[0], u64(out)))
    return out


@gpu
@pytest.mark.parametrize("profile", [False, True])
def test_two_lane_batches_and_profiling(tv, profile):
    """halo_msm_multi, halo_h_msm_with and the batch decider's halo_h_msm_batch with profiling off (msm_multi and h_msm_with on
    two lanes) and on (one lane, event marks): the oracle's points either way; the profiled MSM reports six finite timings."""
    ctx, O = tv["ctx"], tv["O"]
    gs, sc, inf, exp_b = tv["bases"]["dup_cancel_inf"]
    s1, s2 = O.random_scalars(4096, 501), O.random_scalars(33, 502)
    probs = [(gs[:1000], sc[:1000], inf[:1000], 0), (None, s1, None, 100), (None, s2, None, 7)]
    exps = [O.msm_affine(gs[:1000], sc[:1000], inf=inf[:1000], threads=8), O.msm_derived_by_dlog(100, s1, threads=8),
            O.msm_derived_by_dlog(7, s2, threads=8)]
    lanes = 0 if profile else 1
    try:
        ctx.set_profiling(profile)
        ctx.test_msm_route(1)
        got = ctx.msm_multi(probs)
        _route(ctx, 0, two_lanes=lanes)
        assert (ctx.test_msm_route(1)["c"] > 0) == (not profile)
        for g, e in zip(got, exps):
            assert O.pt_eq(g, e)
        lg = 12
        xis = O.random_scalars(lg + 1, 71)
        exp_h = O.msm_derived_by_dlog(0, O.h_get_poly(xis), threads=8)
        out_h, out_s = _h_msm_with(ctx, xis, gs, sc, inf)
        _route(ctx, 0, two_lanes=lanes)
        assert (ctx.test_msm_route(1)["c"] > 0) == (not profile)
        assert O.pt_eq(out_h, exp_h) and O.pt_eq(out_s, exp_b)
        xs = [O.random_scalars(l + 1, 80 + l) for l in (3, 12, 16)]
        w = O.random_scalars(len(xs), 90)
        exp = exp_b
        for x, wj in zip(xs, w):
            exp = O.pt_add(exp, O.pt_mul(O.msm_derived_by_dlog(0, O.h_get_poly(x), threads=8), wj))
        assert O.pt_eq(_h_msm_batch(ctx, xs, w, gs, sc, inf), exp)
        _route(ctx, 0, two_lanes=-1, c=_auto_c(1 << 16))  # generator part on lane 0, companion on lane 1, outside msm_batch
        _route(ctx, 1, two_lanes=-1, c=_auto_c(gs.shape[0]))
        s, off, e = tv["small"]["uniform"]
        assert O.pt_eq(ctx.msm_gens(s, off=off), e)
        t = ctx.last_msm_timings()
        if profile:
            v = list(t.values())
            assert len(v) == 6 and all(math.isfinite(x) and x >= 0 for x in v) and v[5] > 0, t
    finally:
        _restore(ctx)


# ---- opening ---------------------------------------------------------------------------------------------------------------
def _same_proof(O, a, b):
    assert a.lg_n == b.lg_n and a.hiding == b.hiding
    for i in range(a.lg_n):
        assert O.pt_eq(np.array(a.Ls[i]), np.array(b.Ls[i])), f"L[{i}]"
        assert O.pt_eq(np.array(a.Rs[i]), np.array(b.Rs[i])), f"R[{i}]"
    assert O.pt_eq(np.array(a.U), np.array(b.U))
    assert list(a.c) == list(b.c)
    if a.hiding:
        assert O.pt_eq(np.array(a.C_bar), np.array(b.C_bar)) and list(a.w_prime) == list(b.w_prime)


@gpu
@pytest.mark.parametrize("lg,hiding", [(12, False), (12, True), (14, True), (16, False), (16, True)])
def test_open_frozen_tail_window(tv, lg, hiding):
    """pcdl.open with the frozen-tail round MSMs at windows 4, 9, 13, 16 and freeze lengths 256 and 2048: the oracle's
    proof (same L, R, U, c) every time, accepted by pcdl.check; the last round's MSM ran at the window asked for."""
    from halo_accumulation_b200 import pcdl

    ctx, O = tv["ctx"], tv["O"]
    n = 1 << lg
    d = n - 1
    p = O.random_scalars(n - 7, 900 + lg)
    z = O.random_scalars(1, 901)[0]
    w, wb = O.random_scalars(2, 902) if hiding else (None, None)
    q = O.random_scalars(p.shape[0] - 1, 903) if hiding else None
    Cm = pcdl.commit(ctx, p, d, w)
    ref = O.pcdl_open(p, Cm, d, z, w, q, wb, threads=16)
    v = O.scalar_dot(p, O.construct_powers(z, p.shape[0]))
    try:
        for freeze in (256, 2048):
            ctx.set_tuning("ipa_freeze_len", freeze)
            for c in (4, 9, 13, 16):
                ctx.set_tuning("ipa_frozen_c", c)
                ctx.test_msm_route(1)
                pi = pcdl.open(ctx, p, Cm, d, z, w, q, wb)
                # the last round's R ran on lane 1 at the window asked for; U = <s, G> over the frozen tail (lane 0, after
                # the rounds) keeps the automatic window of its length
                _route(ctx, 1, c=c, fixed=0, two_lanes=1)
                _route(ctx, 0, c=_auto_c(min(n, freeze)), fixed=0)
                _same_proof(O, pi, ref)
                pcdl.check(ctx, Cm, d, z, v, pi)
    finally:
        _restore(ctx)


@gpu
def test_open_two_lanes_fixed_deferred(halo, oracle):
    """ipa_two_lanes on FIXED tables with deferred head rounds, at 2^19 where it decides the lanes (smaller L / R pairs share
    two lanes anyway): round 0's L and R against the oracle (<c_hi, G_lo> + <c_hi, z_lo> H' and its mirror, through the
    generators' discrete logs) on one lane and on two, and the full openings of both equal and accepted by pcdl.check."""
    from halo_accumulation_b200 import pcdl
    from halo_accumulation_b200._capi import p64

    O = oracle
    n = 1 << 19
    m = n // 2
    ctx = halo.Context(0, n)
    try:
        ctx.derive_generators(n)
        ctx.precompute_generators(0)
        S, _ = ctx.get_SH()
        p = O.random_scalars(n - 3, 41)
        z = O.random_scalars(1, 42)[0]
        c = np.zeros((n, 4), dtype=np.uint64)
        c[:p.shape[0]] = p
        zp = O.construct_powers(z, n)
        expL = O.pt_add(O.msm_derived_by_dlog(0, c[m:], threads=16), O.pt_mul(S, O.scalar_dot(c[m:], zp[:m])))
        expR = O.pt_add(O.msm_derived_by_dlog(m, c[:m], threads=16), O.pt_mul(S, O.scalar_dot(c[:m], zp[m:])))
        lib = ctx._lib
        lib.halo_ipa_destroy.restype = None
        proofs = []
        for two in (0, 1):
            ctx.set_tuning("ipa_two_lanes", two)
            st = C.c_void_p()
            v = np.zeros(4, dtype=np.uint64)
            ctx.test_msm_route(1)
            ctx._chk(lib.halo_ipa_begin(ctx._h, p64(p), C.c_uint64(p.shape[0]), C.c_uint64(n), p64(np.ascontiguousarray(z)),
                                        C.byref(st), p64(v)))
            try:
                L, R = np.zeros(12, dtype=np.uint64), np.zeros(12, dtype=np.uint64)
                ctx._chk(lib.halo_ipa_set_hprime(st, p64(S)))
                ctx._chk(lib.halo_ipa_round_lr(st, p64(L), p64(R)))
            finally:
                lib.halo_ipa_destroy(st)
            _route(ctx, 0, fixed=1, two_lanes=two)
            assert (ctx.test_msm_route(1)["c"] > 0) == bool(two)
            assert O.pt_eq(L, expL) and O.pt_eq(R, expR), two
            assert v.tolist() == O.scalar_dot(p, zp[:p.shape[0]]).tolist()
            Cm = pcdl.commit(ctx, p, n - 1)
            pi = pcdl.open(ctx, p, Cm, n - 1, z)
            pcdl.check(ctx, Cm, n - 1, z, v, pi)
            proofs.append(pi)
        _same_proof(O, proofs[0], proofs[1])
    finally:
        ctx.close()


# ---- the pipelined sort-ahead --------------------------------------------------------------------------------------------
@gpu
def test_sort_ahead_ctas(halo, oracle):
    """sort_ahead (CTAs per SM of the counting sort that runs beside the previous pipelined MSM, from 2^22 points): off, the
    default and a wider grid give the oracle's point for two calls in flight, variable and FIXED base."""
    O = oracle
    n = 1 << 22
    ctx = halo.Context(0, n)
    try:
        ctx.derive_generators(n)
        a, b = O.random_scalars(n, 51), O.random_scalars(n, 52)
        ea, eb = O.msm_derived_by_dlog(0, a, threads=16), O.msm_derived_by_dlog(0, b, threads=16)
        for fixed in (False, True):
            if fixed:
                ctx.precompute_generators(0)
            ctx.set_fixed_base(fixed)
            for ahead in (0, 1, 4):
                ctx.set_tuning("sort_ahead", ahead)
                t0, t1 = ctx.msm_gens_submit(a), ctx.msm_gens_submit(b)
                assert O.pt_eq(ctx.msm_gens_collect(t0), ea) and O.pt_eq(ctx.msm_gens_collect(t1), eb), (fixed, ahead)
                _route(ctx, 0, fixed=int(fixed), two_lanes=-1)
    finally:
        ctx.close()


# ---- accepted values -------------------------------------------------------------------------------------------------------
@gpu
def test_tuning_values_out_of_range_are_refused(tv, halo):
    """Values that would become a plan or a launch geometry are refused (HALO_EINVAL) instead of cast or replaced; the clamped
    host-buffer knobs keep clamping; 0 stays the automatic value where the header says so."""
    ctx = tv["ctx"]
    bad = {"ipa_frozen_c": [-1, 1, 3, 21, 25], "acc_quad_lanes": [-1, 1, 3, 8], "acc_quad_blocks": [-1, 2, 5, 8],
           "acc_blocks_per_sm": [-1, 33, -2**31], "acc_quad_max_buckets": [-1, -2**31], "pair_passes": [-2, -100],
           "acc_static": [-1, 3, 7]}
    good = {"ipa_frozen_c": [0, 4, 20], "acc_quad_lanes": [0, 2, 4], "acc_quad_blocks": [0, 4, 6], "acc_blocks_per_sm": [0, 1, 32],
            "acc_quad_max_buckets": [0, 1, 2**31 - 1], "pair_passes": [-1, 0, 8, 9], "acc_static": [0, 1, 2],
            "split_first_16ths": [0, 99], "split_second_16ths": [-5, 99], "stage_threads": [0, 99]}
    try:
        for key, vals in bad.items():
            for v in vals:
                with pytest.raises(halo.HaloError) as e:
                    ctx.set_tuning(key, v)
                assert e.value.code == -1, (key, v)
        for key, vals in good.items():
            for v in vals:
                ctx.set_tuning(key, v)
        with pytest.raises(halo.HaloError):
            ctx.set_tuning("no_such_key", 0)
        _restore(ctx)
        ctx.set_tuning("pair_passes", 9)  # above 8 means 8
        _gens(tv, tv["small"], None, names=["uniform"], P=8)
    finally:
        _restore(ctx)
        ctx.set_tuning("split_first_16ths", 2)
        ctx.set_tuning("split_second_16ths", 5)
        ctx.set_tuning("stage_threads", 4)


# ---- the key list stays in step (no GPU) -----------------------------------------------------------------------------------
def _read(*parts):
    with open(os.path.join(ROOT, *parts)) as f:
        return f.read()


def test_every_tuning_key_is_documented_and_covered():
    """The keys halo_set_tuning accepts (csrc/capi.cu) are exactly the keys include/halo_b200.h documents, and every one of them
    is set by a row of this file or by the test module ELSEWHERE names for it.  A knob added without a test fails here."""
    capi = _read("halo-accumulation_b200", "csrc", "capi.cu")
    body = capi[capi.index("int halo_set_tuning("):]
    body = body[:body.index("\n}\n")]
    accepted = set(re.findall(r'!strcmp\(key, "(\w+)"\)\) ctx->', body))
    header = _read("include", "halo_b200.h")
    doc = header[header.index("/* Measurement knobs"):header.index("int halo_set_tuning(")]
    documented = set(re.findall(r'"(\w+)"', doc))
    assert len(accepted) >= 24, accepted
    assert accepted == documented, (sorted(accepted - documented), sorted(documented - accepted))
    here = _read("tests", "test_gpu_tuning.py")
    rows = here[here.index("# ---- accumulation"):here.index("# ---- accepted values")]
    here_keys = set(re.findall(r'set_tuning\("(\w+)"', rows)) | {k for k in re.findall(r'"(\w+)": \d', rows) if k in accepted}
    missing = []
    for key in sorted(accepted):
        if key in here_keys:
            continue
        where = ELSEWHERE.get(key)
        if not where or f'set_tuning("{key}"' not in _read("tests", where):
            missing.append(key)
    assert not missing, f"halo_set_tuning keys no test exercises: {missing}"
    assert set(DEFAULTS) <= accepted and not set(ELSEWHERE) & set(DEFAULTS)
