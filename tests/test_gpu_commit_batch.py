"""Batch commit (pcdl.commit_batch, halo_msm_gens_many; DESIGN.md K2c): k commitments as segmented MSMs over the generators.

Every output is compared with the oracle -- its pcdl_commit at small sizes, the discrete logs of the derived generators
(msm_derived_by_dlog) plus w S at large ones -- and with the single pcdl.commit on the GPU.  The variant rows force kernels with
the existing knobs and assert through halo_test_msm_route that the segmented MSM ran them before they compare points."""
import ctypes as C

import numpy as np
import pytest

from oracle.oracle import R_MOD

gpu = pytest.mark.gpu

N_GENS = 1 << 20
DEFAULTS = {"acc_quad": 1, "pair_passes": -1, "reduce_quad": 1, "sort2_min_lg": 26}
HALO_EINVAL, HALO_ESTATE = -1, -6


def _restore(ctx):
    for k, v in DEFAULTS.items():
        ctx.set_tuning(k, v)
    ctx.set_msm_window(0)
    ctx.set_fixed_base(True)


@pytest.fixture(scope="module")
def env(ctx, oracle, halo):
    from halo_accumulation_b200 import pcdl

    O = oracle
    ctx.derive_generators(N_GENS)
    S, H = ctx.get_SH()
    O.set_params(S, H, ctx.get_generators(0, N_GENS))
    ctx.precompute_generators(0)  # FIXED-base tables for 2^20 generators
    _restore(ctx)
    yield dict(ctx=ctx, O=O, pcdl=pcdl, S=S, halo=halo)
    _restore(ctx)
    ctx.derive_generators(1 << 16)
    S, H = ctx.get_SH()
    O.set_params(S, H, ctx.get_generators(0, 1 << 16))
    bad, live = halo.check_canaries()  # no kernel of this module wrote past a device buffer
    assert bad == 0, (bad, live)


def _expected(env, p, w):
    """sum_i p_i G_i (+ w S) through the discrete logs of the derived generators"""
    O = env["O"]
    e = O.msm_derived_by_dlog(0, p, threads=8) if len(p) else O.pt_from_affine_ints(None)
    return O.pt_add(e, O.pt_mul(env["S"], w)) if w is not None else e


def _check(env, ps, d, ws=None, oracle_commit=False, singles=True):
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    got = pcdl.commit_batch(ctx, ps, d, ws)
    route = ctx.test_msm_route(0)
    assert got.shape == (len(ps), 12)
    for j, p in enumerate(ps):
        w = None if ws is None else ws[j]
        exp = O.pcdl_commit(p, d, w, threads=8) if oracle_commit else _expected(env, p[:d + 1], w)
        assert O.pt_eq(got[j], exp), (j, len(p))
        if singles:
            assert O.pt_eq(got[j], pcdl.commit(ctx, p, d, w)), j
    return got, route


def _edge_polys(O, n, seed):
    big = O.random_scalars(1, seed)[0]
    return [O.random_scalars(n, seed + 1),
            np.zeros((n, 4), dtype=np.uint64),                       # all zero
            np.tile(big, (n, 1)),                                    # all equal: oversized buckets (split hand-off)
            np.tile(O.to_mont([R_MOD - 1])[0], (n, 1)),              # r - 1
            O.random_scalars(n, seed + 1)]                           # a duplicate of the first


@gpu
@pytest.mark.parametrize("hiding", [False, True])
def test_small_against_oracle(env, hiding):
    """k = 1, 2, 3 and a ragged batch with edge inputs (lengths 1, 2, 4095, 4096, empty, zero, equal, r - 1, duplicates, more
    coefficients than d + 1 with a zero tail) against the oracle's pcdl_commit and the single commit."""
    O = env["O"]
    d = 4095
    ws_all = O.random_scalars(16, 7)
    for k in (1, 2, 3):
        ps = [O.random_scalars(4096 - j, 10 + j) for j in range(k)]
        _check(env, ps, d, ws_all[:k] if hiding else None, oracle_commit=True)
    long_zero_tail = np.concatenate([O.random_scalars(4096, 30), np.zeros((5, 4), dtype=np.uint64)])
    ps = [O.random_scalars(1, 20), O.random_scalars(2, 21), O.random_scalars(4095, 22), np.zeros((0, 4), dtype=np.uint64),
          *_edge_polys(O, 4096, 23), long_zero_tail, O.random_scalars(4096, 31)]
    _check(env, ps, d, ws_all[:len(ps)] if hiding else None, oracle_commit=True)


@gpu
def test_k64_and_large_ragged(env):
    """64 polynomials of 2^12 (one group), a ragged batch of 2^16, 2^17 (the FIXED threshold) and 2^20 coefficients, hiding,
    FIXED base on and off."""
    ctx, O = env["ctx"], env["O"]
    ps = [O.random_scalars(4096, 100 + j) for j in range(64)]
    ps[7] = ps[3]
    ws = O.random_scalars(64, 8)
    got, _ = _check(env, ps, 4095, ws, singles=False)
    for j in (0, 3, 7, 63):
        assert O.pt_eq(got[j], env["pcdl"].commit(ctx, ps[j], 4095, ws[j]))
    d = N_GENS - 1
    big = [O.random_scalars(1 << 16, 200), O.random_scalars(1 << 17, 201), O.random_scalars(1 << 17, 202), O.random_scalars(1 << 20, 203),
           O.random_scalars((1 << 16) + 3, 204)]
    try:
        for fixed in (True, False):
            ctx.set_fixed_base(fixed)
            _check(env, big, d, O.random_scalars(len(big), 9))
    finally:
        _restore(ctx)


# ---- variants of the segmented MSM, forced with the existing knobs ----------------------------------------------------------
VARIANTS = [
    # name, knobs, window, polynomial length, count, expected route entries (lengths n .. n + 2, plus zero / equal / r - 1)
    ("fixed_pairs_auto", {}, 0, 1 << 17, 4, dict(fixed=1, c=19)),
    ("fixed_pairs_0", {"pair_passes": 0}, 0, 1 << 17, 3, dict(fixed=1, P=0)),
    ("fixed_pairs_4", {"pair_passes": 4}, 0, 1 << 17, 3, dict(fixed=1, P=4)),
    ("fixed_reduce_quad_0", {"reduce_quad": 0}, 0, 1 << 17, 2, dict(fixed=1, reduce_quad=0)),
    ("variable_c8", {}, 8, 4096, 5, dict(fixed=0, c=8)),
    ("variable_batch_window", {}, 0, 4000, 8, dict(fixed=0, c=8)),  # >= 8 segments of <= 2^12 points: window 8 (K2c policy)
    ("variable_batch_window_7", {}, 0, 4000, 4, dict(fixed=0, c=11)),  # 7 segments: the single-MSM window
    ("variable_c13_pairs_4", {"pair_passes": 4}, 13, 4096, 5, dict(fixed=0, c=13, P=4)),
    ("variable_reduce_quad_0", {"reduce_quad": 0}, 0, 4096, 3, dict(fixed=0, c=11, reduce_quad=0)),
    ("variable_reduce_quad_1", {"reduce_quad": 1}, 0, 4096, 3, dict(fixed=0, c=11, reduce_quad=1)),
    ("variable_acc_quad_0", {"acc_quad": 0}, 8, 100, 2, dict(fixed=0, c=8, acc=0, P=0)),
    ("variable_small_quad", {}, 8, 100, 2, dict(fixed=0, c=8, acc=2, P=0)),
    ("fixed_off", {}, 0, 1 << 17, 2, dict(fixed=0, c=13)),
]


@gpu
@pytest.mark.parametrize("name,knobs,window,n,k,want", VARIANTS, ids=[v[0] for v in VARIANTS])
def test_variants(env, name, knobs, window, n, k, want):
    ctx, O = env["ctx"], env["O"]
    ps = [O.random_scalars(n + (j % 3), 300 + j) for j in range(k)]
    ps += _edge_polys(O, n, 400)[1:4]
    ws = O.random_scalars(len(ps), 11)
    d = (1 << 18) - 1 if n > 4096 else 8191
    try:
        for key, v in knobs.items():
            ctx.set_tuning(key, v)
        ctx.set_msm_window(window)
        if name == "fixed_off":
            ctx.set_fixed_base(False)
        got, route = _check(env, ps, d, ws, singles=False)
        bad = {key: (route[key], v) for key, v in want.items() if route[key] != v}
        assert not bad, f"route {bad} (got, wanted); full record {route}"
        for j in (0, len(ps) - 1):
            assert O.pt_eq(got[j], env["pcdl"].commit(ctx, ps[j], d, ws[j]))
    finally:
        _restore(ctx)


@gpu
def test_two_level_sort(env):
    """The segment term of the two-level counting sort (k_sort_coarse_count / _scatter): the same FIXED-base batch with the sort
    forced on (from 2^20 entries) and off; the two-level sort runs five launches more."""
    ctx, O = env["ctx"], env["O"]
    ps = [O.random_scalars((1 << 17) + j, 450 + j) for j in range(3)] + _edge_polys(O, 1 << 17, 460)[1:4]
    launches = {}
    try:
        for lg in (20, 30):
            ctx.set_tuning("sort2_min_lg", lg)
            l0 = ctx.kernel_launches()
            got = ctx.msm_gens_many(ps)
            launches[lg] = ctx.kernel_launches() - l0
            _route_fixed = ctx.test_msm_route(0)
            assert _route_fixed["fixed"] == 1, _route_fixed
            for j, p in enumerate(ps):
                assert O.pt_eq(got[j], _expected(env, p, None)), (lg, j)
    finally:
        _restore(ctx)
    assert launches[20] == launches[30] + 5, launches


# ---- groups, launches, routes ------------------------------------------------------------------------------------------------
@gpu
def test_groups_keep_order(env):
    """600 outputs of one scalar each: the 256-segment limit cuts them into 3 groups; windows of different plans between them
    add more groups.  Every output stays in place."""
    ctx, O = env["ctx"], env["O"]
    vecs = [O.random_scalars(1, 500 + j) for j in range(600)]
    l0 = ctx.kernel_launches()
    got = ctx.msm_gens_many(vecs)
    many = ctx.kernel_launches() - l0
    l0 = ctx.kernel_launches()
    ctx.msm_gens_many(vecs[:2])
    one_group = ctx.kernel_launches() - l0
    assert many >= 3 * one_group, (many, one_group)
    g0 = ctx.get_generators(0, 1)
    for j in (0, 1, 255, 256, 257, 511, 512, 599):
        assert O.pt_eq(got[j], O.msm_affine(g0, vecs[j])), j
    mixed = [O.random_scalars(n, 600 + j) for j, n in enumerate([4096, 4000, 1, 2, 0, 4096, 3000, 1 << 17, 5])]
    got = ctx.msm_gens_many(mixed)
    for j, v in enumerate(mixed):
        assert O.pt_eq(got[j], _expected(env, v, None)), j


@gpu
def test_one_msm_not_a_loop(env):
    """Inside one group the launch count does not grow with k (k = 2 against k = 32 at 2^12, same route)."""
    ctx, O = env["ctx"], env["O"]
    counts, routes = {}, {}
    try:
        ctx.set_tuning("reduce_quad", 0)  # the policy would pick the quad reduction for the smaller bucket count only
        ctx.set_msm_window(11)  # and the narrow window of a batch of short segments for k >= 8 only
        for k in (2, 32):
            vecs = [O.random_scalars(4096, 700 + j) for j in range(k)]
            ctx.msm_gens_many(vecs)  # warm (buffer growth)
            l0 = ctx.kernel_launches()
            got = ctx.msm_gens_many(vecs)
            counts[k] = ctx.kernel_launches() - l0
            r = ctx.test_msm_route(0)
            r.pop("acc_grid")  # persistent grid sized by the bucket count
            routes[k] = r
            for j in (0, k - 1):
                assert O.pt_eq(got[j], _expected(env, vecs[j], None))
    finally:
        _restore(ctx)
    assert routes[2] == routes[32], routes
    assert counts[32] <= counts[2], counts


@gpu
@pytest.mark.parametrize("n", [4096, 1 << 17])
def test_k1_is_the_single_route(env, n):
    ctx, O = env["ctx"], env["O"]
    p = O.random_scalars(n, 800)
    a = ctx.msm_gens_many([p])[0]
    ra = ctx.test_msm_route(0)
    b = ctx.msm_gens(p)
    rb = ctx.test_msm_route(0)
    assert ra == rb and ra["c"] != 0, (ra, rb)
    assert O.pt_eq(a, b)


# ---- errors ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_errors(env):
    from halo_accumulation_b200 import _host
    from halo_accumulation_b200._capi import HaloError, p64, pack

    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    lib = _host.lib()
    good = O.random_scalars(64, 900)
    high = np.concatenate([O.random_scalars(64, 901), O.random_scalars(1, 902)])  # degree 64 > d = 63

    def raw(ps, d, ws=None):
        packed, lens = pack(ps)
        out = np.full((len(ps), 12), 0x5A5A, dtype=np.uint64)
        wa = np.ascontiguousarray(ws, dtype=np.uint64) if ws is not None else None
        rc = lib.halo_pcdl_commit_batch(ctx._h, p64(packed), p64(lens), C.c_uint64(len(ps)), C.c_uint64(d),
                                        p64(wa) if wa is not None else None, p64(out))
        return rc, out

    for ps, d in (([good, high, good], 63), ([good, good, good], 62), ([good, good, good], 2 * N_GENS - 1)):
        rc, out = raw(ps, d, O.random_scalars(3, 3))
        assert rc == HALO_EINVAL, (rc, d)
        assert (out == 0x5A5A).all(), "an output was written"
        with pytest.raises(HaloError):
            pcdl.commit_batch(ctx, ps, d)
    assert pcdl.commit_batch(ctx, [], 63).shape == (0, 12)
    assert raw([], 63)[0] == 0
    assert ctx.msm_gens_many([]).shape == (0, 12)
    # the C ABI: NULL pointers with k > 0, a length beyond the resident generators
    L = ctx._lib
    lens = np.array([4, 4], dtype=np.uint64)
    out = np.zeros((2, 12), dtype=np.uint64)
    sc = O.random_scalars(8, 903)
    assert L.halo_msm_gens_many(ctx._h, None, p64(lens), C.c_uint64(2), p64(out)) == HALO_EINVAL
    assert L.halo_msm_gens_many(ctx._h, p64(sc), None, C.c_uint64(2), p64(out)) == HALO_EINVAL
    assert L.halo_msm_gens_many(ctx._h, p64(sc), p64(lens), C.c_uint64(2), None) == HALO_EINVAL
    huge = np.array([4, N_GENS + 1], dtype=np.uint64)
    assert L.halo_msm_gens_many(ctx._h, p64(sc), p64(huge), C.c_uint64(2), p64(out)) == HALO_ESTATE
    over = np.array([1 << 62, 1 << 62], dtype=np.uint64)
    assert lib.halo_pcdl_commit_batch(ctx._h, p64(sc), p64(over), C.c_uint64(2), C.c_uint64(63), None, p64(out)) == HALO_EINVAL
    assert L.halo_msm_gens_many(ctx._h, None, None, C.c_uint64(0), None) == 0
