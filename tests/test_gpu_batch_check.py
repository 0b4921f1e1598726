"""GPU tests of the batch decider (DESIGN.md K5b): halo_h_msm_batch against the oracle's MSMs, and pcdl.check_batch /
acc.decider_batch against a loop of the oracle's single checks -- accept on honest claims for every rho, and on a reject the
same (claim index, code) as the first claim the oracle rejects in order; malformed input is an error, not a decision."""
import ctypes as C

import numpy as np
import pytest

from oracle.oracle import R_MOD

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env(ctx, oracle):
    """Context with 2^16 generators and the oracle holding the very same parameters."""
    from halo_accumulation_b200 import acc, pcdl

    ctx.derive_generators(1 << 16)
    S, H = ctx.get_SH()
    oracle.set_params(S, H, ctx.get_generators(0, 1 << 16))
    return dict(ctx=ctx, O=oracle, pcdl=pcdl, acc=acc)


def _h_msm_batch(ctx, xis_list, weights, bases=None, scalars=None, inf=None):
    """(return code, point) of halo_h_msm_batch; bases / scalars None: no companion."""
    lgs = np.array([x.shape[0] - 1 for x in xis_list] or [0], dtype=np.uint32)
    xis = np.ascontiguousarray(np.concatenate(xis_list) if xis_list else np.zeros((1, 4), dtype=np.uint64))
    w = np.ascontiguousarray(weights if len(xis_list) else np.zeros((1, 4)), dtype=np.uint64)
    m = 0 if scalars is None else scalars.shape[0]
    b = np.zeros((1, 8), dtype=np.uint64) if bases is None else np.ascontiguousarray(bases)
    s = np.zeros((1, 4), dtype=np.uint64) if scalars is None else np.ascontiguousarray(scalars)
    infp = None if inf is None else np.ascontiguousarray(inf, dtype=np.uint8).ctypes.data_as(C.POINTER(C.c_uint8))
    out = np.zeros(12, dtype=np.uint64)
    u64 = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint64))  # noqa: E731
    rc = ctx._lib.halo_h_msm_batch(ctx._h, u64(xis), lgs.ctypes.data_as(C.POINTER(C.c_uint32)), u64(w), len(xis_list),
                                   u64(b), infp, u64(s), m, u64(out))
    return rc, out


def test_h_msm_batch_matches_oracle(env):
    """Mixed lg n_j from 1 to 16 (claims of fewer than 8 coefficients and of more than one block), k crossing the kernel's
    claim chunks, weights 0 and 1 among them, with and without a companion: the sum of the oracle's per-claim MSMs."""
    ctx, O = env["ctx"], env["O"]
    gs = ctx.get_generators(0, 1 << 16)
    lgs = [1 + (7 * j) % 16 for j in range(70)]
    xis = [O.random_scalars(lg + 1, 3000 + j) for j, lg in enumerate(lgs)]
    w = O.random_scalars(70, 2999)
    w[0] = O.to_mont([1])[0]
    w[5] = 0
    w[40] = 0
    per_claim = [O.pt_mul(O.msm_affine(gs, O.h_get_poly(x), threads=8), w[j]) for j, x in enumerate(xis)]
    bases = ctx.get_generators(77, 300).copy()
    sc = O.random_scalars(300, 2998)
    inf = np.zeros(300, dtype=np.uint8)
    inf[[0, 17, 299]] = 1
    companion = O.msm_affine(bases, sc, threads=8, inf=inf)
    for k in (1, 2, 33, 70):
        ref = O.pt_from_affine_ints(None)
        for p in per_claim[:k]:
            ref = O.pt_add(ref, p)
        rc, got = _h_msm_batch(ctx, xis[:k], w[:k])
        assert rc == 0 and O.pt_eq(got, ref), k
        rc, got = _h_msm_batch(ctx, xis[:k], w[:k], bases, sc, inf)
        assert rc == 0 and O.pt_eq(got, O.pt_add(ref, companion)), k
    rc, got = _h_msm_batch(ctx, [], [], bases, sc, inf)  # companion alone
    assert rc == 0 and O.pt_eq(got, companion)


def test_h_msm_batch_argument_errors(env):
    ctx, O = env["ctx"], env["O"]
    rc, got = _h_msm_batch(ctx, [], [])
    assert rc == 0 and O.pt_to_affine(got)[1]  # k = m = 0: infinity
    xis = [O.random_scalars(11, 1), O.random_scalars(18, 2)]  # lg 17: above the 2^16 resident generators
    rc, _ = _h_msm_batch(ctx, xis, O.random_scalars(2, 3))
    assert rc < 0
    lib, u64 = ctx._lib, C.POINTER(C.c_uint64)
    out = np.zeros(12, dtype=np.uint64)
    lg = np.array([4], dtype=np.uint32)
    x, w = O.random_scalars(5, 4), O.random_scalars(1, 5)
    lgp = lg.ctypes.data_as(C.POINTER(C.c_uint32))
    assert lib.halo_h_msm_batch(ctx._h, None, lgp, x.ctypes.data_as(u64), 1, None, None, None, 0, out.ctypes.data_as(u64)) == -1
    assert lib.halo_h_msm_batch(ctx._h, x.ctypes.data_as(u64), None, w.ctypes.data_as(u64), 1, None, None, None, 0,
                                out.ctypes.data_as(u64)) == -1
    assert lib.halo_h_msm_batch(ctx._h, x.ctypes.data_as(u64), lgp, w.ctypes.data_as(u64), 1, None, None, w.ctypes.data_as(u64), 1,
                                out.ctypes.data_as(u64)) == -1  # m > 0 without bases
    assert lib.halo_h_msm_batch(ctx._h, x.ctypes.data_as(u64), lgp, w.ctypes.data_as(u64), 1, None, None, None, 0, None) == -1
    assert _h_msm_batch(ctx, [x], w)[0] == 0  # the context still works


def test_h_msm_batch_2_20_fixed_and_variable_base(ctx, oracle):
    """At 2^20 with weights 1: the sum of halo_h_msm over the same claims, with the FIXED-base tables and without."""
    O = oracle
    ctx.derive_generators(1 << 20)
    try:
        ctx.precompute_generators(0)
        xis = [O.random_scalars(lg + 1, 5000 + lg) for lg in (20, 18, 20, 13)]
        one = O.to_mont([1] * len(xis))
        ref = O.pt_from_affine_ints(None)
        for x in xis:
            h = np.zeros(12, dtype=np.uint64)
            ctx._chk(ctx._lib.halo_h_msm(ctx._h, x.ctypes.data_as(C.POINTER(C.c_uint64)), x.shape[0] - 1,
                                         h.ctypes.data_as(C.POINTER(C.c_uint64))))
            ref = O.pt_add(ref, h)
        bases, sc = ctx.get_generators(1000, 100).copy(), O.random_scalars(100, 5100)
        ref_c = O.pt_add(ref, O.msm_affine(bases, sc, threads=8))
        for fixed in (True, False):
            ctx.set_fixed_base(fixed)
            rc, got = _h_msm_batch(ctx, xis, one)
            assert rc == 0 and O.pt_eq(got, ref), fixed
            rc, got = _h_msm_batch(ctx, xis, one, bases, sc)
            assert rc == 0 and O.pt_eq(got, ref_c), fixed
    finally:
        ctx.set_fixed_base(True)
        ctx.derive_generators(1 << 16)


def _claim(env, d, seed, hiding):
    """An honest claim (C, d, z, v, pi) opened on the GPU, hiding or not."""
    ctx, O, pcdl, acc = env["ctx"], env["O"], env["pcdl"], env["acc"]
    n = d + 1
    p = O.random_scalars(max(2, n - n // 3), seed)
    z = O.random_scalars(1, seed + 1)[0]
    w, wb = O.random_scalars(2, seed + 2) if hiding else (None, None)
    q = O.random_scalars(p.shape[0] - 1, seed + 3) if hiding else None
    Cm = pcdl.commit(ctx, p, d, w)
    v = O.scalar_dot(p, O.construct_powers(z, p.shape[0]))
    return acc.new_instance(Cm, d, z, v, pcdl.open(ctx, p, Cm, d, z, w, q, wb))


@pytest.fixture(scope="module")
def pool(env):
    ds = [63, 1023, 15, 255, 1, 4095, 511, 3, 1023, 127]
    return [_claim(env, ds[j % len(ds)], 7000 + 10 * j, j % 2 == 1) for j in range(40)]


@pytest.fixture(scope="module")
def foreign_u(env):
    """A claim whose proof was made under a key with a foreign G_5 (test_gpu_pcdl.py::test_pcdl_full_check_rejects_wrong_U):
    meant to reach the U check; which check trips is whatever the oracle says."""
    import halo_accumulation_b200 as H

    ctx, O, pcdl, acc = env["ctx"], env["O"], env["pcdl"], env["acc"]
    n, d = 64, 63
    S, Hh = ctx.get_SH()
    gs = ctx.get_generators(0, n).copy()
    gs[5] = ctx.get_generators(1000, 1)[0]
    other = H.Context(0, 1 << 10)
    try:
        other.load_generators(S, Hh, gs)
        p, z = O.random_scalars(n, 91), O.random_scalars(1, 92)[0]
        p[5] = 0
        Cm = pcdl.commit(other, p, d)
        v = O.scalar_dot(p, O.construct_powers(z, n))
        return acc.new_instance(Cm, d, z, v, pcdl.open(other, p, Cm, d, z))
    finally:
        other.close()


def _rhos(O):
    return [O.random_scalars(1, 123)[0], O.to_mont([1])[0], O.to_mont([R_MOD - 1])[0], O.random_scalars(1, 456)[0]]


def _oracle_first_reject(O, claims):
    for j, q in enumerate(claims):
        rc = O.pcdl_check(np.array(q.C), q.d, np.array(q.z), np.array(q.v), O.EvalProof.from_buffer_copy(bytes(q.pi)), threads=8)
        if rc != 0:
            return j, rc
    return None


def _same_decision(env, claims, rho, expected):
    pcdl = env["pcdl"]
    if expected is None:
        pcdl.check_batch(env["ctx"], claims, rho)
        return
    with pytest.raises(pcdl.Rejected) as e:
        pcdl.check_batch(env["ctx"], claims, rho)
    assert (e.value.index, e.value.code) == expected


def _copy(q):
    return type(q).from_buffer_copy(bytes(q))


@pytest.mark.parametrize("k", [0, 1, 5, 40])
def test_check_batch_accepts_honest_claims(env, pool, k):
    """Hiding and non-hiding claims of different d; every rho (the accept direction holds for all of them)."""
    claims = pool[:k]
    assert _oracle_first_reject(env["O"], claims) is None
    for rho in _rhos(env["O"]):
        env["pcdl"].check_batch(env["ctx"], claims, rho)


def test_check_batch_200_claims_companion_past_4096_points(env, pool):
    """200 claims (copies of the pool's larger claims) bring 2 lg n + 2 points each: a companion MSM of more than 4096 points."""
    big = [q for q in pool if q.pi.lg_n >= 10]
    claims = [big[j % len(big)] for j in range(200)]
    assert sum(2 * q.pi.lg_n + 2 for q in claims) + 1 > 4096
    for rho in _rhos(env["O"])[:2]:
        env["pcdl"].check_batch(env["ctx"], claims, rho)
    bad = _copy(pool[1])
    bad.v[0] ^= 1
    _same_decision(env, claims[:150] + [bad] + claims[150:], _rhos(env["O"])[0], (150, -10))


@pytest.mark.parametrize("kind", ["v", "z", "foreign_u"])
def test_check_batch_reject_equals_first_single_reject(env, pool, foreign_u, kind):
    """One corrupted claim at the first, middle and last position: (index, code) of the first claim the oracle's single
    check rejects, in order."""
    O = env["O"]
    base = pool[:9]
    if kind == "foreign_u":
        bad = foreign_u
    else:
        bad = _copy(pool[0])
        getattr(bad, kind)[0] ^= 1
    for pos in (0, 4, 8):
        claims = list(base)
        claims[pos] = bad
        expected = _oracle_first_reject(O, claims)
        assert expected is not None and expected[0] == pos
        for rho in _rhos(O)[:2]:
            _same_decision(env, claims, rho, expected)


def test_check_batch_earlier_u_reject_wins_over_later_succinct_reject(env, pool, foreign_u):
    O = env["O"]
    later = _copy(pool[3])
    later.pi.c[0] ^= 1
    claims = [pool[0], foreign_u, pool[2], later, pool[4]]
    expected = _oracle_first_reject(O, claims)
    assert expected[0] == 1 and expected[1] in (-10, -11)
    _same_decision(env, claims, _rhos(O)[0], expected)
    claims = [pool[0], later, pool[2], foreign_u]
    assert _oracle_first_reject(O, claims) == (1, -10)
    _same_decision(env, claims, _rhos(O)[0], (1, -10))


def test_check_batch_malformed_input_is_an_error_wherever_it_sits(env, pool):
    from halo_accumulation_b200 import HaloError

    O, pcdl, ctx = env["O"], env["pcdl"], env["ctx"]
    rho = _rhos(O)[0]
    rejecting = _copy(pool[2])
    rejecting.v[0] ^= 1

    def refused(claims, r=rho):
        with pytest.raises(HaloError) as e:
            pcdl.check_batch(ctx, claims, r)
        assert e.value.code == -1, e.value.code

    off_curve = _copy(pool[1])
    off_curve.pi.Ls[2][5] ^= 4
    not_canonical = _copy(pool[3])
    not_canonical.pi.c[3] = 0x7FFFFFFFFFFFFFFF
    not_pow2 = _copy(pool[0])
    not_pow2.d = 62
    too_large = _copy(pool[0])
    too_large.d = (1 << 17) - 1
    for bad in (off_curve, not_canonical, not_pow2, too_large):
        for pos in (0, 3, 6):
            claims = list(pool[:6])
            claims.insert(pos, bad)
            refused(claims)
        refused([rejecting, bad])  # an error even behind a claim that would be rejected
    refused(pool[:3], np.zeros(4, dtype=np.uint64))  # rho = 0
    pcdl.check_batch(ctx, pool[:6], rho)  # the context still works


def _chain(env, d, steps, seed):
    """Accumulators of a short IVC chain (acc.rs:298-315 shape): one per step."""
    ctx, O, acc = env["ctx"], env["O"], env["acc"]
    n, a, out = d + 1, None, []
    for s in range(steps):
        q = _claim(env, d, seed + 100 * s, True)
        qs = [acc.to_instance(a), q] if a is not None else [q]
        h0, (w, wb), qq = O.random_scalars(2, seed + 100 * s + 50), O.random_scalars(2, seed + 100 * s + 60), \
            O.random_scalars(n - 1, seed + 100 * s + 70)
        a = acc.prover(ctx, d, qs, h0, w, qq, wb)
        acc.verifier(ctx, d, qs, a)
        out.append(a)
    return out


def test_decider_batch_over_chains(env):
    O, acc, ctx = env["O"], env["acc"], env["ctx"]
    accs = _chain(env, 1023, 3, 11000) + _chain(env, 255, 2, 12000) + _chain(env, 63, 2, 13000)
    assert all(O.acc_decider(O.Accumulator.from_buffer_copy(bytes(a)), threads=8) == 0 for a in accs)
    for rho in _rhos(O)[:2]:
        acc.decider_batch(ctx, accs, rho)
    for field, pos in (("z", 0), ("v", 3), ("z", 6)):
        bad = list(accs)
        bad[pos] = _copy(accs[pos])
        getattr(bad[pos], field)[0] ^= 1
        codes = [O.acc_decider(O.Accumulator.from_buffer_copy(bytes(a)), threads=8) for a in bad]
        expected = next((j, c) for j, c in enumerate(codes) if c != 0)
        assert expected[0] == pos
        with pytest.raises(acc.Rejected) as e:
            acc.decider_batch(ctx, bad, _rhos(O)[0])
        assert (e.value.index, e.value.code) == expected
    with pytest.raises(acc.Rejected) as e:  # the single decider keeps its behaviour: no index
        acc.decider(ctx, bad[6])
    assert e.value.index is None
