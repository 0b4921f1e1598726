"""Batch opening at one point (pcdl.open_batch / pcdl.batch_claim; DESIGN.md K3b): k polynomials, one PCDL proof.

The reference restatement of the definition lives here, built from the oracle's own primitives (its SHA3-256, compressed point
serialisation, field arithmetic, scalar_dot and pcdl_open), not through the library: v_j = p_j(z), alpha = rho_0(z, C_0, v_0,
.., C_{k-1}, v_{k-1}), C = sum_j alpha^j C_j, v = sum_j alpha^j v_j, p = sum_j alpha^j p_j, w = sum_j alpha^j w_j and the
single opening of p.  A second, independent restatement of alpha and (C, v) uses oracle/pyref.py (big integers, hashlib).
Montgomery limbs are linear, so sum_j alpha^j p_j of the limbs as integers (alpha canonical) is the Montgomery form of p."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyref
from oracle.oracle import FR, R_MOD

gpu = pytest.mark.gpu

HALO_EINVAL, HALO_ELEN, HALO_ENOMEM, HALO_ESTATE = -1, -2, -5, -6


# ---- the restatement -------------------------------------------------------------------------------------------------------
def _ints(a):
    b = np.ascontiguousarray(a, dtype=np.uint64).tobytes()
    return [int.from_bytes(b[i:i + 32], "little") for i in range(0, len(b), 32)]


def _limbs(vals):
    return np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in vals), dtype=np.uint64).reshape(-1, 4).copy()


def _fr_bytes(O, s):
    r = np.zeros(4, dtype=np.uint64)
    O.lib().orc_fp_to_canon(FR, O._p(np.ascontiguousarray(s, dtype=np.uint64)), O._p(r))
    return r.tobytes()


def _fr_add(O, a, b):
    r = np.zeros(4, dtype=np.uint64)
    O.lib().orc_fp_add(FR, O._p(np.ascontiguousarray(a, dtype=np.uint64)), O._p(np.ascontiguousarray(b, dtype=np.uint64)), O._p(r))
    return r


def orc_alpha(O, Cs, z, vs):
    """rho_0(z, C_0, v_0, ..): the oracle's SHA3-256 over its serialisations, reduced by its from_le_bytes_mod_order"""
    data = _fr_bytes(O, z) + b"".join(O.pt_serialize_compressed(c) + _fr_bytes(O, v) for c, v in zip(Cs, vs))
    dg = O.sha3_256(data + (0).to_bytes(4, "little"))
    a = np.zeros(4, dtype=np.uint64)
    O.lib().orc_fp_from_le_bytes_mod_order(FR, (C.c_uint8 * 32).from_buffer_copy(dg), O._p(a))
    return a


def orc_batch_claim(O, Cs, z, vs):
    """-> (alpha, C, v, [alpha^j]) in the oracle's arithmetic"""
    alpha = orc_alpha(O, Cs, z, vs)
    pw = [O.to_mont([1])[0]]
    for _ in range(1, len(Cs)):
        pw.append(O.fp_mul(pw[-1], alpha, FR))
    Cm, v = O.pt_from_affine_ints(None), np.zeros(4, dtype=np.uint64)
    for j in range(len(Cs)):
        Cm = O.pt_add(Cm, O.pt_mul(Cs[j], pw[j]))
        v = _fr_add(O, v, O.fp_mul(pw[j], vs[j], FR))
    return alpha, Cm, v, pw


def combine(ps, alpha_mont):
    """sum_j alpha^j p_j as Montgomery limbs, by Horner over j on the limbs as integers"""
    a = _canon_int(alpha_mont)
    n = max([len(p) for p in ps] + [1])
    out = [0] * n
    for p in reversed(ps):
        pi = _ints(p)
        out = [(x * a + (pi[i] if i < len(pi) else 0)) % R_MOD for i, x in enumerate(out)]
    return _limbs(out)


def _canon_int(a):
    return _ints(a)[0] * pow(1 << 256, -1, R_MOD) % R_MOD


def degree(p):
    nz = np.flatnonzero(np.asarray(p).reshape(-1, 4).any(axis=1))
    return int(nz[-1]) if len(nz) else 0


def orc_open_batch(O, ps, Cs, d, z, ws=None, q=None, w_bar=None):
    """the definition of K3b, restated -> (vs, C, v, pi, p, w)"""
    ps = [np.asarray(p).reshape(-1, 4)[:d + 1] for p in ps]
    vs = [O.scalar_dot(p, O.construct_powers(z, len(p))) for p in ps]
    alpha, Cm, v, pw = orc_batch_claim(O, Cs, z, vs)
    p = combine(ps, alpha)
    w = None
    if ws is not None:
        w = np.zeros(4, dtype=np.uint64)
        for j in range(len(ps)):
            w = _fr_add(O, w, O.fp_mul(pw[j], ws[j], FR))
    deg = degree(p)
    pi = O.pcdl_open(p, Cm, d, z, w, None if q is None else np.asarray(q)[:deg], w_bar, threads=8)
    return np.array(vs), Cm, v, pi, p, w


def pyref_claim(O, Cs, z, vs):
    """alpha and (C, v) by oracle/pyref.py: affine big-integer points, hashlib"""
    zi = O.from_mont(z)[0]
    vi = O.from_mont(np.asarray(vs).reshape(-1, 4))
    pts = [O.pt_to_affine_ints(c) for c in Cs]
    args = [zi]
    for pt, v in zip(pts, vi):
        args += [pt, v]
    alpha = pyref.rho(0, *args)
    pw = [pow(alpha, j, pyref.R) for j in range(len(Cs))]
    return alpha, pyref.msm(pts, pw), sum(a * v for a, v in zip(pw, vi)) % pyref.R


# ---- CPU: the restatement against itself and pyref -----------------------------------------------------------------------
D_CPU = (1 << 8) - 1


@pytest.fixture(scope="module")
def cpu_env(oracle):
    O = oracle
    saved = O.params() if O.lib().orc_params_n() else None
    O.derive_params(D_CPU + 1)
    yield O
    if saved is not None:  # the oracle's parameters are process-wide
        O.set_params(*saved)


def _cpu_polys(O, seed):
    return [O.random_scalars(D_CPU + 1, seed), O.random_scalars(100, seed + 1), np.zeros((0, 4), dtype=np.uint64),
            np.zeros((7, 4), dtype=np.uint64), np.tile(O.to_mont([R_MOD - 1])[0], (D_CPU + 1, 1))]


@pytest.mark.parametrize("hiding", [False, True])
def test_oracle_open_batch_is_open_of_combined(cpu_env, hiding):
    """the restated batch opening is the oracle's open of the host-combined polynomial against C = commit(p) + w S, and the
    oracle's check accepts the combined claim; each v_j is p_j(z)"""
    O = cpu_env
    ps = _cpu_polys(O, 40)
    ws = O.random_scalars(len(ps), 41) if hiding else None
    Cs = [O.pcdl_commit(p, D_CPU, None if ws is None else ws[j]) for j, p in enumerate(ps)]
    z, wb = O.random_scalars(2, 42)
    q = O.random_scalars(max(degree(p) for p in ps), 43) if hiding else None
    vs, Cm, v, pi, p, w = orc_open_batch(O, ps, Cs, D_CPU, z, ws, q, wb if hiding else None)
    assert O.pt_eq(Cm, O.pcdl_commit(p, D_CPU, w))
    assert list(v) == list(O.scalar_dot(p, O.construct_powers(z, len(p))))
    assert O.pcdl_check(Cm, D_CPU, z, v, pi) == 0
    for j, pj in enumerate(ps):
        assert O.from_mont(vs[j])[0] == sum(a * pow(O.from_mont(z)[0], i, R_MOD) for i, a in enumerate(O.from_mont(pj))) % R_MOD


def test_oracle_claim_matches_pyref(oracle):
    """alpha and (C, v) of the oracle restatement equal pyref's, with C_j = O and duplicate commitments among the inputs"""
    O = oracle
    base = O.affine_to_jac(O.derive_points(2, 3))
    Cs = [O.pt_mul(base[0], O.random_scalars(1, 50)[0]), O.pt_from_affine_ints(None), base[1], base[1], base[2]]
    z = O.random_scalars(1, 51)[0]
    vs = O.random_scalars(len(Cs), 52)
    vs[2] = O.to_mont([R_MOD - 1])[0]
    alpha, Cm, v, _ = orc_batch_claim(O, Cs, z, vs)
    a_py, C_py, v_py = pyref_claim(O, Cs, z, vs)
    assert O.from_mont(alpha)[0] == a_py
    assert O.pt_to_affine_ints(Cm) == C_py
    assert O.from_mont(v)[0] == v_py
    one = orc_batch_claim(O, Cs[:1], z, vs[:1])  # k = 1: alpha^0 = 1
    assert O.pt_eq(one[1], Cs[0]) and list(one[2]) == list(vs[0])


# ---- GPU -------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env(ctx, oracle, halo):
    from halo_accumulation_b200 import acc, pcdl

    O = oracle
    S, H = ctx.get_SH()
    O.set_params(S, H, ctx.get_generators(0, 1 << 16))
    yield dict(ctx=ctx, O=O, pcdl=pcdl, acc=acc, halo=halo)
    bad, live = halo.check_canaries()  # no kernel of this module wrote past a device buffer
    assert bad == 0, (bad, live)


def _same_proof(O, a, b):
    assert a.lg_n == b.lg_n and a.hiding == b.hiding
    for i in range(a.lg_n):
        assert O.pt_eq(np.array(a.Ls[i]), np.array(b.Ls[i])) and O.pt_eq(np.array(a.Rs[i]), np.array(b.Rs[i])), i
    assert O.pt_eq(np.array(a.U), np.array(b.U)) and list(a.c) == list(b.c)
    if a.hiding:
        assert O.pt_eq(np.array(a.C_bar), np.array(b.C_bar)) and list(a.w_prime) == list(b.w_prime)


def _ragged(O, k, n, seed):
    """k polynomials of at most n coefficients: full, shorter, a zero polynomial, an empty list, all r - 1"""
    kinds = [O.random_scalars(n, seed), O.random_scalars(n - 37, seed + 1), np.zeros((n // 2, 4), dtype=np.uint64),
             np.zeros((0, 4), dtype=np.uint64), np.tile(O.to_mont([R_MOD - 1])[0], (n - 1, 1)), O.random_scalars(3, seed + 2),
             O.random_scalars(n, seed + 3), O.random_scalars(n // 4, seed + 4)]
    return kinds[:2] + kinds[2:k] if k > 2 else [kinds[0], kinds[2]]


def _draws(O, ps, hiding, seed):
    if not hiding:
        return None, None, None
    return O.random_scalars(len(ps), seed), O.random_scalars(max(degree(p) for p in ps), seed + 1), O.random_scalars(1, seed + 2)[0]


@gpu
@pytest.mark.parametrize("hiding", [False, True])
@pytest.mark.parametrize("lg", [10, 12])
@pytest.mark.parametrize("k", [2, 3, 8])
def test_against_oracle(env, k, lg, hiding):
    """vs, C, v and every proof field equal the restatement's; the claim is accepted by pcdl.check and the oracle's check, and
    batch_claim gives the same (C, v)"""
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    n = 1 << lg
    d = n - 1
    ps = _ragged(O, k, n, 100 * k + lg)
    ws, q, wb = _draws(O, ps, hiding, 7 + k)
    Cs = pcdl.commit_batch(ctx, ps, d, ws)
    if not hiding:
        assert O.pt_eq(Cs[2 if k > 2 else 1], O.pt_from_affine_ints(None))  # the zero polynomial commits to O
    z = O.random_scalars(1, 300 + k)[0]
    vs, Cm, v, pi = pcdl.open_batch(ctx, ps, Cs, d, z, ws, q, wb)
    evs, eC, ev, epi, _, _ = orc_open_batch(O, ps, Cs, d, z, ws, q, wb)
    assert np.array_equal(vs, evs)
    assert O.pt_eq(Cm, eC) and list(v) == list(ev)
    _same_proof(O, pi, epi)
    pcdl.check(ctx, Cm, d, z, v, pi)
    assert O.pcdl_check(Cm, d, z, v, O.EvalProof.from_buffer_copy(bytes(pi))) == 0
    bC, bv = pcdl.batch_claim(ctx, Cs, z, vs)
    assert O.pt_eq(bC, Cm) and list(bv) == list(v)


@gpu
@pytest.mark.parametrize("hiding", [False, True])
def test_k1_is_open(env, hiding):
    """one polynomial: the proof of pcdl.open (same points, same scalars), C = C_0, v = p(z)"""
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    d = (1 << 12) - 1
    p = O.random_scalars(4000, 400)
    ws, q, wb = _draws(O, [p], hiding, 401)
    Cs = pcdl.commit_batch(ctx, [p], d, ws)
    z = O.random_scalars(1, 402)[0]
    vs, Cm, v, pi = pcdl.open_batch(ctx, [p], Cs, d, z, ws, q, wb)
    ref = pcdl.open(ctx, p, Cs[0], d, z, None if ws is None else ws[0], q, wb)
    _same_proof(O, pi, ref)
    assert O.pt_eq(Cm, Cs[0]) and np.array_equal(v, vs[0])
    assert list(v) == list(O.scalar_dot(p, O.construct_powers(z, len(p))))


@gpu
def test_2_20_hiding(env):
    """k = 4 at 2^20, hiding: the proof equals pcdl.open of the restatement's combined polynomial"""
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    n = 1 << 20
    d = n - 1
    ctx.derive_generators(n)
    ctx.precompute_generators(0)
    try:
        ps = [O.random_scalars(n, 500), O.random_scalars(n - 5, 501), O.random_scalars(1 << 19, 502), O.random_scalars(n, 503)]
        ws, q, wb = _draws(O, ps, True, 504)
        Cs = pcdl.commit_batch(ctx, ps, d, ws)
        z = O.random_scalars(1, 505)[0]
        vs, Cm, v, pi = pcdl.open_batch(ctx, ps, Cs, d, z, ws, q, wb)
        evs = np.array([O.scalar_dot(p, O.construct_powers(z, len(p))) for p in ps])
        assert np.array_equal(vs, evs)
        alpha, eC, ev, pw = orc_batch_claim(O, Cs, z, evs)
        assert O.pt_eq(Cm, eC) and list(v) == list(ev)
        p = combine(ps, alpha)
        w = np.zeros(4, dtype=np.uint64)
        for j in range(4):
            w = _fr_add(O, w, O.fp_mul(pw[j], ws[j], FR))
        ref = pcdl.open(ctx, p, eC, d, z, w, q[:degree(p)], wb)
        _same_proof(O, pi, ref)
        pcdl.check(ctx, Cm, d, z, v, pi)
    finally:
        ctx.derive_generators(1 << 16)


@gpu
def test_accumulation(env):
    """the combined claim as acc.new_instance: prover, verifier and decider on the GPU and in the oracle"""
    ctx, O, pcdl, acc = env["ctx"], env["O"], env["pcdl"], env["acc"]
    d = (1 << 10) - 1
    ps = _ragged(O, 3, d + 1, 600)
    ws, q, wb = _draws(O, ps, True, 601)
    Cs = pcdl.commit_batch(ctx, ps, d, ws)
    z = O.random_scalars(1, 602)[0]
    _, Cm, v, pi = pcdl.open_batch(ctx, ps, Cs, d, z, ws, q, wb)
    inst = acc.new_instance(Cm, d, z, v, pi)
    pcdl.check_batch(ctx, [inst, inst], O.random_scalars(1, 603)[0])
    a = acc.prover(ctx, d, [inst], O.random_scalars(2, 604), O.random_scalars(1, 605)[0], O.random_scalars(d, 606),
                   O.random_scalars(1, 607)[0])
    acc.verifier(ctx, d, [inst], a)
    acc.decider(ctx, a)
    oq = O.Instance.from_buffer_copy(bytes(inst))
    oa = O.Accumulator.from_buffer_copy(bytes(a))
    assert O.acc_verifier(d, [oq], oa) == 0
    assert O.acc_decider(oa) == 0


@gpu
@pytest.mark.parametrize("hiding", [False, True])
def test_soundness(env, hiding):
    """one v_j changed, two commitments swapped or another z: batch_claim + check rejects with the oracle's code"""
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    d = (1 << 10) - 1
    ps = _ragged(O, 3, d + 1, 700)
    ws, q, wb = _draws(O, ps, hiding, 701)
    Cs = pcdl.commit_batch(ctx, ps, d, ws)
    z = O.random_scalars(1, 702)[0]
    vs, Cm, v, pi = pcdl.open_batch(ctx, ps, Cs, d, z, ws, q, wb)
    opi = O.EvalProof.from_buffer_copy(bytes(pi))
    bad_v = vs.copy()
    bad_v[1] = _fr_add(O, bad_v[1], O.to_mont([1])[0])
    swapped = Cs[[1, 0, 2]]
    z2 = O.random_scalars(1, 703)[0]
    for Cs_x, vs_x, z_x in ((Cs, bad_v, z), (swapped, vs, z), (Cs, vs, z2)):
        bC, bv = pcdl.batch_claim(ctx, Cs_x, z_x, vs_x)
        _, eC, ev, _ = orc_batch_claim(O, Cs_x, z_x, vs_x)
        assert O.pt_eq(bC, eC) and list(bv) == list(ev)
        code = O.pcdl_check(eC, d, z_x, ev, opi)
        assert code != 0
        with pytest.raises(pcdl.Rejected) as e:
            pcdl.check(ctx, bC, d, z_x, bv, pi)
        assert e.value.code == code


def _raw_open_batch(env, ps, Cs, d, z, ws=None, q=None, wb=None, k=None):
    """halo_pcdl_open_batch with sentinel outputs -> (rc, outputs untouched)"""
    from halo_accumulation_b200 import _capi, _host

    packed, lens = _capi.pack(ps)
    k = len(lens) if k is None else k
    Cs, z = np.ascontiguousarray(Cs, dtype=np.uint64).reshape(-1, 12), np.ascontiguousarray(z, dtype=np.uint64)
    vs = np.full((max(1, len(lens)), 4), 0xAB, dtype=np.uint64)
    Cm, v = np.full(12, 0xAB, dtype=np.uint64), np.full(4, 0xAB, dtype=np.uint64)
    pi = _host.EvalProof()
    C.memset(C.byref(pi), 0xAB, C.sizeof(pi))
    wa = None if ws is None else np.ascontiguousarray(ws, dtype=np.uint64)
    qa = None if q is None else np.ascontiguousarray(q, dtype=np.uint64).reshape(-1, 4)
    wba = None if wb is None else np.ascontiguousarray(wb, dtype=np.uint64)
    p = _capi.p64
    rc = _host.lib().halo_pcdl_open_batch(env["ctx"]._h, p(packed), p(lens), C.c_uint64(k), p(Cs), C.c_uint64(d), p(z),
                                          None if wa is None else p(wa), None if qa is None else p(qa),
                                          C.c_uint64(0 if qa is None else qa.shape[0]), None if wba is None else p(wba),
                                          p(vs), p(Cm), p(v), C.byref(pi))
    untouched = ((vs == 0xAB).all() and (Cm == 0xAB).all() and (v == 0xAB).all()
                 and bytes(pi) == bytes([0xAB]) * C.sizeof(pi))
    return rc, untouched


@gpu
def test_errors(env, halo):
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    from halo_accumulation_b200 import _capi, _host

    d = (1 << 10) - 1
    ps = [O.random_scalars(d + 1, 800 + j) for j in range(4)]
    ws, q, wb = _draws(O, ps, True, 810)
    Cs = pcdl.commit_batch(ctx, ps, d, ws)
    z = O.random_scalars(1, 811)[0]
    launches = ctx.kernel_launches()
    # a malformed polynomial at position j (degree > d), then d + 1 not a power of two: nothing runs, nothing is written
    for j in range(4):
        bad = list(ps)
        bad[j] = O.random_scalars(d + 2, 820 + j)
        assert _raw_open_batch(env, bad, Cs, d, z, ws, q, wb) == (HALO_EINVAL, True)
    assert _raw_open_batch(env, ps, Cs, d - 1, z, ws, q, wb) == (HALO_EINVAL, True)
    # C_j off the curve and not canonical; w_j and z not canonical; k = 0
    off_curve = Cs.copy()
    off_curve[2, 0] ^= np.uint64(1)
    non_canon = Cs.copy()
    non_canon[1, :4] = np.uint64(0xFFFFFFFFFFFFFFFF)
    big = np.full(4, 0xFFFFFFFFFFFFFFFF, dtype=np.uint64)
    bad_w = ws.copy()
    bad_w[3] = big
    for args in ((ps, off_curve, d, z, ws, q, wb), (ps, non_canon, d, z, ws, q, wb), (ps, Cs, d, z, bad_w, q, wb),
                 (ps, Cs, d, big, ws, q, wb)):
        assert _raw_open_batch(env, *args) == (HALO_EINVAL, True)
    assert _raw_open_batch(env, ps, Cs, d, z, ws, q, wb, k=0) == (HALO_EINVAL, True)
    assert ctx.kernel_launches() == launches
    # n_q != max_j deg(p_j)
    for nq in (len(q) - 1, len(q) + 1):
        assert _raw_open_batch(env, ps, Cs, d, z, ws, O.random_scalars(nq, 830), wb)[0] == HALO_ELEN
    # batch_claim: a non-canonical v_j, an off-curve C_j, k = 0
    vs = O.random_scalars(4, 840)
    bad_v = vs.copy()
    bad_v[0] = big
    for Cs_x, vs_x in ((Cs, bad_v), (off_curve, vs), (Cs[:0], vs[:0])):
        with pytest.raises(_capi.HaloError) as e:
            pcdl.batch_claim(ctx, Cs_x, z, vs_x)
        assert e.value.code == HALO_EINVAL
    # the device layer: combine without a preceding evaluation, k = 0, and an upload the device cannot hold
    lib = _capi.load()
    fresh = halo.Context(0, 1 << 16)
    try:
        fresh.derive_generators(1 << 16)
        deg = C.c_uint64(0)
        alpha = O.random_scalars(1, 850)[0]
        assert lib.halo_poly_combine_resident(fresh._h, _capi.p64(alpha), C.byref(deg)) == HALO_ESTATE
        vs_out = np.zeros((1, 4), dtype=np.uint64)
        one = np.ones(1, dtype=np.uint64)
        assert lib.halo_poly_eval_many(fresh._h, _capi.p64(O.random_scalars(1, 851)), _capi.p64(one), C.c_uint64(0),
                                       C.c_uint64(1024), _capi.p64(z), _capi.p64(vs_out)) == HALO_EINVAL
        k = 1 << 20  # 2^20 polynomials of 2^16 coefficients: 2 TiB, refused before the (one-element) host buffer is read
        lens = np.full(k, 1 << 16, dtype=np.uint64)
        vs_big = np.zeros((k, 4), dtype=np.uint64)
        assert lib.halo_poly_eval_many(fresh._h, _capi.p64(O.random_scalars(1, 852)), _capi.p64(lens), C.c_uint64(k),
                                       C.c_uint64(1 << 16), _capi.p64(z), _capi.p64(vs_big)) == HALO_ENOMEM
        assert not vs_big.any()
        assert lib.halo_poly_combine_resident(fresh._h, _capi.p64(alpha), C.byref(deg)) == HALO_ESTATE
        # the context is still usable after the refused allocation
        p = O.random_scalars(1000, 853)
        vs_out2 = np.zeros((2, 4), dtype=np.uint64)
        lens2 = np.array([1000, 0], dtype=np.uint64)
        assert lib.halo_poly_eval_many(fresh._h, _capi.p64(p), _capi.p64(lens2), C.c_uint64(2), C.c_uint64(1024),
                                       _capi.p64(z), _capi.p64(vs_out2)) == 0
        assert list(vs_out2[0]) == list(O.scalar_dot(p, O.construct_powers(z, 1000))) and not vs_out2[1].any()
    finally:
        fresh.close()
    # and the shared context still opens
    vs, Cm, v, pi = pcdl.open_batch(ctx, ps, Cs, d, z, ws, q, wb)
    pcdl.check(ctx, Cm, d, z, v, pi)
