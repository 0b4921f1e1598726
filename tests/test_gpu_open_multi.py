"""Batch opening at several points (pcdl.open_multi / pcdl.multi_claim; DESIGN.md K3c): k polynomials, T points, one proof.

The restatement of the definition (include/halo_pcdl.h halo_pcdl_open_multi) lives here, built from the oracle's primitives
(its SHA3-256, compressed point serialisation, scalar multiplication, pcdl_commit and pcdl_open) and big integers, not through
the library.  Montgomery limbs are linear, so a combination of the limbs as integers with canonical weights (the challenges,
the points) is the Montgomery form of the combination: the polynomials, their quotients and values are computed that way.
The CPU tests check the restatement against oracle/pyref.py (hashlib, affine big-integer points) and the chunked-scan form of
the division (the kernels' three phases) against plain synthetic division."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from oracle import pyref
from oracle.oracle import R_MOD

gpu = pytest.mark.gpu

HALO_EINVAL, HALO_ELEN, HALO_ENOMEM, HALO_ESTATE = -1, -2, -5, -6
R = R_MOD
MINV = pow(1 << 256, -1, R)


# ---- the restatement -------------------------------------------------------------------------------------------------------
def _ints(a):
    b = np.ascontiguousarray(a, dtype=np.uint64).tobytes()
    return [int.from_bytes(b[i:i + 32], "little") for i in range(0, len(b), 32)]


def _limbs(vals):
    return np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in vals), dtype=np.uint64).reshape(-1, 4).copy()


def _canon(a):
    """Montgomery limbs of one scalar -> its canonical value"""
    return _ints(a)[0] * MINV % R


def _mont(x):
    return _limbs([x * (1 << 256) % R])[0]


def horner(p, z):
    a = 0
    for c in reversed(p):
        a = (a * z + c) % R
    return a


def quot(g, z):
    """synthetic division by X - z from the top: h_{i-1} = g_i + z h_i -> (h, g(z))"""
    n = len(g)
    h, acc = [0] * max(n - 1, 0), 0
    for i in range(n - 1, 0, -1):
        acc = (g[i] + z * acc) % R
        h[i - 1] = acc
    return h, ((g[0] + z * acc) % R if n else 0)


def quot_scan(g, z, B, G):
    """the same division in the kernels' three phases: chunks of B coefficients (S_c by Horner), blocks of G chunks (an
    inclusive suffix scan with Z = z^B gives each chunk's carry from its block and the block's aggregate), a scan of the block
    aggregates in runs of G (each block's carry, and g(z)), then each chunk writes its quotient downward from its carry"""
    n = len(g)
    span = B * G
    nblk = max(1, -(-n // span))
    gp = list(g) + [0] * (nblk * span - n)
    Z, Zb = pow(z, B, R), pow(z, span, R)

    def suffix_scan(v, M):  # Hillis-Steele: v_u <- sum_{w >= u} v_w M^(w - u)
        v, d = list(v), 1
        while d < len(v):
            v = [(v[u] + pow(M, d, R) * v[u + d]) % R if u + d < len(v) else v[u] for u in range(len(v))]
            d *= 2
        return v

    kloc, agg = [], []
    for b in range(nblk):
        S = [horner(gp[(b * G + u) * B:(b * G + u + 1) * B], z) for u in range(G)]
        E = suffix_scan(S, Z)
        kloc += [E[u + 1] if u + 1 < G else 0 for u in range(G)]
        agg.append(E[0])
    r = -(-nblk // G)  # runs of r aggregates per thread of the carry kernel
    runs = [horner(agg[u * r:(u + 1) * r], Zb) for u in range(G)]
    E = suffix_scan(runs, pow(Zb, r, R))
    kblk = [0] * nblk
    for u in range(G):
        c = E[u + 1] if u + 1 < G else 0
        for i in range(min((u + 1) * r, nblk) - 1, u * r - 1, -1):
            kblk[i] = c
            c = (c * Zb + agg[i]) % R
    h = [0] * max(n - 1, 0)
    for c in range(nblk * G):
        b, u = divmod(c, G)
        acc = (kloc[c] + pow(Z, G - 1 - u, R) * kblk[b]) % R
        for i in range((c + 1) * B - 1, c * B - 1, -1):
            if i < n - 1:
                h[i] = acc
            acc = (gp[i] + z * acc) % R
    return h, E[0]


def _u64(x):
    return int(x).to_bytes(8, "little")


def _sc(x):
    return int(x % R).to_bytes(32, "little")


def rho2(O, data):
    return int.from_bytes(O.sha3_256(data + (2).to_bytes(4, "little")), "little") % R


def restate_x1(O, Cs, zs, queries, vs):
    """x1 = rho_2(u64 k, u64 T, u64 m, C_j.., z_t.., (u64 j, u64 t, v_i)..) over canonical zs, vs"""
    data = _u64(len(Cs)) + _u64(len(zs)) + _u64(len(queries))
    data += b"".join(O.pt_serialize_compressed(c) for c in Cs) + b"".join(_sc(z) for z in zs)
    data += b"".join(_u64(j) + _u64(t) + _sc(v) for (j, t), v in zip(queries, vs))
    return rho2(O, data)


def restate_claim(O, Cs, zs, queries, vs, Q, us):
    """the verifier's side (halo_pcdl_multi_claim), canonical scalars in and out -> dict(x1, x2, x3, x4, vh, cs, C, v)"""
    T = len(zs)
    x1 = restate_x1(O, Cs, zs, queries, vs)
    x2 = rho2(O, _sc(x1))
    x3 = rho2(O, _sc(x2) + O.pt_serialize_compressed(Q))
    x4 = rho2(O, _sc(x3) + b"".join(_sc(u) for u in us))
    vh = [0] * T
    cs = [0] * len(Cs)
    for i, (j, t) in enumerate(queries):
        vh[t] = (vh[t] + pow(x1, i, R) * vs[i]) % R
        cs[j] = (cs[j] + pow(x4, t + 1, R) * pow(x1, i, R)) % R
    v = sum(pow(x2, t, R) * (us[t] - vh[t]) * pow(x3 - zs[t], -1, R) + pow(x4, t + 1, R) * us[t] for t in range(T)) % R
    Cm = Q
    for j, c in enumerate(Cs):
        Cm = O.pt_add(Cm, O.pt_mul(c, _mont(cs[j])))
    return dict(x1=x1, x2=x2, x3=x3, x4=x4, vh=vh, cs=cs, C=Cm, v=v)


def degree(p):
    nz = [i for i, c in enumerate(p) if c]
    return nz[-1] if nz else 0


def restate_open(O, ps, Cs, d, zs, queries, ws=None, wQ=None, q=None, wb=None, B=None):
    """the prover's side (halo_pcdl_open_multi) -> dict with vs, Q, us (canonical ints), the claim (C, x3, v), pi, P and q
    (Montgomery integers).  B = (chunk, block): the division in the kernels' scan form as well, asserted equal."""
    pm = [_ints(np.asarray(p).reshape(-1, 4)[:d + 1]) for p in ps]
    zc = [_canon(z) for z in zs]
    n = max(len(p) for p in pm)
    vs = [horner(pm[j], zc[t]) * MINV % R for j, t in queries]
    x1 = restate_x1(O, Cs, zc, queries, vs)
    x2 = rho2(O, _sc(x1))
    T = len(zs)
    f = [[0] * n for _ in range(T)]
    for i, (j, t) in enumerate(queries):
        w = pow(x1, i, R)
        f[t] = [(a + w * (pm[j][l] if l < len(pm[j]) else 0)) % R for l, a in enumerate(f[t])]
    qm = [0] * max(n - 1, 0)
    for t in range(T):
        h, rem = quot(f[t], zc[t])
        if B is not None:
            assert quot_scan(f[t], zc[t], *B) == (h, rem)
        vh = sum(pow(x1, i, R) * vs[i] for i, (_, tt) in enumerate(queries) if tt == t) % R
        assert rem * MINV % R == vh  # f_t(z_t) = v^_t: honest claims divide exactly
        s = pow(x2, t, R)
        qm = [(a + s * b) % R for a, b in zip(qm, h)]
    Q = O.pcdl_commit(_limbs(qm) if qm else np.zeros((0, 4), dtype=np.uint64), d, wQ)
    x3 = rho2(O, _sc(x2) + O.pt_serialize_compressed(Q))
    us = [horner(f[t], x3) * MINV % R for t in range(T)]
    cl = restate_claim(O, Cs, zc, queries, vs, Q, us)
    assert cl["x3"] == x3
    P = list(qm) + [0] * (n - len(qm))
    for j, p in enumerate(pm):
        P = [(a + cl["cs"][j] * (p[l] if l < len(p) else 0)) % R for l, a in enumerate(P)]
    w = None
    if ws is not None:
        w = (_canon(wQ) + sum(cl["cs"][j] * _canon(ws[j]) for j in range(len(ps)))) % R
        w = _mont(w)
    qd = None if q is None else np.asarray(q)[:degree(P)]
    pi = O.pcdl_open(_limbs(P), cl["C"], d, _mont(x3), w, qd, wb, threads=8)
    return dict(vs=vs, Q=Q, us=us, C=cl["C"], x3=x3, v=cl["v"], pi=pi, P=P, q=qm, w=w)


# ---- CPU: the restatement, pyref and the scan form ------------------------------------------------------------------------
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
            np.zeros((7, 4), dtype=np.uint64), np.tile(O.to_mont([R - 1])[0], (D_CPU + 1, 1))]


CPU_SHAPES = {
    1: [(0, 0), (1, 0), (2, 0), (3, 0), (4, 0)],
    2: [(0, 0), (1, 1), (2, 0), (0, 1), (3, 1), (4, 0)],
    3: [(0, 0), (1, 2), (2, 1), (0, 2), (3, 0), (4, 1), (1, 0)],
}


@pytest.mark.parametrize("hiding", [False, True])
@pytest.mark.parametrize("T", [1, 2, 3])
def test_oracle_open_multi(cpu_env, T, hiding):
    """the restated multi-point opening: exact division (plain and in scan form), P(x3) = v, C = commit(P) + w S, and the
    oracle's check accepts the final claim"""
    O = cpu_env
    ps = _cpu_polys(O, 60 + T)
    ws = O.random_scalars(len(ps), 70) if hiding else None
    Cs = [O.pcdl_commit(p, D_CPU, None if ws is None else ws[j]) for j, p in enumerate(ps)]
    zs = O.random_scalars(T, 71 + T)
    wQ, wb = O.random_scalars(2, 72)
    q = O.random_scalars(D_CPU, 73) if hiding else None
    r = restate_open(O, ps, Cs, D_CPU, zs, CPU_SHAPES[T], ws, wQ if hiding else None, q, wb if hiding else None, B=(4, 8))
    assert horner(r["P"], r["x3"]) * MINV % R == r["v"]
    assert O.pt_eq(r["C"], O.pcdl_commit(_limbs(r["P"]), D_CPU, r["w"]))
    assert O.pcdl_check(r["C"], D_CPU, _mont(r["x3"]), _mont(r["v"]), r["pi"]) == 0


def test_scan_form_edges():
    """the three-phase division equals synthetic division at lengths around chunk and block boundaries, z = 0, 1, r - 1"""
    import random

    rnd = random.Random(5)
    for n in (0, 1, 2, 3, 4, 5, 31, 32, 33, 63, 64, 65, 255, 256, 257, 1000):
        g = [rnd.randrange(R) for _ in range(n)]
        for z in (0, 1, R - 1, rnd.randrange(R)):
            assert quot_scan(g, z, 4, 8) == quot(g, z), (n, z)
    g = [rnd.randrange(R) for _ in range(5000)]
    assert quot_scan(g, 3, 16, 16) == quot(g, 3)


def test_transcript_matches_pyref(oracle):
    """x1 .. x4 of the restatement equal hashlib over pyref's serialisation of the affine points"""
    O = oracle
    base = O.affine_to_jac(O.derive_points(2, 3))
    Cs = [O.pt_mul(base[0], O.random_scalars(1, 80)[0]), O.pt_from_affine_ints(None), base[1]]
    zs = [_canon(z) for z in O.random_scalars(2, 81)]
    queries = [(0, 0), (1, 1), (2, 0), (2, 1)]
    vs = [_canon(v) for v in O.random_scalars(4, 82)]
    us = [_canon(u) for u in O.random_scalars(2, 83)]
    Q = O.pt_mul(base[2], O.random_scalars(1, 84)[0])
    cl = restate_claim(O, Cs, zs, queries, vs, Q, us)

    def rho(*parts):
        return int.from_bytes(hashlib.sha3_256(b"".join(parts) + (2).to_bytes(4, "little")).digest(), "little") % pyref.R

    pts = [pyref.serialize_compressed_point(O.pt_to_affine_ints(c)) for c in Cs]
    x1 = rho(_u64(3), _u64(2), _u64(4), *pts, *[pyref.serialize_scalar(z) for z in zs],
             *[_u64(j) + _u64(t) + pyref.serialize_scalar(v) for (j, t), v in zip(queries, vs)])
    x2 = rho(pyref.serialize_scalar(x1))
    x3 = rho(pyref.serialize_scalar(x2), pyref.serialize_compressed_point(O.pt_to_affine_ints(Q)))
    x4 = rho(pyref.serialize_scalar(x3), *[pyref.serialize_scalar(u) for u in us])
    assert (cl["x1"], cl["x2"], cl["x3"], cl["x4"]) == (x1, x2, x3, x4)
    C_py = pyref.pt_add(O.pt_to_affine_ints(Q), pyref.msm([O.pt_to_affine_ints(c) for c in Cs], cl["cs"]))
    assert O.pt_to_affine_ints(cl["C"]) == C_py


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


def _rotations(O, seed):
    """z, omega z, omega^-1 z with omega of order 2^10"""
    z = _canon(O.random_scalars(1, seed)[0])
    om = pow(5, (R - 1) >> 10, R)
    return O.to_mont([z, z * om % R, z * pow(om, -1, R) % R])


def _shape(O, name, n, seed):
    """-> (ps, zs, queries)"""
    if name == "k1T1":
        return [O.random_scalars(n - 3, seed)], O.random_scalars(1, seed + 1), [(0, 0)]
    if name == "k3T2":
        ps = [O.random_scalars(n, seed), O.random_scalars(n - 37, seed + 1), O.random_scalars(5, seed + 2)]
        return ps, O.random_scalars(2, seed + 3), [(j, t) for t in range(2) for j in range(3)]
    if name == "k8T3":  # ragged: polynomials at one, two or three of the rotations
        ps = [O.random_scalars(n, seed), O.random_scalars(n - 37, seed + 1), np.zeros((n // 2, 4), dtype=np.uint64),
              np.zeros((0, 4), dtype=np.uint64), np.tile(O.to_mont([R - 1])[0], (n - 1, 1)), O.random_scalars(3, seed + 2),
              O.random_scalars(n, seed + 3), O.random_scalars(n // 4, seed + 4)]
        qs = [(0, 0), (0, 1), (0, 2), (1, 0), (2, 1), (3, 2), (4, 0), (4, 2), (5, 1), (6, 0), (7, 2), (6, 1)]
        return ps, _rotations(O, seed + 5), qs
    raise ValueError(name)


def _draws(O, ps, hiding, seed):
    if not hiding:
        return None, None, None, None
    deg = max(degree(_ints(p)) for p in ps)
    return (O.random_scalars(len(ps), seed), O.random_scalars(1, seed + 1)[0], O.random_scalars(deg, seed + 2),
            O.random_scalars(1, seed + 3)[0])


def _check_equal(O, out, r):
    vs, Q, us, Cm, x, v, pi = out
    assert [_canon(a) for a in vs] == r["vs"]
    assert O.pt_eq(Q, r["Q"])
    assert [_canon(a) for a in us] == r["us"]
    assert O.pt_eq(Cm, r["C"]) and _canon(x) == r["x3"] and _canon(v) == r["v"]
    _same_proof(O, pi, r["pi"])


@gpu
@pytest.mark.parametrize("hiding", [False, True])
@pytest.mark.parametrize("lg", [10, 12])
@pytest.mark.parametrize("shape", ["k1T1", "k3T2", "k8T3"])
def test_against_restatement(env, shape, lg, hiding):
    """vs, Q, us, C, x3, v and every proof field equal the restatement's; the claim is accepted by pcdl.check and the oracle,
    and multi_claim gives the same (C, x3, v)"""
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    n = 1 << lg
    d = n - 1
    ps, zs, qs = _shape(O, shape, n, 1000 + lg)
    ws, wQ, q, wb = _draws(O, ps, hiding, 1100 + lg)
    Cs = pcdl.commit_batch(ctx, ps, d, ws)
    out = pcdl.open_multi(ctx, ps, Cs, d, zs, qs, ws, wQ, q, wb)
    r = restate_open(O, ps, Cs, d, zs, qs, ws, wQ, q, wb)
    _check_equal(O, out, r)
    vs, Q, us, Cm, x, v, pi = out
    pcdl.check(ctx, Cm, d, x, v, pi)
    assert O.pcdl_check(Cm, d, x, v, O.EvalProof.from_buffer_copy(bytes(pi))) == 0
    mC, mx, mv = pcdl.multi_claim(ctx, Cs, zs, qs, vs, Q, us)
    assert O.pt_eq(mC, Cm) and list(mx) == list(x) and list(mv) == list(v)


def _lib():
    from halo_accumulation_b200 import _capi

    return _capi.load(), _capi.p64


def _upload(env, ps, n):
    from halo_accumulation_b200 import _capi

    lib, p = _lib()
    packed, lens = _capi.pack(ps)
    assert lib.halo_poly_upload(env["ctx"]._h, p(packed), p(lens), C.c_uint64(len(lens)), C.c_uint64(n)) == 0


def _device_quotient(env, zs, scales, queries, weights):
    lib, p = _lib()
    qp = np.array([j for j, _ in queries], dtype=np.uint64)
    qt = np.array([t for _, t in queries], dtype=np.uint64)
    T, m = len(zs), len(queries)
    rems, Q = np.zeros((T, 4), dtype=np.uint64), np.zeros(12, dtype=np.uint64)
    h = env["ctx"]._h
    assert lib.halo_poly_quotient(h, p(np.ascontiguousarray(zs)), p(np.ascontiguousarray(scales)), C.c_uint64(T), p(qp), p(qt),
                                  p(np.ascontiguousarray(weights)), C.c_uint64(m), p(rems), p(Q)) == 0
    nq = C.c_uint64(0)
    assert lib.halo_test_read_quotient(h, None, C.c_uint64(0), C.byref(nq)) == 0
    out = np.zeros((max(1, nq.value), 4), dtype=np.uint64)
    assert lib.halo_test_read_quotient(h, p(out), C.c_uint64(nq.value), C.byref(nq)) == 0
    return rems, Q, out[:nq.value]


@gpu
@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 255, 256, 257, (1 << 16) + 3, 1 << 20])
def test_quotient_kernel(env, n):
    """the resident quotient, coefficient by coefficient, and the remainders equal Python synthetic division at z = 0, 1,
    r - 1 and random points (each its own group, weighted), and Q = <GS, q>"""
    ctx, O = env["ctx"], env["O"]
    if n > 1 << 16:
        ctx.derive_generators(1 << 20)
    try:
        ps = [O.random_scalars(n, 1200 + n % 997), O.random_scalars(max(1, n // 3), 1201)]
        zc = [0, 1, R - 1, _canon(O.random_scalars(1, 1202)[0])]
        if n >= 1 << 16:
            zc = zc[2:]  # two points: the Python division is the slow part
        T = len(zc)
        queries = [(t % 2, t) for t in range(T)] + [((t + 1) % 2, t) for t in range(T)]
        weights = O.random_scalars(len(queries), 1203)
        scales = O.random_scalars(T, 1204)
        _upload(env, ps, max(n, 2))
        rems, Q, qd = _device_quotient(env, O.to_mont(zc), scales, queries, weights)
        pm = [_ints(p) for p in ps]
        qm = [0] * (n - 1)
        for t in range(T):
            f = [0] * n
            for i, (j, tt) in enumerate(queries):
                if tt == t:
                    w = _canon(weights[i])
                    f = [(a + w * (pm[j][l] if l < len(pm[j]) else 0)) % R for l, a in enumerate(f)]
            h, rem = quot(f, zc[t])
            assert _ints(rems[t])[0] == rem, t
            s = _canon(scales[t])
            qm = [(a + s * b) % R for a, b in zip(qm, h)]
        assert _ints(qd) == qm
        if n <= 4096:
            assert O.pt_eq(Q, O.pcdl_commit(qd, (1 << 16) - 1) if n > 1 else O.pt_from_affine_ints(None))
    finally:
        ctx.derive_generators(1 << 16)


@gpu
def test_quotient_max_points(env):
    """HALO_MULTI_MAX_POINTS = 64 points, one polynomial each, against synthetic division"""
    O = env["O"]
    n, T = 300, 64
    ps = [O.random_scalars(n - t, 1300 + t) for t in range(T)]
    zc = [_canon(z) for z in O.random_scalars(T, 1400)]
    queries = [(t, t) for t in range(T)]
    weights, scales = O.random_scalars(T, 1401), O.random_scalars(T, 1402)
    _upload(env, ps, n)
    rems, _, qd = _device_quotient(env, O.to_mont(zc), scales, queries, weights)
    qm = [0] * (n - 1)
    for t in range(T):
        w, s = _canon(weights[t]), _canon(scales[t])
        h, rem = quot([w * c % R for c in _ints(ps[t])] + [0] * t, zc[t])
        assert _ints(rems[t])[0] == rem
        qm = [(a + s * b) % R for a, b in zip(qm, h)]
    assert _ints(qd) == qm


@gpu
def test_eval_queries_kernel(env):
    """halo_poly_eval_queries equals O.scalar_dot with z's powers at lengths around chunk (16) and block (4096) boundaries,
    and the one-point halo_poly_eval_many"""
    ctx, O = env["ctx"], env["O"]
    lib, p = _lib()
    lens = [0, 1, 15, 16, 17, 4095, 4096, 4097, 8193, 12288]
    ps = [O.random_scalars(n, 1500 + n) for n in lens]
    zs = np.concatenate([O.to_mont([0, 1, R - 1]), O.random_scalars(1, 1501)])
    queries = [(j, t) for j in range(len(ps)) for t in range(len(zs))]
    _upload(env, ps, 1 << 14)
    qp = np.array([j for j, _ in queries], dtype=np.uint64)
    qt = np.array([t for _, t in queries], dtype=np.uint64)
    vs = np.zeros((len(queries), 4), dtype=np.uint64)
    assert lib.halo_poly_eval_queries(ctx._h, p(zs), C.c_uint64(len(zs)), p(qp), p(qt), C.c_uint64(len(queries)), p(vs)) == 0
    for i, (j, t) in enumerate(queries):
        ref = O.scalar_dot(ps[j], O.construct_powers(zs[t], len(ps[j]))) if lens[j] else np.zeros(4, dtype=np.uint64)
        assert list(vs[i]) == list(ref), (lens[j], t)
    from halo_accumulation_b200 import _capi

    packed, ln = _capi.pack(ps)
    one = np.zeros((len(ps), 4), dtype=np.uint64)
    assert lib.halo_poly_eval_many(ctx._h, p(packed), p(ln), C.c_uint64(len(ps)), C.c_uint64(1 << 14), p(zs[3]), p(one)) == 0
    assert np.array_equal(one, vs[3::4])


@gpu
def test_accumulation(env):
    """the final claim: check_batch, and acc.prover / verifier / decider on the GPU and in the oracle"""
    ctx, O, pcdl, acc = env["ctx"], env["O"], env["pcdl"], env["acc"]
    d = (1 << 10) - 1
    ps, zs, qs = _shape(O, "k8T3", d + 1, 1600)
    ws, wQ, q, wb = _draws(O, ps, True, 1601)
    Cs = pcdl.commit_batch(ctx, ps, d, ws)
    _, _, _, Cm, x, v, pi = pcdl.open_multi(ctx, ps, Cs, d, zs, qs, ws, wQ, q, wb)
    inst = acc.new_instance(Cm, d, x, v, pi)
    pcdl.check_batch(ctx, [inst, inst], O.random_scalars(1, 1602)[0])
    a = acc.prover(ctx, d, [inst], O.random_scalars(2, 1603), O.random_scalars(1, 1604)[0], O.random_scalars(d, 1605),
                   O.random_scalars(1, 1606)[0])
    acc.verifier(ctx, d, [inst], a)
    acc.decider(ctx, a)
    oq = O.Instance.from_buffer_copy(bytes(inst))
    oa = O.Accumulator.from_buffer_copy(bytes(a))
    assert O.pcdl_check(Cm, d, x, v, O.EvalProof.from_buffer_copy(bytes(pi))) == 0
    assert O.acc_verifier(d, [oq], oa) == 0
    assert O.acc_decider(oa) == 0


@gpu
def test_2_20_fixed_base(env):
    """k = 8, T = 3 at 2^20 over FIXED-base tables, hiding: the claim is accepted, (C, x3, v) is the restated claim, and the
    proof equals pcdl.open of P = q + sum_j c_j p_j restated from the read-back quotient (test_quotient_kernel checks q)"""
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    n = 1 << 20
    d = n - 1
    ctx.derive_generators(n)
    ctx.precompute_generators(0)
    try:
        ps, zs, qs = _shape(O, "k8T3", n, 1700)
        ws, wQ, q, wb = _draws(O, ps, True, 1701)
        Cs = pcdl.commit_batch(ctx, ps, d, ws)
        vs, Q, us, Cm, x, v, pi = pcdl.open_multi(ctx, ps, Cs, d, zs, qs, ws, wQ, q, wb)
        pcdl.check(ctx, Cm, d, x, v, pi)
        cl = restate_claim(O, Cs, [_canon(z) for z in zs], qs, [_canon(a) for a in vs], Q, [_canon(u) for u in us])
        assert O.pt_eq(Cm, cl["C"]) and _canon(x) == cl["x3"] and _canon(v) == cl["v"]
        lib, p = _lib()
        nq = C.c_uint64(0)
        assert lib.halo_test_read_quotient(ctx._h, None, C.c_uint64(0), C.byref(nq)) == 0
        qd = np.zeros((nq.value, 4), dtype=np.uint64)
        assert lib.halo_test_read_quotient(ctx._h, p(qd), C.c_uint64(nq.value), C.byref(nq)) == 0
        P = _ints(qd) + [0]
        for j, pj in enumerate(ps):
            c = cl["cs"][j]
            for l, a in enumerate(_ints(pj)):
                P[l] = (P[l] + c * a) % R
        assert horner(P, cl["x3"]) * MINV % R == _canon(v)
        w = _mont((_canon(wQ) + sum(cl["cs"][j] * _canon(ws[j]) for j in range(8))) % R)
        ref = pcdl.open(ctx, _limbs(P), Cm, d, x, w, q[:degree(P)], wb)
        _same_proof(O, pi, ref)
    finally:
        ctx.derive_generators(1 << 16)


@gpu
@pytest.mark.parametrize("hiding", [False, True])
def test_soundness(env, hiding):
    """one v_i, one u_t or Q changed, a query moved to another point, two queries swapped: multi_claim + check rejects with
    the oracle's code"""
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    d = (1 << 10) - 1
    ps, zs, qs = _shape(O, "k8T3", d + 1, 1800)
    ws, wQ, q, wb = _draws(O, ps, hiding, 1801)
    Cs = pcdl.commit_batch(ctx, ps, d, ws)
    vs, Q, us, Cm, x, v, pi = pcdl.open_multi(ctx, ps, Cs, d, zs, qs, ws, wQ, q, wb)
    opi = O.EvalProof.from_buffer_copy(bytes(pi))
    one = O.to_mont([1])[0]

    def bump(a, i):
        b = a.copy()
        b[i] = _mont((_canon(b[i]) + 1) % R)
        return b

    moved = list(qs)
    moved[4] = (2, 0)  # polynomial 2 at z_0 instead of z_1 (its only query): still a valid query set
    swapped = list(qs)
    swapped[1], swapped[2] = swapped[2], swapped[1]
    Q2 = O.pt_add(Q, O.pt_mul(Cs[0], one))
    for qs_x, vs_x, Q_x, us_x in ((qs, bump(vs, 5), Q, us), (qs, vs, Q, bump(us, 1)), (qs, vs, Q2, us), (moved, vs, Q, us),
                                  (swapped, vs, Q, us)):
        mC, mx, mv = pcdl.multi_claim(ctx, Cs, zs, qs_x, vs_x, Q_x, us_x)
        cl = restate_claim(O, Cs, [_canon(z) for z in zs], qs_x, [_canon(a) for a in vs_x], Q_x, [_canon(u) for u in us_x])
        assert O.pt_eq(mC, cl["C"]) and _canon(mx) == cl["x3"] and _canon(mv) == cl["v"]
        code = O.pcdl_check(mC, d, mx, mv, opi)
        assert code != 0
        with pytest.raises(pcdl.Rejected) as e:
            pcdl.check(ctx, mC, d, mx, mv, pi)
        assert e.value.code == code


def _raw_open_multi(env, ps, Cs, d, zs, queries, ws=None, wQ=None, q=None, wb=None, k=None, T=None, m=None):
    """halo_pcdl_open_multi with sentinel outputs -> (rc, outputs untouched)"""
    from halo_accumulation_b200 import _capi, _host

    packed, lens = _capi.pack(ps)
    k = len(lens) if k is None else k
    zs = np.ascontiguousarray(zs, dtype=np.uint64).reshape(-1, 4)
    T = zs.shape[0] if T is None else T
    qp = np.array([j for j, _ in queries] or [0], dtype=np.uint64)
    qt = np.array([t for _, t in queries] or [0], dtype=np.uint64)
    m = len(queries) if m is None else m
    Cs = None if Cs is None else np.ascontiguousarray(Cs, dtype=np.uint64).reshape(-1, 12)
    vs, us = np.full((max(1, len(queries)), 4), 0xAB, dtype=np.uint64), np.full((max(1, zs.shape[0]), 4), 0xAB, dtype=np.uint64)
    Q, Cm = np.full(12, 0xAB, dtype=np.uint64), np.full(12, 0xAB, dtype=np.uint64)
    x, v = np.full(4, 0xAB, dtype=np.uint64), np.full(4, 0xAB, dtype=np.uint64)
    pi = _host.EvalProof()
    C.memset(C.byref(pi), 0xAB, C.sizeof(pi))

    def opt(a, shape):
        return None if a is None else np.ascontiguousarray(a, dtype=np.uint64).reshape(shape)

    wa, wqa, qa, wba = opt(ws, (-1, 4)), opt(wQ, (4,)), opt(q, (-1, 4)), opt(wb, (4,))
    p = _capi.p64
    P = (lambda a: None if a is None else p(a))
    rc = _host.lib().halo_pcdl_open_multi(env["ctx"]._h, p(packed), p(lens), C.c_uint64(k), P(Cs), C.c_uint64(d), p(zs),
                                          C.c_uint64(T), p(qp), p(qt), C.c_uint64(m), P(wa), P(wqa), P(qa),
                                          C.c_uint64(0 if qa is None else qa.shape[0]), P(wba), p(vs), p(Q), p(us), p(Cm), p(x),
                                          p(v), C.byref(pi))
    untouched = all((a == 0xAB).all() for a in (vs, us, Q, Cm, x, v)) and bytes(pi) == bytes([0xAB]) * C.sizeof(pi)
    return rc, untouched


@gpu
def test_errors(env, halo):
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    from halo_accumulation_b200 import _capi

    d = (1 << 10) - 1
    ps = [O.random_scalars(d + 1, 1900 + j) for j in range(3)]
    ws, wQ, q, wb = _draws(O, ps, True, 1910)
    Cs = pcdl.commit_batch(ctx, ps, d, ws)
    zs = O.random_scalars(2, 1911)
    qs = [(0, 0), (1, 1), (2, 0), (0, 1)]
    good = (ps, Cs, d, zs, qs, ws, wQ, q, wb)
    consts = [O.random_scalars(1, 1931 + j) for j in range(3)]
    C_consts = pcdl.commit_batch(ctx, consts, d, ws)
    launches = ctx.kernel_launches()
    big = np.full(4, 0xFFFFFFFFFFFFFFFF, dtype=np.uint64)

    def with_(i, val):
        a = list(good)
        a[i] = val
        return a

    cases = []
    for j in range(3):  # a malformed polynomial at position j, then d + 1 not a power of two
        bad = list(ps)
        bad[j] = O.random_scalars(d + 2, 1920 + j)
        cases.append(with_(0, bad))
    cases.append(with_(2, d - 1))
    off_curve, non_canon = Cs.copy(), Cs.copy()
    off_curve[2, 0] ^= np.uint64(1)
    non_canon[1, :4] = np.uint64(0xFFFFFFFFFFFFFFFF)
    cases += [with_(1, off_curve), with_(1, non_canon)]
    bad_z = zs.copy()
    bad_z[1] = big
    bad_w = ws.copy()
    bad_w[2] = big
    cases += [with_(3, bad_z), with_(5, bad_w), with_(6, big), with_(8, big)]
    cases.append(with_(3, np.stack([zs[0], zs[0]])))                 # duplicate points
    cases.append(with_(4, qs + [(3, 0)]))                            # polynomial index out of range
    cases.append(with_(4, qs + [(1, 2)]))                            # point index out of range
    cases.append(with_(4, qs + [(2, 0)]))                            # a (j, t) pair twice
    cases.append(with_(4, [(0, 0), (1, 0), (2, 0)]))                 # point 1 unused
    cases.append(with_(4, [(0, 0), (1, 1), (0, 1)]))                 # polynomial 2 unused
    for args in cases:
        assert _raw_open_multi(env, *args) == (HALO_EINVAL, True)
    for kw in (dict(k=0), dict(T=0), dict(m=0)):
        assert _raw_open_multi(env, *good, **kw) == (HALO_EINVAL, True)
    assert _raw_open_multi(env, ps, None, d, zs, qs, ws, wQ, q, wb) == (HALO_EINVAL, True)
    assert _raw_open_multi(env, ps, Cs, d, zs, qs, ws, None, q, wb) == (HALO_EINVAL, True)
    # n_q != max_j deg(p_j); hiding with constant polynomials only
    for nq in (len(q) - 1, len(q) + 1):
        assert _raw_open_multi(env, *with_(7, O.random_scalars(nq, 1930))) == (HALO_ELEN, True)
    assert _raw_open_multi(env, consts, C_consts, d, zs, qs, ws, wQ,
                           np.zeros((0, 4), dtype=np.uint64), wb) == (HALO_ELEN, True)
    assert ctx.kernel_launches() == launches
    # multi_claim: non-canonical v_i, u_t, Q; Q off the curve; the query errors
    vs, Q, us, Cm, x, v, pi = pcdl.open_multi(ctx, *good)
    bad_v, bad_u = vs.copy(), us.copy()
    bad_v[0], bad_u[1] = big, big
    bad_Q = Q.copy()
    bad_Q[0] ^= np.uint64(1)
    for args in ((Cs, zs, qs, bad_v, Q, us), (Cs, zs, qs, vs, Q, bad_u), (Cs, zs, qs, vs, bad_Q, us),
                 (Cs, zs, qs + [(2, 0)], np.concatenate([vs, vs[:1]]), Q, us), (Cs, np.stack([zs[0], zs[0]]), qs, vs, Q, us)):
        with pytest.raises(_capi.HaloError) as e:
            pcdl.multi_claim(ctx, *args)
        assert e.value.code == HALO_EINVAL
    # the device layer: no upload, no quotient, an upload the device cannot hold
    lib, p = _lib()
    fresh = halo.Context(0, 1 << 16)
    try:
        fresh.derive_generators(1 << 16)
        h = fresh._h
        z1 = O.random_scalars(1, 1940)
        zero = np.zeros(1, dtype=np.uint64)
        out = np.zeros((1, 4), dtype=np.uint64)
        Qo = np.zeros(12, dtype=np.uint64)
        deg, nq = C.c_uint64(0), C.c_uint64(0)
        assert lib.halo_poly_eval_queries(h, p(z1), C.c_uint64(1), p(zero), p(zero), C.c_uint64(1), p(out)) == HALO_ESTATE
        assert lib.halo_poly_quotient(h, p(z1), p(z1), C.c_uint64(1), p(zero), p(zero), p(z1), C.c_uint64(1), p(out),
                                      p(Qo)) == HALO_ESTATE
        assert lib.halo_poly_lincomb_resident(h, p(z1), p(z1[0]), C.byref(deg)) == HALO_ESTATE
        assert lib.halo_test_read_quotient(h, None, C.c_uint64(0), C.byref(nq)) == HALO_ESTATE
        _, lens1 = _capi.pack([O.random_scalars(100, 1941)])
        packed1 = O.random_scalars(100, 1941)
        assert lib.halo_poly_upload(h, p(packed1), p(lens1), C.c_uint64(1), C.c_uint64(128)) == 0
        assert lib.halo_poly_lincomb_resident(h, p(z1), p(z1[0]), C.byref(deg)) == HALO_ESTATE  # uploaded, no quotient
        assert lib.halo_poly_eval_queries(h, p(z1), C.c_uint64(1), p(np.ones(1, dtype=np.uint64)), p(zero), C.c_uint64(1),
                                          p(out)) == HALO_EINVAL  # j = 1 >= k
        assert lib.halo_poly_eval_queries(h, p(z1), C.c_uint64(65), p(zero), p(zero), C.c_uint64(1), p(out)) == HALO_EINVAL
        assert not out.any()
        k = 1 << 20  # 2^20 polynomials of 2^16 coefficients: 2 TiB, refused before the (one-element) host buffer is read
        lens = np.full(k, 1 << 16, dtype=np.uint64)
        assert lib.halo_poly_upload(h, p(packed1), p(lens), C.c_uint64(k), C.c_uint64(1 << 16)) == HALO_ENOMEM
        assert lib.halo_poly_eval_queries(h, p(z1), C.c_uint64(1), p(zero), p(zero), C.c_uint64(1), p(out)) == HALO_ESTATE
    finally:
        fresh.close()
    # and the shared context still opens
    vs, Q, us, Cm, x, v, pi = pcdl.open_multi(ctx, *good)
    pcdl.check(ctx, Cm, d, x, v, pi)
