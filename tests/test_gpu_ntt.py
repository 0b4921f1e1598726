"""Polynomials in evaluation form (DESIGN.md K8; definitions in include/halo_b200.h): the batched transform over the scalar field
(Context.ntt / ntt_resident, halo_domain_root) and the PCS entry points that take evaluations (pcdl.commit_evals,
pcdl.open_multi_evals).

The restatement lives here, in big integers: omega_{2^s} = 5^((r - 1) / 2^s), an O(n^2) DFT, a radix-2 FFT and the kernels'
pass decomposition (Stockham passes of at most 2^11 points).  Montgomery limbs are linear, so the transform of the limbs as
integers with canonical twiddles is the Montgomery form of the transform: inputs and outputs are compared as limbs."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle.oracle import R_MOD

gpu = pytest.mark.gpu

HALO_EINVAL, HALO_ELEN, HALO_ESTATE = -1, -2, -6
R = R_MOD
MONT = 1 << 256
MINV = pow(MONT, -1, R)
CURVE = os.environ.get("HALO_B200_CURVE", "pallas")
OMEGA_2_32 = {  # canonical omega_{2^32} of each build's scalar field
    "pallas": 0x2de6a9b8746d3f589e5c4dfd492ae26e9bb97ea3c106f049a70e2c1102b6d05f,
    "vesta": 0x2bce74deac30ebda362120830561f81aea322bf2b7bb7584bdad6fabd87ea32f,
}
FIELDS = {  # scalar-field modulus of each build
    "pallas": 0x40000000000000000000000000000000224698FC0994A8DD8C46EB2100000001,
    "vesta": 0x40000000000000000000000000000000224698FC094CF91B992D30ED00000001,
}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- the restatement -------------------------------------------------------------------------------------------------------
def _ints(a):
    b = np.ascontiguousarray(a, dtype=np.uint64).tobytes()
    return [int.from_bytes(b[i:i + 32], "little") for i in range(0, len(b), 32)]


def _limbs(vals):
    if not len(vals):
        return np.zeros((0, 4), dtype=np.uint64)
    return np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in vals), dtype=np.uint64).reshape(-1, 4).copy()


def _mont(x):
    return _limbs([x * MONT % R])[0]


def root(lg, r=R):
    return pow(5, (r - 1) >> lg, r)


def dft(a, lg, g=1, inverse=False):
    """the definition, O(n^2): forward e_i = sum_j a_j (g w^i)^j; inverse a_j = g^-j n^-1 sum_i e_i w^-ij"""
    n = 1 << lg
    a = list(a) + [0] * (n - len(a))
    if not inverse:
        w = root(lg)
        return [sum(a[j] * pow(g * pow(w, i, R), j, R) for j in range(n)) % R for i in range(n)]
    wi, gi, ni = pow(root(lg), -1, R), pow(g, -1, R), pow(n, -1, R)
    return [ni * pow(gi, j, R) * sum(a[i] * pow(wi, i * j, R) for i in range(n)) % R for j in range(n)]


def _fft(a, w):
    """iterative radix-2 DIT over Z_r, natural order in and out"""
    n = len(a)
    lg = n.bit_length() - 1
    a = [a[int(format(i, f"0{lg}b")[::-1], 2) if lg else 0] for i in range(n)]
    m = 1
    while m < n:
        wm = pow(w, n // (2 * m), R)
        tw = [1] * m
        for j in range(1, m):
            tw[j] = tw[j - 1] * wm % R
        for s in range(0, n, 2 * m):
            for j in range(m):
                u, t = a[s + j], a[s + j + m] * tw[j] % R
                a[s + j], a[s + j + m] = (u + t) % R, (u - t) % R
        m *= 2
    return a


def ntt(a, lg, g=1, inverse=False):
    """the restatement the GPU is compared with: a radix-2 FFT with the coset factors around it"""
    n = 1 << lg
    a = list(a) + [0] * (n - len(a))
    if not inverse:
        return _fft([x * pow(g, j, R) % R for j, x in enumerate(a)], root(lg))
    gi, ni = pow(g, -1, R), pow(n, -1, R)
    e = _fft(a, pow(root(lg), -1, R))
    return [x * ni % R * pow(gi, j, R) % R for j, x in enumerate(e)]


def stockham(a, lg, g=1, inverse=False, max_lg=11):
    """the kernels' decomposition (csrc/ntt.cu): ceil(lg / 11) passes of radix R = 2^lr; group j loads x[j + r n/R] times
    w_{Ns R}^(r (j mod Ns)), runs an R-point DFT (bit-reversed placement, radix-2 stages) and stores to
    y[(j / Ns) Ns R + (j mod Ns) + r Ns]; coset factors at the first loads (forward) or the last stores (inverse)"""
    n = 1 << lg
    P = 1 if lg <= max_lg else -(-lg // max_lg)
    lrs = [lg // P + (1 if p < lg % P else 0) for p in range(P)]
    w = root(lg) if not inverse else pow(root(lg), -1, R)
    x = list(a) + [0] * (n - len(a))
    if not inverse:
        x = [v * pow(g, j, R) % R for j, v in enumerate(x)]
    ns = 1
    for lr in lrs:
        rr = 1 << lr
        y = [0] * n
        for j in range(n // rr):
            k = j % ns
            v = [x[j + r * (n // rr)] * pow(w, r * k * (n // (ns * rr)), R) % R for r in range(rr)]
            v = _fft(v, pow(w, n // rr, R)) if rr > 1 else v
            for r in range(rr):
                y[(j // ns) * ns * rr + k + r * ns] = v[r]
        x, ns = y, ns * rr
    if inverse:
        gi, ni = pow(g, -1, R), pow(n, -1, R)
        x = [v * ni % R * pow(gi, j, R) % R for j, v in enumerate(x)]
    return x


# ---- CPU ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", ["pallas", "vesta"])
def test_domain_root(curve):
    """halo_domain_root of both builds: 5^((r - 1) / 2^lg) in Montgomery form for lg = 0 .. 32, omega_{2^32} as documented,
    omega^(2^31) = -1 and omega^(2^32) = 1; lg = 33 is HALO_EINVAL (no context, no device)"""
    from halo_accumulation_b200 import _build

    _build.build()
    path = os.path.join(ROOT, "halo-accumulation_b200", "lib", "libhalo_b200.so" if curve == "pallas" else "libhalo_b200_vesta.so")
    lib = C.CDLL(path)
    lib.halo_domain_root.argtypes = [C.c_uint32, C.POINTER(C.c_uint64)]
    r = FIELDS[curve]
    out = np.zeros(4, dtype=np.uint64)
    ptr = out.ctypes.data_as(C.POINTER(C.c_uint64))
    for lg in range(33):
        assert lib.halo_domain_root(lg, ptr) == 0
        assert _ints(out)[0] == pow(5, (r - 1) >> lg, r) * MONT % r, lg
    w = _ints(out)[0] * pow(MONT, -1, r) % r
    assert w == OMEGA_2_32[curve]
    assert pow(w, 1 << 31, r) == r - 1 and pow(w, 1 << 32, r) == 1
    assert lib.halo_domain_root(33, ptr) == HALO_EINVAL


def test_restatements_agree():
    """the O(n^2) DFT, the radix-2 FFT and the pass decomposition agree (n <= 64), and FFT = passes at every lg up to 12
    (both directions, cosets included); inverse(forward(x)) = x"""
    import random

    rnd = random.Random(3)
    for lg in range(0, 13):
        n = 1 << lg
        a = [rnd.randrange(R) for _ in range(n)]
        g = rnd.randrange(1, R)
        for inv in (False, True):
            for sh in (1, g):
                f = ntt(a, lg, sh, inv)
                if lg <= 6:
                    assert f == dft(a, lg, sh, inv), (lg, inv)
                assert f == stockham(a, lg, sh, inv), (lg, inv)
                # with a smaller tile the pass boundaries fall inside this range too
                if lg in (5, 9, 12):
                    assert f == stockham(a, lg, sh, inv, max_lg=3)
        assert ntt(ntt(a, lg, g), lg, g, True) == a
    assert ntt([1, 2, 3], 3) == dft([1, 2, 3], 3)  # zero padding


# ---- GPU ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env(ctx, oracle, halo):
    from halo_accumulation_b200 import acc, pcdl

    O = oracle
    S, H = ctx.get_SH()
    O.set_params(S, H, ctx.get_generators(0, 1 << 16))
    yield dict(ctx=ctx, O=O, pcdl=pcdl, acc=acc, halo=halo)
    bad, live = halo.check_canaries()
    assert bad == 0, (bad, live)


def _vectors(O, lg, seed):
    """k = 3 vectors: random, the edge values 0, 1, r - 1 cycled, all equal"""
    n = 1 << lg
    one, rm1 = _ints(O.to_mont([1]))[0], _ints(O.to_mont([R - 1]))[0]
    edge = [[0, one, rm1][i % 3] for i in range(n)]
    same = [_ints(O.random_scalars(1, seed + 1))[0]] * n
    return [_ints(O.random_scalars(n, seed)), edge, same]


def _shifts(O):
    cube = pow(5, (R - 1) // 3, R)  # a primitive cube root of unity (3 divides r - 1)
    assert cube != 1 and pow(cube, 3, R) == 1
    return {"none": None, "5": 5, "cube": cube, "random": _ints(O.random_scalars(1, 77))[0] * MINV % R}


@gpu
@pytest.mark.parametrize("lg", list(range(15)))
def test_against_restatement(env, lg):
    """forward, inverse, coset forward and coset inverse, element by element: lg = 0 .. 14 (every pass-count boundary up to
    there), k = 3 and k = 1, random and edge inputs, shifts 1, 5, a cube root of unity and a random one"""
    ctx, O = env["ctx"], env["O"]
    vs = _vectors(O, lg, 100 + lg)
    a = np.stack([_limbs(v) for v in vs])
    for name, g in _shifts(O).items():
        for inv in (False, True):
            out = ctx.ntt(a, lg, inv, None if g is None else _mont(g))
            for j, v in enumerate(vs):
                assert _ints(out[j]) == ntt(v, lg, 1 if g is None else g, inv), (name, inv, j)
            one = ctx.ntt(a[0], lg, inv, None if g is None else _mont(g))
            assert np.array_equal(one, out[0])


@gpu
@pytest.mark.parametrize("lg", [1, 2, 5, 11, 12, 14])
def test_zero_padded(env, lg):
    """forward with n_in = 0, 1, n/2 and n - 1 coefficients (the rest zero), plain and on a coset"""
    ctx, O = env["ctx"], env["O"]
    n = 1 << lg
    g = _ints(O.random_scalars(1, 90))[0] * MINV % R
    for n_in in sorted({0, 1, n // 2, n - 1}):
        a = _ints(O.random_scalars(max(n_in, 1), 91 + n_in))[:n_in]
        for sh in (None, g):
            out = ctx.ntt(np.stack([_limbs(a), _limbs(a)]) if n_in else np.zeros((2, 0, 4), dtype=np.uint64), lg, False,
                          None if sh is None else _mont(sh))
            want = ntt(a, lg, 1 if sh is None else sh)
            assert _ints(out[0]) == want and _ints(out[1]) == want, (n_in, sh)


def _eval_at_roots(env, coeffs, lg, idxs):
    """p(omega^i) for the given i by halo_poly_eval_queries over the uploaded coefficients (oracle-tested, 64 points a call)"""
    from halo_accumulation_b200 import _capi

    lib, h = _capi.load(), env["ctx"]._h
    n = 1 << lg
    packed = np.ascontiguousarray(coeffs.reshape(-1, 4))
    lens = np.array([n], dtype=np.uint64)
    assert lib.halo_poly_upload(h, _capi.p64(packed), _capi.p64(lens), C.c_uint64(1), C.c_uint64(n)) == 0
    w = root(lg)
    res = []
    for c0 in range(0, len(idxs), 64):
        ch = idxs[c0:c0 + 64]
        zs = np.stack([_mont(pow(w, i, R)) for i in ch])
        qp, qt = np.zeros(len(ch), dtype=np.uint64), np.arange(len(ch), dtype=np.uint64)
        out = np.zeros((len(ch), 4), dtype=np.uint64)
        assert lib.halo_poly_eval_queries(h, _capi.p64(zs), C.c_uint64(len(ch)), _capi.p64(qp), _capi.p64(qt), C.c_uint64(len(ch)),
                                          _capi.p64(out)) == 0
        res += _ints(out)
    return res


@pytest.fixture(scope="module")
def big_ctx(env):
    """a context for transforms up to 2^24 (the session context stops at 2^20)"""
    c = env["halo"].Context(0, 1 << 24)
    yield c
    c.close()


@gpu
@pytest.mark.parametrize("lg", [15, 20, 22, 23, 24])
def test_large(env, big_ctx, lg):
    """2^15 .. 2^24 (2^22 / 2^23: two / three passes): inverse(forward(x)) = x and forward(inverse(x)) = x, coset included; a
    sparse input's forward transform at 64 indices (0, 1, n/2, n - 1 and random ones) against the definition"""
    O, c = env["O"], big_ctx
    n = 1 << lg
    x = O.random_scalars(n, 200 + lg).reshape(1, n, 4)
    g = O.random_scalars(1, 201)[0]
    for sh in (None, g):
        assert np.array_equal(c.ntt(c.ntt(x, lg, False, sh), lg, True, sh), x)
        assert np.array_equal(c.ntt(c.ntt(x, lg, True, sh), lg, False, sh), x)
    rnd = np.random.default_rng(lg)
    pos = sorted(set(int(p) for p in rnd.integers(0, n, 12)) | {0, n - 1})
    vals = _ints(O.random_scalars(len(pos), 202))
    sp = np.zeros((1, n, 4), dtype=np.uint64)
    sp[0, pos] = _limbs(vals)
    idxs = [0, 1, n // 2, n - 1] + [int(i) for i in rnd.integers(0, n, 60)]
    w, gc = root(lg), _ints(g)[0] * MINV % R
    for sh in (1, gc):
        out = c.ntt(sp, lg, False, None if sh == 1 else _mont(sh))
        for i, e in zip(idxs, _ints(out[0, idxs])):
            z = sh * pow(w, i, R) % R
            assert e == sum(v * pow(z, p, R) for p, v in zip(pos, vals)) % R, (sh, i)


@gpu
def test_2_20_against_evaluation(env):
    """a dense forward transform at 2^20 at 64 points by halo_poly_eval_queries at omega^i, one of them by Python Horner"""
    ctx, O = env["ctx"], env["O"]
    lg, n = 20, 1 << 20
    ctx.derive_generators(n)
    try:
        x = O.random_scalars(n, 300)
        e = ctx.ntt(x, lg)
        rnd = np.random.default_rng(5)
        idxs = [0, 1, n // 2, n - 1] + [int(i) for i in rnd.integers(0, n, 60)]
        assert _ints(e[idxs]) == _eval_at_roots(env, x, lg, idxs)
        i = idxs[-1]
        z, acc = pow(root(lg), i, R), 0
        for cf in reversed(_ints(x)):
            acc = (acc * z + cf) % R
        assert _ints(e[i:i + 1])[0] == acc
    finally:
        ctx.derive_generators(1 << 16)


@gpu
@pytest.mark.parametrize("lg,k", [(12, 64), (20, 8)])
def test_batched(env, lg, k):
    """k vectors in one call equal k single calls, both directions and on a coset; the launches for k vectors equal those
    for one"""
    ctx, O = env["ctx"], env["O"]
    n = 1 << lg
    x = O.random_scalars(k * n, 400 + lg).reshape(k, n, 4)
    g = O.random_scalars(1, 401)[0]
    for inv in (False, True):
        for sh in (None, g):
            ctx.ntt(x[:1], lg, inv, sh)  # tables of this size built
            l0 = ctx.kernel_launches()
            one = ctx.ntt(x[:1], lg, inv, sh)
            l1 = ctx.kernel_launches()
            many = ctx.ntt(x, lg, inv, sh)
            assert ctx.kernel_launches() - l1 == l1 - l0
            assert np.array_equal(many[0], one[0])
            for j in range(1, k, max(1, k // 8)):
                assert np.array_equal(many[j], ctx.ntt(x[j], lg, inv, sh))


@gpu
@pytest.mark.parametrize("lg", [3, 12, 23])
def test_resident(env, big_ctx, lg):
    """ntt_resident on a torch CUDA tensor equals ntt on the host (one, two and three passes)"""
    import torch

    O = env["O"]
    c = big_ctx
    k = 3 if lg < 20 else 1
    x = O.random_scalars(k << lg, 500 + lg).reshape(k, 1 << lg, 4)
    g = O.random_scalars(1, 501)[0]
    for inv in (False, True):
        for sh in (None, g):
            t = torch.from_numpy(x.view(np.int64).copy()).cuda()
            torch.cuda.synchronize()
            c.ntt_resident(t.data_ptr(), k, lg, inv, sh)
            got = t.cpu().numpy().view(np.uint64)
            assert np.array_equal(got, c.ntt(x, lg, inv, sh))


@gpu
def test_errors(env):
    """every error path; nothing is written on error"""
    from halo_accumulation_b200 import _capi

    ctx, O = env["ctx"], env["O"]
    lib, p, h = _capi.load(), _capi.p64, ctx._h
    x = O.random_scalars(16, 600)
    out = np.full((16, 4), 7, dtype=np.uint64)
    u = C.c_uint64

    def call(inp, n_in, k, lg, inv, shift, o=out):
        return lib.halo_ntt(h, p(inp) if inp is not None else None, u(n_in), u(k), C.c_uint32(lg), inv, shift, p(o) if o is not None else None)

    good = O.random_scalars(1, 601)[0]
    zero = np.zeros(4, dtype=np.uint64)
    big = _limbs([R])[0]
    assert call(x, 16, 1, 33, 0, None) == HALO_EINVAL
    assert call(x, 16, 1, 21, 0, None) == HALO_EINVAL  # 2^21 > max_n
    assert call(x, 17, 1, 4, 0, None) == HALO_EINVAL
    assert call(x, 8, 1, 4, 1, None) == HALO_ELEN
    assert call(x, 16, 1, 4, 0, p(zero)) == HALO_EINVAL
    assert call(x, 16, 1, 4, 0, p(big)) == HALO_EINVAL
    assert call(None, 16, 1, 4, 0, None) == HALO_EINVAL
    assert call(x, 16, 1, 4, 0, None, None) == HALO_EINVAL
    assert call(x, 16, 1 << 62, 4, 0, None) == HALO_EINVAL  # k 2^lg 32 bytes overflow
    assert (out == 7).all()
    assert call(None, 16, 0, 4, 0, None, None) == 0  # k = 0 does nothing
    assert call(x, 16, 1, 4, 0, p(good)) == 0
    assert lib.halo_ntt_resident(h, None, u(1), C.c_uint32(4), 0, None) == HALO_EINVAL
    assert lib.halo_ntt_resident(h, None, u(0), C.c_uint32(4), 0, None) == 0
    assert lib.halo_ntt_resident(h, C.c_void_p(16), u(1), C.c_uint32(33), 0, None) == HALO_EINVAL
    assert lib.halo_ntt_resident(h, C.c_void_p(16), u(1), C.c_uint32(4), 0, p(zero)) == HALO_EINVAL
    degs = np.full(2, 9, dtype=np.uint64)
    ev = O.random_scalars(32, 602)
    assert lib.halo_poly_upload_evals(h, p(ev), u(2), u(12), p(degs)) == HALO_EINVAL  # not a power of two
    assert lib.halo_poly_upload_evals(h, p(ev), u(0), u(16), p(degs)) == HALO_EINVAL
    assert lib.halo_poly_upload_evals(h, p(ev), u(2), u(1 << 17), p(degs)) == HALO_EINVAL  # beyond the generators
    assert lib.halo_poly_upload_evals(h, None, u(2), u(16), p(degs)) == HALO_EINVAL
    assert (degs == 9).all()
    assert lib.halo_poly_commit_resident(h, None) == HALO_EINVAL
    Cs = np.zeros((2, 12), dtype=np.uint64)
    assert lib.halo_poly_commit_resident(h, p(Cs)) == HALO_ESTATE  # the failed upload left nothing resident


# ---- the PCS entry points ------------------------------------------------------------------------------------------------------
def _intt(E, lg):
    return np.stack([_limbs(ntt(_ints(e), lg, inverse=True)) for e in E])


@gpu
@pytest.mark.parametrize("lg,k", [(10, 1), (10, 8), (16, 1), (16, 8), (20, 1), (20, 8)])
@pytest.mark.parametrize("hiding", [False, True])
def test_commit_evals(env, lg, k, hiding):
    """commit_evals(E) = commit_batch(intt(E)) projectively (FIXED-base tables at 2^20), and the MSM route equals that of
    msm_gens_many on the same lengths"""
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    n, d = 1 << lg, (1 << lg) - 1
    if lg == 20:
        ctx.derive_generators(n)
        ctx.precompute_generators(0)
    try:
        E = O.random_scalars(k * n, 700 + lg + k).reshape(k, n, 4)
        ws = O.random_scalars(k, 701) if hiding else None
        got = pcdl.commit_evals(ctx, E, d, ws)
        route = ctx.test_msm_route()
        coeffs = ctx.ntt(E, lg, inverse=True) if lg > 12 else _intt(E, lg)
        if lg <= 12:
            assert np.array_equal(coeffs, ctx.ntt(E, lg, inverse=True))
        want = pcdl.commit_batch(ctx, list(coeffs), d, ws)
        for j in range(k):
            assert O.pt_eq(got[j], want[j]), j
        ctx.msm_gens_many(list(coeffs))
        assert ctx.test_msm_route() == route
    finally:
        if lg == 20:
            ctx.derive_generators(1 << 16)


@gpu
def test_commit_evals_definition(env):
    """columns of a known polynomial p (E_i = p(omega^i) by the restatement at 2^10) commit to the oracle's pcdl_commit(p)"""
    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    lg, d = 10, (1 << 10) - 1
    ps = [O.random_scalars(1 << lg, 800), O.random_scalars(300, 801), np.zeros((0, 4), dtype=np.uint64)]
    E = np.stack([_limbs(ntt(_ints(p), lg)) for p in ps])
    ws = O.random_scalars(3, 802)
    got = pcdl.commit_evals(ctx, E, d, ws)
    for j, p in enumerate(ps):
        assert O.pt_eq(got[j], O.pcdl_commit(p, d, ws[j]))


def _rot_points(O, lg, seed):
    from halo_accumulation_b200 import domain_root

    w = _ints(domain_root(lg))[0] * MINV % R
    assert w == root(lg)
    z = _ints(O.random_scalars(1, seed))[0] * MINV % R
    return np.stack([_mont(z), _mont(z * w % R), _mont(z * pow(w, -1, R) % R)])


QUERIES = [(0, 0), (0, 1), (0, 2), (1, 0), (2, 1), (3, 2), (4, 0), (4, 2), (5, 1), (6, 0), (7, 2), (6, 1)]


def _same_opening(O, a, b):
    for x, y in zip(a[:6], b[:6]):
        x, y = np.asarray(x), np.asarray(y)
        if x.shape[-1] == 12:
            assert O.pt_eq(x, y)
        else:
            assert np.array_equal(x, y)
    pa, pb = a[6], b[6]  # the proof: points projectively
    assert pa.lg_n == pb.lg_n and pa.hiding == pb.hiding
    for i in range(pa.lg_n):
        assert O.pt_eq(np.array(pa.Ls[i]), np.array(pb.Ls[i])) and O.pt_eq(np.array(pa.Rs[i]), np.array(pb.Rs[i])), i
    assert O.pt_eq(np.array(pa.U), np.array(pb.U)) and list(pa.c) == list(pb.c)
    if pa.hiding:
        assert O.pt_eq(np.array(pa.C_bar), np.array(pb.C_bar)) and list(pa.w_prime) == list(pb.w_prime)


def _columns(O, lg, seed):
    """k = 8 columns: random, a zero column (degree 0), r - 1 everywhere (a constant), and random ones"""
    n = 1 << lg
    E = O.random_scalars(8 * n, seed).reshape(8, n, 4)
    E[2] = 0
    E[4] = O.to_mont([R - 1])[0]
    return E


@gpu
@pytest.mark.parametrize("lg", [10, 20])
@pytest.mark.parametrize("hiding", [False, True])
def test_open_multi_evals(env, lg, hiding):
    """open_multi_evals(E, q) = open_multi(intt(E), q[:max deg]) field by field (vs, Q, us, C, x, v, pi) at z, omega z and
    omega^-1 z with omega = domain_root(lg); k = 8, T = 3; 2^20 over FIXED-base tables.  The claim is accepted by check,
    check_batch and the accumulation scheme, on the GPU and in the oracle."""
    ctx, O, pcdl, acc = env["ctx"], env["O"], env["pcdl"], env["acc"]
    n, d = 1 << lg, (1 << lg) - 1
    if lg == 20:
        ctx.derive_generators(n)
        ctx.precompute_generators(0)
    try:
        E = _columns(O, lg, 900 + lg)
        coeffs = ctx.ntt(E, lg, inverse=True)
        zs = _rot_points(O, lg, 901)
        ws = O.random_scalars(8, 902) if hiding else None
        wQ, wb = (O.random_scalars(2, 903) if hiding else (None, None))
        q = O.random_scalars(d, 904) if hiding else None
        Cs = pcdl.commit_evals(ctx, E, d, ws)
        got = pcdl.open_multi_evals(ctx, E, Cs, d, zs, QUERIES, ws, wQ, q, wb)
        degs = [max([i for i, c in enumerate(_ints(p)) if c] or [0]) for p in coeffs] if lg <= 12 else None
        maxdeg = max(degs) if degs else d
        want = pcdl.open_multi(ctx, list(coeffs), Cs, d, zs, QUERIES, ws, wQ, None if q is None else q[:maxdeg], wb)
        _same_opening(O, got, want)
        vs, Q, us, Cm, x, v, pi = got
        pcdl.check(ctx, Cm, d, x, v, pi)
        if lg == 10:  # the oracle holds the first 2^16 generators
            assert O.pcdl_check(Cm, d, x, v, O.EvalProof.from_buffer_copy(bytes(pi))) == 0
            inst = acc.new_instance(Cm, d, x, v, pi)
            pcdl.check_batch(ctx, [inst, inst], O.random_scalars(1, 905)[0])
            a = acc.prover(ctx, d, [inst], O.random_scalars(2, 906), O.random_scalars(1, 907)[0], O.random_scalars(d, 908),
                           O.random_scalars(1, 909)[0])
            acc.verifier(ctx, d, [inst], a)
            acc.decider(ctx, a)
            oa = O.Accumulator.from_buffer_copy(bytes(a))
            assert O.acc_verifier(d, [O.Instance.from_buffer_copy(bytes(inst))], oa) == 0
            assert O.acc_decider(oa) == 0
    finally:
        if lg == 20:
            ctx.derive_generators(1 << 16)


@gpu
def test_open_multi_evals_errors(env):
    """q of the wrong length (before any device work) and hiding over columns of degree 0 (after the upload) are HALO_ELEN;
    nothing is written"""
    from halo_accumulation_b200 import _capi

    ctx, O, pcdl = env["ctx"], env["O"], env["pcdl"]
    lg, d = 4, 15
    E = np.zeros((2, 16, 4), dtype=np.uint64)
    E[:] = O.to_mont([3])[0]  # constant columns: degree 0
    Cs = pcdl.commit_evals(ctx, E, d)
    zs = O.random_scalars(1, 950)
    ws, wQ, wb = O.random_scalars(2, 951), O.random_scalars(1, 952)[0], O.random_scalars(1, 953)[0]
    for q in (O.random_scalars(d - 1, 954), O.random_scalars(d, 955)):
        with pytest.raises(_capi.HaloError) as e:
            pcdl.open_multi_evals(ctx, E, Cs, d, zs, [(0, 0), (1, 0)], ws, wQ, q, wb)
        assert e.value.code == HALO_ELEN
    with pytest.raises(_capi.HaloError) as e:
        pcdl.open_multi_evals(ctx, np.zeros((2, 12, 4), dtype=np.uint64), Cs, 11, zs, [(0, 0), (1, 0)])
    assert e.value.code == HALO_EINVAL
    with pytest.raises(_capi.HaloError) as e:
        pcdl.commit_evals(ctx, np.zeros((2, 12, 4), dtype=np.uint64), 11)
    assert e.value.code == HALO_EINVAL
