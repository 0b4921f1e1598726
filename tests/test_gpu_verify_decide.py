"""GPU tests of batch verify-and-decide (DESIGN.md K5d): halo_h_msm_batch_submit / _collect against the oracle's MSMs and
halo_h_msm_batch, and acc.verify_decide_batch against the oracle's single verifiers followed by its single deciders --
accept on honest input for every rho, and on a reject the same (position, code) as the first item the oracle rejects in the
order "steps, then decided accumulators"; malformed input anywhere is an error, not a decision."""
import ctypes as C

import numpy as np
import pytest

from oracle.oracle import R_MOD

pytestmark = pytest.mark.gpu

D = 1023
HALO_EINVAL, HALO_ESTATE = -1, -6


@pytest.fixture(scope="module")
def own_ctx(halo):
    """A context of its own: the tests switch "combine_min_outputs"."""
    try:
        import torch

        if not torch.cuda.is_available():
            pytest.skip("no CUDA device in this container")
    except ImportError:
        pytest.skip("no CUDA device in this container")
    c = halo.Context(0, 1 << 20)
    c.derive_generators(1 << 16)
    yield c
    c.close()


@pytest.fixture(scope="module")
def env(own_ctx, oracle):
    """own_ctx with the oracle holding the same parameters."""
    from halo_accumulation_b200 import acc, pcdl

    S, H = own_ctx.get_SH()
    oracle.set_params(S, H, own_ctx.get_generators(0, 1 << 16))
    return dict(ctx=own_ctx, O=oracle, pcdl=pcdl, acc=acc)


u64 = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint64))  # noqa: E731


def _submit(ctx, xis_list, weights):
    """(return code, ticket) of halo_h_msm_batch_submit."""
    lgs = np.array([x.shape[0] - 1 for x in xis_list] or [0], dtype=np.uint32)
    xis = np.ascontiguousarray(np.concatenate(xis_list) if xis_list else np.zeros((1, 4), dtype=np.uint64))
    w = np.ascontiguousarray(weights if len(xis_list) else np.zeros((1, 4)), dtype=np.uint64)
    t = C.c_int(-1)
    rc = ctx._lib.halo_h_msm_batch_submit(ctx._h, u64(xis), lgs.ctypes.data_as(C.POINTER(C.c_uint32)), u64(w), len(xis_list),
                                          C.byref(t))
    return rc, t.value


def _collect(ctx, ticket, bases=None, scalars=None, inf=None):
    """(return code, point) of halo_h_msm_batch_collect; bases / scalars None: no companion."""
    m = 0 if scalars is None else scalars.shape[0]
    b = np.zeros((1, 8), dtype=np.uint64) if bases is None else np.ascontiguousarray(bases)
    s = np.zeros((1, 4), dtype=np.uint64) if scalars is None else np.ascontiguousarray(scalars)
    infp = None if inf is None else np.ascontiguousarray(inf, dtype=np.uint8).ctypes.data_as(C.POINTER(C.c_uint8))
    out = np.zeros(12, dtype=np.uint64)
    rc = ctx._lib.halo_h_msm_batch_collect(ctx._h, ticket, u64(b), infp, u64(s), m, u64(out))
    return rc, out


def _one_call(ctx, xis_list, weights, bases=None, scalars=None, inf=None):
    """(return code, point) of halo_h_msm_batch."""
    lgs = np.array([x.shape[0] - 1 for x in xis_list] or [0], dtype=np.uint32)
    xis = np.ascontiguousarray(np.concatenate(xis_list) if xis_list else np.zeros((1, 4), dtype=np.uint64))
    w = np.ascontiguousarray(weights if len(xis_list) else np.zeros((1, 4)), dtype=np.uint64)
    m = 0 if scalars is None else scalars.shape[0]
    b = np.zeros((1, 8), dtype=np.uint64) if bases is None else np.ascontiguousarray(bases)
    s = np.zeros((1, 4), dtype=np.uint64) if scalars is None else np.ascontiguousarray(scalars)
    infp = None if inf is None else np.ascontiguousarray(inf, dtype=np.uint8).ctypes.data_as(C.POINTER(C.c_uint8))
    out = np.zeros(12, dtype=np.uint64)
    rc = ctx._lib.halo_h_msm_batch(ctx._h, u64(xis), lgs.ctypes.data_as(C.POINTER(C.c_uint32)), u64(w), len(xis_list), u64(b),
                                   infp, u64(s), m, u64(out))
    return rc, out


def _split(ctx, xis_list, weights, bases=None, scalars=None, inf=None):
    rc, t = _submit(ctx, xis_list, weights)
    assert rc == 0
    return _collect(ctx, t, bases, scalars, inf)


def test_submit_collect_matches_oracle_and_one_call(env):
    """Mixed lg n_j from 1 to 16 with weights 0 and 1 among them, with no companion and with one of more than 4096 points
    (infinity flags among them): the oracle's sum, and the point halo_h_msm_batch returns."""
    ctx, O = env["ctx"], env["O"]
    gs = ctx.get_generators(0, 1 << 16)
    lgs = [1 + (5 * j) % 16 for j in range(12)]
    xis = [O.random_scalars(lg + 1, 7000 + j) for j, lg in enumerate(lgs)]
    w = O.random_scalars(len(xis), 6999)
    w[0] = O.to_mont([1])[0]
    w[4] = 0
    ref = O.pt_from_affine_ints(None)
    for j, x in enumerate(xis):
        ref = O.pt_add(ref, O.pt_mul(O.msm_affine(gs, O.h_get_poly(x), threads=8), w[j]))
    bases = ctx.get_generators(300, 5000).copy()
    sc = O.random_scalars(5000, 6998)
    inf = np.zeros(5000, dtype=np.uint8)
    inf[[0, 2048, 4999]] = 1
    companion = O.msm_affine(bases, sc, threads=8, inf=inf)
    for args, want in (((), ref), ((bases, sc, inf), O.pt_add(ref, companion))):
        rc, got = _split(ctx, xis, w, *args)
        assert rc == 0 and O.pt_eq(got, want)
        rc, one = _one_call(ctx, xis, w, *args)
        assert rc == 0 and O.pt_eq(one, got)
    rc, got = _split(ctx, [], [], bases, sc, inf)  # companion alone
    assert rc == 0 and O.pt_eq(got, companion)
    rc, got = _split(ctx, [], [])  # nothing at all: infinity
    assert rc == 0 and O.pt_to_affine(got)[1]


def test_submit_collect_fixed_and_variable_base(halo, oracle):
    """At 2^17 generators with the FIXED-base tables (the generator part takes them from 2^17 points on) and without: the
    same point, which is also the sum of halo_h_msm over the claims plus the oracle's companion."""
    O = oracle
    c = halo.Context(0, 1 << 17)
    try:
        c.derive_generators(1 << 17)
        c.precompute_generators(0)
        xis = [O.random_scalars(lg + 1, 7100 + lg) for lg in (17, 12, 17)]
        one = O.to_mont([1] * len(xis))
        ref = O.pt_from_affine_ints(None)
        for x in xis:
            h = np.zeros(12, dtype=np.uint64)
            c._chk(c._lib.halo_h_msm(c._h, u64(x), x.shape[0] - 1, u64(h)))
            ref = O.pt_add(ref, h)
        bases, sc = c.get_generators(1000, 4500).copy(), O.random_scalars(4500, 7200)
        ref_c = O.pt_add(ref, O.msm_affine(bases, sc, threads=8))
        for fixed in (True, False):
            c.set_fixed_base(fixed)
            rc, got = _split(c, xis, one, bases, sc)
            assert rc == 0 and O.pt_eq(got, ref_c), fixed
            rc, got = _split(c, xis, one)
            assert rc == 0 and O.pt_eq(got, ref), fixed
    finally:
        c.close()


def test_submit_collect_out_of_order(env):
    """A collect without a submit and a second submit are HALO_ESTATE; a wrong ticket is HALO_EINVAL and leaves the batch
    outstanding; collecting with m = 0 drains it; the context works afterwards."""
    ctx, O = env["ctx"], env["O"]
    xis = [O.random_scalars(11, 7300), O.random_scalars(7, 7301)]
    w = O.random_scalars(2, 7302)
    rc, want = _one_call(ctx, xis, w)
    assert rc == 0
    assert _collect(ctx, 0)[0] == HALO_ESTATE
    rc, t = _submit(ctx, xis, w)
    assert rc == 0
    assert _submit(ctx, xis, w)[0] == HALO_ESTATE
    assert _one_call(ctx, xis, w)[0] == HALO_ESTATE  # halo_h_msm_batch is a submit as well
    assert _collect(ctx, t + 1)[0] == HALO_EINVAL
    rc, got = _collect(ctx, t)  # the drain of a caller that gives up
    assert rc == 0 and O.pt_eq(got, want)
    assert _collect(ctx, t)[0] == HALO_ESTATE
    rc, got = _split(ctx, xis, w)
    assert rc == 0 and O.pt_eq(got, want)
    assert _submit(ctx, [O.random_scalars(18, 7303)], w[:1])[0] < 0  # lg 17: above the resident generators
    rc, got = _one_call(ctx, xis, w)  # a refused submit leaves nothing outstanding
    assert rc == 0 and O.pt_eq(got, want)


def _claim(env, d, seed, hiding):
    """An honest instance (C, d, z, v, pi) opened on the GPU, hiding or not."""
    ctx, O, pcdl, acc = env["ctx"], env["O"], env["pcdl"], env["acc"]
    n = d + 1
    p = O.random_scalars(max(2, n - n // 3), seed)
    z = O.random_scalars(1, seed + 1)[0]
    w, wb = O.random_scalars(2, seed + 2) if hiding else (None, None)
    q = O.random_scalars(p.shape[0] - 1, seed + 3) if hiding else None
    Cm = pcdl.commit(ctx, p, d, w)
    v = O.scalar_dot(p, O.construct_powers(z, p.shape[0]))
    return acc.new_instance(Cm, d, z, v, pcdl.open(ctx, p, Cm, d, z, w, q, wb))


def _chain(env, d, steps, seed):
    """(qs, acc) of a short IVC chain (acc.rs:298-315 shape): the first step has m = 1, later ones m = 2 (the previous
    accumulator and a new instance, hiding or not)."""
    ctx, O, acc = env["ctx"], env["O"], env["acc"]
    n, a, out = d + 1, None, []
    for s in range(steps):
        q = _claim(env, d, seed + 100 * s, s % 2 == 0)
        qs = [acc.to_instance(a), q] if a is not None else [q]
        h0, (w, wb), qq = O.random_scalars(2, seed + 100 * s + 50), O.random_scalars(2, seed + 100 * s + 60), \
            O.random_scalars(n - 1, seed + 100 * s + 70)
        a = acc.prover(ctx, d, qs, h0, w, qq, wb)
        out.append((qs, a))
    return out


@pytest.fixture(scope="module")
def steps(env):
    return _chain(env, D, 4, 31000) + _chain(env, D, 3, 32000)


@pytest.fixture(scope="module")
def decided(env):
    """Accumulators of other chains, of several degree bounds."""
    return [a for _, a in _chain(env, 255, 3, 33000) + _chain(env, D, 2, 34000) + _chain(env, 63, 2, 35000)]


@pytest.fixture(scope="module")
def other_d(env):
    return _chain(env, 255, 1, 36000)


def _rhos(O):
    return [O.random_scalars(1, 421)[0], O.to_mont([1])[0], O.to_mont([R_MOD - 1])[0]]


def _copy(x):
    return type(x).from_buffer_copy(bytes(x))


def _oracle_first_reject(O, d, steps, accs):
    """The oracle's single verifiers over the steps, then its single deciders over accs: (position, code) of the first reject."""
    for i, (qs, a) in enumerate(steps):
        rc = O.acc_verifier(d, [O.Instance.from_buffer_copy(bytes(q)) for q in qs], O.Accumulator.from_buffer_copy(bytes(a)),
                            threads=8)
        if rc != 0:
            return i, rc
    for j, a in enumerate(accs):
        rc = O.acc_decider(O.Accumulator.from_buffer_copy(bytes(a)), threads=8)
        if rc != 0:
            return len(steps) + j, rc
    return None


def _same_decision(env, steps, accs, rho, expected, d=D):
    acc = env["acc"]
    if expected is None:
        acc.verify_decide_batch(env["ctx"], d, steps, accs, rho)
        return
    with pytest.raises(acc.Rejected) as e:
        acc.verify_decide_batch(env["ctx"], d, steps, accs, rho)
    assert (e.value.index, e.value.code) == expected


@pytest.mark.parametrize("min_outputs", [0, -1])
def test_accepts_honest_input(env, steps, decided, min_outputs):
    """(k, k_dec) in {(0, 0), (0, 3), (5, 0), (1, 1), (64, 1), (64, 64)} (the 64 are copies of the 7 steps and 7 accumulators),
    for several rho; C' / C* on the device (threshold 0) and on the host (threshold -1: never)."""
    O, ctx = env["O"], env["ctx"]
    assert _oracle_first_reject(O, D, steps, decided) is None
    ctx.set_tuning("combine_min_outputs", min_outputs)
    many_steps = [steps[i % len(steps)] for i in range(64)]
    many_accs = [decided[i % len(decided)] for i in range(64)]
    for k, k_dec in ((0, 0), (0, 3), (5, 0), (1, 1), (64, 1), (64, 64)):
        for rho in _rhos(O):
            _same_decision(env, many_steps[:k], many_accs[:k_dec], rho, None)


def _corrupt_step(steps, other_d, kind, pos):
    """steps with step `pos` corrupted by `kind` (the kinds of test_gpu_batch_verifier.py)."""
    out = list(steps)
    qs, a = steps[pos]
    a = _copy(a)
    qs = [_copy(q) for q in qs]
    if kind == "v":
        a.v[0] ^= 1
    elif kind == "h0":
        a.h0[0][0] ^= 1
    elif kind == "z":
        a.z[0] ^= 1
    elif kind == "C_bar":
        a.C_bar = steps[(pos + 1) % len(steps)][1].C_bar
    elif kind == "U0":
        a.U0 = steps[(pos + 1) % len(steps)][1].U0
    elif kind == "omega":
        a.w[0] ^= 1
    elif kind == "d":
        a.d = 255
    elif kind == "pi_c":
        qs[-1].pi.c[0] ^= 1
    elif kind == "other_d":
        qs[-1] = other_d[0][0][0]  # an honest instance of d = 255
    out[pos] = (qs, a)
    return out


def _corrupt_acc(accs, kind, pos):
    """accs with the claim of accumulator `pos` corrupted: its proof's c or U, or v."""
    out = list(accs)
    a = _copy(accs[pos])
    if kind == "pi_c":
        a.pi.c[0] ^= 1
    elif kind == "v":
        a.v[0] ^= 1
    elif kind == "pi_U":
        a.pi.U = accs[(pos + 1) % len(accs)].pi.U  # a valid point, not this proof's
    out[pos] = a
    return out


@pytest.mark.parametrize("kind", ["v", "h0", "z", "C_bar", "omega", "U0", "d", "pi_c", "other_d"])
def test_step_reject_equals_first_single_reject(env, steps, decided, other_d, kind):
    """One corrupted step at the first, a middle and the last position, honest accumulators behind: (index, code) of the
    oracle's single verifiers then deciders, with C' / C* on the device and on the host."""
    O, ctx = env["O"], env["ctx"]
    for pos in (0, 3, 6):
        bad = _corrupt_step(steps, other_d, kind, pos)
        expected = _oracle_first_reject(O, D, bad, decided)
        assert expected is not None and expected[0] == pos
        for min_outputs in (0, -1):
            ctx.set_tuning("combine_min_outputs", min_outputs)
            _same_decision(env, bad, decided, _rhos(O)[0], expected)


@pytest.mark.parametrize("kind", ["pi_c", "v", "pi_U"])
def test_decided_reject_equals_first_single_reject(env, steps, decided, kind):
    """One corrupted decided accumulator at the first, a middle and the last position behind honest steps: index k + j."""
    O, ctx = env["O"], env["ctx"]
    for pos in (0, 3, len(decided) - 1):
        bad = _corrupt_acc(decided, kind, pos)
        expected = _oracle_first_reject(O, D, steps, bad)
        assert expected == (len(steps) + pos, expected[1]) and expected[1] in (-10, -11)
        for min_outputs in (0, -1):
            ctx.set_tuning("combine_min_outputs", min_outputs)
            _same_decision(env, steps, bad, _rhos(O)[0], expected)
    ctx.set_tuning("combine_min_outputs", 0)
    _same_decision(env, [], _corrupt_acc(decided, kind, 2), _rhos(O)[1], (2, expected[1]))  # no steps: the decider's index


def test_earlier_reject_wins_across_the_boundary(env, steps, decided, other_d):
    O, ctx = env["O"], env["ctx"]
    ctx.set_tuning("combine_min_outputs", 0)
    bad_steps = _corrupt_step(steps, other_d, "pi_c", 5)
    bad_accs = _corrupt_acc(decided, "v", 0)
    assert _oracle_first_reject(O, D, bad_steps, bad_accs) == (5, -10)
    _same_decision(env, bad_steps, bad_accs, _rhos(O)[1], (5, -10))
    bad_accs = _corrupt_acc(_corrupt_acc(decided, "pi_U", 1), "v", 4)
    expected = _oracle_first_reject(O, D, steps, bad_accs)
    assert expected[0] == len(steps) + 1
    _same_decision(env, steps, bad_accs, _rhos(O)[1], expected)


def test_malformed_input_is_an_error_wherever_it_sits(env, steps, decided):
    from halo_accumulation_b200 import HaloError

    O, ctx, acc = env["O"], env["ctx"], env["acc"]
    ctx.set_tuning("combine_min_outputs", 0)
    rho = _rhos(O)[0]
    rejecting_step = _corrupt_step(steps, None, "v", 0)[0]
    rejecting_acc = _corrupt_acc(decided, "v", 0)[0]

    def refused(st, accs, r=rho, d=D):
        with pytest.raises(HaloError) as e:
            acc.verify_decide_batch(ctx, d, st, accs, r)
        assert e.value.code == HALO_EINVAL, e.value.code

    def wrong_lg(pi_owner):
        pi_owner.pi.lg_n -= 1

    def off_curve(pi_owner):
        pi_owner.pi.Ls[2][5] ^= 4

    def not_canonical(pi_owner):
        pi_owner.pi.c[3] = 0x7FFFFFFFFFFFFFFF

    def not_pow2(pi_owner):
        pi_owner.d = 62

    def bad_step(step, fn):
        qs, a = step
        qs = [_copy(q) for q in qs]
        fn(qs[-1])
        return qs, a

    def bad_acc(a, fn):
        a = _copy(a)
        fn(a)
        return a

    for fn in (wrong_lg, off_curve, not_canonical, not_pow2):
        for pos in range(len(steps)):
            st = list(steps)
            st[pos] = bad_step(st[pos], fn)
            refused(st, decided)
        for pos in range(len(decided)):
            accs = list(decided)
            accs[pos] = bad_acc(accs[pos], fn)
            refused(steps, accs)
            refused([], accs)
        # an error even behind an item that would be rejected, within a list and across the boundary
        refused([rejecting_step], [bad_acc(decided[1], fn)])
        refused([], [rejecting_acc, bad_acc(decided[1], fn)])
    refused(steps[:3], decided[:2], d=1022)  # D + 1 not a power of two
    refused(steps[:3], decided[:2], r=np.zeros(4, dtype=np.uint64))  # rho = 0
    refused([], decided[:2], r=np.zeros(4, dtype=np.uint64))
    refused(steps[:3], decided[:2], r=np.array([R_MOD & (2**64 - 1), (R_MOD >> 64) & (2**64 - 1), (R_MOD >> 128) & (2**64 - 1),
                                                  R_MOD >> 192], dtype=np.uint64))  # rho = r: not canonical
    acc.verify_decide_batch(ctx, D, steps, decided, rho)  # the context still decides


def test_chain_verified_and_decided_in_one_call(env, steps):
    """The fast path of a chain: every step verified and the last accumulator decided (it is also the last step's
    accumulator), against verifier_batch followed by decider; then a corrupted last accumulator, which both reject at the
    last step."""
    O, ctx, acc = env["O"], env["ctx"], env["acc"]
    chain = steps[:4]
    ctx.set_tuning("combine_min_outputs", -1)
    for rho in _rhos(O)[:2]:
        acc.verifier_batch(ctx, D, chain, rho)
        acc.decider(ctx, chain[-1][1])
        acc.verify_decide_batch(ctx, D, chain, [chain[-1][1]], rho)
    bad = _corrupt_step(chain, None, "z", 3)
    with pytest.raises(acc.Rejected) as e1:
        acc.verifier_batch(ctx, D, bad, _rhos(O)[0])
    with pytest.raises(acc.Rejected) as e2:
        acc.verify_decide_batch(ctx, D, bad, [bad[-1][1]], _rhos(O)[0])
    assert (e2.value.index, e2.value.code) == (e1.value.index, e1.value.code) == (3, -15)
