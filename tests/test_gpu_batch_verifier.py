"""GPU tests of the batch verifier (DESIGN.md K5c): k_point_combine (halo_test_point_combine) against the oracle's group
law, and acc.verifier_batch against a loop of the oracle's single verifiers -- accept on honest steps for every rho, and on
a reject the same (step index, code) as the first step the oracle rejects in order; malformed input is an error, not a
decision.  Also pcdl.check_batch with its C' computed on the device."""
import ctypes as C

import numpy as np
import pytest

from oracle.oracle import R_MOD

pytestmark = pytest.mark.gpu

D = 1023


@pytest.fixture(scope="session")
def own_ctx(halo):
    """A context of its own: the tests switch "combine_min_outputs".  Session scoped and set up ahead of the session context
    when this file runs alone, so it is closed after the session context's end-of-run canary check, which then covers the
    buffers of k_point_combine as well."""
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
def env(own_ctx, ctx, oracle):
    """own_ctx with the oracle holding the same parameters."""
    from halo_accumulation_b200 import acc, pcdl

    S, H = own_ctx.get_SH()
    oracle.set_params(S, H, own_ctx.get_generators(0, 1 << 16))
    return dict(ctx=own_ctx, O=oracle, pcdl=pcdl, acc=acc, S=S)


def _combine(ctx, path, P, Q, a, b):
    """(return code, [n, 8] affine) of halo_test_point_combine."""
    n = P.shape[0]
    out = np.zeros((max(n, 1), 8), dtype=np.uint64)
    u64 = lambda x: np.ascontiguousarray(x, dtype=np.uint64).ctypes.data_as(C.POINTER(C.c_uint64))  # noqa: E731
    keep = [np.ascontiguousarray(x, dtype=np.uint64) for x in (P, Q, a, b)]
    rc = ctx._lib.halo_test_point_combine(ctx._h, path, *(u64(x) for x in keep), n, u64(out))
    return rc, out[:n]


def _ref(O, S, P, Q, a, b):
    r = O.pt_add(O.pt_add(P, O.pt_mul(Q, a)), O.pt_mul(S, b))
    aff, inf = O.pt_to_affine(r)
    return np.zeros(8, dtype=np.uint64) if inf else aff


def test_point_combine_matches_oracle(env):
    """Scalars 0, 1, r - 1 and random; P and Q at infinity; Q = S; P = -a Q (result O); P equal to the running sum (the final
    addition doubles); N = 1, 7 and 4100.  Device and host paths return the same affine bytes."""
    ctx, O, S = env["ctx"], env["O"], env["S"]
    inf = O.pt_from_affine_ints(None)
    gens = O.affine_to_jac(ctx.get_generators(100, 64))
    one, minus1, zero = O.to_mont([1])[0], O.to_mont([R_MOD - 1])[0], np.zeros(4, dtype=np.uint64)
    rnd = O.random_scalars(64, 901)
    cases = [
        (gens[0], gens[1], rnd[0], rnd[1]),
        (gens[2], gens[3], zero, zero),
        (gens[4], gens[5], one, minus1),
        (gens[6], gens[7], minus1, one),
        (inf, gens[8], rnd[2], rnd[3]),
        (gens[9], inf, rnd[4], rnd[5]),
        (inf, inf, rnd[6], zero),
        (gens[10], S, rnd[7], rnd[7]),  # Q = S, equal scalars: every joint step adds the same point twice
        (gens[11], S, rnd[8], O.to_mont([R_MOD - O.from_mont(rnd[8:9])[0]])[0]),  # Q = S, b = -a
        (O.pt_mul(gens[12], O.to_mont([R_MOD - O.from_mont(rnd[9:10])[0]])[0]), gens[12], rnd[9], zero),  # P = -a Q: O
    ]
    s_part = O.pt_add(O.pt_mul(gens[13], rnd[10]), O.pt_mul(S, rnd[11]))
    cases.append((s_part, gens[13], rnd[10], rnd[11]))  # P = a Q + b S: the last addition is a doubling
    P = np.array([np.asarray(c[0], dtype=np.uint64) for c in cases])
    Q = np.array([np.asarray(c[1], dtype=np.uint64) for c in cases])
    a = np.array([c[2] for c in cases], dtype=np.uint64)
    b = np.array([c[3] for c in cases], dtype=np.uint64)
    ref = np.array([_ref(O, S, P[o], Q[o], a[o], b[o]) for o in range(len(cases))])
    assert not ref[9].any()  # the P = -a Q case is O
    for n in (1, 7, len(cases)):
        for path in (0, 1, -1):
            rc, got = _combine(ctx, path, P[:n], Q[:n], a[:n], b[:n])
            assert rc == 0 and np.array_equal(got, ref[:n]), (n, path)
    # 4100 random outputs (more than one block of every kernel; infinity among them)
    n = 4100
    Pn = O.affine_to_jac(ctx.get_generators(2000, n))
    Qn = O.affine_to_jac(ctx.get_generators(9000, n))
    Qn[[5, 777]] = inf
    an, bn = O.random_scalars(n, 902), O.random_scalars(n, 903)
    an[3] = 0
    rc_d, dev = _combine(ctx, 1, Pn, Qn, an, bn)
    rc_h, host = _combine(ctx, 0, Pn, Qn, an, bn)
    assert rc_d == 0 and rc_h == 0 and np.array_equal(dev, host)
    for o in (0, 3, 5, 777, 2048, n - 1):
        assert np.array_equal(dev[o], _ref(O, S, Pn[o], Qn[o], an[o], bn[o])), o
    assert _combine(ctx, 2, Pn[:1], Qn[:1], an[:1], bn[:1])[0] == -1  # unknown path
    assert _combine(ctx, 1, Pn[:0], Qn[:0], an[:0], bn[:0])[0] == 0  # n = 0


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
    return _chain(env, D, 4, 21000) + _chain(env, D, 3, 22000)


@pytest.fixture(scope="module")
def other_d(env):
    return _chain(env, 255, 2, 23000)


def _rhos(O):
    return [O.random_scalars(1, 321)[0], O.to_mont([1])[0], O.to_mont([R_MOD - 1])[0]]


def _copy(x):
    return type(x).from_buffer_copy(bytes(x))


def _oracle_first_reject(O, d, steps):
    for i, (qs, a) in enumerate(steps):
        rc = O.acc_verifier(d, [O.Instance.from_buffer_copy(bytes(q)) for q in qs], O.Accumulator.from_buffer_copy(bytes(a)),
                            threads=8)
        if rc != 0:
            return i, rc
    return None


def _same_decision(env, steps, rho, expected, d=D):
    acc = env["acc"]
    if expected is None:
        acc.verifier_batch(env["ctx"], d, steps, rho)
        return
    with pytest.raises(acc.Rejected) as e:
        acc.verifier_batch(env["ctx"], d, steps, rho)
    assert (e.value.index, e.value.code) == expected


@pytest.mark.parametrize("min_outputs", [0, -1])
def test_verifier_batch_accepts_honest_steps(env, steps, other_d, min_outputs):
    """k = 0, 1, 7 at D = 1023 and 2 at D = 255, for several rho; C' / C* on the device (threshold 0) and on the host
    (threshold -1: never)."""
    O, ctx, acc = env["O"], env["ctx"], env["acc"]
    assert _oracle_first_reject(O, D, steps) is None and _oracle_first_reject(O, 255, other_d) is None
    ctx.set_tuning("combine_min_outputs", min_outputs)
    for k in (0, 1, 7):
        for rho in _rhos(O):
            acc.verifier_batch(ctx, D, steps[:k], rho)
    acc.verifier_batch(ctx, 255, other_d, _rhos(O)[0])


def test_verifier_batch_200_steps_msm_past_4096_points(env, steps):
    """200 steps (copies of the 7) bring about 48 points each: one MSM of more than 4096 points; a reject deep inside."""
    O, ctx, acc = env["O"], env["ctx"], env["acc"]
    ctx.set_tuning("combine_min_outputs", 0)
    many = [steps[i % len(steps)] for i in range(200)]
    assert sum(len(qs) * (2 * 10 + 3) + 2 for qs, _ in many) > 4096
    for rho in _rhos(O)[:2]:
        acc.verifier_batch(ctx, D, many, rho)
    qs, a = steps[3]
    bad = _copy(a)
    bad.v[0] ^= 1
    _same_decision(env, many[:150] + [(qs, bad)] + many[150:], _rhos(O)[0], (150, -17))


def _corrupt(env, steps, other_d, kind, pos):
    """steps with step `pos` corrupted by `kind`."""
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
        a.C_bar = steps[(pos + 1) % len(steps)][1].C_bar  # a valid point, not this step's
    elif kind == "U0":  # C* and alpha stay as they were: only the combined A_i / B_i terms can reject it
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


@pytest.mark.parametrize("kind", ["v", "h0", "z", "C_bar", "omega", "U0", "d", "pi_c", "other_d"])
def test_verifier_batch_reject_equals_first_single_reject(env, steps, other_d, kind):
    """One corrupted step at the first, middle and last position: (index, code) of the first step the oracle's single
    verifier rejects, in order -- with C' / C* on the device and on the host."""
    O, ctx = env["O"], env["ctx"]
    codes = {"v": -17, "h0": -12, "z": -15, "C_bar": -14, "U0": -12, "d": -13, "pi_c": -10, "other_d": -13}
    for pos in (0, 3, 6):
        bad = _corrupt(env, steps, other_d, kind, pos)
        expected = _oracle_first_reject(O, D, bad)
        assert expected is not None and expected[0] == pos
        if kind in codes:
            assert expected[1] == codes[kind]
        for min_outputs in (0, -1):
            ctx.set_tuning("combine_min_outputs", min_outputs)
            _same_decision(env, bad, _rhos(O)[0], expected)


def test_verifier_batch_earlier_reject_wins(env, steps, other_d):
    O, ctx = env["O"], env["ctx"]
    ctx.set_tuning("combine_min_outputs", 0)
    bad = _corrupt(env, _corrupt(env, steps, other_d, "v", 1), other_d, "pi_c", 4)
    assert _oracle_first_reject(O, D, bad) == (1, -17)
    _same_decision(env, bad, _rhos(O)[1], (1, -17))
    bad = _corrupt(env, _corrupt(env, steps, other_d, "pi_c", 1), other_d, "v", 4)
    assert _oracle_first_reject(O, D, bad) == (1, -10)
    _same_decision(env, bad, _rhos(O)[1], (1, -10))


def test_verifier_batch_malformed_input_is_an_error_wherever_it_sits(env, steps):
    from halo_accumulation_b200 import HaloError

    O, ctx, acc = env["O"], env["ctx"], env["acc"]
    ctx.set_tuning("combine_min_outputs", 0)
    rho = _rhos(O)[0]
    rejecting = _corrupt(env, steps, None, "v", 0)[0]

    def refused(st, r=rho, d=D):
        with pytest.raises(HaloError) as e:
            acc.verifier_batch(ctx, d, st, r)
        assert e.value.code == -1, e.value.code

    def with_bad_instance(step, fn):
        qs, a = step
        qs = [_copy(q) for q in qs]
        fn(qs[-1])
        return qs, a

    def wrong_lg(q):
        q.pi.lg_n -= 1

    def off_curve(q):
        q.pi.Ls[2][5] ^= 4

    def not_canonical(q):
        q.pi.c[3] = 0x7FFFFFFFFFFFFFFF

    def not_pow2(q):
        q.d = 62

    for fn in (wrong_lg, off_curve, not_canonical, not_pow2):
        for pos in (0, 3, 6):
            st = list(steps)
            st[pos] = with_bad_instance(st[pos], fn)
            refused(st)
        refused([rejecting, with_bad_instance(steps[2], fn)])  # an error even behind a step that would be rejected
    refused(steps[:3], d=1022)  # D + 1 not a power of two
    refused(steps[:3], r=np.zeros(4, dtype=np.uint64))  # rho = 0
    acc.verifier_batch(ctx, D, steps, rho)  # the context still verifies


def test_verifier_batch_then_decider_batch(env, steps):
    """The fast path of many accumulators: verifier_batch over the steps, decider_batch over their accumulators."""
    O, ctx, acc = env["O"], env["ctx"], env["acc"]
    ctx.set_tuning("combine_min_outputs", 0)
    acc.verifier_batch(ctx, D, steps, _rhos(O)[0])
    acc.decider_batch(ctx, [a for _, a in steps], _rhos(O)[0])


@pytest.fixture(scope="module")
def pool(env):
    ds = [63, 1023, 15, 255, 1, 4095, 511, 3, 1023, 127]
    return [_claim(env, ds[j % len(ds)], 27000 + 10 * j, j % 2 == 1) for j in range(40)]


def _oracle_first_check_reject(O, claims):
    for j, q in enumerate(claims):
        rc = O.pcdl_check(np.array(q.C), q.d, np.array(q.z), np.array(q.v), O.EvalProof.from_buffer_copy(bytes(q.pi)), threads=8)
        if rc != 0:
            return j, rc
    return None


@pytest.mark.parametrize("min_outputs", [0, -1])
def test_check_batch_with_device_c_prime(env, pool, min_outputs):
    """pcdl.check_batch with C' of its hiding claims from k_point_combine (threshold 0) and from the host (-1): the same
    decisions as the oracle's single checks."""
    O, ctx, pcdl = env["O"], env["ctx"], env["pcdl"]
    ctx.set_tuning("combine_min_outputs", min_outputs)
    assert _oracle_first_check_reject(O, pool) is None
    for k in (1, 2, 40):
        for rho in _rhos(O):
            pcdl.check_batch(ctx, pool[:k], rho)
    for field, pos in (("v", 1), ("z", 20), ("v", 39)):
        claims = list(pool)
        claims[pos] = _copy(pool[pos])
        getattr(claims[pos], field)[0] ^= 1
        expected = _oracle_first_check_reject(O, claims)
        assert expected is not None and expected[0] == pos
        with pytest.raises(pcdl.Rejected) as e:
            pcdl.check_batch(ctx, claims, _rhos(O)[0])
        assert (e.value.index, e.value.code) == expected
