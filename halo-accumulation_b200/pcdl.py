"""Mirror of code/src/pcdl.rs: commit / open / succinct_check / check and HPoly."""
import ctypes as C

import numpy as np

from . import _host
from ._capi import arr, p64, pack
from ._host import EvalProof, Instance, Rejected  # noqa: F401


class HPoly:
    """pcdl.rs:44-92"""

    def __init__(self, xis):
        self.xis = arr(xis).reshape(-1, 4)

    def get_poly(self, ctx):
        lg_n = self.xis.shape[0] - 1
        out = np.zeros((1 << lg_n, 4), dtype=np.uint64)
        ctx._chk(ctx._lib.halo_h_expand(ctx._h, p64(self.xis), lg_n, p64(out)))
        return out

    def eval(self, z):
        z = arr(z, (4,))
        out = np.zeros(4, dtype=np.uint64)
        _host.chk(_host.lib().halo_h_eval(p64(self.xis), self.xis.shape[0] - 1, p64(z), p64(out)))
        return out


def commit(ctx, p, d, w=None):
    """pcdl.rs:99-110"""
    p = arr(p).reshape(-1, 4)
    out = np.zeros(12, dtype=np.uint64)
    wk, wp = _host.opt(w)
    _host.chk(_host.lib().halo_pcdl_commit(ctx._h, p64(p), C.c_uint64(p.shape[0]), C.c_uint64(d), wp, p64(out)))
    return out


def commit_batch(ctx, ps, d, ws=None):
    """`commit` of every polynomial in `ps` (ws: one blinding scalar per polynomial, or None) -> (k, 12) array.  Raises on the
    first malformed polynomial, before any device work, as a loop of `commit` calls would."""
    if len(ps) == 1:  # the single call, exactly (as pcdl::commit_batch does for k = 1)
        return commit(ctx, ps[0], d, None if ws is None else arr(ws).reshape(1, 4)[0])[None]
    packed, lens = pack(ps)
    k = len(lens)
    wa = arr(ws).reshape(k, 4) if ws is not None else None
    out = np.zeros((max(1, k), 12), dtype=np.uint64)
    _host.chk(_host.lib().halo_pcdl_commit_batch(ctx._h, p64(packed), p64(lens), C.c_uint64(k), C.c_uint64(d),
                                                 p64(wa) if wa is not None else None, p64(out)))
    return out[:k]


def open(ctx, p, Cm, d, z, w=None, q=None, w_bar=None):
    """pcdl.rs:120-242.  The reference's rng draws are explicit: q (deg p coefficients) and w_bar when hiding."""
    p, Cm, z = arr(p).reshape(-1, 4), arr(Cm, (12,)), arr(z, (4,))
    pi = EvalProof()
    wk, wp = _host.opt(w)
    wbk, wbp = _host.opt(w_bar)
    qa = arr(q).reshape(-1, 4) if q is not None else None
    _host.chk(_host.lib().halo_pcdl_open(ctx._h, p64(p), C.c_uint64(p.shape[0]), p64(Cm), C.c_uint64(d), p64(z), wp,
                                         p64(qa) if qa is not None else None, C.c_uint64(qa.shape[0] if qa is not None else 0),
                                         wbp, C.byref(pi)))
    return pi


def open_batch(ctx, ps, Cs, d, z, ws=None, q=None, w_bar=None):
    """Opens the polynomials `ps` (commitments Cs, one degree bound d) at one point z with ONE proof (include/halo_pcdl.h
    halo_pcdl_open_batch; the reference has none) -> (vs, C, v, pi): vs[j] = p_j(z), and (C, d, z, v, pi) is an ordinary
    claim for `check`, `check_batch` or acc.new_instance.  Hiding with ws (one w_j per polynomial): q holds
    max_j deg(p_j) coefficients.  With one polynomial this is `open`, bit for bit."""
    packed, lens = pack(ps)
    k = len(lens)
    Cs, z = arr(Cs).reshape(k, 12), arr(z, (4,))
    wa = arr(ws).reshape(k, 4) if ws is not None else None
    qa = arr(q).reshape(-1, 4) if q is not None else None
    wbk, wbp = _host.opt(w_bar)
    vs = np.zeros((max(1, k), 4), dtype=np.uint64)
    Cm, v, pi = np.zeros(12, dtype=np.uint64), np.zeros(4, dtype=np.uint64), EvalProof()
    _host.chk(_host.lib().halo_pcdl_open_batch(ctx._h, p64(packed), p64(lens), C.c_uint64(k), p64(Cs), C.c_uint64(d), p64(z),
                                               p64(wa) if wa is not None else None, p64(qa) if qa is not None else None,
                                               C.c_uint64(qa.shape[0] if qa is not None else 0), wbp, p64(vs), p64(Cm), p64(v),
                                               C.byref(pi)))
    return vs[:k], Cm, v, pi


def batch_claim(ctx, Cs, z, vs):
    """The verifier's reduction of the claims (C_j, z, vs[j]) of `open_batch` to its one claim -> (C, v)."""
    Cs, z = arr(Cs).reshape(-1, 12), arr(z, (4,))
    vs = arr(vs).reshape(Cs.shape[0], 4)
    Cm, v = np.zeros(12, dtype=np.uint64), np.zeros(4, dtype=np.uint64)
    _host.chk(_host.lib().halo_pcdl_batch_claim(ctx._h, p64(Cs), p64(vs), C.c_uint64(Cs.shape[0]), p64(z), p64(Cm), p64(v)))
    return Cm, v


def _queries(queries):
    q = np.ascontiguousarray(queries, dtype=np.uint64).reshape(-1, 2)
    return np.ascontiguousarray(q[:, 0]), np.ascontiguousarray(q[:, 1])


def open_multi(ctx, ps, Cs, d, zs, queries, ws=None, w_Q=None, q=None, w_bar=None):
    """Opens the polynomials `ps` (commitments Cs, one degree bound d) at several points with ONE proof (include/halo_pcdl.h
    halo_pcdl_open_multi; the reference has none).  queries: (j, t) pairs, polynomial j at point zs[t] -> (vs, Q, us, C, x, v,
    pi): vs[i] = p_j(z_t) of query i, Q the quotient's commitment, us[t] = f_t(x), and (C, d, x, v, pi) an ordinary claim for
    `check`, `check_batch` or acc.new_instance.  Hiding with ws (one w_j per polynomial): then w_Q, q (max_j deg(p_j)
    coefficients) and w_bar are the caller's draws."""
    packed, lens = pack(ps)
    k = len(lens)
    Cs, zs = arr(Cs).reshape(k, 12), arr(zs).reshape(-1, 4)
    qp, qt = _queries(queries)
    m, T = qp.shape[0], zs.shape[0]
    wa = arr(ws).reshape(k, 4) if ws is not None else None
    qa = arr(q).reshape(-1, 4) if q is not None else None
    wqk, wqp = _host.opt(w_Q)
    wbk, wbp = _host.opt(w_bar)
    vs, us = np.zeros((max(1, m), 4), dtype=np.uint64), np.zeros((max(1, T), 4), dtype=np.uint64)
    Q, Cm, x, v, pi = np.zeros(12, dtype=np.uint64), np.zeros(12, dtype=np.uint64), np.zeros(4, dtype=np.uint64), \
        np.zeros(4, dtype=np.uint64), EvalProof()
    _host.chk(_host.lib().halo_pcdl_open_multi(ctx._h, p64(packed), p64(lens), C.c_uint64(k), p64(Cs), C.c_uint64(d), p64(zs),
                                               C.c_uint64(T), p64(qp), p64(qt), C.c_uint64(m), p64(wa) if wa is not None else None,
                                               wqp, p64(qa) if qa is not None else None,
                                               C.c_uint64(qa.shape[0] if qa is not None else 0), wbp, p64(vs), p64(Q), p64(us),
                                               p64(Cm), p64(x), p64(v), C.byref(pi)))
    return vs[:m], Q, us[:T], Cm, x, v, pi


def multi_claim(ctx, Cs, zs, queries, vs, Q, us):
    """The verifier's reduction of the claims of `open_multi` (commitments, points, (j, t) queries, their values, the
    quotient's commitment Q and the u_t) to its one claim -> (C, x, v)."""
    Cs, zs = arr(Cs).reshape(-1, 12), arr(zs).reshape(-1, 4)
    qp, qt = _queries(queries)
    vs, Q, us = arr(vs).reshape(qp.shape[0], 4), arr(Q, (12,)), arr(us).reshape(zs.shape[0], 4)
    Cm, x, v = np.zeros(12, dtype=np.uint64), np.zeros(4, dtype=np.uint64), np.zeros(4, dtype=np.uint64)
    _host.chk(_host.lib().halo_pcdl_multi_claim(ctx._h, p64(Cs), C.c_uint64(Cs.shape[0]), p64(zs), C.c_uint64(zs.shape[0]),
                                                p64(qp), p64(qt), p64(vs), C.c_uint64(qp.shape[0]), p64(Q), p64(us), p64(Cm),
                                                p64(x), p64(v)))
    return Cm, x, v


def succinct_check(ctx, Cm, d, z, v, pi):
    """pcdl.rs:252-314 -> (HPoly, U); raises Rejected"""
    Cm, z, v = arr(Cm, (12,)), arr(z, (4,)), arr(v, (4,))
    lg = max(int(d + 1).bit_length() - 1, 0)
    xis = np.zeros((lg + 1, 4), dtype=np.uint64)
    U = np.zeros(12, dtype=np.uint64)
    _host.chk(_host.lib().halo_pcdl_succinct_check(ctx._h, p64(Cm), C.c_uint64(d), p64(z), p64(v), C.byref(pi), p64(xis), p64(U)))
    return HPoly(xis), U


def check(ctx, Cm, d, z, v, pi):
    """pcdl.rs:323-342; raises Rejected"""
    Cm, z, v = arr(Cm, (12,)), arr(z, (4,)), arr(v, (4,))
    _host.chk(_host.lib().halo_pcdl_check(ctx._h, p64(Cm), C.c_uint64(d), p64(z), p64(v), C.byref(pi)))


def check_batch(ctx, claims, rho):
    """Batch decider over claims built by acc.new_instance (include/halo_pcdl.h halo_pcdl_check_batch; the reference has
    none): one MSM over the generators for all claims, combined with the caller's random rho != 0.  Raises Rejected with
    .code and .index of the first claim that `check` rejects, exactly as a loop of `check` calls would."""
    a = (Instance * max(1, len(claims)))(*claims)
    rho = arr(rho, (4,))
    idx = C.c_uint64()
    rc = _host.lib().halo_pcdl_check_batch(ctx._h, a, C.c_uint64(len(claims)), p64(rho), C.byref(idx))
    _host.chk(rc, idx.value)
