"""Mirror of code/src/acc.rs: Instance, Accumulator, prover / verifier / decider."""
import ctypes as C

import numpy as np

from . import _host
from ._capi import arr, p64
from ._host import Accumulator, Instance, Rejected  # noqa: F401


def new_instance(Cm, d, z, v, pi):
    """Instance::new, acc.rs:109-119"""
    q = Instance()
    C.memmove(q.C, arr(Cm, (12,)).ctypes.data, 96)
    q.d = d
    C.memmove(q.z, arr(z, (4,)).ctypes.data, 32)
    C.memmove(q.v, arr(v, (4,)).ctypes.data, 32)
    q.pi = pi
    return q


def to_instance(acc):
    """impl From<Accumulator> for Instance, acc.rs:121-131"""
    q = Instance()
    _host.lib().halo_acc_to_instance(C.byref(acc), C.byref(q))
    return q


def prover(ctx, d, qs, h0, w, q, w_bar):
    """acc.rs:190-220; rng draws explicit in the reference's order: h0 (2 coefficients), w, open's q and w_bar."""
    a = (Instance * max(1, len(qs)))(*qs)
    h0, w, w_bar, q = arr(h0, (2, 4)), arr(w, (4,)), arr(w_bar, (4,)), arr(q).reshape(-1, 4)
    out = Accumulator()
    _host.chk(_host.lib().halo_acc_prover(ctx._h, C.c_uint64(d), a, C.c_uint64(len(qs)), p64(h0), p64(w), p64(q),
                                          C.c_uint64(q.shape[0]), p64(w_bar), C.byref(out)))
    return out


def verifier(ctx, d, qs, acc):
    """acc.rs:223-243; raises Rejected"""
    a = (Instance * max(1, len(qs)))(*qs)
    _host.chk(_host.lib().halo_acc_verifier(ctx._h, C.c_uint64(d), a, C.c_uint64(len(qs)), C.byref(acc)))


def decider(ctx, acc):
    """acc.rs:245-255; raises Rejected"""
    _host.chk(_host.lib().halo_acc_decider(ctx._h, C.byref(acc)))


def decider_batch(ctx, accs, rho):
    """check_batch over (C_bar, d, z, v, pi) of every accumulator (include/halo_pcdl.h halo_acc_decider_batch); raises
    Rejected with .code and .index exactly as a loop of `decider` calls would."""
    a = (Accumulator * max(1, len(accs)))(*accs)
    rho = arr(rho, (4,))
    idx = C.c_uint64()
    rc = _host.lib().halo_acc_decider_batch(ctx._h, a, C.c_uint64(len(accs)), p64(rho), C.byref(idx))
    _host.chk(rc, idx.value)


def verifier_batch(ctx, d, steps, rho):
    """k `verifier` calls at once (include/halo_pcdl.h halo_acc_verifier_batch): steps = [(qs, acc), ..], each checked against
    d; one MSM for all steps, combined with the caller's random rho != 0.  Raises Rejected with .code and .index (the step)
    exactly as a loop of `verifier` calls would."""
    qs = [q for s in steps for q in s[0]]
    a = (Instance * max(1, len(qs)))(*qs)
    accs = (Accumulator * max(1, len(steps)))(*[s[1] for s in steps])
    ms = np.array([len(s[0]) for s in steps] or [0], dtype=np.uint64)
    rho = arr(rho, (4,))
    idx = C.c_uint64()
    rc = _host.lib().halo_acc_verifier_batch(ctx._h, C.c_uint64(d), a, p64(ms), accs, C.c_uint64(len(steps)), p64(rho),
                                             C.byref(idx))
    _host.chk(rc, idx.value)


def verify_decide_batch(ctx, d, steps, decide_accs, rho):
    """verifier_batch(ctx, d, steps, rho) followed by decider_batch(ctx, decide_accs, rho) in one call
    (include/halo_pcdl.h halo_acc_verify_decide_batch).  Raises Rejected with .code and .index exactly as a loop of `verifier`
    calls followed by a loop of `decider` calls would: step i is index i, decided accumulator j is index len(steps) + j."""
    qs = [q for s in steps for q in s[0]]
    a = (Instance * max(1, len(qs)))(*qs)
    accs = (Accumulator * max(1, len(steps)))(*[s[1] for s in steps])
    dec = (Accumulator * max(1, len(decide_accs)))(*decide_accs)
    ms = np.array([len(s[0]) for s in steps] or [0], dtype=np.uint64)
    rho = arr(rho, (4,))
    idx = C.c_uint64()
    rc = _host.lib().halo_acc_verify_decide_batch(ctx._h, C.c_uint64(d), a, p64(ms), accs, C.c_uint64(len(steps)), dec,
                                                  C.c_uint64(len(decide_accs)), p64(rho), C.byref(idx))
    _host.chk(rc, idx.value)
