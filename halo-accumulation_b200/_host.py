"""ctypes binding of libhalo_host.so (include/halo_pcdl.h): the C++ host layer mirroring the reference's
pedersen / pcdl / acc modules on top of the CUDA ABI."""
import ctypes as C
import os

import numpy as np

from . import _build
from ._capi import HaloError, arr, load, p64, u64p

MAX_LG = 32
REJECT_SUCCINCT, REJECT_U, REJECT_U0, REJECT_D, REJECT_CBAR, REJECT_Z, REJECT_V = -10, -11, -12, -13, -14, -15, -17

_REJECT_TEXT = {
    REJECT_SUCCINCT: "C_(log_n) != CM.Commit_Sigma(c || v')",
    REJECT_U: "U != CM.Commit(ck, h_vec)",
    REJECT_U0: "U_0 != PCDL.Commit_rho0(ck^(1)_PC, h_0; w = bot)",
    REJECT_D: "d_i != d",
    REJECT_CBAR: "C_bar' != C_bar",
    REJECT_Z: "z' = z",
    REJECT_V: "h(z) = v",
}


class Rejected(Exception):
    """The analogue of the reference's `ensure!` Err (anyhow::Error) from a verifier-style function.  `index`: the
    rejected claim of a batch decision (check_batch / decider_batch) or step (verifier_batch), None for the single calls."""

    def __init__(self, code, index=None):
        super().__init__(_REJECT_TEXT.get(code, f"rejected ({code})"))
        self.code = code
        self.index = index


class EvalProof(C.Structure):  # pcdl.rs:22-30
    _fields_ = [
        ("lg_n", C.c_uint32),
        ("hiding", C.c_uint32),
        ("Ls", (C.c_uint64 * 12) * MAX_LG),
        ("Rs", (C.c_uint64 * 12) * MAX_LG),
        ("U", C.c_uint64 * 12),
        ("c", C.c_uint64 * 4),
        ("C_bar", C.c_uint64 * 12),
        ("w_prime", C.c_uint64 * 4),
    ]


class Instance(C.Structure):  # acc.rs:21-28
    _fields_ = [("C", C.c_uint64 * 12), ("d", C.c_uint64), ("z", C.c_uint64 * 4), ("v", C.c_uint64 * 4), ("pi", EvalProof)]


class Accumulator(C.Structure):  # acc.rs:43-59
    _fields_ = [
        ("C_bar", C.c_uint64 * 12),
        ("d", C.c_uint64),
        ("z", C.c_uint64 * 4),
        ("v", C.c_uint64 * 4),
        ("pi", EvalProof),
        ("h0", (C.c_uint64 * 4) * 2),
        ("U0", C.c_uint64 * 12),
        ("w", C.c_uint64 * 4),
    ]


_lib = None


def lib():
    global _lib
    if _lib is None:
        load()  # libhalo_b200.so first (RTLD_GLOBAL not needed: rpath $ORIGIN resolves the dependency)
        path = _build.HOST_LIB
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: build it with __graft_entry__.build()")
        _lib = C.CDLL(path)
        _lib.halo_host_last_error.restype = C.c_char_p
        _lib.halo_pcdl_commit_batch.argtypes = [C.c_void_p, u64p, u64p, C.c_uint64, C.c_uint64, u64p, u64p]
        _lib.halo_pcdl_open_batch.argtypes = [C.c_void_p, u64p, u64p, C.c_uint64, u64p, C.c_uint64, u64p, u64p, u64p, C.c_uint64,
                                              u64p, u64p, u64p, u64p, C.POINTER(EvalProof)]
        _lib.halo_pcdl_batch_claim.argtypes = [C.c_void_p, u64p, u64p, C.c_uint64, u64p, u64p, u64p]
        _lib.halo_pcdl_open_multi.argtypes = [C.c_void_p, u64p, u64p, C.c_uint64, u64p, C.c_uint64, u64p, C.c_uint64, u64p, u64p,
                                              C.c_uint64, u64p, u64p, u64p, C.c_uint64, u64p, u64p, u64p, u64p, u64p, u64p, u64p,
                                              C.POINTER(EvalProof)]
        _lib.halo_pcdl_commit_evals.argtypes = [C.c_void_p, u64p, C.c_uint64, C.c_uint64, u64p, u64p]
        _lib.halo_pcdl_open_multi_evals.argtypes = [C.c_void_p, u64p, C.c_uint64, u64p, C.c_uint64, u64p, C.c_uint64, u64p, u64p,
                                                    C.c_uint64, u64p, u64p, u64p, C.c_uint64, u64p, u64p, u64p, u64p, u64p, u64p,
                                                    u64p, C.POINTER(EvalProof)]
        _lib.halo_pcdl_multi_claim.argtypes = [C.c_void_p, u64p, C.c_uint64, u64p, C.c_uint64, u64p, u64p, u64p, C.c_uint64, u64p,
                                               u64p, u64p, u64p, u64p]
        _lib.halo_pcdl_check_batch.argtypes = [C.c_void_p, C.POINTER(Instance), C.c_uint64, u64p, u64p]
        _lib.halo_acc_decider_batch.argtypes = [C.c_void_p, C.POINTER(Accumulator), C.c_uint64, u64p, u64p]
        _lib.halo_acc_verifier_batch.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(Instance), u64p, C.POINTER(Accumulator),
                                                 C.c_uint64, u64p, u64p]
        _lib.halo_acc_verify_decide_batch.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(Instance), u64p, C.POINTER(Accumulator),
                                                      C.c_uint64, C.POINTER(Accumulator), C.c_uint64, u64p, u64p]
    return _lib


def chk(rc, index=None):
    """0 -> ok; HALO_REJECT_* -> Rejected (Err in the reference); HALO_E* -> HaloError (panic in the reference)."""
    if rc == 0:
        return
    if rc <= -10:
        raise Rejected(rc, index)
    raise HaloError(rc, lib().halo_host_last_error().decode())


def opt(a):
    if a is None:
        return None, None
    a = arr(a, (4,))
    return a, p64(a)
