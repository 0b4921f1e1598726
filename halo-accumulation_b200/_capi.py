"""ctypes binding of libhalo_b200.so (include/halo_b200.h).  This is the same C ABI a Rust shim binds
(INTEGRATION.md); Python only marshals numpy buffers.  There is no fallback: a missing library or a
failing CUDA call raises."""
import ctypes as C
import os

import numpy as np

from . import _build

u64p = C.POINTER(C.c_uint64)
u8p = C.POINTER(C.c_uint8)

HALO_OK, HALO_EINVAL, HALO_ELEN, HALO_ECUDA, HALO_ENCCL, HALO_ENOMEM, HALO_ESTATE, HALO_EIO = 0, -1, -2, -3, -4, -5, -6, -7
HALO_EINTERNAL = -8


class HaloError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libhalo_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load():
    """Loads the CUDA library; raises if it has not been built (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the hot path has no CPU fallback)")
    lib = C.CDLL(path)
    lib.halo_ctx_create.argtypes = [C.c_int, C.c_uint64, C.POINTER(C.c_void_p)]
    lib.halo_ctx_destroy.argtypes = [C.c_void_p]
    lib.halo_ctx_destroy.restype = None
    lib.halo_last_error.argtypes = [C.c_void_p]
    lib.halo_last_error.restype = C.c_char_p
    lib.halo_kernel_launches.argtypes = [C.c_void_p]
    lib.halo_kernel_launches.restype = C.c_uint64
    lib.halo_curve_name.restype = C.c_char_p
    lib.halo_num_generators.argtypes = [C.c_void_p]
    lib.halo_num_generators.restype = C.c_uint64
    lib.halo_save_generators.argtypes = [C.c_void_p, C.c_char_p]
    lib.halo_load_generators_file.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64]
    lib.halo_comm_slice.argtypes = [C.c_uint64, C.c_int, C.c_int, u64p, u64p]
    lib.halo_comm_slice.restype = None
    lib.halo_comm_destroy.argtypes = [C.c_void_p]
    lib.halo_comm_destroy.restype = None
    lib.halo_comm_init_rank.argtypes = [C.c_void_p, C.POINTER(C.c_uint8), C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    lib.halo_comm_derive_generators.argtypes = [C.c_void_p, C.c_uint64]
    lib.halo_comm_precompute_generators.argtypes = [C.c_void_p, C.c_int]
    lib.halo_msm_gens_sharded.argtypes = [C.c_void_p, u64p, C.c_uint64, C.c_uint64, C.c_uint64, u64p]
    lib.halo_msm_gens_sharded_resident.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, u64p]
    lib.halo_comm_allgather_sum.argtypes = [C.c_void_p, u64p, u64p]
    lib.halo_mgpu_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]
    lib.halo_mgpu_destroy.argtypes = [C.c_void_p]
    lib.halo_mgpu_destroy.restype = None
    lib.halo_mgpu_msm_gens.argtypes = [C.c_void_p, u64p, C.c_uint64, u64p]
    lib.halo_mgpu_last_error.argtypes = [C.c_void_p]
    lib.halo_mgpu_last_error.restype = C.c_char_p
    lib.halo_h_msm_batch.argtypes = [C.c_void_p, u64p, C.POINTER(C.c_uint32), u64p, C.c_uint64, u64p, u8p, u64p, C.c_uint64, u64p]
    lib.halo_h_msm_batch_submit.argtypes = [C.c_void_p, u64p, C.POINTER(C.c_uint32), u64p, C.c_uint64, C.POINTER(C.c_int)]
    lib.halo_h_msm_batch_collect.argtypes = [C.c_void_p, C.c_int, u64p, u8p, u64p, C.c_uint64, u64p]
    lib.halo_msm_gens_many.argtypes = [C.c_void_p, u64p, u64p, C.c_uint64, u64p]
    lib.halo_test_point_combine.argtypes = [C.c_void_p, C.c_int, u64p, u64p, u64p, u64p, C.c_uint64, u64p]
    if lib.halo_curve_name().decode() != _build.CURVE:
        raise RuntimeError(f"{path} was built for {lib.halo_curve_name().decode()}, HALO_B200_CURVE asks for {_build.CURVE}")
    _lib = lib
    return lib


def p64(a):
    assert a.dtype == np.uint64 and a.flags["C_CONTIGUOUS"], (a.dtype, a.flags)
    return a.ctypes.data_as(u64p)


def pack(vectors):
    """Scalar vectors -> (packed [sum len][4] array, lengths [k]) for the batch entry points.  A (k, n, 4) array is used in
    place; a list is copied into one buffer."""
    if isinstance(vectors, np.ndarray) and vectors.ndim == 3:
        k, n = vectors.shape[:2]
        packed = arr(vectors).reshape(-1, 4) if k * n else np.zeros((1, 4), dtype=np.uint64)
        return packed, np.full(k, n, dtype=np.uint64)
    vs = [arr(v).reshape(-1, 4) for v in vectors]
    lens = np.array([v.shape[0] for v in vs], dtype=np.uint64)
    packed = np.concatenate(vs) if vs and int(lens.sum()) else np.zeros((1, 4), dtype=np.uint64)
    return np.ascontiguousarray(packed), lens


def arr(x, shape=None):
    a = np.ascontiguousarray(x, dtype=np.uint64)
    return a.reshape(shape) if shape is not None else a
