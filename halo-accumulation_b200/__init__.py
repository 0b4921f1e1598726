"""halo-accumulation on B200: host-side mirror of the reference's hot-path interface.

`Context` wraps the C ABI of libhalo_b200.so (include/halo_b200.h): hand-written sm_100a CUDA for the
Pallas MSMs, IPA folds and h-expansion behind PCDL / ASDL.  The submodules `group`, `pedersen`, `pcdl`
and `acc` mirror the reference's Rust modules of the same names (code/src/*.rs) on top of it.
"""
import ctypes as C
import os

import numpy as np

from . import _build
from ._capi import HaloError, arr, load, p64, pack, u8p

__all__ = ["Context", "Comm", "MultiGpu", "HaloError", "build", "points_sum", "points_equal", "comm_slice"]


def points_sum(points_jac):
    """Sum of Jacobian points in index order (combining per-GPU partial MSM results)."""
    pts = arr(points_jac).reshape(-1, 12)
    out = np.zeros(12, dtype=np.uint64)
    rc = load().halo_points_sum(p64(pts), C.c_uint64(pts.shape[0]), p64(out))
    if rc != 0:
        raise HaloError(rc, "halo_points_sum")
    return out


def build(force=False):
    return _build.build(force=force)


def points_equal(a, b):
    """`==` on Projective: same group element regardless of representation."""
    a, b = arr(a, (12,)), arr(b, (12,))
    return bool(load().halo_points_equal(p64(a), p64(b)))


def check_canaries():
    """(overwritten, live): how many live device buffers had the 256-byte canary behind their end overwritten (test hook;
    compute-sanitizer is not available on this pool)."""
    live = C.c_int()
    bad = load().halo_test_check_canaries(C.byref(live))
    return int(bad), live.value


def comm_slice(n_total, rank, size):
    """halo_comm_slice: the contiguous point slice [first, first + count) of rank `rank` of `size`."""
    first, count = C.c_uint64(), C.c_uint64()
    load().halo_comm_slice(C.c_uint64(n_total), int(rank), int(size), C.byref(first), C.byref(count))
    return first.value, count.value


class Comm:
    """Rank form of the sharded MSM (include/halo_b200.h, "multi-GPU"): one communicator per context, NCCL inside the library."""

    ID_BYTES = 128

    @staticmethod
    def unique_id():
        buf = (C.c_uint8 * Comm.ID_BYTES)()
        rc = load().halo_comm_unique_id(buf)
        if rc != 0:
            raise HaloError(rc, "halo_comm_unique_id failed (libnccl.so.2 not loadable?)")
        return bytes(buf)

    def __init__(self, ctx, uid, nranks, rank):
        self._lib, self.ctx = load(), ctx
        assert len(uid) == Comm.ID_BYTES
        h = C.c_void_p()
        buf = (C.c_uint8 * Comm.ID_BYTES).from_buffer_copy(uid)
        ctx._chk(self._lib.halo_comm_init_rank(ctx._h, buf, int(nranks), int(rank), C.byref(h)))
        self._h, self.rank, self.size = h, rank, nranks

    def close(self):
        if getattr(self, "_h", None):
            self._lib.halo_comm_destroy(self._h)
            self._h = None

    def derive_generators(self, n_total):
        self.ctx._chk(self._lib.halo_comm_derive_generators(self._h, C.c_uint64(n_total)))

    def precompute_generators(self, window=0):
        self.ctx._chk(self._lib.halo_comm_precompute_generators(self._h, int(window)))

    def msm_gens_sharded(self, local_scalars, n_global, off_local=0):
        s = arr(local_scalars).reshape(-1, 4)
        out = np.zeros(12, dtype=np.uint64)
        self.ctx._chk(self._lib.halo_msm_gens_sharded(self._h, p64(s), C.c_uint64(off_local), C.c_uint64(s.shape[0]), C.c_uint64(n_global), p64(out)))
        return out

    def msm_gens_sharded_resident(self, d_ptr, n_local, n_global, off_local=0):
        out = np.zeros(12, dtype=np.uint64)
        self.ctx._chk(self._lib.halo_msm_gens_sharded_resident(self._h, C.c_void_p(d_ptr), C.c_uint64(off_local), C.c_uint64(n_local),
                                                               C.c_uint64(n_global), p64(out)))
        return out

    def allgather_sum(self, point_jac):
        p = arr(point_jac, (12,))
        out = np.zeros(12, dtype=np.uint64)
        self.ctx._chk(self._lib.halo_comm_allgather_sum(self._h, p64(p), p64(out)))
        return out


class MultiGpu:
    """Node form: one caller thread, g devices (halo_mgpu_*); the multi-GPU body of `point_dot_affine` over GS[0..n)."""

    def __init__(self, devices, n_total, precompute_window=0):
        self._lib = load()
        devs = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        rc = self._lib.halo_mgpu_create(devs, len(devices), C.c_uint64(n_total), int(precompute_window), C.byref(h))
        if rc != 0:
            raise HaloError(rc, "halo_mgpu_create failed")
        self._h, self.size, self.n_total = h, len(devices), n_total

    def close(self):
        if getattr(self, "_h", None):
            self._lib.halo_mgpu_destroy(self._h)
            self._h = None

    def msm_gens(self, scalars):
        s = arr(scalars).reshape(-1, 4)
        out = np.zeros(12, dtype=np.uint64)
        rc = self._lib.halo_mgpu_msm_gens(self._h, p64(s), C.c_uint64(s.shape[0]), p64(out))
        if rc != 0:
            raise HaloError(rc, self._lib.halo_mgpu_last_error(self._h).decode())
        return out


class _MsmDesc(C.Structure):  # halo_msm_desc, include/halo_b200.h
    _fields_ = [("bases_affine", C.POINTER(C.c_uint64)), ("inf_flags", u8p), ("scalars", C.POINTER(C.c_uint64)),
                ("n", C.c_uint64), ("off", C.c_uint64)]


class Context:
    """One CUDA device + resident public parameters (replaces consts.rs:23-68)."""

    def __init__(self, device=0, max_n=1 << 20):
        self._lib = load()
        h = C.c_void_p()
        rc = self._lib.halo_ctx_create(int(device), C.c_uint64(max_n), C.byref(h))
        if rc != 0:
            raise HaloError(rc, "halo_ctx_create failed (no usable CUDA device? there is no CPU fallback)")
        self._h = h
        self.device = device
        self.max_n = max_n

    def close(self):
        if getattr(self, "_h", None):
            self._lib.halo_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != 0:
            raise HaloError(rc, self._lib.halo_last_error(self._h).decode())

    # ---- parameters ----
    def derive_generators(self, n):
        self._chk(self._lib.halo_derive_generators(self._h, C.c_uint64(n)))

    def derive_generators_range(self, first, n):
        """Resident generators become G_first .. G_{first+n-1} (point slice of the sharded MSM)."""
        self._chk(self._lib.halo_derive_generators_range(self._h, C.c_uint64(first), C.c_uint64(n)))

    def precompute_generators(self, c=0):
        """FIXED-base tables for the resident generators (optional accelerator; same results)."""
        self._chk(self._lib.halo_precompute_generators(self._h, int(c)))

    def set_fixed_base(self, on):
        self._chk(self._lib.halo_set_fixed_base(self._h, int(bool(on))))

    def timer_start(self):
        self._chk(self._lib.halo_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float()
        self._chk(self._lib.halo_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def load_generators(self, S, H, gs):
        S, H, gs = arr(S, (12,)), arr(H, (12,)), arr(gs).reshape(-1, 8)
        self._chk(self._lib.halo_load_generators(self._h, p64(S), p64(H), p64(gs), C.c_uint64(gs.shape[0])))

    def save_generators(self, path):
        """Writes S, H and the resident generators to a generator store (flat file of the 64-byte device records)."""
        self._chk(self._lib.halo_save_generators(self._h, os.fsencode(path)))

    def load_generators_file(self, path, n=0):
        """The first n generators of a store (0 = all) become the resident set; checksum and on-curve check included."""
        self._chk(self._lib.halo_load_generators_file(self._h, os.fsencode(path), C.c_uint64(n)))

    def num_generators(self):
        return int(self._lib.halo_num_generators(self._h))

    def get_generators(self, off, n):
        out = np.zeros((n, 8), dtype=np.uint64)
        self._chk(self._lib.halo_get_generators(self._h, C.c_uint64(off), C.c_uint64(n), p64(out)))
        return out

    def get_SH(self):
        S, H = np.zeros(12, dtype=np.uint64), np.zeros(12, dtype=np.uint64)
        self._chk(self._lib.halo_get_SH(self._h, p64(S), p64(H)))
        return S, H

    def derive_points(self, start, count):
        out = np.zeros((count, 8), dtype=np.uint64)
        self._chk(self._lib.halo_derive_points(self._h, C.c_uint64(start), C.c_uint64(count), p64(out)))
        return out

    # ---- MSM ----
    def msm_gens(self, scalars, off=0):
        s = arr(scalars).reshape(-1, 4)
        out = np.zeros(12, dtype=np.uint64)
        self._chk(self._lib.halo_msm_gens(self._h, p64(s), C.c_uint64(off), C.c_uint64(s.shape[0]), p64(out)))
        return out

    def msm_gens_many(self, scalar_vectors):
        """halo_msm_gens_many: row j of the (k, 12) result is sum_i scalar_vectors[j][i] * G_i (one segmented MSM per group)."""
        packed, lens = pack(scalar_vectors)
        out = np.zeros((max(1, len(lens)), 12), dtype=np.uint64)
        self._chk(self._lib.halo_msm_gens_many(self._h, p64(packed), p64(lens), C.c_uint64(len(lens)), p64(out)))
        return out[:len(lens)]

    def msm_gens_submit(self, scalars, off=0):
        """Pipelined halo_msm_gens: returns a ticket; `scalars` must stay alive (ideally pinned) until collect."""
        s = arr(scalars).reshape(-1, 4)
        t = C.c_int()
        self._chk(self._lib.halo_msm_gens_submit(self._h, p64(s), C.c_uint64(off), C.c_uint64(s.shape[0]), C.byref(t)))
        return t.value, s

    def msm_gens_submit_resident(self, d_ptr, n, off=0):
        """Pipelined MSM over device-resident scalars (CUDA pointer); returns a ticket for msm_gens_collect."""
        t = C.c_int()
        self._chk(self._lib.halo_msm_gens_submit_resident(self._h, C.c_void_p(d_ptr), C.c_uint64(off), C.c_uint64(n), C.byref(t)))
        return t.value, None

    def msm_gens_collect(self, ticket):
        out = np.zeros(12, dtype=np.uint64)
        self._chk(self._lib.halo_msm_gens_collect(self._h, int(ticket[0]), p64(out)))
        return out

    def msm_gens_resident(self, d_ptr, n, off=0):
        out = np.zeros(12, dtype=np.uint64)
        self._chk(self._lib.halo_msm_gens_resident(self._h, C.c_void_p(d_ptr), C.c_uint64(off), C.c_uint64(n), p64(out)))
        return out

    def msm(self, bases_affine, scalars, inf_flags=None):
        b, s = arr(bases_affine).reshape(-1, 8), arr(scalars).reshape(-1, 4)
        n = min(b.shape[0], s.shape[0])  # msm_unchecked truncates to the shorter input
        out = np.zeros(12, dtype=np.uint64)
        infp = None
        if inf_flags is not None:
            inf_flags = np.ascontiguousarray(inf_flags, dtype=np.uint8)
            infp = inf_flags.ctypes.data_as(u8p)
        self._chk(self._lib.halo_msm(self._h, p64(b), infp, p64(s), C.c_uint64(n), p64(out)))
        return out

    def msm_multi(self, problems):
        """A batch of small independent MSMs with one host round trip (halo_msm_multi).  problems: list of
        (bases_affine or None, scalars, inf_flags or None, off); None bases = resident generators from `off`."""
        descs = (_MsmDesc * max(1, len(problems)))()
        keep = []
        for d, (b, sc, inf, off) in zip(descs, problems):
            sc = arr(sc).reshape(-1, 4)
            keep.append(sc)
            d.scalars, d.n, d.off = p64(sc), sc.shape[0], off
            if b is not None:
                b = arr(b).reshape(-1, 8)
                assert b.shape[0] == sc.shape[0]
                keep.append(b)
                d.bases_affine = p64(b)
                if inf is not None:
                    inf = np.ascontiguousarray(inf, dtype=np.uint8)
                    keep.append(inf)
                    d.inf_flags = inf.ctypes.data_as(u8p)
        out = np.zeros((max(1, len(problems)), 12), dtype=np.uint64)
        self._chk(self._lib.halo_msm_multi(self._h, descs, C.c_uint32(len(problems)), p64(out)))
        return out[:len(problems)]

    def msm_jac(self, bases_jac, scalars):
        b, s = arr(bases_jac).reshape(-1, 12), arr(scalars).reshape(-1, 4)
        n = min(b.shape[0], s.shape[0])
        out = np.zeros(12, dtype=np.uint64)
        self._chk(self._lib.halo_msm_jac(self._h, p64(b), p64(s), C.c_uint64(n), p64(out)))
        return out

    # ---- tuning / accounting ----
    def set_msm_window(self, c):
        self._chk(self._lib.halo_set_msm_window(self._h, int(c)))

    def set_tuning(self, key, value):
        self._chk(self._lib.halo_set_tuning(self._h, key.encode(), int(value)))

    def set_profiling(self, on):
        self._chk(self._lib.halo_set_profiling(self._h, int(bool(on))))

    def last_msm_timings(self):
        t = (C.c_float * 6)()
        self._chk(self._lib.halo_last_msm_timings(self._h, t))
        return dict(zip(["digits", "scan", "scatter", "accumulate", "reduce", "total"], list(t)))

    def kernel_launches(self):
        return int(self._lib.halo_kernel_launches(self._h))

    # ---- test hooks (include/halo_b200_test.h) ----
    def test_fp_op(self, which, op, a, b=None):
        a = arr(a).reshape(-1, 4)
        out = np.zeros_like(a)
        bp = None
        if b is not None:
            b = arr(b).reshape(-1, 4)
            bp = p64(b)
        self._chk(self._lib.halo_test_fp_op(self._h, which, op, p64(a), bp, p64(out), C.c_uint64(a.shape[0])))
        return out

    def test_madd_chain(self, affine, neg=None):
        a = arr(affine).reshape(-1, 8)
        out = np.zeros(12, dtype=np.uint64)
        negp = None
        if neg is not None:
            neg = np.ascontiguousarray(neg, dtype=np.uint8)
            negp = neg.ctypes.data_as(u8p)
        self._chk(self._lib.halo_test_madd_chain(self._h, p64(a), negp, C.c_uint64(a.shape[0]), p64(out)))
        return out

    def test_add_chain(self, jac, dbls=0):
        a = arr(jac).reshape(-1, 12)
        out = np.zeros(12, dtype=np.uint64)
        self._chk(self._lib.halo_test_add_chain(self._h, p64(a), C.c_uint64(a.shape[0]), int(dbls), p64(out)))
        return out

    MSM_ROUTE_KEYS = ("c", "fixed", "P", "pass0_async", "acc", "quad_lanes", "quad_blocks", "acc_grid", "reduce_quad", "two_lanes")

    def test_msm_route(self, lane=0):
        """What the last MSM on `lane` ran (halo_test_msm_route); acc: 2 quad, 1 static, 0 lane claiming.  Reading clears it."""
        out = (C.c_int * 10)()
        self._chk(self._lib.halo_test_msm_route(self._h, int(lane), out))
        return dict(zip(self.MSM_ROUTE_KEYS, list(out)))

    def test_fp_mul_throughput(self, blocks, threads, iters, ilp=1):
        ms, ck = C.c_float(), C.c_uint64()
        self._chk(self._lib.halo_test_fp_mul_throughput(self._h, blocks, threads, iters, ilp, C.byref(ms), C.byref(ck)))
        return ms.value

    def test_vec_bench(self, kind, n):
        ms = C.c_float()
        self._chk(self._lib.halo_test_vec_bench(self._h, int(kind), C.c_uint64(n), C.byref(ms)))
        return ms.value

    def test_gather_throughput(self, table_bytes, blocks, threads, iters, nbytes=64):
        ms = C.c_float()
        self._chk(self._lib.halo_test_gather_throughput(self._h, C.c_uint64(table_bytes), blocks, threads, iters, nbytes, C.byref(ms)))
        return ms.value

    def test_imad_throughput(self, kind, blocks, threads, iters):
        ms, ck = C.c_float(), C.c_uint64()
        self._chk(self._lib.halo_test_imad_throughput(self._h, kind, blocks, threads, iters, C.byref(ms), C.byref(ck)))
        return ms.value
