/*
 * halo_b200.h -- C ABI of libhalo_b200.so: the B200 (sm_100a) implementation of the data-parallel hot
 * path of rasmus-kirk/halo-accumulation (PCDL commit / open / succinct check / check, ASDL decider).
 *
 * This is the drop-in boundary: exactly the entry points a Rust FFI shim inside the reference crate
 * would bind to replace the bodies of group.rs:13-37 and the loops of pcdl.rs:195-227 / pcdl.rs:56-77,338
 * (see INTEGRATION.md for the `extern "C"` block and the marshalling code).  Plain pointers and sizes
 * only; no C++ or torch types.  Paths below are relative to the reference tree (code/src/...).
 *
 * Data layout (identical to arkworks' in-memory representation, consts.rs:4-21, main.rs:47-53,91-100):
 *   scalar  (PallasScalar, Fr)  : uint64_t[4], little-endian limbs, Montgomery form, R = 2^256
 *   base-field element (Fq)     : uint64_t[4], same
 *   affine point (PallasAffine) : uint64_t[8] = x[4] | y[4]; infinity via a separate flag byte
 *   Jacobian point (PallasPoint): uint64_t[12] = x[4] | y[4] | z[4]; infinity <=> z == 0
 * Points returned by the library are valid Jacobian representatives of the same group element the
 * reference computes; compare with `==` on `Projective` (cross-multiplied) or after `into_affine()`.
 *
 * Conventions: every function returns 0 (HALO_OK) or a negative error code; nothing unwinds across
 * the ABI; `halo_last_error(ctx)` returns a human-readable message for the last failure on that
 * context.  Verifier-style rejections are NOT errors at this level: the library returns points and
 * scalars, the host layer above (pcdl / acc) raises the reference's `ensure!` failures.
 * A context is bound to one CUDA device and one stream; it is not thread-safe (the reference is
 * single-threaded), but different contexts may be used from different host threads at the same time, on the same
 * device or not; calls are synchronous except the `_submit` / `_collect` pairs.  All host buffers are
 * owned by the caller; all device memory is owned by the context.  There is no CPU fallback: if
 * no CUDA device is usable, halo_ctx_create fails with HALO_ECUDA.
 */
#ifndef HALO_B200_H
#define HALO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HALO_OK 0
#define HALO_EINVAL (-1) /* n not a power of two / exceeds the context's max_n (pcdl.rs:102-104, :261-262) */
#define HALO_ELEN (-2)   /* length mismatch (pedersen.rs:7-12) */
#define HALO_ECUDA (-3)  /* CUDA runtime failure; see halo_last_error */
#define HALO_ENCCL (-4)  /* NCCL failure (libnccl.so.2 missing, communicator error, ranks disagreeing on the MSM plan) */
#define HALO_ENOMEM (-5)
#define HALO_ESTATE (-6) /* call out of order (e.g. generators not loaded) */
#define HALO_EIO (-7)    /* generator store: file cannot be opened / read / written */
#define HALO_EINTERNAL (-8) /* the library contradicts itself (a batch decision that its one-by-one checks do not confirm) */

typedef struct halo_ctx halo_ctx;

/* ---- context ------------------------------------------------------------------------------------- */
/* Creates a context on CUDA device `device` able to handle vectors up to `max_n` elements. */
int halo_ctx_create(int device, uint64_t max_n, halo_ctx **out);
void halo_ctx_destroy(halo_ctx *ctx);
const char *halo_last_error(halo_ctx *ctx);
/* The curve this library was built for: "pallas" (libhalo_b200.so, the reference's `ark_pallas` types) or "vesta"
 * (libhalo_b200_vesta.so: same sources and entry points with coordinate and scalar field swapped, SURVEY 8(f).4).
 * A process that needs both halves of the Pasta cycle loads the two libraries with dlopen(RTLD_LOCAL). */
const char *halo_curve_name(void);
/* Count of this library's kernel launches on the context since creation (bench accounting). */
uint64_t halo_kernel_launches(halo_ctx *ctx);
/* Tuning / diagnostics: force the Pippenger window width (0 = automatic). */
int halo_set_msm_window(halo_ctx *ctx, int c);
/* Measurement knobs: they select alternative kernels, launch geometries and schedules, not results.  The MSM and opening
 * variants are compared with the oracle, and with each other, in tests/test_gpu_tuning.py (which also checks that this list
 * matches the keys the library accepts); the host-buffer, sort and batch-check knobs in the tests named there.  Keys and values:
 *   accumulation   "acc_static" 0 .. 2: 1 / 2 = force thread-per-bucket / lane-level bucket claiming (0 = automatic);
 *                  "acc_blocks_per_sm" 0 .. 32 (CTAs per SM of the lane-claiming kernel, 0 = 4); "acc_quad" 0 / other (four
 *                  lanes per bucket for small MSMs); "acc_quad_max_buckets" >= 0; "acc_quad_lanes" 0 / 2 / 4 and "acc_quad_blocks"
 *                  0 / 4 / 6 (CTAs per SM; 0 = policy); "pair_passes" >= -1 (-1 = policy by bucket fill, above 8 means 8);
 *                  "pair_bwd_async" 0 / other; "reduce_quad" 0 / other (refused above the size limit of the quad reduction)
 *   counting sort  "sort_ahead" (CTAs per SM of the sort of the next pipelined call, 0 = off), "sort2" 0 / other, "sort2_min_lg"
 *                  (two-level staged sort)
 *   host buffers   "split_blocking" (lg of the size from which the blocking call runs as point slices, 0 = never),
 *                  "split_first_16ths" (clamped to 1 .. 15), "split_second_16ths" (clamped to 0 .. 14; 0 = two slices),
 *                  "stage_pageable" 0 / other, "stage_threads" (clamped to 1 .. 8)
 *   opening        "ipa_defer_rounds" (-1 = automatic), "ipa_defer2_rounds", "ipa_two_lanes" 0 / other, "ipa_freeze_len" (0 = 8192),
 *                  "ipa_frozen_c" 0 or 4 .. 20 (0 = automatic window), "ipa_fold_call_min_lg" (folds of >= 2^v outputs use the
 *                  kernel copy with the multiplication out of line; -1 = never)
 *   batch checks   "combine_min_outputs" (the exact C' = C + alpha C_bar - w' S of hiding claims and C* = C_bar - omega S of
 *                  accumulation steps run as one device launch from this many points on, on host threads below; -1 = never)
 * Unknown keys and values outside the ranges given return HALO_EINVAL. */
int halo_set_tuning(halo_ctx *ctx, const char *key, int value);
/* Enable per-phase CUDA-event timing of the MSM; read back with halo_last_msm_timings (ms):
 * [digits, scan, scatter, accumulate, bucket_reduce, total]. */
int halo_set_profiling(halo_ctx *ctx, int on);
int halo_last_msm_timings(halo_ctx *ctx, float out_ms[6]);

/* ---- public parameters: replaces consts.rs:23-68 (N, S, H, GS) ----------------------------------- */
/* K6. Derives S = P_0, H = P_1, G_i = P_{i+2}, i < n, on the device by the rule of main.rs:18-45
 * (P_k = [SHA3-256(genesis || k as u64 LE) mod r] * (-1, 2)) and keeps them resident. */
int halo_derive_generators(halo_ctx *ctx, uint64_t n);
/* Point-slice variant for the sharded MSM: S, H as above, resident generators are G_first .. G_{first+n-1}
 * (rank r of g holds the slice [r n/g, (r+1) n/g); halo_msm_gens offsets are relative to `first`). */
int halo_derive_generators_range(halo_ctx *ctx, uint64_t first, uint64_t n);
/* FIXED-base acceleration for halo_msm_gens / halo_h_msm: precomputes the multiples 2^(off_w) G_i of every resident
 * generator (W x the generator memory) so all windows share one bucket set.  c = window width, 0 = automatic.
 * Optional; results are identical with or without it.  Invalidated when the generators change. */
int halo_precompute_generators(halo_ctx *ctx, int c);
/* Switch the FIXED-base path off / on without dropping the tables (A/B measurements). */
int halo_set_fixed_base(halo_ctx *ctx, int on);
/* Alternative: take the reference's own constants (consts::S, consts::H as Jacobian, consts::GS affine). */
int halo_load_generators(halo_ctx *ctx, const uint64_t S_jac[12], const uint64_t H_jac[12],
                         const uint64_t *gs_affine /*[n][8]*/, uint64_t n);
/* Generator store (SURVEY 8(f).3; the reference's analogue is main.rs:47-67 writing consts.rs / points.txt, and
 * report.md:2081-2086 names the generated source as what limits n): S, H and the resident G_i as one flat file of
 * 64-byte Montgomery affine records behind a 64-byte header (magic, curve, n, checksum).  `load` reads the first n
 * generators of a store (0 = all of them) through pinned double buffers, verifies the checksum when the whole file is
 * read, and checks ON THE DEVICE that every record is a canonical point on the curve; on failure the context is left
 * without generators.  HALO_EIO: file problems; HALO_EINVAL: not a store, other curve, too short, corrupt. */
int halo_save_generators(halo_ctx *ctx, const char *path);
int halo_load_generators_file(halo_ctx *ctx, const char *path, uint64_t n);
/* Reads generators back (tests / caching): out_affine[i] = G_{off+i}. */
int halo_get_generators(halo_ctx *ctx, uint64_t off, uint64_t n, uint64_t *out_affine /*[n][8]*/);
int halo_get_SH(halo_ctx *ctx, uint64_t S_jac[12], uint64_t H_jac[12]);
/* Number of resident generators: the reference's N (consts.rs:23); D = N - 1. */
uint64_t halo_num_generators(halo_ctx *ctx);
/* Raw derivation without installing: out_affine[i] = P_{start+i}. */
int halo_derive_points(halo_ctx *ctx, uint64_t start, uint64_t count, uint64_t *out_affine /*[count][8]*/);

/* ---- K2: multi-scalar multiplication ------------------------------------------------------------- */
/* sum_i scalars[i] * G_{off+i}, i < n.   Replaces group.rs:24-26 `point_dot_affine` as called by
 * pedersen.rs:14 over GS[0..n] (pcdl.rs:109, :338; acc.rs:153, :195). */
int halo_msm_gens(halo_ctx *ctx, const uint64_t *scalars /*[n][4]*/, uint64_t off, uint64_t n, uint64_t out_jac[12]);
/* k MSMs over the resident generators: out_jac[j] = sum_{i < lens[j]} scalars_j[i] * G_i, the scalar vectors packed back to
 * back in output order (a batch of commitments: ark-poly-commit's `commit` over a list, the columns of a circuit).  Runs as
 * segmented MSMs -- one sort, accumulation and bucket reduction for a group of outputs -- with the copy of the next group and
 * the host finish of the previous one beside each group's kernels (DESIGN.md K2c); a group of one output is a halo_msm_gens
 * call.  lens[j] = 0 gives infinity; k = 0 does nothing.  HALO_EINVAL: NULL pointers with k > 0, a packed size that
 * overflows; HALO_ESTATE: a length beyond the resident generators (nothing runs in either case). */
int halo_msm_gens_many(halo_ctx *ctx, const uint64_t *scalars /*packed, [sum lens][4]*/, const uint64_t *lens /*[k]*/, uint64_t k,
                       uint64_t *out_jac /*[k][12]*/);
/* sum_i scalars[i] * bases[i] for caller-supplied affine bases; inf_flags may be NULL.
 * Replaces group.rs:24-26 for arbitrary bases and, after the caller's normalisation, group.rs:18-21. */
int halo_msm(halo_ctx *ctx, const uint64_t *bases_affine /*[n][8]*/, const uint8_t *inf_flags /*[n] or NULL*/,
             const uint64_t *scalars /*[n][4]*/, uint64_t n, uint64_t out_jac[12]);
/* Same as group.rs:18-21 `point_dot`: Jacobian bases, normalised on the device (batched inversion). */
int halo_msm_jac(halo_ctx *ctx, const uint64_t *bases_jac /*[n][12]*/, const uint64_t *scalars /*[n][4]*/, uint64_t n,
                 uint64_t out_jac[12]);
/* Pipelined form of halo_msm_gens for streams of commitments (an IVC chain, a batch of polynomials): submit enqueues
 * the host-to-device copy on a copy stream and the MSM behind it and returns at once; collect waits for that MSM and
 * finishes it.  Two tickets may be in flight, so the copy of call k+1 overlaps the kernels of call k, and (n >= 2^22) the
 * counting sort of call k+1 runs on a high-priority stream beside the bucket accumulation of call k (the sort is bound
 * by L2 atomics, the accumulation by the integer pipe).  `scalars` must stay valid (and should be pinned) until the
 * ticket is collected. */
int halo_msm_gens_submit(halo_ctx *ctx, const uint64_t *scalars /*[n][4]*/, uint64_t off, uint64_t n, int *ticket);
int halo_msm_gens_collect(halo_ctx *ctx, int ticket, uint64_t out_jac[12]);
/* Device-resident variants for throughput measurement: d_scalars is a CUDA device pointer to n scalars (complete when
 * the call is made; for submit_resident untouched until the ticket is collected). */
int halo_msm_gens_resident(halo_ctx *ctx, const void *d_scalars, uint64_t off, uint64_t n, uint64_t out_jac[12]);
int halo_msm_gens_submit_resident(halo_ctx *ctx, const void *d_scalars, uint64_t off, uint64_t n, int *ticket);

/* Sum of g Jacobian points on the host, in index order. */
int halo_points_sum(const uint64_t *points_jac /*[g][12]*/, uint64_t g, uint64_t out_jac[12]);
/* Projective equality of two Jacobian points (cross-multiplied, as `==` on arkworks' Projective): 1 / 0. */
int halo_points_equal(const uint64_t a_jac[12], const uint64_t b_jac[12]);
/* CUDA-event stopwatch on the context's stream (the stream every kernel of this library is launched on). */
int halo_timer_start(halo_ctx *ctx);
int halo_timer_stop(halo_ctx *ctx, float *elapsed_ms);

/* ---- multi-GPU: the MSM sharded by point slice (SURVEY 8e) ---------------------------------------------------------
 * Only the MSM shards.  Rank r of g holds the contiguous slice [first_r, first_r + count_r) of the generators
 * (halo_comm_slice) and the matching slice of the scalars; every rank runs the Pippenger on its slice and the partial
 * results meet in ONE ncclAllGather over NVLink / NVSwitch, enqueued by the library on the context's stream; the ranks'
 * partials are added in rank order and finished once, so every rank returns the same point.  Replaces group.rs:24-26 at scale.
 * NCCL is loaded at run time (dlopen "libnccl.so.2", or the path in HALO_NCCL_LIB) the first time one of these is called.
 *
 * Rank form: one process or thread per GPU (torchrun, MPI, a thread pool).  Rank 0 calls halo_comm_unique_id, the caller
 * distributes the 128 bytes by its own means, then EVERY rank calls halo_comm_init_rank (a collective: it returns when all
 * ranks have joined).  Every halo_msm_gens_sharded* / halo_comm_allgather_sum call is a collective as well: all ranks must
 * make it, in the same order, with the same n_global. */
#define HALO_COMM_ID_BYTES 128
typedef struct halo_comm halo_comm;
int halo_comm_unique_id(uint8_t id[HALO_COMM_ID_BYTES]);
int halo_comm_init_rank(halo_ctx *ctx, const uint8_t id[HALO_COMM_ID_BYTES], int nranks, int rank, halo_comm **out);
void halo_comm_destroy(halo_comm *comm);
int halo_comm_rank(const halo_comm *comm);
int halo_comm_size(const halo_comm *comm);
int halo_nccl_version(void); /* e.g. 22809; 0 if NCCL cannot be loaded */
/* The contiguous point slice of rank `rank` of `size` over n_total points: [*first, *first + *count). */
void halo_comm_slice(uint64_t n_total, int rank, int size, uint64_t *first, uint64_t *count);
/* Derives this rank's slice of the n_total generators (halo_derive_generators_range over halo_comm_slice). */
int halo_comm_derive_generators(halo_comm *comm, uint64_t n_total);
/* halo_precompute_generators with a window chosen from the LARGEST slice, so that every rank builds tables for the same
 * plan (window = 0: automatic). */
int halo_comm_precompute_generators(halo_comm *comm, int window);
/* sum over ALL ranks of sum_{i < n_local} local_scalars[i] * G_{first_rank + off_local + i}: this rank contributes its
 * n_local points (0 allowed); n_global = the total number of points of the whole MSM (sum of the ranks' n_local), from
 * which every rank derives the same window plan.  Result on every rank. */
int halo_msm_gens_sharded(halo_comm *comm, const uint64_t *local_scalars /*[n_local][4]*/, uint64_t off_local, uint64_t n_local,
                          uint64_t n_global, uint64_t out_jac[12]);
/* Same with this rank's scalars already on its device (CUDA pointer). */
int halo_msm_gens_sharded_resident(halo_comm *comm, const void *d_local_scalars, uint64_t off_local, uint64_t n_local,
                                   uint64_t n_global, uint64_t out_jac[12]);
/* All-gather of one Jacobian point per rank and their sum in rank order: combines per-rank results that were computed by
 * other calls (e.g. the pipelined halo_msm_gens_submit / _collect on every rank). */
int halo_comm_allgather_sum(halo_comm *comm, const uint64_t point_jac[12], uint64_t out_jac[12]);

/* Node form: ONE caller thread, g devices.  The library owns a context, a communicator (ncclCommInitAll) and a worker
 * thread per device, derives each device's slice of the n_total generators and (precompute_window >= 0; 0 = automatic
 * window) its FIXED-base tables.  halo_mgpu_msm_gens then is the multi-GPU body of `point_dot_affine` over GS[0..n):
 * every device copies its part of the caller's scalar vector, runs its slice and joins the all-gather. */
typedef struct halo_mgpu halo_mgpu;
int halo_mgpu_create(const int *devices, int g, uint64_t n_total, int precompute_window, halo_mgpu **out);
void halo_mgpu_destroy(halo_mgpu *m);
int halo_mgpu_size(const halo_mgpu *m);
halo_ctx *halo_mgpu_ctx(halo_mgpu *m, int i);
const char *halo_mgpu_last_error(halo_mgpu *m);
int halo_mgpu_msm_gens(halo_mgpu *m, const uint64_t *scalars /*[n][4]*/, uint64_t n, uint64_t out_jac[12]);

/* ---- scalar vectors -------------------------------------------------------------------------------- */
/* sum_i xs[i] * ys[i] in Fr.  Replaces group.rs:13-15 `scalar_dot`. */
int halo_scalar_dot(halo_ctx *ctx, const uint64_t *xs, const uint64_t *ys, uint64_t n, uint64_t out[4]);
/* out[j] = z^j, j < n.  Replaces group.rs:29-37 `construct_powers`. */
int halo_construct_powers(halo_ctx *ctx, const uint64_t z[4], uint64_t n, uint64_t *out /*[n][4]*/);

/* ---- K5: the polynomial h(X) = prod_{i<lg n} (1 + xi_{lg n - i} X^{2^i}) ---------------------------- */
/* Coefficient vector of h.  xis = [xi_0 .. xi_{lg n}] (xi_0 is carried but unused, as in the reference).
 * Replaces HPoly::get_poly, pcdl.rs:56-77. */
int halo_h_expand(halo_ctx *ctx, const uint64_t *xis /*[lg_n+1][4]*/, uint32_t lg_n, uint64_t *out /*[2^lg_n][4]*/);
/* U' = <GS[0..n), coeffs(h)>: expansion and MSM without the coefficients ever leaving the device.
 * Replaces pcdl.rs:338 (`pedersen::commit(None, &GS[0..n], &h.get_poly().coeffs)`), the decider's MSM. */
int halo_h_msm(halo_ctx *ctx, const uint64_t *xis /*[lg_n+1][4]*/, uint32_t lg_n, uint64_t out_jac[12]);
/* pcdl::check (pcdl.rs:323-342) in one call: <G, coeffs(h)> as above AND the k-point MSM that succinct_check's group
 * equation reduces to (pcdl.rs:285-310: k = 2 lg n + 2 points L_i, R_i, H, U with host-computed scalars), run
 * concurrently on two streams; the challenges need only the transcript, so neither waits for the other. */
int halo_h_msm_with(halo_ctx *ctx, const uint64_t *xis /*[lg_n+1][4]*/, uint32_t lg_n, const uint64_t *bases_affine /*[k][8]*/,
                    const uint8_t *inf_flags /*[k] or NULL*/, const uint64_t *scalars /*[k][4]*/, uint64_t k,
                    uint64_t out_h_jac[12], uint64_t out_small_jac[12]);
/* Batch decider core (K5b): ONE point
 *   <GS[0..n), sum_j weights[j] coeffs(h_j)> + sum_{i<m} scalars[i] * bases[i],   n = max_j 2^lg_ns[j],
 * where h_j is the h(X) of claim j with challenges xi_0 .. xi_{lg_ns[j]} (the next lg_ns[j] + 1 rows of xis, concatenated
 * in claim order; xi_0 unused as in halo_h_expand) and its coefficients are zero from 2^lg_ns[j] on.  The coefficient sum
 * is built on the device in one kernel, then the generator MSM (FIXED-base tables under the same condition as halo_h_msm)
 * and the companion MSM over caller-supplied affine points run on two streams.  m is not limited to 4096 (k claims at
 * lg n = 20 bring 42 k + 1 points, DESIGN.md K5b).  Each lg_ns[j] is checked like halo_h_msm's lg_n; k, m < 2^32.
 * k = m = 0 gives infinity.  Same as halo_h_msm_batch_submit followed by halo_h_msm_batch_collect. */
int halo_h_msm_batch(halo_ctx *ctx, const uint64_t *xis /*sum_j (lg_ns[j]+1) rows of [4]*/, const uint32_t *lg_ns /*[k]*/,
                     const uint64_t *weights /*[k][4]*/, uint64_t k, const uint64_t *bases_affine /*[m][8]*/,
                     const uint8_t *inf_flags /*[m] or NULL*/, const uint64_t *scalars /*[m][4]*/, uint64_t m, uint64_t out_jac[12]);
/* halo_h_msm_batch in two calls (K5d), so that the caller's host work runs while the device computes the generator part.
 * submit enqueues the coefficient sum and the generator MSM and returns without waiting for the device; the caller's
 * buffers are read before it returns.  collect runs the companion MSM on the second stream, waits for both and returns
 * their sum, which is what halo_h_msm_batch returns for the same arguments.  One batch may be outstanding per context:
 * a second submit, or a collect without a submit, is HALO_ESTATE.  A caller that gives up after a submit collects with
 * m = 0 to leave the context idle.  Other calls of the library may be made between the two. */
int halo_h_msm_batch_submit(halo_ctx *ctx, const uint64_t *xis /*sum_j (lg_ns[j]+1) rows of [4]*/, const uint32_t *lg_ns /*[k]*/,
                            const uint64_t *weights /*[k][4]*/, uint64_t k, int *ticket);
int halo_h_msm_batch_collect(halo_ctx *ctx, int ticket, const uint64_t *bases_affine /*[m][8]*/, const uint8_t *inf_flags /*[m] or NULL*/,
                             const uint64_t *scalars /*[m][4]*/, uint64_t m, uint64_t out_jac[12]);
/* A batch of small, independent MSMs with ONE host round trip (SURVEY 8(f).2): the accumulation verifier's
 * common_subroutine (acc.rs:135-188) needs commit(h_0) (acc.rs:153) and, per instance q_i, the 2 lg n + 2 point MSM that
 * succinct_check's group equation reduces to (pcdl.rs:285-310); none depends on another's result, so they are enqueued
 * together (alternating between the context's two streams) and synchronised once.  Each result is kept separate: the
 * reference checks every instance on its own, and so does the caller.
 * bases_affine == NULL: the resident generators G_off .. G_{off+n-1}.  n <= 4096 per MSM.  out_jac: [count][12]. */
typedef struct halo_msm_desc {
    const uint64_t *bases_affine; /* [n][8] Montgomery affine, or NULL */
    const uint8_t *inf_flags;     /* [n] or NULL (only with bases_affine) */
    const uint64_t *scalars;      /* [n][4] */
    uint64_t n;
    uint64_t off;                 /* first resident generator when bases_affine == NULL */
} halo_msm_desc;
int halo_msm_multi(halo_ctx *ctx, const halo_msm_desc *descs, uint32_t count, uint64_t *out_jac /*[count][12]*/);
/* out = h_0 + sum_{i<m} alphas[i+1] * coeffs(h_i), zero-padded to n = 2^lg_n.
 * Replaces AccumulatedHPolys::get_poly, acc.rs:85-94. */
int halo_h_lincomb(halo_ctx *ctx, const uint64_t *h0 /*[n_h0][4]*/, uint64_t n_h0, const uint64_t *alphas /*[m+1][4]*/,
                   const uint64_t *xis /*[m][lg_n+1][4]*/, uint64_t m, uint32_t lg_n, uint64_t *out /*[2^lg_n][4]*/);

/* Same, but the polynomial stays on the device for a following halo_ipa_begin_resident (acc.rs:209 opens h.get_poly():
 * no reason to move 32 n bytes to the host and back); *degree_out = its degree (DensePolynomial::degree). */
int halo_h_lincomb_resident(halo_ctx *ctx, const uint64_t *h0, uint64_t n_h0, const uint64_t *alphas, const uint64_t *xis,
                            uint64_t m, uint32_t lg_n, uint64_t *degree_out);

/* ---- K3b: k polynomials opened at one point (halo_pcdl_open_batch, include/halo_pcdl.h) ----------------- */
/* vs_out[j] = p_j(z) for k polynomials packed back to back (polynomial j has n_coeffs[j] <= n coefficients), in one segmented
 * evaluation: the coefficients are uploaded once (pageable memory staged as by halo_msm_gens), z^0 .. z^(max_j n_coeffs[j] - 1)
 * built on the device, then two launches for all k.  The polynomials stay on the device for halo_poly_combine_resident; their
 * buffer (sum_j n_coeffs[j] * 32 bytes) stays in the context until it is destroyed, like the opening's buffers.
 * HALO_EINVAL: NULL pointers, k = 0 or k >= 2^31, n beyond the resident generators, n_coeffs[j] > n (nothing runs).
 * HALO_ENOMEM: no device memory for the upload; nothing is written and no evaluation is left to combine. */
int halo_poly_eval_many(halo_ctx *ctx, const uint64_t *coeffs /*packed, [sum n_coeffs][4]*/, const uint64_t *n_coeffs /*[k]*/,
                        uint64_t k, uint64_t n, const uint64_t z[4], uint64_t *vs_out /*[k][4]*/);
/* p = sum_j alpha^j p_j over the polynomials of the last halo_poly_eval_many (one launch; coefficients of p_j past
 * n_coeffs[j] are zero), left on the device for halo_ipa_begin_resident; *degree_out = its degree (DensePolynomial::degree).
 * May be called again with another alpha.  HALO_ESTATE: no preceding evaluation on this context.  HALO_ENOMEM: no device
 * memory for p; the context then holds no resident polynomial. */
int halo_poly_combine_resident(halo_ctx *ctx, const uint64_t alpha[4], uint64_t *degree_out);

/* ---- K3c: k polynomials opened at several points (halo_pcdl_open_multi, include/halo_pcdl.h) ----------- */
#define HALO_MULTI_MAX_POINTS 64
/* The upload half of halo_poly_eval_many: the k packed polynomials become the context's resident polynomials, with the same
 * errors; an earlier upload and its quotient are gone whatever the outcome. */
int halo_poly_upload(halo_ctx *ctx, const uint64_t *coeffs /*packed, [sum n_coeffs][4]*/, const uint64_t *n_coeffs /*[k]*/,
                     uint64_t k, uint64_t n);
/* vs_out[i] = p_{q_poly[i]}(zs[q_point[i]]) over the resident polynomials, for m queries in two launches (k_quot_chunks,
 * k_quot_carry).  HALO_EINVAL: NULL pointers, T = 0 or T > HALO_MULTI_MAX_POINTS, m = 0 or m >= 2^31, q_poly[i] >= k or
 * q_point[i] >= T.  HALO_ESTATE: nothing uploaded.  HALO_ENOMEM: no device memory for the scratch; nothing is written. */
int halo_poly_eval_queries(halo_ctx *ctx, const uint64_t *zs /*[T][4]*/, uint64_t T, const uint64_t *q_poly /*[m]*/,
                           const uint64_t *q_point /*[m]*/, uint64_t m, uint64_t *vs_out /*[m][4]*/);
/* With f_t = sum_{i: q_point[i] = t} weights[i] p_{q_poly[i]} over the resident polynomials (n = the longest of them):
 *   q = sum_t scales[t] (f_t - f_t(z_t)) / (X - z_t), n - 1 coefficients, kept on the device;
 *   rems_out[t] = f_t(z_t), the remainders;  Q_out = <GS[0..n-1), q> by the generator-MSM route of halo_msm_gens.
 * The division is a chunked scan in three launches (k_quot_chunks, k_quot_carry, k_quot_write).  Errors as
 * halo_poly_eval_queries; on any error no quotient is left for halo_poly_lincomb_resident. */
int halo_poly_quotient(halo_ctx *ctx, const uint64_t *zs /*[T][4]*/, const uint64_t *scales /*[T][4]*/, uint64_t T,
                       const uint64_t *q_poly /*[m]*/, const uint64_t *q_point /*[m]*/, const uint64_t *weights /*[m][4]*/, uint64_t m,
                       uint64_t *rems_out /*[T][4]*/, uint64_t Q_out[12]);
/* P = sum_j cs[j] p_j + c_q q over the resident polynomials and the quotient of the last halo_poly_quotient (one launch,
 * k_poly_lincomb), left on the device for halo_ipa_begin_resident; *degree_out = its degree.  HALO_ESTATE: no quotient of
 * the current upload.  HALO_ENOMEM: no device memory for P; the context then holds no resident polynomial. */
int halo_poly_lincomb_resident(halo_ctx *ctx, const uint64_t *cs /*[k][4]*/, const uint64_t c_q[4], uint64_t *degree_out);

/* ---- K3 / K4 / K7: the rounds of PCDL.open (pcdl.rs:183-231) ----------------------------------------- */
typedef struct halo_ipa halo_ipa;
/* Uploads the coefficients of p (zero-padded to n, pcdl.rs:183-184), copies GS[0..n) (pcdl.rs:185), builds
 * (1, z, .., z^{n-1}) on the device (pcdl.rs:186) and returns v = p(z) (pcdl.rs:135). */
int halo_ipa_begin(halo_ctx *ctx, const uint64_t *coeffs /*[n_coeffs][4]*/, uint64_t n_coeffs, uint64_t n,
                   const uint64_t z[4], halo_ipa **out, uint64_t v_out[4]);
/* halo_ipa_begin on the polynomial left on the device by halo_h_lincomb_resident. */
int halo_ipa_begin_resident(halo_ctx *ctx, uint64_t n, const uint64_t z[4], halo_ipa **out, uint64_t v_out[4]);
void halo_ipa_destroy(halo_ipa *st);
/* Hiding (pcdl.rs:137-164): p_bar = q (X - z) on the device, returns <GS, p_bar> (the caller adds w_bar * S). */
int halo_ipa_blind_commit(halo_ipa *st, const uint64_t *q /*[n_q][4]*/, uint64_t n_q, uint64_t out_jac[12]);
/* p' = p + alpha p_bar (pcdl.rs:156). */
int halo_ipa_blind_apply(halo_ipa *st, const uint64_t alpha[4]);
/* H' = xi_0 * H (pcdl.rs:181), computed by the caller. */
int halo_ipa_set_hprime(halo_ipa *st, const uint64_t Hprime_jac[12]);
/* L = <c_hi, G_lo> + <c_hi, z_lo> H', R = <c_lo, G_hi> + <c_lo, z_hi> H' for the current round (pcdl.rs:199-209). */
int halo_ipa_round_lr(halo_ipa *st, uint64_t L_jac[12], uint64_t R_jac[12]);
/* G <- G_lo + xi G_hi, c <- c_lo + xi^-1 c_hi, z <- z_lo + xi z_hi (pcdl.rs:216-224). */
int halo_ipa_round_fold(halo_ipa *st, const uint64_t xi[4], const uint64_t xi_inv[4]);
/* U = G[0], c = c[0] after lg n rounds (pcdl.rs:230-231). */
int halo_ipa_finish(halo_ipa *st, uint64_t U_jac[12], uint64_t c[4]);

#ifdef __cplusplus
}
#endif
#endif /* HALO_B200_H */
