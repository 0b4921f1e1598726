/*
 * halo_b200_test.h -- test hooks exported by libhalo_b200.so so the parity suite can exercise the
 * device field core (K1) and group law in isolation against the oracle.  Not part of the drop-in
 * boundary; a Rust shim never binds these.
 */
#ifndef HALO_B200_TEST_H
#define HALO_B200_TEST_H
#include "halo_b200.h"
#ifdef __cplusplus
extern "C" {
#endif
/* Element-wise field op on the device: which = 0 (coordinate field Fq) / 1 (scalar field Fr) of the build's curve; op = 0 mul, 1 add, 2 sub, 3 sqr, 4 inv,
 * 5 neg, 6 to_canonical, 7 from_canonical.  a, b, out: host arrays of n elements (uint64_t[4] each). */
int halo_test_fp_op(halo_ctx *ctx, int which, int op, const uint64_t *a, const uint64_t *b, uint64_t *out, uint64_t n);
/* Single device thread: sum_i (neg[i] ? -P_i : P_i) over affine points via mixed adds -> Jacobian. */
int halo_test_madd_chain(halo_ctx *ctx, const uint64_t *affine /*[n][8]*/, const uint8_t *neg, uint64_t n,
                         uint64_t out_jac[12]);
/* Single device thread: sum of Jacobian points via full XYZZ adds followed by `dbls` doublings. */
int halo_test_add_chain(halo_ctx *ctx, const uint64_t *jac /*[n][12]*/, uint64_t n, int dbls, uint64_t out_jac[12]);
/* Modular-multiplication throughput microbenchmark (K1): `iters` dependent Fq multiplications per thread
 * on blocks x threads threads; returns elapsed ms and a checksum limb. */
int halo_test_fp_mul_throughput(halo_ctx *ctx, int blocks, int threads, int iters, int ilp, float *ms, uint64_t *checksum);
/* Integer-pipe peak microbenchmark: 16 independent multiply-add chains per thread whose multiplicand is the running
 * accumulator (nothing is loop invariant).  kind 0 = mad.lo.u32 (IMAD), 1 = mad.wide.u32 (IMAD.WIDE), 2 = mad.hi.u32
 * (IMAD.HI): ops = blocks * threads * iters * 16.  kinds 3-7: carry-chain forms, 8 (7: 16) ops per iteration. */
int halo_test_imad_throughput(halo_ctx *ctx, int kind, int blocks, int threads, int iters, float *ms, uint64_t *checksum);
/* Every device buffer of the library is allocated with a 256-byte canary behind its end.  Returns the number of live
 * buffers whose canary was overwritten (0 = no kernel wrote past a buffer); *live_buffers = how many were checked. */
int halo_test_check_canaries(int *live_buffers);
/* Route of the last MSM enqueued on `lane` (0: the context's stream; 1: the second stream of two-lane batches and of the
 * companion MSM of halo_h_msm_batch), as the host code chose it from the plan, the size and halo_set_tuning:
 *   out[0] window c            out[1] 1 = FIXED base, 0 = variable base     out[2] P, pair-tree passes (after the clamp to 8)
 *   out[3] pass-0 kernel of the pair tree: 1 = k_pair_bwd0 (cp.async), 0 = k_pair_bwd<true> (per-lane gathers), -1 = P == 0
 *   out[4] accumulation kernel: 2 = k_accumulate_quad, 1 = k_accumulate_static, 0 = k_accumulate (lane claiming)
 *   out[5] lanes per bucket and out[6] CTAs per SM of k_accumulate_quad (0 for the other kernels)
 *   out[7] grid of k_accumulate (0 for the other kernels)
 *   out[8] bucket reduction: 1 = k_reduce_slabs_quad, 0 = k_reduce_slabs (one lane per addition)
 *   out[9] 1 / 0: the msm_batch that enqueued it ran on two lanes / one; -1: enqueued outside msm_batch
 * Reading clears the record (out[0] = 0 until the next MSM on that lane).  Host bookkeeping only: no kernel, launch or device
 * memory. */
int halo_test_msm_route(halo_ctx *ctx, int lane, int out[10]);
/* Random-gather ceiling of HBM: blocks * threads threads each read `iters` pseudo-random 64-byte-aligned slots (16, 32 or
 * 64 bytes of each; bytes = -64: four adjacent lanes fetch one 64-byte slot with one instruction, blocks * threads / 4 *
 * iters gathers; bytes = -32: two adjacent lanes fetch one 32-byte slot, blocks * threads / 2 * iters gathers) of a table of
 * `table_bytes` bytes; ms = best of 2 timed launches.  The denominator for the first
 * pair-tree pass and for the gathers of k_accumulate (DESIGN.md, K2b). */
int halo_test_gather_throughput(halo_ctx *ctx, uint64_t table_bytes, int blocks, int threads, int iters, int bytes, float *ms);
/* Times one HBM-bound Fr vector kernel on synthetic device-resident data (ms, best of 5): kind 0 = the c / z folds of
 * one IPA round over 2 x n/2 outputs (pcdl.rs:221-223), 1 = h-expansion to 2^floor(lg n) coefficients (pcdl.rs:56-77),
 * 2 = dot product of two n-vectors (group.rs:13-15), 3 = powers of z (group.rs:29-37). */
int halo_test_vec_bench(halo_ctx *ctx, int kind, uint64_t n, float *ms);
/* Times k_h_lincomb (DESIGN.md K5b) over k claims of 2^lg_n coefficients each, lg_n <= 30 (ms, best of 5, CUDA events; the
 * copy of the claim descriptors included). */
int halo_test_h_lincomb_bench(halo_ctx *ctx, uint32_t lg_n, uint64_t k, float *ms);
/* Host-side GLV decomposition of a challenge used by the generator fold (K4): xi = k1 + k2 * lambda (mod r), written in
 * joint sparse form (digits in {0, +-1}, LSB first; at most half of the positions non-zero on average).  Runs without a GPU. */
int halo_test_glv_decompose_jsf(const uint64_t xi[4], int8_t d1[136], int8_t d2[136], int *top);
/* K5c (DESIGN.md): R_o = P_o + a_o Q_o + b_o S for o < n, S of the context's parameters, each exact, returned affine
 * (out_affine[n][8], infinity = (0, 0)).  P, Q: Jacobian [n][12]; a, b: [n][4].  path 1: k_point_combine, one launch for all
 * outputs (GLV + joint sparse form digits written on the host); 0: host GLV on up to 16 threads; -1: the device from
 * "combine_min_outputs" outputs on (halo_set_tuning), the host below.
 * Unlike the other hooks this one is load-bearing: the batch checks of libhalo_host.so (halo_pcdl_check_batch,
 * halo_acc_decider_batch, halo_acc_verifier_batch) take every C' and C* through it with path -1.  It stays out of
 * halo_b200.h because only that library calls it; removing or changing it breaks those entry points. */
int halo_test_point_combine(halo_ctx *ctx, int path, const uint64_t *P_jac, const uint64_t *Q_jac, const uint64_t *a,
                            const uint64_t *b, uint64_t n, uint64_t *out_affine);
/* K3c: *n_out = the number of coefficients of the quotient q that the last halo_poly_quotient left on the device; when
 * cap >= *n_out they are copied to out[*n_out][4] (Montgomery limbs).  HALO_ESTATE: no quotient of the current upload. */
int halo_test_read_quotient(halo_ctx *ctx, uint64_t *out, uint64_t cap, uint64_t *n_out);
#ifdef __cplusplus
}
#endif
#endif
