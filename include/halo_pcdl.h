/*
 * halo_pcdl.h -- C view of the host layer above the CUDA ABI: the reference's public API for the hot
 * path, same names, argument meaning and error behaviour (code/src/pedersen.rs, pcdl.rs, acc.rs), with the
 * data-parallel work dispatched to libhalo_b200.so (include/halo_b200.h).
 *
 * The reference is Rust; no Rust toolchain exists in this image, so the host side is C++
 * (halo-accumulation_b200/host/ *.hpp, namespaces halo::pedersen / halo::pcdl / halo::acc) and this header
 * exposes it to C / ctypes for the parity tests and the benchmark.  A Rust build would keep its own
 * pcdl.rs / acc.rs and bind halo_b200.h directly (INTEGRATION.md).
 *
 * Randomness: the reference draws from `rng` inside open (pcdl.rs:141,146) and prover (acc.rs:192,198).
 * Here the caller passes those draws explicitly, in the reference's draw order, so that results are
 * reproducible and comparable bit for bit.
 *
 * Return value: HALO_OK (accept / success), a HALO_E* error (halo_b200.h) -- the analogue of the
 * reference's assert!/panic -- or a HALO_REJECT_* code -- the analogue of its `ensure!` Err.
 */
#ifndef HALO_PCDL_H
#define HALO_PCDL_H
#include "halo_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define HALO_MAX_LG 32

#define HALO_REJECT_SUCCINCT (-10) /* "C_(log_n) != CM.Commit_Sigma(c || v')"         pcdl.rs:307-310 */
#define HALO_REJECT_U (-11)        /* "U != CM.Commit(ck, h_vec)"                      pcdl.rs:339    */
#define HALO_REJECT_U0 (-12)       /* "U_0 != PCDL.Commit(ck, h_0; w = bot)"           acc.rs:152-155 */
#define HALO_REJECT_D (-13)        /* "d_i != d" / "d' = d"                            acc.rs:169,239 */
#define HALO_REJECT_CBAR (-14)     /* "C_bar' != C_bar"                                acc.rs:237     */
#define HALO_REJECT_Z (-15)        /* "z' = z"                                         acc.rs:238     */
#define HALO_REJECT_V (-17)        /* "h(z) = v"                                       acc.rs:240     */

/* pcdl.rs:22-30 EvalProof */
typedef struct {
    uint32_t lg_n;
    uint32_t hiding; /* C_bar / w_prime are Some(..) */
    uint64_t Ls[HALO_MAX_LG][12];
    uint64_t Rs[HALO_MAX_LG][12];
    uint64_t U[12];
    uint64_t c[4];
    uint64_t C_bar[12];
    uint64_t w_prime[4];
} halo_eval_proof;

/* acc.rs:21-28 Instance */
typedef struct {
    uint64_t C[12];
    uint64_t d;
    uint64_t z[4];
    uint64_t v[4];
    halo_eval_proof pi;
} halo_instance;

/* acc.rs:43-59 Accumulator with pi_V = AccumulatorHiding { h (degree 1), U, w } */
typedef struct {
    uint64_t C_bar[12];
    uint64_t d;
    uint64_t z[4];
    uint64_t v[4];
    halo_eval_proof pi;
    uint64_t h0[2][4];
    uint64_t U0[12];
    uint64_t w[4];
} halo_accumulator;

/* pedersen.rs:6-20  commit(w, Gs, ms); gs_affine == NULL means GS[0..n_gs) of the context. */
int halo_pedersen_commit(halo_ctx *ctx, const uint64_t *w /*nullable*/, const uint64_t *gs_affine, uint64_t n_gs,
                         const uint64_t *ms, uint64_t n_ms, uint64_t out_jac[12]);
/* pcdl.rs:99-110 */
int halo_pcdl_commit(halo_ctx *ctx, const uint64_t *coeffs, uint64_t n_coeffs, uint64_t d, const uint64_t *w /*nullable*/,
                     uint64_t out_jac[12]);
/* halo_pcdl_commit of k polynomials of one degree bound d (the reference has no batch form): polynomial j has n_coeffs[j]
 * coefficients, packed back to back in `coeffs`; ws holds w_j for every output (hiding) or is NULL.  The polynomials are
 * validated in order as commit does, and the first malformed one fails the call with HALO_EINVAL before any device work and
 * before any output is written.  One halo_msm_gens_many for all of them; the hiding terms w_j S in one combined step. */
int halo_pcdl_commit_batch(halo_ctx *ctx, const uint64_t *coeffs /*packed*/, const uint64_t *n_coeffs /*[k]*/, uint64_t k, uint64_t d,
                           const uint64_t *ws /*[k][4] or NULL*/, uint64_t *out_jac /*[k][12]*/);
/* K8: halo_pcdl_commit_batch of the k polynomials whose d + 1 evaluations over H_{d+1} are evals[j] (include/halo_b200.h K8):
 * one batched inverse transform (halo_poly_upload_evals), one segmented MSM over the resident coefficients
 * (halo_poly_commit_resident), then C_j + w_j S for the hiding ones in one combine.  d + 1 must be a power of two within the
 * resident generators (HALO_EINVAL, checked before any device work); every degree is <= d by construction.  k = 0 does nothing. */
int halo_pcdl_commit_evals(halo_ctx *ctx, const uint64_t *evals /*[k][d+1][4]*/, uint64_t k, uint64_t d, const uint64_t *ws /*[k][4] or NULL*/,
                           uint64_t *out_jac /*[k][12]*/);
/* pcdl.rs:120-242; hiding iff w != NULL, then q (n_q = deg p coefficients) and w_bar are the rng draws. */
int halo_pcdl_open(halo_ctx *ctx, const uint64_t *coeffs, uint64_t n_coeffs, const uint64_t C_jac[12], uint64_t d,
                   const uint64_t z[4], const uint64_t *w /*nullable*/, const uint64_t *q, uint64_t n_q,
                   const uint64_t *w_bar, halo_eval_proof *pi);
/* Batch opening at one point (an extension: the reference opens one polynomial at a time, DESIGN.md K3b).  For k >= 1
 * polynomials p_j of one degree bound d, packed as in halo_pcdl_commit_batch, their commitments C_j (as commit returns them,
 * C_j = commit(p_j) + w_j S) and one point z:
 *   v_j   = p_j(z)                                                  -> vs_out[j]
 *   alpha = rho_0(z, C_0, v_0, C_1, v_1, .., C_{k-1}, v_{k-1})      (tag 0; z, every v_j as a scalar, every C_j compressed)
 *   C = sum_j alpha^j C_j, v = sum_j alpha^j v_j                    -> C_out, v_out
 *   p = sum_j alpha^j p_j, and with ws: w = sum_j alpha^j w_j
 *   pi = halo_pcdl_open(p, C, d, z, w, q, w_bar)                    -> pi
 * (C, d, z, v, pi) is an ordinary PCDL claim: halo_pcdl_check, halo_pcdl_check_batch and the accumulation scheme take it
 * unchanged.  alpha binds every v_j.  If some p_j(z) != v_j, the combined claim is true for at most k - 1 values of alpha,
 * so a false batch passes with probability <= (k - 1) / r plus the soundness error of one PCDL check.
 * Hiding iff ws != NULL: then q holds n_q = max_j deg(p_j) coefficients (what is known before alpha exists; the opening
 * uses the first deg(p) of them, all of them unless the top coefficients cancel) and w_bar is the second draw.  k = 1 is
 * halo_pcdl_open itself, bit for bit (C = C_0, v = v_0).  The uploaded polynomials stay in the context's pooled buffer
 * (halo_poly_eval_many).
 * Returns HALO_EINVAL, before any device work and before any output is written, for k = 0, NULL pointers, the first
 * malformed polynomial in order (d + 1 not a power of two, deg > d, d >= the resident generators), a C_j off the curve or
 * not canonical, a w_j or z not canonical; HALO_ELEN for n_q != max_j deg(p_j) or deg = 0 with hiding (as open);
 * HALO_EINTERNAL when the opening's own p(z) differs from v (a bug, not a decision). */
int halo_pcdl_open_batch(halo_ctx *ctx, const uint64_t *coeffs /*packed*/, const uint64_t *n_coeffs /*[k]*/, uint64_t k,
                         const uint64_t *Cs /*[k][12]*/, uint64_t d, const uint64_t z[4], const uint64_t *ws /*[k][4] or NULL*/,
                         const uint64_t *q, uint64_t n_q, const uint64_t *w_bar, uint64_t *vs_out /*[k][4]*/, uint64_t C_out[12],
                         uint64_t v_out[4], halo_eval_proof *pi);
/* The verifier's side of halo_pcdl_open_batch: the claims (C_j, z, v_j) reduced to the one claim (C, v) above (alpha from the
 * same transcript), to be decided by halo_pcdl_check / _succinct_check / _check_batch or accumulated.  C_j = O (the zero
 * polynomial without hiding) is allowed.  HALO_EINVAL: k = 0, NULL pointers, a C_j off the curve or not canonical, a v_j or
 * z not canonical. */
int halo_pcdl_batch_claim(halo_ctx *ctx, const uint64_t *Cs /*[k][12]*/, const uint64_t *vs /*[k][4]*/, uint64_t k,
                          const uint64_t z[4], uint64_t C_out[12], uint64_t v_out[4]);
/* Batch opening at several points (an extension: the reference opens one polynomial at one point, DESIGN.md K3c; the
 * multi-point reduction of Halo 2, after Boneh-Drake-Fisch-Gabizon 2020).
 *
 * Inputs: k >= 1 polynomials p_0 .. p_{k-1} of one degree bound d, packed as in halo_pcdl_commit_batch; their commitments
 * C_j, as commit returns them; T >= 1 distinct points z_0 .. z_{T-1} (T <= HALO_MULTI_MAX_POINTS); m >= 1 queries
 * (j_i, t_i) = (q_poly[i], q_point[i]): polynomial j_i is opened at point z_{t_i}; optionally the blinding scalars w_j.
 * Every point and every polynomial must appear in at least one query, and no (j, t) pair may repeat.
 * All challenges use the transcript of host/group.hpp with tag 2 (rho_2), apart from PCDL's tag 0 and ASDL's tag 1; each
 * record is a u64 little-endian, a compressed point or a canonical scalar.
 *   1. v_i = p_{j_i}(z_{t_i}) for i < m                                                      -> vs_out[i]
 *   2. x1 = rho_2(u64 k, u64 T, u64 m, C_0 .. C_{k-1}, z_0 .. z_{T-1}, then for each query i: u64 j_i, u64 t_i, v_i)
 *   3. for each point t, over its queries in query order: f_t = sum_{i: t_i = t} x1^i p_{j_i}, v^_t = sum x1^i v_i,
 *      C^_t = sum x1^i C_{j_i}, w^_t = sum x1^i w_{j_i}
 *   4. x2 = rho_2(x1)
 *   5. q = sum_t x2^t (f_t - v^_t) / (X - z_t): exact division for honest claims, deg q <= d - 1.  The quotient of f_t by
 *      (X - z_t) does not depend on v^_t; the remainder of that division is f_t(z_t) and must equal v^_t.
 *   6. Q = commit(q, d, w_Q), the ordinary PCDL commitment (hiding with the caller's draw w_Q)       -> Q_out
 *   7. x3 = rho_2(x2, Q); if x3 equals some z_t the call fails with HALO_EINTERNAL (probability <= T / r)  -> x_out
 *   8. u_t = f_t(x3) for t < T                                                                 -> us_out[t]
 *   9. x4 = rho_2(x3, u_0 .. u_{T-1})
 *  10. the final claim: P = q + sum_t x4^(t+1) f_t = q + sum_j c_j p_j with c_j = sum_{i: j_i = j} x4^(t_i+1) x1^i;
 *      C = Q + sum_j c_j C_j; v = q^ + sum_t x4^(t+1) u_t with q^ = sum_t x2^t (u_t - v^_t) / (x3 - z_t);
 *      w = w_Q + sum_j c_j w_j when hiding                                                     -> C_out, v_out
 *  11. pi = halo_pcdl_open(P, C, d, x3, w, q_rand, w_bar), the opening unchanged               -> pi
 * (C, d, x3, v, pi) is an ordinary PCDL claim: halo_pcdl_check, halo_pcdl_check_batch and the accumulation scheme take it
 * unchanged.  The verifier's side is halo_pcdl_multi_claim.
 * Hiding applies iff ws != NULL; the caller's draws are, in order, w_Q, q_rand with n_q = max_j deg(p_j) coefficients (as
 * in halo_pcdl_open_batch; the opening takes the first deg(P) of them) and w_bar.
 * Soundness: if some v_i is false, then with probability >= 1 - (m - 1)/r over x1 some f_t(z_t) != v^_t; then with
 * probability >= 1 - (T - 1)/r over x2 the sum of step 5 has a pole and is no polynomial; Q is bound before x3; over x4 the
 * final claim forces q'(x3) = q^ and u_t = f_t(x3) for every t, except with probability T/r; and the committed q' agrees with
 * the rational function at x3 with probability at most (d + T)/r.  Total <= (m + 3T + d)/r plus the soundness error of one
 * PCDL check (DESIGN.md K3c).
 * Returns, before any device work and before any output is written: HALO_EINVAL for k, T or m = 0, NULL pointers, the first
 * malformed polynomial in order (as halo_pcdl_open_batch), a C_j off the curve or not canonical, a z_t, w_j, w_Q or w_bar
 * that is not canonical, duplicate points, a query index out of range, a duplicate (j, t) pair, an unused point or
 * polynomial; HALO_ELEN for n_q != max_j deg(p_j) or max deg = 0 with hiding.  HALO_EINTERNAL when a remainder differs from
 * v^_t or the opening's own P(x3) from v (bugs, not decisions), or x3 is one of the points. */
int halo_pcdl_open_multi(halo_ctx *ctx, const uint64_t *coeffs /*packed*/, const uint64_t *n_coeffs /*[k]*/, uint64_t k,
                         const uint64_t *Cs /*[k][12]*/, uint64_t d, const uint64_t *zs /*[T][4]*/, uint64_t T,
                         const uint64_t *q_poly /*[m]*/, const uint64_t *q_point /*[m]*/, uint64_t m,
                         const uint64_t *ws /*[k][4] or NULL*/, const uint64_t *w_Q, const uint64_t *q, uint64_t n_q,
                         const uint64_t *w_bar, uint64_t *vs_out /*[m][4]*/, uint64_t Q_out[12], uint64_t *us_out /*[T][4]*/,
                         uint64_t C_out[12], uint64_t x_out[4], uint64_t v_out[4], halo_eval_proof *pi);
/* K8: the same opening of k polynomials given in evaluation form (include/halo_b200.h K8): evals[j] holds p_j(omega^i),
 * i < d + 1, omega = omega_{d+1}.  The polynomials come from ONE batched inverse transform on the device
 * (halo_poly_upload_evals); everything after that is halo_pcdl_open_multi's code.  Hiding: q holds n_q = d coefficients, the
 * most any degree can be (halo_pcdl_open_multi: max_j deg p_j); the opening uses its first deg(P) <= max_j deg p_j, so the result
 * equals halo_pcdl_open_multi of the interpolated polynomials with q[0 .. max_j deg p_j) field by field.  Errors as
 * halo_pcdl_open_multi, with d + 1 a power of two and HALO_ELEN for n_q != d before any device work; a maximum degree of 0
 * with hiding is HALO_ELEN after the upload (the degrees are known only then), with nothing written. */
int halo_pcdl_open_multi_evals(halo_ctx *ctx, const uint64_t *evals /*[k][d+1][4]*/, uint64_t k, const uint64_t *Cs /*[k][12]*/,
                               uint64_t d, const uint64_t *zs /*[T][4]*/, uint64_t T, const uint64_t *q_poly /*[m]*/,
                               const uint64_t *q_point /*[m]*/, uint64_t m, const uint64_t *ws /*[k][4] or NULL*/, const uint64_t *w_Q,
                               const uint64_t *q /*[n_q][4]*/, uint64_t n_q, const uint64_t *w_bar, uint64_t *vs_out /*[m][4]*/,
                               uint64_t Q_out[12], uint64_t *us_out /*[T][4]*/, uint64_t C_out[12], uint64_t x_out[4], uint64_t v_out[4],
                               halo_eval_proof *pi);
/* The verifier's side of halo_pcdl_open_multi: recomputes x1 .. x4 and reduces the claims (C_j, z_t, v_i) with the prover's
 * Q and u_t to the one claim (C, x3, v) above (host arithmetic and one point_dot of k + 1 points), to be decided by
 * halo_pcdl_check / _check_batch or accumulated.  HALO_EINVAL as halo_pcdl_open_multi for the commitments, points and
 * queries, and for a v_i, u_t or Q that is not canonical; HALO_EINTERNAL when x3 is one of the points. */
int halo_pcdl_multi_claim(halo_ctx *ctx, const uint64_t *Cs /*[k][12]*/, uint64_t k, const uint64_t *zs /*[T][4]*/, uint64_t T,
                          const uint64_t *q_poly /*[m]*/, const uint64_t *q_point /*[m]*/, const uint64_t *vs /*[m][4]*/, uint64_t m,
                          const uint64_t Q[12], const uint64_t *us /*[T][4]*/, uint64_t C_out[12], uint64_t x_out[4],
                          uint64_t v_out[4]);
/* pcdl.rs:252-314; on accept writes the HPoly challenges xis[lg_n+1][4] and U. */
int halo_pcdl_succinct_check(halo_ctx *ctx, const uint64_t C_jac[12], uint64_t d, const uint64_t z[4], const uint64_t v[4],
                             const halo_eval_proof *pi, uint64_t *xis_out, uint64_t U_out[12]);
/* pcdl.rs:323-342 */
int halo_pcdl_check(halo_ctx *ctx, const uint64_t C_jac[12], uint64_t d, const uint64_t z[4], const uint64_t v[4],
                    const halo_eval_proof *pi);
/* Batch decider (an extension: the reference decides one claim at a time, DESIGN.md K5b).  Decides the k claims
 * (C, d, z, v, pi) -- each what halo_pcdl_check takes -- with ONE MSM over the generators: with the caller's rho != 0 the
 * succinct equations E_j (pcdl.rs:307-310) and the U checks F_j (pcdl.rs:339) of all claims are combined into
 *   sum_j (rho^2j E_j + rho^(2j+1) F_j) = O.
 * Honest claims satisfy it for every rho; if some E_j or F_j != O it holds for at most 2k - 1 values of rho, so a false
 * accept has probability <= (2k - 1) / r when rho is drawn after the claims are fixed (from a CSPRNG, or by hashing all k
 * claims).  rho is an explicit argument like every other random draw here.
 * Returns
 *   HALO_OK         accept, iff the combined point is O;
 *   HALO_REJECT_*   otherwise halo_pcdl_check runs on claims 0, 1, .. in order and the first reject is returned, with
 *                   *rejected_index = its claim: the (index, code) pair a loop of single checks returns;
 *   HALO_EINTERNAL  the combined equation failed but every claim accepts on its own (a bug, not a decision);
 *   HALO_EINVAL     before any decision, wherever the claim sits: a point or scalar of a claim that is not canonical / not
 *                   on the curve, d + 1 not a power of two, d >= the resident generators, a proof with the wrong number
 *                   of rounds, a zero challenge; rho = 0 or not canonical; claims / rho / rejected_index NULL with k > 0.
 * k = 0 accepts and reads no other argument.  *rejected_index is written on a reject only. */
int halo_pcdl_check_batch(halo_ctx *ctx, const halo_instance *claims, uint64_t k, const uint64_t rho[4],
                          uint64_t *rejected_index);
/* HPoly::eval pcdl.rs:79-91 */
int halo_h_eval(const uint64_t *xis, uint32_t lg_n, const uint64_t z[4], uint64_t out[4]);

/* acc.rs:190-220; draws in order: h0 (2 coefficients), w, then open's q and w_bar. */
int halo_acc_prover(halo_ctx *ctx, uint64_t d, const halo_instance *qs, uint64_t m, const uint64_t h0[2][4],
                    const uint64_t w[4], const uint64_t *q, uint64_t n_q, const uint64_t w_bar[4], halo_accumulator *acc);
/* acc.rs:223-243 */
int halo_acc_verifier(halo_ctx *ctx, uint64_t d, const halo_instance *qs, uint64_t m, const halo_accumulator *acc);
/* acc.rs:245-255 */
int halo_acc_decider(halo_ctx *ctx, const halo_accumulator *acc);
/* halo_pcdl_check_batch over (C_bar, d, z, v, pi) of each accumulator (the claim of acc.rs:254), same results and errors;
 * every accumulator is validated like halo_acc_decider's. */
int halo_acc_decider_batch(halo_ctx *ctx, const halo_accumulator *accs, uint64_t k, const uint64_t rho[4],
                           uint64_t *rejected_index);
/* Batch verifier (an extension: the reference verifies one accumulation step at a time, DESIGN.md K5c).  Verifies the k
 * steps (qs_i, accs[i]) against D -- each what halo_acc_verifier takes, step i owning the next ms[i] instances of qs -- with
 * ONE variable-base MSM: with the caller's rho != 0 the group equations of all steps, in the order
 *   A_i = U0_i - h0_i[0] G_0 - h0_i[1] G_1                        (acc.rs:152-155)
 *   E_ij = the succinct equation of instance j                    (pcdl.rs:307-310), j = 1 .. ms[i]
 *   B_i = sum_{j=0..m_i} alpha_i^j U_ij + omega_i S - C_bar_i     (acc.rs:178, :184, :237; U_i0 = U0_i, omega_i = accs[i].w)
 * for i = 0, 1, .., are combined into sum_t rho^t X_t = O over T = sum_i (ms[i] + 2) equations; the host checks d_ij = D,
 * d_i = D, z_i = rho_1(C_bar_i - omega_i S, alpha_i) and h_i(z_i) = v_i.  Honest steps pass for every rho; if some equation
 * != O the sum is O for at most T - 1 values of rho, so a false accept has probability <= (T - 1) / r when rho is drawn after
 * the steps are fixed (from a CSPRNG, or by hashing all steps).
 * Returns
 *   HALO_OK         accept, iff the combined point is O and every host check holds;
 *   HALO_REJECT_*   otherwise halo_acc_verifier runs on steps 0, 1, .. in order and the first reject is returned, with
 *                   *rejected_index = its step: the (index, code) pair a loop of single verifiers returns;
 *   HALO_EINTERNAL  the combined check failed but every step accepts on its own (a bug, not a decision);
 *   HALO_EINVAL     before any decision, wherever the step sits: a point or scalar that is not canonical / not on the
 *                   curve, d + 1 or D + 1 not a power of two, d or D >= the resident generators, a proof with the wrong
 *                   number of rounds, a zero challenge, h_0 of degree > D; rho = 0 or not canonical; qs / ms / accs / rho /
 *                   rejected_index NULL with k > 0 (qs may be NULL when every ms[i] is 0).
 * k = 0 accepts and reads no other argument.  *rejected_index is written on a reject only. */
int halo_acc_verifier_batch(halo_ctx *ctx, uint64_t d, const halo_instance *qs /*[sum ms]*/, const uint64_t *ms /*[k]*/,
                            const halo_accumulator *accs /*[k]*/, uint64_t k, const uint64_t rho[4], uint64_t *rejected_index);
/* Batch verify-and-decide (DESIGN.md K5d): halo_acc_verifier_batch(d, qs, ms, steps_accs, k) followed by
 * halo_acc_decider_batch(decide_accs, k_dec) in ONE call, with the same decisions and errors as that pair.  The combined
 * equation is the T_v = sum_i (ms[i] + 2) equations of the steps, in the order of halo_acc_verifier_batch, followed by the
 * pair E_j, F_j of halo_acc_decider_batch for each decided accumulator, the powers of rho running on across the boundary;
 * a false accept has probability <= (T - 1) / r, T = T_v + 2 k_dec, when rho is drawn after both lists are fixed.  The
 * generator MSM of the decided accumulators runs on the device while the steps' transcripts run on the host.
 * Returns
 *   HALO_OK         accept, iff the combined point is O and every host check of every step holds;
 *   HALO_REJECT_*   otherwise halo_acc_verifier runs on steps 0, 1, .., then halo_acc_decider on the decided accumulators
 *                   0, 1, .., and the first reject is returned with *rejected_index = its position in the sequence "steps,
 *                   then decided accumulators": step i is i, decided accumulator j is k + j;
 *   HALO_EINTERNAL  the combined check failed but every item accepts on its own (a bug, not a decision);
 *   HALO_EINVAL     before any decision, for malformed input anywhere in either list (what either batch call refuses), the
 *                   error of the first malformed item in the same order; rho = 0 or not canonical; ms / steps_accs NULL with
 *                   k > 0, decide_accs NULL with k_dec > 0, rho / rejected_index NULL.
 * k = k_dec = 0 accepts and reads no other argument.  A decided accumulator may also be one of the steps' accumulators. */
int halo_acc_verify_decide_batch(halo_ctx *ctx, uint64_t d, const halo_instance *qs /*[sum ms]*/, const uint64_t *ms /*[k]*/,
                                 const halo_accumulator *steps_accs /*[k]*/, uint64_t k, const halo_accumulator *decide_accs /*[k_dec]*/,
                                 uint64_t k_dec, const uint64_t rho[4], uint64_t *rejected_index);
/* impl From<Accumulator> for Instance, acc.rs:121-131 */
void halo_acc_to_instance(const halo_accumulator *acc, halo_instance *q);

/* Fiat-Shamir helpers exposed for the parity tests (group.rs:41-89). */
void halo_point_serialize_compressed(const uint64_t p_jac[12], uint8_t out[33]);

#ifdef __cplusplus
}
#endif
#endif /* HALO_PCDL_H */
