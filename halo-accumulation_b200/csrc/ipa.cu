// ipa.cu -- K3/K4/K7: the IPA rounds of PCDL.open on the device.
//
// Replaces the loop body pcdl.rs:195-227.  Per round, with m = cur / 2:
//   K3  dot_l = <c_hi, z_lo>, dot_r = <c_lo, z_hi>                       (group.rs:13-15, pcdl.rs:203,207)
//       L = <c_hi, G_lo> + dot_l H',  R = <c_lo, G_hi> + dot_r H'        (pcdl.rs:204,208) -- two Pippenger MSMs
//       whose H' term rides along as a one-element tail, enqueued back to back with one synchronisation
//   K4  G_j <- G_j + xi G_{j+m}   (shared-scalar multiply-add, signed NAF digits of xi broadcast to all
//       threads -> divergence-free), c_j <- c_j + xi^-1 c_{j+m}, z_j <- z_j + xi z_{j+m}   (pcdl.rs:216-224)
//   K7  the folded generators are normalised back to affine inside the fold kernel so every later MSM keeps the
//       8M+2S mixed addition (the reference instead pays one inversion per element per MSM, group.rs:19).
// Folds and MSM rounds stay on one GPU by design (sequential rounds with a hash between them, pcdl.rs:212).
#include "ipa.cuh"

#include <cstring>
#include <functional>

#include "../../include/halo_b200.h"
#include "glv.cuh"
#include "msm.cuh"
#include "vec.cuh"

using namespace halo;

namespace halo {

// This file is compiled twice (see ipa_fold.cu): the second unit holds only k_fold_multi, under the name k_fold_multi_call and
// with the field multiplication as an out-of-line call, for folds with many outputs.
#ifndef HALO_FOLD_MIN_BLOCKS
#define HALO_FOLD_MIN_BLOCKS 3  // 4 CTAs per SM (128 registers) spills and measures 10 % slower
#endif
#ifndef HALO_IPA_FOLD_TU

#ifndef HALO_IPA_FREEZE_LEN
#define HALO_IPA_FREEZE_LEN 8192
#endif
constexpr uint64_t IPA_FREEZE_LEN = HALO_IPA_FREEZE_LEN;

// ---- GLV: xi * P = k1 * P + k2 * phi(P), phi(x, y) = (beta x, y) = lambda * P, |k1|, |k2| < 2^129 ------------------
// Pallas has j-invariant 0, so Fq contains a primitive cube root of unity beta and Fr the matching lambda
// (lambda * (x, y) = (beta x, y); pair fixed by checking lambda * G on the generator).  The shared challenge of a
// round is decomposed once on the host (Babai rounding against the reduced basis (a1, b1), (a2, b2) of the lattice
// {(a, b): a + b lambda = 0 mod r}); the kernel then needs 129 doublings instead of 255.

__device__ __constant__ uint32_t c_beta_mont[8] = HALO_GLV_BETA_MONT;  // glv.cuh

// K4 point part: G[j] <- affine(G[j] + xi * G[j + m]) with xi = k1 + k2 lambda is the D = 1 case of k_fold_multi below
// (joint digit loop uniform across the grid: same xi for every element of a round).  The sum is left in XYZZ coordinates
// with den[j] = ZZ * ZZZ (1 for infinity); the normalisation shares its inversions across the whole round (batch_invert:
// 3 multiplications per element instead of a 255-squaring Fermat chain each) and k_fold_finish writes the affine point
// back (K7).
// x = X / ZZ = X * ZZZ * inv, y = Y / ZZZ = Y * ZZ * inv with inv = 1 / (ZZ * ZZZ)
__global__ void __launch_bounds__(128) k_fold_finish(const xyzz_t* __restrict__ sums, const fq_t* __restrict__ inv, uint64_t m,
                                                     affine_t* __restrict__ G) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    xyzz_t p = sums[j];
    affine_t out;
    if (xyzz_is_inf(p)) {
        affine_set_inf(out);
    } else {
        fq_t i = inv[j], t;
        fp_mul(t, i, p.zzz);
        fp_mul(out.x, p.x, t);
        fp_mul(t, i, p.zz);
        fp_mul(out.y, p.y, t);
    }
    G[j] = out;
}

// ---- deferred head: several fold rounds in one joint pass ---------------------------------------------------------------
// Folding round by round pays ~129 doublings per element per round.  When the first D rounds are deferred (their L / R
// are MSMs over the untouched generators with per-index coefficients, like the frozen tail below), the generator vector
// after round D - 1 is, for j < n / 2^D,
//     G^(D)_j = sum_{t < 2^D} s_t G_{j + off_t},   s_t = prod_k xi_k^{bit_k(t)},   off_t = sum_k bit_k(t) n / 2^(k+1)
// (pcdl.rs:216-218 unrolled D times), a 2^D-term multi-scalar multiplication with SHARED scalars: one joint
// double-and-add (Straus) pays the 129 doublings once per output instead of once per term.  The host decomposes every
// s_t by GLV (k1, k2), writes each pair in joint sparse form (half of the positions carry an addition instead of two
// thirds for separate NAFs; the combinations P +- phi(P) are one free point and one precomputed affine point per
// term), merges all terms into one operation list (uniform across the grid, so the loop is divergence free) and uploads it.
constexpr int FOLD_MAX_DEFER = 4;
constexpr int FOLD_MAX_OPS = 3072;
// The operation list is per CONTEXT (halo_ctx::fold_ops on the host, halo_ctx::ipa_ops on the device): two contexts may run
// openings concurrently from two host threads, on the same device or not (INTEGRATION.md "threading"), so neither a
// process-wide host buffer nor a __constant__ symbol (one per device, shared by every stream) may hold it.  The kernel
// reads it with uniform addresses (one L1 broadcast per operation, negligible beside the ~10 multiplications that follow).
static_assert(FOLD_MAX_OPS == sizeof(halo::FoldOpsHost::code), "halo_ctx::fold_ops capacity");

#endif  // HALO_IPA_FOLD_TU

__device__ __forceinline__ uint64_t fold_term_offset(uint64_t n, int D, int t) {
    uint64_t off = 0;
    for (int k = 0; k < D; k++)
        if ((t >> k) & 1) off += n >> (k + 1);
    return off;
}
#ifndef HALO_IPA_FOLD_TU
// Per term t >= 1 and output j: beta x (so phi(P) = (beta x, y)) and the denominator x - beta x of P - phi(P); the joint
// sparse form below adds P, phi(P), P + phi(P) = (-(x + beta x), -y) [= -phi^2(P), free] or P - phi(P) [one affine
// addition per term, inversions shared by batch_invert].
__global__ void __launch_bounds__(128) k_fold_prep1(const affine_t* __restrict__ G0, uint64_t n, int D, fq_t* __restrict__ bx,
                                                    fq_t* __restrict__ den) {
    const uint64_t m = n >> D;
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int t = blockIdx.y + 1;
    if (j >= m) return;
    fq_t beta;
#pragma unroll
    for (int i = 0; i < 8; i++) beta.v[i] = c_beta_mont[i];
    const affine_t p = G0[j + fold_term_offset(n, D, t)];
    fq_t r, d;
    fp_mul(r, p.x, beta);
    fp_sub(d, p.x, r);
    if (fp_is_zero(d)) fp_one(d);  // infinity, or x = 0 (then phi(P) = P and the difference is infinity): no inversion
    bx[(uint64_t)(t - 1) * m + j] = r;
    den[(uint64_t)(t - 1) * m + j] = d;
}
__global__ void __launch_bounds__(128) k_fold_prep2(const affine_t* __restrict__ G0, uint64_t n, int D, const fq_t* __restrict__ bx,
                                                    const fq_t* __restrict__ inv, affine_t* __restrict__ diff) {
    const uint64_t m = n >> D;
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int t = blockIdx.y + 1;
    if (j >= m) return;
    const affine_t p = G0[j + fold_term_offset(n, D, t)];
    const fq_t b = bx[(uint64_t)(t - 1) * m + j];
    affine_t out;
    fq_t d;
    fp_sub(d, p.x, b);
    if (affine_is_inf(p) || fp_is_zero(d)) {
        affine_set_inf(out);
    } else {  // (x, y) + (beta x, -y): lambda = (-y - y) / (beta x - x) = 2 y / (x - beta x)
        fq_t lam, t1;
        fp_dbl(t1, p.y);
        fp_mul(lam, t1, inv[(uint64_t)(t - 1) * m + j]);
        fp_sqr(t1, lam);
        fp_sub(t1, t1, p.x);
        fp_sub(out.x, t1, b);
        fp_sub(t1, p.x, out.x);
        fp_mul(t1, lam, t1);
        fp_sub(out.y, t1, p.y);
    }
    diff[(uint64_t)(t - 1) * m + j] = out;
}

#endif  // HALO_IPA_FOLD_TU

// op code: 0xff = double; else (t - 1) | kind << 4 | sign << 7 with kind 0: P_t, 1: phi(P_t), 2: P_t + phi(P_t), 3: P_t - phi(P_t)
#ifdef HALO_IPA_FOLD_TU
#define k_fold_multi k_fold_multi_call
#endif
__global__ void __launch_bounds__(128, HALO_FOLD_MIN_BLOCKS) k_fold_multi(const affine_t* __restrict__ G0, uint64_t n, int D,
                                                                         const fq_t* __restrict__ bx,
                                                                         const affine_t* __restrict__ diff,
                                                                         const uint8_t* __restrict__ ops, int n_ops,
                                                                         xyzz_t* __restrict__ sums, fq_t* __restrict__ den) {
    const uint64_t m = n >> D;
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    xyzz_t acc;
    xyzz_set_inf(acc);
#pragma unroll 1
    for (int o = 0; o < n_ops; o++) {
        const uint32_t code = __ldg(ops + o);
        if (code == 0xffu) {
            xyzz_dbl(acc, acc);
        } else {
            const int t = (int)(code & 0xf) + 1, kind = (code >> 4) & 3;
            bool neg = (code >> 7) != 0;
            const uint64_t slot = (uint64_t)(t - 1) * m + j;
            affine_t p;
            if (kind == 3) {
                p = diff[slot];
            } else {
                p = G0[j + fold_term_offset(n, D, t)];
                if (kind != 0 && !affine_is_inf(p)) {
                    const fq_t b = bx[slot];
                    if (kind == 1) {
                        p.x = b;
                    } else {  // P + phi(P) = (-(x + beta x), -y)
                        fq_t sx;
                        fp_add(sx, p.x, b);
                        fp_neg(p.x, sx);
                        neg = !neg;
                    }
                }
            }
            xyzz_madd(acc, p, neg);
        }
    }
    affine_t lo = G0[j];
    xyzz_madd(acc, lo, false);
    sums[j] = acc;
    fq_t d;
    if (xyzz_is_inf(acc))
        fp_one(d);
    else
        fp_mul(d, acc.zz, acc.zzz);
    den[j] = d;
}

#ifdef HALO_IPA_FOLD_TU
#undef k_fold_multi
void launch_fold_multi_call(cudaStream_t st, unsigned grid, const affine_t* G0, uint64_t n, int D, const fq_t* bx, const affine_t* diff,
                            const uint8_t* ops, int n_ops, xyzz_t* sums, fq_t* den) {
    k_fold_multi_call<<<grid, 128, 0, st>>>(G0, n, D, bx, diff, ops, n_ops, sums, den);
}
}  // namespace halo
#else  // the rest of the file belongs to the normal unit

// ---- frozen tail: once the vectors are short the generators stop being folded -------------------------------------
// Folding m elements costs one ~2300-modmul serial chain per element no matter how small m is (about a millisecond of
// latency per round), so for the last rounds the generator vector is frozen at G0 = G^(r0) (M0 elements) and only the
// coefficient s_j with which G0_j enters the current folded generator is tracked (s_j <- xi s_j when j falls in the high
// half, pcdl.rs:218 unrolled).  Then, with cur the logical length and m = cur / 2,
//   L = <c_hi, G_lo> = sum_{j: j mod cur <  m} c[(j mod cur) + m] s_j G0_j ,
//   R = <c_lo, G_hi> = sum_{j: j mod cur >= m} c[(j mod cur) - m] s_j G0_j ,   U = sum_j s_j G0_j
// are MSMs over the fixed affine vector G0: same group elements as folding, without the folds.
__global__ void __launch_bounds__(256) k_frozen_scalars(const fr_t* __restrict__ c, const fr_t* __restrict__ s, uint32_t M0,
                                                        uint32_t cur, fr_t* __restrict__ tL, fr_t* __restrict__ tR) {
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= M0) return;
    const uint32_t m = cur >> 1, jj = j & (cur - 1);
    fr_t zero, v;
    fp_zero(zero);
    if (jj < m) {
        fp_mul(v, c[jj + m], s[j]);
        tL[j] = v;
        tR[j] = zero;
    } else {
        fp_mul(v, c[jj - m], s[j]);
        tL[j] = zero;
        tR[j] = v;
    }
}
__global__ void __launch_bounds__(256) k_frozen_fold_s(fr_t* __restrict__ s, uint32_t M0, uint32_t cur, fr_t xi) {
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= M0) return;
    if ((j & (cur - 1)) >= (cur >> 1)) {
        fr_t v = s[j];
        fp_mul(v, v, xi);
        s[j] = v;
    }
}
__global__ void __launch_bounds__(256) k_fill_one(fr_t* __restrict__ s, uint32_t n) {
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    fr_t one;
    fp_one(one);
    s[j] = one;
}

// ---- host: decomposition and joint sparse form: glv.cuh ---------------------------------------------------------------

}  // namespace halo

namespace halo {
// Materialises G^(D) from the untouched generators after D deferred rounds (see k_fold_multi).
// src: the vector being folded (n elements), xis: the D challenges, oldest first.  D = 1 is the ordinary round.
static void fold_multi(halo_ctx* ctx, const affine_t* src, uint64_t n, const fr_t* xis, int D) {
    const int T = 1 << D;
    const uint64_t m = n >> D;
    // s_t = prod_k xi_k^{bit_k(t)}
    std::vector<fr_t> coef(T);
    fp_one(coef[0]);
    for (int t = 1; t < T; t++) {
        int k = 31 - __builtin_clz((unsigned)t);  // highest set bit: s_t = s_{t - 2^k} * xi_k
        fp_mul(coef[t], coef[t ^ (1 << k)], xis[k]);
    }
    std::vector<GlvDigits> dg(T);
    int top = -1;
    for (int t = 1; t < T; t++) {
        make_glv_jsf(coef[t], dg[t]);
        if (dg[t].top > top) top = dg[t].top;
    }
    FoldOpsHost& ops = ctx->fold_ops;  // one opening per context at a time; the copy below is staged before the call returns
    int no = 0;
    if ((top + 1) * T > FOLD_MAX_OPS) throw CudaError{cudaErrorInvalidValue, "fold_multi: operation list too long", __FILE__, __LINE__};
    for (int i = top; i >= 0; i--) {
        ops.code[no++] = 0xff;
        for (int t = 1; t < T; t++) {
            const int d1 = dg[t].d1[i], d2 = dg[t].d2[i];
            if (!d1 && !d2) continue;
            int kind, neg;
            if (d1 && !d2) kind = 0, neg = d1 < 0;
            else if (!d1 && d2) kind = 1, neg = d2 < 0;
            else if (d1 == d2) kind = 2, neg = d1 < 0;
            else kind = 3, neg = d1 < 0;  // d1 = -d2: +-(P - phi(P))
            ops.code[no++] = (uint8_t)((t - 1) | (kind << 4) | (neg ? 0x80 : 0));
        }
    }
    ctx->ipa_ops.reserve(FOLD_MAX_OPS);
    HALO_CUDA(cudaMemcpyAsync(ctx->ipa_ops.p, ops.code, (size_t)no, cudaMemcpyHostToDevice, ctx->stream));
    ctx->ipa_bx.reserve((size_t)(T - 1) * m * sizeof(fq_t));
    ctx->ipa_diff.reserve((size_t)(T - 1) * m * sizeof(affine_t));
    ctx->ipa_den2.reserve((size_t)(T - 1) * m * sizeof(fq_t));
    ctx->ipa_sums.reserve(m * sizeof(xyzz_t));
    ctx->ipa_den.reserve(m * sizeof(fq_t));
    const affine_t* G0 = src;
    const dim3 pgrid((unsigned)((m + 127) / 128), (unsigned)(T - 1));
    k_fold_prep1<<<pgrid, 128, 0, ctx->stream>>>(G0, n, D, ctx->ipa_bx.as<fq_t>(), ctx->ipa_den2.as<fq_t>());
    batch_invert(ctx, ctx->stream, ctx->ipa_den2.as<fq_t>(), (uint32_t)((T - 1) * m), ctx->ipa_inv_scratch);
    k_fold_prep2<<<pgrid, 128, 0, ctx->stream>>>(G0, n, D, ctx->ipa_bx.as<fq_t>(), ctx->ipa_den2.as<fq_t>(), ctx->ipa_diff.as<affine_t>());
    // Many outputs: the copy of the kernel with the multiplication out of line (ipa_fold.cu).  The loop body inlines a doubling
    // and a mixed addition behind four kinds of operand selection, ~75 KiB of code that every warp walks at its own pace; out of
    // line the 2^17-output joint fold of an opening at 2^20 takes 12.7 instead of 15.0 ms, while folds of <= 2^15 outputs
    // (latency bound, a warp or two per SM) are 5-10 % faster inlined (profiles/r02_fold_multi_call_ab.txt).
    if (ctx->tune_fold_call_min_lg >= 0 && m >= ((uint64_t)1 << ctx->tune_fold_call_min_lg))
        launch_fold_multi_call(ctx->stream, (unsigned)((m + 127) / 128), G0, n, D, ctx->ipa_bx.as<fq_t>(), ctx->ipa_diff.as<affine_t>(),
                               ctx->ipa_ops.as<uint8_t>(), no, ctx->ipa_sums.as<xyzz_t>(), ctx->ipa_den.as<fq_t>());
    else
        k_fold_multi<<<(unsigned)((m + 127) / 128), 128, 0, ctx->stream>>>(G0, n, D, ctx->ipa_bx.as<fq_t>(), ctx->ipa_diff.as<affine_t>(),
                                                                           ctx->ipa_ops.as<uint8_t>(), no,
                                                                           ctx->ipa_sums.as<xyzz_t>(), ctx->ipa_den.as<fq_t>());
    batch_invert(ctx, ctx->stream, ctx->ipa_den.as<fq_t>(), (uint32_t)m, ctx->ipa_inv_scratch);
    k_fold_finish<<<(unsigned)((m + 127) / 128), 128, 0, ctx->stream>>>(ctx->ipa_sums.as<xyzz_t>(), ctx->ipa_den.as<fq_t>(), m,
                                                                        ctx->ipa_G.as<affine_t>());
    ctx->kernel_launches += 4;
    HALO_CUDA(cudaGetLastError());
}
}  // namespace halo

extern "C" int halo_test_glv_decompose_jsf(const uint64_t xi[4], int8_t d1[136], int8_t d2[136], int* top) {
    fr_t x;
    memcpy(&x, xi, 32);
    GlvDigits dg;
    make_glv_jsf(x, dg);
    memcpy(d1, dg.d1, 136);
    memcpy(d2, dg.d2, 136);
    *top = dg.top;
    return 0;
}

#define IPA_TRY(st)  \
    halo_ctx* ctx = (st)->ctx; \
    try {             \
        HALO_CUDA(cudaSetDevice(ctx->device));
#define IPA_CATCH                                           \
    }                                                       \
    catch (const halo::CudaError& e) {                      \
        ctx->last_error = std::string("CUDA error: ") + cudaGetErrorString(e.err) + " (" + e.what + ")"; \
        return HALO_ECUDA;                                  \
    }                                                       \
    catch (...) { /* nothing unwinds across the C ABI */    \
        ctx->last_error = "unexpected internal exception";  \
        return HALO_ECUDA;                                  \
    }                                                       \
    return HALO_OK;

static inline bool is_pow2(uint64_t n) { return n && !(n & (n - 1)); }

extern "C" {

static int ipa_begin_impl(halo_ctx* ctx, const uint64_t* coeffs, bool resident, uint64_t n_coeffs, uint64_t n, const uint64_t z[4],
                          halo_ipa** out, uint64_t v_out[4]) {
    if (!ctx || !out || !z || (!coeffs && !resident && n_coeffs)) return HALO_EINVAL;
    *out = nullptr;
    if (!is_pow2(n) || n > ctx->n_gens || n_coeffs > n) {  // pcdl.rs:128-132
        ctx->last_error = "halo_ipa_begin: n must be a power of two <= resident generators and >= n_coeffs";
        return HALO_EINVAL;
    }
    if (ctx->ipa_busy) {
        ctx->last_error = "halo_ipa_begin: another opening is in flight on this context";
        return HALO_ESTATE;
    }
    halo_ipa* st = new halo_ipa();
    st->ctx = ctx;
    try {
        HALO_CUDA(cudaSetDevice(ctx->device));
        st->n = st->cur = n;
        while (((uint64_t)1 << st->lg_n) < n) st->lg_n++;
        // deferred head (k_fold_multi): pays when the L / R of the deferred rounds can take the FIXED-base path
        st->fixed_ok = gens_use_fixed(ctx, n);
        st->defer = ctx->tune_ipa_defer >= 0 ? ctx->tune_ipa_defer : (st->fixed_ok ? 3 : 0);
        if (st->defer > FOLD_MAX_DEFER) st->defer = FOLD_MAX_DEFER;
        if (st->defer > (int)st->lg_n) st->defer = (int)st->lg_n;
        memcpy(&st->z, z, 32);
        ctx->ipa_G.reserve(n * sizeof(affine_t));
        ctx->ipa_cs.reserve(n * sizeof(fr_t));
        ctx->ipa_zs.reserve(n * sizeof(fr_t));
        ctx->ipa_tail.reserve(sizeof(affine_t) + (2 + VEC_DOT_MAX_BLOCKS) * sizeof(fr_t));
        cudaStream_t s = ctx->stream;
        HALO_CUDA(cudaMemcpyAsync(ctx->ipa_G.p, ctx->gens.p, n * sizeof(affine_t), cudaMemcpyDeviceToDevice, s));  // pcdl.rs:185
        HALO_CUDA(cudaMemsetAsync(ctx->ipa_cs.p, 0, n * sizeof(fr_t), s));                                         // pcdl.rs:183-184
        if (n_coeffs)
            HALO_CUDA(cudaMemcpyAsync(ctx->ipa_cs.p, resident ? ctx->poly_dev.p : (const void*)coeffs, n_coeffs * sizeof(fr_t),
                                      resident ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
        vec_powers(ctx, st->z, n, ctx->ipa_zs.as<fr_t>());  // pcdl.rs:186
        if (v_out) {                                   // v = p(z) = <c, z-powers>  (pcdl.rs:135)
            fr_t* scal = reinterpret_cast<fr_t*>(reinterpret_cast<char*>(ctx->ipa_tail.p) + sizeof(affine_t));
            vec_dot(ctx, ctx->ipa_cs.as<fr_t>(), ctx->ipa_zs.as<fr_t>(), n, scal + 2, scal);
            HALO_CUDA(cudaMemcpyAsync(v_out, scal, 32, cudaMemcpyDeviceToHost, s));
        }
        HALO_CUDA(cudaStreamSynchronize(s));
    } catch (const halo::CudaError& e) {
        ctx->last_error = std::string("CUDA error: ") + cudaGetErrorString(e.err) + " (" + e.what + ")";
        delete st;
        return HALO_ECUDA;
    }
    ctx->ipa_busy = true;
    *out = st;
    return HALO_OK;
}

int halo_ipa_begin(halo_ctx* ctx, const uint64_t* coeffs, uint64_t n_coeffs, uint64_t n, const uint64_t z[4], halo_ipa** out,
                   uint64_t v_out[4]) {
    return ipa_begin_impl(ctx, coeffs, false, n_coeffs, n, z, out, v_out);
}

int halo_ipa_begin_resident(halo_ctx* ctx, uint64_t n, const uint64_t z[4], halo_ipa** out, uint64_t v_out[4]) {
    if (!ctx || ctx->poly_n == 0 || ctx->poly_n > n) {
        if (ctx) ctx->last_error = "halo_ipa_begin_resident: no resident polynomial (call halo_h_lincomb_resident first)";
        return HALO_ESTATE;
    }
    return ipa_begin_impl(ctx, nullptr, true, ctx->poly_n, n, z, out, v_out);
}

void halo_ipa_destroy(halo_ipa* st) {
    if (!st) return;
    cudaSetDevice(st->ctx->device);
    cudaStreamSynchronize(st->ctx->stream);
    st->ctx->ipa_busy = false;  // the buffers stay with the context for the next opening
    delete st;
}

int halo_ipa_blind_commit(halo_ipa* st, const uint64_t* q, uint64_t n_q, uint64_t out_jac[12]) {
    if (!st || !q || !out_jac) return HALO_EINVAL;
    if (n_q == 0 || n_q >= st->n || st->round != 0) {
        st->ctx->last_error = "halo_ipa_blind_commit: need 0 < n_q < n before the first round";
        return HALO_EINVAL;
    }
    IPA_TRY(st)
    ctx->ipa_pbar.reserve(st->n * sizeof(fr_t));
    ctx->stage_scalars.reserve(n_q * sizeof(fr_t));
    HALO_CUDA(cudaMemcpyAsync(ctx->stage_scalars.p, q, n_q * sizeof(fr_t), cudaMemcpyHostToDevice, ctx->stream));
    vec_pbar(ctx, ctx->stage_scalars.as<fr_t>(), n_q, st->z, st->n, ctx->ipa_pbar.as<fr_t>());
    xyzz_t r;
    msm_gens_device(ctx, ctx->ipa_pbar.as<fr_t>(), 0, st->n, r);  // commit(p_bar) without the w_bar S term
    jac_t j;
    xyzz_to_jac(j, r);
    memcpy(out_jac, &j, 96);
    st->have_pbar = true;
    IPA_CATCH
}

int halo_ipa_blind_apply(halo_ipa* st, const uint64_t alpha[4]) {
    if (!st || !alpha || !st->have_pbar || st->round != 0) return HALO_EINVAL;
    IPA_TRY(st)
    fr_t a;
    memcpy(&a, alpha, 32);
    vec_axpy(ctx, ctx->ipa_cs.as<fr_t>(), ctx->ipa_pbar.as<fr_t>(), a, st->n);  // p' = p + alpha p_bar  (pcdl.rs:156)
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    st->have_pbar = false;
    IPA_CATCH
}

int halo_ipa_set_hprime(halo_ipa* st, const uint64_t Hprime_jac[12]) {
    if (!st || !Hprime_jac) return HALO_EINVAL;
    IPA_TRY(st)
    jac_t j;
    memcpy(&j, Hprime_jac, 96);
    xyzz_t x;
    jac_to_xyzz(x, j);
    affine_t a;
    xyzz_to_affine(a, x);
    HALO_CUDA(cudaMemcpyAsync(ctx->ipa_tail.p, &a, sizeof a, cudaMemcpyHostToDevice, ctx->stream));
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    st->hprime = a;
    st->have_hprime = true;
    IPA_CATCH
}

int halo_ipa_round_lr(halo_ipa* st, uint64_t L_jac[12], uint64_t R_jac[12]) {
    if (!st || !L_jac || !R_jac) return HALO_EINVAL;
    if (!st->have_hprime || st->cur < 2 || st->lr_done) {
        st->ctx->last_error = "halo_ipa_round_lr: call order (set_hprime, then lr/fold alternating, lg n rounds)";
        return HALO_ESTATE;
    }
    IPA_TRY(st)
    const uint64_t m = st->cur / 2;
    affine_t* G = ctx->ipa_G.as<affine_t>();
    fr_t* c = ctx->ipa_cs.as<fr_t>();
    fr_t* z = ctx->ipa_zs.as<fr_t>();
    affine_t* Hp = ctx->ipa_tail.as<affine_t>();
    fr_t* scal = reinterpret_cast<fr_t*>(reinterpret_cast<char*>(ctx->ipa_tail.p) + sizeof(affine_t));
    vec_dot(ctx, c + m, z, m, scal + 2, scal);          // dot_l = <c_r, z_l>
    vec_dot(ctx, c, z + m, m, scal + 2, scal + 1);      // dot_r = <c_l, z_r>
    const uint64_t freeze_len = ctx->tune_ipa_freeze_len > 0 ? (uint64_t)ctx->tune_ipa_freeze_len : IPA_FREEZE_LEN;
    if (!st->frozen) {  // between stages: decide how the coming rounds treat the generator vector (see k_frozen_scalars)
        int D = 0;
        bool over_gens = false;
        if (st->cur > freeze_len) {
            if (st->round == 0 && st->defer > 0) {
                D = st->defer;  // head stage over GS itself
                over_gens = true;
            } else if (ctx->tune_ipa_defer2 > 0 && ctx->tune_ipa_defer != 0) {  // ("ipa_defer_rounds" = 0 switches every stage off)
                int room = 0;  // rounds until the frozen-tail length is reached
                while ((st->cur >> (room + 1)) >= freeze_len) room++;
                D = room < ctx->tune_ipa_defer2 ? room : ctx->tune_ipa_defer2;
                if (D > FOLD_MAX_DEFER) D = FOLD_MAX_DEFER;
                if (D < 2) D = 0;  // a single round is the ordinary fold
            }
        }
        if (D > 0 || st->cur <= freeze_len) {
            st->frozen = true;
            st->deferred = D > 0;  // a deferred stage is undone by k_fold_multi after D rounds; the tail freeze is final
            st->stage_D = D;
            st->stage_first = st->round;
            st->stage_over_gens = over_gens;
            st->M0 = (uint32_t)st->cur;
            st->defer_xis.clear();
            ctx->ipa_frozen.reserve((size_t)3 * st->M0 * sizeof(fr_t));
            k_fill_one<<<(st->M0 + 255) / 256, 256, 0, ctx->stream>>>(ctx->ipa_frozen.as<fr_t>(), st->M0);
            ctx->kernel_launches++;
        }
    }
    MsmInput in[2];
    if (st->frozen) {
        fr_t* sv = ctx->ipa_frozen.as<fr_t>();
        fr_t* tL = sv + st->M0;
        fr_t* tR = tL + st->M0;
        k_frozen_scalars<<<(st->M0 + 255) / 256, 256, 0, ctx->stream>>>(c, sv, st->M0, (uint32_t)st->cur, tL, tR);
        ctx->kernel_launches++;
        in[0].bases = G;
        in[0].scalars = tL;
        in[1].bases = G;
        in[1].scalars = tR;
        if (st->deferred && st->stage_over_gens && st->fixed_ok)  // G is still GS[0..n): shared bucket set over the precomputed multiples
            for (int k = 0; k < 2; k++) in[k] = gens_msm_input(ctx, true, in[k].scalars, 0, st->M0);
    } else {
        in[0].bases = G;       // L = <c_r, g_l> + dot_l H'
        in[0].scalars = c + m;
        in[1].bases = G + m;   // R = <c_l, g_r> + dot_r H'
        in[1].scalars = c;
    }
    const bool host_tail = in[0].fixed_stride != 0;  // the FIXED-base path has no tail: dot * H' is added on the host
    fr_t dots[2];
    for (int k = 0; k < 2; k++) {
        in[k].n = st->frozen ? st->M0 : (uint32_t)m;
        if (!host_tail) {
            in[k].tail_bases = Hp;
            in[k].tail_scalars = scal + k;
            in[k].n_tail = 1;
        }
    }
    const int saved_c = ctx->force_c;
    if (st->frozen && !st->deferred && ctx->tune_ipa_frozen_c > 0) ctx->force_c = ctx->tune_ipa_frozen_c;
    xyzz_t out[2], tails[2];
    std::function<void()> tail_fn = [&]() {  // dot_l H', dot_r H' on the host while the MSM kernels run
        xyzz_t hp;
        xyzz_from_affine(hp, st->hprime);
        for (int k = 0; k < 2; k++) xyzz_mul_glv(tails[k], hp, dots[k]);
    };
    if (host_tail) {
        HALO_CUDA(cudaMemcpyAsync(dots, scal, sizeof dots, cudaMemcpyDeviceToHost, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));  // two dot products: microseconds
    }
    ctx->force_two_lanes = host_tail && ctx->tune_ipa_two_lanes != 0;
    msm_batch(ctx, in, 2, out, host_tail ? &tail_fn : nullptr);
    ctx->force_two_lanes = false;
    ctx->force_c = saved_c;
    if (host_tail)
        for (int k = 0; k < 2; k++) xyzz_add(out[k], tails[k]);
    jac_t j;
    xyzz_to_jac(j, out[0]);
    memcpy(L_jac, &j, 96);
    xyzz_to_jac(j, out[1]);
    memcpy(R_jac, &j, 96);
    st->lr_done = true;
    IPA_CATCH
}

int halo_ipa_round_fold(halo_ipa* st, const uint64_t xi[4], const uint64_t xi_inv[4]) {
    if (!st || !xi || !xi_inv) return HALO_EINVAL;
    if (!st->lr_done) {
        st->ctx->last_error = "halo_ipa_round_fold: round_lr must precede fold";
        return HALO_ESTATE;
    }
    IPA_TRY(st)
    const uint64_t m = st->cur / 2;
    fr_t x, xinv;
    memcpy(&x, xi, 32);
    memcpy(&xinv, xi_inv, 32);
    if (st->deferred) st->defer_xis.push_back(x);
    if (st->frozen) {
        k_frozen_fold_s<<<(st->M0 + 255) / 256, 256, 0, ctx->stream>>>(ctx->ipa_frozen.as<fr_t>(), st->M0, (uint32_t)st->cur, x);
    } else {
        fold_multi(ctx, ctx->ipa_G.as<affine_t>(), st->cur, &x, 1);  // G_j + xi G_{j+m}, joint-sparse-form digits of xi
    }
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
    vec_fold_scalars(ctx, ctx->ipa_cs.as<fr_t>(), ctx->ipa_zs.as<fr_t>(), m, x, xinv);
    st->cur = m;
    st->round++;
    st->lr_done = false;
    if (st->deferred && (int)(st->round - st->stage_first) == st->stage_D && st->cur > 1) {
        // the stage's rounds in one joint pass: G^(first + D) from G^(first) (ipa_G still holds it: nothing was folded)
        fold_multi(ctx, ctx->ipa_G.as<affine_t>(), st->M0, st->defer_xis.data(), st->stage_D);
        st->frozen = st->deferred = false;
        st->defer_xis.clear();
    }
    IPA_CATCH
}

int halo_ipa_finish(halo_ipa* st, uint64_t U_jac[12], uint64_t c_out[4]) {
    if (!st || !U_jac || !c_out) return HALO_EINVAL;
    if (st->cur != 1) {
        st->ctx->last_error = "halo_ipa_finish: rounds remaining";
        return HALO_ESTATE;
    }
    IPA_TRY(st)
    xyzz_t x;
    if (st->frozen) {  // U = sum_j s_j G0_j
        HALO_CUDA(cudaMemcpyAsync(c_out, ctx->ipa_cs.p, 32, cudaMemcpyDeviceToHost, ctx->stream));
        msm_device(ctx, ctx->ipa_G.as<affine_t>(), ctx->ipa_frozen.as<fr_t>(), st->M0, x);
    } else {
        affine_t u;
        HALO_CUDA(cudaMemcpyAsync(&u, ctx->ipa_G.p, sizeof u, cudaMemcpyDeviceToHost, ctx->stream));
        HALO_CUDA(cudaMemcpyAsync(c_out, ctx->ipa_cs.p, 32, cudaMemcpyDeviceToHost, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));
        xyzz_from_affine(x, u);
    }
    jac_t j;
    xyzz_to_jac(j, x);
    memcpy(U_jac, &j, 96);  // U = G_(lg n)[0]  (pcdl.rs:230)
    IPA_CATCH
}

}  // extern "C"
#endif  // HALO_IPA_FOLD_TU
