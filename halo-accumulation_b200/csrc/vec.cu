// vec.cu -- Fr vector kernels: dot products, powers, folds, and the expansion of h(X) and of sums of them (K5, K5b).
//
// Replaces the serial scalar loops of the reference:
//   group.rs:13-15  scalar_dot            -> k_dot_partial + k_dot_final
//   group.rs:29-37  construct_powers      -> k_powers
//   pcdl.rs:221-223 c / z folds           -> k_fold_scalars   (HBM bound: 2 x (64 B read + 32 B write) per j)
//   pcdl.rs:56-77   HPoly::get_poly       -> k_h_lincomb, one claim of weight 1 (closed form pinned by pcdl.rs:496-508:
//                                             coeff[j] = prod_{b: bit b of j set} xi_{lg n - b})
//   acc.rs:85-94    AccumulatedHPolys::get_poly -> k_h_lincomb with weights alpha^{i+1}, accumulating onto h_0
//   (batch decider)  sum_j w_j coeffs(h_j) over claims of mixed size -> k_h_lincomb (DESIGN.md K5b)
//   pcdl.rs:140-142,156  p_bar = q (X - z), p' = p + alpha p_bar -> k_pbar, k_axpy
//   (batch opening)  p_j(z) of k polynomials, sum_j alpha^j p_j   -> k_poly_eval_many + k_poly_eval_final, k_poly_combine (K3b)
//   (multi-point opening) sum_t s_t (f_t - f_t(z_t)) / (X - z_t), p_j(z_t) of m queries, sum_j c_j p_j + c_q q
//                    -> k_quot_chunks + k_quot_carry (+ k_quot_write), k_poly_lincomb (K3c)
#include "common.cuh"
#include "vec.cuh"

namespace halo {

constexpr int VEC_THREADS = 256;

// ---- powers ------------------------------------------------------------------------------------
struct PowTable {
    fr_t p[40];  // p[i] = z^(2^i)
};
constexpr int POW_CHUNK = 32;

__global__ void __launch_bounds__(VEC_THREADS) k_powers(PowTable tab, uint64_t n, fr_t* __restrict__ out) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t j0 = t * POW_CHUNK;
    if (j0 >= n) return;
    fr_t cur;
    fp_one(cur);
#pragma unroll 1
    for (int i = 0; i < 40; i++)
        if ((j0 >> i) & 1) fp_mul(cur, cur, tab.p[i]);
    fr_t z = tab.p[0];
#pragma unroll 1
    for (int k = 0; k < POW_CHUNK && j0 + k < n; k++) {
        out[j0 + k] = cur;
        fp_mul(cur, cur, z);
    }
}

void vec_powers(halo_ctx* ctx, const fr_t& z, uint64_t n, fr_t* d_out) {
    if (n == 0) return;
    PowTable tab;
    tab.p[0] = z;
    for (int i = 1; i < 40; i++) fp_sqr(tab.p[i], tab.p[i - 1]);
    uint64_t threads = (n + POW_CHUNK - 1) / POW_CHUNK;
    k_powers<<<(unsigned)((threads + VEC_THREADS - 1) / VEC_THREADS), VEC_THREADS, 0, ctx->stream>>>(tab, n, d_out);
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
}

// ---- dot product ---------------------------------------------------------------------------------
__device__ __forceinline__ void block_sum_fr(fr_t& v, fr_t* sm) {
    const int j = threadIdx.x;
    sm[j] = v;
    __syncthreads();
    for (int stride = VEC_THREADS / 2; stride >= 1; stride >>= 1) {
        if (j < stride) {
            fp_add(v, v, sm[j + stride]);
            sm[j] = v;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(VEC_THREADS) k_dot_partial(const fr_t* __restrict__ a, const fr_t* __restrict__ b, uint64_t n,
                                                             fr_t* __restrict__ partials) {
    __shared__ fr_t sm[VEC_THREADS];
    fr_t acc, t;
    fp_zero(acc);
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        fp_mul(t, a[i], b[i]);
        fp_add(acc, acc, t);
    }
    block_sum_fr(acc, sm);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}
__global__ void __launch_bounds__(VEC_THREADS) k_dot_final(const fr_t* __restrict__ partials, uint32_t count, fr_t* __restrict__ out) {
    __shared__ fr_t sm[VEC_THREADS];
    fr_t acc;
    fp_zero(acc);
    for (uint32_t i = threadIdx.x; i < count; i += blockDim.x) fp_add(acc, acc, partials[i]);
    block_sum_fr(acc, sm);
    if (threadIdx.x == 0) *out = acc;
}

void vec_dot(halo_ctx* ctx, const fr_t* d_a, const fr_t* d_b, uint64_t n, fr_t* d_partials, fr_t* d_out) {
    uint32_t blocks = (uint32_t)((n + VEC_THREADS - 1) / VEC_THREADS);
    if (blocks > VEC_DOT_MAX_BLOCKS) blocks = VEC_DOT_MAX_BLOCKS;
    if (blocks == 0) blocks = 1;
    k_dot_partial<<<blocks, VEC_THREADS, 0, ctx->stream>>>(d_a, d_b, n, d_partials);
    k_dot_final<<<1, VEC_THREADS, 0, ctx->stream>>>(d_partials, blocks, d_out);
    ctx->kernel_launches += 2;
    HALO_CUDA(cudaGetLastError());
}

// ---- k polynomials at one point (K3b) ------------------------------------------------------------------------
// Polynomial j owns coeffs[off[j] .. off[j+1]).  A segment of bps blocks per polynomial, grid-strided over its coefficients:
// partials[j bps + b]; then one block per polynomial adds its bps partials.
__global__ void __launch_bounds__(VEC_THREADS) k_poly_eval_many(const fr_t* __restrict__ coeffs, const uint64_t* __restrict__ off,
                                                                const fr_t* __restrict__ pows, uint32_t bps,
                                                                fr_t* __restrict__ partials) {
    __shared__ fr_t sm[VEC_THREADS];
    const uint32_t seg = blockIdx.x / bps, b = blockIdx.x % bps;
    const uint64_t o = off[seg], len = off[seg + 1] - o;
    fr_t acc, t;
    fp_zero(acc);
    for (uint64_t i = (uint64_t)b * blockDim.x + threadIdx.x; i < len; i += (uint64_t)bps * blockDim.x) {
        fp_mul(t, coeffs[o + i], pows[i]);
        fp_add(acc, acc, t);
    }
    block_sum_fr(acc, sm);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}
__global__ void __launch_bounds__(VEC_THREADS) k_poly_eval_final(const fr_t* __restrict__ partials, uint32_t bps, fr_t* __restrict__ out) {
    __shared__ fr_t sm[VEC_THREADS];
    const fr_t* p = partials + (uint64_t)blockIdx.x * bps;
    fr_t acc;
    fp_zero(acc);
    for (uint32_t i = threadIdx.x; i < bps; i += blockDim.x) fp_add(acc, acc, p[i]);
    block_sum_fr(acc, sm);
    if (threadIdx.x == 0) out[blockIdx.x] = acc;
}

uint32_t vec_eval_many_blocks(uint64_t k, uint64_t n_max) {
    uint64_t b = (n_max + VEC_THREADS - 1) / VEC_THREADS, cap = VEC_DOT_MAX_BLOCKS / k;
    if (b > cap) b = cap;
    return b ? (uint32_t)b : 1;
}

void vec_eval_many(halo_ctx* ctx, const fr_t* d_coeffs, const uint64_t* d_off, uint64_t k, uint64_t n_max, const fr_t* d_pows,
                   fr_t* d_partials, fr_t* d_out) {
    const uint32_t bps = vec_eval_many_blocks(k, n_max);
    k_poly_eval_many<<<(unsigned)(k * bps), VEC_THREADS, 0, ctx->stream>>>(d_coeffs, d_off, d_pows, bps, d_partials);
    k_poly_eval_final<<<(unsigned)k, VEC_THREADS, 0, ctx->stream>>>(d_partials, bps, d_out);
    ctx->kernel_launches += 2;
    HALO_CUDA(cudaGetLastError());
}

// out[i] = sum_j alpha^j p_j[i] by Horner over j (p_j[i] = 0 from off[j+1] - off[j] on): k multiplications per coefficient
__global__ void __launch_bounds__(VEC_THREADS) k_poly_combine(const fr_t* __restrict__ coeffs, const uint64_t* __restrict__ off,
                                                              uint32_t k, fr_t alpha, uint64_t n, fr_t* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fr_t acc;
    fp_zero(acc);
#pragma unroll 1
    for (uint32_t j = k; j-- > 0;) {
        fp_mul(acc, acc, alpha);
        const uint64_t o = off[j];
        if (i < off[j + 1] - o) fp_add(acc, acc, coeffs[o + i]);
    }
    out[i] = acc;
}

void vec_poly_combine(halo_ctx* ctx, const fr_t* d_coeffs, const uint64_t* d_off, uint64_t k, const fr_t& alpha, uint64_t n,
                      fr_t* d_out) {
    k_poly_combine<<<(unsigned)((n + VEC_THREADS - 1) / VEC_THREADS), VEC_THREADS, 0, ctx->stream>>>(d_coeffs, d_off, (uint32_t)k,
                                                                                                     alpha, n, d_out);
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
}

// ---- K3c: division by X - z and evaluation, as a chunked scan ---------------------------------------------------------
// A group is g = sum of its terms w p_j (coefficients synthesised on the fly, never stored).  The quotient h = g / (X - z)
// obeys h_{i-1} = g_i + z h_i from the top down; the remainder is g(z).  A thread owns QB consecutive coefficients (its chunk
// c), a block QT chunks:
//   k_quot_chunks: S_c = sum_l g_{cB+l} z^l (Horner), then a block suffix scan gives the carry into each chunk from the chunks
//                  above it in the block (kloc) and the block's aggregate (agg);
//   k_quot_carry:  one block per group scans the aggregates: the carry into each block (kblk) and g(z) = the full suffix (rem);
//   k_quot_write:  each chunk starts from its carry kloc + z^(QB (QT - 1 - t)) kblk and writes h downward; q (+)= s h.
// Evaluation is the first two kernels without kloc / kblk.
constexpr int QB = 16;
constexpr int QT = 256;

__device__ __forceinline__ void quot_synth(fr_t& g, const fr_t* __restrict__ coeffs, const QuotTerm* __restrict__ terms,
                                           uint32_t first, uint32_t count, uint64_t i) {
    fp_zero(g);
#pragma unroll 1
    for (uint32_t e = first; e < first + count; e++) {
        const QuotTerm& tm = terms[e];
        if (i >= tm.len) continue;
        if (tm.unit) {
            fp_add(g, g, coeffs[tm.off + i]);
        } else {
            fr_t t;
            fp_mul(t, coeffs[tm.off + i], tm.w);
            fp_add(g, g, t);
        }
    }
}

// In-block inclusive suffix scan of v over the QT threads: v_t <- sum_{u >= t} v_u Z^(u - t), where pw[d] = Z^d for d < QT
__device__ __forceinline__ void block_suffix_scan(fr_t& v, fr_t* sm, const fr_t* __restrict__ pw) {
    const int t = threadIdx.x;
    sm[t] = v;
    __syncthreads();
#pragma unroll 1
    for (int d = 1; d < QT; d <<= 1) {
        fr_t o;
        const bool has = t + d < QT;
        if (has) {
            fp_mul(o, sm[t + d], pw[d]);
            fp_add(v, v, o);
        }
        __syncthreads();
        sm[t] = v;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(QT) k_quot_chunks(const fr_t* __restrict__ coeffs, const QuotGroup* __restrict__ groups,
                                                    const QuotTerm* __restrict__ terms, const fr_t* __restrict__ zthr,
                                                    uint32_t nblk, fr_t* __restrict__ kloc, fr_t* __restrict__ agg) {
    __shared__ fr_t sm[QT];
    const uint32_t g = blockIdx.x / nblk, b = blockIdx.x % nblk;
    const QuotGroup& gr = groups[g];
    const fr_t z = gr.z;
    const uint64_t lo = ((uint64_t)b * QT + threadIdx.x) * QB;
    fr_t acc, x;
    fp_zero(acc);
#pragma unroll 1
    for (int l = QB - 1; l >= 0; l--) {
        quot_synth(x, coeffs, terms, gr.first, gr.count, lo + l);
        fp_mul(acc, acc, z);
        fp_add(acc, acc, x);
    }
    const fr_t* pw = zthr + (uint64_t)gr.tab * QT;
    block_suffix_scan(acc, sm, pw);
    if (kloc) {
        fr_t c;
        if (threadIdx.x + 1 < QT)
            c = sm[threadIdx.x + 1];
        else
            fp_zero(c);
        kloc[(uint64_t)g * nblk * QT + (uint64_t)b * QT + threadIdx.x] = c;
    }
    if (threadIdx.x == 0) agg[(uint64_t)g * nblk + b] = acc;
}

__global__ void __launch_bounds__(QT) k_quot_carry(const QuotGroup* __restrict__ groups, const fr_t* __restrict__ agg, uint32_t nblk,
                                                   fr_t* __restrict__ kblk, fr_t* __restrict__ rem) {
    __shared__ fr_t sm[QT];
    __shared__ fr_t pw[QT];
    const uint32_t g = blockIdx.x, t = threadIdx.x;
    const fr_t zb = groups[g].zblk;  // z^(QB QT): one block's span
    const fr_t* a = agg + (uint64_t)g * nblk;
    const uint32_t r = (nblk + QT - 1) / QT, lo = t * r, hi = min(lo + r, nblk);
    fr_t acc;
    fp_zero(acc);
#pragma unroll 1
    for (uint32_t i = hi; i-- > lo;) {
        fp_mul(acc, acc, zb);
        fp_add(acc, acc, a[i]);
    }
    if (t == 0) {  // pw[d] = zb^(r d): the distance of d runs
        fr_t m, e;
        fp_one(m);
        e = zb;
        for (uint32_t s = r; s; s >>= 1) {
            if (s & 1) fp_mul(m, m, e);
            fp_sqr(e, e);
        }
        fp_one(e);
        for (int d = 0; d < QT; d++) {
            pw[d] = e;
            fp_mul(e, e, m);
        }
    }
    __syncthreads();
    block_suffix_scan(acc, sm, pw);
    if (t == 0) rem[g] = acc;
    if (!kblk) return;
    fr_t c;
    if (t + 1 < QT)
        c = sm[t + 1];
    else
        fp_zero(c);
#pragma unroll 1
    for (uint32_t i = hi; i-- > lo;) {
        kblk[(uint64_t)g * nblk + i] = c;
        fp_mul(c, c, zb);
        fp_add(c, c, a[i]);
    }
}

__global__ void __launch_bounds__(QT) k_quot_write(const fr_t* __restrict__ coeffs, const QuotGroup* __restrict__ groups,
                                                   uint32_t n_groups, const QuotTerm* __restrict__ terms, const fr_t* __restrict__ zthr,
                                                   uint32_t nblk, const fr_t* __restrict__ kloc, const fr_t* __restrict__ kblk,
                                                   uint64_t n_q, fr_t* __restrict__ q) {
    const uint32_t b = blockIdx.x, t = threadIdx.x;
    const uint64_t lo = ((uint64_t)b * QT + t) * QB;
    if (lo >= n_q) return;
#pragma unroll 1
    for (uint32_t g = 0; g < n_groups; g++) {
        const QuotGroup& gr = groups[g];
        const fr_t z = gr.z, s = gr.s;
        fr_t acc, x, o;
        fp_mul(acc, kblk[(uint64_t)g * nblk + b], zthr[(uint64_t)gr.tab * QT + (QT - 1 - t)]);
        fp_add(acc, acc, kloc[(uint64_t)g * nblk * QT + (uint64_t)b * QT + t]);  // h_{lo + QB - 1}
#pragma unroll 1
        for (int l = QB - 1; l >= 0; l--) {
            const uint64_t i = lo + l;  // acc = h_i
            if (i < n_q) {
                fp_mul(o, acc, s);
                if (g) fp_add(o, o, q[i]);
                q[i] = o;
            }
            if (l) {
                quot_synth(x, coeffs, terms, gr.first, gr.count, i);
                fp_mul(acc, acc, z);
                fp_add(acc, acc, x);
            }
        }
    }
}

uint32_t vec_quot_blocks(uint64_t n) {
    const uint64_t b = (n + (uint64_t)QB * QT - 1) / ((uint64_t)QB * QT);
    return b ? (uint32_t)b : 1;
}

void vec_quot_tables(const fr_t& z, fr_t& zblk, fr_t* zthr) {
    fr_t zq = z;
    for (int i = 1; i < QB; i <<= 1) fp_sqr(zq, zq);  // z^QB (QB a power of two)
    fp_one(zthr[0]);
    for (int u = 1; u < QT; u++) fp_mul(zthr[u], zthr[u - 1], zq);
    fp_mul(zblk, zthr[QT - 1], zq);
}

void vec_quot_eval(halo_ctx* ctx, const fr_t* d_coeffs, const QuotGroup* d_groups, uint32_t n_groups, const QuotTerm* d_terms,
                   const fr_t* d_zthr, uint64_t n, fr_t* d_agg, fr_t* d_rem) {
    const uint32_t nblk = vec_quot_blocks(n);
    k_quot_chunks<<<(unsigned)((uint64_t)n_groups * nblk), QT, 0, ctx->stream>>>(d_coeffs, d_groups, d_terms, d_zthr, nblk, nullptr,
                                                                                 d_agg);
    k_quot_carry<<<n_groups, QT, 0, ctx->stream>>>(d_groups, d_agg, nblk, nullptr, d_rem);
    ctx->kernel_launches += 2;
    HALO_CUDA(cudaGetLastError());
}

void vec_quotient(halo_ctx* ctx, const fr_t* d_coeffs, const QuotGroup* d_groups, uint32_t n_groups, const QuotTerm* d_terms,
                  const fr_t* d_zthr, uint64_t n, fr_t* d_kloc, fr_t* d_agg, fr_t* d_kblk, fr_t* d_rem, fr_t* d_q) {
    const uint32_t nblk = vec_quot_blocks(n);
    k_quot_chunks<<<(unsigned)((uint64_t)n_groups * nblk), QT, 0, ctx->stream>>>(d_coeffs, d_groups, d_terms, d_zthr, nblk, d_kloc,
                                                                                 d_agg);
    k_quot_carry<<<n_groups, QT, 0, ctx->stream>>>(d_groups, d_agg, nblk, d_kblk, d_rem);
    ctx->kernel_launches += 2;
    if (n > 1) {
        k_quot_write<<<nblk, QT, 0, ctx->stream>>>(d_coeffs, d_groups, n_groups, d_terms, d_zthr, nblk, d_kloc, d_kblk, n - 1, d_q);
        ctx->kernel_launches++;
    }
    HALO_CUDA(cudaGetLastError());
}

// out[i] = sum_j c_j p_j[i] + c_q q[i] (p_j[i] = 0 from off[j+1] - off[j] on, q[i] = 0 from n_q on)
__global__ void __launch_bounds__(VEC_THREADS) k_poly_lincomb(const fr_t* __restrict__ coeffs, const uint64_t* __restrict__ off,
                                                              const fr_t* __restrict__ cs, uint32_t k, const fr_t* __restrict__ q,
                                                              uint64_t n_q, fr_t c_q, uint64_t n, fr_t* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fr_t acc, t;
    fp_zero(acc);
    if (i < n_q) fp_mul(acc, q[i], c_q);
#pragma unroll 1
    for (uint32_t j = 0; j < k; j++) {
        const uint64_t o = off[j];
        if (i < off[j + 1] - o) {
            fp_mul(t, coeffs[o + i], cs[j]);
            fp_add(acc, acc, t);
        }
    }
    out[i] = acc;
}

void vec_poly_lincomb(halo_ctx* ctx, const fr_t* d_coeffs, const uint64_t* d_off, const fr_t* d_cs, uint64_t k, const fr_t* d_q,
                      uint64_t n_q, const fr_t& c_q, uint64_t n, fr_t* d_out) {
    k_poly_lincomb<<<(unsigned)((n + VEC_THREADS - 1) / VEC_THREADS), VEC_THREADS, 0, ctx->stream>>>(d_coeffs, d_off, d_cs, (uint32_t)k,
                                                                                                     d_q, n_q, c_q, n, d_out);
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
}

// ---- scalar folds (pcdl.rs:221-223) ------------------------------------------------------------------
__global__ void __launch_bounds__(VEC_THREADS) k_fold_scalars(fr_t* __restrict__ c, fr_t* __restrict__ z, uint64_t m, fr_t xi,
                                                              fr_t xi_inv) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    fr_t lo, hi, t;
    lo = c[j];
    hi = c[j + m];
    fp_mul(t, hi, xi_inv);
    fp_add(lo, lo, t);
    c[j] = lo;
    lo = z[j];
    hi = z[j + m];
    fp_mul(t, hi, xi);
    fp_add(lo, lo, t);
    z[j] = lo;
}
void vec_fold_scalars(halo_ctx* ctx, fr_t* d_c, fr_t* d_z, uint64_t m, const fr_t& xi, const fr_t& xi_inv) {
    if (m == 0) return;
    k_fold_scalars<<<(unsigned)((m + VEC_THREADS - 1) / VEC_THREADS), VEC_THREADS, 0, ctx->stream>>>(d_c, d_z, m, xi, xi_inv);
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
}

// ---- sum of weighted h(X) of several claims (K5b) ------------------------------------------------------------
// out[i] (+)= sum_j w_j prod_{b: bit b of i} x_j[b] for i < 2^lg_j.  A block owns 2^11 consecutive coefficients, a thread 8
// of them: bits 0-2 of the index are the thread's own, bits 3-10 its thread index, the bits above the block's.  Per chunk of
// claims the block first builds, in shared memory, the block-uniform product of the high bits with w_j folded in, two
// 16-entry tables over the thread-index bits (the high one with that product folded in) and an 8-entry table over the low
// bits; a thread then pays 1 multiplication for its base and 7 for its 8 coefficients, about 1 per coefficient and claim.
constexpr int LC_THREADS = 256;
constexpr int LC_SPAN_LG = 11;  // lg of the coefficients of one block: 8 per thread
constexpr int LC_CHUNK = 32;    // claims whose tables are in shared memory at a time (41 KiB)
constexpr uint32_t LC_DEAD = 0xFFFFFFFFu;

__global__ void __launch_bounds__(LC_THREADS) k_h_lincomb(const LincombClaim* __restrict__ claims, uint32_t k, uint64_t n_out,
                                                          int accumulate, fr_t* __restrict__ out) {
    __shared__ fr_t t_hi[LC_CHUNK][16];   // w_j * (high bits) * subset products of x[7..10]
    __shared__ fr_t t_mid[LC_CHUNK][16];  // subset products of x[3..6]
    __shared__ fr_t t_lo[LC_CHUNK][8];    // subset products of x[0..2]
    __shared__ fr_t high[LC_CHUNK];
    __shared__ uint32_t lgs[LC_CHUNK];    // lg n_j, or LC_DEAD when the claim ends below this block
    const uint32_t tid = threadIdx.x;
    const uint64_t base = (uint64_t)blockIdx.x << LC_SPAN_LG;
    const uint64_t i0 = base + 8 * (uint64_t)tid;
    fr_t acc[8];
#pragma unroll
    for (int s = 0; s < 8; s++) fp_zero(acc[s]);
#pragma unroll 1
    for (uint32_t c0 = 0; c0 < k; c0 += LC_CHUNK) {
        const uint32_t cn = k - c0 < (uint32_t)LC_CHUNK ? k - c0 : (uint32_t)LC_CHUNK;
        __syncthreads();  // the previous chunk's tables are consumed
        if (tid < cn) {
            const LincombClaim& cl = claims[c0 + tid];
            const uint32_t lg = cl.lg_n;
            const bool live = (base >> lg) == 0;
            fr_t h = cl.w;
#pragma unroll 1
            for (uint32_t b = LC_SPAN_LG; live && b < lg; b++)
                if ((base >> b) & 1) fp_mul(h, h, cl.x[b]);
            high[tid] = h;
            lgs[tid] = live ? lg : LC_DEAD;
        }
        __syncthreads();
#pragma unroll 1
        for (uint32_t e = tid; e < cn * 40; e += LC_THREADS) {
            const uint32_t c = e / 40, r = e % 40;
            if (lgs[c] == LC_DEAD) continue;
            const fr_t* x = claims[c0 + c].x;
            fr_t v;
            uint32_t sub, first;
            if (r < 16) {
                v = high[c];
                sub = r, first = 7;
            } else if (r < 32) {
                fp_one(v);
                sub = r - 16, first = 3;
            } else {
                fp_one(v);
                sub = r - 32, first = 0;
            }
#pragma unroll 1
            for (uint32_t b = 0; b < 4; b++)
                if ((sub >> b) & 1) fp_mul(v, v, x[first + b]);
            if (r < 16)
                t_hi[c][sub] = v;
            else if (r < 32)
                t_mid[c][sub] = v;
            else
                t_lo[c][sub] = v;
        }
        __syncthreads();
#pragma unroll 1
        for (uint32_t c = 0; c < cn; c++) {
            const uint32_t lg = lgs[c];
            if (lg == LC_DEAD || (i0 >> lg) != 0) continue;
            const uint32_t cnt = lg < 3 ? 1u << lg : 8u;  // claims shorter than 8 coefficients
            fr_t b, v;
            fp_mul(b, t_hi[c][tid >> 4], t_mid[c][tid & 15]);
            fp_add(acc[0], acc[0], b);
#pragma unroll
            for (uint32_t s = 1; s < 8; s++) {
                if (s < cnt) {
                    fp_mul(v, b, t_lo[c][s]);
                    fp_add(acc[s], acc[s], v);
                }
            }
        }
    }
#pragma unroll
    for (int s = 0; s < 8; s++) {
        if (i0 + s < n_out) {
            if (accumulate) {
                fr_t o = out[i0 + s];
                fp_add(o, o, acc[s]);
                out[i0 + s] = o;
            } else {
                out[i0 + s] = acc[s];
            }
        }
    }
}

void vec_h_lincomb(halo_ctx* ctx, const fr_t* xis, const uint32_t* lg_ns, const fr_t* weights, uint64_t k, uint64_t n_out,
                   bool accumulate, fr_t* d_out) {
    if (n_out == 0) return;
    std::vector<LincombClaim> h(k ? k : 1);
    fr_t one;
    fp_one(one);
    const fr_t* x = xis;
    for (uint64_t j = 0; j < k; j++) {
        const uint32_t lg = lg_ns[j];
        h[j].w = weights[j];
        for (uint32_t b = 0; b < LINCOMB_MAX_LG; b++) h[j].x[b] = b < lg ? x[lg - b] : one;
        h[j].lg_n = lg;
        x += lg + 1;
    }
    ctx->lincomb_claims.reserve(h.size() * sizeof(LincombClaim));
    HALO_CUDA(cudaMemcpyAsync(ctx->lincomb_claims.p, h.data(), k * sizeof(LincombClaim), cudaMemcpyHostToDevice, ctx->stream));
    const unsigned blocks = (unsigned)((n_out + (1u << LC_SPAN_LG) - 1) >> LC_SPAN_LG);
    k_h_lincomb<<<blocks, LC_THREADS, 0, ctx->stream>>>(ctx->lincomb_claims.as<LincombClaim>(), (uint32_t)k, n_out,
                                                        accumulate ? 1 : 0, d_out);
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
}

// ---- hiding polynomial helpers ---------------------------------------------------------------------------
// p_bar = q * (X - z), zero-padded to n: p_bar[i] = q[i-1] - z q[i]   (pcdl.rs:140-142)
__global__ void __launch_bounds__(VEC_THREADS) k_pbar(const fr_t* __restrict__ q, uint64_t n_q, fr_t z, uint64_t n,
                                                      fr_t* __restrict__ out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fr_t acc, t;
    fp_zero(acc);
    if (i >= 1 && i - 1 < n_q) acc = q[i - 1];
    if (i < n_q) {
        fp_mul(t, z, q[i]);
        fp_sub(acc, acc, t);
    }
    out[i] = acc;
}
void vec_pbar(halo_ctx* ctx, const fr_t* d_q, uint64_t n_q, const fr_t& z, uint64_t n, fr_t* d_out) {
    k_pbar<<<(unsigned)((n + VEC_THREADS - 1) / VEC_THREADS), VEC_THREADS, 0, ctx->stream>>>(d_q, n_q, z, n, d_out);
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
}

// y += alpha * x   (pcdl.rs:156)
__global__ void __launch_bounds__(VEC_THREADS) k_axpy(fr_t* __restrict__ y, const fr_t* __restrict__ x, fr_t alpha, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fr_t t, o = y[i];
    fp_mul(t, x[i], alpha);
    fp_add(o, o, t);
    y[i] = o;
}
void vec_axpy(halo_ctx* ctx, fr_t* d_y, const fr_t* d_x, const fr_t& alpha, uint64_t n) {
    if (n == 0) return;
    k_axpy<<<(unsigned)((n + VEC_THREADS - 1) / VEC_THREADS), VEC_THREADS, 0, ctx->stream>>>(d_y, d_x, alpha, n);
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
}

}  // namespace halo
