// combine.cu -- K5c: many independent exact combinations R_o = P_o + a_o Q_o + b_o S in one launch.
//
// The batch verifier and the batch decider (DESIGN.md K5b, K5c) need, per hiding claim, C' = C + alpha C_bar - w' S
// (pcdl.rs:272-279) and, per accumulation step, C* = C_bar - omega S.  Both points are hashed, so they must be exact; on
// the host each costs one or two GLV scalar multiplications.  Here the division of labour of k_fold_multi (ipa.cu) applies:
// the host splits a_o and b_o by GLV and writes each pair in joint sparse form (glv.cuh, microseconds per scalar); one device
// thread per output runs the joint double-and-add over the four terms Q, phi(Q), S, phi(S) with 129 shared doublings.
// phi(Q) = (beta x, y) and Q + phi(Q) = (-(x + beta x), -y) are free; Q - phi(Q) comes from one batched affine addition
// per point (inversions shared by batch_invert).  Unlike the fold, outputs have different scalars, so every thread reads its
// own digit column from global memory (coalesced: digit position major).  The sums are normalised with one batch_invert.
#include <algorithm>
#include <cstring>
#include <system_error>
#include <thread>
#include <vector>

#include "../../include/halo_b200_test.h"
#include "common.cuh"
#include "glv.cuh"
#include "msm.cuh"

using namespace halo;

namespace halo {

__device__ __constant__ uint32_t c_combine_beta[8] = HALO_GLV_BETA_MONT;  // glv.cuh

constexpr int COMBINE_POS = 136;  // digit positions of GlvDigits

// beta x and the denominator x - beta x of Q - phi(Q) for every base (the n points Q_o, then S)
__global__ void __launch_bounds__(128) k_combine_prep1(const affine_t* __restrict__ Q, uint32_t n, fq_t* __restrict__ bx,
                                                       fq_t* __restrict__ den) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    fq_t beta;
#pragma unroll
    for (int i = 0; i < 8; i++) beta.v[i] = c_combine_beta[i];
    const affine_t p = Q[j];
    fq_t r, d;
    fp_mul(r, p.x, beta);
    fp_sub(d, p.x, r);
    if (fp_is_zero(d)) fp_one(d);  // infinity, or x = 0 (phi(Q) = Q, the difference is infinity): no inversion
    bx[j] = r;
    den[j] = d;
}
// Q - phi(Q) = (x, y) + (beta x, -y): lambda = 2 y / (x - beta x)
__global__ void __launch_bounds__(128) k_combine_prep2(const affine_t* __restrict__ Q, uint32_t n, const fq_t* __restrict__ bx,
                                                       const fq_t* __restrict__ inv, affine_t* __restrict__ diff) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const affine_t p = Q[j];
    const fq_t b = bx[j];
    affine_t out;
    fq_t d;
    fp_sub(d, p.x, b);
    if (affine_is_inf(p) || fp_is_zero(d)) {
        affine_set_inf(out);
    } else {
        fq_t lam, t1;
        fp_dbl(t1, p.y);
        fp_mul(lam, t1, inv[j]);
        fp_sqr(t1, lam);
        fp_sub(t1, t1, p.x);
        fp_sub(out.x, t1, b);
        fp_sub(t1, p.x, out.x);
        fp_mul(t1, lam, t1);
        fp_sub(out.y, t1, p.y);
    }
    diff[j] = out;
}

// acc += d1 B + d2 phi(B) for joint digits d1, d2 in {-1, 0, 1}; B at index j of Q / bx / diff
static __device__ __forceinline__ void combine_term(xyzz_t& acc, const affine_t* __restrict__ Q, const fq_t* __restrict__ bx,
                                                    const affine_t* __restrict__ diff, uint32_t j, int d1, int d2) {
    if (!d1 && !d2) return;
    affine_t p;
    bool neg;
    if (d1 && d2 && d1 != d2) {  // +-(B - phi(B))
        p = diff[j];
        neg = d1 < 0;
    } else {
        p = Q[j];
        neg = (d1 ? d1 : d2) < 0;
        if (d2 && !affine_is_inf(p)) {
            const fq_t b = bx[j];
            if (!d1) {  // phi(B) = (beta x, y)
                p.x = b;
            } else {  // B + phi(B) = (-(x + beta x), -y)
                fq_t sx;
                fp_add(sx, p.x, b);
                fp_neg(p.x, sx);
                neg = !neg;
            }
        }
    }
    xyzz_madd(acc, p, neg);
}

// One thread per output: joint double-and-add over the digits of (a_o: Q_o, phi(Q_o)) and (b_o: S, phi(S)), then + P_o.
// digit byte at [pos * n + o]: bits 0-1 / 2-3 / 4-5 / 6-7 = k1(a), k2(a), k1(b), k2(b), each 0 (0), 1 (+1) or 3 (-1).
// xyzz_madd is exact for infinity and for a running sum equal to +- the addend, so crafted inputs stay exact.
__global__ void __launch_bounds__(32) k_point_combine(const affine_t* __restrict__ P, const affine_t* __restrict__ Q,
                                                      const fq_t* __restrict__ bx, const affine_t* __restrict__ diff,
                                                      const uint8_t* __restrict__ digits, const int16_t* __restrict__ tops,
                                                      uint32_t n, xyzz_t* __restrict__ sums, fq_t* __restrict__ den) {
    const uint32_t o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n) return;
    xyzz_t acc;
    xyzz_set_inf(acc);
#pragma unroll 1
    for (int i = tops[o]; i >= 0; i--) {
        xyzz_dbl(acc, acc);
        const uint32_t c = digits[(size_t)i * n + o];
        if (!c) continue;
        auto dig = [](uint32_t v) { return v == 1 ? 1 : v == 3 ? -1 : 0; };
        combine_term(acc, Q, bx, diff, o, dig(c & 3), dig((c >> 2) & 3));
        combine_term(acc, Q, bx, diff, n, dig((c >> 4) & 3), dig(c >> 6));
    }
    xyzz_madd(acc, P[o], false);
    sums[o] = acc;
    fq_t d;
    if (xyzz_is_inf(acc))
        fp_one(d);
    else
        fp_mul(d, acc.zz, acc.zzz);
    den[o] = d;
}

// x = X / ZZ = X * ZZZ * inv, y = Y / ZZZ = Y * ZZ * inv with inv = 1 / (ZZ * ZZZ); infinity -> (0, 0)
__global__ void __launch_bounds__(128) k_combine_finish(const xyzz_t* __restrict__ sums, const fq_t* __restrict__ inv, uint32_t n,
                                                        affine_t* __restrict__ out) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const xyzz_t p = sums[j];
    affine_t r;
    if (xyzz_is_inf(p)) {
        affine_set_inf(r);
    } else {
        fq_t i = inv[j], t;
        fp_mul(t, i, p.zzz);
        fp_mul(r.x, p.x, t);
        fp_mul(t, i, p.zz);
        fp_mul(r.y, p.y, t);
    }
    out[j] = r;
}

static uint8_t digit_code(int d) { return d > 0 ? 1 : d < 0 ? 3 : 0; }

// XYZZ -> affine for many points with one inversion (Montgomery's trick); infinity -> (0, 0)
static std::vector<affine_t> to_affine_batch(const std::vector<xyzz_t>& pts) {
    const size_t n = pts.size();
    std::vector<fq_t> pre(n);
    fq_t acc, inv, t;
    fp_one(acc);
    for (size_t i = 0; i < n; i++) {
        pre[i] = acc;
        if (!xyzz_is_inf(pts[i])) {
            fp_mul(t, pts[i].zz, pts[i].zzz);
            fp_mul(acc, acc, t);
        }
    }
    fp_inv(inv, acc);
    std::vector<affine_t> out(n);
    for (size_t i = n; i-- > 0;) {
        const xyzz_t& p = pts[i];
        if (xyzz_is_inf(p)) {
            affine_set_inf(out[i]);
            continue;
        }
        fq_t d, id;
        fp_mul(d, p.zz, p.zzz);
        fp_mul(id, inv, pre[i]);  // 1 / (ZZ * ZZZ)
        fp_mul(inv, inv, d);
        fp_mul(t, id, p.zzz);
        fp_mul(out[i].x, p.x, t);
        fp_mul(t, id, p.zz);
        fp_mul(out[i].y, p.y, t);
    }
    return out;
}

static void combine_device(halo_ctx* ctx, const std::vector<xyzz_t>& Px, const std::vector<xyzz_t>& Qx, const fr_t* a,
                           const fr_t* b, uint32_t n, affine_t* out) {
    std::vector<xyzz_t> pq(Px);
    pq.insert(pq.end(), Qx.begin(), Qx.end());
    const std::vector<affine_t> pqa = to_affine_batch(pq);
    const affine_t* P = pqa.data();
    const affine_t* Q = pqa.data() + n;
    // one upload: P [n] | Q [n] + S | digits [136][n] | tops [n]
    const size_t offQ = (size_t)n * sizeof(affine_t), offD = offQ + (size_t)(n + 1) * sizeof(affine_t);
    const size_t offT = offD + (size_t)COMBINE_POS * n, bytes = offT + (size_t)n * sizeof(int16_t);
    std::vector<uint8_t> host(bytes, 0);
    std::memcpy(host.data(), P, offQ);
    std::memcpy(host.data() + offQ, Q, (size_t)n * sizeof(affine_t));
    std::memcpy(host.data() + offQ + (size_t)n * sizeof(affine_t), &ctx->S, sizeof(affine_t));
    uint8_t* dig = host.data() + offD;
    int16_t* tops = reinterpret_cast<int16_t*>(host.data() + offT);
    for (uint32_t o = 0; o < n; o++) {
        GlvDigits da, db;
        make_glv_jsf(a[o], da);
        make_glv_jsf(b[o], db);
        tops[o] = std::max(da.top, db.top);
        for (int i = 0; i <= tops[o]; i++)
            dig[(size_t)i * n + o] = (uint8_t)(digit_code(da.d1[i]) | digit_code(da.d2[i]) << 2 | digit_code(db.d1[i]) << 4 |
                                               digit_code(db.d2[i]) << 6);
    }
    ctx->combine_in.reserve(bytes);
    // work: bx [n + 1] | den [n + 1] | diff [n + 1] | sums [n] | den2 [n] | out [n]
    const size_t wbx = 0, wden = wbx + (size_t)(n + 1) * sizeof(fq_t), wdiff = wden + (size_t)(n + 1) * sizeof(fq_t);
    const size_t wsums = wdiff + (size_t)(n + 1) * sizeof(affine_t), wden2 = wsums + (size_t)n * sizeof(xyzz_t);
    const size_t wout = wden2 + (size_t)n * sizeof(fq_t), wbytes = wout + (size_t)n * sizeof(affine_t);
    ctx->combine_work.reserve(wbytes);
    char* in = static_cast<char*>(ctx->combine_in.p);
    char* w = static_cast<char*>(ctx->combine_work.p);
    const affine_t* dP = reinterpret_cast<const affine_t*>(in);
    const affine_t* dQ = reinterpret_cast<const affine_t*>(in + offQ);
    fq_t* bx = reinterpret_cast<fq_t*>(w + wbx);
    fq_t* den = reinterpret_cast<fq_t*>(w + wden);
    affine_t* diff = reinterpret_cast<affine_t*>(w + wdiff);
    xyzz_t* sums = reinterpret_cast<xyzz_t*>(w + wsums);
    fq_t* den2 = reinterpret_cast<fq_t*>(w + wden2);
    affine_t* dout = reinterpret_cast<affine_t*>(w + wout);
    cudaStream_t st = ctx->stream;
    HALO_CUDA(cudaMemcpyAsync(in, host.data(), bytes, cudaMemcpyHostToDevice, st));
    const unsigned g1 = (n + 1 + 127) / 128;
    k_combine_prep1<<<g1, 128, 0, st>>>(dQ, n + 1, bx, den);
    batch_invert(ctx, st, den, n + 1, ctx->combine_inv_scratch);
    k_combine_prep2<<<g1, 128, 0, st>>>(dQ, n + 1, bx, den, diff);
    // 32 threads per CTA: few outputs are a latency-bound chain each, so they are spread over as many SMs as possible
    k_point_combine<<<(n + 31) / 32, 32, 0, st>>>(dP, dQ, bx, diff, reinterpret_cast<const uint8_t*>(in + offD),
                                                 reinterpret_cast<const int16_t*>(in + offT), n, sums, den2);
    batch_invert(ctx, st, den2, n, ctx->combine_inv_scratch);
    k_combine_finish<<<(n + 127) / 128, 128, 0, st>>>(sums, den2, n, dout);
    ctx->kernel_launches += 4;
    HALO_CUDA(cudaGetLastError());
    HALO_CUDA(cudaMemcpyAsync(out, dout, (size_t)n * sizeof(affine_t), cudaMemcpyDeviceToHost, st));
    HALO_CUDA(cudaStreamSynchronize(st));
}

// The host path: P + a Q + b S by GLV (xyzz_mul_glv, as `Projective * Fr` of the host layer), outputs spread over up to 16
// host threads, each normalised with its own inversion.
static void combine_host(const std::vector<xyzz_t>& P, const std::vector<xyzz_t>& Q, const affine_t& S_aff, const fr_t* a,
                         const fr_t* b, uint32_t n, affine_t* out) {
    xyzz_t S;
    xyzz_from_affine(S, S_aff);
    auto work = [&](size_t t, size_t T) {
        for (size_t o = t; o < n; o += T) {
            xyzz_t r = P[o], u;
            xyzz_mul_glv(u, Q[o], a[o]);
            xyzz_add(r, u);
            xyzz_mul_glv(u, S, b[o]);
            xyzz_add(r, u);
            xyzz_to_affine(out[o], r);
        }
    };
    const size_t hw = std::thread::hardware_concurrency();
    const size_t T = std::min<size_t>(n, std::max<size_t>(1, std::min<size_t>(hw, 16)));
    std::vector<std::thread> th;
    std::vector<size_t> unspawned;
    for (size_t t = 1; t < T; t++) {
        try {
            th.emplace_back(work, t, T);
        } catch (const std::system_error&) {
            unspawned.push_back(t);  // no thread available: this thread takes that share as well
        }
    }
    work(0, T);
    for (size_t t : unspawned) work(t, T);
    for (auto& x : th) x.join();
}

}  // namespace halo

extern "C" int halo_test_point_combine(halo_ctx* ctx, int path, const uint64_t* P_jac, const uint64_t* Q_jac, const uint64_t* a,
                                       const uint64_t* b, uint64_t n, uint64_t* out_affine) {
    if (!ctx || path < -1 || path > 1 || (n && (!P_jac || !Q_jac || !a || !b || !out_affine))) return HALO_EINVAL;
    if (n >> 31) {
        ctx->last_error = "halo_test_point_combine: n is 2^31 or more";
        return HALO_EINVAL;
    }
    if (!ctx->have_SH) {
        ctx->last_error = "halo_test_point_combine: parameters not loaded";
        return HALO_ESTATE;
    }
    if (n == 0) return HALO_OK;
    try {
        HALO_CUDA(cudaSetDevice(ctx->device));
        std::vector<xyzz_t> P(n), Q(n);
        for (uint64_t o = 0; o < n; o++) {
            jac_t j;
            std::memcpy(&j, P_jac + 12 * o, 96);
            jac_to_xyzz(P[o], j);
            std::memcpy(&j, Q_jac + 12 * o, 96);
            jac_to_xyzz(Q[o], j);
        }
        const fr_t* as = reinterpret_cast<const fr_t*>(a);
        const fr_t* bs = reinterpret_cast<const fr_t*>(b);
        affine_t* out = reinterpret_cast<affine_t*>(out_affine);
        const int m = ctx->tune_combine_min_outputs;
        const bool device = path == 1 || (path == -1 && m >= 0 && n >= (uint64_t)m);
        if (device)
            combine_device(ctx, P, Q, as, bs, (uint32_t)n, out);
        else
            combine_host(P, Q, ctx->S, as, bs, (uint32_t)n, out);
    } catch (const CudaError& e) {
        ctx->last_error = cudaGetErrorString(e.err);
        return HALO_ECUDA;
    } catch (const std::bad_alloc&) {
        ctx->last_error = "out of host memory";
        return HALO_ENOMEM;
    }
    return HALO_OK;
}
