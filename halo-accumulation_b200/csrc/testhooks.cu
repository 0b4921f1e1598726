// testhooks.cu -- device test hooks and integer-pipe microbenchmarks (include/halo_b200_test.h).
#include <cstring>

#include "../../include/halo_b200_test.h"
#include "common.cuh"
#include "vec.cuh"

using namespace halo;

namespace halo {

template <class P>
__global__ void __launch_bounds__(128) k_fp_op(int op, const fp_t<P>* a, const fp_t<P>* b, fp_t<P>* out, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fp_t<P> x = a[i], y = b ? b[i] : a[i], r;
    switch (op) {
        case 0: fp_mul(r, x, y); break;
        case 1: fp_add(r, x, y); break;
        case 2: fp_sub(r, x, y); break;
        case 3: fp_sqr(r, x); break;
        case 4: fp_inv(r, x); break;
        case 5: fp_neg(r, x); break;
        case 6: fp_to_canon(r.v, x); break;
        default: fp_from_canon(r, x.v); break;
    }
    out[i] = r;
}

__global__ void k_madd_chain(const affine_t* pts, const uint8_t* neg, uint64_t n, jac_t* out) {
    if (threadIdx.x || blockIdx.x) return;
    xyzz_t acc;
    xyzz_set_inf(acc);
    for (uint64_t i = 0; i < n; i++) xyzz_madd(acc, pts[i], neg && neg[i]);
    jac_t j;
    xyzz_to_jac(j, acc);
    *out = j;
}
__global__ void k_add_chain(const jac_t* pts, uint64_t n, int dbls, jac_t* out) {
    if (threadIdx.x || blockIdx.x) return;
    xyzz_t acc;
    xyzz_set_inf(acc);
    for (uint64_t i = 0; i < n; i++) {
        xyzz_t q;
        jac_to_xyzz(q, pts[i]);
        xyzz_add(acc, q);
    }
    for (int i = 0; i < dbls; i++) xyzz_dbl(acc, acc);
    jac_t j;
    xyzz_to_jac(j, acc);
    *out = j;
}


// Random 64-byte gathers (the access pattern of the bucket accumulation: one affine base per entry) from a table far
// larger than the L2: every thread walks `iters` pseudo-random 64-byte-aligned slots and xors what it reads.
__global__ void __launch_bounds__(256) k_gather_tp(const uint4* __restrict__ table, uint64_t slots, int iters, int bytes, uint32_t* sink) {
    uint64_t x = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 0x9e3779b97f4a7c15ull + 0x1234567ull;
    uint4 acc = make_uint4(0, 0, 0, 0);
    for (int i = 0; i < iters; i += 4) {  // four independent gathers in flight per thread
        const uint4* p[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            x ^= x << 13;
            x ^= x >> 7;
            x ^= x << 17;
            p[k] = table + __umul64hi(x, slots) * 4;  // uniform in [0, slots)
        }
        uint4 v[4][4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            v[k][0] = p[k][0];
            if (bytes >= 32) v[k][1] = p[k][1];
            if (bytes >= 64) {
                v[k][2] = p[k][2];
                v[k][3] = p[k][3];
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            acc.x ^= v[k][0].x; acc.y ^= v[k][0].y; acc.z ^= v[k][0].z; acc.w ^= v[k][0].w;
            if (bytes >= 32) { acc.x ^= v[k][1].x; acc.y ^= v[k][1].y; acc.z ^= v[k][1].z; acc.w ^= v[k][1].w; }
            if (bytes >= 64) { acc.x ^= v[k][2].x ^ v[k][3].x; acc.y ^= v[k][2].y ^ v[k][3].y; acc.z ^= v[k][2].z ^ v[k][3].z; acc.w ^= v[k][2].w ^ v[k][3].w; }
        }
    }
    if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x5a5a5a5au) sink[0] = acc.x;
}

// Cooperative variant: 4 adjacent lanes fetch one 64-byte slot with ONE instruction (16 bytes each), so both 32-byte
// sectors of the slot are requested together; 8 slots per warp-instruction.  gathers = blocks * threads * iters / 4 * 4
// (each lane still walks `iters` slots, shared with its 3 neighbours: count blocks * threads / 4 * iters).
// LANES = 2: two adjacent lanes fetch one 32-byte slot (an x coordinate alone), 16 slots per warp-instruction.
template <int LANES>
__global__ void __launch_bounds__(256) k_gather_coop_tp(const uint4* __restrict__ table, uint64_t slots, int iters, uint32_t* sink) {
    const unsigned lane = threadIdx.x & 31u, sub = lane & (LANES - 1u);
    uint64_t x = (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) / LANES) * 0x9e3779b97f4a7c15ull + 0x1234567ull;  // same for the lanes of a group
    uint4 acc = make_uint4(0, 0, 0, 0);
    for (int i = 0; i < iters; i += 4) {
        const uint4* p[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            x ^= x << 13;
            x ^= x >> 7;
            x ^= x << 17;
            p[k] = table + __umul64hi(x, slots) * LANES + sub;
        }
        uint4 v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) v[k] = *p[k];
#pragma unroll
        for (int k = 0; k < 4; k++) { acc.x ^= v[k].x; acc.y ^= v[k].y; acc.z ^= v[k].z; acc.w ^= v[k].w; }
    }
    if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x5a5a5a5au) sink[0] = acc.x;
}

template <int ILP, int V>
__global__ void __launch_bounds__(512) k_fp_mul_tp(int iters, uint32_t* sink) {
    fq_t x[ILP], y;
    uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
    for (int k = 0; k < ILP; k++) {
        fp_one(x[k]);
        x[k].v[0] ^= tid + k;
        x[k].v[7] &= 0x0fffffffu;
    }
    fp_one(y);
    y.v[1] ^= tid * 2654435761u;
    y.v[7] &= 0x0fffffffu;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < ILP; k++) {
            if (V < 0) {
                fp_mul_portable(x[k], x[k], y);
            } else {
                uint32_t o[8];
                fp_mul_asm<FqParams, (V < 0 ? 0 : V)>(o, x[k].v, y.v);
#pragma unroll
                for (int j = 0; j < 8; j++) x[k].v[j] = o[j];
            }
        }
    }
    uint32_t acc = 0;
#pragma unroll
    for (int k = 0; k < ILP; k++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc ^= x[k].v[j];
    if (acc == 0x12345678u) sink[0] = acc;  // keep the chain alive without a store per thread
    if (tid == 0) sink[1] = acc;
}

template <int KIND>
__global__ void __launch_bounds__(1024) k_imad_tp(int iters, uint32_t* sink) {
    uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t a = tid * 2654435761u + 12345u, b = tid ^ 0x9e3779b9u;
    uint32_t r[16], cnt[8];
    uint64_t w[16];
#pragma unroll
    for (int k = 0; k < 16; k++) {
        r[k] = tid + k;
        w[k] = tid + 7 * k;
        cnt[k & 7] = k;
    }
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            // the multiplicand is the accumulator itself, so no product is loop invariant (ptxas otherwise hoists a * b and
            // the loop degenerates into additions)
            if (KIND == 0) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(r[k]) : "r"(a), "r"(b));
            if (KIND == 1) asm volatile("{.reg .u32 lo, hi; mov.b64 {lo, hi}, %0; mad.wide.u32 %0, lo, %1, %0;}" : "+l"(w[k]) : "r"(a));
            if (KIND == 2) asm volatile("mad.hi.u32 %0, %0, %1, %2;" : "+r"(r[k]) : "r"(a), "r"(b));
        }
        if (KIND == 3) {  // 8 independent wide MADs with carry-OUT captured by an ADDC (IMAD.WIDE P-out + IADD3.X)
#pragma unroll
            for (int k = 0; k < 8; k++)
                asm volatile("mad.lo.cc.u32 %0, %3, %4, %0;\n\tmadc.hi.cc.u32 %1, %3, %4, %1;\n\taddc.u32 %2, %2, 0;"
                             : "+r"(r[2 * k]), "+r"(r[2 * k + 1]), "+r"(cnt[k]) : "r"(a), "r"(b));
        }
        if (KIND == 4) {  // 2 independent carry chains of 4 fused pairs each (IMAD.WIDE.X with carry in and out)
#pragma unroll
            for (int k = 0; k < 2; k++)
                asm volatile("mad.lo.cc.u32 %0, %9, %10, %0;\n\tmadc.hi.cc.u32 %1, %9, %10, %1;\n\t"
                             "madc.lo.cc.u32 %2, %9, %10, %2;\n\tmadc.hi.cc.u32 %3, %9, %10, %3;\n\t"
                             "madc.lo.cc.u32 %4, %9, %10, %4;\n\tmadc.hi.cc.u32 %5, %9, %10, %5;\n\t"
                             "madc.lo.cc.u32 %6, %9, %10, %6;\n\tmadc.hi.cc.u32 %7, %9, %10, %7;\n\t"
                             "addc.u32 %8, %8, 0;"
                             : "+r"(r[8 * k]), "+r"(r[8 * k + 1]), "+r"(r[8 * k + 2]), "+r"(r[8 * k + 3]), "+r"(r[8 * k + 4]),
                               "+r"(r[8 * k + 5]), "+r"(r[8 * k + 6]), "+r"(r[8 * k + 7]), "+r"(cnt[k])
                             : "r"(a), "r"(b));
        }
        if (KIND == 5) {  // 8 independent fused pairs, no carry in or out (plain IMAD.WIDE through the .cc idiom)
#pragma unroll
            for (int k = 0; k < 8; k++)
                asm volatile("mad.lo.cc.u32 %0, %2, %3, %0;\n\tmadc.hi.u32 %1, %2, %3, %1;"
                             : "+r"(r[2 * k]), "+r"(r[2 * k + 1]) : "r"(a), "r"(b));
        }
        if (KIND == 6) {  // 8 independent wide MADs with carry-IN only (ADD.CC feeding IMAD.WIDE.X, no carry out)
#pragma unroll
            for (int k = 0; k < 8; k++)
                asm volatile("add.cc.u32 %2, %2, %3;\n\tmadc.lo.cc.u32 %0, %3, %4, %0;\n\tmadc.hi.u32 %1, %3, %4, %1;"
                             : "+r"(r[2 * k]), "+r"(r[2 * k + 1]), "+r"(cnt[k]) : "r"(a), "r"(b));
        }
        if (KIND == 7) {  // 16 independent 3-input adds with carry chains of length 2 (ALU pipe reference)
#pragma unroll
            for (int k = 0; k < 8; k++)
                asm volatile("add.cc.u32 %0, %0, %2;\n\taddc.u32 %1, %1, %3;" : "+r"(r[2 * k]), "+r"(r[2 * k + 1]) : "r"(a), "r"(b));
        }
    }
    uint32_t acc = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) acc ^= r[k] ^ (uint32_t)w[k] ^ (uint32_t)(w[k] >> 32) ^ cnt[k & 7];
    if (acc == 0x12345678u) sink[0] = acc;
    if (tid == 0) sink[1] = acc;
}

}  // namespace halo

#define T_TRY(ctx) try { HALO_CUDA(cudaSetDevice((ctx)->device));
#define T_CATCH(ctx)                                        \
    }                                                       \
    catch (const halo::CudaError& e) {                      \
        (ctx)->last_error = cudaGetErrorString(e.err);      \
        return HALO_ECUDA;                                  \
    }                                                       \
    return HALO_OK;

extern "C" {

int halo_test_fp_op(halo_ctx* ctx, int which, int op, const uint64_t* a, const uint64_t* b, uint64_t* out, uint64_t n) {
    if (!ctx || !a || !out) return HALO_EINVAL;
    T_TRY(ctx)
    DevBuf da, db, dout;
    da.reserve(n * 32);
    dout.reserve(n * 32);
    HALO_CUDA(cudaMemcpy(da.p, a, n * 32, cudaMemcpyHostToDevice));
    if (b) {
        db.reserve(n * 32);
        HALO_CUDA(cudaMemcpy(db.p, b, n * 32, cudaMemcpyHostToDevice));
    }
    unsigned grid = (unsigned)((n + 127) / 128);
    if (which)
        k_fp_op<ScalarParams><<<grid, 128, 0, ctx->stream>>>(op, da.as<fr_t>(), b ? db.as<fr_t>() : nullptr, dout.as<fr_t>(), n);
    else
        k_fp_op<BaseParams><<<grid, 128, 0, ctx->stream>>>(op, da.as<fq_t>(), b ? db.as<fq_t>() : nullptr, dout.as<fq_t>(), n);
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    HALO_CUDA(cudaMemcpy(out, dout.p, n * 32, cudaMemcpyDeviceToHost));
    da.release();
    db.release();
    dout.release();
    T_CATCH(ctx)
}

int halo_test_madd_chain(halo_ctx* ctx, const uint64_t* affine, const uint8_t* neg, uint64_t n, uint64_t out_jac[12]) {
    if (!ctx || !out_jac) return HALO_EINVAL;
    T_TRY(ctx)
    DevBuf dp, dn, dout;
    dp.reserve((n ? n : 1) * 64);
    dout.reserve(96);
    if (n) HALO_CUDA(cudaMemcpy(dp.p, affine, n * 64, cudaMemcpyHostToDevice));
    if (neg && n) {
        dn.reserve(n);
        HALO_CUDA(cudaMemcpy(dn.p, neg, n, cudaMemcpyHostToDevice));
    }
    k_madd_chain<<<1, 32, 0, ctx->stream>>>(dp.as<affine_t>(), neg ? dn.as<uint8_t>() : nullptr, n, dout.as<jac_t>());
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    HALO_CUDA(cudaMemcpy(out_jac, dout.p, 96, cudaMemcpyDeviceToHost));
    dp.release();
    dn.release();
    dout.release();
    T_CATCH(ctx)
}

int halo_test_add_chain(halo_ctx* ctx, const uint64_t* jac, uint64_t n, int dbls, uint64_t out_jac[12]) {
    if (!ctx || !out_jac) return HALO_EINVAL;
    T_TRY(ctx)
    DevBuf dp, dout;
    dp.reserve((n ? n : 1) * 96);
    dout.reserve(96);
    if (n) HALO_CUDA(cudaMemcpy(dp.p, jac, n * 96, cudaMemcpyHostToDevice));
    k_add_chain<<<1, 32, 0, ctx->stream>>>(dp.as<jac_t>(), n, dbls, dout.as<jac_t>());
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    HALO_CUDA(cudaMemcpy(out_jac, dout.p, 96, cudaMemcpyDeviceToHost));
    dp.release();
    dout.release();
    T_CATCH(ctx)
}

int halo_test_fp_mul_throughput(halo_ctx* ctx, int blocks, int threads, int iters, int ilp, float* ms, uint64_t* checksum) {
    if (!ctx || !ms) return HALO_EINVAL;
    T_TRY(ctx)
    DevBuf sink;
    sink.reserve(16);
    cudaEvent_t e0, e1;
    HALO_CUDA(cudaEventCreate(&e0));
    HALO_CUDA(cudaEventCreate(&e1));
    for (int rep = 0; rep < 2; rep++) {
        HALO_CUDA(cudaEventRecord(e0, ctx->stream));
        // ilp encodes (ilp, variant): ilp % 10 = independent chains per thread, ilp / 10 = variant + 1 (0 = portable C++)
        int var = ilp / 10 - 1, il = ilp % 10;
#define TP(I, V) k_fp_mul_tp<I, V><<<blocks, threads, 0, ctx->stream>>>(iters, sink.as<uint32_t>())
        if (il == 1) { if (var < 0) TP(1, -1); else if (var == 0) TP(1, 0); else if (var == 1) TP(1, 1); else if (var == 2) TP(1, 2); else if (var == 3) TP(1, 3); else TP(1, 4); }
        else { if (var < 0) TP(2, -1); else if (var == 0) TP(2, 0); else if (var == 1) TP(2, 1); else if (var == 2) TP(2, 2); else if (var == 3) TP(2, 3); else TP(2, 4); }
#undef TP
        HALO_CUDA(cudaEventRecord(e1, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    ctx->kernel_launches += 2;
    HALO_CUDA(cudaGetLastError());
    HALO_CUDA(cudaEventElapsedTime(ms, e0, e1));
    uint32_t h[4] = {0, 0, 0, 0};
    HALO_CUDA(cudaMemcpy(h, sink.p, 8, cudaMemcpyDeviceToHost));
    if (checksum) *checksum = h[1];
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    sink.release();
    T_CATCH(ctx)
}

int halo_test_check_canaries(int* live_buffers) {
    cudaDeviceSynchronize();
    int bad = 0;
    const auto& r = halo::devbuf_registry();
    for (const halo::DevBuf* b : r)
        if (!b->canary_ok()) bad++;
    if (live_buffers) *live_buffers = (int)r.size();
    return bad;
}

int halo_test_msm_route(halo_ctx* ctx, int lane, int out[10]) {
    if (!ctx || !out || lane < 0 || lane > 1) return HALO_EINVAL;
    memcpy(out, ctx->msm_route[lane], sizeof ctx->msm_route[lane]);
    memset(ctx->msm_route[lane], 0, sizeof ctx->msm_route[lane]);  // c = 0 until the next MSM on this lane
    return HALO_OK;
}

int halo_test_gather_throughput(halo_ctx* ctx, uint64_t table_bytes, int blocks, int threads, int iters, int bytes, float* ms) {
    if (!ctx || !ms || table_bytes < 4096 || threads > 256) return HALO_EINVAL;
    T_TRY(ctx)
    DevBuf table, sink;
    table.reserve(table_bytes);
    sink.reserve(16);
    HALO_CUDA(cudaMemsetAsync(table.p, 0x3c, table_bytes, ctx->stream));
    cudaEvent_t e0, e1;
    HALO_CUDA(cudaEventCreate(&e0));
    HALO_CUDA(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 3; rep++) {
        HALO_CUDA(cudaEventRecord(e0, ctx->stream));
        if (bytes == -32)
            k_gather_coop_tp<2><<<blocks, threads, 0, ctx->stream>>>(table.as<uint4>(), table_bytes / 32, iters, sink.as<uint32_t>());
        else if (bytes < 0)
            k_gather_coop_tp<4><<<blocks, threads, 0, ctx->stream>>>(table.as<uint4>(), table_bytes / 64, iters, sink.as<uint32_t>());
        else
            k_gather_tp<<<blocks, threads, 0, ctx->stream>>>(table.as<uint4>(), table_bytes / 64, iters, bytes, sink.as<uint32_t>());
        HALO_CUDA(cudaEventRecord(e1, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));
        float t;
        HALO_CUDA(cudaEventElapsedTime(&t, e0, e1));
        if (rep > 0 && t < best) best = t;
    }
    ctx->kernel_launches += 3;
    HALO_CUDA(cudaGetLastError());
    *ms = best;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    table.release();
    sink.release();
    T_CATCH(ctx)
}

int halo_test_imad_throughput(halo_ctx* ctx, int kind, int blocks, int threads, int iters, float* ms, uint64_t* checksum) {
    if (!ctx || !ms) return HALO_EINVAL;
    T_TRY(ctx)
    DevBuf sink;
    sink.reserve(16);
    cudaEvent_t e0, e1;
    HALO_CUDA(cudaEventCreate(&e0));
    HALO_CUDA(cudaEventCreate(&e1));
    for (int rep = 0; rep < 2; rep++) {
        HALO_CUDA(cudaEventRecord(e0, ctx->stream));
        if (kind == 0) k_imad_tp<0><<<blocks, threads, 0, ctx->stream>>>(iters, sink.as<uint32_t>());
        else if (kind == 1) k_imad_tp<1><<<blocks, threads, 0, ctx->stream>>>(iters, sink.as<uint32_t>());
        else if (kind == 2) k_imad_tp<2><<<blocks, threads, 0, ctx->stream>>>(iters, sink.as<uint32_t>());
        else if (kind == 3) k_imad_tp<3><<<blocks, threads, 0, ctx->stream>>>(iters, sink.as<uint32_t>());
        else if (kind == 4) k_imad_tp<4><<<blocks, threads, 0, ctx->stream>>>(iters, sink.as<uint32_t>());
        else if (kind == 5) k_imad_tp<5><<<blocks, threads, 0, ctx->stream>>>(iters, sink.as<uint32_t>());
        else if (kind == 6) k_imad_tp<6><<<blocks, threads, 0, ctx->stream>>>(iters, sink.as<uint32_t>());
        else k_imad_tp<7><<<blocks, threads, 0, ctx->stream>>>(iters, sink.as<uint32_t>());
        HALO_CUDA(cudaEventRecord(e1, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    ctx->kernel_launches += 2;
    HALO_CUDA(cudaGetLastError());
    HALO_CUDA(cudaEventElapsedTime(ms, e0, e1));
    uint32_t h[4] = {0, 0, 0, 0};
    HALO_CUDA(cudaMemcpy(h, sink.p, 8, cudaMemcpyDeviceToHost));
    if (checksum) *checksum = h[1];
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    sink.release();
    T_CATCH(ctx)
}

// Times one Fr vector kernel on device-resident synthetic data (CUDA events on the context stream, best of 5):
// kind 0 = scalar folds (pcdl.rs:221-223), 1 = h-expansion, 2 = dot product, 3 = powers of z.
int halo_test_vec_bench(halo_ctx* ctx, int kind, uint64_t n, float* ms) {
    if (!ctx || !ms || n < 8) return HALO_EINVAL;
    T_TRY(ctx)
    DevBuf a, b, scratch;
    a.reserve(n * sizeof(fr_t));
    b.reserve(n * sizeof(fr_t));
    scratch.reserve((2 + VEC_DOT_MAX_BLOCKS) * sizeof(fr_t));
    fr_t z;
    fp_one(z);
    z.v[0] ^= 0x1234567u;
    z.v[5] ^= 0x0abcdefu;
    vec_powers(ctx, z, n, a.as<fr_t>());
    vec_powers(ctx, z, n, b.as<fr_t>());
    fr_t xis[33];
    for (int i = 0; i < 33; i++) {
        xis[i] = z;
        xis[i].v[1] ^= (uint32_t)i * 2654435761u;
        xis[i].v[7] &= 0x0fffffffu;
    }
    int lg = 0;
    while (((uint64_t)2 << lg) <= n) lg++;
    cudaEvent_t e0, e1;
    HALO_CUDA(cudaEventCreate(&e0));
    HALO_CUDA(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 6; rep++) {
        HALO_CUDA(cudaEventRecord(e0, ctx->stream));
        if (kind == 0) vec_fold_scalars(ctx, a.as<fr_t>(), b.as<fr_t>(), n / 2, z, xis[3]);
        else if (kind == 1) {
            const uint32_t ulg = (uint32_t)lg;
            vec_h_lincomb(ctx, xis, &ulg, &z, 1, (uint64_t)1 << lg, false, a.as<fr_t>());
        }
        else if (kind == 2) vec_dot(ctx, a.as<fr_t>(), b.as<fr_t>(), n, scratch.as<fr_t>() + 2, scratch.as<fr_t>());
        else vec_powers(ctx, z, n, a.as<fr_t>());
        HALO_CUDA(cudaEventRecord(e1, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));
        float t;
        HALO_CUDA(cudaEventElapsedTime(&t, e0, e1));
        if (rep > 0 && t < best) best = t;
    }
    *ms = best;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    a.release();
    b.release();
    scratch.release();
    T_CATCH(ctx)
}

// k_h_lincomb over k claims of 2^lg_n coefficients, writing (CUDA events on the context stream, best of 5 after a warm-up;
// the H2D copy of the claim descriptors included).
int halo_test_h_lincomb_bench(halo_ctx* ctx, uint32_t lg_n, uint64_t k, float* ms) {
    if (!ctx || !ms || lg_n > LINCOMB_MAX_LG || k == 0) return HALO_EINVAL;
    T_TRY(ctx)
    const uint64_t n = (uint64_t)1 << lg_n;
    DevBuf a;
    a.reserve(n * sizeof(fr_t));
    std::vector<fr_t> xis(k * (lg_n + 1)), w(k);
    std::vector<uint32_t> lgs(k, lg_n);
    for (size_t i = 0; i < xis.size(); i++) {
        fp_one(xis[i]);
        xis[i].v[1] ^= (uint32_t)i * 2654435761u;
        xis[i].v[7] &= 0x0fffffffu;
    }
    for (uint64_t j = 0; j < k; j++) w[j] = xis[j * (lg_n + 1)];
    cudaEvent_t e0, e1;
    HALO_CUDA(cudaEventCreate(&e0));
    HALO_CUDA(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 6; rep++) {
        HALO_CUDA(cudaEventRecord(e0, ctx->stream));
        vec_h_lincomb(ctx, xis.data(), lgs.data(), w.data(), k, n, false, a.as<fr_t>());
        HALO_CUDA(cudaEventRecord(e1, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));
        float t;
        HALO_CUDA(cudaEventElapsedTime(&t, e0, e1));
        if (rep > 0 && t < best) best = t;
    }
    *ms = best;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    a.release();
    T_CATCH(ctx)
}

int halo_test_read_quotient(halo_ctx* ctx, uint64_t* out, uint64_t cap, uint64_t* n_out) {
    if (!ctx || !n_out || (!out && cap)) return HALO_EINVAL;
    if (!ctx->quot_ready) return HALO_ESTATE;
    T_TRY(ctx)
    *n_out = ctx->quot_n;
    if (cap >= ctx->quot_n && ctx->quot_n) {
        HALO_CUDA(cudaMemcpyAsync(out, ctx->quot_dev.p, ctx->quot_n * sizeof(fr_t), cudaMemcpyDeviceToHost, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    T_CATCH(ctx)
}
}
