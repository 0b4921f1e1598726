// capi.cu -- extern "C" entry points of libhalo_b200.so (include/halo_b200.h).
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <system_error>
#include <thread>

#include "../../include/halo_b200.h"
#include "common.cuh"
#include "msm.cuh"
#include "params.cuh"
#include "vec.cuh"

using namespace halo;

namespace halo {
// Registry behind DevBuf's canaries: one process-wide list, guarded by a mutex (a context is single-threaded like the
// reference, but several contexts may live on several host threads).
std::vector<DevBuf*>& devbuf_registry() {
    static std::vector<DevBuf*> r;
    return r;
}
std::mutex& devbuf_registry_mutex() {
    static std::mutex m;
    return m;
}

__global__ void __launch_bounds__(256) k_mark_infinity(affine_t* __restrict__ bases, const uint8_t* __restrict__ inf, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && inf[i]) affine_set_inf(bases[i]);
}

// The caller's infinity flags of n staged bases to d_inf, then the flagged bases set to infinity, on `st`
static void mark_infinity(halo_ctx* ctx, cudaStream_t st, affine_t* d_bases, uint8_t* d_inf, const uint8_t* inf_flags, uint64_t n) {
    HALO_CUDA(cudaMemcpyAsync(d_inf, inf_flags, n, cudaMemcpyHostToDevice, st));
    k_mark_infinity<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_bases, d_inf, n);
    ctx->kernel_launches++;
}

__global__ void __launch_bounds__(128) k_jac_to_affine(const jac_t* __restrict__ in, affine_t* __restrict__ out, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    jac_t p = in[i];
    xyzz_t q;
    jac_to_xyzz(q, p);
    affine_t a;
    xyzz_to_affine(a, q);
    out[i] = a;
}

int set_error(halo_ctx* ctx, int code, const char* fmt, const char* a, const char* b, int line) {
    if (ctx) {
        char buf[512];
        snprintf(buf, sizeof buf, fmt, a, b, line);
        ctx->last_error = buf;
    }
    return code;
}

}  // namespace halo

namespace halo {
void h2d_copy(halo_ctx* ctx, void* dst, const void* src, size_t bytes, cudaStream_t st) {
    if (bytes == 0) return;
    constexpr size_t CH = halo_ctx::STAGE_CHUNK;
    bool pageable = false;
    if (ctx->tune_stage_pageable && bytes >= 4 * CH) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, src) == cudaSuccess)
            pageable = at.type == cudaMemoryTypeUnregistered;
        else
            cudaGetLastError();
    }
    if (!pageable) {
        HALO_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
        return;
    }
    constexpr int TMAX = halo_ctx::STAGE_THREADS, S = halo_ctx::STAGE_SLOTS;
    const int T = ctx->tune_stage_threads < 1 ? 1 : ctx->tune_stage_threads > TMAX ? TMAX : ctx->tune_stage_threads;
    for (int i = 0; i < T * S; i++)
        if (!ctx->stage_pinned[i]) {
            HALO_CUDA(cudaMallocHost(&ctx->stage_pinned[i], CH));
            HALO_CUDA(cudaEventCreateWithFlags(&ctx->stage_ev[i], cudaEventDisableTiming));
        }
    const size_t nchunks = (bytes + CH - 1) / CH;
    cudaError_t errs[TMAX];
    auto work = [&](int t) {
        errs[t] = cudaSetDevice(ctx->device);
        size_t use = 0;
        for (size_t k = (size_t)t; k < nchunks && errs[t] == cudaSuccess; k += T, use++) {
            const int slot = t * S + (int)(use % S);
            if (use >= (size_t)S) errs[t] = cudaEventSynchronize(ctx->stage_ev[slot]);  // the DMA out of this slot two chunks ago
            const size_t off = k * CH, len = bytes - off < CH ? bytes - off : CH;
            memcpy(ctx->stage_pinned[slot], static_cast<const char*>(src) + off, len);
            if (errs[t] == cudaSuccess)
                errs[t] = cudaMemcpyAsync(static_cast<char*>(dst) + off, ctx->stage_pinned[slot], len, cudaMemcpyHostToDevice, st);
            if (errs[t] == cudaSuccess) errs[t] = cudaEventRecord(ctx->stage_ev[slot], st);
        }
    };
    // the ring may still be draining from the previous staged copy (a different stream): wait before refilling it
    for (int i = 0; i < TMAX * S; i++)
        if (ctx->stage_ev[i]) HALO_CUDA(cudaEventSynchronize(ctx->stage_ev[i]));
    std::thread th[TMAX];
    int spawned = 0;
    for (int t = 1; t < T; t++) {
        try {
            th[t] = std::thread(work, t);
            spawned |= 1 << t;
        } catch (const std::system_error&) {
        }
    }
    work(0);
    for (int t = 1; t < T; t++) {
        if (spawned & (1 << t))
            th[t].join();
        else
            work(t);  // no thread available: this thread takes the chunks as well
    }
    for (int t = 0; t < T; t++)
        if (errs[t] != cudaSuccess) throw CudaError{errs[t], "staged host-to-device copy", __FILE__, __LINE__};
}

void async_init(halo_ctx* ctx) {
    if (ctx->copy_stream) return;
    HALO_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    int prio_lo = 0, prio_hi = 0;
    HALO_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    HALO_CUDA(cudaStreamCreateWithPriority(&ctx->sort_stream, cudaStreamNonBlocking, prio_hi));
    for (auto& s : ctx->slots) {
        HALO_CUDA(cudaEventCreateWithFlags(&s.sorted, cudaEventDisableTiming));
        HALO_CUDA(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
        HALO_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
        HALO_CUDA(cudaMallocHost(reinterpret_cast<void**>(&s.h_parts), 3 * MSM_MAX_WINDOWS * sizeof(xyzz_t)));
    }
}
}  // namespace halo

#define HALO_TRY(ctx) \
    try {             \
        HALO_CUDA(cudaSetDevice((ctx)->device));
#define HALO_CATCH(ctx)                                                                                        \
    }                                                                                                          \
    catch (const halo::CudaError& e) {                                                                         \
        return halo::set_error(ctx, HALO_ECUDA, "CUDA error: %s at %s:%d", cudaGetErrorString(e.err), e.file, e.line); \
    }                                                                                                          \
    catch (const std::bad_alloc&) {                                                                            \
        return halo::set_error(ctx, HALO_ENOMEM, "out of host memory%s%s%d", "", "", 0);                        \
    }                                                                                                          \
    catch (...) { /* nothing unwinds across the C ABI */                                                       \
        return halo::set_error(ctx, HALO_ECUDA, "unexpected internal exception%s%s%d", "", "", 0);              \
    }                                                                                                          \
    return HALO_OK;

static int fail(halo_ctx* ctx, int code, const char* msg) {
    if (ctx) ctx->last_error = msg;
    return code;
}

static void out_jac_from_xyzz(const xyzz_t& p, uint64_t out[12]) {
    jac_t j;
    xyzz_to_jac(j, p);
    memcpy(out, &j, 96);
}

extern "C" {

int halo_ctx_create(int device, uint64_t max_n, halo_ctx** out) {
    if (!out) return HALO_EINVAL;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) return HALO_ECUDA;
    halo_ctx* ctx = new halo_ctx();
    ctx->device = device;
    ctx->max_n = max_n;
    try {
        HALO_CUDA(cudaSetDevice(device));
        HALO_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        HALO_CUDA(cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device));
        {  // staging threads for pageable host buffers: the host's hardware threads shared among the visible GPUs, 4 .. 8
            int ndev = 1;
            if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) ndev = 1;
            const int hw = (int)std::thread::hardware_concurrency();
            const int t = hw / ndev;
            ctx->tune_stage_threads = t < 4 ? 4 : t > halo_ctx::STAGE_THREADS ? halo_ctx::STAGE_THREADS : t;
        }
        HALO_CUDA(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
        HALO_CUDA(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
        HALO_CUDA(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
        for (auto& e : ctx->ev) HALO_CUDA(cudaEventCreate(&e));
    } catch (const halo::CudaError&) {
        delete ctx;
        return HALO_ECUDA;
    }
    *out = ctx;
    return HALO_OK;
}

void halo_ctx_destroy(halo_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->gens.release();
    ctx->fixed_table.release();
    ctx->gens_pre.release();
    ctx->stage_scalars.release();
    ctx->stage_bases.release();
    ctx->stage_misc.release();
    ctx->poly_dev.release();
    ctx->polys_dev.release();
    ctx->polys_off.release();
    ctx->quot_dev.release();
    ctx->quot_scratch.release();
    ctx->lincomb_claims.release();
    for (halo::DevBuf* b : {&ctx->combine_in, &ctx->combine_work, &ctx->combine_inv_scratch}) b->release();
    for (halo::DevBuf* b : {&ctx->ipa_G, &ctx->ipa_cs, &ctx->ipa_zs, &ctx->ipa_pbar, &ctx->ipa_tail, &ctx->ipa_frozen,
                           &ctx->ipa_sums, &ctx->ipa_den, &ctx->ipa_inv_scratch, &ctx->ipa_bx, &ctx->ipa_diff, &ctx->ipa_den2, &ctx->ipa_ops}) b->release();
    for (MsmWorkspace* wsp : {&ctx->ws, &ctx->ws2}) {
    MsmWorkspace& ws = *wsp;
    for (DevBuf* b : {&ws.counts, &ws.offsets, &ws.cursor, &ws.entries, &ws.buckets, &ws.wsums, &ws.scan_tmp,
                      &ws.task_bucket, &ws.task_partial, &ws.split_ctrl, &ws.split_tasks, &ws.split_buckets, &ws.split_partials,
                      &ws.pt_a, &ws.pt_b, &ws.pt_prefix, &ws.pt_levels, &ws.sort_tmp, &ws.sort_coarse, &ws.sort_fine})
        b->release();
    }
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    for (auto& e : ctx->ev)
        if (e) cudaEventDestroy(e);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    for (void* p : ctx->stage_pinned)
        if (p) cudaFreeHost(p);
    for (cudaEvent_t e : ctx->stage_ev)
        if (e) cudaEventDestroy(e);
    for (auto& s : ctx->slots) {
        s.scalars.release();
        for (DevBuf* b : {&s.sort_ws.counts, &s.sort_ws.offsets, &s.sort_ws.entries, &s.sort_ws.scan_tmp, &s.sort_ws.sort_tmp, &s.sort_ws.sort_coarse, &s.sort_ws.sort_fine}) b->release();
        if (s.sorted) cudaEventDestroy(s.sorted);
        if (s.copied) cudaEventDestroy(s.copied);
        if (s.done) cudaEventDestroy(s.done);
        if (s.h_parts) cudaFreeHost(s.h_parts);
    }
    for (DevBuf* b : {&ctx->hb.scalars, &ctx->hb.companion, &ctx->hb.parts}) b->release();
    if (ctx->hb.done) cudaEventDestroy(ctx->hb.done);
    if (ctx->hb.h_parts) cudaFreeHost(ctx->hb.h_parts);
    for (auto& b : ctx->many) {
        for (DevBuf* d : {&b.scalars, &b.seg_off, &b.parts}) d->release();
        if (b.h_seg_off) cudaFreeHost(b.h_seg_off);
        if (b.h_parts) cudaFreeHost(b.h_parts);
        if (b.copied) cudaEventDestroy(b.copied);
        if (b.done) cudaEventDestroy(b.done);
    }
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->sort_stream) cudaStreamDestroy(ctx->sort_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* halo_last_error(halo_ctx* ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }
const char* halo_curve_name(void) { return HALO_CURVE_NAME; }
uint64_t halo_kernel_launches(halo_ctx* ctx) { return ctx ? ctx->kernel_launches : 0; }
uint64_t halo_num_generators(halo_ctx* ctx) { return ctx ? ctx->n_gens : 0; }
int halo_set_msm_window(halo_ctx* ctx, int c) {
    if (!ctx || c < 0 || c > 20) return HALO_EINVAL;
    ctx->force_c = c;
    return HALO_OK;
}
int halo_set_tuning(halo_ctx* ctx, const char* key, int value) {
    if (!ctx || !key) return HALO_EINVAL;
    // values that become a plan or a launch geometry are checked, not cast or silently replaced
    bool ok = true;
    if (!strcmp(key, "acc_static")) ok = value >= 0 && value <= 2;
    else if (!strcmp(key, "acc_blocks_per_sm")) ok = value >= 0 && value <= 32;
    else if (!strcmp(key, "acc_quad_max_buckets")) ok = value >= 0;
    else if (!strcmp(key, "acc_quad_lanes")) ok = value == 0 || value == 2 || value == 4;
    else if (!strcmp(key, "acc_quad_blocks")) ok = value == 0 || value == 4 || value == 6;
    else if (!strcmp(key, "pair_passes")) ok = value >= -1;
    else if (!strcmp(key, "ipa_frozen_c")) ok = value == 0 || (value >= 4 && value <= 20);  // the range of halo_set_msm_window
    if (!ok) return fail(ctx, HALO_EINVAL, "halo_set_tuning: value out of range for this key (include/halo_b200.h)");
    if (!strcmp(key, "acc_static")) ctx->tune_acc_static = value;
    else if (!strcmp(key, "acc_blocks_per_sm")) ctx->tune_acc_blocks_per_sm = value;
    else if (!strcmp(key, "acc_quad")) ctx->tune_acc_quad = value;
    else if (!strcmp(key, "acc_quad_max_buckets")) ctx->tune_acc_quad_max_buckets = value;
    else if (!strcmp(key, "acc_quad_lanes")) ctx->tune_acc_quad_lanes = value;
    else if (!strcmp(key, "acc_quad_blocks")) ctx->tune_acc_quad_blocks = value;
    else if (!strcmp(key, "pair_passes")) ctx->tune_pair_passes = value;
    else if (!strcmp(key, "split_blocking")) ctx->tune_split_blocking = value;
    else if (!strcmp(key, "split_first_16ths")) ctx->tune_split_first_16ths = value < 1 ? 1 : value > 15 ? 15 : value;
    else if (!strcmp(key, "split_second_16ths")) ctx->tune_split_second_16ths = value < 0 ? 0 : value > 14 ? 14 : value;
    else if (!strcmp(key, "sort_ahead")) ctx->tune_sort_ahead = value;
    else if (!strcmp(key, "stage_pageable")) ctx->tune_stage_pageable = value;
    else if (!strcmp(key, "stage_threads")) ctx->tune_stage_threads = value;
    else if (!strcmp(key, "reduce_quad")) ctx->tune_reduce_quad = value;
    else if (!strcmp(key, "sort2")) ctx->tune_sort2 = value;
    else if (!strcmp(key, "sort2_min_lg")) ctx->tune_sort2_min_lg = value;
    else if (!strcmp(key, "pair_bwd_async")) ctx->tune_pair_bwd_async = value;
    else if (!strcmp(key, "ipa_defer_rounds")) ctx->tune_ipa_defer = value;
    else if (!strcmp(key, "ipa_fold_call_min_lg")) ctx->tune_fold_call_min_lg = value;
    else if (!strcmp(key, "ipa_defer2_rounds")) ctx->tune_ipa_defer2 = value;
    else if (!strcmp(key, "ipa_two_lanes")) ctx->tune_ipa_two_lanes = value;
    else if (!strcmp(key, "ipa_freeze_len")) ctx->tune_ipa_freeze_len = value;
    else if (!strcmp(key, "ipa_frozen_c")) ctx->tune_ipa_frozen_c = value;
    else if (!strcmp(key, "combine_min_outputs")) ctx->tune_combine_min_outputs = value;
    else return fail(ctx, HALO_EINVAL, "halo_set_tuning: unknown key");
    return HALO_OK;
}
int halo_set_profiling(halo_ctx* ctx, int on) {
    if (!ctx) return HALO_EINVAL;
    ctx->profile = on != 0;
    return HALO_OK;
}
int halo_last_msm_timings(halo_ctx* ctx, float out_ms[6]) {
    if (!ctx) return HALO_EINVAL;
    const Timings& t = ctx->last;
    out_ms[0] = t.digits_ms;
    out_ms[1] = t.scan_ms;
    out_ms[2] = t.scatter_ms;
    out_ms[3] = t.accumulate_ms;
    out_ms[4] = t.reduce_ms;
    out_ms[5] = t.total_ms;
    return HALO_OK;
}

int halo_derive_generators(halo_ctx* ctx, uint64_t n) { return halo_derive_generators_range(ctx, 0, n); }

int halo_points_sum(const uint64_t* points_jac, uint64_t g, uint64_t out_jac[12]) {
    if (!out_jac || (!points_jac && g)) return HALO_EINVAL;
    xyzz_t acc;
    xyzz_set_inf(acc);
    for (uint64_t i = 0; i < g; i++) {
        jac_t j;
        memcpy(&j, points_jac + 12 * i, 96);
        xyzz_t q;
        jac_to_xyzz(q, j);
        xyzz_add(acc, q);
    }
    out_jac_from_xyzz(acc, out_jac);
    return HALO_OK;
}

int halo_points_equal(const uint64_t a_jac[12], const uint64_t b_jac[12]) {
    jac_t a, b;
    memcpy(&a, a_jac, 96);
    memcpy(&b, b_jac, 96);
    bool ia = fp_is_zero(a.z), ib = fp_is_zero(b.z);
    if (ia || ib) return ia && ib;
    fq_t za2, zb2, l, r;
    fp_sqr(za2, a.z);
    fp_sqr(zb2, b.z);
    fp_mul(l, a.x, zb2);
    fp_mul(r, b.x, za2);
    if (!fp_eq(l, r)) return 0;
    fp_mul(l, a.y, zb2);
    fp_mul(l, l, b.z);
    fp_mul(r, b.y, za2);
    fp_mul(r, r, a.z);
    return fp_eq(l, r) ? 1 : 0;
}

int halo_timer_start(halo_ctx* ctx) {
    if (!ctx) return HALO_EINVAL;
    HALO_TRY(ctx)
    HALO_CUDA(cudaEventRecord(ctx->ev[6], ctx->stream));
    HALO_CATCH(ctx)
}
int halo_timer_stop(halo_ctx* ctx, float* elapsed_ms) {
    if (!ctx || !elapsed_ms) return HALO_EINVAL;
    HALO_TRY(ctx)
    HALO_CUDA(cudaEventRecord(ctx->ev[7], ctx->stream));
    HALO_CUDA(cudaEventSynchronize(ctx->ev[7]));
    HALO_CUDA(cudaEventElapsedTime(elapsed_ms, ctx->ev[6], ctx->ev[7]));
    HALO_CATCH(ctx)
}

int halo_derive_generators_range(halo_ctx* ctx, uint64_t first, uint64_t n) {
    if (!ctx) return HALO_EINVAL;
    if (n == 0 || n > ctx->max_n) return fail(ctx, HALO_EINVAL, "halo_derive_generators: n exceeds max_n");
    HALO_TRY(ctx)
    // P_0 = S, P_1 = H land in a small staging buffer; G_i = P_{i+2} directly in the resident array
    ctx->gens.reserve(n * sizeof(affine_t));
    ctx->stage_misc.reserve(2 * sizeof(affine_t));
    params_derive_points(ctx, 0, 2, ctx->stage_misc.as<affine_t>());
    params_derive_points(ctx, 2 + first, n, ctx->gens.as<affine_t>());
    affine_t sh[2];
    HALO_CUDA(cudaMemcpyAsync(sh, ctx->stage_misc.p, sizeof sh, cudaMemcpyDeviceToHost, ctx->stream));
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->S = sh[0];
    ctx->H = sh[1];
    ctx->have_SH = true;
    ctx->n_gens = n;
    ctx->pre_n = 0;  // tables of precomputed multiples are stale
    HALO_CATCH(ctx)
}

int halo_precompute_generators(halo_ctx* ctx, int c) {
    if (!ctx) return HALO_EINVAL;
    if (ctx->n_gens == 0) return fail(ctx, HALO_ESTATE, "halo_precompute_generators: no generators resident");
    if (c != 0 && (c < 8 || c > 24)) return fail(ctx, HALO_EINVAL, "halo_precompute_generators: window must be 0 (auto) or 8..24");
    HALO_TRY(ctx)
    msm_precompute_tables(ctx, c);
    HALO_CATCH(ctx)
}

int halo_set_fixed_base(halo_ctx* ctx, int on) {
    if (!ctx) return HALO_EINVAL;
    ctx->use_fixed = on != 0;
    return HALO_OK;
}

int halo_load_generators(halo_ctx* ctx, const uint64_t S_jac[12], const uint64_t H_jac[12], const uint64_t* gs_affine,
                         uint64_t n) {
    if (!ctx || !gs_affine) return HALO_EINVAL;
    if (n == 0 || n > ctx->max_n) return fail(ctx, HALO_EINVAL, "halo_load_generators: n exceeds max_n");
    HALO_TRY(ctx)
    ctx->gens.reserve(n * sizeof(affine_t));
    HALO_CUDA(cudaMemcpyAsync(ctx->gens.p, gs_affine, n * sizeof(affine_t), cudaMemcpyHostToDevice, ctx->stream));
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    if (S_jac && H_jac) {
        jac_t s, h;
        memcpy(&s, S_jac, 96);
        memcpy(&h, H_jac, 96);
        xyzz_t t;
        jac_to_xyzz(t, s);
        xyzz_to_affine(ctx->S, t);
        jac_to_xyzz(t, h);
        xyzz_to_affine(ctx->H, t);
        ctx->have_SH = true;
    }
    ctx->n_gens = n;
    ctx->pre_n = 0;
    HALO_CATCH(ctx)
}

// ---- generator store (SURVEY 8(f).3) ---------------------------------------------------------------------------------
// The reference keeps its public parameters as generated source (main.rs:47-67 writes them, consts.rs holds 16 386 of
// them, and report.md:2081-2086 names that as the limit on n).  Here they are a flat file of the device records:
//   header (64 B): magic "HALOGEN1", curve name (8 B, zero padded), n, record size (64), checksum, 24 B reserved
//   S, H           2 x 64 B Montgomery affine
//   G_0 .. G_{n-1} n x 64 B Montgomery affine (x | y, little-endian limbs: the bytes of consts.rs' mk_aff! arguments)
// Loading streams the file through two pinned buffers (the read of chunk k+1 overlaps the copy of chunk k), verifies
// the checksum and checks on the device that every record is a canonical point on the curve.
namespace {
constexpr char STORE_MAGIC[8] = {'H', 'A', 'L', 'O', 'G', 'E', 'N', '1'};
constexpr size_t STORE_CHUNK = 32u << 20;
struct StoreHeader {
    char magic[8];
    char curve[8];
    uint64_t n;
    uint64_t record_bytes;
    uint64_t checksum;
    uint64_t reserved[3];
};
static_assert(sizeof(StoreHeader) == 64, "store header layout");
// 64-bit multiply-rotate checksum over the u64 words of S, H and the records, in file order
inline uint64_t store_mix(uint64_t h, const void* data, size_t bytes) {
    const uint64_t* w = static_cast<const uint64_t*>(data);
    for (size_t i = 0; i < bytes / 8; i++) {
        h ^= w[i];
        h *= 0x9e3779b97f4a7c15ull;
        h = (h << 29) | (h >> 35);
    }
    return h;
}
struct FileCloser {
    FILE* f;
    ~FileCloser() {
        if (f) fclose(f);
    }
};
struct PinnedPair {
    void* p[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    ~PinnedPair() {
        for (int i = 0; i < 2; i++) {
            if (p[i]) cudaFreeHost(p[i]);
            if (ev[i]) cudaEventDestroy(ev[i]);
        }
    }
};
}  // namespace

int halo_save_generators(halo_ctx* ctx, const char* path) {
    if (!ctx || !path) return HALO_EINVAL;
    if (ctx->n_gens == 0 || !ctx->have_SH) return fail(ctx, HALO_ESTATE, "halo_save_generators: no generators resident");
    HALO_TRY(ctx)
    FileCloser fc{fopen(path, "wb")};
    if (!fc.f) return fail(ctx, HALO_EIO, "halo_save_generators: cannot open the file for writing");
    StoreHeader hd = {};
    memcpy(hd.magic, STORE_MAGIC, 8);
    strncpy(hd.curve, HALO_CURVE_NAME, 8);
    hd.n = ctx->n_gens;
    hd.record_bytes = sizeof(affine_t);
    affine_t sh[2] = {ctx->S, ctx->H};
    uint64_t sum = store_mix(0, sh, sizeof sh);
    if (fwrite(&hd, sizeof hd, 1, fc.f) != 1 || fwrite(sh, sizeof sh, 1, fc.f) != 1)
        return fail(ctx, HALO_EIO, "halo_save_generators: write failed");
    PinnedPair pp;
    for (int i = 0; i < 2; i++) {
        HALO_CUDA(cudaMallocHost(&pp.p[i], STORE_CHUNK));
        HALO_CUDA(cudaEventCreateWithFlags(&pp.ev[i], cudaEventDisableTiming));
    }
    const size_t total = ctx->n_gens * sizeof(affine_t);
    const char* src = ctx->gens.as<char>();
    size_t issued = 0, written = 0;
    int k = 0;
    auto issue = [&](int b) {
        size_t len = total - issued < STORE_CHUNK ? total - issued : STORE_CHUNK;
        HALO_CUDA(cudaMemcpyAsync(pp.p[b], src + issued, len, cudaMemcpyDeviceToHost, ctx->stream));
        HALO_CUDA(cudaEventRecord(pp.ev[b], ctx->stream));
        issued += len;
    };
    if (issued < total) issue(0);
    while (written < total) {  // the device-to-host copy of chunk k+1 runs while chunk k is hashed and written
        int b = k & 1;
        if (issued < total) issue(b ^ 1);
        HALO_CUDA(cudaEventSynchronize(pp.ev[b]));
        size_t len = total - written < STORE_CHUNK ? total - written : STORE_CHUNK;
        sum = store_mix(sum, pp.p[b], len);
        if (fwrite(pp.p[b], 1, len, fc.f) != len) return fail(ctx, HALO_EIO, "halo_save_generators: write failed");
        written += len;
        k++;
    }
    hd.checksum = sum;
    if (fseek(fc.f, 0, SEEK_SET) != 0 || fwrite(&hd, sizeof hd, 1, fc.f) != 1 || fflush(fc.f) != 0)
        return fail(ctx, HALO_EIO, "halo_save_generators: write failed");
    HALO_CATCH(ctx)
}

int halo_load_generators_file(halo_ctx* ctx, const char* path, uint64_t n) {
    if (!ctx || !path) return HALO_EINVAL;
    HALO_TRY(ctx)
    FileCloser fc{fopen(path, "rb")};
    if (!fc.f) return fail(ctx, HALO_EIO, "halo_load_generators_file: cannot open the file");
    StoreHeader hd;
    affine_t sh[2];
    if (fread(&hd, sizeof hd, 1, fc.f) != 1 || fread(sh, sizeof sh, 1, fc.f) != 1)
        return fail(ctx, HALO_EIO, "halo_load_generators_file: truncated header");
    char curve[8] = {};
    strncpy(curve, HALO_CURVE_NAME, 8);
    if (memcmp(hd.magic, STORE_MAGIC, 8) != 0 || hd.record_bytes != sizeof(affine_t))
        return fail(ctx, HALO_EINVAL, "halo_load_generators_file: not a generator store");
    if (memcmp(hd.curve, curve, 8) != 0)
        return fail(ctx, HALO_EINVAL, "halo_load_generators_file: the store holds points of the other curve");
    if (n == 0) n = hd.n;
    if (n > hd.n) return fail(ctx, HALO_EINVAL, "halo_load_generators_file: the store holds fewer generators than requested");
    if (n > ctx->max_n) return fail(ctx, HALO_EINVAL, "halo_load_generators_file: n exceeds max_n");
    ctx->n_gens = 0;  // the resident set is replaced; a failure below leaves the context without generators
    ctx->pre_n = 0;
    ctx->gens.reserve(n * sizeof(affine_t));
    PinnedPair pp;
    for (int i = 0; i < 2; i++) {
        HALO_CUDA(cudaMallocHost(&pp.p[i], STORE_CHUNK));
        HALO_CUDA(cudaEventCreateWithFlags(&pp.ev[i], cudaEventDisableTiming));
    }
    // a prefix of the store is a valid parameter set (G_0..G_{n-1}); the checksum covers the whole file, so it is
    // verified only when all of it is read -- the on-curve check below covers every record either way
    const size_t total = n * sizeof(affine_t);
    uint64_t sum = store_mix(0, sh, sizeof sh);
    size_t done = 0;
    for (int k = 0; done < total; k++) {
        int b = k & 1;
        if (k >= 2) HALO_CUDA(cudaEventSynchronize(pp.ev[b]));  // the copy out of this buffer two chunks ago
        size_t len = total - done < STORE_CHUNK ? total - done : STORE_CHUNK;
        if (fread(pp.p[b], 1, len, fc.f) != len) return fail(ctx, HALO_EIO, "halo_load_generators_file: truncated file");
        sum = store_mix(sum, pp.p[b], len);
        HALO_CUDA(cudaMemcpyAsync(ctx->gens.as<char>() + done, pp.p[b], len, cudaMemcpyHostToDevice, ctx->stream));
        HALO_CUDA(cudaEventRecord(pp.ev[b], ctx->stream));
        done += len;
    }
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    if (n == hd.n && sum != hd.checksum) return fail(ctx, HALO_EINVAL, "halo_load_generators_file: checksum mismatch");
    ctx->stage_bases.reserve(sizeof sh);
    HALO_CUDA(cudaMemcpyAsync(ctx->stage_bases.p, sh, sizeof sh, cudaMemcpyHostToDevice, ctx->stream));
    if (params_count_off_curve(ctx, ctx->stage_bases.as<affine_t>(), 2) != 0 ||
        params_count_off_curve(ctx, ctx->gens.as<affine_t>(), n) != 0)
        return fail(ctx, HALO_EINVAL, "halo_load_generators_file: the store holds records that are not points on the curve");
    ctx->S = sh[0];
    ctx->H = sh[1];
    ctx->have_SH = true;
    ctx->n_gens = n;
    HALO_CATCH(ctx)
}

int halo_get_generators(halo_ctx* ctx, uint64_t off, uint64_t n, uint64_t* out_affine) {
    if (!ctx || !out_affine) return HALO_EINVAL;
    if (off + n > ctx->n_gens) return fail(ctx, HALO_EINVAL, "halo_get_generators: range exceeds resident generators");
    HALO_TRY(ctx)
    HALO_CUDA(cudaMemcpyAsync(out_affine, ctx->gens.as<affine_t>() + off, n * sizeof(affine_t), cudaMemcpyDeviceToHost,
                              ctx->stream));
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    HALO_CATCH(ctx)
}

int halo_get_SH(halo_ctx* ctx, uint64_t S_jac[12], uint64_t H_jac[12]) {
    if (!ctx || !ctx->have_SH) return fail(ctx, HALO_ESTATE, "halo_get_SH: parameters not loaded");
    xyzz_t t;
    xyzz_from_affine(t, ctx->S);
    out_jac_from_xyzz(t, S_jac);
    xyzz_from_affine(t, ctx->H);
    out_jac_from_xyzz(t, H_jac);
    return HALO_OK;
}

int halo_derive_points(halo_ctx* ctx, uint64_t start, uint64_t count, uint64_t* out_affine) {
    if (!ctx || !out_affine) return HALO_EINVAL;
    HALO_TRY(ctx)
    ctx->stage_bases.reserve(count * sizeof(affine_t));
    params_derive_points(ctx, start, count, ctx->stage_bases.as<affine_t>());
    HALO_CUDA(cudaMemcpyAsync(out_affine, ctx->stage_bases.p, count * sizeof(affine_t), cudaMemcpyDeviceToHost, ctx->stream));
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    HALO_CATCH(ctx)
}

int halo_msm_gens_resident(halo_ctx* ctx, const void* d_scalars, uint64_t off, uint64_t n, uint64_t out_jac[12]) {
    if (!ctx || !out_jac || (!d_scalars && n)) return HALO_EINVAL;
    if (off + n > ctx->n_gens) return fail(ctx, HALO_ESTATE, "halo_msm_gens: range exceeds resident generators");
    HALO_TRY(ctx)
    xyzz_t r;
    msm_gens_device(ctx, reinterpret_cast<const fr_t*>(d_scalars), off, n, r);
    out_jac_from_xyzz(r, out_jac);
    HALO_CATCH(ctx)
}

int halo_msm_gens(halo_ctx* ctx, const uint64_t* scalars, uint64_t off, uint64_t n, uint64_t out_jac[12]) {
    if (!ctx || !out_jac || (!scalars && n)) return HALO_EINVAL;
    if (off + n > ctx->n_gens) return fail(ctx, HALO_ESTATE, "halo_msm_gens: range exceeds resident generators");
    // Large calls are split into point slices that go through the two pipeline slots: the host-to-device copies of the later
    // slices overlap the kernels of the earlier ones (2^24 scalars from pinned memory, round 1: 45.4 ms unsplit, 41.1 ms with
    // two halves, 38.2 ms with 5/16 + 11/16; round 2: 37.0 ms with 5/16 + 11/16, 36.05 ms with 2/16 + 5/16 + 9/16; from
    // pageable memory 41.9 -> 39.8 ms); the partial sums are added on the host.
    if (ctx->tune_split_blocking > 0 && n >= ((uint64_t)1 << ctx->tune_split_blocking) && !ctx->slots[0].active && !ctx->slots[1].active) {
        // slices in sixteenths of n: the first slice's copy is the exposed one; with a second cut the third slice is submitted
        // into the first slice's slot as soon as that one is collected (two slots in flight at any time)
        const int a = ctx->tune_split_first_16ths, b = ctx->tune_split_second_16ths;
        uint64_t cut[4] = {0, n / 16 * (uint64_t)a, 0, n};
        int ns = 2;
        if (b > 0 && a + b < 16) {
            cut[2] = n / 16 * (uint64_t)(a + b);
            ns = 3;
        } else {
            cut[2] = n;
        }
        int tk[3];
        uint64_t parts[36];
        int rc = 0, submitted = 0, collected = 0;
        for (int i = 0; i < ns && !rc; i++) {
            if (i == 2) {
                rc = halo_msm_gens_collect(ctx, tk[0], parts);
                collected = 1;
                if (rc) break;
            }
            rc = halo_msm_gens_submit(ctx, scalars + 4 * cut[i], off + cut[i], cut[i + 1] - cut[i], &tk[i]);
            if (!rc) submitted = i + 1;
        }
        for (int i = collected; i < submitted; i++) {  // on failure this drains what is in flight; the first error is the one returned
            const int rci = halo_msm_gens_collect(ctx, tk[i], parts + 12 * i);
            if (!rc) rc = rci;
        }
        if (rc) return rc;
        return halo_points_sum(parts, (uint64_t)ns, out_jac);
    }
    HALO_TRY(ctx)
    ctx->stage_scalars.reserve((n ? n : 1) * sizeof(fr_t));
    if (n) h2d_copy(ctx, ctx->stage_scalars.p, scalars, n * sizeof(fr_t), ctx->stream);
    xyzz_t r;
    msm_gens_device(ctx, ctx->stage_scalars.as<fr_t>(), off, n, r);
    out_jac_from_xyzz(r, out_jac);
    HALO_CATCH(ctx)
}

// ---- halo_msm_gens_many (DESIGN.md K2c): k MSMs over the resident generators as segmented MSMs ----
namespace {
constexpr uint64_t MANY_MAX_SCALARS = (uint64_t)1 << 24;  // per group: the scalars, entries and buckets of the library's 2^24-point MSM
constexpr uint64_t MANY_MAX_ENTRIES = (uint64_t)1 << 28;
constexpr uint64_t MANY_MAX_BUCKETS = (uint64_t)1 << 23;  // the scan's limit, (NB + 4095) / 4096 <= 2048
constexpr uint64_t MANY_SORT2_BUCKETS = (uint64_t)1 << 21;  // the two-level sort's 2048 coarse bins of 1024 buckets
constexpr uint32_t MANY_MAX_SEGS = 256;  // bounds the window partials of a group (3 W segs points, pinned on the host)

// One segmented MSM: the non-empty outputs jobs[j0 .. j1) (their scalars are adjacent in the packed buffer, from s0 on).
struct ManyGroup {
    size_t j0, j1;
    uint64_t s0, ns, max_len;
    MsmPlan plan;
};

// Outputs in caller order, cut into groups of one plan within the limits above; a group of one output is an ordinary MSM.
// Each output's plan is that of a single MSM of its length; groups of short segments then narrow it.
std::vector<ManyGroup> many_groups(halo_ctx* ctx, const std::vector<uint64_t>& jobs, const uint64_t* lens, const uint64_t* starts) {
    std::vector<ManyGroup> gs;
    for (size_t j = 0; j < jobs.size(); j++) {
        const uint64_t len = lens[jobs[j]];
        const MsmPlan p = msm_plan(ctx, len, gens_use_fixed(ctx, len));
        if (!gs.empty()) {
            ManyGroup& g = gs.back();
            const uint64_t segs = g.j1 - g.j0 + 1, ns = g.ns + len, nb = segs * g.plan.NB, entries = ns * (uint64_t)p.W;
            const bool fits = p.c == g.plan.c && p.fixed == g.plan.fixed && segs <= MANY_MAX_SEGS && ns <= MANY_MAX_SCALARS &&
                              entries <= MANY_MAX_ENTRIES && nb <= MANY_MAX_BUCKETS &&
                              (entries < ((uint64_t)1 << ctx->tune_sort2_min_lg) || nb <= MANY_SORT2_BUCKETS);
            if (fits) {
                g.j1++;
                g.ns = ns;
                g.max_len = std::max(g.max_len, len);
                continue;
            }
        }
        gs.push_back(ManyGroup{j, j + 1, starts[jobs[j]], len, len, p});
    }
    for (ManyGroup& g : gs) {
        const uint32_t segs = (uint32_t)(g.j1 - g.j0);
        if (segs == 1) continue;
        // Window sweep of the segmented MSM (profiles/r06_commit_batch.jsonl, B200): 2^12-point segments, window 7 .. 13, best
        // at 8 -- 8 segments 0.77 ms (c = 11, the single-MSM window: 1.07), 64 segments 2.98 ms (4.56).  A batch fills the
        // machine, so the narrow window's smaller bucket reduction wins over the latency-bound single MSM's choice.  At 2^16 (8 /
        // 64 segments) the single-MSM window is within 3 % of the best: kept.  (2^13 .. 2^15: not measured.)
        const bool narrow = !g.plan.fixed && !ctx->force_c && segs >= 8 && g.max_len <= 4096 && g.plan.c > 8;
        g.plan = msm_plan(ctx, g.max_len, g.plan.fixed, narrow ? 8 : g.plan.c, segs);
    }
    return gs;
}

}  // namespace

int halo_msm_gens_many(halo_ctx* ctx, const uint64_t* scalars, const uint64_t* lens, uint64_t k, uint64_t* out_jac) {
    if (!ctx) return HALO_EINVAL;
    if (k == 0) return HALO_OK;
    if (!scalars || !lens || !out_jac) return HALO_EINVAL;
    std::vector<uint64_t> starts, jobs;  // packed position of every output; the outputs with scalars
    try {
        starts.resize(k);
        uint64_t total = 0;
        for (uint64_t j = 0; j < k; j++) {
            if (lens[j] > ctx->n_gens) return fail(ctx, HALO_ESTATE, "halo_msm_gens_many: length exceeds resident generators");
            starts[j] = total;
            total += lens[j];
            if (total < lens[j] || total > UINT64_MAX / sizeof(fr_t)) return fail(ctx, HALO_EINVAL, "halo_msm_gens_many: packed size overflows");
            if (lens[j]) jobs.push_back(j);
        }
    } catch (const std::bad_alloc&) {
        return fail(ctx, HALO_ENOMEM, "out of host memory");
    }
    HALO_TRY(ctx)
    for (uint64_t j = 0; j < k; j++)
        if (!lens[j]) {
            xyzz_t inf;
            xyzz_set_inf(inf);
            out_jac_from_xyzz(inf, out_jac + 12 * j);
        }
    std::vector<ManyGroup> groups = many_groups(ctx, jobs, lens, starts.data());
    const size_t G = groups.size();
    auto multi = [&](size_t g) { return groups[g].j1 - groups[g].j0 > 1; };
    // both buffers at the size of the largest group, before anything is in flight
    uint64_t max_ns = 0;
    size_t max_parts = 0;
    for (size_t g = 0; g < G; g++)
        if (multi(g)) {
            max_ns = std::max(max_ns, groups[g].ns);
            max_parts = std::max(max_parts, msm_parts(groups[g].plan));
        }
    if (max_ns) {
        async_init(ctx);
        for (auto& b : ctx->many) {
            if (!b.copied) {
                HALO_CUDA(cudaEventCreateWithFlags(&b.copied, cudaEventDisableTiming));
                HALO_CUDA(cudaEventCreateWithFlags(&b.done, cudaEventDisableTiming));
                HALO_CUDA(cudaMallocHost(reinterpret_cast<void**>(&b.h_seg_off), (size_t)(MANY_MAX_SEGS + 1) * 4));
            }
            b.scalars.reserve(max_ns * sizeof(fr_t));
            b.seg_off.reserve((size_t)(MANY_MAX_SEGS + 1) * 4);
            b.parts.reserve(max_parts * sizeof(xyzz_t));
            if (b.h_parts_cap < max_parts) {
                if (b.h_parts) HALO_CUDA(cudaFreeHost(b.h_parts));
                b.h_parts = nullptr;
                b.h_parts_cap = 0;
                HALO_CUDA(cudaMallocHost(reinterpret_cast<void**>(&b.h_parts), max_parts * sizeof(xyzz_t)));
                b.h_parts_cap = max_parts;
            }
        }
    }
    // Whatever happens below, nothing may still read the caller's scalars or write its outputs once this call returns.
    struct Drain {
        halo_ctx* c;
        ~Drain() {
            if (!c) return;
            cudaStreamSynchronize(c->copy_stream);
            cudaStreamSynchronize(c->stream);
        }
    } drain{max_ns ? ctx : nullptr};
    // group g's scalars and segment starts into buffer g & 1 on the copy stream, once the group two back has released it
    auto issue_copy = [&](size_t g) {
        const ManyGroup& gr = groups[g];
        halo_ctx::ManyBuf& b = ctx->many[g & 1];
        const uint32_t segs = (uint32_t)(gr.j1 - gr.j0);
        HALO_CUDA(cudaEventSynchronize(b.copied));  // the pinned segment starts of that group have left
        HALO_CUDA(cudaStreamWaitEvent(ctx->copy_stream, b.done, 0));
        for (uint32_t s = 0; s <= segs; s++) b.h_seg_off[s] = (uint32_t)((s < segs ? starts[jobs[gr.j0 + s]] : gr.s0 + gr.ns) - gr.s0);
        HALO_CUDA(cudaMemcpyAsync(b.seg_off.p, b.h_seg_off, (size_t)(segs + 1) * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
        h2d_copy(ctx, b.scalars.p, scalars + 4 * gr.s0, gr.ns * sizeof(fr_t), ctx->copy_stream);
        HALO_CUDA(cudaEventRecord(b.copied, ctx->copy_stream));
    };
    // group g's segmented MSM on the context stream, its window partials to the pinned host buffer
    auto launch = [&](size_t g) {
        const ManyGroup& gr = groups[g];
        halo_ctx::ManyBuf& b = ctx->many[g & 1];
        // FIXED base as the group's plan, which the segment lengths chose, not by the length of the whole group
        MsmInput in = gens_msm_input(ctx, gr.plan.fixed, b.scalars.as<fr_t>(), 0, gr.ns);
        in.segs = gr.plan.segs;
        in.seg_off = b.seg_off.as<uint32_t>();
        HALO_CUDA(cudaStreamWaitEvent(ctx->stream, b.copied, 0));
        msm_enqueue_to_host(ctx, in, gr.plan, b.parts.as<xyzz_t>(), b.h_parts);
        HALO_CUDA(cudaEventRecord(b.done, ctx->stream));
    };
    // host finish of group g, one segment per task (a variable-base finish is ~255 doublings)
    auto finish = [&](size_t g) {
        const ManyGroup& gr = groups[g];
        halo_ctx::ManyBuf& b = ctx->many[g & 1];
        HALO_CUDA(cudaEventSynchronize(b.done));
        const size_t per = msm_parts(gr.plan) / gr.plan.segs;
        auto one = [&](size_t s) {
            xyzz_t r;
            msm_finish_host(b.h_parts + per * s, gr.plan, r);
            out_jac_from_xyzz(r, out_jac + 12 * jobs[gr.j0 + s]);
        };
        if (gr.plan.fixed)
            for (size_t s = 0; s < gr.plan.segs; s++) one(s);
        else
            host_parallel(gr.plan.segs, one);
    };
    // Pipeline: the copy of group g+1 and the host finish of group g-1 run while group g is on the device.  A group of one
    // output drains the pipeline and takes the halo_msm_gens route.
    if (G && multi(0)) issue_copy(0);
    size_t pend = SIZE_MAX;  // group whose partials are outstanding
    for (size_t g = 0; g < G; g++) {
        if (!multi(g)) {
            if (pend != SIZE_MAX) finish(pend);
            pend = SIZE_MAX;
            const uint64_t j = jobs[groups[g].j0];
            const int rc = halo_msm_gens(ctx, scalars + 4 * starts[j], 0, lens[j], out_jac + 12 * j);
            if (rc) return rc;
        } else {
            launch(g);
        }
        if (g + 1 < G && multi(g + 1)) issue_copy(g + 1);
        if (multi(g)) {
            if (pend != SIZE_MAX) finish(pend);
            pend = g;
        }
    }
    if (pend != SIZE_MAX) finish(pend);
    HALO_CATCH(ctx)
}

// Shared body of the two submit entry points: host scalars are copied on the copy stream first; device-resident
// scalars (resident = true) are used in place and must stay untouched until the ticket is collected.
static int submit_impl(halo_ctx* ctx, const uint64_t* scalars, bool resident, uint64_t off, uint64_t n, int* ticket) {
    if (!ctx || !ticket || (!scalars && n)) return HALO_EINVAL;
    if (off + n > ctx->n_gens) return fail(ctx, HALO_ESTATE, "halo_msm_gens_submit: range exceeds resident generators");
    HALO_TRY(ctx)
    async_init(ctx);
    const int si = ctx->next_slot;
    halo_ctx::AsyncSlot& s = ctx->slots[si];
    if (s.active) return fail(ctx, HALO_ESTATE, "halo_msm_gens_submit: both pipeline slots are in flight; collect one first");
    s.empty = n == 0;
    if (!s.empty) {
        const bool ahead_on = ctx->tune_sort_ahead > 0 && n >= ((uint64_t)1 << 22);
        // (delaying the sort until the HBM-bound pass-0 gathers of the MSM in front are over measured slower: the
        // throttled sort then no longer fits under what is left of that MSM)
        // resident: the caller's producer of the scalars ran on a stream we do not know; like halo_msm_gens_resident, the
        // contract is that they are complete when this call is made
        const fr_t* d_scalars = reinterpret_cast<const fr_t*>(scalars);
        if (!resident) {
            s.scalars.reserve(n * sizeof(fr_t));
            h2d_copy(ctx, s.scalars.p, scalars, n * sizeof(fr_t), ctx->copy_stream);
            HALO_CUDA(cudaEventRecord(s.copied, ctx->copy_stream));
            HALO_CUDA(cudaStreamWaitEvent(ahead_on ? ctx->sort_stream : ctx->stream, s.copied, 0));
            d_scalars = s.scalars.as<fr_t>();
        }
        const bool fixed = gens_use_fixed(ctx, n);
        s.plan = msm_plan(ctx, n, fixed);
        ctx->ws.wsums.reserve((size_t)6 * 3 * MSM_MAX_WINDOWS * sizeof(xyzz_t));
        xyzz_t* d_parts = ctx->ws.wsums.as<xyzz_t>() + (size_t)(4 + si) * 3 * MSM_MAX_WINDOWS;  // slots 0-3 belong to msm_batch
        // the sort buffers of this slot were last read by the accumulation of the MSM two submits ago, which the caller
        // has collected (slot free) -- so the sort may start as soon as the scalars have arrived
        SortAhead ahead{&s.sort_ws, ctx->sort_stream, s.sorted, ctx->tune_sort_ahead};
        msm_enqueue_to_host(ctx, gens_msm_input(ctx, fixed, d_scalars, off, n), s.plan, d_parts, s.h_parts, 0, ahead_on ? &ahead : nullptr);
        HALO_CUDA(cudaEventRecord(s.done, ctx->stream));
    }
    s.active = true;
    *ticket = si;
    ctx->next_slot = si ^ 1;
    HALO_CATCH(ctx)
}

int halo_msm_gens_submit(halo_ctx* ctx, const uint64_t* scalars, uint64_t off, uint64_t n, int* ticket) {
    return submit_impl(ctx, scalars, false, off, n, ticket);
}

int halo_msm_gens_submit_resident(halo_ctx* ctx, const void* d_scalars, uint64_t off, uint64_t n, int* ticket) {
    return submit_impl(ctx, reinterpret_cast<const uint64_t*>(d_scalars), true, off, n, ticket);
}

int halo_msm_gens_collect(halo_ctx* ctx, int ticket, uint64_t out_jac[12]) {
    if (!ctx || !out_jac || ticket < 0 || ticket > 1) return HALO_EINVAL;
    halo_ctx::AsyncSlot& s = ctx->slots[ticket];
    if (!s.active) return fail(ctx, HALO_ESTATE, "halo_msm_gens_collect: ticket not in flight");
    HALO_TRY(ctx)
    xyzz_t r;
    if (s.empty) {
        xyzz_set_inf(r);
    } else {
        HALO_CUDA(cudaEventSynchronize(s.done));
        msm_finish_host(s.h_parts, s.plan, r);
    }
    s.active = false;
    out_jac_from_xyzz(r, out_jac);
    HALO_CATCH(ctx)
}

int halo_msm(halo_ctx* ctx, const uint64_t* bases_affine, const uint8_t* inf_flags, const uint64_t* scalars, uint64_t n,
             uint64_t out_jac[12]) {
    if (!ctx || !out_jac || ((!scalars || !bases_affine) && n)) return HALO_EINVAL;
    if (n > ctx->max_n) return fail(ctx, HALO_EINVAL, "halo_msm: n exceeds max_n");
    HALO_TRY(ctx)
    ctx->stage_scalars.reserve((n ? n : 1) * sizeof(fr_t));
    ctx->stage_bases.reserve((n ? n : 1) * sizeof(affine_t));
    if (n) {
        h2d_copy(ctx, ctx->stage_scalars.p, scalars, n * sizeof(fr_t), ctx->stream);
        h2d_copy(ctx, ctx->stage_bases.p, bases_affine, n * sizeof(affine_t), ctx->stream);
        if (inf_flags) {
            ctx->stage_misc.reserve(n);
            mark_infinity(ctx, ctx->stream, ctx->stage_bases.as<affine_t>(), ctx->stage_misc.as<uint8_t>(), inf_flags, n);
        }
    }
    xyzz_t r;
    msm_device(ctx, ctx->stage_bases.as<affine_t>(), ctx->stage_scalars.as<fr_t>(), n, r);
    out_jac_from_xyzz(r, out_jac);
    HALO_CATCH(ctx)
}

int halo_msm_jac(halo_ctx* ctx, const uint64_t* bases_jac, const uint64_t* scalars, uint64_t n, uint64_t out_jac[12]) {
    if (!ctx || !out_jac || ((!scalars || !bases_jac) && n)) return HALO_EINVAL;
    if (n > ctx->max_n) return fail(ctx, HALO_EINVAL, "halo_msm_jac: n exceeds max_n");
    HALO_TRY(ctx)
    ctx->stage_scalars.reserve((n ? n : 1) * sizeof(fr_t));
    ctx->stage_bases.reserve((n ? n : 1) * sizeof(affine_t));
    ctx->stage_misc.reserve((n ? n : 1) * sizeof(jac_t));
    if (n) {
        HALO_CUDA(cudaMemcpyAsync(ctx->stage_scalars.p, scalars, n * sizeof(fr_t), cudaMemcpyHostToDevice, ctx->stream));
        HALO_CUDA(cudaMemcpyAsync(ctx->stage_misc.p, bases_jac, n * sizeof(jac_t), cudaMemcpyHostToDevice, ctx->stream));
        k_jac_to_affine<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(ctx->stage_misc.as<jac_t>(),
                                                                             ctx->stage_bases.as<affine_t>(), n);
        ctx->kernel_launches++;
    }
    xyzz_t r;
    msm_device(ctx, ctx->stage_bases.as<affine_t>(), ctx->stage_scalars.as<fr_t>(), n, r);
    out_jac_from_xyzz(r, out_jac);
    HALO_CATCH(ctx)
}


// ---- scalar vectors (group.rs:13-15, :29-37) ----------------------------------------------------------
int halo_scalar_dot(halo_ctx* ctx, const uint64_t* xs, const uint64_t* ys, uint64_t n, uint64_t out[4]) {
    if (!ctx || !out || ((!xs || !ys) && n)) return HALO_EINVAL;
    HALO_TRY(ctx)
    ctx->stage_scalars.reserve((2 * (n ? n : 1) + 1 + VEC_DOT_MAX_BLOCKS) * sizeof(fr_t));
    fr_t* a = ctx->stage_scalars.as<fr_t>();
    fr_t* b = a + n;
    fr_t* res = b + n;
    if (n) {
        HALO_CUDA(cudaMemcpyAsync(a, xs, n * sizeof(fr_t), cudaMemcpyHostToDevice, ctx->stream));
        HALO_CUDA(cudaMemcpyAsync(b, ys, n * sizeof(fr_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    vec_dot(ctx, a, b, n, res + 1, res);
    HALO_CUDA(cudaMemcpyAsync(out, res, 32, cudaMemcpyDeviceToHost, ctx->stream));
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    HALO_CATCH(ctx)
}

int halo_construct_powers(halo_ctx* ctx, const uint64_t z[4], uint64_t n, uint64_t* out) {
    if (!ctx || !z || (!out && n)) return HALO_EINVAL;
    HALO_TRY(ctx)
    if (n) {
        ctx->stage_scalars.reserve(n * sizeof(fr_t));
        fr_t zz;
        memcpy(&zz, z, 32);
        vec_powers(ctx, zz, n, ctx->stage_scalars.as<fr_t>());
        HALO_CUDA(cudaMemcpyAsync(out, ctx->stage_scalars.p, n * sizeof(fr_t), cudaMemcpyDeviceToHost, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    HALO_CATCH(ctx)
}

// ---- K5: h(X) (pcdl.rs:56-77, :338; acc.rs:85-94) --------------------------------------------------------
static int check_lg(halo_ctx* ctx, uint32_t lg_n, bool need_gens) {
    if (lg_n > 30 || ((uint64_t)1 << lg_n) > ctx->max_n) return fail(ctx, HALO_EINVAL, "h: 2^lg_n exceeds max_n");
    if (need_gens && ((uint64_t)1 << lg_n) > ctx->n_gens) return fail(ctx, HALO_ESTATE, "h: 2^lg_n exceeds resident generators");
    return HALO_OK;
}

// d = coeffs(h), the n = 2^lg_n coefficients of one claim
static void h_expand_one(halo_ctx* ctx, const uint64_t* xis, uint32_t lg_n, fr_t* d) {
    fr_t one;
    fp_one(one);
    vec_h_lincomb(ctx, reinterpret_cast<const fr_t*>(xis), &lg_n, &one, 1, (uint64_t)1 << lg_n, false, d);
}

int halo_h_expand(halo_ctx* ctx, const uint64_t* xis, uint32_t lg_n, uint64_t* out) {
    if (!ctx || !xis || !out) return HALO_EINVAL;
    if (int rc = check_lg(ctx, lg_n, false)) return rc;
    HALO_TRY(ctx)
    uint64_t n = (uint64_t)1 << lg_n;
    ctx->stage_scalars.reserve(n * sizeof(fr_t));
    h_expand_one(ctx, xis, lg_n, ctx->stage_scalars.as<fr_t>());
    HALO_CUDA(cudaMemcpyAsync(out, ctx->stage_scalars.p, n * sizeof(fr_t), cudaMemcpyDeviceToHost, ctx->stream));
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    HALO_CATCH(ctx)
}

int halo_h_msm(halo_ctx* ctx, const uint64_t* xis, uint32_t lg_n, uint64_t out_jac[12]) {
    if (!ctx || !xis || !out_jac) return HALO_EINVAL;
    if (int rc = check_lg(ctx, lg_n, true)) return rc;
    HALO_TRY(ctx)
    uint64_t n = (uint64_t)1 << lg_n;
    ctx->stage_scalars.reserve(n * sizeof(fr_t));
    h_expand_one(ctx, xis, lg_n, ctx->stage_scalars.as<fr_t>());
    xyzz_t r;
    msm_gens_device(ctx, ctx->stage_scalars.as<fr_t>(), 0, n, r);
    out_jac_from_xyzz(r, out_jac);
    HALO_CATCH(ctx)
}

// <GS[0..n), stage_scalars> and the companion MSM sum_i scalars[i] * bases[i] (i < m, staged in stage_misc) on the two lanes
// of msm_batch.
static void h_msm_pair(halo_ctx* ctx, uint64_t n, const uint64_t* bases_affine, const uint8_t* inf_flags, const uint64_t* scalars,
                       uint64_t m, xyzz_t out[2]) {
    MsmInput in[2];
    in[0] = gens_msm_input(ctx, gens_use_fixed(ctx, n), ctx->stage_scalars.as<fr_t>(), 0, n);
    // companion: bases | scalars | infinity flags staged in stage_misc
    const size_t mm = m ? m : 1;
    ctx->stage_misc.reserve(mm * (sizeof(affine_t) + sizeof(fr_t) + 1));
    affine_t* d_b = ctx->stage_misc.as<affine_t>();
    fr_t* d_s = reinterpret_cast<fr_t*>(d_b + mm);
    uint8_t* d_i = reinterpret_cast<uint8_t*>(d_s + mm);
    if (m) {
        HALO_CUDA(cudaMemcpyAsync(d_b, bases_affine, m * sizeof(affine_t), cudaMemcpyHostToDevice, ctx->stream));
        HALO_CUDA(cudaMemcpyAsync(d_s, scalars, m * sizeof(fr_t), cudaMemcpyHostToDevice, ctx->stream));
        if (inf_flags) mark_infinity(ctx, ctx->stream, d_b, d_i, inf_flags, m);
    }
    in[1].bases = d_b;
    in[1].scalars = d_s;
    in[1].n = (uint32_t)m;
    ctx->force_two_lanes = m > 0;
    try {
        msm_batch(ctx, in, 2, out);
    } catch (...) {
        ctx->force_two_lanes = false;
        throw;
    }
    ctx->force_two_lanes = false;
}

int halo_h_msm_with(halo_ctx* ctx, const uint64_t* xis, uint32_t lg_n, const uint64_t* bases_affine, const uint8_t* inf_flags,
                    const uint64_t* scalars, uint64_t k, uint64_t out_h_jac[12], uint64_t out_small_jac[12]) {
    if (!ctx || !xis || !out_h_jac || !out_small_jac || ((!bases_affine || !scalars) && k)) return HALO_EINVAL;
    if (int rc = check_lg(ctx, lg_n, true)) return rc;
    if (k > 4096) return fail(ctx, HALO_EINVAL, "halo_h_msm_with: the companion MSM is meant to be small (k <= 4096)");
    HALO_TRY(ctx)
    uint64_t n = (uint64_t)1 << lg_n;
    ctx->stage_scalars.reserve(n * sizeof(fr_t));
    h_expand_one(ctx, xis, lg_n, ctx->stage_scalars.as<fr_t>());
    xyzz_t out[2];
    h_msm_pair(ctx, n, bases_affine, inf_flags, scalars, k, out);
    out_jac_from_xyzz(out[0], out_h_jac);
    out_jac_from_xyzz(out[1], out_small_jac);
    HALO_CATCH(ctx)
}

// The generator half (k_h_lincomb, then the generator MSM on lane 0) is enqueued by submit; collect runs the companion on
// lane 1, so it starts at once even while the generator MSM still runs, and finishes both.
static constexpr size_t HB_SLOT = 3 * MSM_MAX_WINDOWS;

int halo_h_msm_batch_submit(halo_ctx* ctx, const uint64_t* xis, const uint32_t* lg_ns, const uint64_t* weights, uint64_t k,
                            int* ticket) {
    if (!ctx || !ticket || ((!xis || !lg_ns || !weights) && k)) return HALO_EINVAL;
    if (k >> 32) return fail(ctx, HALO_EINVAL, "halo_h_msm_batch_submit: k is 2^32 or more");
    if (ctx->hb.active) return fail(ctx, HALO_ESTATE, "halo_h_msm_batch_submit: a batch is outstanding; collect it first");
    uint64_t n = 0;
    for (uint64_t j = 0; j < k; j++) {
        if (int rc = check_lg(ctx, lg_ns[j], true)) return rc;
        if (((uint64_t)1 << lg_ns[j]) > n) n = (uint64_t)1 << lg_ns[j];
    }
    HALO_TRY(ctx)
    halo_ctx::HBatch& b = ctx->hb;
    if (!b.h_parts) {
        HALO_CUDA(cudaEventCreateWithFlags(&b.done, cudaEventDisableTiming));
        HALO_CUDA(cudaMallocHost(reinterpret_cast<void**>(&b.h_parts), 2 * HB_SLOT * sizeof(xyzz_t)));
    }
    b.parts.reserve(2 * HB_SLOT * sizeof(xyzz_t));
    b.empty = n == 0;
    if (!b.empty) {
        b.scalars.reserve(n * sizeof(fr_t));
        vec_h_lincomb(ctx, reinterpret_cast<const fr_t*>(xis), lg_ns, reinterpret_cast<const fr_t*>(weights), k, n, false,
                      b.scalars.as<fr_t>());
        const bool fixed = gens_use_fixed(ctx, n);
        b.plan = msm_plan(ctx, n, fixed);
        msm_enqueue_to_host(ctx, gens_msm_input(ctx, fixed, b.scalars.as<fr_t>(), 0, n), b.plan, b.parts.as<xyzz_t>(), b.h_parts);
        HALO_CUDA(cudaEventRecord(b.done, ctx->stream));
    }
    b.active = true;
    *ticket = 0;
    HALO_CATCH(ctx)
}

int halo_h_msm_batch_collect(halo_ctx* ctx, int ticket, const uint64_t* bases_affine, const uint8_t* inf_flags,
                             const uint64_t* scalars, uint64_t m, uint64_t out_jac[12]) {
    if (!ctx || !out_jac || ticket != 0 || ((!bases_affine || !scalars) && m)) return HALO_EINVAL;
    if (m >> 32) return fail(ctx, HALO_EINVAL, "halo_h_msm_batch_collect: m is 2^32 or more");
    halo_ctx::HBatch& b = ctx->hb;
    if (!b.active) return fail(ctx, HALO_ESTATE, "halo_h_msm_batch_collect: no batch submitted");
    b.active = false;  // from here on the batch is collected, whatever the outcome
    HALO_TRY(ctx)
    xyzz_t gen, comp;
    xyzz_set_inf(gen);
    xyzz_set_inf(comp);
    if (m) {
        b.companion.reserve(m * (sizeof(affine_t) + sizeof(fr_t) + 1));
        affine_t* d_b = b.companion.as<affine_t>();
        fr_t* d_s = reinterpret_cast<fr_t*>(d_b + m);
        uint8_t* d_i = reinterpret_cast<uint8_t*>(d_s + m);
        HALO_CUDA(cudaMemcpyAsync(d_b, bases_affine, m * sizeof(affine_t), cudaMemcpyHostToDevice, ctx->stream2));
        HALO_CUDA(cudaMemcpyAsync(d_s, scalars, m * sizeof(fr_t), cudaMemcpyHostToDevice, ctx->stream2));
        if (inf_flags) mark_infinity(ctx, ctx->stream2, d_b, d_i, inf_flags, m);
        MsmInput in;
        in.bases = d_b;
        in.scalars = d_s;
        in.n = (uint32_t)m;
        const MsmPlan plan = msm_plan(ctx, m, false);
        msm_enqueue_to_host(ctx, in, plan, b.parts.as<xyzz_t>() + HB_SLOT, b.h_parts + HB_SLOT, 1);
        // the companion is the smaller MSM as a rule: its host finish overlaps the generator MSM
        HALO_CUDA(cudaStreamSynchronize(ctx->stream2));
        msm_finish_host(b.h_parts + HB_SLOT, plan, comp);
    }
    if (!b.empty) {
        HALO_CUDA(cudaEventSynchronize(b.done));
        msm_finish_host(b.h_parts, b.plan, gen);
        if (ctx->profile) msm_read_timings(ctx);  // the generator MSM (lane 0)
    }
    xyzz_add(gen, comp);
    out_jac_from_xyzz(gen, out_jac);
    HALO_CATCH(ctx)
}

int halo_h_msm_batch(halo_ctx* ctx, const uint64_t* xis, const uint32_t* lg_ns, const uint64_t* weights, uint64_t k,
                     const uint64_t* bases_affine, const uint8_t* inf_flags, const uint64_t* scalars, uint64_t m,
                     uint64_t out_jac[12]) {
    // the companion's arguments are checked ahead of the submit: a refused collect would leave the batch outstanding
    if (!ctx || !out_jac || ((!bases_affine || !scalars) && m)) return HALO_EINVAL;
    if (m >> 32) return fail(ctx, HALO_EINVAL, "halo_h_msm_batch: m is 2^32 or more");
    int ticket = 0;
    if (int rc = halo_h_msm_batch_submit(ctx, xis, lg_ns, weights, k, &ticket)) return rc;
    return halo_h_msm_batch_collect(ctx, ticket, bases_affine, inf_flags, scalars, m, out_jac);
}

int halo_msm_multi(halo_ctx* ctx, const halo_msm_desc* descs, uint32_t count, uint64_t* out_jac) {
    if (!ctx || (!descs && count) || (!out_jac && count)) return HALO_EINVAL;
    size_t bytes = 0;
    for (uint32_t k = 0; k < count; k++) {
        const halo_msm_desc& d = descs[k];
        if (d.n && !d.scalars) return HALO_EINVAL;
        if (d.n > 4096) return fail(ctx, HALO_EINVAL, "halo_msm_multi: the MSMs of a batch are meant to be small (n <= 4096)");
        if (!d.bases_affine && d.off + d.n > ctx->n_gens)
            return fail(ctx, HALO_EINVAL, "halo_msm_multi: range exceeds the resident generators");
        bytes += d.n * (sizeof(fr_t) + (d.bases_affine ? sizeof(affine_t) + 16 : 0)) + 64;
    }
    HALO_TRY(ctx)
    // one staging area for the whole batch: per MSM  scalars | bases | infinity flags  (16-byte aligned pieces)
    ctx->stage_misc.reserve(bytes ? bytes : 64);
    char* cur = ctx->stage_misc.as<char>();
    auto take = [&](size_t len) {
        char* p = cur;
        cur += (len + 15) & ~(size_t)15;
        return p;
    };
    std::vector<MsmInput> ins(count);
    for (uint32_t k = 0; k < count; k++) {
        const halo_msm_desc& d = descs[k];
        if (!d.n) continue;
        fr_t* d_s = reinterpret_cast<fr_t*>(take(d.n * sizeof(fr_t)));
        HALO_CUDA(cudaMemcpyAsync(d_s, d.scalars, d.n * sizeof(fr_t), cudaMemcpyHostToDevice, ctx->stream));
        ins[k].scalars = d_s;
        ins[k].n = (uint32_t)d.n;
        if (d.bases_affine) {
            affine_t* d_b = reinterpret_cast<affine_t*>(take(d.n * sizeof(affine_t)));
            HALO_CUDA(cudaMemcpyAsync(d_b, d.bases_affine, d.n * sizeof(affine_t), cudaMemcpyHostToDevice, ctx->stream));
            if (d.inf_flags) mark_infinity(ctx, ctx->stream, d_b, reinterpret_cast<uint8_t*>(take(d.n)), d.inf_flags, d.n);
            ins[k].bases = d_b;
        } else {
            ins[k].bases = ctx->gens.as<affine_t>() + d.off;
        }
    }
    for (uint32_t k0 = 0; k0 < count; k0 += 4) {  // msm_batch: up to 4 MSMs on two lanes, one synchronisation
        const int c = (int)(count - k0 < 4 ? count - k0 : 4);
        xyzz_t out[4];
        msm_batch(ctx, ins.data() + k0, c, out);
        for (int k = 0; k < c; k++) out_jac_from_xyzz(out[k], out_jac + 12 * (k0 + k));
    }
    HALO_CATCH(ctx)
}

// DensePolynomial::degree of the n device coefficients d (index of the highest non-zero one, 0 for the zero polynomial):
// scanned down from the top in chunks (the leading coefficient is non-zero except with negligible probability)
static uint64_t device_degree(halo_ctx* ctx, const fr_t* d, uint64_t n) {
    uint64_t hi = n;
    std::vector<fr_t> chunk(64);
    while (hi > 0) {
        uint64_t lo = hi > 64 ? hi - 64 : 0;
        HALO_CUDA(cudaMemcpyAsync(chunk.data(), d + lo, (hi - lo) * sizeof(fr_t), cudaMemcpyDeviceToHost, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));
        for (uint64_t i = hi; i-- > lo;)
            if (!fp_is_zero(chunk[i - lo])) return i;
        hi = lo;
    }
    return 0;
}

// out != NULL: coefficients to the host.  out == NULL: the polynomial stays on the device (ctx->poly_dev) and
// *degree_out receives its degree (DensePolynomial::degree: index of the highest non-zero coefficient).
static int h_lincomb_impl(halo_ctx* ctx, const uint64_t* h0, uint64_t n_h0, const uint64_t* alphas, const uint64_t* xis,
                          uint64_t m, uint32_t lg_n, uint64_t* out, uint64_t* degree_out) {
    if (!ctx || (!out && !degree_out) || (!h0 && n_h0) || ((!alphas || !xis) && m)) return HALO_EINVAL;
    if (int rc = check_lg(ctx, lg_n, false)) return rc;
    uint64_t n = (uint64_t)1 << lg_n;
    if (n_h0 > n) return fail(ctx, HALO_EINVAL, "halo_h_lincomb: h_0 longer than n");
    HALO_TRY(ctx)
    DevBuf& buf = out ? ctx->stage_scalars : ctx->poly_dev;
    buf.reserve(n * sizeof(fr_t));
    fr_t* d = buf.as<fr_t>();
    HALO_CUDA(cudaMemsetAsync(d, 0, n * sizeof(fr_t), ctx->stream));
    if (n_h0) HALO_CUDA(cudaMemcpyAsync(d, h0, n_h0 * sizeof(fr_t), cudaMemcpyHostToDevice, ctx->stream));
    std::vector<uint32_t> lgs(m, lg_n);
    if (m)  // acc.rs:90-92: h_0 + sum_i alphas[i + 1] coeffs(h_i)
        vec_h_lincomb(ctx, reinterpret_cast<const fr_t*>(xis), lgs.data(), reinterpret_cast<const fr_t*>(alphas) + 1, m, n, true, d);
    if (out) {
        HALO_CUDA(cudaMemcpyAsync(out, d, n * sizeof(fr_t), cudaMemcpyDeviceToHost, ctx->stream));
        HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    } else {
        ctx->poly_n = n;
        *degree_out = device_degree(ctx, d, n);
    }
    HALO_CATCH(ctx)
}

int halo_h_lincomb(halo_ctx* ctx, const uint64_t* h0, uint64_t n_h0, const uint64_t* alphas, const uint64_t* xis, uint64_t m,
                   uint32_t lg_n, uint64_t* out) {
    if (!out) return HALO_EINVAL;
    return h_lincomb_impl(ctx, h0, n_h0, alphas, xis, m, lg_n, out, nullptr);
}

int halo_h_lincomb_resident(halo_ctx* ctx, const uint64_t* h0, uint64_t n_h0, const uint64_t* alphas, const uint64_t* xis,
                            uint64_t m, uint32_t lg_n, uint64_t* degree_out) {
    if (!degree_out) return HALO_EINVAL;
    return h_lincomb_impl(ctx, h0, n_h0, alphas, xis, m, lg_n, nullptr, degree_out);
}

// ---- K3b: k polynomials opened at one point ------------------------------------------------------------------
// Grows a buffer; false when the device has no memory for it (the error is cleared: the context stays usable)
static bool reserve_or_nomem(DevBuf& b, size_t bytes) {
    try {
        b.reserve(bytes);
        return true;
    } catch (const CudaError& e) {
        if (e.err != cudaErrorMemoryAllocation) throw;
        cudaGetLastError();
        return false;
    }
}

// Validates k packed polynomials of at most n coefficients and uploads them into the pooled polys_dev; on success they are the
// context's resident polynomials (polys_k, polys_n = the longest), the quotient of an earlier upload is gone.  The caller's
// scratch, n_max * extra_per_poly + extra_fixed elements of stage_scalars, is reserved before anything is uploaded.
static int poly_upload(halo_ctx* ctx, const char* fn, const uint64_t* coeffs, const uint64_t* n_coeffs, uint64_t k, uint64_t n,
                       uint64_t extra_per_poly, uint64_t extra_fixed) {
    std::string e(fn);
    if (!ctx || !n_coeffs) return HALO_EINVAL;
    if (k == 0 || (k >> 31)) return fail(ctx, HALO_EINVAL, (e + ": k must be 1 .. 2^31 - 1").c_str());
    if (n > ctx->n_gens) return fail(ctx, HALO_EINVAL, (e + ": n exceeds the resident generators").c_str());
    std::vector<uint64_t> off(k + 1, 0);
    uint64_t n_max = 0;
    for (uint64_t j = 0; j < k; j++) {
        if (n_coeffs[j] > n) return fail(ctx, HALO_EINVAL, (e + ": a polynomial has more than n coefficients").c_str());
        off[j + 1] = off[j] + n_coeffs[j];  // k < 2^31 polynomials of at most n < 2^32 coefficients: no wrap
        n_max = std::max(n_max, n_coeffs[j]);
    }
    const uint64_t total = off[k];
    if (!coeffs && total) return HALO_EINVAL;
    if (total > (UINT64_MAX >> 6)) return fail(ctx, HALO_ENOMEM, (e + ": out of device memory").c_str());
    ctx->polys_k = 0;  // the previous upload is gone from here on, whatever the outcome
    ctx->quot_ready = false;
    HALO_TRY(ctx)
    if (!reserve_or_nomem(ctx->polys_dev, (total ? total : 1) * sizeof(fr_t)) ||
        !reserve_or_nomem(ctx->polys_off, (k + 1) * sizeof(uint64_t)) ||
        !reserve_or_nomem(ctx->stage_scalars, (n_max * extra_per_poly + extra_fixed) * sizeof(fr_t) + 1))
        return fail(ctx, HALO_ENOMEM, (e + ": out of device memory").c_str());
    HALO_CUDA(cudaMemcpyAsync(ctx->polys_off.p, off.data(), (k + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    h2d_copy(ctx, ctx->polys_dev.p, coeffs, total * sizeof(fr_t), ctx->stream);
    ctx->polys_k = k;
    ctx->polys_n = n_max;
    ctx->polys_starts = std::move(off);
    HALO_CATCH(ctx)
}

int halo_poly_upload(halo_ctx* ctx, const uint64_t* coeffs, const uint64_t* n_coeffs, uint64_t k, uint64_t n) {
    return poly_upload(ctx, "halo_poly_upload", coeffs, n_coeffs, k, n, 0, 0);
}

int halo_poly_eval_many(halo_ctx* ctx, const uint64_t* coeffs, const uint64_t* n_coeffs, uint64_t k, uint64_t n, const uint64_t z[4],
                        uint64_t* vs_out) {
    if (!ctx || !n_coeffs || !z || !vs_out) return HALO_EINVAL;
    if (k == 0 || (k >> 31)) return fail(ctx, HALO_EINVAL, "halo_poly_eval_many: k must be 1 .. 2^31 - 1");
    uint64_t n_max = 0;
    for (uint64_t j = 0; j < k; j++) n_max = std::max(n_max, std::min(n_coeffs[j], n));
    const uint32_t bps = vec_eval_many_blocks(k, n_max);
    const int rc = poly_upload(ctx, "halo_poly_eval_many", coeffs, n_coeffs, k, n, 1, (uint64_t)bps * k + k);
    if (rc) return rc;
    HALO_TRY(ctx)
    fr_t zz;
    memcpy(&zz, z, 32);
    fr_t* pows = ctx->stage_scalars.as<fr_t>();
    fr_t* partials = pows + n_max;
    fr_t* vs = partials + (uint64_t)bps * k;
    vec_powers(ctx, zz, n_max, pows);
    vec_eval_many(ctx, ctx->polys_dev.as<fr_t>(), ctx->polys_off.as<uint64_t>(), k, n_max, pows, partials, vs);
    HALO_CUDA(cudaMemcpyAsync(vs_out, vs, k * sizeof(fr_t), cudaMemcpyDeviceToHost, ctx->stream));
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    HALO_CATCH(ctx)
}

int halo_poly_combine_resident(halo_ctx* ctx, const uint64_t alpha[4], uint64_t* degree_out) {
    if (!ctx || !alpha || !degree_out) return HALO_EINVAL;
    if (!ctx->polys_k) return fail(ctx, HALO_ESTATE, "halo_poly_combine_resident: no polynomials (call halo_poly_eval_many first)");
    HALO_TRY(ctx)
    const uint64_t n = ctx->polys_n ? ctx->polys_n : 1;  // k empty polynomials combine to one zero coefficient
    ctx->poly_n = 0;
    if (!reserve_or_nomem(ctx->poly_dev, n * sizeof(fr_t))) return fail(ctx, HALO_ENOMEM, "halo_poly_combine_resident: out of device memory");
    fr_t a;
    memcpy(&a, alpha, 32);
    vec_poly_combine(ctx, ctx->polys_dev.as<fr_t>(), ctx->polys_off.as<uint64_t>(), ctx->polys_k, a, n, ctx->poly_dev.as<fr_t>());
    ctx->poly_n = n;
    *degree_out = device_degree(ctx, ctx->poly_dev.as<fr_t>(), n);
    HALO_CATCH(ctx)
}

// ---- K3c: k polynomials opened at several points ---------------------------------------------------------------
// Descriptors and scratch of one run of the K3c kernels, carved out of ctx->quot_scratch.  Points t < T each get a power
// table; group g sums its terms (j, w) over the resident polynomials.
struct QuotRun {
    std::vector<QuotGroup> groups;
    std::vector<QuotTerm> terms;
    std::vector<fr_t> zthr;
    QuotGroup* d_groups = nullptr;
    QuotTerm* d_terms = nullptr;
    fr_t *d_zthr = nullptr, *d_kloc = nullptr, *d_agg = nullptr, *d_kblk = nullptr, *d_rem = nullptr;
};

// One table per point; the points are checked by the caller
static void quot_points(QuotRun& r, const uint64_t* zs, uint64_t T) {
    r.zthr.resize(T * VEC_QUOT_ZTHR);
    for (uint64_t t = 0; t < T; t++) {
        fr_t z, zb;
        memcpy(&z, zs + 4 * t, 32);
        vec_quot_tables(z, zb, &r.zthr[t * VEC_QUOT_ZTHR]);
    }
}

static QuotGroup quot_group(const uint64_t* zs, uint64_t t, const fr_t& s, uint32_t first, uint32_t count, const std::vector<fr_t>& zthr) {
    QuotGroup g{};
    memcpy(&g.z, zs + 4 * t, 32);
    g.s = s;
    fp_mul(g.zblk, zthr[t * VEC_QUOT_ZTHR + VEC_QUOT_ZTHR - 1], zthr[t * VEC_QUOT_ZTHR + 1]);
    g.first = first;
    g.count = count;
    g.tab = (uint32_t)t;
    return g;
}

static QuotTerm quot_term(const std::vector<uint64_t>& off, uint64_t j, const fr_t* w) {  // w = NULL: weight one
    QuotTerm e{};
    e.off = off[j];
    e.len = off[j + 1] - off[j];
    if (w) {
        e.w = *w;
    } else {
        fp_one(e.w);
        e.unit = 1;
    }
    return e;
}

// Reserves the scratch (false: no device memory) and uploads the descriptors
static bool quot_stage(halo_ctx* ctx, QuotRun& r, uint64_t nblk, bool carries) {
    const uint64_t G = r.groups.size();
    auto al = [](uint64_t b) { return (b + 255) & ~(uint64_t)255; };
    const uint64_t b_groups = al(G * sizeof(QuotGroup)), b_terms = al(r.terms.size() * sizeof(QuotTerm)),
                   b_zthr = al(r.zthr.size() * sizeof(fr_t)), b_kloc = carries ? al(G * nblk * VEC_QUOT_ZTHR * sizeof(fr_t)) : 0,
                   b_agg = al(G * nblk * sizeof(fr_t)), b_kblk = carries ? b_agg : 0, b_rem = al(G * sizeof(fr_t));
    if (!reserve_or_nomem(ctx->quot_scratch, b_groups + b_terms + b_zthr + b_kloc + b_agg + b_kblk + b_rem)) return false;
    char* p = static_cast<char*>(ctx->quot_scratch.p);
    r.d_groups = reinterpret_cast<QuotGroup*>(p);
    r.d_terms = reinterpret_cast<QuotTerm*>(p += b_groups);
    r.d_zthr = reinterpret_cast<fr_t*>(p += b_terms);
    r.d_kloc = carries ? reinterpret_cast<fr_t*>(p + b_zthr) : nullptr;
    r.d_agg = reinterpret_cast<fr_t*>(p += b_zthr + b_kloc);
    r.d_kblk = carries ? reinterpret_cast<fr_t*>(p + b_agg) : nullptr;
    r.d_rem = reinterpret_cast<fr_t*>(p += b_agg + b_kblk);
    HALO_CUDA(cudaMemcpyAsync(r.d_groups, r.groups.data(), G * sizeof(QuotGroup), cudaMemcpyHostToDevice, ctx->stream));
    HALO_CUDA(cudaMemcpyAsync(r.d_terms, r.terms.data(), r.terms.size() * sizeof(QuotTerm), cudaMemcpyHostToDevice, ctx->stream));
    HALO_CUDA(cudaMemcpyAsync(r.d_zthr, r.zthr.data(), r.zthr.size() * sizeof(fr_t), cudaMemcpyHostToDevice, ctx->stream));
    return true;
}

static int check_queries(halo_ctx* ctx, const char* fn, const uint64_t* zs, uint64_t T, const uint64_t* q_poly, const uint64_t* q_point,
                         uint64_t m) {
    std::string e(fn);
    if (!zs || !q_poly || !q_point) return fail(ctx, HALO_EINVAL, (e + ": NULL pointer").c_str());
    if (T == 0 || T > HALO_MULTI_MAX_POINTS) return fail(ctx, HALO_EINVAL, (e + ": T must be 1 .. HALO_MULTI_MAX_POINTS").c_str());
    if (m == 0 || (m >> 31)) return fail(ctx, HALO_EINVAL, (e + ": m must be 1 .. 2^31 - 1").c_str());
    if (!ctx->polys_k) return fail(ctx, HALO_ESTATE, (e + ": no resident polynomials (call halo_poly_upload first)").c_str());
    for (uint64_t i = 0; i < m; i++)
        if (q_poly[i] >= ctx->polys_k || q_point[i] >= T) return fail(ctx, HALO_EINVAL, (e + ": a query index is out of range").c_str());
    return HALO_OK;
}

int halo_poly_eval_queries(halo_ctx* ctx, const uint64_t* zs, uint64_t T, const uint64_t* q_poly, const uint64_t* q_point, uint64_t m,
                           uint64_t* vs_out) {
    if (!ctx || !vs_out) return HALO_EINVAL;
    if (int rc = check_queries(ctx, "halo_poly_eval_queries", zs, T, q_poly, q_point, m)) return rc;
    HALO_TRY(ctx)
    const std::vector<uint64_t>& off = ctx->polys_starts;
    QuotRun r;
    quot_points(r, zs, T);
    fr_t one;
    fp_one(one);
    for (uint64_t i = 0; i < m; i++) {
        r.groups.push_back(quot_group(zs, q_point[i], one, (uint32_t)i, 1, r.zthr));
        r.terms.push_back(quot_term(off, q_poly[i], nullptr));
    }
    const uint64_t n = ctx->polys_n, nblk = vec_quot_blocks(n);
    if (!quot_stage(ctx, r, nblk, false)) return fail(ctx, HALO_ENOMEM, "halo_poly_eval_queries: out of device memory");
    vec_quot_eval(ctx, ctx->polys_dev.as<fr_t>(), r.d_groups, (uint32_t)m, r.d_terms, r.d_zthr, n, r.d_agg, r.d_rem);
    HALO_CUDA(cudaMemcpyAsync(vs_out, r.d_rem, m * sizeof(fr_t), cudaMemcpyDeviceToHost, ctx->stream));
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    HALO_CATCH(ctx)
}

int halo_poly_quotient(halo_ctx* ctx, const uint64_t* zs, const uint64_t* scales, uint64_t T, const uint64_t* q_poly,
                       const uint64_t* q_point, const uint64_t* weights, uint64_t m, uint64_t* rems_out, uint64_t Q_out[12]) {
    if (!ctx || !scales || !weights || !rems_out || !Q_out) return HALO_EINVAL;
    if (int rc = check_queries(ctx, "halo_poly_quotient", zs, T, q_poly, q_point, m)) return rc;
    ctx->quot_ready = false;
    HALO_TRY(ctx)
    const std::vector<uint64_t>& off = ctx->polys_starts;
    QuotRun r;
    quot_points(r, zs, T);
    for (uint64_t t = 0; t < T; t++) {  // point t's terms in query order
        const uint32_t first = (uint32_t)r.terms.size();
        for (uint64_t i = 0; i < m; i++)
            if (q_point[i] == t) r.terms.push_back(quot_term(off, q_poly[i], reinterpret_cast<const fr_t*>(weights + 4 * i)));
        fr_t s;
        memcpy(&s, scales + 4 * t, 32);
        r.groups.push_back(quot_group(zs, t, s, first, (uint32_t)r.terms.size() - first, r.zthr));
    }
    const uint64_t n = ctx->polys_n, nblk = vec_quot_blocks(n), n_q = n ? n - 1 : 0;
    if (!quot_stage(ctx, r, nblk, true) || !reserve_or_nomem(ctx->quot_dev, (n_q ? n_q : 1) * sizeof(fr_t)))
        return fail(ctx, HALO_ENOMEM, "halo_poly_quotient: out of device memory");
    vec_quotient(ctx, ctx->polys_dev.as<fr_t>(), r.d_groups, (uint32_t)T, r.d_terms, r.d_zthr, n, r.d_kloc, r.d_agg, r.d_kblk, r.d_rem,
                 ctx->quot_dev.as<fr_t>());
    std::vector<fr_t> rems(T);
    HALO_CUDA(cudaMemcpyAsync(rems.data(), r.d_rem, T * sizeof(fr_t), cudaMemcpyDeviceToHost, ctx->stream));
    xyzz_t Q;
    msm_gens_device(ctx, ctx->quot_dev.as<fr_t>(), 0, n_q, Q);  // synchronises the stream
    memcpy(rems_out, rems.data(), T * sizeof(fr_t));
    out_jac_from_xyzz(Q, Q_out);
    ctx->quot_n = n_q;
    ctx->quot_ready = true;
    HALO_CATCH(ctx)
}

int halo_poly_lincomb_resident(halo_ctx* ctx, const uint64_t* cs, const uint64_t c_q[4], uint64_t* degree_out) {
    if (!ctx || !cs || !c_q || !degree_out) return HALO_EINVAL;
    if (!ctx->polys_k || !ctx->quot_ready)
        return fail(ctx, HALO_ESTATE, "halo_poly_lincomb_resident: no quotient of the resident polynomials (call halo_poly_quotient first)");
    HALO_TRY(ctx)
    const uint64_t n = ctx->polys_n ? ctx->polys_n : 1;
    ctx->poly_n = 0;
    if (!reserve_or_nomem(ctx->poly_dev, n * sizeof(fr_t)) || !reserve_or_nomem(ctx->stage_scalars, ctx->polys_k * sizeof(fr_t)))
        return fail(ctx, HALO_ENOMEM, "halo_poly_lincomb_resident: out of device memory");
    HALO_CUDA(cudaMemcpyAsync(ctx->stage_scalars.p, cs, ctx->polys_k * sizeof(fr_t), cudaMemcpyHostToDevice, ctx->stream));
    fr_t cq;
    memcpy(&cq, c_q, 32);
    vec_poly_lincomb(ctx, ctx->polys_dev.as<fr_t>(), ctx->polys_off.as<uint64_t>(), ctx->stage_scalars.as<fr_t>(), ctx->polys_k,
                     ctx->quot_dev.as<fr_t>(), ctx->quot_n, cq, n, ctx->poly_dev.as<fr_t>());
    ctx->poly_n = n;
    *degree_out = device_degree(ctx, ctx->poly_dev.as<fr_t>(), n);
    HALO_CATCH(ctx)
}

}  // extern "C"
