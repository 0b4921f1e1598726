// comm.cu -- the MSM sharded over the GPUs of one node, behind the C ABI (include/halo_b200.h, "multi-GPU").
//
// Replaces group.rs:24-26 (`point_dot_affine` -> VariableBaseMSM::msm_unchecked) at scale.  Only the MSM shards (SURVEY
// 8e): rank r of g owns the contiguous point slice [r n / g, (r + 1) n / g) of the resident generators and the matching
// slice of the scalars, runs the single-GPU Pippenger of msm.cu on it, and the per-rank partial results meet in ONE
// ncclAllGather over NVLink / NVSwitch, enqueued on the library's own stream right behind the bucket reduction.  What is
// gathered are not finished points but each rank's reduction partials (E, A2, R2 per window, XYZZ, msm.cu): every rank
// uses the same plan, the recombination S = E + slab (A2 - R2) and the Horner over the windows are linear, so the ranks'
// partials are added component by component, in rank order, and the host finish (<= 255 doublings) runs ONCE, not once
// per rank.  Folds, h-expansion and the transcript stay on one GPU (sequential rounds, pcdl.rs:212).
//
// NCCL is not a link-time dependency: libnccl.so.2 is dlopen'ed the first time a communicator is made (a process that
// already holds a copy, e.g. through torch, shares it), so single-GPU users of libhalo_b200.so need no NCCL at all.
// Two forms:
//   rank form    halo_comm_unique_id / halo_comm_init_rank   one process (or thread) per GPU: torchrun, MPI, a thread pool
//   node form    halo_mgpu_create ..                          one caller thread, the library owns one worker thread, context
//                                                             and communicator per device (ncclCommInitAll)
#include <dlfcn.h>

#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/halo_b200.h"
#include "common.cuh"
#include "msm.cuh"

using namespace halo;

// ---- the handful of NCCL entry points we use, resolved at run time (declarations restated from nccl.h 2.27) ----------
namespace {
struct ncclComm;
typedef ncclComm* ncclComm_t;
struct ncclUniqueId {
    char internal[128];
};
typedef int ncclResult_t;  // ncclSuccess = 0
constexpr int NCCL_UINT8 = 1;  // ncclDataType_t: ncclInt8 = 0, ncclUint8 = 1

struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetVersion)(int*) = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string error;
};

NcclApi* nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {getenv("HALO_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char* nm : names) {
            if (!nm || !*nm) continue;
            api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);  // a copy already in the process (torch's) is reused by soname
            if (api.handle) break;
        }
        if (!api.handle) {
            api.error = std::string("cannot load libnccl.so.2: ") + (dlerror() ? dlerror() : "not found");
            return;
        }
        auto sym = [&](const char* s) {
            void* p = dlsym(api.handle, s);
            if (!p && api.error.empty()) api.error = std::string("libnccl lacks ") + s;
            return p;
        };
        api.GetVersion = reinterpret_cast<decltype(api.GetVersion)>(sym("ncclGetVersion"));
        api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
        api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
        api.CommInitAll = reinterpret_cast<decltype(api.CommInitAll)>(sym("ncclCommInitAll"));
        api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
        api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
        api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
    });
    return api.error.empty() ? &api : nullptr;
}
const char* nccl_load_error() { return "libnccl.so.2 could not be loaded or lacks a symbol (set HALO_NCCL_LIB to its path)"; }

struct NcclError {
    ncclResult_t rc;
    const char* what;
};
#define HALO_NCCL(api, expr)                                 \
    do {                                                     \
        ncclResult_t _r = (api)->expr;                       \
        if (_r != 0) throw NcclError{_r, #expr};             \
    } while (0)

// Every rank must run the SAME plan for the component-wise sum to be valid; the plan signature travels with the partials.
struct alignas(16) PartHeader {
    uint32_t magic, c, W, fixed, red_slabs, red_T, red_log_s, n_sets;  // n_sets: point slices (partial sets) in the block
    uint32_t pad[24];
};
static_assert(sizeof(PartHeader) == sizeof(xyzz_t), "header occupies one XYZZ slot");
constexpr uint32_t PART_MAGIC = 0x48414c4fu;  // "HALO"
constexpr int PART_SLOTS = 1 + 3 * MSM_MAX_WINDOWS;  // header + (E, A2, R2) per window
}  // namespace

struct halo_comm {
    halo_ctx* ctx = nullptr;
    ncclComm_t comm = nullptr;
    int rank = 0, size = 1;
    uint64_t n_total = 0;  // generators of the whole set (0: slices were installed by the caller)
    DevBuf send, recv;     // [PART_SLOTS] and [size][PART_SLOTS] XYZZ slots (only the used prefix is gathered)
    xyzz_t* h_recv = nullptr;    // pinned, [size][PART_SLOTS]
    PartHeader* h_hdr = nullptr;  // pinned
    // halo_comm_allgather_sum runs here, not on the context's stream: in the pipelined pattern (submit k + 1, collect k,
    // combine k) the context's stream already holds the kernels of MSM k + 1, and a collective queued behind them would make
    // every step wait for the next one
    cudaStream_t side = nullptr;
    DevBuf side_send, side_recv;
    uint64_t* h_side = nullptr;  // pinned, [size][12]
    cudaEvent_t copied[3] = {};  // host-to-device copies of the point slices of a host-scalar call
};

namespace {
int comm_fail(halo_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->last_error = msg;
    return code;
}

#define COMM_TRY(ctx) \
    try {             \
        HALO_CUDA(cudaSetDevice((ctx)->device));
#define COMM_CATCH(ctx)                                                                                              \
    }                                                                                                                \
    catch (const halo::CudaError& e) {                                                                               \
        return comm_fail(ctx, HALO_ECUDA, std::string("CUDA error: ") + cudaGetErrorString(e.err) + " (" + e.what + ")"); \
    }                                                                                                                \
    catch (const NcclError& e) {                                                                                     \
        NcclApi* a_ = nccl_api();                                                                                    \
        return comm_fail(ctx, HALO_ENCCL, std::string("NCCL error: ") + (a_ ? a_->GetErrorString(e.rc) : "?") + " (" + e.what + ")"); \
    }                                                                                                                \
    catch (const std::bad_alloc&) {                                                                                  \
        return comm_fail(ctx, HALO_ENOMEM, "out of host memory");                                                    \
    }                                                                                                                \
    catch (...) { /* nothing unwinds across the C ABI */                                                             \
        return comm_fail(ctx, HALO_ECUDA, "unexpected internal exception");                                          \
    }                                                                                                                \
    return HALO_OK;

void comm_alloc(halo_comm* c) {
    c->send.reserve((size_t)PART_SLOTS * sizeof(xyzz_t));
    c->recv.reserve((size_t)c->size * PART_SLOTS * sizeof(xyzz_t));
    HALO_CUDA(cudaMallocHost(reinterpret_cast<void**>(&c->h_recv), (size_t)c->size * PART_SLOTS * sizeof(xyzz_t)));
    HALO_CUDA(cudaMallocHost(reinterpret_cast<void**>(&c->h_hdr), sizeof(PartHeader)));
    int prio_lo = 0, prio_hi = 0;
    HALO_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    HALO_CUDA(cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, prio_hi));  // its one-CTA kernels go ahead of queued MSM CTAs
    c->side_send.reserve(96);
    c->side_recv.reserve((size_t)96 * c->size);
    HALO_CUDA(cudaMallocHost(reinterpret_cast<void**>(&c->h_side), (size_t)96 * c->size));
}

// The plan every rank uses for an MSM over `n_global` points: FIXED-base when every rank holds tables built with the
// same window (halo_comm_precompute_generators) and the per-rank slice is large enough, else the variable-base plan of the
// LARGEST slice -- a function of (n_global, size) only, hence identical on all ranks whatever their own slice length.
MsmPlan comm_plan(const halo_comm* c, uint64_t n_global) {
    const uint64_t slice = (n_global + c->size - 1) / c->size;
    return msm_plan(c->ctx, slice ? slice : 1, gens_use_fixed(c->ctx, slice));
}

// local MSM -> partials behind a header in `send` -> all-gather -> host: check headers, add the ranks' partials
// component-wise in rank order, finish once.  The local part may come as up to three point slices (`nsl`), each with its own
// device scalars and an optional event that its host-to-device copy has landed: both run the same plan, so their partials
// simply join the sum -- this is how the host-scalar call overlaps the copies of the later slices with the kernels of the earlier ones.
struct LocalSlice {
    const fr_t* d_scalars;
    uint64_t off, n;
    cudaEvent_t ready;      // may be null
    const uint64_t* h_src;  // host scalars still to be copied to d_scalars on the copy stream (then `ready` is recorded), or null
};
void sharded_msm(halo_comm* c, const LocalSlice* sl, int nsl, uint64_t n_global, xyzz_t& out) {
    halo_ctx* ctx = c->ctx;
    NcclApi* api = nccl_api();
    const MsmPlan plan = comm_plan(c, n_global);
    const size_t parts = msm_parts(plan);
    const size_t used = 1 + parts * nsl;
    if (used > PART_SLOTS) throw NcclError{5, "too many windows for a sliced sharded MSM"};
    xyzz_t* d_send = c->send.as<xyzz_t>();
    cudaStream_t st = ctx->stream;
    PartHeader& h = *c->h_hdr;
    memset(&h, 0, sizeof h);
    h.magic = PART_MAGIC;
    h.c = (uint32_t)plan.c, h.W = (uint32_t)plan.W, h.fixed = plan.fixed, h.red_slabs = plan.red_slabs;
    h.red_T = (uint32_t)plan.red_T, h.red_log_s = (uint32_t)plan.red_log_s, h.n_sets = (uint32_t)nsl;
    HALO_CUDA(cudaMemcpyAsync(d_send, &h, sizeof h, cudaMemcpyHostToDevice, st));
    for (int k = 0; k < nsl; k++) {
        xyzz_t* d_parts = d_send + 1 + parts * k;
        if (sl[k].h_src) {
            // the copy is issued here, slice by slice: staging a PAGEABLE slice blocks this thread, and the kernels of the
            // slices already enqueued run meanwhile
            h2d_copy(ctx, const_cast<fr_t*>(sl[k].d_scalars), sl[k].h_src, sl[k].n * sizeof(fr_t), ctx->copy_stream);
            HALO_CUDA(cudaEventRecord(sl[k].ready, ctx->copy_stream));
        }
        if (sl[k].ready) HALO_CUDA(cudaStreamWaitEvent(st, sl[k].ready, 0));
        if (sl[k].n)
            msm_enqueue(ctx, gens_msm_input(ctx, plan.fixed, sl[k].d_scalars, sl[k].off, sl[k].n), plan, d_parts);
        else
            HALO_CUDA(cudaMemsetAsync(d_parts, 0, parts * sizeof(xyzz_t), st));  // zz = 0: infinity
    }
    const size_t bytes = used * sizeof(xyzz_t);
    HALO_NCCL(api, AllGather(d_send, c->recv.p, bytes, NCCL_UINT8, c->comm, st));
    HALO_CUDA(cudaMemcpyAsync(c->h_recv, c->recv.p, bytes * c->size, cudaMemcpyDeviceToHost, st));
    HALO_CUDA(cudaStreamSynchronize(st));
    // rank r's block starts at h_recv + r * used
    std::vector<xyzz_t> sum(parts);
    for (auto& p : sum) xyzz_set_inf(p);
    for (int r = 0; r < c->size; r++) {
        const xyzz_t* blk = c->h_recv + r * used;
        PartHeader hr;
        memcpy(&hr, blk, sizeof hr);
        if (hr.magic != PART_MAGIC || hr.c != h.c || hr.W != h.W || hr.fixed != h.fixed || hr.red_slabs != h.red_slabs ||
            hr.red_T != h.red_T || hr.red_log_s != h.red_log_s || hr.n_sets != h.n_sets)
            throw NcclError{5 /* ncclInvalidUsage */, "ranks disagree on the MSM plan (different n_global, tables, window or call on some rank)"};
        for (int k = 0; k < nsl; k++)
            for (size_t j = 0; j < parts; j++) xyzz_add(sum[j], blk[1 + parts * k + j]);
    }
    msm_finish_host(sum.data(), plan, out);
}
void sharded_msm(halo_comm* c, const fr_t* d_scalars, uint64_t off_local, uint64_t n_local, uint64_t n_global, xyzz_t& out) {
    LocalSlice one{d_scalars, off_local, n_local, nullptr, nullptr};
    sharded_msm(c, &one, 1, n_global, out);
}
}  // namespace

extern "C" {

void halo_comm_slice(uint64_t n_total, int rank, int size, uint64_t* first, uint64_t* count) {
    const uint64_t base = n_total / (uint64_t)size, rem = n_total % (uint64_t)size;
    const uint64_t r = (uint64_t)rank;
    if (first) *first = r * base + (r < rem ? r : rem);
    if (count) *count = base + (r < rem ? 1 : 0);
}

int halo_comm_unique_id(uint8_t id[HALO_COMM_ID_BYTES]) {
    if (!id) return HALO_EINVAL;
    NcclApi* api = nccl_api();
    if (!api) return HALO_ENCCL;
    ncclUniqueId u;
    if (api->GetUniqueId(&u) != 0) return HALO_ENCCL;
    memcpy(id, u.internal, HALO_COMM_ID_BYTES);
    return HALO_OK;
}

int halo_comm_init_rank(halo_ctx* ctx, const uint8_t id[HALO_COMM_ID_BYTES], int nranks, int rank, halo_comm** out) {
    if (!ctx || !id || !out || nranks < 1 || rank < 0 || rank >= nranks) return HALO_EINVAL;
    *out = nullptr;
    NcclApi* api = nccl_api();
    if (!api) return comm_fail(ctx, HALO_ENCCL, nccl_load_error());
    halo_comm* c = new halo_comm();
    c->ctx = ctx;
    c->rank = rank;
    c->size = nranks;
    try {
        HALO_CUDA(cudaSetDevice(ctx->device));
        ncclUniqueId u;
        memcpy(u.internal, id, HALO_COMM_ID_BYTES);
        HALO_NCCL(api, CommInitRank(&c->comm, nranks, u, rank));
        comm_alloc(c);
    } catch (const halo::CudaError& e) {
        halo_comm_destroy(c);
        return comm_fail(ctx, HALO_ECUDA, std::string("CUDA error: ") + cudaGetErrorString(e.err) + " (" + e.what + ")");
    } catch (const NcclError& e) {
        halo_comm_destroy(c);
        return comm_fail(ctx, HALO_ENCCL, std::string("NCCL error: ") + api->GetErrorString(e.rc) + " (" + e.what + ")");
    } catch (...) {
        halo_comm_destroy(c);
        return comm_fail(ctx, HALO_ECUDA, "unexpected internal exception");
    }
    *out = c;
    return HALO_OK;
}

void halo_comm_destroy(halo_comm* c) {
    if (!c) return;
    if (c->ctx) cudaSetDevice(c->ctx->device);
    if (c->ctx && c->ctx->stream) cudaStreamSynchronize(c->ctx->stream);
    NcclApi* api = nccl_api();
    if (c->comm && api) api->CommDestroy(c->comm);
    if (c->side) {
        cudaStreamSynchronize(c->side);
        cudaStreamDestroy(c->side);
    }
    c->send.release();
    c->recv.release();
    c->side_send.release();
    c->side_recv.release();
    if (c->h_recv) cudaFreeHost(c->h_recv);
    if (c->h_hdr) cudaFreeHost(c->h_hdr);
    if (c->h_side) cudaFreeHost(c->h_side);
    for (cudaEvent_t e : c->copied)
        if (e) cudaEventDestroy(e);
    delete c;
}

int halo_comm_rank(const halo_comm* c) { return c ? c->rank : -1; }
int halo_comm_size(const halo_comm* c) { return c ? c->size : 0; }
int halo_nccl_version(void) {
    NcclApi* api = nccl_api();
    int v = 0;
    return (api && api->GetVersion(&v) == 0) ? v : 0;
}

int halo_comm_derive_generators(halo_comm* c, uint64_t n_total) {
    if (!c || n_total == 0) return HALO_EINVAL;
    uint64_t first, count;
    halo_comm_slice(n_total, c->rank, c->size, &first, &count);
    if (count == 0) return comm_fail(c->ctx, HALO_EINVAL, "halo_comm_derive_generators: fewer generators than ranks");
    int rc = halo_derive_generators_range(c->ctx, first, count);
    if (rc == HALO_OK) c->n_total = n_total;
    return rc;
}

int halo_comm_precompute_generators(halo_comm* c, int window) {
    if (!c) return HALO_EINVAL;
    halo_ctx* ctx = c->ctx;
    if (ctx->n_gens == 0) return comm_fail(ctx, HALO_ESTATE, "halo_comm_precompute_generators: no generators resident");
    if (window == 0) {  // the automatic choice is a function of the largest slice, so that every rank builds the same tables
        const uint64_t total = c->n_total ? c->n_total : ctx->n_gens * (uint64_t)c->size;
        window = msm_make_fixed_plan((total + c->size - 1) / c->size, 0).c;
    }
    return halo_precompute_generators(ctx, window);
}

int halo_msm_gens_sharded_resident(halo_comm* c, const void* d_local_scalars, uint64_t off_local, uint64_t n_local, uint64_t n_global,
                                   uint64_t out_jac[12]) {
    if (!c || !out_jac || (!d_local_scalars && n_local)) return HALO_EINVAL;
    halo_ctx* ctx = c->ctx;
    if (off_local + n_local > ctx->n_gens) return comm_fail(ctx, HALO_ESTATE, "halo_msm_gens_sharded: slice exceeds this rank's resident generators");
    if (n_global < n_local) return comm_fail(ctx, HALO_EINVAL, "halo_msm_gens_sharded: n_global < n_local");
    COMM_TRY(ctx)
    xyzz_t r;
    sharded_msm(c, reinterpret_cast<const fr_t*>(d_local_scalars), off_local, n_local, n_global, r);
    jac_t j;
    xyzz_to_jac(j, r);
    memcpy(out_jac, &j, 96);
    COMM_CATCH(ctx)
}

int halo_msm_gens_sharded(halo_comm* c, const uint64_t* local_scalars, uint64_t off_local, uint64_t n_local, uint64_t n_global,
                          uint64_t out_jac[12]) {
    if (!c || !out_jac || (!local_scalars && n_local)) return HALO_EINVAL;
    halo_ctx* ctx = c->ctx;
    if (off_local + n_local > ctx->n_gens) return comm_fail(ctx, HALO_ESTATE, "halo_msm_gens_sharded: slice exceeds this rank's resident generators");
    if (n_global < n_local) return comm_fail(ctx, HALO_EINVAL, "halo_msm_gens_sharded: n_global < n_local");
    COMM_TRY(ctx)
    ctx->stage_scalars.reserve((n_local ? n_local : 1) * sizeof(fr_t));
    xyzz_t r;
    // Large calls go as two or three point slices (the cuts of the single-GPU blocking call, in sixteenths of n_global / size):
    // the copies of the later slices run on the copy stream beside the kernels of the earlier ones.  The cuts are a function of
    // n_global and the communicator size only, so every rank makes the same number of slices whatever its own n_local.
    const uint64_t slice = (n_global + c->size - 1) / c->size;
    const size_t parts = msm_parts(comm_plan(c, n_global));
    const int a16 = ctx->tune_split_first_16ths, b16 = ctx->tune_split_second_16ths;
    const int nsl = (b16 > 0 && a16 + b16 < 16 && 1 + 3 * parts <= PART_SLOTS) ? 3 : 2;
    if (ctx->tune_split_blocking > 0 && slice >= ((uint64_t)1 << ctx->tune_split_blocking) && 1 + nsl * parts <= PART_SLOTS &&
        !ctx->slots[0].active && !ctx->slots[1].active) {
        async_init(ctx);
        uint64_t cut[4] = {0, slice / 16 * (uint64_t)a16, nsl == 3 ? slice / 16 * (uint64_t)(a16 + b16) : n_local, n_local};
        for (int k = 1; k < 3; k++)
            if (cut[k] > n_local) cut[k] = n_local;
        if (nsl == 2) cut[2] = n_local;
        fr_t* d = ctx->stage_scalars.as<fr_t>();
        LocalSlice sl[3];
        for (int k = 0; k < nsl; k++) {
            if (!c->copied[k]) HALO_CUDA(cudaEventCreateWithFlags(&c->copied[k], cudaEventDisableTiming));
            const uint64_t lo = cut[k], hi = k + 1 == nsl ? n_local : cut[k + 1];
            sl[k] = LocalSlice{d + lo, off_local + lo, hi - lo, c->copied[k], local_scalars + 4 * lo};
        }
        sharded_msm(c, sl, nsl, n_global, r);
    } else {
        if (n_local) h2d_copy(ctx, ctx->stage_scalars.p, local_scalars, n_local * sizeof(fr_t), ctx->stream);
        sharded_msm(c, ctx->stage_scalars.as<fr_t>(), off_local, n_local, n_global, r);
    }
    jac_t j;
    xyzz_to_jac(j, r);
    memcpy(out_jac, &j, 96);
    COMM_CATCH(ctx)
}

// One all-gather of a Jacobian point per rank + ordered sum: combines results of calls that already finished per rank
// (the pipelined halo_msm_gens_submit / _collect path of a weak-scaling run).
int halo_comm_allgather_sum(halo_comm* c, const uint64_t point_jac[12], uint64_t out_jac[12]) {
    if (!c || !point_jac || !out_jac) return HALO_EINVAL;
    halo_ctx* ctx = c->ctx;
    NcclApi* api = nccl_api();
    if (!api) return comm_fail(ctx, HALO_ENCCL, nccl_load_error());
    COMM_TRY(ctx)
    cudaStream_t st = c->side;
    HALO_CUDA(cudaMemcpyAsync(c->side_send.p, point_jac, 96, cudaMemcpyHostToDevice, st));
    HALO_NCCL(api, AllGather(c->side_send.p, c->side_recv.p, 96, NCCL_UINT8, c->comm, st));
    HALO_CUDA(cudaMemcpyAsync(c->h_side, c->side_recv.p, (size_t)96 * c->size, cudaMemcpyDeviceToHost, st));
    HALO_CUDA(cudaStreamSynchronize(st));
    int rc = halo_points_sum(c->h_side, (uint64_t)c->size, out_jac);
    if (rc) return rc;
    COMM_CATCH(ctx)
}

}  // extern "C"

// ---- node form: one caller, g devices ----------------------------------------------------------------------------------
struct halo_mgpu {
    int g = 0;
    uint64_t n_total = 0;
    std::vector<halo_ctx*> ctxs;
    std::vector<halo_comm*> comms;
    std::vector<uint64_t> first, count;
    // one persistent worker per device: NCCL collectives of one process must be issued concurrently, one thread per
    // communicator (or inside a group call); the workers also keep each device's CUDA context current on its own thread
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_job, cv_done;
    uint64_t job_seq = 0;
    int pending = 0;
    bool quit = false;
    std::function<int(int)> job;  // job(rank) -> status
    std::vector<int> status;
    std::vector<uint64_t> results;  // [g][12]
    std::string last_error;
};

namespace {
void mgpu_worker(halo_mgpu* m, int r) {
    uint64_t seen = 0;
    cudaSetDevice(m->ctxs[r]->device);
    for (;;) {
        std::function<int(int)> job;
        {
            std::unique_lock<std::mutex> lk(m->mu);
            m->cv_job.wait(lk, [&] { return m->quit || m->job_seq != seen; });
            if (m->quit) return;
            seen = m->job_seq;
            job = m->job;
        }
        int rc = HALO_ECUDA;
        try {
            rc = job(r);
        } catch (...) {
        }
        {
            std::lock_guard<std::mutex> lk(m->mu);
            m->status[r] = rc;
            if (--m->pending == 0) m->cv_done.notify_all();
        }
    }
}
// Runs job(r) on every worker and waits; returns the first failing status.
int mgpu_run(halo_mgpu* m, std::function<int(int)> job) {
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->job = std::move(job);
        m->pending = m->g;
        m->job_seq++;
    }
    m->cv_job.notify_all();
    std::unique_lock<std::mutex> lk(m->mu);
    m->cv_done.wait(lk, [&] { return m->pending == 0; });
    for (int r = 0; r < m->g; r++)
        if (m->status[r] != HALO_OK) {
            m->last_error = std::string("device ") + std::to_string(m->ctxs[r]->device) + ": " + m->ctxs[r]->last_error;
            return m->status[r];
        }
    return HALO_OK;
}
}  // namespace

extern "C" {

int halo_mgpu_create(const int* devices, int g, uint64_t n_total, int precompute_window, halo_mgpu** out) {
    if (!devices || !out || g < 1 || g > 64 || n_total < (uint64_t)g) return HALO_EINVAL;
    *out = nullptr;
    NcclApi* api = nccl_api();
    if (!api) return HALO_ENCCL;
    halo_mgpu* m = new halo_mgpu();
    m->g = g;
    m->n_total = n_total;
    m->ctxs.assign(g, nullptr);
    m->comms.assign(g, nullptr);
    m->first.resize(g), m->count.resize(g), m->status.assign(g, HALO_OK), m->results.assign((size_t)g * 12, 0);
    int rc = HALO_OK;
    std::vector<ncclComm_t> nc(g, nullptr);
    for (int r = 0; r < g && rc == HALO_OK; r++) {
        halo_comm_slice(n_total, r, g, &m->first[r], &m->count[r]);
        rc = halo_ctx_create(devices[r], m->count[r], &m->ctxs[r]);
    }
    if (rc == HALO_OK && api->CommInitAll(nc.data(), g, devices) != 0) rc = HALO_ENCCL;
    if (rc == HALO_OK) {
        try {
            for (int r = 0; r < g; r++) {
                halo_comm* c = new halo_comm();
                m->comms[r] = c;
                c->ctx = m->ctxs[r];
                c->comm = nc[r];
                c->rank = r;
                c->size = g;
                c->n_total = n_total;
                HALO_CUDA(cudaSetDevice(c->ctx->device));
                comm_alloc(c);
            }
        } catch (...) {
            rc = HALO_ECUDA;
        }
    }
    if (rc != HALO_OK) {
        for (int r = 0; r < g; r++) {
            if (m->comms[r]) halo_comm_destroy(m->comms[r]);
            else if (nc[r]) api->CommDestroy(nc[r]);
            if (m->ctxs[r]) halo_ctx_destroy(m->ctxs[r]);
        }
        delete m;
        return rc;
    }
    for (int r = 0; r < g; r++) m->workers.emplace_back(mgpu_worker, m, r);
    // public parameters: every device derives its own slice of the generators (K6) and, optionally, its tables
    rc = mgpu_run(m, [m, precompute_window](int r) {
        int s = halo_derive_generators_range(m->ctxs[r], m->first[r], m->count[r]);
        if (s == HALO_OK && precompute_window >= 0) s = halo_comm_precompute_generators(m->comms[r], precompute_window);
        return s;
    });
    if (rc != HALO_OK) {
        halo_mgpu_destroy(m);
        return rc;
    }
    *out = m;
    return HALO_OK;
}

void halo_mgpu_destroy(halo_mgpu* m) {
    if (!m) return;
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->quit = true;
    }
    m->cv_job.notify_all();
    for (auto& t : m->workers)
        if (t.joinable()) t.join();
    for (int r = 0; r < m->g; r++) {
        if (m->comms[r]) halo_comm_destroy(m->comms[r]);
        if (m->ctxs[r]) halo_ctx_destroy(m->ctxs[r]);
    }
    delete m;
}

int halo_mgpu_size(const halo_mgpu* m) { return m ? m->g : 0; }
halo_ctx* halo_mgpu_ctx(halo_mgpu* m, int i) { return (m && i >= 0 && i < m->g) ? m->ctxs[i] : nullptr; }
const char* halo_mgpu_last_error(halo_mgpu* m) { return m ? m->last_error.c_str() : "null handle"; }

// sum_{i<n} scalars[i] * G_i over the first n generators of the sharded set: device r takes the part of [0, n) that falls
// into its slice, copies those scalars itself (g concurrent H2D copies from the caller's buffer), and all devices meet in
// the one all-gather.  The drop-in for group.rs:24-26 as called by pedersen.rs:14 with more than one GPU.
int halo_mgpu_msm_gens(halo_mgpu* m, const uint64_t* scalars, uint64_t n, uint64_t out_jac[12]) {
    if (!m || !out_jac || (!scalars && n)) return HALO_EINVAL;
    if (n > m->n_total) {
        m->last_error = "halo_mgpu_msm_gens: n exceeds the sharded generator set";
        return HALO_EINVAL;
    }
    int rc = mgpu_run(m, [m, scalars, n](int r) {
        const uint64_t lo = m->first[r];
        const uint64_t n_local = n > lo ? (n - lo < m->count[r] ? n - lo : m->count[r]) : 0;
        // n_global is passed as the FULL set size: every call then uses one plan (and the tables) however short n is
        return halo_msm_gens_sharded(m->comms[r], scalars + 4 * lo, 0, n_local, m->n_total, m->results.data() + 12 * (size_t)r);
    });
    if (rc != HALO_OK) return rc;
    memcpy(out_jac, m->results.data(), 96);  // every rank holds the same sum
    return HALO_OK;
}

}  // extern "C"
