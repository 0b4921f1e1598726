// common.cuh -- shared host-side declarations for libhalo_b200.so (context, workspaces, error plumbing).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>
#include <string>
#include <vector>

#include "ec.cuh"

namespace halo {

// Error codes cross the C ABI as ints; see include/halo_b200.h.
enum : int {
    E_OK = 0,
    E_INVAL = -1,
    E_LEN = -2,
    E_CUDA = -3,
    E_NCCL = -4,
    E_NOMEM = -5,
    E_STATE = -6,
    E_IO = -7,
};

struct CudaError {
    cudaError_t err;
    const char* what;
    const char* file;
    int line;
};

#define HALO_CUDA(expr)                                                      \
    do {                                                                     \
        cudaError_t _e = (expr);                                             \
        if (_e != cudaSuccess) throw halo::CudaError{_e, #expr, __FILE__, __LINE__}; \
    } while (0)

// Device buffer that only grows; owned by a context, never handed across the ABI.  Every allocation carries a 256-byte
// canary behind its end (compute-sanitizer is not available on this pool): halo_test_check_canaries() verifies that no
// kernel wrote past any live buffer.
struct DevBuf;
std::vector<DevBuf*>& devbuf_registry();
std::mutex& devbuf_registry_mutex();  // contexts on different host threads grow / release buffers concurrently
struct DevBuf {
    static constexpr size_t CANARY = 256;
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void reserve(size_t bytes) {
        if (bytes <= cap) return;
        release();
        HALO_CUDA(cudaMalloc(&p, bytes + CANARY));
        cap = bytes;
        HALO_CUDA(cudaMemset(static_cast<char*>(p) + cap, 0xA5, CANARY));
        std::lock_guard<std::mutex> lock(devbuf_registry_mutex());
        devbuf_registry().push_back(this);
    }
    void release() {
        if (p) {
            cudaFree(p);
            std::lock_guard<std::mutex> lock(devbuf_registry_mutex());
            auto& r = devbuf_registry();
            for (size_t i = 0; i < r.size(); i++)
                if (r[i] == this) {
                    r[i] = r.back();
                    r.pop_back();
                    break;
                }
        }
        p = nullptr;
        cap = 0;
    }
    bool canary_ok() const {
        if (!p) return true;
        unsigned char h[CANARY];
        if (cudaMemcpy(h, static_cast<const char*>(p) + cap, CANARY, cudaMemcpyDeviceToHost) != cudaSuccess) return false;
        for (size_t i = 0; i < CANARY; i++)
            if (h[i] != 0xA5) return false;
        return true;
    }
    template <class T>
    T* as() const {
        return reinterpret_cast<T*>(p);
    }
};

// MSM plan: window width c, W windows, M = 2^(c-1) buckets per window (signed digits).
// The 255 scalar bits are split into W windows of near-equal width (<= c, top window <= c - 1) so that
// for uniform scalars every window fills its buckets evenly; a short top window would otherwise pile
// n / 2^t entries into a handful of buckets and serialise their accumulation.
constexpr int MSM_MAX_WINDOWS = 64;
struct MsmWidths {
    uint8_t w[MSM_MAX_WINDOWS];
};
struct MsmPlan {
    int c = 0;
    int W = 0;
    uint32_t M = 0;
    uint32_t NB = 0;  // segs * (W * M (variable base) or M (fixed base: one shared bucket set))
    uint32_t segs = 1;  // segmented MSM (halo_msm_gens_many): one bucket set per segment, segment s owns buckets [s NB / segs, ..)
    bool fixed = false;
    MsmWidths widths;
    // bucket reduction geometry: slabs of red_T << red_log_s buckets
    int red_T = 0, red_log_s = 0;
    uint32_t red_slabs = 0;
    bool red_quad = true;  // k_reduce_slabs_quad (quad-cooperative additions) or the one-lane k_reduce_slabs
};

struct MsmWorkspace {
    DevBuf counts, offsets, cursor, entries, buckets, wsums, scan_tmp;
    DevBuf task_bucket, task_partial;  // slab partials of the bucket reduction
    DevBuf split_ctrl, split_tasks, split_buckets, split_partials;  // oversized-bucket splitting
    DevBuf sort_tmp, sort_coarse, sort_fine;  // two-level counting sort: (fine bucket | entry) records grouped by coarse bin, per-CTA bin rows + directory, per-chunk bucket rows
    DevBuf pt_a, pt_b, pt_prefix, pt_levels;  // pair-tree passes (msm_pairs.cu): ping-pong slot arrays, prefixes, product hierarchy
};

// Operation list of the generator fold (ipa.cu, k_fold_multi), built on the host per opening round.
struct FoldOpsHost {
    uint8_t code[3072];
};

struct Timings {
    float digits_ms = 0, scan_ms = 0, scatter_ms = 0, accumulate_ms = 0, reduce_ms = 0, total_ms = 0;
};

}  // namespace halo

struct halo_ctx;
namespace halo {
// Host-to-device copy of a caller buffer on `st`.  Pinned (or registered) memory goes to cudaMemcpyAsync directly.  Large
// PAGEABLE buffers -- a Rust Vec<Fr>, a numpy array -- would be staged by the driver through one small bounce buffer at a
// fraction of the PCIe rate; they are instead copied by a few host threads into a ring of pinned chunks, each chunk's DMA
// enqueued as soon as it is filled.  Returns when the caller's buffer has been read completely (the DMAs may still run).
void h2d_copy(halo_ctx* ctx, void* dst, const void* src, size_t bytes, cudaStream_t st);
// Creates the copy / sort streams and the two pipeline slots of the context on first use (capi.cu).
void async_init(halo_ctx* ctx);
}  // namespace halo

// The opaque handle behind `halo_ctx*` (include/halo_b200.h).
struct halo_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    uint64_t max_n = 0;
    // public parameters (consts.rs:23-68): G_0..G_{n_gens-1} resident in HBM as Montgomery affine, S and H on host
    halo::DevBuf gens;
    uint64_t n_gens = 0;
    halo::affine_t S, H;
    bool have_SH = false;
    halo::DevBuf fixed_table;  // fixed-base table for generator derivation (K6)
    halo::DevBuf gens_pre;     // precomputed multiples 2^(off_w) G_i for the FIXED-base MSM
    halo::MsmPlan pre_plan;
    uint64_t pre_n = 0;
    bool use_fixed = true;
    // scratch
    halo::MsmWorkspace ws, ws2;  // ws2 / stream2: second lane for a pair of small MSMs (msm_batch)
    cudaStream_t stream2 = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    halo::DevBuf stage_scalars, stage_bases, stage_misc;
    halo::DevBuf poly_dev;  // polynomial left on the device by halo_h_lincomb_resident for halo_ipa_begin_resident
    halo::DevBuf lincomb_claims;  // claim descriptors of vec_h_lincomb
    halo::DevBuf combine_in, combine_work, combine_inv_scratch;  // k_point_combine (combine.cu): inputs, work and outputs, inversions
    uint64_t poly_n = 0;
    // halo_poly_upload / halo_poly_eval_many: the k uploaded polynomials and their k + 1 segment starts, kept for the
    // evaluations, the quotient and the combinations (polys_k = 0: none resident); polys_n = the longest of them
    halo::DevBuf polys_dev, polys_off;
    uint64_t polys_k = 0, polys_n = 0;
    std::vector<uint64_t> polys_starts;  // host copy of polys_off
    // halo_poly_quotient: q of the resident polynomials, kept for halo_poly_lincomb_resident (quot_ready: q belongs to the
    // current upload), and the scratch of the K3c kernels (descriptors, carries)
    halo::DevBuf quot_dev, quot_scratch;
    uint64_t quot_n = 0;
    bool quot_ready = false;
    // buffers of the (single) in-flight PCDL opening, kept across openings: cudaMalloc / cudaFree of 100+ MB per open
    // costs tens of milliseconds
    halo::DevBuf ipa_G, ipa_cs, ipa_zs, ipa_pbar, ipa_tail, ipa_frozen;
    halo::DevBuf ipa_ops;          // device copy of fold_ops
    halo::FoldOpsHost fold_ops;    // per context: two contexts may open concurrently from two host threads
    halo::DevBuf ipa_sums, ipa_den, ipa_inv_scratch, ipa_bx, ipa_diff, ipa_den2;  // generator fold: XYZZ sums, ZZ * ZZZ and the batched inversion's hierarchy
    bool ipa_busy = false;
    // asynchronous MSM pipeline (halo_msm_gens_submit / _collect): two in-flight slots, H2D on its own stream so the copy
    // of call k+1 overlaps the kernels of call k
    struct AsyncSlot {
        halo::DevBuf scalars;
        halo::MsmWorkspace sort_ws;  // counts / offsets / entries of this slot's counting sort (SortAhead)
        cudaEvent_t copied = nullptr, done = nullptr, sorted = nullptr;
        halo::xyzz_t* h_parts = nullptr;  // pinned
        halo::MsmPlan plan;
        bool active = false;
        bool empty = false;
    } slots[2];
    cudaStream_t copy_stream = nullptr, sort_stream = nullptr;  // sort_stream: highest priority
    int next_slot = 0;
    // the outstanding batch of halo_h_msm_batch_submit / _collect: its own buffers, so that calls made between the two
    // (the verifier's C' on the device, other MSMs) neither wait for nor overwrite it
    struct HBatch {
        halo::DevBuf scalars;    // sum_j w_j coeffs(h_j)
        halo::DevBuf companion;  // bases | scalars | infinity flags of the companion MSM
        halo::DevBuf parts;      // window partials: generator MSM | companion MSM
        halo::xyzz_t* h_parts = nullptr;  // pinned, same layout
        cudaEvent_t done = nullptr;
        halo::MsmPlan plan;
        bool active = false;
        bool empty = false;  // no claims: the generator part is infinity
    } hb;
    // halo_msm_gens_many: two group buffers, so that the copy of group g+1 and the host finish of group g-1 overlap the
    // kernels of group g
    struct ManyBuf {
        halo::DevBuf scalars, seg_off, parts;
        uint32_t* h_seg_off = nullptr;  // pinned
        halo::xyzz_t* h_parts = nullptr;  // pinned
        size_t h_parts_cap = 0;  // points; h_seg_off holds MANY_MAX_SEGS + 1 starts
        cudaEvent_t copied = nullptr, done = nullptr;
    } many[2];
    // staging ring for host-to-device copies out of PAGEABLE caller memory (h2d_copy, capi.cu)
    static constexpr int STAGE_THREADS = 8, STAGE_SLOTS = 2;  // upper bound of threads; tune_stage_threads of them work
    static constexpr size_t STAGE_CHUNK = 8u << 20;
    void* stage_pinned[STAGE_THREADS * STAGE_SLOTS] = {};
    cudaEvent_t stage_ev[STAGE_THREADS * STAGE_SLOTS] = {};
    int tune_stage_pageable = 1;  // 0: hand pageable pointers to cudaMemcpyAsync as they are
    int tune_acc_quad_lanes = 0, tune_acc_quad_blocks = 0;  // k_accumulate_quad: lanes per bucket (2 / 4) and CTAs per SM (4 / 6); 0 = policy
    int tune_stage_threads = 4;   // host threads that copy pageable chunks into the pinned ring (1 .. STAGE_THREADS)
    void* pinned = nullptr;
    size_t pinned_cap = 0;
    int force_c = 0;
    int tune_acc_static = 0, tune_acc_blocks_per_sm = 0;
    int tune_acc_quad = 1;  // small MSMs: four lanes per bucket (k_accumulate_quad); 0: one lane per bucket
    int tune_acc_quad_max_buckets = 1 << 15;
    bool force_two_lanes = false;  // run a pair of large MSMs (deferred IPA rounds) on the two lanes as well
    int tune_ipa_two_lanes = 1, tune_ipa_freeze_len = 0;
    int tune_ipa_frozen_c = 9;   // window of the frozen-tail MSMs (8192 points): round 1 measured 10 best with the one-lane single-slab reduction;
                                 // with the two-level quad reduction 11 was (8192-point MSM 0.46 / 0.38 / 0.41 ms at c = 10 / 11 / 12), with
                                 // four lanes per bucket 10 again (0.32 / 0.35 ms at c = 10 / 11), and once the host's Horner finish halved
                                 // (assembly field core) 9: open at 2^20 46.0 -> 45.6 ms in three alternating runs
    int tune_combine_min_outputs = 1024;  // halo_test_point_combine: the device from this many outputs on, host GLV below (-1: never); measured crossover, DESIGN.md K5c
    int tune_fold_call_min_lg = 17;  // generator folds of >= 2^this outputs use the copy of k_fold_multi with the multiplication out of line (-1: never)
    int tune_ipa_defer = -1;    // -1: automatic (3 rounds when the FIXED-base tables cover the opening); 0: off; D: force
    int tune_ipa_defer2 = 0;    // later deferred stages over the materialised vector, at most this many rounds each; 0 = off: measured slower at 2^20
                                // (rounds 3-6 as one stage: 4 x 2.1 ms L / R + 5.3 ms latency-bound fold of 8192 outputs against 4.9 + 6.2 ms; profiles/r02_ipa_stage2_probe.txt)
    int tune_sort_ahead = 1;  // pipelined submit: CTAs per SM of the counting sort running beside the previous MSM (0: off)
    int tune_split_blocking = 23;  // halo_msm_gens: two point slices through the pipeline slots for n >= 2^this (0: never)
    int tune_split_second_16ths = 5;  // > 0: three slices (first, second, rest); the third copy starts when the first slice is collected
    int tune_split_first_16ths = 2;  // size of the first slice in sixteenths of n: its H2D copy is exposed, the second slice's copy hides behind
                                     // the first slice's kernels (2^24: 8 -> 41.1 ms, 6 -> 38.4, 5 -> 38.2, 4 -> 39.7, 3 -> 41.0; scripts/gpu_split_probe.py)
    bool sort2_attr = false;     // dynamic shared-memory opt-in of the staged sort kernels done on this context's device
    int tune_sort2 = 1;          // two-level counting sort with staged, coalesced writes for inputs of >= 2^tune_sort2_min_lg entries
    int tune_sort2_min_lg = 26;  // measured: 2^24 FIXED 6.15 -> 4.45 ms, 2^23 2.76 -> 2.31, 2^22 1.26 -> 1.29 (profiles/r02_sort2_v3_ab.jsonl)
    int tune_pair_bwd_async = 1;  // pass 0 of the pair tree: 1 = cp.async-staged operands + prefix loaded a step ahead (k_pair_bwd0, 5 CTAs per SM:
                                  // accumulation phase at 2^24 27.39 -> 26.75 ms; profiles/r02_pair_bwd_async_ab.jsonl), 0 = per-lane gathers
    int tune_reduce_quad = 1;   // 0: one-lane bucket reduction (k_reduce_slabs), for A/B measurements; applied by msm_plan
    int tune_pair_passes = -1;  // -1: automatic; 0: XYZZ accumulation only; P > 0: force P pair-tree passes
    // what msm_enqueue chose for the last MSM on each lane (halo_test_msm_route, layout in include/halo_b200_test.h); host
    // bookkeeping only, written next to the decisions themselves
    int msm_route[2][10] = {};
    uint64_t kernel_launches = 0;
    halo::Timings last;
    bool profile = false;
    cudaEvent_t ev[8] = {};
    std::string last_error;
};
