// msm.cuh -- internal interface of the MSM engine (msm.cu).
#pragma once
#include <functional>

#include "common.cuh"

namespace halo {
// One MSM problem, all pointers device resident: sum_{i<n} scalars[i] * bases[i] plus an optional short "tail"
// of extra (base, scalar) pairs held elsewhere in memory (used for the H' term of the IPA rounds, pcdl.rs:204,208).
struct MsmInput {
    const affine_t* bases = nullptr;
    const fr_t* scalars = nullptr;
    uint32_t n = 0;
    const affine_t* tail_bases = nullptr;
    const fr_t* tail_scalars = nullptr;
    uint32_t n_tail = 0;
    // FIXED-base mode: bases = table of precomputed multiples, table[w * fixed_stride + fixed_first + i]
    uint32_t fixed_stride = 0;
    uint32_t fixed_first = 0;
    // Segmented MSM (segs > 1, no tail): segs independent MSMs over the same bases in one pass.  The scalar at packed position
    // seg_off[s] <= i < seg_off[s + 1] (device array of segs + 1 entries) multiplies base i - seg_off[s]; segment s has its own
    // bucket set and its own window partials (msm_enqueue: 3 W partials per segment, segment-major).
    uint32_t segs = 1;
    const uint32_t* seg_off = nullptr;
};
MsmPlan msm_make_fixed_plan(uint64_t n, int force_c);
// The plan of an MSM of n points: the FIXED-base tables' plan or the variable-base window of n points (c, else the context's
// forced window, else the measured choice), over `segs` segments, with the context's reduction kernel.  Plans are final when
// made: msm_enqueue and msm_finish_host read them as they are.
MsmPlan msm_plan(const halo_ctx* ctx, uint64_t n, bool fixed, int c = 0, uint32_t segs = 1);
// Window partials an MSM leaves in d_out: (E, A2, R2) per window (one window in FIXED mode) and segment, segment-major
inline size_t msm_parts(const MsmPlan& p) { return (size_t)3 * (p.fixed ? 1 : p.W) * p.segs; }
// FIXED base for an MSM of n points over the resident generators (tables present, enough points to amortise the wide window)
bool gens_use_fixed(const halo_ctx* ctx, uint64_t n);
// The MSM of n scalars over the resident generators G_first..: over their precomputed multiples when `fixed`
MsmInput gens_msm_input(const halo_ctx* ctx, bool fixed, const fr_t* scalars, uint64_t first, uint64_t n);
// Counting sort of an MSM ahead of its accumulation: own stream (high priority), own sort buffers, throttled grid.
struct SortAhead {
    MsmWorkspace* ws;
    cudaStream_t stream;
    cudaEvent_t sorted;
    int ctas_per_sm;  // 0: full grid
};
// Device part of one MSM: its msm_parts(plan) partial points into d_out (see msm.cu).
void msm_enqueue(halo_ctx* ctx, const MsmInput& in, const MsmPlan& plan, xyzz_t* d_out, int lane = 0, const SortAhead* ahead = nullptr);
// msm_enqueue, then the copy of its partials from d_out to the pinned h_out on the lane's stream
void msm_enqueue_to_host(halo_ctx* ctx, const MsmInput& in, const MsmPlan& plan, xyzz_t* d_out, xyzz_t* h_out, int lane = 0,
                         const SortAhead* ahead = nullptr);
// Phase timings of the last MSM on lane 0 under profiling (events recorded by msm_enqueue, complete) into ctx->last
void msm_read_timings(halo_ctx* ctx);
// f(0) .. f(k - 1) on up to 16 host threads (host finishes of variable-base MSMs: ~255 doublings each)
void host_parallel(size_t k, const std::function<void(size_t)>& f);
// First `passes` levels of the bucket sums as flat pairwise affine additions with batched inversion (msm_pairs.cu).
const affine_t* pair_tree_enqueue(halo_ctx* ctx, MsmWorkspace& ws, cudaStream_t st, const MsmInput& in, const uint32_t* entries,
                                  const uint32_t* total_slots, uint64_t slots_max, int passes);
// vals[i] <- 1 / vals[i] for n non-zero elements of Fq, in place (Montgomery's trick over a product hierarchy, msm_pairs.cu)
void batch_invert(halo_ctx* ctx, cudaStream_t st, fq_t* vals, uint32_t n, DevBuf& scratch);
// Builds the table of precomputed multiples for the resident generators (FIXED-base mode).
void msm_precompute_tables(halo_ctx* ctx, int force_c);
// MSM over resident generators G_first.., FIXED-base when available.
void msm_gens_device(halo_ctx* ctx, const fr_t* d_scalars, uint64_t first, uint64_t n, xyzz_t& out);
// Up to 4 MSMs enqueued back to back with a single synchronisation; results on the host.
void msm_batch(halo_ctx* ctx, const MsmInput* ins, int count, xyzz_t* outs, const std::function<void()>* while_running = nullptr);
void msm_finish_host(const xyzz_t* wsums, const MsmPlan& plan, xyzz_t& out);
// Full MSM with device-resident inputs; synchronises the context stream and returns the point on the host.
void msm_device(halo_ctx* ctx, const affine_t* d_bases, const fr_t* d_scalars, uint64_t n, xyzz_t& out);
// Kernels of the second translation unit of msm.cu (msm_small.cu: out-of-line field multiplication): four (or two) lanes per
// bucket for the accumulation of small MSMs, and the quad-cooperative bucket reduction.
void launch_accumulate_quad(cudaStream_t st, int lanes, int minb, const affine_t* bases, uint32_t n, const affine_t* tail_bases,
                            const uint32_t* offsets, const uint32_t* entries, uint32_t NB, xyzz_t* buckets, uint32_t split_len);
void launch_reduce_slabs_quad(cudaStream_t st, dim3 grid, int T, int log_s, const xyzz_t* in, const xyzz_t* extra, size_t in_stride,
                              xyzz_t* outA, xyzz_t* outR, xyzz_t* outE, int out_stride);
}  // namespace halo
