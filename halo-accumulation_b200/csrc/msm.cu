// msm.cu -- K2: Pippenger multi-scalar multiplication on sm_100a.
//
// Replaces `VariableBaseMSM::msm_unchecked` as called from group.rs:20 and group.rs:25 (callers:
// pedersen.rs:14, pcdl.rs:109,204,208,338, acc.rs:153,178,195).  Pipeline (all on one stream):
//   1. k_digits<COUNT>   scalars (Montgomery) -> canonical -> signed radix-2^c digits; histogram per bucket
//   2. exclusive scan    bucket offsets
//   3. k_digits<SCATTER> counting-sort scatter of (point index | sign) into bucket order
//   4. k_accumulate      one thread per bucket: XYZZ accumulator in registers, mixed adds of gathered bases
//   5. k_reduce_slabs    bucket reduction sum_k k * B_k: CTAs over slabs of buckets (running sums + block suffix scan),
//                        then one CTA per window over the slab partials
//   6. host              slab recombination and Horner over the window sums (O(255) doublings, independent of n)
// Two modes.  VARIABLE base (halo_msm, IPA rounds): W windows, W bucket sets.  FIXED base (resident generators with
// precomputed multiples 2^(off_w) G_i, halo_precompute_generators): every window's digit indexes ONE shared bucket set
// and selects the precomputed multiple instead, so the bucket reduction and the Horner doublings are paid once, not W
// times, and the window can be as wide as the bucket memory allows.
// Integer pipe bound (IMAD); see DESIGN.md for the roofline accounting.
#include <functional>

#include <system_error>
#include <thread>

#include "common.cuh"
#include "msm.cuh"

namespace halo {

// This file is compiled twice (see msm_small.cu): the normal translation unit holds everything except the two kernels whose
// lanes are few and out of step (k_accumulate_quad, k_reduce_slabs_quad); those live in the second unit, where the field
// multiplication is an out-of-line call (HALO_FP_MUL_CALL).
#ifndef HALO_MSM_SMALL_TU

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
static void plan_set_reduce(MsmPlan& p, bool quad);
static void plan_fill(MsmPlan& p, int c, bool fixed) {
    p.c = c;
    p.fixed = fixed;
    p.W = 255 / c + 1;  // c * W >= 256 > 255: the top window absorbs the final carry
    p.M = 1u << (c - 1);
    p.NB = fixed ? p.M : (uint32_t)p.W * p.M;
    // near-equal widths summing to 255; the low windows take the remainder so the top window is the narrow one
    int base = 255 / p.W, rem = 255 - base * p.W;
    for (int w = 0; w < MSM_MAX_WINDOWS; w++) p.widths.w[w] = w < p.W ? (uint8_t)(base + (w < rem ? 1 : 0)) : 0;
    plan_set_reduce(p, true);
}
// bucket reduction geometry: slabs of T * s buckets, T (logical) threads per CTA.  quad: k_reduce_slabs_quad (T <= 128
// quads, slabs of up to 2048 buckets); else k_reduce_slabs (T <= 256 threads).
static void plan_set_reduce(MsmPlan& p, bool quad) {
    // Measured (scripts/gpu_reduce_probe.py, profiles/r02_reduce_*): the reduction of one slab is a job for ONE CTA, and a
    // CTA's arithmetic runs on one SM (~0.4 G multiplications/s): with a slab per window, a 22-window MSM of 2048 buckets
    // per window kept 22 of the 148 SMs busy for 0.3 ms.  So windows of >= 1024 buckets are cut into slabs until every SM
    // has a CTA or two; a second launch (one CTA per window, 0.07 ms at 32-128 slabs, 0.31 ms at 1024) combines the slab
    // partials, hence at most 128 slabs per window and none for small windows.  The quad-cooperative kernel has the
    // shorter dependent chain but issues ~40 % more instructions per addition: it wins while the reduction is latency
    // bound (<= 3 * 2^17 buckets in all), the one-lane kernel wins beyond (2^22 variable base: 0.69 against 0.83 ms).
    const uint32_t nwin = (p.fixed ? 1u : (uint32_t)p.W) * p.segs;  // every window of every segment
    quad = quad && (uint64_t)nwin * p.M <= (p.fixed ? 524288u : 393216u);  // (one bucket set of 2^19: 0.80 -> 0.67 ms)
    p.red_quad = quad;
    if (!quad) {
        p.red_T = p.M < 256u ? (int)p.M : 256;
        p.red_log_s = 0;
        while (((uint32_t)p.red_T << p.red_log_s) < p.M && p.red_log_s < 3) p.red_log_s++;
        p.red_slabs = p.M / ((uint32_t)p.red_T << p.red_log_s);
        return;
    }
    uint32_t G = 1;
    if (p.M >= 512u)
        while (G * nwin < 296u && G < 128u && p.M / (2 * G) >= 256u) G *= 2;
    uint32_t B = p.M / G;                  // buckets per slab (power of two)
    while (B > 128u * 16u) B >>= 1;        // at most 16 items per logical thread
    uint32_t T = B / 8 ? B / 8 : 1;        // ~8 items per logical thread, 16 .. 128 quads per CTA
    if (B <= 512u) T = B / 4 ? B / 4 : 1;  // single-slab windows (frozen IPA rounds): 4 items, the shortest chain measured
    if (T < 16) T = B < 16 ? B : 16;
    if (T > 128) T = 128;
    p.red_T = (int)T;
    p.red_log_s = 0;
    while ((T << p.red_log_s) < B) p.red_log_s++;
    p.red_slabs = p.M / (T << p.red_log_s);
}

static int ceil_lg(uint64_t n) {
    int l = 0;
    while (((uint64_t)1 << l) < n) l++;
    return l;
}

// Window widths below are the measured optima on B200 (scripts/gpu_msm_probe.py sweeps: profiles/r01_msm_window_sweep.txt,
// re-measured with the two-level / quad-cooperative bucket reduction in profiles/r02_msm_window_sweep_variable.txt):
// total cost = W * (n mixed adds) + bucket reduction (~2.5 full adds per bucket).
static MsmPlan msm_make_plan(uint64_t n, int force_c) {
    const int lg = ceil_lg(n);
    // (third sweep, with four lanes per bucket below 2^15 buckets and the pair-pass policy by bucket fill:
    // profiles/r02_msm_window_sweep_variable_v3.txt -- smaller windows pay once their buckets are full enough for tree passes)
    int c = lg <= 6 ? 4 : lg <= 8 ? 7 : lg <= 10 ? 8 : lg <= 12 ? 11 : lg <= 15 ? 10 : lg <= 16 ? 11 : lg <= 19 ? 13 : 16;
    if (force_c) c = force_c;
    if (c < 4) c = 4;  // W = 255 / c + 1 <= MSM_MAX_WINDOWS
    if (c > 20) c = 20;
    MsmPlan p;
    plan_fill(p, c, false);
    return p;
}

// Fixed-base plan for `n` resident generators: one bucket set, W precomputed multiples per generator.
MsmPlan msm_make_fixed_plan(uint64_t n, int force_c) {
    const int lg = ceil_lg(n);
    int c = lg <= 17 ? 16 : lg <= 22 ? 19 : 20;
    if (force_c) c = force_c;
    if (c < 8) c = 8;
    if (c > 24) c = 24;
    while ((double)(255 / c + 1) * (double)n >= 2147483648.0 && c < 24) c++;  // entry = index | sign << 31
    MsmPlan p;
    plan_fill(p, c, true);
    return p;
}

// The reduction kernel is part of the plan (msm_finish_host undoes its slab geometry), so the reduce_quad knob is applied
// here, once, and not where the plan is run.
MsmPlan msm_plan(const halo_ctx* ctx, uint64_t n, bool fixed, int c, uint32_t segs) {
    MsmPlan p = fixed ? ctx->pre_plan : msm_make_plan(n, c ? c : ctx->force_c);
    p.NB *= segs;
    p.segs = segs;
    plan_set_reduce(p, ctx->tune_reduce_quad != 0);
    return p;
}

// ------------------------------------------------------------------------------------------------
// 1/3. digit extraction: count or scatter
// ------------------------------------------------------------------------------------------------
// VARIABLE: bucket = w * M + |d| - 1, entry = i.   FIXED: bucket = |d| - 1, entry = w * stride + first + i (the index of
// the precomputed multiple 2^(off_w) G_{first+i}).
// SEG (segmented MSM): scalar i of segment s (seg_off[s] <= i < seg_off[s + 1]) goes to bucket s * NB1 + (the bucket above)
// with i - seg_off[s] in place of i; the entry does not record the segment, so every later stage reads bases unchanged.
__device__ __forceinline__ uint32_t seg_of(const uint32_t* __restrict__ seg_off, uint32_t segs, uint32_t i) {
    uint32_t a = 0, b = segs;  // the last segment starting at or before i
    while (b - a > 1) {
        const uint32_t m = (a + b) >> 1;
        if (seg_off[m] <= i) a = m; else b = m;
    }
    return a;
}
// (the segmented scatter needs ~47 registers: at the 32 that full occupancy leaves it spilled; minBlocks 0 = no bound)
template <bool SCATTER, bool SEG>
__global__ void __launch_bounds__(256, SEG ? 4 : 0) k_digits(const fr_t* __restrict__ scalars, uint32_t n,
                                                const fr_t* __restrict__ tail_scalars, uint32_t n_tail, const MsmWidths widths,
                                                int W, uint32_t M, uint32_t fixed_stride, uint32_t fixed_first,
                                                uint32_t* __restrict__ counts, uint32_t* __restrict__ entries,
                                                const uint32_t* __restrict__ seg_off, uint32_t segs, uint32_t NB1) {
    // grid-stride: the launch normally covers every scalar with one thread; the pipelined path (SortAhead) runs the sort
    // of the NEXT MSM with a few CTAs per SM beside the accumulation kernels of the current one
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n + n_tail; i += gridDim.x * blockDim.x) {
    fr_t s = i < n ? scalars[i] : tail_scalars[i - n];
    uint32_t li = i, bofs = 0;  // index of the base, first bucket of the segment
    if (SEG) {
        const uint32_t sg = seg_of(seg_off, segs, i);
        li = i - seg_off[sg];
        bofs = sg * NB1;
    }
    uint32_t k[8];
    fp_to_canon(k, s);  // arkworks `into_bigint`
    uint32_t carry = 0;
    for (int w = 0; w < W; w++) {
        const uint32_t c = widths.w[w];
        uint32_t d = (k[0] & ((1u << c) - 1u)) + carry;
#pragma unroll
        for (int j = 0; j < 7; j++) k[j] = __funnelshift_r(k[j], k[j + 1], c);
        k[7] >>= c;
        carry = 0;
        uint32_t neg = 0;
        if (d > (1u << (c - 1))) {  // digit in (-2^(c-1), 2^(c-1)]; never taken in the top window (scalar < 2^255)
            d = (1u << c) - d;
            neg = 1;
            carry = 1;
        }
        if (d != 0) {
            uint32_t b = bofs + (fixed_stride ? (d - 1) : (uint32_t)w * M + (d - 1));
            // COUNT: histogram (a fire-and-forget RED).  SCATTER: `counts` holds the running write cursor of every bucket,
            // initialised to the bucket offsets, so the returned value is the absolute slot (one random L2 access less per
            // entry than offsets[b] + slot).
            uint32_t pos = atomicAdd(&counts[b], 1u);
            if (SCATTER) {
                uint32_t idx = fixed_stride ? (uint32_t)w * fixed_stride + fixed_first + li : li;
                entries[pos] = idx | (neg << 31);
            }
        }
    }
    }
}

// ------------------------------------------------------------------------------------------------
// 2. exclusive scan of u32 (three small kernels; NB <= 4096 * 2048)
// ------------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 16;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {
    __shared__ uint32_t warp_sums[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint32_t ws = lane < (int)(blockDim.x >> 5) ? warp_sums[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, ws, o);
            if (lane >= o) ws += y;
        }
        warp_sums[lane] = ws;
    }
    __syncthreads();
    uint32_t base = wid ? warp_sums[wid - 1] : 0;
    *total = warp_sums[(blockDim.x >> 5) - 1];
    return base + x - v;
}

// `round_mask` = 2^P - 1 rounds every count up to a multiple of 2^P first (padded segments for the pair tree, msm_pairs.cu)
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_local(const uint32_t* __restrict__ in, uint32_t* __restrict__ out,
                                                             uint32_t n, uint32_t round_mask, uint32_t* __restrict__ tile_sums) {
    uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint32_t sum = 0;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; j++) {
        v[j] = (base + j < n) ? ((in[base + j] + round_mask) & ~round_mask) : 0;
        sum += v[j];
    }
    uint32_t total;
    uint32_t ex = block_exclusive_scan(sum, &total);
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; j++) {
        if (base + j < n) out[base + j] = ex;
        ex += v[j];
    }
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}
// single CTA: exclusive scan of up to 2048 tile sums, also writes the grand total to out_total
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tiles(uint32_t* tile_sums, uint32_t ntiles, uint32_t* out_total) {
    constexpr int PER = 8;  // 256 * 8 = 2048 tiles
    uint32_t v[PER], sum = 0;
#pragma unroll
    for (int j = 0; j < PER; j++) {
        uint32_t idx = threadIdx.x * PER + j;
        v[j] = idx < ntiles ? tile_sums[idx] : 0;
        sum += v[j];
    }
    uint32_t total;
    uint32_t ex = block_exclusive_scan(sum, &total);
#pragma unroll
    for (int j = 0; j < PER; j++) {
        uint32_t idx = threadIdx.x * PER + j;
        if (idx < ntiles) tile_sums[idx] = ex;
        ex += v[j];
    }
    if (threadIdx.x == 0) *out_total = total;
}
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_add(uint32_t* __restrict__ out, uint32_t n,
                                                           const uint32_t* __restrict__ tile_sums) {
    uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    uint32_t add = tile_sums[blockIdx.x];
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; j++)
        if (base + j < n) out[base + j] += add;
}

// Pad slots [offsets[b] + counts[b], offsets[b + 1]) of every bucket segment get the "infinity" entry (pair tree only).
__global__ void __launch_bounds__(256) k_fill_pads(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ offsets, uint32_t NB,
                                                   uint32_t* __restrict__ entries) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= NB) return;
    for (uint32_t e = offsets[b] + counts[b], end = offsets[b + 1]; e < end; e++) entries[e] = 0xffffffffu;
}
__global__ void __launch_bounds__(256) k_shift_offsets(const uint32_t* __restrict__ in, uint32_t n, int shift, uint32_t* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i] >> shift;
}

// offsets[0..n] = exclusive scan of counts[0..n) with offsets[n] = total
static void exclusive_scan(const uint32_t* counts, uint32_t* offsets, uint32_t n, uint32_t round_mask, uint32_t* tmp,
                           cudaStream_t st, uint64_t* launches) {
    uint32_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    k_scan_local<<<ntiles, SCAN_THREADS, 0, st>>>(counts, offsets, n, round_mask, tmp);
    k_scan_tiles<<<1, SCAN_THREADS, 0, st>>>(tmp, ntiles, offsets + n);
    k_scan_add<<<ntiles, SCAN_THREADS, 0, st>>>(offsets, n, tmp);
    *launches += 3;
}

// ------------------------------------------------------------------------------------------------
// 1-3 (large MSMs): two-level counting sort with shared-memory atomics and STAGED, COALESCED writes.  The one-pass sort above
// pays two L2 atomics per entry (a RED for the histogram, an atomic with return for the write cursor) plus a random 4-byte
// store: 6.1 ms of a 34 ms MSM at 2^24.  What bounds it is not the atomics but the number of scattered store transactions
// (~45-50 G/s to HBM-backed lines whatever their size; ~94 G/s inside an L2-resident region): two earlier versions of this
// sort that only moved the atomics into shared memory measured 8.6 and 9.5 ms (profiles/r02_sort2_v1_ab.jsonl, _v2_).  So
// here every record leaves a CTA as part of a run.  Buckets are grouped into NC coarse bins of NF = 1024 consecutive buckets;
//   A   k_sort_coarse_count    every CTA counts the entries of ITS tiles (tile = 1024 scalars, CTA c owns tiles c, c + grid, ..)
//                              per coarse bin in shared memory and writes the row cta_hist[cta][bin]
//   S1  k_sort_coarse_scan     per bin: total, offset, chunk directory (chunks of 8192 records), and the row turned into the
//                              CTA's first slot inside the bin (no global atomic anywhere: every slot is known in advance)
//   B   k_sort_coarse_scatter  the same tiles again: count, scan, place the tile's records into shared memory IN BIN ORDER,
//                              write them out so that consecutive threads write consecutive (fine bucket | entry) records of
//                              a bin's run (26 records = 208 bytes per bin and tile at 2^24)
//   C   k_sort_fine_count      per chunk: histogram over the bin's 1024 fine buckets -> row fine[chunk][bucket]
//   S2a k_sort_fine_total      per bucket: sum over its bin's chunks -> the global bucket counts (the array the one-pass sort
//                              produces; scan, rounding to 2^P slots and padding are shared with it)
//   S3  k_sort_fine_base       per bucket: rows turned into each chunk's first slot inside the bucket
//   D   k_sort_fine_scatter    per chunk: records placed into shared memory IN BUCKET ORDER and written out in that order (the
//                              ~8 entries a bucket gets from a chunk leave as one or two transactions, inside the bin's own
//                              L2-resident region)
// Chunks make C / D insensitive to skew (all scalars equal puts every entry into a handful of bins: such a bin is cut into
// many chunks whose shared-memory atomics serialise, nothing worse).  Output (counts, offsets, entries, pad slots) is what
// the downstream kernels expect from the one-pass sort, up to the order inside a bucket, which no consumer depends on.
// Measured at 2^24 FIXED: 0.46 (A) + 0.03 + 1.56 (B) + 0.48 (C) + 0.1 + 1.65 (D) = 4.45 ms against 6.15; used from 2^26 entries.
// ------------------------------------------------------------------------------------------------
constexpr int S2_THREADS = 512;
constexpr int S2_MAX_W = 20;        // windows per scalar (c >= 13)
constexpr uint32_t S2_NF_LOG = 10;  // fine buckets per coarse bin
constexpr uint32_t S2_NF = 1u << S2_NF_LOG;
constexpr uint32_t S2_MAX_NC = 2048;
constexpr uint32_t S2_CHUNK = 8192;  // entries per chunk
constexpr uint32_t S2_MAX_CTAS = 592;
constexpr int S2_SPT = 2;                                // scalars per thread and tile (coarse passes)
constexpr uint32_t S2_TILE = S2_THREADS * S2_SPT;        // scalars per tile: CTA c owns the tiles c, c + grid, ..
constexpr int S2_BIN_SHIFT = 42;                         // staged record: entry (32) | fine bucket (10) | coarse bin (12)
constexpr uint64_t S2_REC_MASK = ((uint64_t)1 << S2_BIN_SHIFT) - 1;

// Calls f(bucket, entry) for every non-zero digit of scalar i (the digit rule of k_digits; bofs: first bucket of the scalar's
// segment, i: its index in the segment).  Bits are picked straight out of the canonical limbs (no 256-bit shift per window).
template <class F>
__device__ __forceinline__ void s2_for_digits(const fr_t& s, uint32_t i, uint32_t bofs, const MsmWidths& widths, int W, uint32_t M,
                                              uint32_t fixed_stride, uint32_t fixed_first, F&& f) {
    uint32_t k[9];
    fp_to_canon(k, s);
    k[8] = 0;
    uint32_t carry = 0, off = 0;
    for (int w = 0; w < W; w++) {
        const uint32_t c = widths.w[w];
        const uint32_t lo = off >> 5, sh = off & 31u;
        const uint32_t bits = __funnelshift_r(k[lo], k[lo + 1], sh);  // k[lo] >> sh | k[lo + 1] << (32 - sh)
        uint32_t d = (bits & ((1u << c) - 1u)) + carry;
        off += c;
        carry = 0;
        uint32_t neg = 0;
        if (d > (1u << (c - 1))) {
            d = (1u << c) - d;
            neg = 1;
            carry = 1;
        }
        if (d != 0) {
            const uint32_t b = bofs + (fixed_stride ? (d - 1) : (uint32_t)w * M + (d - 1));
            const uint32_t idx = fixed_stride ? (uint32_t)w * fixed_stride + fixed_first + i : i;
            f(b, idx | (neg << 31));
        }
    }
}

// s2_for_digits on packed scalar i of a (SEG: segmented) MSM
template <bool SEG, class F>
__device__ __forceinline__ void s2_for_digits_at(const fr_t& s, uint32_t i, const uint32_t* __restrict__ seg_off, uint32_t segs, uint32_t NB1,
                                                 const MsmWidths& widths, int W, uint32_t M, uint32_t fixed_stride, uint32_t fixed_first, F&& f) {
    uint32_t li = i, bofs = 0;
    if (SEG) {
        const uint32_t sg = seg_of(seg_off, segs, i);
        li = i - seg_off[sg];
        bofs = sg * NB1;
    }
    s2_for_digits(s, li, bofs, widths, W, M, fixed_stride, fixed_first, f);
}

template <bool SEG>
__global__ void __launch_bounds__(S2_THREADS) k_sort_coarse_count(const fr_t* __restrict__ scalars, uint32_t n,
                                                                  const fr_t* __restrict__ tail_scalars, uint32_t n_tail,
                                                                  const MsmWidths widths, int W, uint32_t M, uint32_t fixed_stride,
                                                                  uint32_t fixed_first, uint32_t NC, uint32_t* __restrict__ cta_hist,
                                                                  const uint32_t* __restrict__ seg_off, uint32_t segs, uint32_t NB1) {
    __shared__ uint32_t hist[S2_MAX_NC];
    for (uint32_t t = threadIdx.x; t < NC; t += blockDim.x) hist[t] = 0;
    __syncthreads();
    const uint32_t ntot = n + n_tail, ntiles = (ntot + S2_TILE - 1) / S2_TILE;
    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
#pragma unroll
        for (int r = 0; r < S2_SPT; r++) {
            const uint32_t i = tile * S2_TILE + (uint32_t)r * S2_THREADS + threadIdx.x;
            if (i < ntot) {
                const fr_t s = i < n ? scalars[i] : tail_scalars[i - n];
                s2_for_digits_at<SEG>(s, i, seg_off, segs, NB1, widths, W, M, fixed_stride, fixed_first,
                                      [&](uint32_t b, uint32_t) { atomicAdd(&hist[b >> S2_NF_LOG], 1u); });
            }
        }
    __syncthreads();
    for (uint32_t t = threadIdx.x; t < NC; t += blockDim.x) cta_hist[(size_t)blockIdx.x * NC + t] = hist[t];
}

// one CTA of 1024 threads, up to 2 bins per thread
__global__ void __launch_bounds__(1024) k_sort_coarse_scan(uint32_t* __restrict__ cta_hist, uint32_t nctas, uint32_t NC,
                                                           uint32_t* __restrict__ coarse_off, uint32_t* __restrict__ chunk_pre) {
    uint32_t tot[2] = {0, 0};
    for (int r = 0; r < 2; r++) {
        const uint32_t t = threadIdx.x * 2 + r;
        if (t < NC) {
            uint32_t acc = 0;
#pragma unroll 8
            for (uint32_t c = 0; c < nctas; c++) acc += cta_hist[(size_t)c * NC + t];
            tot[r] = acc;
        }
    }
    uint32_t total, ctotal;
    const uint32_t ch0 = (tot[0] + S2_CHUNK - 1) / S2_CHUNK, ch1 = (tot[1] + S2_CHUNK - 1) / S2_CHUNK;
    uint32_t ex = block_exclusive_scan(tot[0] + tot[1], &total);
    __syncthreads();
    uint32_t cex = block_exclusive_scan(ch0 + ch1, &ctotal);
    __syncthreads();
    for (int r = 0; r < 2; r++) {
        const uint32_t t = threadIdx.x * 2 + r;
        if (t < NC) {
            const uint32_t off = ex + (r ? tot[0] : 0), coff = cex + (r ? ch0 : 0);
            coarse_off[t] = off;
            chunk_pre[t] = coff;
            uint32_t base = off;
            for (uint32_t c = 0; c < nctas; c += 8) {
                uint32_t v[8];
#pragma unroll
                for (int j = 0; j < 8; j++) v[j] = c + j < nctas ? cta_hist[(size_t)(c + j) * NC + t] : 0;
#pragma unroll
                for (int j = 0; j < 8; j++)
                    if (c + j < nctas) {
                        cta_hist[(size_t)(c + j) * NC + t] = base;
                        base += v[j];
                    }
            }
        }
    }
    if (threadIdx.x == 0) {
        coarse_off[NC] = total;
        chunk_pre[NC] = ctotal;
    }
}

// exclusive scan of v[0 .. len) (len <= 4 * blockDim) into out[0 .. len], out[len] = total; every thread of the CTA calls it
__device__ __forceinline__ void s2_block_scan(const uint32_t* __restrict__ v, uint32_t len, uint32_t* __restrict__ out) {
    const uint32_t per = (len + blockDim.x - 1) / blockDim.x;  // <= 4
    const uint32_t b0 = threadIdx.x * per;
    uint32_t loc[4], sum = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        loc[j] = ((uint32_t)j < per && b0 + j < len) ? v[b0 + j] : 0;
        sum += loc[j];
    }
    uint32_t total;
    uint32_t ex = block_exclusive_scan(sum, &total);
    __syncthreads();  // (block_exclusive_scan's own scratch may be reused by the next call)
#pragma unroll
    for (int j = 0; j < 4; j++)
        if ((uint32_t)j < per && b0 + j < len) {
            out[b0 + j] = ex;
            ex += loc[j];
        }
    if (threadIdx.x == 0) out[len] = total;
}

// B: the CTA's tiles again.  Per tile: count per bin, scan, place every record into a shared-memory staging area IN BIN ORDER,
// then write the staged records out so that consecutive threads write consecutive addresses of a bin's run (26 records =
// 208 bytes per bin and tile at 2^24): what limits a scatter on this part is the number of store transactions, ~45 G/s,
// whatever their size, so a record must not be its own transaction.  Dynamic shared memory: gcur[NC] | hist[NC] | toff[NC + 1]
// | stage[S2_TILE * W] (8 bytes each).
template <bool SEG>
__global__ void __launch_bounds__(S2_THREADS) k_sort_coarse_scatter(const fr_t* __restrict__ scalars, uint32_t n,
                                                                    const fr_t* __restrict__ tail_scalars, uint32_t n_tail,
                                                                    const MsmWidths widths, int W, uint32_t M, uint32_t fixed_stride,
                                                                    uint32_t fixed_first, uint32_t NC, const uint32_t* __restrict__ cta_base,
                                                                    uint64_t* __restrict__ tmp, const uint32_t* __restrict__ seg_off,
                                                                    uint32_t segs, uint32_t NB1) {
    extern __shared__ __align__(16) unsigned char s2_smem[];
    uint32_t* gcur = reinterpret_cast<uint32_t*>(s2_smem);
    uint32_t* hist = gcur + NC;
    uint32_t* toff = hist + NC;
    uint64_t* stage = reinterpret_cast<uint64_t*>(s2_smem + (((size_t)(3 * NC + 1) * 4 + 15) & ~(size_t)15));
    for (uint32_t t = threadIdx.x; t < NC; t += blockDim.x) gcur[t] = cta_base[(size_t)blockIdx.x * NC + t];
    const uint32_t ntot = n + n_tail, ntiles = (ntot + S2_TILE - 1) / S2_TILE;
    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (uint32_t t = threadIdx.x; t < NC; t += blockDim.x) hist[t] = 0;
        __syncthreads();
#pragma unroll
        for (int r = 0; r < S2_SPT; r++) {
            const uint32_t i = tile * S2_TILE + (uint32_t)r * S2_THREADS + threadIdx.x;
            if (i < ntot) {
                const fr_t s = i < n ? scalars[i] : tail_scalars[i - n];
                s2_for_digits_at<SEG>(s, i, seg_off, segs, NB1, widths, W, M, fixed_stride, fixed_first,
                                      [&](uint32_t b, uint32_t) { atomicAdd(&hist[b >> S2_NF_LOG], 1u); });
            }
        }
        __syncthreads();
        s2_block_scan(hist, NC, toff);
        __syncthreads();
        for (uint32_t t = threadIdx.x; t < NC; t += blockDim.x) hist[t] = 0;  // now the placement cursor inside the tile
        __syncthreads();
#pragma unroll
        for (int r = 0; r < S2_SPT; r++) {
            const uint32_t i = tile * S2_TILE + (uint32_t)r * S2_THREADS + threadIdx.x;
            if (i < ntot) {
                const fr_t s = i < n ? scalars[i] : tail_scalars[i - n];
                s2_for_digits_at<SEG>(s, i, seg_off, segs, NB1, widths, W, M, fixed_stride, fixed_first, [&](uint32_t b, uint32_t ent) {
                    const uint32_t bin = b >> S2_NF_LOG;
                    const uint32_t pos = toff[bin] + atomicAdd(&hist[bin], 1u);
                    stage[pos] = ((uint64_t)bin << S2_BIN_SHIFT) | ((uint64_t)(b & (S2_NF - 1u)) << 32) | ent;
                });
            }
        }
        __syncthreads();
        const uint32_t total = toff[NC];
        for (uint32_t t = threadIdx.x; t < total; t += blockDim.x) {
            const uint64_t rec = stage[t];
            const uint32_t bin = (uint32_t)(rec >> S2_BIN_SHIFT);
            tmp[gcur[bin] + (t - toff[bin])] = rec & S2_REC_MASK;
        }
        __syncthreads();
        for (uint32_t t = threadIdx.x; t < NC; t += blockDim.x) gcur[t] += hist[t];
        __syncthreads();
    }
}

// chunk -> (bin, entry range): binary search in the chunk directory
__device__ __forceinline__ void s2_chunk_range(uint32_t chunk, const uint32_t* __restrict__ chunk_pre, const uint32_t* __restrict__ coarse_off,
                                               uint32_t NC, uint32_t& bin, uint32_t& lo, uint32_t& hi) {
    uint32_t a = 0, b = NC;  // largest bin with chunk_pre[bin] <= chunk
    while (b - a > 1) {
        const uint32_t m = (a + b) >> 1;
        if (chunk_pre[m] <= chunk) a = m; else b = m;
    }
    bin = a;
    lo = coarse_off[a] + (chunk - chunk_pre[a]) * S2_CHUNK;
    const uint32_t end = coarse_off[a + 1];
    hi = lo + S2_CHUNK < end ? lo + S2_CHUNK : end;
}

__global__ void __launch_bounds__(S2_THREADS) k_sort_fine_count(const uint64_t* __restrict__ tmp, const uint32_t* __restrict__ chunk_pre,
                                                                const uint32_t* __restrict__ coarse_off, uint32_t NC,
                                                                uint32_t* __restrict__ fine) {
    __shared__ uint32_t hist[S2_NF];
    __shared__ uint32_t sh[3];
    const uint32_t nchunks = chunk_pre[NC];
    for (uint32_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        if (threadIdx.x == 0) s2_chunk_range(chunk, chunk_pre, coarse_off, NC, sh[0], sh[1], sh[2]);
        for (uint32_t t = threadIdx.x; t < S2_NF; t += blockDim.x) hist[t] = 0;
        __syncthreads();
        const uint32_t lo = sh[1], hi = sh[2];
        for (uint32_t q = lo + threadIdx.x; q < hi; q += blockDim.x) atomicAdd(&hist[(uint32_t)(tmp[q] >> 32)], 1u);
        __syncthreads();
        for (uint32_t t = threadIdx.x; t < S2_NF; t += blockDim.x) fine[(size_t)chunk * S2_NF + t] = hist[t];
        __syncthreads();
    }
}
// per bucket: total over the chunks of its bin
__global__ void __launch_bounds__(256) k_sort_fine_total(const uint32_t* __restrict__ fine, const uint32_t* __restrict__ chunk_pre, uint32_t NB,
                                                         uint32_t* __restrict__ counts) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= NB) return;
    const uint32_t bin = b >> S2_NF_LOG, f = b & (S2_NF - 1u);
    uint32_t acc = 0;
    for (uint32_t c = chunk_pre[bin], c1 = chunk_pre[bin + 1]; c < c1; c++) acc += fine[(size_t)c * S2_NF + f];
    counts[b] = acc;
}
// per bucket: fine[chunk][bucket] <- first slot of the chunk's entries inside the bucket.  Loads go in batches of 8 ahead of
// the stores (read and written array are the same, so the compiler would otherwise serialise one global round trip per chunk).
__global__ void __launch_bounds__(256) k_sort_fine_base(uint32_t* __restrict__ fine, const uint32_t* __restrict__ chunk_pre, uint32_t NB,
                                                        const uint32_t* __restrict__ offsets) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= NB) return;
    const uint32_t bin = b >> S2_NF_LOG, f = b & (S2_NF - 1u);
    uint32_t base = offsets[b];
    const uint32_t c1 = chunk_pre[bin + 1];
    for (uint32_t c = chunk_pre[bin]; c < c1; c += 8) {
        uint32_t v[8];
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = c + j < c1 ? fine[(size_t)(c + j) * S2_NF + f] : 0;
#pragma unroll
        for (int j = 0; j < 8; j++)
            if (c + j < c1) {
                fine[(size_t)(c + j) * S2_NF + f] = base;
                base += v[j];
            }
    }
}

// D: per chunk the records are placed into shared memory IN BUCKET ORDER and written out in that order, so the (on average 8)
// entries a bucket receives from a chunk leave as one or two transactions instead of eight.
__global__ void __launch_bounds__(S2_THREADS) k_sort_fine_scatter(const uint64_t* __restrict__ tmp, const uint32_t* __restrict__ chunk_pre,
                                                                  const uint32_t* __restrict__ coarse_off, uint32_t NC,
                                                                  const uint32_t* __restrict__ fine, uint32_t* __restrict__ entries) {
    extern __shared__ __align__(16) unsigned char s2_smem[];  // stage[S2_CHUNK] (8 B) | hist[NF] | coff[NF + 1] | base[NF]
    uint64_t* stage = reinterpret_cast<uint64_t*>(s2_smem);
    uint32_t* hist = reinterpret_cast<uint32_t*>(stage + S2_CHUNK);
    uint32_t* coff = hist + S2_NF;
    uint32_t* base = coff + S2_NF + 1;
    __shared__ uint32_t sh[3];
    constexpr int PER = S2_CHUNK / S2_THREADS;  // 16
    const uint32_t nchunks = chunk_pre[NC];
    for (uint32_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        if (threadIdx.x == 0) s2_chunk_range(chunk, chunk_pre, coarse_off, NC, sh[0], sh[1], sh[2]);
        for (uint32_t t = threadIdx.x; t < S2_NF; t += blockDim.x) {
            hist[t] = 0;
            base[t] = fine[(size_t)chunk * S2_NF + t];
        }
        __syncthreads();
        const uint32_t lo = sh[1], hi = sh[2];
        uint64_t v[PER];
#pragma unroll
        for (int j = 0; j < PER; j++) {
            const uint32_t q = lo + (uint32_t)j * S2_THREADS + threadIdx.x;
            v[j] = 0;
            if (q < hi) {
                v[j] = tmp[q];
                atomicAdd(&hist[(uint32_t)(v[j] >> 32)], 1u);
            }
        }
        __syncthreads();
        s2_block_scan(hist, S2_NF, coff);
        __syncthreads();
        for (uint32_t t = threadIdx.x; t < S2_NF; t += blockDim.x) hist[t] = 0;
        __syncthreads();
#pragma unroll
        for (int j = 0; j < PER; j++) {
            const uint32_t q = lo + (uint32_t)j * S2_THREADS + threadIdx.x;
            if (q < hi) {
                const uint32_t f = (uint32_t)(v[j] >> 32);
                stage[coff[f] + atomicAdd(&hist[f], 1u)] = v[j];
            }
        }
        __syncthreads();
        const uint32_t total = hi - lo;
        for (uint32_t t = threadIdx.x; t < total; t += blockDim.x) {
            const uint64_t rec = stage[t];
            const uint32_t f = (uint32_t)(rec >> 32);
            entries[base[f] + (t - coff[f])] = (uint32_t)rec;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// 4. bucket accumulation: one thread per bucket, accumulator in registers
// ------------------------------------------------------------------------------------------------
// Lanes do not own a fixed bucket: a lane that has drained its bucket stores it and claims the next unprocessed one
// (one warp-aggregated atomicAdd per claim round), so every lane of a warp stays busy until the work runs out.  With
// a static thread-per-bucket mapping the warp waits for its fullest bucket: bucket loads are Poisson, which costs
// 10 % at 416 entries per bucket and 21 % at 96 (c = 22).
#endif  // HALO_MSM_SMALL_TU
// Entry / base fetch of the accumulation kernels.  Indirect: entries[e] = (index | sign << 31) into bases (or the tail).
// DIRECT (after the pair-tree passes, msm_pairs.cu): slot e itself holds an affine partial sum, infinity is marked by
// x = 2^256 - 1 and is mapped to the (0, 0) encoding xyzz_madd skips.
template <bool DIRECT>
__device__ __forceinline__ uint32_t acc_entry(const uint32_t* __restrict__ entries, uint32_t e) {
    return DIRECT ? e : entries[e];
}
template <bool DIRECT>
__device__ __forceinline__ affine_t acc_base(const affine_t* __restrict__ bases, uint32_t n, const affine_t* __restrict__ tail_bases,
                                             uint32_t ent) {
    if (DIRECT) {  // slot arrays are SoA: x[0 .. n) | y[0 .. n), n = capacity of the last pair-tree pass
        const fq_t* xs = reinterpret_cast<const fq_t*>(bases);
        affine_t p;
        p.x = xs[ent];
        p.y = xs[(size_t)n + ent];
        if (p.x.v[7] == 0xffffffffu) affine_set_inf(p);
        return p;
    }
    const uint32_t idx = ent & 0x7fffffffu;
    return idx < n ? bases[idx] : tail_bases[idx - n];
}

#ifndef HALO_MSM_SMALL_TU
#ifndef HALO_ACC_MIN_BLOCKS
#define HALO_ACC_MIN_BLOCKS 4
#endif
template <bool DIRECT>
__global__ void __launch_bounds__(128, HALO_ACC_MIN_BLOCKS) k_accumulate(const affine_t* __restrict__ bases, uint32_t n,
                                                                         const affine_t* __restrict__ tail_bases,
                                                                         const uint32_t* __restrict__ offsets,
                                                                         const uint32_t* __restrict__ entries, uint32_t NB,
                                                                         xyzz_t* __restrict__ buckets,
                                                                         uint32_t* __restrict__ next_bucket, uint32_t split_len) {
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    uint32_t b = 0xffffffffu;  // no bucket yet
    uint32_t e = 0, end = 0;
    bool exhausted = false;
    xyzz_t acc;
    xyzz_set_inf(acc);
    uint32_t ent1 = 0, ent2 = 0;
    affine_t p1;
    affine_set_inf(p1);
    while (true) {
        const bool need = !exhausted && e == end;
        if (need && b < 0xfffffffeu) buckets[b] = acc;
        const unsigned want = __ballot_sync(0xffffffffu, need);
        if (want) {
            uint32_t base = 0;
            const int leader = __ffs(want) - 1;
            if ((int)lane == leader) base = atomicAdd(next_bucket, (uint32_t)__popc(want));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (need) {
                b = base + (uint32_t)__popc(want & lt_mask);
                if (b < NB) {
                    e = offsets[b];
                    end = offsets[b + 1];
                    xyzz_set_inf(acc);
                    if (end - e > split_len) {  // oversized bucket: handled by k_accumulate_split, never stored here
                        b = 0xfffffffeu;
                        end = e;
                    }
                    // refill the software pipeline (entry two ahead, base one ahead)
                    if (e < end) {
                        ent1 = acc_entry<DIRECT>(entries, e);
                        if (e + 1 < end) ent2 = acc_entry<DIRECT>(entries, e + 1);
                        p1 = acc_base<DIRECT>(bases, n, tail_bases, ent1);
                    }
                } else {
                    b = 0xffffffffu;
                    e = end = 0;
                    exhausted = true;
                }
            }
        }
        if (__all_sync(0xffffffffu, exhausted)) break;
        if (e < end) {
            const uint32_t ent0 = ent1;
            const affine_t p0 = p1;
            ent1 = ent2;
            if (e + 2 < end) ent2 = acc_entry<DIRECT>(entries, e + 2);
            if (e + 1 < end) p1 = acc_base<DIRECT>(bases, n, tail_bases, ent1);
            xyzz_madd(acc, p0, !DIRECT && (ent0 >> 31) != 0);
            e++;
        }
    }
}

// Static mapping (one thread per bucket) kept for A/B measurements: halo_set_tuning(ctx, "acc_static", 1).
template <bool DIRECT>
__global__ void __launch_bounds__(128, HALO_ACC_MIN_BLOCKS) k_accumulate_static(const affine_t* __restrict__ bases, uint32_t n,
                                                                                const affine_t* __restrict__ tail_bases,
                                                                                const uint32_t* __restrict__ offsets,
                                                                                const uint32_t* __restrict__ entries, uint32_t NB,
                                                                                xyzz_t* __restrict__ buckets, uint32_t split_len) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= NB) return;
    uint32_t beg = offsets[b], end = offsets[b + 1];
    if (end - beg > split_len) return;  // oversized bucket: k_accumulate_split
    xyzz_t acc;
    xyzz_set_inf(acc);
    // software pipeline: the entry two steps ahead and the base one step ahead are in flight during each mixed add
    uint32_t ent1 = beg < end ? acc_entry<DIRECT>(entries, beg) : 0;
    uint32_t ent2 = beg + 1 < end ? acc_entry<DIRECT>(entries, beg + 1) : 0;
    affine_t p1;
    if (beg < end) p1 = acc_base<DIRECT>(bases, n, tail_bases, ent1);
    for (uint32_t e = beg; e < end; e++) {
        const uint32_t ent0 = ent1;
        const affine_t p0 = p1;
        ent1 = ent2;
        if (e + 2 < end) ent2 = acc_entry<DIRECT>(entries, e + 2);
        if (e + 1 < end) p1 = acc_base<DIRECT>(bases, n, tail_bases, ent1);
        xyzz_madd(acc, p0, !DIRECT && (ent0 >> 31) != 0);
    }
    buckets[b] = acc;
}

#endif  // HALO_MSM_SMALL_TU

// Four lanes per bucket (small MSMs).  With one lane per bucket a small MSM's accumulation lasts as long as its LONGEST
// bucket: fills are Poisson, so at a mean of 8-16 entries some bucket has ~35 and the kernel takes 35 dependent mixed additions
// (3.6 us each) while the average lane is done after 8 (ncu, 2^13 points: SMs active 56 % of the kernel, 18.5 of 32 lanes active
// per instruction).  Here lane k of a quad adds the entries k, k + 4, .. of the bucket and the four partial sums are merged by
// two shuffle steps (two full additions): chains of ~9 + 2 instead of ~35.  Used while four lanes per bucket fit about one wave
// of the machine (<= 2^15 buckets, no pair-tree passes); oversized buckets go to the split kernels as before.
__device__ __forceinline__ void xyzz_shfl_xor(xyzz_t& dst, const xyzz_t& src, int mask) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
        dst.x.v[i] = __shfl_xor_sync(0xffffffffu, src.x.v[i], mask);
        dst.y.v[i] = __shfl_xor_sync(0xffffffffu, src.y.v[i], mask);
        dst.zz.v[i] = __shfl_xor_sync(0xffffffffu, src.zz.v[i], mask);
        dst.zzz.v[i] = __shfl_xor_sync(0xffffffffu, src.zzz.v[i], mask);
    }
}
static __device__ __noinline__ void xyzz_add_nl(xyzz_t& acc, const xyzz_t& q);
#ifdef HALO_MSM_SMALL_TU
// L = 4 or 2 lanes per bucket; MINB CTAs of 128 threads per SM (4: 128 registers; 6: 80 registers -- enough resident lanes to
// run 2^16 points' 24 576 buckets x 4 lanes in ONE wave instead of 1.3, measured slower: see the launch site)
template <int L, int MINB>
__global__ void __launch_bounds__(128, MINB) k_accumulate_quad(const affine_t* __restrict__ bases, uint32_t n,
                                                               const affine_t* __restrict__ tail_bases,
                                                               const uint32_t* __restrict__ offsets,
                                                               const uint32_t* __restrict__ entries, uint32_t NB,
                                                               xyzz_t* __restrict__ buckets, uint32_t split_len) {
    static_assert(L == 2 || L == 4, "lanes per bucket");
    const uint32_t gt = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t b = gt / L, k = gt % L;
    uint32_t beg = 0, end = 0;
    if (b < NB) {
        beg = offsets[b];
        end = offsets[b + 1];
        if (end - beg > split_len) end = beg;  // oversized bucket: k_accumulate_split
    }
    xyzz_t acc;
    xyzz_set_inf(acc);
    // software pipeline as in k_accumulate_static, stride L
    uint32_t e = beg + k;
    uint32_t ent1 = e < end ? entries[e] : 0, ent2 = e + L < end ? entries[e + L] : 0;
    affine_t p1;
    affine_set_inf(p1);
    if (e < end) p1 = acc_base<false>(bases, n, tail_bases, ent1);
    for (; e < end; e += L) {
        const uint32_t ent0 = ent1;
        const affine_t p0 = p1;
        ent1 = ent2;
        if (e + 2 * L < end) ent2 = entries[e + 2 * L];
        if (e + L < end) p1 = acc_base<false>(bases, n, tail_bases, ent1);
        xyzz_madd(acc, p0, (ent0 >> 31) != 0);
    }
    // merge the lanes of a bucket: every lane of the warp takes part in the shuffles
    xyzz_t other;
    xyzz_shfl_xor(other, acc, 1);
    xyzz_add_nl(acc, other);
    if (L == 4) {
        xyzz_shfl_xor(other, acc, 2);
        xyzz_add_nl(acc, other);
    }
    if (b < NB && k == 0 && !(offsets[b + 1] - offsets[b] > split_len)) buckets[b] = acc;
}

#endif  // HALO_MSM_SMALL_TU
static __device__ __noinline__ void xyzz_add_nl(xyzz_t& acc, const xyzz_t& q) { xyzz_add(acc, q); }
static __device__ __noinline__ void xyzz_dbl_nl(xyzz_t& acc) { xyzz_dbl(acc, acc); }

#ifndef HALO_MSM_SMALL_TU
// ------------------------------------------------------------------------------------------------
// 4b. oversized buckets.  Uniform scalars fill buckets evenly, but legal inputs can pile everything into a few buckets
//     (all scalars equal, tiny scalars, a constant polynomial): one lane would then add millions of points serially.
//     Buckets deeper than split_len are cut into chunks of split_len entries ("split tasks"), accumulated by lane-level
//     claiming like ordinary buckets, and merged by one warp per bucket.  Costs three near-empty launches when no bucket
//     is oversized.
// ------------------------------------------------------------------------------------------------
struct SplitTask {
    uint32_t beg, end;  // entry range
};
struct SplitBucket {
    uint32_t bucket, first_task, n_tasks;
};
// ctrl[0] = number of split tasks, ctrl[1] = number of split buckets, ctrl[2] = claim counter
__global__ void __launch_bounds__(256) k_split_plan(const uint32_t* __restrict__ offsets, uint32_t NB, uint32_t split_len,
                                                    uint32_t max_tasks, uint32_t max_buckets, uint32_t* __restrict__ ctrl,
                                                    SplitTask* __restrict__ tasks, SplitBucket* __restrict__ sbuckets) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= NB) return;
    uint32_t beg = offsets[b], end = offsets[b + 1];
    uint32_t cnt = end - beg;
    if (cnt <= split_len) return;
    uint32_t nt = (cnt + split_len - 1) / split_len;
    uint32_t first = atomicAdd(&ctrl[0], nt);
    uint32_t slot = atomicAdd(&ctrl[1], 1u);
    if (first + nt > max_tasks || slot >= max_buckets) {
        ctrl[3] = 1;  // capacity exceeded (cannot happen: capacities are sized from the entry count), flagged for the host
        return;
    }
    sbuckets[slot] = SplitBucket{b, first, nt};
    for (uint32_t t = 0; t < nt; t++) {
        uint32_t tb = beg + t * split_len;
        uint32_t te = tb + split_len < end ? tb + split_len : end;
        tasks[first + t] = SplitTask{tb, te};
    }
}

template <bool DIRECT>
__global__ void __launch_bounds__(128, HALO_ACC_MIN_BLOCKS) k_accumulate_split(const affine_t* __restrict__ bases, uint32_t n,
                                                                               const affine_t* __restrict__ tail_bases,
                                                                               const uint32_t* __restrict__ entries,
                                                                               const SplitTask* __restrict__ tasks,
                                                                               uint32_t* __restrict__ ctrl,
                                                                               xyzz_t* __restrict__ partials) {
    const uint32_t NT = ctrl[0];
    if (NT == 0) return;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    uint32_t t = 0xffffffffu, e = 0, end = 0;
    bool exhausted = false;
    xyzz_t acc;
    xyzz_set_inf(acc);
    while (true) {
        const bool need = !exhausted && e == end;
        if (need && t != 0xffffffffu) partials[t] = acc;
        const unsigned want = __ballot_sync(0xffffffffu, need);
        if (want) {
            uint32_t base = 0;
            const int leader = __ffs(want) - 1;
            if ((int)lane == leader) base = atomicAdd(&ctrl[2], (uint32_t)__popc(want));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (need) {
                t = base + (uint32_t)__popc(want & lt_mask);
                if (t < NT) {
                    SplitTask tk = tasks[t];
                    e = tk.beg;
                    end = tk.end;
                    xyzz_set_inf(acc);
                } else {
                    t = 0xffffffffu;
                    e = end = 0;
                    exhausted = true;
                }
            }
        }
        if (__all_sync(0xffffffffu, exhausted)) break;
        if (e < end) {
            uint32_t ent = acc_entry<DIRECT>(entries, e);
            affine_t p = acc_base<DIRECT>(bases, n, tail_bases, ent);
            xyzz_madd(acc, p, !DIRECT && (ent >> 31) != 0);
            e++;
        }
    }
}

// one warp per oversized bucket: lanes stride over the bucket's partial sums, then a shuffle tree
__device__ __forceinline__ void xyzz_shfl_down(xyzz_t& dst, const xyzz_t& src, int delta) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
        dst.x.v[i] = __shfl_down_sync(0xffffffffu, src.x.v[i], delta);
        dst.y.v[i] = __shfl_down_sync(0xffffffffu, src.y.v[i], delta);
        dst.zz.v[i] = __shfl_down_sync(0xffffffffu, src.zz.v[i], delta);
        dst.zzz.v[i] = __shfl_down_sync(0xffffffffu, src.zzz.v[i], delta);
    }
}
__global__ void __launch_bounds__(128) k_merge_split(const SplitBucket* __restrict__ sbuckets, const uint32_t* __restrict__ ctrl,
                                                     const xyzz_t* __restrict__ partials, xyzz_t* __restrict__ buckets) {
    const uint32_t NS = ctrl[1];
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t s = warp; s < NS; s += nwarps) {
        SplitBucket sb = sbuckets[s];
        xyzz_t acc;
        xyzz_set_inf(acc);
        for (uint32_t t = lane; t < sb.n_tasks; t += 32) {
            xyzz_t q = partials[sb.first_task + t];
            xyzz_add_nl(acc, q);
        }
        for (int delta = 16; delta >= 1; delta >>= 1) {
            xyzz_t other;
            xyzz_shfl_down(other, acc, delta);
            xyzz_add_nl(acc, other);
        }
        if (lane == 0) buckets[sb.bucket] = acc;
    }
}

// ------------------------------------------------------------------------------------------------
// 5. bucket reduction.  For a slab of T * s items Q_t (s = 2^log_s per thread) a CTA of T threads produces
//      A = sum_t (t + 1) Q_t ,   R = sum_t Q_t ,   E = sum_t X_t  (plain sum of a second array, optional)
//    by per-thread running sums, a block-wide suffix scan of the per-thread totals and tree sums.
//    Level 1: grid (slabs, windows) over the buckets -> (A_g, R_g) per slab g.
//    Level 2 (slabs > 1): one CTA per window over Q = R_g, X = A_g -> (A2, R2, E).
//    Window sum  S = sum_k (k+1) B_k = sum_g A_g + slab * sum_g g R_g = E + slab * (A2 - R2)      [host, msm_finish_host]
// ------------------------------------------------------------------------------------------------

constexpr int REDUCE_THREADS = 256;

__device__ __forceinline__ void block_tree_sum(xyzz_t& v, xyzz_t* sm, int T) {
    const int j = threadIdx.x;
    sm[j] = v;
    __syncthreads();
    for (int stride = T >> 1; stride >= 1; stride >>= 1) {
        if (j < stride) {
            xyzz_t other = sm[j + stride];
            xyzz_add_nl(v, other);
            sm[j] = v;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(REDUCE_THREADS) k_reduce_slabs(const xyzz_t* __restrict__ in, const xyzz_t* __restrict__ extra,
                                                                 size_t in_stride, int T, int log_s,
                                                                 xyzz_t* __restrict__ outA, xyzz_t* __restrict__ outR,
                                                                 xyzz_t* __restrict__ outE, int out_stride) {
    __shared__ xyzz_t sm[REDUCE_THREADS];
    const int j = threadIdx.x;
    const uint32_t s = 1u << log_s;
    const size_t base = (size_t)blockIdx.y * in_stride + (((size_t)blockIdx.x * T + j) << log_s);
    const xyzz_t* Q = in + base;
    // running sums from the top: R = sum Q_t, A = sum (t + 1) Q_t over this thread's s items
    xyzz_t R, A;
    xyzz_set_inf(R);
    xyzz_set_inf(A);
    for (int t = (int)s - 1; t >= 0; t--) {
        xyzz_t q = Q[t];
        xyzz_add_nl(R, q);
        xyzz_add_nl(A, R);
    }
    // inclusive suffix scan of R over the CTA: Suf_j = sum_{i >= j} R_i
    xyzz_t Suf = R;
    sm[j] = Suf;
    __syncthreads();
    for (int stride = 1; stride < T; stride <<= 1) {
        bool has = j + stride < T;
        xyzz_t other;
        if (has) other = sm[j + stride];
        __syncthreads();
        if (has) xyzz_add_nl(Suf, other);
        sm[j] = Suf;
        __syncthreads();
    }
    xyzz_t total = sm[0];  // sum of all R_j
    __syncthreads();
    // sum_{j >= 1} Suf_j = sum_j j R_j: thread j's items carry the extra weight j * s
    if (j == 0) xyzz_set_inf(Suf);
    block_tree_sum(Suf, sm, T);
    if (j == 0)
        for (int t = 0; t < log_s; t++) xyzz_dbl_nl(Suf);
    block_tree_sum(A, sm, T);
    const size_t o = ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * out_stride;
    if (j == 0) {
        xyzz_add_nl(A, Suf);
        outA[o] = A;
        outR[o] = total;
    }
    if (extra) {
        xyzz_t e;
        xyzz_set_inf(e);
        for (uint32_t t = 0; t < s; t++) {
            xyzz_t q = extra[base + t];
            xyzz_add_nl(e, q);
        }
        block_tree_sum(e, sm, T);
        if (j == 0) outE[o] = e;
    }
}

#endif  // HALO_MSM_SMALL_TU

constexpr int RQ_MAX_T = 128;  // logical threads (quads) per CTA of k_reduce_slabs_quad: 512 physical threads
#ifdef HALO_MSM_SMALL_TU
// ------------------------------------------------------------------------------------------------
// 5b. the same reduction with QUAD-COOPERATIVE point additions (the default; "reduce_quad" = 0 selects the kernel above).
//     The reduction is a chain of ~30-70 dependent point additions per CTA with almost nothing to run beside it: its cost
//     is latency, 14 dependent multiplications of ~0.3 us per addition.  Here one point lives in four adjacent lanes (lane
//     k holds coordinate k of (X, Y, ZZ, ZZZ)) and the 12M + 2S of add-2008-s are issued as FOUR levels of one
//     multiplication per lane, operands and results moving between the lanes of the quad by shuffles:
//        level 1   U1 = X1 ZZ2 | S1 = Y1 ZZZ2 | U2 = X2 ZZ1 | S2 = Y2 ZZZ1          (operand: xor-2 shuffle of point 2)
//                  P = U2 - U1 on lanes 0, 2;  R = S2 - S1 on lanes 1, 3            (xor-2 shuffle of the products)
//        level 2   PP = P^2   | RR = R^2     | ZZ1 ZZ2     | ZZZ1 ZZZ2
//        level 3   PPP = P PP |     -        | Q = U1 PP   |     -                  (PP broadcast from lane 0)
//        level 4   ZZZ3 = ZZZ1 ZZZ2 PPP | V = R (Q - X3), X3 = RR - PPP - 2Q | ZZ3 = ZZ1 ZZ2 PP | T = S1 PPP
//                  X3 -> lane 0, Y3 = V - T on lane 1, ZZ3 on lane 2, ZZZ3 -> lane 3
//     Infinity operands are resolved by selects; equal or opposite operands (P = 0) fall back to the one-lane routine on
//     a replicated copy -- rare (crafted inputs), exact.  Every lane of a warp must call quad_add (full-mask shuffles).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ fq_t fq_shfl(const fq_t& v, int src) {
    fq_t r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = __shfl_sync(0xffffffffu, v.v[i], src);
    return r;
}
__device__ __forceinline__ fq_t fq_shfl_xor(const fq_t& v, int m) {
    fq_t r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = __shfl_xor_sync(0xffffffffu, v.v[i], m);
    return r;
}
__device__ __forceinline__ fq_t fq_sel(bool c, const fq_t& a, const fq_t& b) {
    fq_t r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = c ? a.v[i] : b.v[i];
    return r;
}
__device__ __forceinline__ fq_t xyzz_coord(const xyzz_t& p, unsigned k) {
    return k == 0 ? p.x : k == 1 ? p.y : k == 2 ? p.zz : p.zzz;
}
static __device__ __noinline__ fq_t quad_add(fq_t acc, fq_t q) {
    const unsigned FULL = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31u, k = lane & 3u, qb = lane & ~3u;
    // infinity <=> ZZ == 0: the flag lives on lane 2 of the quad
    const unsigned za = __ballot_sync(FULL, fp_is_zero(acc)), zq = __ballot_sync(FULL, fp_is_zero(q));
    const bool acc_inf = (za >> (qb + 2)) & 1u, q_inf = (zq >> (qb + 2)) & 1u;
    fq_t t = fq_shfl_xor(q, 2);  // ZZ2 | ZZZ2 | X2 | Y2
    fq_t m1;
    fp_mul(m1, acc, t);          // U1 | S1 | U2 | S2
    fq_t o1 = fq_shfl_xor(m1, 2);  // U2 | S2 | U1 | S1
    fq_t d;
    {
        const fq_t hi = fq_sel(k < 2, o1, m1), lo = fq_sel(k < 2, m1, o1);
        fp_sub(d, hi, lo);       // P | R | P | R
    }
    const unsigned zd = __ballot_sync(FULL, fp_is_zero(d));
    const bool p_zero = (zd >> qb) & 1u;
    fq_t m2;
    {
        const fq_t a2 = fq_sel(k < 2, d, acc), b2 = fq_sel(k < 2, d, q);
        fp_mul(m2, a2, b2);      // PP | RR | ZZ1 ZZ2 | ZZZ1 ZZZ2
    }
    const fq_t PPb = fq_shfl(m2, (int)qb);
    fq_t m3;
    {
        const fq_t a3 = fq_sel(k == 2, o1, d);
        fp_mul(m3, a3, PPb);     // PPP | (unused) | Q | (unused)
    }
    const fq_t PPPb = fq_shfl(m3, (int)qb), Qb = fq_shfl(m3, (int)qb + 2);
    const fq_t zzz12 = fq_shfl(m2, (int)qb + 3);  // used by lane 0
    fq_t x3, w;
    fp_sub(x3, m2, PPPb);  // meaningful on lane 1 (m2 = RR)
    fp_sub(x3, x3, Qb);
    fp_sub(x3, x3, Qb);
    fp_sub(w, Qb, x3);
    fq_t m4;
    {
        const fq_t a4 = k == 0 ? zzz12 : k == 1 ? d : k == 2 ? m2 : o1;
        const fq_t b4 = k == 0 ? PPPb : k == 1 ? w : k == 2 ? PPb : PPPb;
        fp_mul(m4, a4, b4);      // ZZZ3 | V | ZZ3 | T
    }
    const fq_t e = fq_sel(k == 1, x3, m4);
    const int src = (int)qb + (k == 0 ? 1 : k == 1 ? 3 : k == 2 ? 2 : 0);
    const fq_t g = fq_shfl(e, src);  // X3 | T | ZZ3 | ZZZ3
    fq_t res;
    fp_sub(res, m4, g);              // lane 1: Y3 = V - T
    res = fq_sel(k == 1, res, g);
    res = fq_sel(q_inf, acc, fq_sel(acc_inf, q, res));
    const bool special = p_zero && !acc_inf && !q_inf;  // doubling or cancellation
    if (__any_sync(FULL, special)) {
        xyzz_t A, B;
        A.x = fq_shfl(acc, (int)qb), A.y = fq_shfl(acc, (int)qb + 1), A.zz = fq_shfl(acc, (int)qb + 2), A.zzz = fq_shfl(acc, (int)qb + 3);
        B.x = fq_shfl(q, (int)qb), B.y = fq_shfl(q, (int)qb + 1), B.zz = fq_shfl(q, (int)qb + 2), B.zzz = fq_shfl(q, (int)qb + 3);
        if (special) {
            xyzz_add_nl(A, B);
            res = xyzz_coord(A, k);
        }
    }
    return res;
}

// Same contract as k_reduce_slabs; blockDim.x = max(32, 4 * T), logical thread j = threadIdx.x / 4.
__global__ void __launch_bounds__(4 * RQ_MAX_T) k_reduce_slabs_quad(const xyzz_t* __restrict__ in, const xyzz_t* __restrict__ extra,
                                                                    size_t in_stride, int T, int log_s, xyzz_t* __restrict__ outA,
                                                                    xyzz_t* __restrict__ outR, xyzz_t* __restrict__ outE, int out_stride) {
    __shared__ xyzz_t smA[RQ_MAX_T], smB[RQ_MAX_T];
    fq_t* cA = reinterpret_cast<fq_t*>(smA);  // coordinate k of logical thread j: c[4 j + k]
    fq_t* cB = reinterpret_cast<fq_t*>(smB);
    const int j = (int)(threadIdx.x >> 2);
    const unsigned k = threadIdx.x & 3u;
    const bool act = j < T;
    const uint32_t s = 1u << log_s;
    const size_t base = (size_t)blockIdx.y * in_stride + (((size_t)blockIdx.x * T + (act ? j : 0)) << log_s);
    const fq_t* Q = reinterpret_cast<const fq_t*>(in + base);
    fq_t zero;
    fp_zero(zero);
    // running sums from the top: R = sum Q_t, A = sum (t + 1) Q_t over this logical thread's s items
    fq_t R = zero, A = zero;
    for (int t = (int)s - 1; t >= 0; t--) {
        const fq_t q = act ? Q[4 * t + k] : zero;
        R = quad_add(R, q);
        A = quad_add(A, R);
    }
    // inclusive suffix scan of R over the CTA: Suf_j = sum_{i >= j} R_i
    fq_t Suf = R;
    if (act) cA[4 * j + k] = Suf;
    __syncthreads();
    for (int stride = 1; stride < T; stride <<= 1) {
        const bool has = act && j + stride < T;
        const fq_t other = has ? cA[4 * (j + stride) + k] : zero;
        __syncthreads();
        if (__any_sync(0xffffffffu, has)) Suf = quad_add(Suf, other);  // warps with nothing to add skip the call (warp uniform)
        if (act) cA[4 * j + k] = Suf;
        __syncthreads();
    }
    const fq_t total = cA[k];  // logical thread 0: sum of all R_j
    __syncthreads();
    // two tree sums at once, in disjoint halves of the CTA: F = sum_{j >= 1} Suf_j (= sum_j j R_j) and sum_j A_j
    if (act) {
        cA[4 * j + k] = j == 0 ? zero : Suf;
        cB[4 * j + k] = A;
    }
    __syncthreads();
    if (T >= 2) {
        const int half = T >> 1;
        const int tree = j >= half ? 1 : 0, jj = j & (half - 1);
        fq_t* c = tree ? cB : cA;
        for (int stride = half; stride >= 1; stride >>= 1) {
            const bool on = act && jj < stride;
            const fq_t x = on ? c[4 * jj + k] : zero, y = on ? c[4 * (jj + stride) + k] : zero;
            fq_t r = zero;
            if (__any_sync(0xffffffffu, on)) r = quad_add(x, y);
            __syncthreads();
            if (on) c[4 * jj + k] = r;
            __syncthreads();
        }
    }
    const size_t o = ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * out_stride;
    fq_t* oR = reinterpret_cast<fq_t*>(outR + o);
    if (j == 0) oR[k] = total;
    if (threadIdx.x == 0) {  // slab result A = sum_j A_j + 2^log_s F: a handful of one-lane operations
        xyzz_t F = smA[0], S = smB[0];
        for (int t = 0; t < log_s; t++) xyzz_dbl_nl(F);
        xyzz_add_nl(S, F);
        outA[o] = S;
    }
    if (extra) {  // plain sum of a second array (level 2: the slabs' A partials)
        __syncthreads();
        const fq_t* X = reinterpret_cast<const fq_t*>(extra + base);
        fq_t e = zero;
        for (uint32_t t = 0; t < s; t++) {
            const fq_t q = act ? X[4 * t + k] : zero;
            e = quad_add(e, q);
        }
        if (act) cA[4 * j + k] = e;
        __syncthreads();
        for (int stride = T >> 1; stride >= 1; stride >>= 1) {
            const bool on = act && j < stride;
            const fq_t x = on ? cA[4 * j + k] : zero, y = on ? cA[4 * (j + stride) + k] : zero;
            fq_t r = zero;
            if (__any_sync(0xffffffffu, on)) r = quad_add(x, y);
            __syncthreads();
            if (on) cA[4 * j + k] = r;
            __syncthreads();
        }
        fq_t* oE = reinterpret_cast<fq_t*>(outE + o);
        if (j == 0) oE[k] = cA[k];
    }
}

// Launchers of this unit's kernels (declared in msm.cuh, called by msm_enqueue in the normal unit).
void launch_accumulate_quad(cudaStream_t st, int lanes, int minb, const affine_t* bases, uint32_t n, const affine_t* tail_bases,
                            const uint32_t* offsets, const uint32_t* entries, uint32_t NB, xyzz_t* buckets, uint32_t split_len) {
    const unsigned qgrid = (unsigned)(((uint64_t)NB * lanes + 127) / 128);
#define HALO_ACCQ(LL, MB) k_accumulate_quad<LL, MB><<<qgrid, 128, 0, st>>>(bases, n, tail_bases, offsets, entries, NB, buckets, split_len)
    if (lanes == 4 && minb == 4) HALO_ACCQ(4, 4);
    else if (lanes == 4) HALO_ACCQ(4, 6);
    else if (minb == 4) HALO_ACCQ(2, 4);
    else HALO_ACCQ(2, 6);
#undef HALO_ACCQ
}
void launch_reduce_slabs_quad(cudaStream_t st, dim3 grid, int T, int log_s, const xyzz_t* in, const xyzz_t* extra, size_t in_stride,
                              xyzz_t* outA, xyzz_t* outR, xyzz_t* outE, int out_stride) {
    k_reduce_slabs_quad<<<grid, 4 * T < 32 ? 32 : 4 * T, 0, st>>>(in, extra, in_stride, T, log_s, outA, outR, outE, out_stride);
}
#endif  // HALO_MSM_SMALL_TU

#ifndef HALO_MSM_SMALL_TU
// ------------------------------------------------------------------------------------------------
// fixed-base tables: table[w * n + i] = 2^(off_w) * G_i (affine), w = 0 .. W-1, off_w = sum of the lower window widths
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_precompute(const affine_t* __restrict__ gens, uint32_t n, const MsmWidths widths, int W,
                                                    affine_t* __restrict__ table) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    affine_t g = gens[i];
    table[i] = g;
    xyzz_t p;
    xyzz_from_affine(p, g);
    for (int w = 1; w < W; w++) {
        const int c = widths.w[w - 1];
        for (int k = 0; k < c; k++) xyzz_dbl_nl(p);
        affine_t a;
        xyzz_to_affine(a, p);
        table[(size_t)w * n + i] = a;
        xyzz_from_affine(p, a);
    }
}

void msm_precompute_tables(halo_ctx* ctx, int force_c) {
    if (ctx->n_gens == 0) throw CudaError{cudaErrorInvalidValue, "precompute: no generators", __FILE__, __LINE__};
    MsmPlan plan = msm_make_fixed_plan(ctx->n_gens, force_c);
    uint32_t n = (uint32_t)ctx->n_gens;
    ctx->gens_pre.reserve((size_t)plan.W * n * sizeof(affine_t));
    k_precompute<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->gens.as<affine_t>(), n, plan.widths, plan.W,
                                                          ctx->gens_pre.as<affine_t>());
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
    HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->pre_plan = plan;
    ctx->pre_n = n;
}

// ------------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------------
// Device part of one MSM.  d_out receives 3 points per window (one "window" in FIXED mode): [E, A2, R2] with
// window sum S = E + slab * (A2 - R2); a single-slab plan writes S into E and leaves A2 = R2 = infinity.
void msm_enqueue(halo_ctx* ctx, const MsmInput& in, const MsmPlan& plan, xyzz_t* d_out, int lane, const SortAhead* ahead) {
    const uint32_t n = in.n;
    const uint32_t ntot = in.n + in.n_tail;
    // lane 0: the context's stream and workspace.  lane 1: a second stream and workspace, so two latency-bound MSMs of
    // one IPA round (L and R) overlap instead of queueing behind each other.
    MsmWorkspace& ws = lane ? ctx->ws2 : ctx->ws;
    cudaStream_t st = lane ? ctx->stream2 : ctx->stream;
    // SortAhead (pipelined submit): the counting sort runs on its own high-priority stream with its own buffers and a
    // throttled grid, so it proceeds beside the accumulation kernels of the previous MSM (the sort is bound by L2 atomics
    // and leaves the integer pipe idle; the accumulation is the opposite); the accumulation below waits for it.
    MsmWorkspace& sws = ahead ? *ahead->ws : ws;
    cudaStream_t sst = ahead ? ahead->stream : st;
    const uint32_t NB = plan.NB;
    // a segmented MSM is one MSM over segs bucket sets: from the sort on, windows of all segments are handled alike
    const bool seg = in.segs > 1;
    if (in.segs != plan.segs || (seg && (in.n_tail || !in.seg_off)))
        throw CudaError{cudaErrorInvalidValue, "segmented MSM: plan / input mismatch", __FILE__, __LINE__};
    const uint32_t NB1 = NB / plan.segs;
    const int nwin = (plan.fixed ? 1 : plan.W) * (int)plan.segs;
    const uint64_t total_entries_max = (uint64_t)ntot * plan.W;
    // pair-tree passes (msm_pairs.cu): worthwhile once the per-pass fixed costs (7 launches and one ~0.1 ms inversion
    // latency) are small against the additions saved; bucket segments are then padded to multiples of 2^P slots
    int P = 0;
    if (ctx->tune_pair_passes >= 0) {
        P = ctx->tune_pair_passes;
    } else if (total_entries_max >= ((uint64_t)1 << 21)) {
        // measured per size and mode (profiles/r02_pair_passes_sweep.jsonl; round 1: profiles/r01_pair_tree_sweep.jsonl): what
        // decides is the mean bucket fill -- every pass halves it at 6.2 instead of 10 multiplications per addition but costs
        // ~0.1 ms of hierarchy latency and pads every bucket to a multiple of 2^P slots.
        //   FIXED 2^18 .. 2^24: fill 14 / 28 / 56 / 112 / 224 / 416 -> best P = 2 / 2 / 3 / 3 / 4 / 4;  variable 2^19 .. 2^22: 16 / 32 / 64 / 128 -> 2 / 2 / 3 / 4
        const uint64_t fill = total_entries_max / NB;
        P = fill < 12 ? 0 : fill < 48 ? 2 : fill < 120 ? 3 : 4;
    }
    if (P > 8) P = 8;
    const uint32_t rmask = (1u << P) - 1u;
    uint64_t slots_max = total_entries_max + (uint64_t)rmask * NB;
    slots_max = (slots_max + rmask) & ~(uint64_t)rmask;
    if (slots_max >= 0xfffffff0ull) throw CudaError{cudaErrorInvalidValue, "MSM too large for 32-bit slot indices", __FILE__, __LINE__};
    sws.counts.reserve((size_t)(NB + 1) * 4);
    sws.offsets.reserve((size_t)(NB + 1) * 4);
    sws.entries.reserve((size_t)slots_max * 4);
    ws.buckets.reserve((size_t)NB * sizeof(xyzz_t));
    sws.scan_tmp.reserve(4096 * 4);
    ws.task_partial.reserve((size_t)(2 * plan.red_slabs + 3) * nwin * sizeof(xyzz_t));
    if ((NB + SCAN_TILE - 1) / SCAN_TILE > 2048) throw CudaError{cudaErrorInvalidValue, "bucket count too large for scan", __FILE__, __LINE__};
    if (plan.red_slabs > (uint32_t)(plan.red_quad ? RQ_MAX_T : REDUCE_THREADS) * 64) throw CudaError{cudaErrorInvalidValue, "too many reduction slabs", __FILE__, __LINE__};

    uint32_t* counts = sws.counts.as<uint32_t>();
    uint32_t* offsets = sws.offsets.as<uint32_t>();
    uint32_t* entries = sws.entries.as<uint32_t>();
    xyzz_t* buckets = ws.buckets.as<xyzz_t>();
    const bool prof = ctx->profile && lane == 0;
    auto mark = [&](int i) {
        if (prof) HALO_CUDA(cudaEventRecord(ctx->ev[i], st));
    };
    const uint32_t fstride = plan.fixed ? in.fixed_stride : 0;

    mark(0);
    HALO_CUDA(cudaMemsetAsync(counts, 0, (size_t)(NB + 1) * 4, sst));
    const int TPB = 256;
    uint32_t grid = (ntot + TPB - 1) / TPB;
    uint32_t cap = 0;
    if (ahead && ahead->ctas_per_sm > 0) {
        cap = (uint32_t)ctx->sm_count * (uint32_t)ahead->ctas_per_sm;
        if (grid > cap) grid = cap;
    }
    // two-level sort (shared-memory atomics) for large inputs whose geometry fits; else the one-pass counting sort
    const uint32_t NC = (NB + S2_NF - 1) / S2_NF;
    const bool sort2 = ctx->tune_sort2 != 0 && total_entries_max >= ((uint64_t)1 << ctx->tune_sort2_min_lg) && plan.W <= S2_MAX_W &&
                       plan.M >= S2_NF && NC <= S2_MAX_NC;
    if (sort2) {
        const uint32_t max_chunks = (uint32_t)(total_entries_max / S2_CHUNK) + NC + 1;
        uint32_t g1 = (ntot + S2_TILE - 1) / S2_TILE, g2 = max_chunks;
        const uint32_t full1 = (uint32_t)ctx->sm_count * 2u, full2 = (uint32_t)ctx->sm_count * 4u;  // persistent grids
        if (g1 > full1) g1 = full1;
        if (g1 > S2_MAX_CTAS) g1 = S2_MAX_CTAS;
        if (g2 > full2) g2 = full2;
        if (cap) {
            if (g1 > cap) g1 = cap;
            if (g2 > cap) g2 = cap;
        }
        sws.sort_tmp.reserve((size_t)total_entries_max * 8);
        sws.sort_fine.reserve((size_t)max_chunks * S2_NF * 4);
        sws.sort_coarse.reserve(((size_t)S2_MAX_CTAS * S2_MAX_NC + 2 * (S2_MAX_NC + 1)) * 4);
        uint32_t* cta_hist = sws.sort_coarse.as<uint32_t>();
        uint32_t* coarse_off = cta_hist + (size_t)S2_MAX_CTAS * S2_MAX_NC;
        uint32_t* chunk_pre = coarse_off + (S2_MAX_NC + 1);
        uint64_t* tmp = sws.sort_tmp.as<uint64_t>();
        uint32_t* fine = sws.sort_fine.as<uint32_t>();
        if (seg)
            k_sort_coarse_count<true><<<g1, S2_THREADS, 0, sst>>>(in.scalars, n, in.tail_scalars, in.n_tail, plan.widths, plan.W, plan.M, fstride,
                                                                   in.fixed_first, NC, cta_hist, in.seg_off, in.segs, NB1);
        else
            k_sort_coarse_count<false><<<g1, S2_THREADS, 0, sst>>>(in.scalars, n, in.tail_scalars, in.n_tail, plan.widths, plan.W, plan.M, fstride,
                                                                    in.fixed_first, NC, cta_hist, nullptr, 1, NB1);
        k_sort_coarse_scan<<<1, 1024, 0, sst>>>(cta_hist, g1, NC, coarse_off, chunk_pre);
        const size_t smem_b = (((size_t)(3 * NC + 1) * 4 + 15) & ~(size_t)15) + (size_t)S2_TILE * plan.W * 8;
        const size_t smem_d = (size_t)S2_CHUNK * 8 + (size_t)(3 * S2_NF + 1) * 4;
        if (!ctx->sort2_attr) {  // per device: opt in to more than 48 KiB of dynamic shared memory
            HALO_CUDA(cudaFuncSetAttribute(k_sort_coarse_scatter<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            HALO_CUDA(cudaFuncSetAttribute(k_sort_coarse_scatter<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            HALO_CUDA(cudaFuncSetAttribute(k_sort_fine_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
            ctx->sort2_attr = true;
        }
        if (seg)
            k_sort_coarse_scatter<true><<<g1, S2_THREADS, smem_b, sst>>>(in.scalars, n, in.tail_scalars, in.n_tail, plan.widths, plan.W, plan.M,
                                                                          fstride, in.fixed_first, NC, cta_hist, tmp, in.seg_off, in.segs, NB1);
        else
            k_sort_coarse_scatter<false><<<g1, S2_THREADS, smem_b, sst>>>(in.scalars, n, in.tail_scalars, in.n_tail, plan.widths, plan.W, plan.M,
                                                                           fstride, in.fixed_first, NC, cta_hist, tmp, nullptr, 1, NB1);
        mark(1);
        k_sort_fine_count<<<g2, S2_THREADS, 0, sst>>>(tmp, chunk_pre, coarse_off, NC, fine);
        k_sort_fine_total<<<(NB + 255) / 256, 256, 0, sst>>>(fine, chunk_pre, NB, counts);
        exclusive_scan(counts, offsets, NB, rmask, sws.scan_tmp.as<uint32_t>(), sst, &ctx->kernel_launches);
        if (P) {
            k_fill_pads<<<(NB + 255) / 256, 256, 0, sst>>>(counts, offsets, NB, entries);
            ctx->kernel_launches++;
        }
        HALO_CUDA(cudaMemsetAsync(counts + NB, 0, 4, sst));  // the claim counter of k_accumulate
        k_sort_fine_base<<<(NB + 255) / 256, 256, 0, sst>>>(fine, chunk_pre, NB, offsets);
        mark(2);
        k_sort_fine_scatter<<<g2, S2_THREADS, smem_d, sst>>>(tmp, chunk_pre, coarse_off, NC, fine, entries);
        ctx->kernel_launches += 7;
    } else {
    if (seg)
        k_digits<false, true><<<grid, TPB, 0, sst>>>(in.scalars, n, in.tail_scalars, in.n_tail, plan.widths, plan.W, plan.M, fstride,
                                                     in.fixed_first, counts, nullptr, in.seg_off, in.segs, NB1);
    else
        k_digits<false, false><<<grid, TPB, 0, sst>>>(in.scalars, n, in.tail_scalars, in.n_tail, plan.widths, plan.W, plan.M, fstride,
                                                      in.fixed_first, counts, nullptr, nullptr, 1, NB1);
    mark(1);
    exclusive_scan(counts, offsets, NB, rmask, sws.scan_tmp.as<uint32_t>(), sst, &ctx->kernel_launches);
    if (P) {  // pad slots of every bucket segment stand for the point at infinity
        k_fill_pads<<<(NB + 255) / 256, 256, 0, sst>>>(counts, offsets, NB, entries);
        ctx->kernel_launches++;
    }
    // the histogram array becomes the write cursor of every bucket; its spare slot [NB] the claim counter of k_accumulate
    HALO_CUDA(cudaMemcpyAsync(counts, offsets, (size_t)NB * 4, cudaMemcpyDeviceToDevice, sst));
    HALO_CUDA(cudaMemsetAsync(counts + NB, 0, 4, sst));
    mark(2);
    if (seg)
        k_digits<true, true><<<grid, TPB, 0, sst>>>(in.scalars, n, in.tail_scalars, in.n_tail, plan.widths, plan.W, plan.M, fstride,
                                                    in.fixed_first, counts, entries, in.seg_off, in.segs, NB1);
    else
        k_digits<true, false><<<grid, TPB, 0, sst>>>(in.scalars, n, in.tail_scalars, in.n_tail, plan.widths, plan.W, plan.M, fstride,
                                                     in.fixed_first, counts, entries, nullptr, 1, NB1);
    ctx->kernel_launches += 2;
    }
    if (ahead) {
        HALO_CUDA(cudaEventRecord(ahead->sorted, sst));
        HALO_CUDA(cudaStreamWaitEvent(st, ahead->sorted, 0));
    }
    mark(3);
    // P > 0: the first P levels of every bucket's sum as flat pairwise affine additions (msm_pairs.cu); the XYZZ kernels
    // below then see bucket b as the slots [offsets[b] >> P, offsets[b + 1] >> P) of the returned array.
    const affine_t* acc_bases = in.bases;
    const uint32_t* acc_offsets = offsets;
    uint32_t acc_n = plan.fixed ? 0x7fffffffu : n;
    uint64_t acc_entries_max = total_entries_max;
    if (P) {
        acc_bases = pair_tree_enqueue(ctx, ws, st, in, entries, offsets + NB, slots_max, P);
        ws.cursor.reserve((size_t)(NB + 1) * 4);
        k_shift_offsets<<<(NB + 1 + 255) / 256, 256, 0, st>>>(offsets, NB + 1, P, ws.cursor.as<uint32_t>());
        ctx->kernel_launches++;
        acc_offsets = ws.cursor.as<uint32_t>();
        acc_n = (uint32_t)(slots_max >> P);  // DIRECT mode: the y array starts this many elements behind the x array
        acc_entries_max = slots_max >> P;
    }
    // oversized-bucket threshold: 4x the mean fill, at least 1024 entries (uniform scalars never reach it)
    uint32_t split_len = (uint32_t)(4 * (acc_entries_max / NB + 1));
    if (split_len < 1024) split_len = 1024;
    const uint32_t max_split_tasks = (uint32_t)(acc_entries_max / split_len + 1) * 2 + 16;  // sum ceil(cnt/L) <= E/L + #split
    const uint32_t max_split_buckets = (uint32_t)(acc_entries_max / split_len + 1);
    ws.split_ctrl.reserve(16);
    ws.split_tasks.reserve((size_t)max_split_tasks * sizeof(SplitTask));
    ws.split_buckets.reserve((size_t)max_split_buckets * sizeof(SplitBucket));
    ws.split_partials.reserve((size_t)max_split_tasks * sizeof(xyzz_t));
    uint32_t* split_ctrl = ws.split_ctrl.as<uint32_t>();
    HALO_CUDA(cudaMemsetAsync(split_ctrl, 0, 16, st));
    // thread-per-bucket is ~8 % faster when buckets are deep and evenly filled (variable base, large n); lane-level
    // claiming wins everywhere else (measured: profiles/r01_accumulate_static_vs_dynamic.txt)
    const bool deep = !P && !plan.fixed && (uint64_t)ntot * plan.W >= (uint64_t)NB * 256;
    // measured (profiles/r02_acc_quad_ab.jsonl): 2^8 .. 2^14 points (<= 24 576 buckets) 0.080 -> 0.041, 0.108 -> 0.055, 0.197 -> 0.165,
    // 0.324 -> 0.229 ms; at 2^15 / 2^16 (82 k buckets: 4.3 waves of quads, two extra full additions per bucket) it loses
    const bool quad_lanes = !P && ctx->tune_acc_quad != 0 && NB <= (uint32_t)ctx->tune_acc_quad_max_buckets && ctx->tune_acc_static == 0 && !deep;
    int acc_kind = 0, acc_lanes = 0, acc_minb = 0;  // 2 = k_accumulate_quad, 1 = k_accumulate_static, 0 = k_accumulate
    uint32_t acc_grid = 0;
    if (quad_lanes) {
        // lanes per bucket and CTAs per SM (tunables acc_quad_lanes / acc_quad_blocks; 0 = the policy below)
        int lanes = ctx->tune_acc_quad_lanes, minb = ctx->tune_acc_quad_blocks;
        // measured (profiles/r02_acc_quad_lanes_blocks_ab.jsonl, 2^12 .. 2^16 points): 6 CTAs per SM (80 registers, one wave at
        // 2^16 instead of 1.3) is 4-9 % slower than 4 CTAs (128 registers) at every size, 2 lanes 9-25 % slower than 4: the
        // kernel is bound by issue slots and by the deepest lane of each warp, not by the partial second wave
        if (lanes != 2 && lanes != 4) lanes = 4;
        if (minb != 4 && minb != 6) minb = 4;
        launch_accumulate_quad(st, lanes, minb, acc_bases, acc_n, in.tail_bases, acc_offsets, entries, NB, buckets, split_len);
        acc_kind = 2, acc_lanes = lanes, acc_minb = minb;
    } else if (ctx->tune_acc_static == 1 || (ctx->tune_acc_static == 0 && deep)) {
        acc_kind = 1;
        if (P)
            k_accumulate_static<true><<<(NB + 127) / 128, 128, 0, st>>>(acc_bases, acc_n, in.tail_bases, acc_offsets, entries, NB,
                                                                       buckets, split_len);
        else
            k_accumulate_static<false><<<(NB + 127) / 128, 128, 0, st>>>(acc_bases, acc_n, in.tail_bases, acc_offsets, entries, NB,
                                                                        buckets, split_len);
    } else {
        // persistent lanes: enough CTAs to fill the machine, capped by the amount of work
        uint32_t want_blocks = (NB + 127) / 128;
        uint32_t max_blocks = (uint32_t)ctx->sm_count * (ctx->tune_acc_blocks_per_sm ? ctx->tune_acc_blocks_per_sm : HALO_ACC_MIN_BLOCKS);
        uint32_t blocks = want_blocks < max_blocks ? want_blocks : max_blocks;
        acc_grid = blocks;
        uint32_t* next_bucket = counts + NB;  // spare slot at the end of the counter array (zeroed above)
        if (P)
            k_accumulate<true><<<blocks, 128, 0, st>>>(acc_bases, acc_n, in.tail_bases, acc_offsets, entries, NB, buckets, next_bucket,
                                                       split_len);
        else
            k_accumulate<false><<<blocks, 128, 0, st>>>(acc_bases, acc_n, in.tail_bases, acc_offsets, entries, NB, buckets, next_bucket,
                                                        split_len);
    }
    {
        k_split_plan<<<(NB + 255) / 256, 256, 0, st>>>(acc_offsets, NB, split_len, max_split_tasks, max_split_buckets, split_ctrl,
                                                       ws.split_tasks.as<SplitTask>(), ws.split_buckets.as<SplitBucket>());
        uint32_t sblocks = (uint32_t)ctx->sm_count * HALO_ACC_MIN_BLOCKS;
        uint32_t cap = (max_split_tasks + 127) / 128;
        if (sblocks > cap) sblocks = cap;
        if (P)
            k_accumulate_split<true><<<sblocks, 128, 0, st>>>(acc_bases, acc_n, in.tail_bases, entries, ws.split_tasks.as<SplitTask>(),
                                                              split_ctrl, ws.split_partials.as<xyzz_t>());
        else
            k_accumulate_split<false><<<sblocks, 128, 0, st>>>(acc_bases, acc_n, in.tail_bases, entries, ws.split_tasks.as<SplitTask>(),
                                                               split_ctrl, ws.split_partials.as<xyzz_t>());
        uint32_t mblocks = (max_split_buckets + 3) / 4;
        if (mblocks > (uint32_t)ctx->sm_count * 4) mblocks = (uint32_t)ctx->sm_count * 4;
        k_merge_split<<<mblocks, 128, 0, st>>>(ws.split_buckets.as<SplitBucket>(), split_ctrl, ws.split_partials.as<xyzz_t>(), buckets);
        ctx->kernel_launches += 3;
    }
    mark(4);
    HALO_CUDA(cudaMemsetAsync(d_out, 0, msm_parts(plan) * sizeof(xyzz_t), st));
    const bool quad = plan.red_quad;
    const int maxT = quad ? RQ_MAX_T : REDUCE_THREADS;
    auto reduce = [&](dim3 grid, int T, int log_s, const xyzz_t* src, const xyzz_t* extra, size_t stride, xyzz_t* oA, xyzz_t* oR, xyzz_t* oE,
                      int ostride) {
        if (quad)
            launch_reduce_slabs_quad(st, grid, T, log_s, src, extra, stride, oA, oR, oE, ostride);
        else
            k_reduce_slabs<<<grid, T, 0, st>>>(src, extra, stride, T, log_s, oA, oR, oE, ostride);
    };
    if (plan.red_slabs == 1) {
        // A is the window sum; R goes to scratch (at stride 3)
        reduce(dim3(1, nwin), plan.red_T, plan.red_log_s, buckets, nullptr, plan.M, d_out, ws.task_partial.as<xyzz_t>(), nullptr, 3);
        ctx->kernel_launches += 1;
    } else {
        xyzz_t* slabA = ws.task_partial.as<xyzz_t>();
        xyzz_t* slabR = slabA + (size_t)nwin * plan.red_slabs;
        reduce(dim3(plan.red_slabs, nwin), plan.red_T, plan.red_log_s, buckets, nullptr, plan.M, slabA, slabR, nullptr, 1);
        // the second level is one CTA per window: with few windows its cost is the latency of its dependent chain, which is
        // shortest when every scheduler of the SM runs one warp (32 quads); a full 128-quad CTA queues 4 warps per scheduler
        // and measured 0.17 ms for 128 slabs (profiles/r02_reduce_launches.csv)
        const int maxT2 = quad ? 32 : maxT;
        int T2 = plan.red_slabs < (uint32_t)maxT2 ? (int)plan.red_slabs : maxT2;
        int log_s2 = 0;
        while (((uint32_t)T2 << log_s2) < plan.red_slabs) log_s2++;
        reduce(dim3(1, nwin), T2, log_s2, slabR, slabA, plan.red_slabs, d_out + 1, d_out + 2, d_out, 3);
        ctx->kernel_launches += 2;
    }
    mark(5);
    ctx->kernel_launches += 1;  // the accumulation kernel (the sort counted its own above)
    HALO_CUDA(cudaGetLastError());
    int* route = ctx->msm_route[lane ? 1 : 0];
    route[0] = plan.c;
    route[1] = plan.fixed ? 1 : 0;
    route[2] = P;
    route[3] = P ? (ctx->tune_pair_bwd_async ? 1 : 0) : -1;
    route[4] = acc_kind;
    route[5] = acc_kind == 2 ? acc_lanes : 0;
    route[6] = acc_kind == 2 ? acc_minb : 0;
    route[7] = acc_kind == 0 ? (int)acc_grid : 0;
    route[8] = plan.red_quad ? 1 : 0;
    route[9] = -1;  // msm_batch overwrites it with its lane decision
}

// Host finish: per window S = E + slab * (A2 - R2), then Horner over the windows (a single term in FIXED mode).
void msm_finish_host(const xyzz_t* parts, const MsmPlan& plan, xyzz_t& out) {
    const int nwin = plan.fixed ? 1 : plan.W;
    const int log_slab = plan.red_log_s + (plan.red_T > 1 ? 31 - __builtin_clz((unsigned)plan.red_T) : 0);
    xyzz_t total;
    xyzz_set_inf(total);
    for (int w = nwin - 1; w >= 0; w--) {
        xyzz_t S = parts[3 * w];
        if (plan.red_slabs > 1) {
            xyzz_t d = parts[3 * w + 2];
            if (!xyzz_is_inf(d)) xyzz_neg(d);
            xyzz_add(d, parts[3 * w + 1]);
            for (int k = 0; k < log_slab; k++) xyzz_dbl(d, d);
            xyzz_add(S, d);
        }
        xyzz_add(total, S);
        if (w > 0)
            for (int k = 0; k < plan.widths.w[w - 1]; k++) xyzz_dbl(total, total);
    }
    out = total;
}

void msm_enqueue_to_host(halo_ctx* ctx, const MsmInput& in, const MsmPlan& plan, xyzz_t* d_out, xyzz_t* h_out, int lane,
                         const SortAhead* ahead) {
    msm_enqueue(ctx, in, plan, d_out, lane, ahead);
    HALO_CUDA(cudaMemcpyAsync(h_out, d_out, msm_parts(plan) * sizeof(xyzz_t), cudaMemcpyDeviceToHost, lane ? ctx->stream2 : ctx->stream));
}

void msm_read_timings(halo_ctx* ctx) {
    float t[5];
    for (int i = 0; i < 5; i++) HALO_CUDA(cudaEventElapsedTime(&t[i], ctx->ev[i], ctx->ev[i + 1]));
    ctx->last.digits_ms = t[0];
    ctx->last.scan_ms = t[1];
    ctx->last.scatter_ms = t[2];
    ctx->last.accumulate_ms = t[3];
    ctx->last.reduce_ms = t[4];
    HALO_CUDA(cudaEventElapsedTime(&ctx->last.total_ms, ctx->ev[0], ctx->ev[5]));
}

void host_parallel(size_t k, const std::function<void(size_t)>& f) {
    const size_t hw = std::thread::hardware_concurrency();
    const size_t T = std::min(k, std::max<size_t>(1, std::min<size_t>(hw, 16)));
    std::vector<std::thread> th;
    std::vector<size_t> unspawned;
    auto work = [&](size_t t) {
        for (size_t j = t; j < k; j += T) f(j);
    };
    for (size_t t = 1; t < T; t++) {
        try {
            th.emplace_back(work, t);
        } catch (const std::system_error&) {
            unspawned.push_back(t);  // no thread available: this thread takes that share as well (nothing may unwind across the ABI)
        }
    }
    work(0);
    for (size_t t : unspawned) work(t);
    for (auto& x : th) x.join();
}

// Enqueue `count` MSMs back to back on the context stream (they share the workspace, so they serialise on the
// stream), then one D2H of all partial sums, one synchronisation, and the host finish per MSM.
void msm_batch(halo_ctx* ctx, const MsmInput* ins, int count, xyzz_t* outs, const std::function<void()>* while_running) {
    constexpr int MAXB = 4, SLOT = 3 * MSM_MAX_WINDOWS;
    if (count > MAXB) throw CudaError{cudaErrorInvalidValue, "msm_batch: count > 4", __FILE__, __LINE__};
    MsmPlan plans[MAXB];
    ctx->ws.wsums.reserve((size_t)6 * SLOT * sizeof(xyzz_t));  // 4 batch slots + 2 asynchronous pipeline slots
    xyzz_t* d_parts = ctx->ws.wsums.as<xyzz_t>();
    if (!ctx->pinned) {
        HALO_CUDA(cudaMallocHost(&ctx->pinned, (size_t)MAXB * SLOT * sizeof(xyzz_t)));
        ctx->pinned_cap = (size_t)MAXB * SLOT * sizeof(xyzz_t);
    }
    xyzz_t* h_parts = reinterpret_cast<xyzz_t*>(ctx->pinned);
    bool any = false;
    // two MSMs in a batch that are small enough to be latency bound run on two streams with separate workspaces
    // (a batch of 3 or 4 alternates between the two lanes)
    bool two_lanes = false;
    uint64_t n_sum = 0;
    int n_live = 0;
    for (int k = 0; k < count; k++) {
        n_sum += ins[k].n;
        n_live += ins[k].n + ins[k].n_tail > 0;
    }
    if (count >= 2 && n_live == count && ctx->stream2 && (n_sum <= (1u << 19) || ctx->force_two_lanes) && !ctx->profile) {
        two_lanes = true;
        HALO_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));       // inputs produced on the main stream are complete
        HALO_CUDA(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
    }
    for (int k = 0; k < count; k++) {
        if (ins[k].n + ins[k].n_tail == 0) continue;
        plans[k] = msm_plan(ctx, ins[k].n + ins[k].n_tail, ins[k].fixed_stride != 0);
        const int lane = two_lanes ? (k & 1) : 0;
        msm_enqueue_to_host(ctx, ins[k], plans[k], d_parts + k * SLOT, h_parts + k * SLOT, lane);
        ctx->msm_route[lane][9] = two_lanes ? 1 : 0;
        any = true;
    }
    if (two_lanes) {
        HALO_CUDA(cudaEventRecord(ctx->ev_join, ctx->stream2));
        HALO_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));  // later main-stream work (the fold) is ordered after lane 1
    }
    if (while_running) (*while_running)();  // host work that overlaps the kernels enqueued above
    // A pair of very unequal MSMs on the two lanes (pcdl::check: <G, h> of 2^20 points beside the 2 lg n + 2 point MSM of the
    // succinct check): the small one is done long before the large one, so its ~255 host doublings are finished while the
    // large one still runs instead of after it.
    bool early[MAXB] = {false, false, false, false};
    if (two_lanes && count == 2 && !plans[1].fixed && (uint64_t)ins[1].n * 64 <= ins[0].n) {
        HALO_CUDA(cudaEventSynchronize(ctx->ev_join));  // lane 1's partials are on the host
        msm_finish_host(h_parts + 1 * SLOT, plans[1], outs[1]);
        early[1] = true;
    }
    if (any) HALO_CUDA(cudaStreamSynchronize(ctx->stream));
    if (any && ctx->profile) msm_read_timings(ctx);
    // the Horner combination of a variable-base MSM is ~255 host doublings (~0.1 ms): the two results of an IPA round
    // (L and R) are finished on two host threads
    auto finish = [&](size_t k) {
        if (early[k]) return;
        if (ins[k].n + ins[k].n_tail == 0)
            xyzz_set_inf(outs[k]);
        else
            msm_finish_host(h_parts + k * SLOT, plans[k], outs[k]);
    };
    // (the results of an IPA round, L and R, and the up to four small MSMs of a verifier batch: one host thread each)
    int heavy = 0;
    for (int k = 0; k < count; k++) heavy += ins[k].n + ins[k].n_tail > 0 && !plans[k].fixed;
    if (count >= 2 && heavy == count)
        host_parallel((size_t)count, finish);
    else
        for (int k = 0; k < count; k++) finish(k);
}

void msm_device(halo_ctx* ctx, const affine_t* d_bases, const fr_t* d_scalars, uint64_t n, xyzz_t& out) {
    MsmInput in;
    in.bases = d_bases;
    in.scalars = d_scalars;
    in.n = (uint32_t)n;
    msm_batch(ctx, &in, 1, &out);
}

// sum_i scalars[i] * G_{first+i} over the resident generators; takes the FIXED-base path when tables exist and the
// problem is large enough to amortise the (n-independent) bucket reduction of the wide window.  (pre_n != 0: an MSM of n <=
// n_gens points implies it, but the sharded MSM asks with a slice of n_global, which a rank's resident set need not cover.)
bool gens_use_fixed(const halo_ctx* ctx, uint64_t n) {
    return ctx->use_fixed && ctx->pre_n == ctx->n_gens && ctx->pre_n != 0 && ctx->gens_pre.p && n >= (1u << 17) && n * 8 >= ctx->pre_n;
}

MsmInput gens_msm_input(const halo_ctx* ctx, bool fixed, const fr_t* scalars, uint64_t first, uint64_t n) {
    MsmInput in;
    in.scalars = scalars;
    in.n = (uint32_t)n;
    if (fixed) {
        in.bases = ctx->gens_pre.as<affine_t>();
        in.fixed_stride = (uint32_t)ctx->pre_n;
        in.fixed_first = (uint32_t)first;
    } else {
        in.bases = ctx->gens.as<affine_t>() + first;
    }
    return in;
}

void msm_gens_device(halo_ctx* ctx, const fr_t* d_scalars, uint64_t first, uint64_t n, xyzz_t& out) {
    const MsmInput in = gens_msm_input(ctx, gens_use_fixed(ctx, n), d_scalars, first, n);
    msm_batch(ctx, &in, 1, &out);
}

#endif  // HALO_MSM_SMALL_TU
}  // namespace halo
