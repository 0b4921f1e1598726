// ntt.cu -- K8: batched number-theoretic transforms over the scalar field (DESIGN.md K8).
//
// A transform of n = 2^lg scalars runs as ceil(lg / 11) Stockham passes over HBM.  Pass p takes a radix R = 2^lr with
// sum lr = lg; with Ns = the product of the radices before it, group j < n / R of a vector
//   loads v_r = x[j + r n / R] * omega_{Ns R}^(r (j mod Ns)),  r < R       (the twiddle of the previous passes)
//   computes the R-point DFT of v in shared memory (bit-reversed placement, lr radix-2 stages)
//   stores V_r to y[(j / Ns) Ns R + (j mod Ns) + r Ns]
// so input and output are in natural order and no pass reorders data on its own.  A block holds 2^11 scalars (64 KiB): 2^(11 - lr)
// adjacent groups, which are adjacent vectors when R = n.  The grid covers every group of all k vectors, so the number of
// launches does not depend on k.  The coset powers g^j of a forward transform are applied as the first pass loads, the factors
// g^-j n^-1 of an inverse one as the last pass stores.
//
// Tables (built on the device by k_ntt_pows, kept in the context): omega_{2^11}^x for the stages inside a block, and per size a
// two-level table of omega_n: omega_n^e = lo[e mod 2^B] * hi[e >> B], B = ceil(lg / 2) -- at 2^24 2 x 4096 entries (256 KiB)
// instead of 2^24 (512 MiB).  The coset / scale factors of one call use the same two-level split.  An inverse transform reads
// the same tables at the negated exponent.
#include "ntt.cuh"

namespace halo {

constexpr uint32_t NTT_THREADS = 256;
constexpr uint32_t NTT_TILE = 1u << NTT_TILE_LG;

// ---- host: roots and plans -------------------------------------------------------------------------------------------
fr_t ntt_root(uint32_t lg) {
    // t = (r - 1) / 2^32: the modulus' 32-bit limbs shifted down by one limb (its low limb is 1)
    const uint32_t t[8] = {ScalarParams::P1, ScalarParams::P2, ScalarParams::P3, 0, 0, 0, 0x40000000u, 0};
    fr_t base, w;
    fp_from_u32(base, 5);
    fp_one(w);
    for (int i = 255; i >= 0; i--) {
        fp_sqr(w, w);
        if ((t[i >> 5] >> (i & 31)) & 1u) fp_mul(w, w, base);
    }
    for (uint32_t i = lg; i < NTT_MAX_LG; i++) fp_sqr(w, w);  // omega_{2^lg} = omega_{2^32}^(2^(32 - lg))
    return w;
}

uint32_t ntt_passes(uint32_t lg) { return lg <= NTT_TILE_LG ? 1 : (lg + NTT_TILE_LG - 1) / NTT_TILE_LG; }
bool ntt_stage_in_a(uint32_t lg) { return ntt_passes(lg) % 2 == 0; }

static uint32_t pass_lg(uint32_t lg, uint32_t p) {  // radices as equal as possible, the larger ones first
    const uint32_t P = ntt_passes(lg);
    return lg / P + (p < lg % P ? 1 : 0);
}
static uint32_t split_lg(uint32_t lg) { return (lg + 1) / 2; }  // B of the two-level tables

static fr_t fr_pow2k(fr_t x, uint32_t k) {  // x^(2^k)
    for (uint32_t i = 0; i < k; i++) fp_sqr(x, x);
    return x;
}
static fr_t fr_inv_two_pow(uint32_t k) {  // 2^-k
    fr_t x;
    fp_one(x);
    for (uint32_t i = 0; i < k; i++) fp_add(x, x, x);
    fp_inv(x, x);
    return x;
}

// ---- kernels --------------------------------------------------------------------------------------------------------
// out[i] = lo_base^i (i < lo_n), out[lo_n + i] = hi_scale * hi_base^i (i < hi_n); exponents below 2^17
__global__ void __launch_bounds__(NTT_THREADS) k_ntt_pows(fr_t lo_base, uint32_t lo_n, fr_t hi_base, fr_t hi_scale, uint32_t hi_n,
                                                          fr_t* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= lo_n + hi_n) return;
    const bool hi = i >= lo_n;
    uint32_t e = hi ? i - lo_n : i;
    fr_t b = hi ? hi_base : lo_base, acc;
    if (hi)
        acc = hi_scale;
    else
        fp_one(acc);
#pragma unroll 1
    for (; e; e >>= 1) {
        if (e & 1) fp_mul(acc, acc, b);
        fp_sqr(b, b);
    }
    out[i] = acc;
}

struct NttPass {
    const fr_t* in;
    fr_t* out;
    const fr_t* tw;     // two-level table of omega_n: 2^tw_b entries, then the high part
    const fr_t* dit;    // omega_{2^11}^x
    const fr_t* scale;  // two-level table of the coset / scale factors (same split), or NULL
    fr_t c;             // the constant factor of an inverse transform without a shift (n^-1)
    uint64_t groups;    // k n / R
    uint64_t in_stride, n_in;  // input vector stride and its valid prefix (first pass), n otherwise
    uint32_t lg_n, lr, lg_ns, lg_g, tw_b;
    uint32_t inverse;
    uint32_t pre;   // 1: multiply the loads by scale[index]
    uint32_t post;  // 1: multiply the stores by c; 2: by scale[index]
};

__device__ __forceinline__ fr_t ntt_two_level(const fr_t* __restrict__ t, uint32_t b, uint64_t e) {
    fr_t r;
    fp_mul(r, t[e & ((1ull << b) - 1)], t[(1ull << b) + (e >> b)]);
    return r;
}

__global__ void __launch_bounds__(NTT_THREADS) k_ntt_pass(NttPass p) {
    extern __shared__ uint4 ntt_smem[];
    fr_t* s = reinterpret_cast<fr_t*>(ntt_smem);
    const uint32_t lr = p.lr, lg = p.lg_g, tile = 1u << (lr + lg);
    const uint64_t n = 1ull << p.lg_n, g0 = (uint64_t)blockIdx.x << lg;
    const uint32_t lg_gpv = p.lg_n - lr;  // log2 of the groups of one vector
    const uint64_t gpv_mask = (1ull << lg_gpv) - 1, ns_mask = (1ull << p.lg_ns) - 1;
    // loads: consecutive threads read consecutive groups, or consecutive r when a group is a whole vector
    const bool load_r_fast = lg_gpv == 0;
    for (uint32_t f = threadIdx.x; f < tile; f += NTT_THREADS) {
        const uint32_t gi = load_r_fast ? f >> lr : f & ((1u << lg) - 1), r = load_r_fast ? f & ((1u << lr) - 1) : f >> lg;
        const uint64_t gam = g0 + gi;
        if (gam >= p.groups) continue;
        const uint64_t b = gam >> lg_gpv, j = gam & gpv_mask, idx = j + ((uint64_t)r << lg_gpv);
        fr_t v;
        if (idx < p.n_in)
            v = p.in[b * p.in_stride + idx];
        else
            fp_zero(v);
        if (p.pre) fp_mul(v, v, ntt_two_level(p.scale, p.tw_b, idx));
        if (p.lg_ns) {  // omega_{Ns R}^(r k) = omega_n^(r k n / (Ns R))
            uint64_t e = ((uint64_t)r * (j & ns_mask)) << (p.lg_n - p.lg_ns - lr);
            if (p.inverse) e = (n - e) & (n - 1);
            if (e) fp_mul(v, v, ntt_two_level(p.tw, p.tw_b, e));
        }
        s[(gi << lr) + (lr ? __brev(r) >> (32 - lr) : 0)] = v;
    }
    __syncthreads();
    // radix-2 DIT stages on bit-reversed data: natural order out
#pragma unroll 1
    for (uint32_t st = 0; st < lr; st++) {
        const uint32_t m = 1u << st;
#pragma unroll 1
        for (uint32_t bf = threadIdx.x; bf < tile / 2; bf += NTT_THREADS) {
            const uint32_t gi = bf >> (lr - 1), bb = bf & ((1u << (lr - 1)) - 1);
            const uint32_t jj = bb & (m - 1), i = ((bb >> st) << (st + 1)) + jj;
            uint32_t e = jj << (NTT_TILE_LG - 1 - st);
            if (p.inverse) e = (NTT_TILE - e) & (NTT_TILE - 1);
            fr_t* x = s + (gi << lr);
            fr_t u = x[i], t = x[i + m];
            fp_mul(t, t, p.dit[e]);
            fr_t a, d;
            fp_add(a, u, t);
            fp_sub(d, u, t);
            x[i] = a;
            x[i + m] = d;
        }
        __syncthreads();
    }
    // stores: consecutive threads write consecutive r when Ns = 1 (y[j R + r]), consecutive groups otherwise
    const bool store_r_fast = p.lg_ns == 0;
    for (uint32_t f = threadIdx.x; f < tile; f += NTT_THREADS) {
        const uint32_t gi = store_r_fast ? f >> lr : f & ((1u << lg) - 1), r = store_r_fast ? f & ((1u << lr) - 1) : f >> lg;
        const uint64_t gam = g0 + gi;
        if (gam >= p.groups) continue;
        const uint64_t b = gam >> lg_gpv, j = gam & gpv_mask;
        const uint64_t idx = ((j >> p.lg_ns) << (p.lg_ns + lr)) + (j & ns_mask) + ((uint64_t)r << p.lg_ns);
        fr_t v = s[(gi << lr) + r];
        if (p.post == 1) fp_mul(v, v, p.c);
        if (p.post == 2) fp_mul(v, v, ntt_two_level(p.scale, p.tw_b, idx));
        p.out[b * n + idx] = v;
    }
}

// d_deg[b] = max(1 + index of a non-zero scalar) over chunks of NTT_DEG_CHUNK scalars of vector b; one atomic per block
constexpr uint32_t NTT_DEG_CHUNK = 8192;
__global__ void __launch_bounds__(NTT_THREADS) k_ntt_degree(const fr_t* __restrict__ d, uint64_t n, uint64_t bpv,
                                                            unsigned long long* __restrict__ deg) {
    __shared__ unsigned long long red[NTT_THREADS / 32];
    const uint64_t b = blockIdx.x / bpv, lo = (blockIdx.x % bpv) * NTT_DEG_CHUNK;
    const uint64_t hi = lo + NTT_DEG_CHUNK < n ? lo + NTT_DEG_CHUNK : n;
    unsigned long long best = 0;
    for (uint64_t i = lo + threadIdx.x; i < hi; i += NTT_THREADS)
        if (!fp_is_zero(d[b * n + i])) best = i + 1;  // i grows: the last hit is this thread's highest
    for (int o = 16; o; o >>= 1) {
        const unsigned long long x = __shfl_down_sync(0xffffffffu, best, o);
        best = x > best ? x : best;
    }
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (uint32_t w = 1; w < NTT_THREADS / 32; w++) best = red[w] > best ? red[w] : best;
        if (best) atomicMax(deg + b, best);
    }
}

// ---- host: tables, passes -----------------------------------------------------------------------------------------
static bool reserve_ok(DevBuf& b, size_t bytes) {
    try {
        b.reserve(bytes);
        return true;
    } catch (const CudaError& e) {
        if (e.err != cudaErrorMemoryAllocation) throw;
        cudaGetLastError();
        return false;
    }
}

static void launch_pows(halo_ctx* ctx, const fr_t& lo_base, uint32_t lo_n, const fr_t& hi_base, const fr_t& hi_scale, uint32_t hi_n,
                        fr_t* out) {
    const uint32_t total = lo_n + hi_n;
    k_ntt_pows<<<(total + NTT_THREADS - 1) / NTT_THREADS, NTT_THREADS, 0, ctx->stream>>>(lo_base, lo_n, hi_base, hi_scale, hi_n, out);
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
}

bool ntt_prepare(halo_ctx* ctx, uint32_t lg, bool inverse, const fr_t* shift) {
    const uint32_t B = split_lg(lg), lo_n = 1u << B, hi_n = 1u << (lg - B);
    fr_t one;
    fp_one(one);
    if (!ctx->ntt_dit.p) {
        if (!reserve_ok(ctx->ntt_dit, NTT_TILE * sizeof(fr_t))) return false;
        launch_pows(ctx, ntt_root(NTT_TILE_LG), NTT_TILE, one, one, 0, ctx->ntt_dit.as<fr_t>());
    }
    DevBuf& tw = ctx->ntt_tw[lg];
    if (!tw.p) {
        if (!reserve_ok(tw, (size_t)(lo_n + hi_n) * sizeof(fr_t))) return false;
        const fr_t w = ntt_root(lg);
        launch_pows(ctx, w, lo_n, fr_pow2k(w, B), one, hi_n, tw.as<fr_t>());
    }
    if (!shift) return true;
    // forward: g^i; inverse: n^-1 g^-i, split as lo[i mod 2^B] * hi[i >> B]
    if (!reserve_ok(ctx->ntt_scale, (size_t)(lo_n + hi_n) * sizeof(fr_t))) return false;
    fr_t g = *shift, c = one;
    if (inverse) {
        fp_inv(g, g);
        c = fr_inv_two_pow(lg);
    }
    launch_pows(ctx, g, lo_n, fr_pow2k(g, B), c, hi_n, ctx->ntt_scale.as<fr_t>());
    return true;
}

void ntt_run(halo_ctx* ctx, const fr_t* src, uint64_t n_in, fr_t* a, fr_t* b, uint64_t k, uint32_t lg, bool inverse, bool shifted) {
    if (k == 0) return;
    if (!ctx->ntt_attr) {
        HALO_CUDA(cudaFuncSetAttribute(k_ntt_pass, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(NTT_TILE * sizeof(fr_t))));
        ctx->ntt_attr = true;
    }
    const uint32_t P = ntt_passes(lg);
    const uint64_t n = 1ull << lg;
    const fr_t ninv = fr_inv_two_pow(lg);
    const fr_t* in = src;
    uint32_t lg_ns = 0;
    for (uint32_t q = 0; q < P; q++) {
        NttPass p{};
        const uint32_t lr = pass_lg(lg, q);
        p.in = in;
        p.out = (P - 1 - q) % 2 == 0 ? a : b;
        p.tw = ctx->ntt_tw[lg].as<fr_t>();
        p.dit = ctx->ntt_dit.as<fr_t>();
        p.scale = shifted ? ctx->ntt_scale.as<fr_t>() : nullptr;
        p.c = ninv;
        p.groups = k << (lg - lr);
        p.in_stride = q == 0 ? n_in : n;
        p.n_in = q == 0 ? n_in : n;
        p.lg_n = lg;
        p.lr = lr;
        p.lg_ns = lg_ns;
        p.lg_g = NTT_TILE_LG - lr;
        p.tw_b = split_lg(lg);
        p.inverse = inverse;
        p.pre = q == 0 && !inverse && shifted;
        p.post = q + 1 == P && inverse ? (shifted ? 2 : 1) : 0;
        const uint64_t blocks = (p.groups + (1ull << p.lg_g) - 1) >> p.lg_g;
        k_ntt_pass<<<(unsigned)blocks, NTT_THREADS, NTT_TILE * sizeof(fr_t), ctx->stream>>>(p);
        ctx->kernel_launches++;
        HALO_CUDA(cudaGetLastError());
        in = p.out;
        lg_ns += lr;
    }
}

void ntt_degrees(halo_ctx* ctx, const fr_t* d, uint64_t k, uint64_t n, uint64_t* d_deg) {
    HALO_CUDA(cudaMemsetAsync(d_deg, 0, k * sizeof(uint64_t), ctx->stream));
    if (k == 0 || n == 0) return;
    const uint64_t bpv = (n + NTT_DEG_CHUNK - 1) / NTT_DEG_CHUNK;
    k_ntt_degree<<<(unsigned)(k * bpv), NTT_THREADS, 0, ctx->stream>>>(d, n, bpv, reinterpret_cast<unsigned long long*>(d_deg));
    ctx->kernel_launches++;
    HALO_CUDA(cudaGetLastError());
}

}  // namespace halo
