// ntt.cuh -- internal interface of ntt.cu (K8: batched number-theoretic transforms over the scalar field).
#pragma once
#include "common.cuh"
namespace halo {
constexpr uint32_t NTT_MAX_LG = 32;   // the 2-adicity of both scalar fields
constexpr uint32_t NTT_TILE_LG = 11;  // largest sub-transform of one pass: 2^11 scalars (64 KiB of shared memory)
// omega_{2^lg} = 5^((r - 1) / 2^lg) in Montgomery form, lg <= 32
fr_t ntt_root(uint32_t lg);
// Number of passes over HBM of a transform of 2^lg scalars: ceil(lg / 11), at least one
uint32_t ntt_passes(uint32_t lg);
// The buffer that ntt_run's first pass reads when its input is staged: the pass writes the other one of (a, b), so a staged
// input goes here.  (One pass with n_in = n may also read and write a in place.)
bool ntt_stage_in_a(uint32_t lg);
// Builds the twiddle tables of 2^lg (once per size and context) and the coset / scale table of this call; false when the device
// has no memory for them (nothing else is touched)
bool ntt_prepare(halo_ctx* ctx, uint32_t lg, bool inverse, const fr_t* shift);
// k transforms of 2^lg scalars on the context stream; the result lands in a.  src holds k vectors of n_in scalars (n_in < 2^lg:
// forward only, the missing coefficients are zero) and is b, or a when ntt_stage_in_a(lg) (or one pass with n_in = 2^lg).
// b holds k * 2^lg scalars when there is more than one pass.  ntt_prepare must have been called with the same lg, inverse
// and shift.
void ntt_run(halo_ctx* ctx, const fr_t* src, uint64_t n_in, fr_t* a, fr_t* b, uint64_t k, uint32_t lg, bool inverse, bool shifted);
// d_deg[j] = DensePolynomial::degree of vector j of k vectors of n scalars (one launch; d_deg is zeroed first)
void ntt_degrees(halo_ctx* ctx, const fr_t* d, uint64_t k, uint64_t n, uint64_t* d_deg);
}  // namespace halo
