// vec.cuh -- internal interface of vec.cu (Fr vector kernels and the expansion of sums of h(X)).
#pragma once
#include "common.cuh"
namespace halo {
constexpr uint32_t VEC_DOT_MAX_BLOCKS = 1184;  // 8 CTAs per SM x 148 SMs
// d_out[j] = z^j, j < n
void vec_powers(halo_ctx* ctx, const fr_t& z, uint64_t n, fr_t* d_out);
// *d_out = sum a[i] b[i]; d_partials: scratch of VEC_DOT_MAX_BLOCKS elements; everything device resident
void vec_dot(halo_ctx* ctx, const fr_t* d_a, const fr_t* d_b, uint64_t n, fr_t* d_partials, fr_t* d_out);
// K3b: k polynomials packed back to back, polynomial j = d_coeffs[d_off[j] .. d_off[j+1]) (d_off: k + 1 device starts), its
// length <= n_max.  vec_eval_many: d_out[j] = <p_j, d_pows> (d_pows: z^0 .. z^(n_max-1)); d_partials holds
// k * vec_eval_many_blocks(k, n_max) elements.  vec_poly_combine: d_out[i] = sum_j alpha^j p_j[i], i < n.  k < 2^32.
uint32_t vec_eval_many_blocks(uint64_t k, uint64_t n_max);
void vec_eval_many(halo_ctx* ctx, const fr_t* d_coeffs, const uint64_t* d_off, uint64_t k, uint64_t n_max, const fr_t* d_pows,
                   fr_t* d_partials, fr_t* d_out);
void vec_poly_combine(halo_ctx* ctx, const fr_t* d_coeffs, const uint64_t* d_off, uint64_t k, const fr_t& alpha, uint64_t n,
                      fr_t* d_out);
// K3c: groups g = sum of terms w p_j over the polynomials packed in d_coeffs, divided by X - z or evaluated at z (vec.cu).
// Group gi owns the terms [first, first + count); zthr: 256 entries per point, zthr[u] = z^(16 u) (vec_quot_tables).
struct QuotTerm {
    fr_t w;
    uint64_t off, len;  // the polynomial's coefficients d_coeffs[off .. off + len)
    uint32_t unit;      // w = 1: added without a multiplication
    uint32_t pad[3];
};
struct QuotGroup {
    fr_t z, s, zblk;  // the point, the quotient's weight in q, z^(16 * 256)
    uint32_t first, count;
    uint32_t tab;     // the point's row of zthr
    uint32_t pad[5];
};
constexpr uint32_t VEC_QUOT_ZTHR = 256;
// blocks of 2^12 coefficients over n (at least one): kloc holds n_groups * blocks * 256 elements, agg / kblk n_groups * blocks
uint32_t vec_quot_blocks(uint64_t n);
void vec_quot_tables(const fr_t& z, fr_t& zblk, fr_t* zthr);
// d_rem[gi] = g(z) for every group, two launches
void vec_quot_eval(halo_ctx* ctx, const fr_t* d_coeffs, const QuotGroup* d_groups, uint32_t n_groups, const QuotTerm* d_terms,
                   const fr_t* d_zthr, uint64_t n, fr_t* d_agg, fr_t* d_rem);
// d_rem as above and d_q[i] = sum_g s_g quot(g, X - z_g)[i] for i < n - 1 (n >= every term's len), three launches
void vec_quotient(halo_ctx* ctx, const fr_t* d_coeffs, const QuotGroup* d_groups, uint32_t n_groups, const QuotTerm* d_terms,
                  const fr_t* d_zthr, uint64_t n, fr_t* d_kloc, fr_t* d_agg, fr_t* d_kblk, fr_t* d_rem, fr_t* d_q);
// d_out[i] = sum_j d_cs[j] p_j[i] + c_q d_q[i], i < n (p_j as in vec_eval_many; d_q[i] = 0 from n_q on)
void vec_poly_lincomb(halo_ctx* ctx, const fr_t* d_coeffs, const uint64_t* d_off, const fr_t* d_cs, uint64_t k, const fr_t* d_q,
                      uint64_t n_q, const fr_t& c_q, uint64_t n, fr_t* d_out);
// c[j] += xi_inv c[j+m]; z[j] += xi z[j+m], j < m
void vec_fold_scalars(halo_ctx* ctx, fr_t* d_c, fr_t* d_z, uint64_t m, const fr_t& xi, const fr_t& xi_inv);
// One claim of vec_h_lincomb on the device: weight, x[b] = xi_{lg_n - b} for b < lg_n (one above), lg_n.
constexpr uint32_t LINCOMB_MAX_LG = 30;
struct LincombClaim {
    fr_t w;
    fr_t x[LINCOMB_MAX_LG];
    uint32_t lg_n;
    uint32_t pad[7];
};
// d_out[i] (+)= sum_j weights[j] * coeffs(h_j)[i], i < n_out (coefficients of h_j zero from 2^lg_ns[j] on); claim j's
// challenges xi_0 .. xi_{lg_ns[j]} are the next lg_ns[j] + 1 rows of xis; xis, lg_ns, weights on the host, lg_ns[j] <= 30
void vec_h_lincomb(halo_ctx* ctx, const fr_t* xis, const uint32_t* lg_ns, const fr_t* weights, uint64_t k, uint64_t n_out,
                   bool accumulate, fr_t* d_out);
void vec_pbar(halo_ctx* ctx, const fr_t* d_q, uint64_t n_q, const fr_t& z, uint64_t n, fr_t* d_out);
void vec_axpy(halo_ctx* ctx, fr_t* d_y, const fr_t* d_x, const fr_t& alpha, uint64_t n);
}  // namespace halo
