// host/capi_host.cpp -- C view (include/halo_pcdl.h) of the C++ host layer, for ctypes / C callers.
#include <functional>

#include "../../include/halo_pcdl.h"

#include "acc.hpp"
#include "pcdl.hpp"
#include "pedersen.hpp"

using namespace halo;

namespace {
thread_local std::string g_host_error;
template <class F>
int guarded(F&& f) {
    try {
        f();
        return HALO_OK;
    } catch (const HaloFailure& e) {
        g_host_error = e.what();
        return e.code;
    } catch (const std::bad_alloc&) {
        g_host_error = "out of host memory";
        return HALO_ENOMEM;
    } catch (const std::exception& e) {
        g_host_error = e.what();
        return HALO_EINVAL;
    } catch (...) {  // nothing unwinds across the C ABI
        g_host_error = "unexpected internal exception";
        return HALO_EINVAL;
    }
}
// Verifier-side inputs are raw limbs from the caller: canonical residues and points on the curve, or HALO_EINVAL
// (see host/group.hpp "validation at the C boundary").
void validate(const halo_eval_proof& pi) {
    ensure(pi.lg_n <= HALO_MAX_LG, HALO_EINVAL, "proof: lg_n out of range");
    for (uint32_t i = 0; i < pi.lg_n; i++)
        ensure(point_valid(pi.Ls[i]) && point_valid(pi.Rs[i]), HALO_EINVAL, "proof: L / R is not a canonical point on the curve");
    ensure(point_valid(pi.U), HALO_EINVAL, "proof: U is not a canonical point on the curve");
    ensure(scalar_valid(pi.c), HALO_EINVAL, "proof: c is not a canonical scalar");
    if (pi.hiding) {
        ensure(point_valid(pi.C_bar), HALO_EINVAL, "proof: C_bar is not a canonical point on the curve");
        ensure(scalar_valid(pi.w_prime), HALO_EINVAL, "proof: w' is not a canonical scalar");
    }
}
void validate(const halo_instance& q) {
    ensure(point_valid(q.C), HALO_EINVAL, "instance: C is not a canonical point on the curve");
    ensure(scalar_valid(q.z) && scalar_valid(q.v), HALO_EINVAL, "instance: z / v is not a canonical scalar");
    validate(q.pi);
}
void validate(const halo_accumulator& a) {
    ensure(point_valid(a.C_bar) && point_valid(a.U0), HALO_EINVAL, "accumulator: C_bar / U_0 is not a canonical point on the curve");
    ensure(scalar_valid(a.z) && scalar_valid(a.v) && scalar_valid(a.w) && scalar_valid(a.h0[0]) && scalar_valid(a.h0[1]), HALO_EINVAL,
           "accumulator: z / v / w / h_0 is not a canonical scalar");
    validate(a.pi);
}
PolyView poly_from(const uint64_t* c, uint64_t n) { return PolyView(reinterpret_cast<const PallasScalar*>(c), n); }
}  // namespace

extern "C" {

const char* halo_host_last_error(void) { return g_host_error.c_str(); }

int halo_pedersen_commit(halo_ctx* ctx, const uint64_t* w, const uint64_t* gs_affine, uint64_t n_gs, const uint64_t* ms,
                         uint64_t n_ms, uint64_t out_jac[12]) {
    return guarded([&] {
        PallasScalar ws;
        if (w) ws = scalar_load(w);
        PallasPoint r = pedersen::commit(ctx, w ? &ws : nullptr, gs_affine, n_gs, reinterpret_cast<const PallasScalar*>(ms), n_ms);
        point_store(out_jac, r);
    });
}

int halo_pcdl_commit(halo_ctx* ctx, const uint64_t* coeffs, uint64_t n_coeffs, uint64_t d, const uint64_t* w, uint64_t out_jac[12]) {
    return guarded([&] {
        PallasScalar ws;
        if (w) ws = scalar_load(w);
        point_store(out_jac, pcdl::commit(ctx, poly_from(coeffs, n_coeffs), d, w ? &ws : nullptr));
    });
}

int halo_pcdl_commit_batch(halo_ctx* ctx, const uint64_t* coeffs, const uint64_t* n_coeffs, uint64_t k, uint64_t d, const uint64_t* ws,
                           uint64_t* out_jac) {
    return guarded([&] {
        if (k == 0) return;
        ensure(coeffs && n_coeffs && out_jac, HALO_EINVAL, "halo_pcdl_commit_batch: NULL pointer");
        std::vector<PolyView> ps;
        ps.reserve(k);
        uint64_t off = 0;
        for (uint64_t j = 0; j < k; j++) {
            ensure(n_coeffs[j] <= UINT64_MAX / 32 - off, HALO_EINVAL, "halo_pcdl_commit_batch: packed size overflows");
            ps.push_back(poly_from(coeffs + 4 * off, n_coeffs[j]));
            off += n_coeffs[j];
        }
        const std::vector<PallasPoint> C = pcdl::commit_batch(ctx, ps, d, reinterpret_cast<const PallasScalar*>(ws));
        for (uint64_t j = 0; j < k; j++) point_store(out_jac + 12 * j, C[j]);
    });
}

int halo_pcdl_commit_evals(halo_ctx* ctx, const uint64_t* evals, uint64_t k, uint64_t d, const uint64_t* ws, uint64_t* out_jac) {
    return guarded([&] {
        if (k == 0) return;
        ensure(evals && out_jac, HALO_EINVAL, "halo_pcdl_commit_evals: NULL pointer");
        ensure(d < UINT64_MAX && k <= UINT64_MAX / 32 / (d + 1), HALO_EINVAL, "halo_pcdl_commit_evals: k (d + 1) scalars overflow");
        const std::vector<PallasPoint> C = pcdl::commit_evals(ctx, reinterpret_cast<const PallasScalar*>(evals), k, d,
                                                              reinterpret_cast<const PallasScalar*>(ws));
        for (uint64_t j = 0; j < k; j++) point_store(out_jac + 12 * j, C[j]);
    });
}

int halo_pcdl_open(halo_ctx* ctx, const uint64_t* coeffs, uint64_t n_coeffs, const uint64_t C_jac[12], uint64_t d,
                   const uint64_t z[4], const uint64_t* w, const uint64_t* q, uint64_t n_q, const uint64_t* w_bar,
                   halo_eval_proof* pi) {
    return guarded([&] {
        PallasScalar ws, wbs;
        PolyView qp(nullptr, 0);
        if (w) {
            ensure(q && w_bar, HALO_EINVAL, "hiding open needs q and w_bar");
            ws = scalar_load(w);
            wbs = scalar_load(w_bar);
            qp = poly_from(q, n_q);
        }
        pcdl::EvalProof p = pcdl::open(ctx, poly_from(coeffs, n_coeffs), point_load(C_jac), d, scalar_load(z), w ? &ws : nullptr,
                                       w ? &qp : nullptr, w ? &wbs : nullptr);
        pcdl::proof_to_c(p, *pi);
    });
}

int halo_pcdl_open_batch(halo_ctx* ctx, const uint64_t* coeffs, const uint64_t* n_coeffs, uint64_t k, const uint64_t* Cs, uint64_t d,
                         const uint64_t z[4], const uint64_t* ws, const uint64_t* q, uint64_t n_q, const uint64_t* w_bar,
                         uint64_t* vs_out, uint64_t C_out[12], uint64_t v_out[4], halo_eval_proof* pi) {
    return guarded([&] {
        ensure(k >= 1, HALO_EINVAL, "halo_pcdl_open_batch: nothing to open (k = 0)");
        ensure(n_coeffs && Cs && vs_out && C_out && v_out && pi, HALO_EINVAL, "halo_pcdl_open_batch: NULL pointer");
        std::vector<PolyView> ps;
        std::vector<PallasPoint> C(k);
        std::vector<PallasScalar> w(ws ? k : 0);
        ps.reserve(k);
        uint64_t off = 0;
        for (uint64_t j = 0; j < k; j++) {
            ensure(n_coeffs[j] <= UINT64_MAX / 32 - off, HALO_EINVAL, "halo_pcdl_open_batch: packed size overflows");
            ps.push_back(poly_from(coeffs + 4 * off, n_coeffs[j]));
            off += n_coeffs[j];
            C[j] = point_load_checked(Cs + 12 * j, "C_j is not a canonical point on the curve");
            if (ws) w[j] = scalar_load_checked(ws + 4 * j, "w_j is not a canonical scalar");
        }
        ensure(coeffs || off == 0, HALO_EINVAL, "halo_pcdl_open_batch: NULL coefficients");
        const PallasScalar zs = scalar_load_checked(z, "z is not a canonical scalar");
        PallasScalar wbs;
        PolyView qp(nullptr, 0);
        if (ws) {
            ensure(w_bar && (q || n_q == 0), HALO_EINVAL, "hiding open needs q and w_bar");
            wbs = scalar_load(w_bar);
            qp = poly_from(q, n_q);
        }
        pcdl::BatchOpening r = pcdl::open_batch(ctx, ps, C, d, zs, ws ? w.data() : nullptr, ws ? &qp : nullptr, ws ? &wbs : nullptr);
        for (uint64_t j = 0; j < k; j++) scalar_store(vs_out + 4 * j, r.vs[j]);
        point_store(C_out, r.C);
        scalar_store(v_out, r.v);
        pcdl::proof_to_c(r.pi, *pi);
    });
}

int halo_pcdl_batch_claim(halo_ctx* ctx, const uint64_t* Cs, const uint64_t* vs, uint64_t k, const uint64_t z[4], uint64_t C_out[12],
                          uint64_t v_out[4]) {
    return guarded([&] {
        ensure(k >= 1, HALO_EINVAL, "halo_pcdl_batch_claim: no claim (k = 0)");
        ensure(Cs && vs && C_out && v_out, HALO_EINVAL, "halo_pcdl_batch_claim: NULL pointer");
        std::vector<PallasPoint> C(k);
        std::vector<PallasScalar> v(k);
        for (uint64_t j = 0; j < k; j++) {
            C[j] = point_load_checked(Cs + 12 * j, "C_j is not a canonical point on the curve");
            v[j] = scalar_load_checked(vs + 4 * j, "v_j is not a canonical scalar");
        }
        const pcdl::BatchClaim r = pcdl::batch_claim(ctx, C, v, scalar_load_checked(z, "z is not a canonical scalar"));
        point_store(C_out, r.C);
        scalar_store(v_out, r.v);
    });
}

// The caller's points and queries of a multi-point opening (validated in pcdl::multi_validate)
static void multi_inputs(const uint64_t* zs, uint64_t T, const uint64_t* q_poly, const uint64_t* q_point, uint64_t m,
                         std::vector<PallasScalar>& z, std::vector<uint64_t>& qp, std::vector<uint64_t>& qt) {
    z.resize(T);
    for (uint64_t t = 0; t < T; t++) z[t] = scalar_load_checked(zs + 4 * t, "z_t is not a canonical scalar");
    qp.assign(q_poly, q_poly + m);
    qt.assign(q_point, q_point + m);
}

// The body of the two multi-point entry points after their polynomials: the caller's commitments, points, queries and draws
// in, the opening of `open` out
using MultiOpen = std::function<pcdl::MultiOpening(const std::vector<PallasPoint>&, const std::vector<PallasScalar>&, const std::vector<uint64_t>&,
                                                   const std::vector<uint64_t>&, const PallasScalar*, const PallasScalar*, const PolyView*,
                                                   const PallasScalar*)>;
static void open_multi_c(uint64_t k, const uint64_t* Cs, const uint64_t* zs, uint64_t T, const uint64_t* q_poly, const uint64_t* q_point,
                         uint64_t m, const uint64_t* ws, const uint64_t* w_Q, const uint64_t* q, uint64_t n_q, const uint64_t* w_bar,
                         uint64_t* vs_out, uint64_t Q_out[12], uint64_t* us_out, uint64_t C_out[12], uint64_t x_out[4], uint64_t v_out[4],
                         halo_eval_proof* pi, const MultiOpen& open) {
    std::vector<PallasPoint> C(k);
    std::vector<PallasScalar> w(ws ? k : 0);
    for (uint64_t j = 0; j < k; j++) {
        C[j] = point_load_checked(Cs + 12 * j, "C_j is not a canonical point on the curve");
        if (ws) w[j] = scalar_load_checked(ws + 4 * j, "w_j is not a canonical scalar");
    }
    std::vector<PallasScalar> z;
    std::vector<uint64_t> qp, qt;
    multi_inputs(zs, T, q_poly, q_point, m, z, qp, qt);
    PallasScalar wq, wbs;
    PolyView qv(nullptr, 0);
    if (ws) {
        ensure(w_Q && w_bar && (q || n_q == 0), HALO_EINVAL, "hiding open needs w_Q, q and w_bar");
        wq = scalar_load_checked(w_Q, "w_Q is not a canonical scalar");
        wbs = scalar_load_checked(w_bar, "w_bar is not a canonical scalar");
        qv = poly_from(q, n_q);
    }
    const pcdl::MultiOpening r = open(C, z, qp, qt, ws ? w.data() : nullptr, ws ? &wq : nullptr, ws ? &qv : nullptr, ws ? &wbs : nullptr);
    for (uint64_t i = 0; i < m; i++) scalar_store(vs_out + 4 * i, r.vs[i]);
    point_store(Q_out, r.Q);
    for (uint64_t t = 0; t < T; t++) scalar_store(us_out + 4 * t, r.us[t]);
    point_store(C_out, r.claim.C);
    scalar_store(x_out, r.claim.x3);
    scalar_store(v_out, r.claim.v);
    pcdl::proof_to_c(r.pi, *pi);
}

int halo_pcdl_open_multi(halo_ctx* ctx, const uint64_t* coeffs, const uint64_t* n_coeffs, uint64_t k, const uint64_t* Cs, uint64_t d,
                         const uint64_t* zs, uint64_t T, const uint64_t* q_poly, const uint64_t* q_point, uint64_t m, const uint64_t* ws,
                         const uint64_t* w_Q, const uint64_t* q, uint64_t n_q, const uint64_t* w_bar, uint64_t* vs_out, uint64_t Q_out[12],
                         uint64_t* us_out, uint64_t C_out[12], uint64_t x_out[4], uint64_t v_out[4], halo_eval_proof* pi) {
    return guarded([&] {
        ensure(k >= 1 && T >= 1 && m >= 1, HALO_EINVAL, "halo_pcdl_open_multi: k, T and m must be at least 1");
        ensure(n_coeffs && Cs && zs && q_poly && q_point && vs_out && Q_out && us_out && C_out && x_out && v_out && pi, HALO_EINVAL,
               "halo_pcdl_open_multi: NULL pointer");
        std::vector<PolyView> ps;
        ps.reserve(k);
        uint64_t off = 0;
        for (uint64_t j = 0; j < k; j++) {
            ensure(n_coeffs[j] <= UINT64_MAX / 32 - off, HALO_EINVAL, "halo_pcdl_open_multi: packed size overflows");
            ps.push_back(poly_from(coeffs + 4 * off, n_coeffs[j]));
            off += n_coeffs[j];
        }
        ensure(coeffs || off == 0, HALO_EINVAL, "halo_pcdl_open_multi: NULL coefficients");
        open_multi_c(k, Cs, zs, T, q_poly, q_point, m, ws, w_Q, q, n_q, w_bar, vs_out, Q_out, us_out, C_out, x_out, v_out, pi,
                     [&](auto& C, auto& z, auto& qp, auto& qt, auto w, auto wq, auto qv, auto wb) {
                         return pcdl::open_multi(ctx, ps, C, d, z, qp, qt, w, wq, qv, wb);
                     });
    });
}

int halo_pcdl_open_multi_evals(halo_ctx* ctx, const uint64_t* evals, uint64_t k, const uint64_t* Cs, uint64_t d, const uint64_t* zs,
                               uint64_t T, const uint64_t* q_poly, const uint64_t* q_point, uint64_t m, const uint64_t* ws,
                               const uint64_t* w_Q, const uint64_t* q, uint64_t n_q, const uint64_t* w_bar, uint64_t* vs_out,
                               uint64_t Q_out[12], uint64_t* us_out, uint64_t C_out[12], uint64_t x_out[4], uint64_t v_out[4],
                               halo_eval_proof* pi) {
    return guarded([&] {
        ensure(k >= 1 && T >= 1 && m >= 1, HALO_EINVAL, "halo_pcdl_open_multi_evals: k, T and m must be at least 1");
        ensure(evals && Cs && zs && q_poly && q_point && vs_out && Q_out && us_out && C_out && x_out && v_out && pi, HALO_EINVAL,
               "halo_pcdl_open_multi_evals: NULL pointer");
        const PallasScalar* e = reinterpret_cast<const PallasScalar*>(evals);
        open_multi_c(k, Cs, zs, T, q_poly, q_point, m, ws, w_Q, q, n_q, w_bar, vs_out, Q_out, us_out, C_out, x_out, v_out, pi,
                     [&](auto& C, auto& z, auto& qp, auto& qt, auto w, auto wq, auto qv, auto wb) {
                         return pcdl::open_multi_evals(ctx, e, C, d, z, qp, qt, w, wq, qv, wb);
                     });
    });
}

int halo_pcdl_multi_claim(halo_ctx* ctx, const uint64_t* Cs, uint64_t k, const uint64_t* zs, uint64_t T, const uint64_t* q_poly,
                          const uint64_t* q_point, const uint64_t* vs, uint64_t m, const uint64_t Q[12], const uint64_t* us,
                          uint64_t C_out[12], uint64_t x_out[4], uint64_t v_out[4]) {
    return guarded([&] {
        ensure(k >= 1 && T >= 1 && m >= 1, HALO_EINVAL, "halo_pcdl_multi_claim: k, T and m must be at least 1");
        ensure(Cs && zs && q_poly && q_point && vs && Q && us && C_out && x_out && v_out, HALO_EINVAL, "halo_pcdl_multi_claim: NULL pointer");
        std::vector<PallasPoint> C(k);
        for (uint64_t j = 0; j < k; j++) C[j] = point_load_checked(Cs + 12 * j, "C_j is not a canonical point on the curve");
        std::vector<PallasScalar> z, v(m), u(T);
        std::vector<uint64_t> qp, qt;
        multi_inputs(zs, T, q_poly, q_point, m, z, qp, qt);
        for (uint64_t i = 0; i < m; i++) v[i] = scalar_load_checked(vs + 4 * i, "v_i is not a canonical scalar");
        const PallasPoint Qp = point_load_checked(Q, "Q is not a canonical point on the curve");
        for (uint64_t t = 0; t < T; t++) u[t] = scalar_load_checked(us + 4 * t, "u_t is not a canonical scalar");
        const pcdl::MultiClaim r = pcdl::multi_claim(ctx, C, z, qp, qt, v, Qp, u);
        point_store(C_out, r.C);
        scalar_store(x_out, r.x3);
        scalar_store(v_out, r.v);
    });
}

int halo_pcdl_succinct_check(halo_ctx* ctx, const uint64_t C_jac[12], uint64_t d, const uint64_t z[4], const uint64_t v[4],
                             const halo_eval_proof* pi, uint64_t* xis_out, uint64_t U_out[12]) {
    return guarded([&] {
        ensure(pi != nullptr, HALO_EINVAL, "null proof");
        validate(*pi);
        auto hu = pcdl::succinct_check(ctx, point_load_checked(C_jac, "C is not a canonical point on the curve"), d,
                                       scalar_load_checked(z, "z is not a canonical scalar"),
                                       scalar_load_checked(v, "v is not a canonical scalar"), pcdl::proof_from_c(*pi));
        if (xis_out) std::memcpy(xis_out, hu.first.xis.data(), hu.first.xis.size() * 32);
        if (U_out) point_store(U_out, hu.second);
    });
}

int halo_pcdl_check(halo_ctx* ctx, const uint64_t C_jac[12], uint64_t d, const uint64_t z[4], const uint64_t v[4],
                    const halo_eval_proof* pi) {
    return guarded([&] {
        ensure(pi != nullptr, HALO_EINVAL, "null proof");
        validate(*pi);
        pcdl::check(ctx, point_load_checked(C_jac, "C is not a canonical point on the curve"), d,
                    scalar_load_checked(z, "z is not a canonical scalar"), scalar_load_checked(v, "v is not a canonical scalar"),
                    pcdl::proof_from_c(*pi));
    });
}

int halo_pcdl_check_batch(halo_ctx* ctx, const halo_instance* claims, uint64_t k, const uint64_t rho[4], uint64_t* rejected_index) {
    return guarded([&] {
        if (k == 0) return;
        ensure(claims && rho && rejected_index, HALO_EINVAL, "null claims / rho / rejected_index");
        const PallasScalar r = scalar_load_checked(rho, "rho is not a canonical scalar");
        std::vector<acc::Instance> v;
        v.reserve(k);
        for (uint64_t j = 0; j < k; j++) {
            validate(claims[j]);
            v.push_back(acc::instance_from_c(claims[j]));
        }
        std::vector<pcdl::Query> qs;
        qs.reserve(k);
        for (const acc::Instance& q : v) qs.push_back(pcdl::Query{&q.C, q.d, &q.z, &q.v, &q.pi});
        pcdl::check_batch(ctx, qs, r, rejected_index);
    });
}

int halo_h_eval(const uint64_t* xis, uint32_t lg_n, const uint64_t z[4], uint64_t out[4]) {
    return guarded([&] {
        std::vector<PallasScalar> x(lg_n + 1);
        std::memcpy(x.data(), xis, (lg_n + 1) * 32);
        scalar_store(out, pcdl::HPoly(x).eval(scalar_load(z)));
    });
}

int halo_acc_prover(halo_ctx* ctx, uint64_t d, const halo_instance* qs, uint64_t m, const uint64_t h0[2][4], const uint64_t w[4],
                    const uint64_t* q, uint64_t n_q, const uint64_t w_bar[4], halo_accumulator* acc) {
    return guarded([&] {
        ensure(qs != nullptr || m == 0, HALO_EINVAL, "null instance list");
        std::vector<acc::Instance> v;
        for (uint64_t i = 0; i < m; i++) {
            validate(qs[i]);
            v.push_back(acc::instance_from_c(qs[i]));
        }
        acc::Accumulator a = acc::prover(ctx, d, v, PallasPoly{scalar_load(h0[0]), scalar_load(h0[1])}, scalar_load(w),
                                         poly_from(q, n_q), scalar_load(w_bar));
        acc::accumulator_to_c(a, *acc);
    });
}

int halo_acc_verifier(halo_ctx* ctx, uint64_t d, const halo_instance* qs, uint64_t m, const halo_accumulator* acc) {
    return guarded([&] {
        ensure(acc != nullptr && (qs != nullptr || m == 0), HALO_EINVAL, "null accumulator / instance list");
        validate(*acc);
        std::vector<acc::Instance> v;
        for (uint64_t i = 0; i < m; i++) {
            validate(qs[i]);
            v.push_back(acc::instance_from_c(qs[i]));
        }
        acc::verifier(ctx, d, v, acc::accumulator_from_c(*acc));
    });
}

int halo_acc_decider(halo_ctx* ctx, const halo_accumulator* acc) {
    return guarded([&] {
        ensure(acc != nullptr, HALO_EINVAL, "null accumulator");
        validate(*acc);
        acc::decider(ctx, acc::accumulator_from_c(*acc));
    });
}

int halo_acc_decider_batch(halo_ctx* ctx, const halo_accumulator* accs, uint64_t k, const uint64_t rho[4], uint64_t* rejected_index) {
    return guarded([&] {
        if (k == 0) return;
        ensure(accs && rho && rejected_index, HALO_EINVAL, "null accumulators / rho / rejected_index");
        const PallasScalar r = scalar_load_checked(rho, "rho is not a canonical scalar");
        std::vector<acc::Accumulator> v;
        v.reserve(k);
        for (uint64_t j = 0; j < k; j++) {
            validate(accs[j]);
            v.push_back(acc::accumulator_from_c(accs[j]));
        }
        acc::decider_batch(ctx, v, r, rejected_index);
    });
}

int halo_acc_verifier_batch(halo_ctx* ctx, uint64_t d, const halo_instance* qs, const uint64_t* ms, const halo_accumulator* accs,
                            uint64_t k, const uint64_t rho[4], uint64_t* rejected_index) {
    return halo_acc_verify_decide_batch(ctx, d, qs, ms, accs, k, nullptr, 0, rho, rejected_index);
}

int halo_acc_verify_decide_batch(halo_ctx* ctx, uint64_t d, const halo_instance* qs, const uint64_t* ms,
                                 const halo_accumulator* steps_accs, uint64_t k, const halo_accumulator* decide_accs, uint64_t k_dec,
                                 const uint64_t rho[4], uint64_t* rejected_index) {
    return guarded([&] {
        if (k == 0 && k_dec == 0) return;
        ensure((ms && steps_accs) || k == 0, HALO_EINVAL, "null ms / step accumulators");
        ensure(decide_accs || k_dec == 0, HALO_EINVAL, "null decided accumulators");
        ensure(rho && rejected_index, HALO_EINVAL, "null rho / rejected_index");
        const PallasScalar r = scalar_load_checked(rho, "rho is not a canonical scalar");
        uint64_t total = 0;
        for (uint64_t i = 0; i < k; i++) {
            ensure(ms[i] <= UINT64_MAX - total, HALO_EINVAL, "instance count overflows");
            total += ms[i];
        }
        ensure(qs != nullptr || total == 0, HALO_EINVAL, "null instance list");
        std::vector<std::vector<acc::Instance>> qv(k);
        std::vector<acc::Accumulator> av;
        av.reserve(k);
        uint64_t at = 0;
        for (uint64_t i = 0; i < k; i++) {
            validate(steps_accs[i]);
            av.push_back(acc::accumulator_from_c(steps_accs[i]));
            for (uint64_t j = 0; j < ms[i]; j++, at++) {
                validate(qs[at]);
                qv[i].push_back(acc::instance_from_c(qs[at]));
            }
        }
        std::vector<acc::Accumulator> dv;
        dv.reserve(k_dec);
        for (uint64_t j = 0; j < k_dec; j++) {
            validate(decide_accs[j]);
            dv.push_back(acc::accumulator_from_c(decide_accs[j]));
        }
        std::vector<acc::Step> steps(k);
        for (uint64_t i = 0; i < k; i++) steps[i] = acc::Step{&qv[i], &av[i]};
        std::vector<pcdl::Query> claims;
        claims.reserve(k_dec);
        for (const acc::Accumulator& a : dv) claims.push_back(pcdl::Query{&a.C_bar, a.d, &a.z, &a.v, &a.pi});
        acc::verify_decide_batch(ctx, d, steps, claims, r, rejected_index);
    });
}

void halo_acc_to_instance(const halo_accumulator* acc, halo_instance* q) {
    std::memcpy(q->C, acc->C_bar, 96);
    q->d = acc->d;
    std::memcpy(q->z, acc->z, 32);
    std::memcpy(q->v, acc->v, 32);
    q->pi = acc->pi;
}

void halo_point_serialize_compressed(const uint64_t p_jac[12], uint8_t out[33]) { serialize_compressed(point_load(p_jac), out); }

}  // extern "C"
