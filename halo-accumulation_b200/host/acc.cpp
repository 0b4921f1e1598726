// host/acc.cpp -- see acc.hpp.  Control flow follows code/src/acc.rs step by step.
#include "acc.hpp"

#include <algorithm>
#include <cstdint>
#include <optional>

namespace halo {
namespace acc {

static uint32_t ilog2(uint64_t n) {
    uint32_t l = 0;
    while (((uint64_t)1 << (l + 1)) <= n) l++;
    return l;
}

PallasPoly AccumulatedHPolys::get_poly(halo_ctx* ctx, uint32_t lg_n) const {
    size_t n = (size_t)1 << lg_n;
    PallasPoly out(n);
    std::vector<PallasScalar> xis;
    xis.reserve(hs.size() * (lg_n + 1));
    for (const auto& h : hs) {
        ensure(h.xis.size() == lg_n + 1, HALO_EINVAL, "HPoly size mismatch");
        xis.insert(xis.end(), h.xis.begin(), h.xis.end());
    }
    size_t n_h0 = have_h0 ? (h_0.size() < n ? h_0.size() : n) : 0;
    check_rc(ctx, halo_h_lincomb(ctx, reinterpret_cast<const uint64_t*>(h_0.data()), n_h0,
                                 reinterpret_cast<const uint64_t*>(alphas.data()),
                                 reinterpret_cast<const uint64_t*>(xis.data()), hs.size(), lg_n,
                                 reinterpret_cast<uint64_t*>(out.data())));
    return out;
}

uint64_t AccumulatedHPolys::get_poly_resident(halo_ctx* ctx, uint32_t lg_n) const {
    size_t n = (size_t)1 << lg_n;
    std::vector<PallasScalar> xis;
    xis.reserve(hs.size() * (lg_n + 1));
    for (const auto& h : hs) {
        ensure(h.xis.size() == lg_n + 1, HALO_EINVAL, "HPoly size mismatch");
        xis.insert(xis.end(), h.xis.begin(), h.xis.end());
    }
    size_t n_h0 = have_h0 ? (h_0.size() < n ? h_0.size() : n) : 0;
    uint64_t deg = 0;
    check_rc(ctx, halo_h_lincomb_resident(ctx, reinterpret_cast<const uint64_t*>(h_0.data()), n_h0,
                                          reinterpret_cast<const uint64_t*>(alphas.data()),
                                          reinterpret_cast<const uint64_t*>(xis.data()), hs.size(), lg_n, &deg));
    return deg;
}

PallasScalar AccumulatedHPolys::eval(const PallasScalar& z) const {
    PallasScalar v = scalar_zero();
    if (have_h0) {  // h_0.evaluate(z), Horner
        PallasScalar acc = scalar_zero();
        for (size_t i = h_0.size(); i-- > 0;) acc = acc * z + h_0[i];
        v = v + acc;
    }
    for (size_t i = 0; i < hs.size(); i++) v = v + hs[i].eval(z) * alphas[i + 1];
    return v;
}

// Field order of the derive: h_0: Option<PallasPoly>, hs: Vec<HPoly>, alpha: Option<PallasScalar>, alphas: Vec<PallasScalar>.
// Option -> 1 byte then the value; Vec -> u64 LE length then elements; DensePolynomial -> its coeffs Vec (trailing
// zeros trimmed by from_coefficients_vec); HPoly -> its xis Vec.  [ark-serialize 0.5, restated; parity unpinned]
void AccumulatedHPolys::serialize(Transcript& t) const {
    t.u8(have_h0 ? 1 : 0);
    if (have_h0) {
        size_t len = h_0.size();
        while (len > 0 && fp_is_zero(h_0[len - 1])) len--;
        t.u64(len);
        for (size_t i = 0; i < len; i++) t.scalar(h_0[i]);
    }
    t.u64(hs.size());
    for (const auto& h : hs) {
        t.u64(h.xis.size());
        for (const auto& x : h.xis) t.scalar(x);
    }
    t.u8(have_alpha ? 1 : 0);
    if (have_alpha) t.scalar(alpha);
    t.u64(alphas.size());
    for (const auto& a : alphas) t.scalar(a);
}

struct CommonOut {
    PallasPoint C_bar;
    uint64_t d;
    PallasScalar z;
    AccumulatedHPolys hs;
};

// acc.rs:135-188
static CommonOut common_subroutine(halo_ctx* ctx, uint64_t d, const std::vector<Instance>& qs, const AccumulatorHiding& pi_V) {
    size_t m = qs.size();
    AccumulatedHPolys hs(m);
    std::vector<PallasPoint> Us;
    Us.reserve(m + 1);
    // (2) parse pi_V (:146-149)
    hs.h_0 = pi_V.h;
    hs.have_h0 = true;
    Us.push_back(pi_V.U);
    // (3) and (4) need m + 1 small MSMs, none of which depends on another's result: one device round trip for all of
    // them (pcdl::succinct_check_many), the `ensure!`s raised afterwards in the reference's order.  Input that the
    // reference would panic on goes through the one-by-one path so that the first failure is the reference's.
    bool batched = false;
    if (m >= 1 && pi_V.h.size() <= 4096) {
        try {
            std::vector<pcdl::Query> queries;
            for (const auto& q : qs) queries.push_back(pcdl::Query{&q.C, q.d, &q.z, &q.v, &q.pi});
            PolyView h0(pi_V.h);
            pcdl::SuccinctMany sm = pcdl::succinct_check_many(ctx, queries, &h0, d);
            batched = true;
            // (3) U_0 == PCDL.Commit(h_0, d, None) (:152-155)
            ensure(pi_V.U == sm.commitment, HALO_REJECT_U0, "U_0 != PCDL.Commit_rho0(ck^(1)_PC, h_0; w = bot)");
            // (4) (:158-170)
            for (size_t i = 0; i < m; i++) {
                ensure(sm.accept[i], HALO_REJECT_SUCCINCT, "C_(log_n) != CM.Commit_Sigma(c || v')");  // pcdl.rs:307-310
                hs.hs.push_back(sm.hu[i].first);
                Us.push_back(sm.hu[i].second);
                ensure(qs[i].d == d, HALO_REJECT_D, "d_i != d");  // :169
            }
        } catch (const HaloFailure& e) {
            if (batched || e.code <= HALO_REJECT_SUCCINCT) throw;  // a decision, already in the reference's order
            hs.hs.clear();
            Us.resize(1);
        }
    }
    if (!batched) {
        // (3) U_0 == PCDL.Commit(h_0, d, None) (:152-155)
        ensure(pi_V.U == pcdl::commit(ctx, pi_V.h, d, nullptr), HALO_REJECT_U0, "U_0 != PCDL.Commit_rho0(ck^(1)_PC, h_0; w = bot)");
        // (4) (:158-170)
        for (const auto& q : qs) {
            auto hu = pcdl::succinct_check(ctx, q.C, q.d, q.z, q.v, q.pi);
            hs.hs.push_back(hu.first);
            Us.push_back(hu.second);
            ensure(q.d == d, HALO_REJECT_D, "d_i != d");  // :169
        }
    }
    // (6) alpha = rho_1(hs) (:173)
    Transcript t;
    hs.serialize(t);
    hs.set_alpha(t.finish(1));
    // (8) C = sum alpha^i U_i (:178)
    PallasPoint C = point_dot(ctx, hs.alphas.data(), Us, Us.size() < hs.alphas.size() ? Us.size() : hs.alphas.size());
    // (9) z = rho_1(C, alpha) (:181)
    PallasScalar z = Transcript().point(C).scalar(hs.alpha).finish(1);
    // (10) C_bar = C + w S (:184)
    PallasPoint S, H;
    params_SH(ctx, S, H);
    PallasPoint C_bar = C + S * pi_V.w;
    return CommonOut{C_bar, d, z, std::move(hs)};
}

Accumulator prover(halo_ctx* ctx, uint64_t d, const std::vector<Instance>& qs, const PallasPoly& h_0, const PallasScalar& w,
                   PolyView q, const PallasScalar& w_bar) {
    ensure(h_0.size() == 2, HALO_EINVAL, "h_0 must be PallasPoly::rand(1): two coefficients");  // :192
    // U_0 = PCDL.Commit(h_0, d, None) (:195)
    PallasPoint U_0 = pcdl::commit(ctx, h_0, d, nullptr);
    AccumulatorHiding pi_V{h_0, U_0, w};  // :198-199
    CommonOut c = common_subroutine(ctx, d, qs, pi_V);  // :202
    PallasScalar v = c.hs.eval(c.z);                    // :205
    // pi = PCDL.Open(h(X), C_bar, d, z; w) (:209)
    // h.get_poly() (:85-94) is expanded on the device and opened from there
    uint64_t deg = c.hs.get_poly_resident(ctx, ilog2(d + 1));
    pcdl::EvalProof pi = pcdl::open_resident(ctx, deg, c.C_bar, d, c.z, &w, &q, &w_bar);
    return Accumulator{c.C_bar, c.d, c.z, v, pi, pi_V};  // :212-219
}

void verifier(halo_ctx* ctx, uint64_t D, const std::vector<Instance>& qs, const Accumulator& acc) {
    CommonOut c = common_subroutine(ctx, D, qs, acc.pi_V);  // :234
    ensure(c.C_bar == acc.C_bar, HALO_REJECT_CBAR, "C_bar' != C_bar");  // :237
    ensure(c.z == acc.z, HALO_REJECT_Z, "z' = z");                       // :238
    ensure(c.d == acc.d, HALO_REJECT_D, "d' = d");                       // :239
    ensure(c.hs.eval(acc.z) == acc.v, HALO_REJECT_V, "h(z) = v");        // :240
}

void decider(halo_ctx* ctx, const Accumulator& acc) {
    pcdl::check(ctx, acc.C_bar, acc.d, acc.z, acc.v, acc.pi);  // :254
}

void decider_batch(halo_ctx* ctx, const std::vector<Accumulator>& accs, const PallasScalar& rho, uint64_t* rejected_index) {
    std::vector<pcdl::Query> qs;
    qs.reserve(accs.size());
    for (const Accumulator& a : accs) qs.push_back(pcdl::Query{&a.C_bar, a.d, &a.z, &a.v, &a.pi});
    pcdl::check_batch(ctx, qs, rho, rejected_index);
}

// DESIGN.md K5c.  Step i (instances q_{i,j}, accumulator acc_i) holds iff the group equations
//   A_i = U0_i - h0_i[0] G_0 - h0_i[1] G_1                       (acc.rs:152-155)
//   E_ij = the succinct equation of q_{i,j}                       (pcdl.rs:307-310)
//   B_i = sum_{j=0..m_i} alpha_i^j U_{i,j} + omega_i S - C_bar_i  (acc.rs:178, :184, :237; U_{i,0} = U0_i)
// are O and the host checks d_{i,j} = D, d_i = D, rho_1(C*_i, alpha_i) = z_i with C*_i = C_bar_i - omega_i S, h_i(z_i) = v_i
// hold.  z' = rho_1(C_i, alpha_i) hashes C_i = sum_j alpha_i^j U_{i,j} itself, which a random combination cannot stand for;
// C*_i is the only C_i that passes (B_i = O <=> C_i = C*_i), so it is hashed instead.  The T_v = sum_i (m_i + 2) equations
// are combined in the order A_0, E_0*, B_0, A_1, .. with the powers of rho.  DESIGN.md K5d: the decided claims' E_j, F_j
// (pcdl::check_batch) follow with rho^(T_v + 2j), rho^(T_v + 2j + 1), and everything is ONE halo_h_msm_batch.
void verify_decide_batch(halo_ctx* ctx, uint64_t D, const std::vector<Step>& steps, const std::vector<pcdl::Query>& claims,
                         const PallasScalar& rho, uint64_t* rejected_index) {
    ensure(!fp_is_zero(rho), HALO_EINVAL, "rho is zero");
    const size_t k = steps.size();
    if (k == 0 && claims.empty()) return;
    PallasPoint S, H;
    params_SH(ctx, S, H);  // missing parameters fail here, before any worker thread reads the context
    const uint64_t n = D + 1;
    affine_t g[2];
    pcdl::QueryBatch inst, dec;  // the steps' instances, the decided claims
    std::vector<size_t> first(k + 1, 0);
    if (k > 0) {
        // what the single verifier refuses as malformed, wherever it sits (pcdl::commit of h_0: pcdl.rs:102-104)
        ensure(n != 0 && !(n & (n - 1)), HALO_EINVAL, "d+1 is not a power of 2");
        ensure(n <= halo_num_generators(ctx), HALO_EINVAL, "d > D");
        for (size_t i = 0; i < k; i++) {
            const Accumulator& a = *steps[i].acc;
            ensure(a.pi_V.h.size() == 2, HALO_EINVAL, "h_0 must have two coefficients");
            ensure(D >= 1 || fp_is_zero(a.pi_V.h[1]), HALO_EINVAL, "p.degree() > d");
            first[i] = inst.qs.size();
            for (const Instance& q : *steps[i].qs) inst.qs.push_back(pcdl::Query{&q.C, q.d, &q.z, &q.v, &q.pi});
        }
        // G_0, G_1 of the A_i: read now, as the read waits for the context's stream, which the generator part will occupy
        check_rc(ctx, halo_get_generators(ctx, 0, n >= 2 ? 2 : 1, reinterpret_cast<uint64_t*>(g)));
    }
    first[k] = inst.qs.size();
    dec.qs = claims;

    // validation + alpha of every query; then C' of the hiding ones and C*_i of every step in ONE combine call
    inst.validate(ctx, false);
    dec.validate(ctx, true);
    pcdl::CombineList cl;
    inst.request(cl);
    dec.request(cl);
    const size_t star = cl.P.size();
    for (size_t i = 0; i < k; i++) cl.push(steps[i].acc->C_bar, point_zero(), scalar_zero(), -steps[i].acc->pi_V.w);
    const std::vector<affine_t> c_out = cl.run(ctx);

    // the decided claims' transcripts; their generator part then runs on the device while the steps' transcripts run here
    pcdl::parallel_each(dec.valid, [&](size_t j) { dec.finish(ctx, j, c_out); });
    PallasScalar r_dec = scalar_one();  // rho^T_v
    for (size_t t = 0; t < inst.qs.size() + 2 * k; t++) r_dec = r_dec * rho;
    pcdl::BatchTerms terms;
    pcdl::GeneratorPart gen(ctx);
    if (!inst.failed() && !dec.failed()) {
        terms.add_claims(dec, dec.c_prime_affine(c_out), r_dec, rho);
        gen.submit(terms);
    }

    // per step: the rest of every transcript, alpha_i = rho_1(hs_i) (acc.rs:173) and the host checks
    std::vector<std::vector<PallasScalar>> step_alphas(k);
    std::vector<uint8_t> host_ok(k, 0);
    const auto step_errs = pcdl::parallel_each(k, [&](size_t i) {
        const Accumulator& a = *steps[i].acc;
        const size_t m = first[i + 1] - first[i];
        AccumulatedHPolys hs(m);
        hs.h_0 = a.pi_V.h;
        hs.have_h0 = true;
        bool ok = a.d == D;  // acc.rs:239
        for (size_t j = first[i]; j < first[i + 1]; j++) {
            if (j >= inst.valid) return;
            inst.finish(ctx, j, c_out);
            if (!inst.preps[j]) return;
            hs.hs.push_back(inst.preps[j]->h);
            ok = ok && inst.qs[j].d == D;  // acc.rs:169
        }
        Transcript t;
        hs.serialize(t);
        hs.set_alpha(t.finish(1));
        ok = ok && Transcript().point_affine(c_out[star + i]).scalar(hs.alpha).finish(1) == a.z;  // acc.rs:181, :238
        ok = ok && hs.eval(a.z) == a.v;                                                            // acc.rs:240
        host_ok[i] = ok;
        step_alphas[i] = std::move(hs.alphas);
    });
    inst.rethrow_first();
    if (pcdl::first_error(step_errs) < k) std::rethrow_exception(step_errs[pcdl::first_error(step_errs)]);
    dec.rethrow_first();

    // sum_t rho^t X_t over A_i, E_i1 .. E_im_i, B_i
    std::vector<PallasPoint> acc_pts;  // U0_i, C_bar_i of every step, normalised together
    for (size_t i = 0; i < k; i++) {
        acc_pts.push_back(steps[i].acc->pi_V.U);
        acc_pts.push_back(steps[i].acc->C_bar);
    }
    const std::vector<affine_t> acc_aff = batch_to_affine(acc_pts);
    const std::vector<affine_t> cp_aff = inst.c_prime_affine(c_out);
    PallasScalar s_G0 = scalar_zero(), s_G1 = scalar_zero(), s_S = scalar_zero();
    PallasScalar r_t = scalar_one();  // rho^t of the current equation
    for (size_t i = 0; i < k; i++) {
        const Accumulator& a = *steps[i].acc;
        const PallasScalar rA = r_t;
        r_t = r_t * rho;
        std::vector<PallasScalar> rE;
        for (size_t j = first[i]; j < first[i + 1]; j++) {
            rE.push_back(r_t);
            r_t = r_t * rho;
        }
        const PallasScalar rB = r_t;
        r_t = r_t * rho;
        const std::vector<PallasScalar>& al = step_alphas[i];
        // A_i and B_i's alpha^0 U0_i
        s_G0 = s_G0 - rA * a.pi_V.h[0];
        s_G1 = s_G1 - rA * a.pi_V.h[1];
        terms.aff.push_back(acc_aff[2 * i]);
        terms.sc.push_back(rA + rB * al[0]);
        // E_ij, and U_ij's + rho^tB alpha_i^j from B_i
        for (size_t j = first[i]; j < first[i + 1]; j++) terms.add_succinct(*inst.preps[j], cp_aff[j], rE[j - first[i]], rB * al[j - first[i] + 1]);
        s_S = s_S + rB * a.pi_V.w;
        terms.aff.push_back(acc_aff[2 * i + 1]);  // - C_bar_i
        terms.sc.push_back(-rB);
    }
    const std::vector<affine_t> sh = batch_to_affine({S, H});
    if (k > 0) {
        terms.aff.push_back(g[0]);
        terms.sc.push_back(s_G0);
        if (n >= 2) {
            terms.aff.push_back(g[1]);
            terms.sc.push_back(s_G1);
        }
        terms.aff.push_back(sh[0]);
        terms.sc.push_back(s_S);
    }
    const bool zero = gen.is_zero(terms, sh[1]);
    bool all_ok = true;
    for (size_t i = 0; i < k; i++) all_ok = all_ok && host_ok[i];
    if (all_ok && zero) return;

    // rejected: the steps one by one, in order, then the claims, so that (index, code) is what a loop of single verifiers
    // followed by a loop of single deciders returns
    for (size_t i = 0; i < k; i++) {
        try {
            verifier(ctx, D, *steps[i].qs, *steps[i].acc);
        } catch (const HaloFailure& e) {
            if (e.code <= HALO_REJECT_SUCCINCT && rejected_index) *rejected_index = i;
            throw;
        }
    }
    pcdl::check_in_order(ctx, claims, k, rejected_index);
    throw HaloFailure(HALO_EINTERNAL, "verify_decide_batch: the combined equation fails but every item accepts on its own");
}

void verifier_batch(halo_ctx* ctx, uint64_t D, const std::vector<Step>& steps, const PallasScalar& rho, uint64_t* rejected_index) {
    verify_decide_batch(ctx, D, steps, {}, rho, rejected_index);
}

Instance instance_from_c(const halo_instance& q) {
    return Instance{point_load(q.C), q.d, scalar_load(q.z), scalar_load(q.v), pcdl::proof_from_c(q.pi)};
}
Accumulator accumulator_from_c(const halo_accumulator& a) {
    AccumulatorHiding pv{{scalar_load(a.h0[0]), scalar_load(a.h0[1])}, point_load(a.U0), scalar_load(a.w)};
    return Accumulator{point_load(a.C_bar), a.d, scalar_load(a.z), scalar_load(a.v), pcdl::proof_from_c(a.pi), pv};
}
void accumulator_to_c(const Accumulator& a, halo_accumulator& out) {
    std::memset(&out, 0, sizeof out);
    point_store(out.C_bar, a.C_bar);
    out.d = a.d;
    scalar_store(out.z, a.z);
    scalar_store(out.v, a.v);
    pcdl::proof_to_c(a.pi, out.pi);
    for (size_t i = 0; i < 2 && i < a.pi_V.h.size(); i++) scalar_store(out.h0[i], a.pi_V.h[i]);
    point_store(out.U0, a.pi_V.U);
    scalar_store(out.w, a.pi_V.w);
}

}  // namespace acc
}  // namespace halo
