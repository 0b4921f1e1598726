// host/pcdl.cpp -- see pcdl.hpp.  Control flow follows code/src/pcdl.rs step by step; every O(n) step is a
// call into libhalo_b200.so.
#include "pcdl.hpp"

#include <algorithm>
#include <cstdint>
#include <exception>
#include <functional>
#include <optional>
#include <system_error>
#include <thread>

#include "../../include/halo_b200_test.h"
#include "pedersen.hpp"

namespace halo {
namespace pcdl {

static bool is_pow2(uint64_t n) { return n && !(n & (n - 1)); }
static uint32_t ilog2(uint64_t n) {
    uint32_t l = 0;
    while (((uint64_t)1 << (l + 1)) <= n) l++;
    return l;
}
static uint64_t degree(PolyView p) {  // DensePolynomial::degree (trailing zeros trimmed)
    uint64_t n = p.size();
    while (n > 0 && fp_is_zero(p[n - 1])) n--;
    return n ? n - 1 : 0;
}

PallasPoly HPoly::get_poly(halo_ctx* ctx) const {
    uint32_t lg_n = (uint32_t)xis.size() - 1;
    PallasPoly out((size_t)1 << lg_n);
    check_rc(ctx, halo_h_expand(ctx, reinterpret_cast<const uint64_t*>(xis.data()), lg_n, reinterpret_cast<uint64_t*>(out.data())));
    return out;
}

PallasScalar HPoly::eval(const PallasScalar& z) const {
    size_t lg_n = xis.size() - 1;
    PallasScalar one = scalar_one();
    PallasScalar v = one + xis[lg_n] * z;
    PallasScalar z_i = z;
    for (size_t i = 1; i < lg_n; i++) {
        z_i = z_i * z_i;
        v = v * (one + xis[lg_n - i] * z_i);
    }
    return v;
}

PallasPoint commit(halo_ctx* ctx, PolyView p, uint64_t d, const PallasScalar* w) {
    uint64_t n = d + 1;
    ensure(is_pow2(n), HALO_EINVAL, "d+1 is not a power of 2");  // pcdl.rs:102
    ensure(degree(p) <= d, HALO_EINVAL, "p.degree() > d");       // pcdl.rs:103
    ensure(n <= halo_num_generators(ctx), HALO_EINVAL, "d > D");  // pcdl.rs:104
    uint64_t n_coeffs = p.size() < n ? p.size() : n;
    // coeffs.resize(n, ZERO) (pcdl.rs:106-107): the zero tail is implied, not uploaded
    return pedersen::commit(ctx, w, nullptr, n, p.data(), n_coeffs, true);
}

// The polynomials of a batch of degree bound d, validated in order as commit does (the first malformed one throws), and the
// number of coefficients each uploads: coeffs.resize(n, ZERO) (pcdl.rs:106-107) implies the zero tail.
static std::vector<uint64_t> batch_lens(halo_ctx* ctx, const std::vector<PolyView>& ps, uint64_t d) {
    const uint64_t n = d + 1;
    std::vector<uint64_t> lens(ps.size());
    for (size_t j = 0; j < ps.size(); j++) {
        ensure(is_pow2(n), HALO_EINVAL, "d+1 is not a power of 2");  // pcdl.rs:102
        ensure(degree(ps[j]) <= d, HALO_EINVAL, "p.degree() > d");   // pcdl.rs:103
        ensure(n <= halo_num_generators(ctx), HALO_EINVAL, "d > D");  // pcdl.rs:104
        lens[j] = ps[j].size() < n ? ps[j].size() : n;
    }
    return lens;
}

// The uploaded prefixes (lens[j] coefficients of ps[j]) as one packed array: in place when they already lie back to back in
// memory, else copied into `copy`.  Null when there is nothing to upload.
static const PallasScalar* packed_prefixes(const std::vector<PolyView>& ps, const std::vector<uint64_t>& lens,
                                           std::vector<PallasScalar>& copy) {
    const size_t k = ps.size();
    bool packed = true;
    const PallasScalar* end = nullptr;  // one past the uploaded prefix of the last non-empty polynomial
    for (size_t j = 0; j < k; j++) {
        if (!lens[j]) continue;  // an empty polynomial uploads nothing, wherever its view points
        if (end && ps[j].data() != end) packed = false;
        end = ps[j].data() + lens[j];
    }
    size_t first = 0;  // the first polynomial with coefficients to upload anchors the packed buffer
    while (first < k && !lens[first]) first++;
    if (packed) return first < k ? ps[first].data() : nullptr;
    uint64_t total = 0;
    for (uint64_t l : lens) total += l;
    copy.resize(total);
    uint64_t o = 0;
    for (size_t j = 0; j < k; j++) {
        std::copy(ps[j].data(), ps[j].data() + lens[j], copy.begin() + o);
        o += lens[j];
    }
    return copy.data();
}

std::vector<PallasPoint> commit_batch(halo_ctx* ctx, const std::vector<PolyView>& ps, uint64_t d, const PallasScalar* ws) {
    const size_t k = ps.size();
    const std::vector<uint64_t> lens = batch_lens(ctx, ps, d);
    if (k == 0) return {};
    if (k == 1) return {commit(ctx, ps[0], d, ws)};  // the single call, exactly
    std::vector<PallasScalar> copy;
    const PallasScalar* base = packed_prefixes(ps, lens, copy);
    std::vector<uint64_t> out(12 * k);
    static const PallasScalar none = scalar_zero();
    check_rc(ctx, halo_msm_gens_many(ctx, reinterpret_cast<const uint64_t*>(base ? base : &none), lens.data(), k, out.data()));
    std::vector<PallasPoint> C(k);
    for (size_t j = 0; j < k; j++) C[j] = point_load(&out[12 * j]);
    if (ws) {  // pedersen.rs:15-16: C_j + w_j S for every j in ONE combine (host threads or k_point_combine by the output count)
        CombineList cl;
        for (size_t j = 0; j < k; j++) cl.push(C[j], point_zero(), scalar_zero(), ws[j]);
        const std::vector<affine_t> r = cl.run(ctx);
        for (size_t j = 0; j < k; j++) xyzz_from_affine(C[j].p, r[j]);
    }
    return C;
}

static EvalProof open_impl(halo_ctx* ctx, const PolyView* p, uint64_t deg, const PallasPoint& C, uint64_t d, const PallasScalar& z,
                           const PallasScalar* w, const PolyView* q, const PallasScalar* w_bar, PallasScalar* v_out);

EvalProof open(halo_ctx* ctx, PolyView p, const PallasPoint& C, uint64_t d, const PallasScalar& z, const PallasScalar* w,
               const PolyView* q, const PallasScalar* w_bar, PallasScalar* v_out) {
    return open_impl(ctx, &p, degree(p), C, d, z, w, q, w_bar, v_out);
}
EvalProof open_resident(halo_ctx* ctx, uint64_t deg, const PallasPoint& C, uint64_t d, const PallasScalar& z,
                        const PallasScalar* w, const PolyView* q, const PallasScalar* w_bar, PallasScalar* v_out) {
    return open_impl(ctx, nullptr, deg, C, d, z, w, q, w_bar, v_out);
}

BatchClaim batch_claim(halo_ctx* ctx, const std::vector<PallasPoint>& Cs, const std::vector<PallasScalar>& vs, const PallasScalar& z) {
    const size_t k = Cs.size();
    ensure(k >= 1 && vs.size() == k, HALO_EINVAL, "batch claim: no polynomial");
    // alpha binds every v_j: a prover could otherwise trade a false v_j against another
    const std::vector<affine_t> aff = batch_to_affine(Cs);
    Transcript t;
    t.scalar(z);
    for (size_t j = 0; j < k; j++) t.point_affine(aff[j]).scalar(vs[j]);
    BatchClaim r;
    r.alpha = t.finish(0);
    r.powers.resize(k);
    r.powers[0] = scalar_one();
    for (size_t j = 1; j < k; j++) r.powers[j] = r.powers[j - 1] * r.alpha;
    r.v = scalar_zero();
    for (size_t j = 0; j < k; j++) r.v = r.v + r.powers[j] * vs[j];
    r.C = point_dot(ctx, r.powers.data(), Cs, k);
    return r;
}

BatchOpening open_batch(halo_ctx* ctx, const std::vector<PolyView>& ps, const std::vector<PallasPoint>& Cs, uint64_t d,
                        const PallasScalar& z, const PallasScalar* ws, const PolyView* q, const PallasScalar* w_bar) {
    const size_t k = ps.size();
    ensure(k >= 1 && Cs.size() == k, HALO_EINVAL, "open_batch: no polynomial");
    const std::vector<uint64_t> lens = batch_lens(ctx, ps, d);
    if (ws) {  // q is drawn before alpha exists: max_j deg(p_j) coefficients, as `open` wants deg(p) >= 1 of them
        ensure(q && w_bar, HALO_EINVAL, "hiding open needs the random polynomial q and w_bar");
        uint64_t max_deg = 0;
        for (const PolyView& p : ps) max_deg = std::max(max_deg, degree(p));
        ensure(max_deg >= 1 && q->size() == max_deg, HALO_ELEN, "q must have max_j deg(p_j) coefficients");
    }
    BatchOpening r;
    if (k == 1) {  // the single call, exactly: alpha^0 = 1 makes the claim (C_0, v_0)
        r.pi = open(ctx, ps[0], Cs[0], d, z, ws, q, w_bar, &r.v);
        r.vs = {r.v};
        r.C = Cs[0];
        return r;
    }
    std::vector<PallasScalar> copy;
    const PallasScalar* base = packed_prefixes(ps, lens, copy);
    r.vs.resize(k);
    check_rc(ctx, halo_poly_eval_many(ctx, reinterpret_cast<const uint64_t*>(base), lens.data(), k, d + 1,
                                      reinterpret_cast<const uint64_t*>(&z), reinterpret_cast<uint64_t*>(r.vs.data())));
    const BatchClaim bc = batch_claim(ctx, Cs, r.vs, z);
    PallasScalar w = scalar_zero();
    if (ws)
        for (size_t j = 0; j < k; j++) w = w + bc.powers[j] * ws[j];
    uint64_t deg = 0;
    check_rc(ctx, halo_poly_combine_resident(ctx, reinterpret_cast<const uint64_t*>(&bc.alpha), &deg));
    // the top coefficients of p cancel only with negligible probability; the opening then takes the first deg(p) of q
    const PolyView qd = ws ? PolyView(q->data(), std::min<uint64_t>(deg, q->size())) : PolyView(nullptr, 0);
    PallasScalar v_dev;
    r.pi = open_resident(ctx, deg, bc.C, d, z, ws ? &w : nullptr, ws ? &qd : nullptr, w_bar, &v_dev);
    // the opening evaluates p(z) itself; it must be the claim's sum_j alpha^j v_j
    ensure(v_dev == bc.v, HALO_EINTERNAL, "open_batch: p(z) of the combined polynomial differs from sum_j alpha^j v_j");
    r.C = bc.C;
    r.v = bc.v;
    return r;
}

// ---- K3c: several points -------------------------------------------------------------------------------------------
// Every point and polynomial in some query, points distinct, no (j, t) pair twice
static void multi_validate(size_t k, const std::vector<PallasScalar>& zs, const std::vector<uint64_t>& q_poly,
                           const std::vector<uint64_t>& q_point) {
    const size_t T = zs.size(), m = q_poly.size();
    ensure(k >= 1 && T >= 1 && m >= 1 && q_point.size() == m, HALO_EINVAL, "multi-point opening: k, T and m must be at least 1");
    ensure(T <= HALO_MULTI_MAX_POINTS, HALO_EINVAL, "multi-point opening: more than HALO_MULTI_MAX_POINTS points");
    for (size_t t = 0; t < T; t++)
        for (size_t u = 0; u < t; u++) ensure(!(zs[t] == zs[u]), HALO_EINVAL, "multi-point opening: duplicate points");
    std::vector<std::pair<uint64_t, uint64_t>> pairs(m);
    std::vector<uint8_t> poly_used(k, 0), point_used(T, 0);
    for (size_t i = 0; i < m; i++) {
        ensure(q_poly[i] < k && q_point[i] < T, HALO_EINVAL, "multi-point opening: a query index is out of range");
        pairs[i] = {q_poly[i], q_point[i]};
        poly_used[q_poly[i]] = point_used[q_point[i]] = 1;
    }
    std::sort(pairs.begin(), pairs.end());
    ensure(std::adjacent_find(pairs.begin(), pairs.end()) == pairs.end(), HALO_EINVAL, "multi-point opening: a (j, t) pair repeats");
    ensure(std::count(poly_used.begin(), poly_used.end(), 0) == 0, HALO_EINVAL, "multi-point opening: a polynomial is in no query");
    ensure(std::count(point_used.begin(), point_used.end(), 0) == 0, HALO_EINVAL, "multi-point opening: a point is in no query");
}

static std::vector<PallasScalar> powers_of(const PallasScalar& x, size_t n) {
    std::vector<PallasScalar> p(n);
    if (n) p[0] = scalar_one();
    for (size_t i = 1; i < n; i++) p[i] = p[i - 1] * x;
    return p;
}

// x1 = rho_2(u64 k, u64 T, u64 m, C_0 .. C_{k-1}, z_0 .. z_{T-1}, (u64 j_i, u64 t_i, v_i) for every query)
static PallasScalar multi_x1(const std::vector<PallasPoint>& Cs, const std::vector<PallasScalar>& zs, const std::vector<uint64_t>& q_poly,
                             const std::vector<uint64_t>& q_point, const std::vector<PallasScalar>& vs) {
    Transcript t;
    t.u64(Cs.size()).u64(zs.size()).u64(q_poly.size());
    for (const affine_t& a : batch_to_affine(Cs)) t.point_affine(a);
    for (const PallasScalar& z : zs) t.scalar(z);
    for (size_t i = 0; i < q_poly.size(); i++) t.u64(q_poly[i]).u64(q_point[i]).scalar(vs[i]);
    return t.finish(2);
}

// v_hat_t = sum_{i: t_i = t} x1^i v_i
static std::vector<PallasScalar> multi_vhat(size_t T, const std::vector<uint64_t>& q_point, const std::vector<PallasScalar>& vs,
                                            const std::vector<PallasScalar>& pw1) {
    std::vector<PallasScalar> vh(T, scalar_zero());
    for (size_t i = 0; i < q_point.size(); i++) vh[q_point[i]] = vh[q_point[i]] + pw1[i] * vs[i];
    return vh;
}

static void multi_x3_check(const PallasScalar& x3, const std::vector<PallasScalar>& zs) {
    for (const PallasScalar& z : zs) ensure(!(x3 == z), HALO_EINTERNAL, "multi-point opening: x3 is one of the points");
}

// Steps 9-10 of the definition from x1, x2, x3 and the u_t
static MultiClaim multi_final(halo_ctx* ctx, const std::vector<PallasPoint>& Cs, const std::vector<PallasScalar>& zs,
                              const std::vector<uint64_t>& q_poly, const std::vector<uint64_t>& q_point, const std::vector<PallasScalar>& pw1,
                              const std::vector<PallasScalar>& vh, const PallasScalar& x2, const PallasScalar& x3, const PallasPoint& Q,
                              const std::vector<PallasScalar>& us) {
    const size_t k = Cs.size(), T = zs.size();
    Transcript tr;
    tr.scalar(x3);
    for (const PallasScalar& u : us) tr.scalar(u);
    const PallasScalar x4 = tr.finish(2);
    const std::vector<PallasScalar> pw2 = powers_of(x2, T), pw4 = powers_of(x4, T + 1);
    std::vector<PallasScalar> den(T);
    for (size_t t = 0; t < T; t++) den[t] = x3 - zs[t];
    batch_inverse(den);
    MultiClaim r;
    r.x3 = x3;
    r.v = scalar_zero();
    for (size_t t = 0; t < T; t++) r.v = r.v + pw2[t] * (us[t] - vh[t]) * den[t] + pw4[t + 1] * us[t];  // q_hat + sum x4^(t+1) u_t
    r.cs.assign(k, scalar_zero());
    for (size_t i = 0; i < q_poly.size(); i++) r.cs[q_poly[i]] = r.cs[q_poly[i]] + pw4[q_point[i] + 1] * pw1[i];
    std::vector<PallasPoint> pts(1, Q);
    pts.insert(pts.end(), Cs.begin(), Cs.end());
    std::vector<PallasScalar> sc(1, scalar_one());
    sc.insert(sc.end(), r.cs.begin(), r.cs.end());
    r.C = point_dot(ctx, sc.data(), pts, k + 1);
    return r;
}

MultiClaim multi_claim(halo_ctx* ctx, const std::vector<PallasPoint>& Cs, const std::vector<PallasScalar>& zs,
                       const std::vector<uint64_t>& q_poly, const std::vector<uint64_t>& q_point, const std::vector<PallasScalar>& vs,
                       const PallasPoint& Q, const std::vector<PallasScalar>& us) {
    multi_validate(Cs.size(), zs, q_poly, q_point);
    ensure(vs.size() == q_poly.size() && us.size() == zs.size(), HALO_EINVAL, "multi_claim: one v per query and one u per point");
    const PallasScalar x1 = multi_x1(Cs, zs, q_poly, q_point, vs);
    const std::vector<PallasScalar> pw1 = powers_of(x1, q_poly.size());
    const PallasScalar x2 = Transcript().scalar(x1).finish(2);
    const PallasScalar x3 = Transcript().scalar(x2).point(Q).finish(2);
    multi_x3_check(x3, zs);
    return multi_final(ctx, Cs, zs, q_poly, q_point, pw1, multi_vhat(zs.size(), q_point, vs, pw1), x2, x3, Q, us);
}

MultiOpening open_multi(halo_ctx* ctx, const std::vector<PolyView>& ps, const std::vector<PallasPoint>& Cs, uint64_t d,
                        const std::vector<PallasScalar>& zs, const std::vector<uint64_t>& q_poly, const std::vector<uint64_t>& q_point,
                        const PallasScalar* ws, const PallasScalar* w_Q, const PolyView* q, const PallasScalar* w_bar) {
    const size_t k = ps.size(), T = zs.size(), m = q_poly.size();
    ensure(k >= 1 && Cs.size() == k, HALO_EINVAL, "open_multi: no polynomial");
    const std::vector<uint64_t> lens = batch_lens(ctx, ps, d);
    multi_validate(k, zs, q_poly, q_point);
    if (ws) {  // q is drawn before any challenge exists: max_j deg(p_j) coefficients, as in open_batch
        ensure(w_Q && q && w_bar, HALO_EINVAL, "hiding open needs w_Q, the random polynomial q and w_bar");
        uint64_t max_deg = 0;
        for (const PolyView& p : ps) max_deg = std::max(max_deg, degree(p));
        ensure(max_deg >= 1 && q->size() == max_deg, HALO_ELEN, "q must have max_j deg(p_j) coefficients");
    }
    std::vector<PallasScalar> copy;
    const PallasScalar* base = packed_prefixes(ps, lens, copy);
    check_rc(ctx, halo_poly_upload(ctx, reinterpret_cast<const uint64_t*>(base), lens.data(), k, d + 1));
    const uint64_t* zp = reinterpret_cast<const uint64_t*>(zs.data());
    MultiOpening r;
    r.vs.resize(m);
    check_rc(ctx, halo_poly_eval_queries(ctx, zp, T, q_poly.data(), q_point.data(), m, reinterpret_cast<uint64_t*>(r.vs.data())));

    const PallasScalar x1 = multi_x1(Cs, zs, q_poly, q_point, r.vs);
    const std::vector<PallasScalar> pw1 = powers_of(x1, m), vh = multi_vhat(T, q_point, r.vs, pw1);
    const PallasScalar x2 = Transcript().scalar(x1).finish(2);
    const std::vector<PallasScalar> pw2 = powers_of(x2, T);
    std::vector<PallasScalar> rems(T);
    uint64_t Qb[12];
    check_rc(ctx, halo_poly_quotient(ctx, zp, reinterpret_cast<const uint64_t*>(pw2.data()), T, q_poly.data(), q_point.data(),
                                     reinterpret_cast<const uint64_t*>(pw1.data()), m, reinterpret_cast<uint64_t*>(rems.data()), Qb));
    for (size_t t = 0; t < T; t++)  // f_t(z_t), the remainder of the division, must be the claimed v_hat_t
        ensure(rems[t] == vh[t], HALO_EINTERNAL, "open_multi: a remainder of the division differs from sum x1^i v_i");
    r.Q = point_load(Qb);
    if (ws) {
        PallasPoint S, H;
        params_SH(ctx, S, H);
        r.Q = r.Q + S * (*w_Q);
    }
    const PallasScalar x3 = Transcript().scalar(x2).point(r.Q).finish(2);
    multi_x3_check(x3, zs);

    // u_t = f_t(x3) from every polynomial at x3
    std::vector<uint64_t> all(k), zero(k, 0);
    for (size_t j = 0; j < k; j++) all[j] = j;
    std::vector<PallasScalar> ev(k);
    check_rc(ctx, halo_poly_eval_queries(ctx, reinterpret_cast<const uint64_t*>(&x3), 1, all.data(), zero.data(), k,
                                         reinterpret_cast<uint64_t*>(ev.data())));
    r.us.assign(T, scalar_zero());
    for (size_t i = 0; i < m; i++) r.us[q_point[i]] = r.us[q_point[i]] + pw1[i] * ev[q_poly[i]];
    r.claim = multi_final(ctx, Cs, zs, q_poly, q_point, pw1, vh, x2, x3, r.Q, r.us);

    PallasScalar w = scalar_zero();
    if (ws) {
        w = *w_Q;
        for (size_t j = 0; j < k; j++) w = w + r.claim.cs[j] * ws[j];
    }
    const PallasScalar one = scalar_one();
    uint64_t deg = 0;
    check_rc(ctx, halo_poly_lincomb_resident(ctx, reinterpret_cast<const uint64_t*>(r.claim.cs.data()),
                                             reinterpret_cast<const uint64_t*>(&one), &deg));
    const PolyView qd = ws ? PolyView(q->data(), std::min<uint64_t>(deg, q->size())) : PolyView(nullptr, 0);
    PallasScalar v_dev;
    r.pi = open_resident(ctx, deg, r.claim.C, d, x3, ws ? &w : nullptr, ws ? &qd : nullptr, w_bar, &v_dev);
    // the opening evaluates P(x3) itself; it must be the claim's v
    ensure(v_dev == r.claim.v, HALO_EINTERNAL, "open_multi: P(x3) of the combined polynomial differs from v");
    return r;
}

static EvalProof open_impl(halo_ctx* ctx, const PolyView* p, uint64_t deg, const PallasPoint& C, uint64_t d, const PallasScalar& z,
                           const PallasScalar* w, const PolyView* q, const PallasScalar* w_bar, PallasScalar* v_out) {
    uint64_t n = d + 1;
    ensure(is_pow2(n), HALO_EINVAL, "d+1 is not a power of 2");  // pcdl.rs:130
    ensure(deg <= d, HALO_EINVAL, "p.degree() > d");             // pcdl.rs:131
    ensure(n <= halo_num_generators(ctx), HALO_EINVAL, "d > D");  // pcdl.rs:132
    uint32_t lg_n = ilog2(n);
    PallasPoint S, H;
    params_SH(ctx, S, H);

    // device state: c (zero padded), G, z-powers; v = p(z) (pcdl.rs:135, :183-186)
    halo_ipa* st = nullptr;
    uint64_t vbuf[4];
    if (p) {
        uint64_t n_coeffs = p->size() < n ? p->size() : n;
        check_rc(ctx, halo_ipa_begin(ctx, reinterpret_cast<const uint64_t*>(p->data()), n_coeffs, n,
                                     reinterpret_cast<const uint64_t*>(&z), &st, vbuf));
    } else {
        check_rc(ctx, halo_ipa_begin_resident(ctx, n, reinterpret_cast<const uint64_t*>(&z), &st, vbuf));
    }
    struct Guard {
        halo_ipa* s;
        ~Guard() { halo_ipa_destroy(s); }
    } guard{st};
    PallasScalar v = scalar_load(vbuf);
    if (v_out) *v_out = v;

    EvalProof pi;
    PallasPoint C_prime = C;
    if (w) {  // pcdl.rs:137-164
        ensure(q && w_bar, HALO_EINVAL, "hiding open needs the random polynomial q and w_bar");
        ensure(deg >= 1 && q->size() == deg, HALO_ELEN, "q must have deg(p) coefficients (PallasPoly::rand(p.degree() - 1))");
        // p_bar = q (X - z); C_bar = commit(p_bar, d, w_bar)  (:140-149)
        uint64_t cb[12];
        check_rc(ctx, halo_ipa_blind_commit(st, reinterpret_cast<const uint64_t*>(q->data()), q->size(), cb));
        PallasPoint C_bar = S * (*w_bar) + point_load(cb);
        // alpha = rho_0(C, z, v, C_bar)  (:153)
        PallasScalar a = Transcript().point(C).scalar(z).scalar(v).point(C_bar).finish(0);
        // p' = p + alpha p_bar  (:156)
        check_rc(ctx, halo_ipa_blind_apply(st, reinterpret_cast<const uint64_t*>(&a)));
        // w' = w_bar alpha + w ; C' = C + alpha C_bar - w' S  (:159-162)
        PallasScalar w_prime = (*w_bar) * a + (*w);
        C_prime = C + C_bar * a - S * w_prime;
        pi.hiding = true;
        pi.C_bar = C_bar;
        pi.w_prime = w_prime;
    }

    // xi_0 = rho_0(C', z, v); H' = xi_0 H  (:180-181)
    PallasScalar xi_i = Transcript().point(C_prime).scalar(z).scalar(v).finish(0);
    PallasPoint H_prime = H * xi_i;
    uint64_t hp[12];
    point_store(hp, H_prime);
    check_rc(ctx, halo_ipa_set_hprime(st, hp));

    pi.Ls.reserve(lg_n);
    pi.Rs.reserve(lg_n);
    for (uint32_t round = 0; round < lg_n; round++) {  // :195-227
        uint64_t Lb[12], Rb[12];
        check_rc(ctx, halo_ipa_round_lr(st, Lb, Rb));  // :199-209
        PallasPoint L = point_load(Lb), R = point_load(Rb);
        pi.Ls.push_back(L);
        pi.Rs.push_back(R);
        PallasScalar xi_next = Transcript().scalar(xi_i).point(L).point(R).finish(0);  // :212
        ensure(!fp_is_zero(xi_next), HALO_EINVAL, "challenge is zero (inverse().unwrap())");  // :213
        PallasScalar xi_next_inv = scalar_inverse(xi_next);
        xi_i = xi_next;
        check_rc(ctx, halo_ipa_round_fold(st, reinterpret_cast<const uint64_t*>(&xi_next),
                                          reinterpret_cast<const uint64_t*>(&xi_next_inv)));  // :216-224
    }
    uint64_t Ub[12], cb[4];
    check_rc(ctx, halo_ipa_finish(st, Ub, cb));  // :230-231
    pi.U = point_load(Ub);
    pi.c = scalar_load(cb);
    return pi;
}

// succinct_check (pcdl.rs:252-314) up to its group equation is succinct_alpha, C' (:272-279) and succinct_finish; the group
// equation is left as one small MSM:
//   C_lg == c U + v' H'   <=>   C' + sum_k scalars[k] * aff[k] == 0
PallasScalar succinct_alpha(halo_ctx* ctx, const PallasPoint& C, uint64_t d, const PallasScalar& z, const PallasScalar& v,
                            const EvalProof& pi) {
    uint64_t n = d + 1;
    ensure(is_pow2(n), HALO_EINVAL, "d+1 is not a power of 2!");           // :261
    ensure(n <= halo_num_generators(ctx), HALO_EINVAL, "d was larger than D!");  // :262
    uint32_t lg_n = ilog2(n);
    ensure(pi.Ls.size() == lg_n && pi.Rs.size() == lg_n, HALO_EINVAL, "proof has the wrong number of rounds");
    return pi.hiding ? Transcript().point(C).scalar(z).scalar(v).point(pi.C_bar).finish(0) : scalar_zero();  // :272-276
}

SuccinctPrep succinct_finish(halo_ctx* ctx, const PallasPoint& C_prime, uint64_t d, const PallasScalar& z, const PallasScalar& v,
                             const EvalProof& pi) {
    uint32_t lg_n = ilog2(d + 1);
    PallasPoint S, H;
    params_SH(ctx, S, H);
    // xi_0, challenges (:282-293); the group arithmetic of :285-298 and :307-310 is one small MSM:
    //   C_lg == c U + v' H'   <=>   C' + (xi_0 v - xi_0 v') H + sum_i (xi_{i+1}^-1 L_i + xi_{i+1} R_i) - c U == 0
    // all points that enter the transcript or the MSM are normalised with ONE field inversion (the reference normalises
    // each point separately inside serialize_compressed; same bytes)
    std::vector<PallasPoint> pts;
    pts.reserve(2 * (size_t)lg_n + 2);
    for (uint32_t i = 0; i < lg_n; i++) {
        pts.push_back(pi.Ls[i]);
        pts.push_back(pi.Rs[i]);
    }
    pts.push_back(H);
    pts.push_back(pi.U);
    std::vector<affine_t> aff = batch_to_affine(pts);
    std::vector<uint8_t> inf(aff.size());
    for (size_t i = 0; i < aff.size(); i++) inf[i] = affine_is_inf(aff[i]) ? 1 : 0;
    std::vector<PallasScalar> xis;
    xis.reserve(lg_n + 1);
    xis.push_back(Transcript().point(C_prime).scalar(z).scalar(v).finish(0));
    for (uint32_t i = 0; i < lg_n; i++) {
        PallasScalar xi_next = Transcript().scalar(xis[i]).point_affine(aff[2 * i]).point_affine(aff[2 * i + 1]).finish(0);  // :293
        ensure(!fp_is_zero(xi_next), HALO_EINVAL, "challenge is zero (inverse().unwrap())");                                 // :297
        xis.push_back(xi_next);
    }
    std::vector<PallasScalar> inv(xis.begin() + 1, xis.end());
    batch_inverse(inv);  // xi_{i+1}^-1, one inversion for all rounds
    std::vector<PallasScalar> scalars;
    scalars.reserve(2 * (size_t)lg_n + 2);
    for (uint32_t i = 0; i < lg_n; i++) {
        scalars.push_back(inv[i]);      // xi_{i+1}^-1 L_i
        scalars.push_back(xis[i + 1]);  // xi_{i+1}   R_i
    }
    HPoly h(xis);                                   // :301
    PallasScalar v_prime = pi.c * h.eval(z);        // :304
    scalars.push_back(xis[0] * v - xis[0] * v_prime);  // v H' - v' H' with H' = xi_0 H  (:285, :288, :308)
    scalars.push_back(-pi.c);                          // - c U
    return SuccinctPrep{std::move(h), pi.U, C_prime, std::move(aff), std::move(inf), std::move(scalars)};
}

static SuccinctPrep succinct_prepare(halo_ctx* ctx, const PallasPoint& C, uint64_t d, const PallasScalar& z, const PallasScalar& v,
                                     const EvalProof& pi) {
    PallasScalar a = succinct_alpha(ctx, C, d, z, v, pi);
    // C' = C + alpha C_bar - w' S  (:272-279)
    PallasPoint C_prime = C;
    if (pi.hiding) {
        PallasPoint S, H;
        params_SH(ctx, S, H);
        C_prime = C + pi.C_bar * a - S * pi.w_prime;
    }
    return succinct_finish(ctx, C_prime, d, z, v, pi);
}

std::vector<affine_t> combine(halo_ctx* ctx, const std::vector<PallasPoint>& P, const std::vector<PallasPoint>& Q,
                              const std::vector<PallasScalar>& a, const std::vector<PallasScalar>& b) {
    const size_t n = P.size();
    std::vector<uint64_t> pj(12 * n), qj(12 * n);
    for (size_t o = 0; o < n; o++) {
        point_store(&pj[12 * o], P[o]);
        point_store(&qj[12 * o], Q[o]);
    }
    std::vector<affine_t> out(n);
    check_rc(ctx, halo_test_point_combine(ctx, -1, pj.data(), qj.data(), reinterpret_cast<const uint64_t*>(a.data()),
                                          reinterpret_cast<const uint64_t*>(b.data()), n, reinterpret_cast<uint64_t*>(out.data())));
    return out;
}

std::vector<std::exception_ptr> parallel_each(size_t k, const std::function<void(size_t)>& f) {
    std::vector<std::exception_ptr> errs(k);
    auto work = [&](size_t t, size_t T) {
        for (size_t j = t; j < k; j += T) {
            try {
                f(j);
            } catch (...) {
                errs[j] = std::current_exception();
            }
        }
    };
    const size_t hw = std::thread::hardware_concurrency();
    const size_t T = std::min(k, std::max<size_t>(1, std::min<size_t>(hw, 16)));
    std::vector<std::thread> th;
    std::vector<size_t> unspawned;
    for (size_t t = 1; t < T; t++) {
        try {
            th.emplace_back(work, t, T);
        } catch (const std::system_error&) {
            unspawned.push_back(t);  // no thread available: this thread takes that share as well
        }
    }
    work(0, T);
    for (size_t t : unspawned) work(t, T);
    for (auto& x : th) x.join();
    return errs;
}

size_t first_error(const std::vector<std::exception_ptr>& errs) {
    for (size_t j = 0; j < errs.size(); j++)
        if (errs[j]) return j;
    return errs.size();
}

std::pair<HPoly, PallasPoint> succinct_check(halo_ctx* ctx, const PallasPoint& C, uint64_t d, const PallasScalar& z,
                                             const PallasScalar& v, const EvalProof& pi) {
    SuccinctPrep sp = succinct_prepare(ctx, C, d, z, v, pi);
    uint64_t out[12];
    check_rc(ctx, halo_msm(ctx, reinterpret_cast<const uint64_t*>(sp.aff.data()), sp.inf.data(),
                           reinterpret_cast<const uint64_t*>(sp.scalars.data()), sp.aff.size(), out));
    PallasPoint lhs = sp.C_prime + point_load(out);
    ensure(xyzz_is_inf(lhs.p), HALO_REJECT_SUCCINCT, "C_(log_n) != CM.Commit_Sigma(c || v')");  // :307-310
    return {sp.h, sp.U};                                                                        // :313
}

SuccinctMany succinct_check_many(halo_ctx* ctx, const std::vector<Query>& qs, const PolyView* commit_p, uint64_t commit_d) {
    std::vector<SuccinctPrep> preps;
    preps.reserve(qs.size());
    for (const Query& q : qs) preps.push_back(succinct_prepare(ctx, *q.C, q.d, *q.z, *q.v, *q.pi));
    std::vector<halo_msm_desc> descs;
    for (const SuccinctPrep& sp : preps)
        descs.push_back(halo_msm_desc{reinterpret_cast<const uint64_t*>(sp.aff.data()), sp.inf.data(),
                                      reinterpret_cast<const uint64_t*>(sp.scalars.data()), sp.aff.size(), 0});
    if (commit_p) {  // pcdl::commit without hiding: <coeffs, GS[0..)> over the resident generators
        uint64_t n = commit_d + 1;
        ensure(is_pow2(n), HALO_EINVAL, "d+1 is not a power of 2");          // pcdl.rs:102
        ensure(degree(*commit_p) <= commit_d, HALO_EINVAL, "p.degree() > d");  // pcdl.rs:103
        ensure(n <= halo_num_generators(ctx), HALO_EINVAL, "d > D");          // pcdl.rs:104
        uint64_t n_coeffs = commit_p->size() < n ? commit_p->size() : n;
        ensure(n_coeffs <= 4096, HALO_EINVAL, "succinct_check_many: the commitment riding along must be short");
        descs.push_back(halo_msm_desc{nullptr, nullptr, reinterpret_cast<const uint64_t*>(commit_p->data()), n_coeffs, 0});
    }
    std::vector<uint64_t> out(12 * descs.size() + 12);
    check_rc(ctx, halo_msm_multi(ctx, descs.data(), (uint32_t)descs.size(), out.data()));
    SuccinctMany r;
    for (size_t i = 0; i < preps.size(); i++) {
        PallasPoint lhs = preps[i].C_prime + point_load(&out[12 * i]);
        r.accept.push_back(xyzz_is_inf(lhs.p));  // :307-310
        r.hu.emplace_back(preps[i].h, preps[i].U);
    }
    if (commit_p) r.commitment = point_load(&out[12 * preps.size()]);
    return r;
}

void check(halo_ctx* ctx, const PallasPoint& C, uint64_t d, const PallasScalar& z, const PallasScalar& v,
           const EvalProof& pi) {
    // succinct_check (:332) and comm = pedersen::commit(None, GS[0..d+1], h.get_poly().coeffs) (:338).  The challenges
    // (hence h) need only the transcript, so the small MSM of the succinct check and the expansion + MSM <G, h> run
    // concurrently on the device; the two `ensure!`s are evaluated in the reference's order.
    SuccinctPrep sp = succinct_prepare(ctx, C, d, z, v, pi);
    uint64_t out_h[12], out_s[12];
    check_rc(ctx, halo_h_msm_with(ctx, reinterpret_cast<const uint64_t*>(sp.h.xis.data()), (uint32_t)sp.h.xis.size() - 1,
                                  reinterpret_cast<const uint64_t*>(sp.aff.data()), sp.inf.data(),
                                  reinterpret_cast<const uint64_t*>(sp.scalars.data()), sp.aff.size(), out_h, out_s));
    PallasPoint lhs = sp.C_prime + point_load(out_s);
    ensure(xyzz_is_inf(lhs.p), HALO_REJECT_SUCCINCT, "C_(log_n) != CM.Commit_Sigma(c || v')");  // :307-310
    ensure(sp.U == point_load(out_h), HALO_REJECT_U, "U != CM.Commit(ck, h_vec)");                // :339
}

void QueryBatch::validate(halo_ctx* ctx, bool finish_plain) {
    const size_t k = qs.size();
    alphas.assign(k, scalar_zero());
    errs2.assign(k, nullptr);
    slot.assign(k, SIZE_MAX);
    preps.clear();
    preps.resize(k);
    errs1 = parallel_each(k, [&](size_t j) {
        const Query& q = qs[j];
        alphas[j] = succinct_alpha(ctx, *q.C, q.d, *q.z, *q.v, *q.pi);
        if (finish_plain && !q.pi->hiding) finish(ctx, j, {});
    });
    valid = first_error(errs1);
}

void QueryBatch::request(CombineList& cl) {
    for (size_t j = 0; j < valid; j++)
        if (qs[j].pi->hiding && !errs2[j]) slot[j] = cl.push(*qs[j].C, qs[j].pi->C_bar, alphas[j], -qs[j].pi->w_prime);
}

void QueryBatch::finish(halo_ctx* ctx, size_t j, const std::vector<affine_t>& c_out) {
    if (preps[j] || errs2[j]) return;
    const Query& q = qs[j];
    PallasPoint C_prime = *q.C;
    if (slot[j] != SIZE_MAX) xyzz_from_affine(C_prime.p, c_out[slot[j]]);
    try {
        preps[j].emplace(succinct_finish(ctx, C_prime, q.d, *q.z, *q.v, *q.pi));
    } catch (...) {
        errs2[j] = std::current_exception();
    }
}

bool QueryBatch::failed() const { return valid < qs.size() || first_error(errs2) < qs.size(); }

void QueryBatch::rethrow_first() const {
    for (size_t j = 0; j < valid; j++)
        if (errs2[j]) std::rethrow_exception(errs2[j]);
    if (valid < qs.size()) std::rethrow_exception(errs1[valid]);
}

std::vector<affine_t> QueryBatch::c_prime_affine(const std::vector<affine_t>& c_out) const {
    std::vector<affine_t> out(qs.size());  // the combined ones as they come, the others (C' = C) normalised together
    std::vector<PallasPoint> plain;
    std::vector<size_t> plain_at;
    for (size_t j = 0; j < qs.size(); j++) {
        if (slot[j] != SIZE_MAX)
            out[j] = c_out[slot[j]];
        else
            plain.push_back(preps[j]->C_prime), plain_at.push_back(j);
    }
    const std::vector<affine_t> plain_aff = batch_to_affine(plain);
    for (size_t i = 0; i < plain_at.size(); i++) out[plain_at[i]] = plain_aff[i];
    return out;
}

void BatchTerms::add_succinct(const SuccinctPrep& sp, const affine_t& c_prime, const PallasScalar& re, const PallasScalar& u_extra) {
    const size_t lr = sp.aff.size() - 2;  // L_0, R_0, .., then H, U
    for (size_t l = 0; l < lr; l++) {
        aff.push_back(sp.aff[l]);
        sc.push_back(re * sp.scalars[l]);
    }
    s_H = s_H + re * sp.scalars[lr];
    aff.push_back(sp.aff[lr + 1]);
    sc.push_back(re * sp.scalars[lr + 1] + u_extra);
    aff.push_back(c_prime);
    sc.push_back(re);
}

void BatchTerms::add_claims(const QueryBatch& qb, const std::vector<affine_t>& c_aff, PallasScalar r, const PallasScalar& rho) {
    for (size_t j = 0; j < qb.qs.size(); j++) {
        const SuccinctPrep& sp = *qb.preps[j];
        const PallasScalar rf = r * rho;
        add_succinct(sp, c_aff[j], r, rf);  // U_j: - rho^t c_j from E_j, + rho^(t+1) from F_j
        lgs.push_back((uint32_t)sp.h.xis.size() - 1);
        xis.insert(xis.end(), sp.h.xis.begin(), sp.h.xis.end());
        weights.push_back(-rf);
        r = rf * rho;
    }
}

GeneratorPart::~GeneratorPart() {
    if (ticket_ < 0) return;
    uint64_t out[12];
    halo_h_msm_batch_collect(ctx_, ticket_, nullptr, nullptr, nullptr, 0, out);
}

void GeneratorPart::submit(const BatchTerms& t) {
    check_rc(ctx_, halo_h_msm_batch_submit(ctx_, reinterpret_cast<const uint64_t*>(t.xis.data()), t.lgs.data(),
                                           reinterpret_cast<const uint64_t*>(t.weights.data()), t.lgs.size(), &ticket_));
}

bool GeneratorPart::is_zero(BatchTerms& t, const affine_t& H) {
    t.aff.push_back(H);  // H, the same point in every succinct equation
    t.sc.push_back(t.s_H);
    std::vector<uint8_t> inf(t.aff.size());
    for (size_t i = 0; i < t.aff.size(); i++) inf[i] = affine_is_inf(t.aff[i]) ? 1 : 0;
    const int ticket = ticket_;
    ticket_ = -1;
    uint64_t out[12];
    check_rc(ctx_, halo_h_msm_batch_collect(ctx_, ticket, reinterpret_cast<const uint64_t*>(t.aff.data()), inf.data(),
                                            reinterpret_cast<const uint64_t*>(t.sc.data()), t.aff.size(), out));
    return xyzz_is_inf(point_load(out).p);
}

void check_in_order(halo_ctx* ctx, const std::vector<Query>& qs, uint64_t index_base, uint64_t* rejected_index) {
    for (size_t j = 0; j < qs.size(); j++) {
        try {
            check(ctx, *qs[j].C, qs[j].d, *qs[j].z, *qs[j].v, *qs[j].pi);
        } catch (const HaloFailure& e) {
            if (e.code <= HALO_REJECT_SUCCINCT && rejected_index) *rejected_index = index_base + j;
            throw;
        }
    }
}

void check_batch(halo_ctx* ctx, const std::vector<Query>& qs, const PallasScalar& rho, uint64_t* rejected_index) {
    ensure(!fp_is_zero(rho), HALO_EINVAL, "rho is zero");
    if (qs.empty()) return;
    PallasPoint S, H;
    params_SH(ctx, S, H);  // missing parameters fail here, before any worker thread reads the context
    // the transcript of check, unchanged, spread over host threads: the claims without hiding in one pass; C' = C + alpha C_bar
    // - w' S of the hiding ones in ONE combine call (on the device from "combine_min_outputs"), then their transcripts
    QueryBatch qb;
    qb.qs = qs;
    qb.validate(ctx, true);
    CombineList cl;
    qb.request(cl);
    const std::vector<affine_t> c_out = cl.run(ctx);
    parallel_each(qb.valid, [&](size_t j) { qb.finish(ctx, j, c_out); });
    qb.rethrow_first();

    // sum_j rho^2j E_j + rho^(2j+1) F_j with E_j = C'_j + sum_i s_{j,i} P_{j,i} (L, R, H, U) and F_j = U_j - <G, h_j>
    BatchTerms t;
    t.add_claims(qb, qb.c_prime_affine(c_out), scalar_one(), rho);
    GeneratorPart gen(ctx);
    gen.submit(t);
    if (gen.is_zero(t, batch_to_affine({S, H})[1])) return;

    // rejected: the claims one by one, in order, so that (index, code) is what a loop of single deciders returns
    check_in_order(ctx, qs, 0, rejected_index);
    throw HaloFailure(HALO_EINTERNAL, "check_batch: the combined equation fails but every claim accepts on its own");
}

EvalProof proof_from_c(const halo_eval_proof& p) {
    EvalProof r;
    ensure(p.lg_n <= HALO_MAX_LG, HALO_EINVAL, "lg_n too large");
    for (uint32_t i = 0; i < p.lg_n; i++) {
        r.Ls.push_back(point_load(p.Ls[i]));
        r.Rs.push_back(point_load(p.Rs[i]));
    }
    r.U = point_load(p.U);
    r.c = scalar_load(p.c);
    r.hiding = p.hiding != 0;
    if (r.hiding) {
        r.C_bar = point_load(p.C_bar);
        r.w_prime = scalar_load(p.w_prime);
    }
    return r;
}
void proof_to_c(const EvalProof& p, halo_eval_proof& out) {
    std::memset(&out, 0, sizeof out);
    out.lg_n = (uint32_t)p.Ls.size();
    out.hiding = p.hiding ? 1 : 0;
    for (size_t i = 0; i < p.Ls.size(); i++) {
        point_store(out.Ls[i], p.Ls[i]);
        point_store(out.Rs[i], p.Rs[i]);
    }
    point_store(out.U, p.U);
    scalar_store(out.c, p.c);
    if (p.hiding) {
        point_store(out.C_bar, p.C_bar);
        scalar_store(out.w_prime, p.w_prime);
    }
}

}  // namespace pcdl
}  // namespace halo
