// host/pcdl.hpp -- host mirror of code/src/pcdl.rs (Bulletproofs-style polynomial commitment, DL based).
#pragma once
#include <exception>
#include <functional>
#include <optional>

#include "../../include/halo_pcdl.h"
#include "group.hpp"

namespace halo {
namespace pcdl {

// pcdl.rs:22-30
struct EvalProof {
    std::vector<PallasPoint> Ls, Rs;
    PallasPoint U;
    PallasScalar c;
    bool hiding = false;  // C_bar / w_prime are Some(..)
    PallasPoint C_bar;
    PallasScalar w_prime;
};

// pcdl.rs:44-92
struct HPoly {
    std::vector<PallasScalar> xis;
    explicit HPoly(std::vector<PallasScalar> x) : xis(std::move(x)) {}
    // pcdl.rs:56-77: coefficient vector (n = 2^lg n elements), expanded on the device
    PallasPoly get_poly(halo_ctx* ctx) const;
    // pcdl.rs:79-91
    PallasScalar eval(const PallasScalar& z) const;
};

// pcdl.rs:99-110
PallasPoint commit(halo_ctx* ctx, PolyView p, uint64_t d, const PallasScalar* w);
// `commit` of every polynomial (w: one blinding scalar per polynomial, or null): validated in order as commit does, then one
// halo_msm_gens_many over all of them and w_j S added by one `combine` call (DESIGN.md K2c)
std::vector<PallasPoint> commit_batch(halo_ctx* ctx, const std::vector<PolyView>& ps, uint64_t d, const PallasScalar* ws);
// pcdl.rs:120-242; rng draws made explicit: q (deg p coefficients), w_bar.  v_out (nullable) receives v = p(z).
EvalProof open(halo_ctx* ctx, PolyView p, const PallasPoint& C, uint64_t d, const PallasScalar& z, const PallasScalar* w,
               const PolyView* q, const PallasScalar* w_bar, PallasScalar* v_out = nullptr);
// Same for a polynomial of degree `deg` that already sits on the device (halo_h_lincomb_resident): acc.rs:209.
EvalProof open_resident(halo_ctx* ctx, uint64_t deg, const PallasPoint& C, uint64_t d, const PallasScalar& z,
                        const PallasScalar* w, const PolyView* q, const PallasScalar* w_bar, PallasScalar* v_out = nullptr);

// Batch opening at one point (DESIGN.md K3b; the reference has none).  batch_claim reduces the claims (C_j, z, v_j) to one:
// alpha = rho_0(z, C_0, v_0, .., C_{k-1}, v_{k-1}), C = sum_j alpha^j C_j, v = sum_j alpha^j v_j; powers[j] = alpha^j.
struct BatchClaim {
    PallasScalar alpha, v;
    PallasPoint C;
    std::vector<PallasScalar> powers;
};
BatchClaim batch_claim(halo_ctx* ctx, const std::vector<PallasPoint>& Cs, const std::vector<PallasScalar>& vs, const PallasScalar& z);
// v_j = p_j(z) for every polynomial, then `open` of p = sum_j alpha^j p_j against the batch claim (C, v), with
// w = sum_j alpha^j w_j when ws is given; q carries max_j deg(p_j) coefficients, of which the opening uses the first deg(p).
// The polynomials are validated in order as commit_batch does, before any device work.  k = 1 is `open` itself.
struct BatchOpening {
    std::vector<PallasScalar> vs;
    PallasPoint C;
    PallasScalar v;
    EvalProof pi;
};
BatchOpening open_batch(halo_ctx* ctx, const std::vector<PolyView>& ps, const std::vector<PallasPoint>& Cs, uint64_t d,
                        const PallasScalar& z, const PallasScalar* ws, const PolyView* q, const PallasScalar* w_bar);

// Batch opening at several points (DESIGN.md K3c, include/halo_pcdl.h halo_pcdl_open_multi; the reference has none).  Query i
// opens polynomial q_poly[i] at zs[q_point[i]].  multi_claim is the verifier's side: the claims (C_j, z_t, v_i) with the
// prover's Q and u_t reduced to the one PCDL claim (C, x3, v); c_j are the weights of P = q + sum_j c_j p_j.  Both validate
// the queries (HALO_EINVAL) and fail with HALO_EINTERNAL when x3 is one of the points.
struct MultiClaim {
    PallasPoint C;
    PallasScalar x3, v;
    std::vector<PallasScalar> cs;
};
MultiClaim multi_claim(halo_ctx* ctx, const std::vector<PallasPoint>& Cs, const std::vector<PallasScalar>& zs,
                       const std::vector<uint64_t>& q_poly, const std::vector<uint64_t>& q_point, const std::vector<PallasScalar>& vs,
                       const PallasPoint& Q, const std::vector<PallasScalar>& us);
// vs[i] = p_{q_poly[i]}(z_{q_point[i]}), the quotient's commitment Q, us[t] = f_t(x3) and the proof of the final claim.  Hiding
// iff ws is given: w_Q blinds Q, q holds max_j deg(p_j) coefficients (the opening uses the first deg(P)), w_bar as in open.
struct MultiOpening {
    std::vector<PallasScalar> vs, us;
    PallasPoint Q;
    MultiClaim claim;
    EvalProof pi;
};
MultiOpening open_multi(halo_ctx* ctx, const std::vector<PolyView>& ps, const std::vector<PallasPoint>& Cs, uint64_t d,
                        const std::vector<PallasScalar>& zs, const std::vector<uint64_t>& q_poly, const std::vector<uint64_t>& q_point,
                        const PallasScalar* ws, const PallasScalar* w_Q, const PolyView* q, const PallasScalar* w_bar);
// succinct_check (pcdl.rs:252-314) without its group equation, in two halves around C' = C + alpha C_bar - w' S (:272-279) so
// that a batch can compute every C' with one `combine` call.  succinct_alpha validates (d + 1 a power of two, d <= D, the
// number of rounds) and returns alpha = rho_0(C, z, v, C_bar) of a hiding proof (zero otherwise); succinct_finish runs the rest
// of the transcript from C' and leaves the group equation as C' + sum_k scalars[k] aff[k] == O (aff: L_0, R_0, .., H, U).
struct SuccinctPrep {
    HPoly h;
    PallasPoint U, C_prime;
    std::vector<affine_t> aff;
    std::vector<uint8_t> inf;
    std::vector<PallasScalar> scalars;
};
PallasScalar succinct_alpha(halo_ctx* ctx, const PallasPoint& C, uint64_t d, const PallasScalar& z, const PallasScalar& v,
                            const EvalProof& pi);
SuccinctPrep succinct_finish(halo_ctx* ctx, const PallasPoint& C_prime, uint64_t d, const PallasScalar& z, const PallasScalar& v,
                             const EvalProof& pi);
// R_o = P_o + a_o Q_o + b_o S for every o, exact and affine: halo_test_point_combine, on the device from "combine_min_outputs"
// outputs on (one launch), on host threads below
std::vector<affine_t> combine(halo_ctx* ctx, const std::vector<PallasPoint>& P, const std::vector<PallasPoint>& Q,
                              const std::vector<PallasScalar>& a, const std::vector<PallasScalar>& b);
// f(0) .. f(k - 1) spread over up to 16 host threads; returns what each call threw (null: nothing)
std::vector<std::exception_ptr> parallel_each(size_t k, const std::function<void(size_t)>& f);
// index of the first non-null entry (errs.size() if none)
size_t first_error(const std::vector<std::exception_ptr>& errs);

// pcdl.rs:252-314; throws HaloFailure(HALO_REJECT_SUCCINCT) on reject
std::pair<HPoly, PallasPoint> succinct_check(halo_ctx* ctx, const PallasPoint& C, uint64_t d, const PallasScalar& z,
                                             const PallasScalar& v, const EvalProof& pi);
// SURVEY 8(f).2: the succinct checks of several instances (acc.rs:158-170) and one unhidden commitment (acc.rs:153) with a
// single device round trip (halo_msm_multi).  Nothing is decided here: `accept[i]` is instance i's group equation
// (pcdl.rs:307-310) and the caller raises the reference's `ensure!`s in the reference's order.  Malformed input throws
// exactly as succinct_check / commit would, but possibly out of order -- callers fall back to the one-by-one path then.
struct Query {
    const PallasPoint* C;
    uint64_t d;
    const PallasScalar* z;
    const PallasScalar* v;
    const EvalProof* pi;
};
struct SuccinctMany {
    std::vector<std::pair<HPoly, PallasPoint>> hu;  // what succinct_check returns per instance
    std::vector<bool> accept;
    PallasPoint commitment;                          // commit(commit_p, commit_d, None) when commit_p != nullptr
};
SuccinctMany succinct_check_many(halo_ctx* ctx, const std::vector<Query>& qs, const PolyView* commit_p, uint64_t commit_d);
// pcdl.rs:323-342
void check(halo_ctx* ctx, const PallasPoint& C, uint64_t d, const PallasScalar& z, const PallasScalar& v,
           const EvalProof& pi);

// Batch decider (DESIGN.md K5b; the reference has none): the claims' succinct equations E_j and U checks F_j are combined
// with powers of the caller's rho != 0 into sum_j (rho^2j E_j + rho^(2j+1) F_j) = O, ONE halo_h_msm_batch.  Accepts iff that
// point is O.  Otherwise runs `check` on the claims in order and throws the first reject with *rejected_index = its claim;
// if every claim then accepts, the batch contradicted them: HALO_EINTERNAL.  Malformed input in any claim throws
// HALO_EINVAL before any decision.
void check_batch(halo_ctx* ctx, const std::vector<Query>& claims, const PallasScalar& rho, uint64_t* rejected_index);

// ---- the stages shared by the batch checks (check_batch, acc::verifier_batch, acc::verify_decide_batch; DESIGN.md K5d) ----
// Inputs of ONE `combine` call, gathered from every part of a batch.
struct CombineList {
    std::vector<PallasPoint> P, Q;
    std::vector<PallasScalar> a, b;
    size_t push(const PallasPoint& p, const PallasPoint& q, const PallasScalar& x, const PallasScalar& y) {
        P.push_back(p), Q.push_back(q), a.push_back(x), b.push_back(y);
        return P.size() - 1;
    }
    std::vector<affine_t> run(halo_ctx* ctx) const { return combine(ctx, P, Q, a, b); }
};
// The succinct equations of a list of queries, prepared in three steps around the one `combine` call of the batch:
// validate() (every query's validation and alpha, on host threads), request() (C' of the hiding queries that passed) and
// finish(j) (query j's transcript from its C').  The error of a batch is that of its first malformed query in order:
// rethrow_first() raises it, whichever step found it.
struct QueryBatch {
    std::vector<Query> qs;
    std::vector<PallasScalar> alphas;
    std::vector<std::exception_ptr> errs1, errs2;  // validate() / finish() failures
    size_t valid = 0;                              // queries ahead of the first one validate() refused
    std::vector<size_t> slot;                      // C' in the combine output (SIZE_MAX: C' = C)
    std::vector<std::optional<SuccinctPrep>> preps;
    void validate(halo_ctx* ctx, bool finish_plain);  // finish_plain: finish the queries without hiding in the same pass
    void request(CombineList& cl);
    void finish(halo_ctx* ctx, size_t j, const std::vector<affine_t>& c_out);  // j < valid
    bool failed() const;                           // some query is malformed
    void rethrow_first() const;                    // no-op if none is
    std::vector<affine_t> c_prime_affine(const std::vector<affine_t>& c_out) const;  // C'_j of every query, affine
};
// Terms of one combined equation sum_t rho^t X_t = O: the companion MSM (points and scalars; H once, with its scalars summed)
// and the generator part <GS, sum_j w_j coeffs(h_j)> (the claims' xi rows, lg n and weights).
struct BatchTerms {
    std::vector<affine_t> aff;
    std::vector<PallasScalar> sc;
    PallasScalar s_H = scalar_zero();
    std::vector<PallasScalar> xis, weights;
    std::vector<uint32_t> lgs;
    // re E + u_extra U for the succinct equation E = C' + sum_i s_i P_i (L, R, H, U) of one query
    void add_succinct(const SuccinctPrep& sp, const affine_t& c_prime, const PallasScalar& re, const PallasScalar& u_extra);
    // the claims' E_j and F_j = U_j - <G, h_j> with rho^t, rho^(t+1) for claim j, t = 2 j from rho_first on
    void add_claims(const QueryBatch& qb, const std::vector<affine_t>& c_aff, PallasScalar rho_first, const PallasScalar& rho);
};
// The decide stage: the generator part is submitted ahead of the host work that builds the companion terms; is_zero()
// collects with them and tells whether the combined point is O.  A batch left outstanding (the caller threw) is drained on
// destruction.
class GeneratorPart {
  public:
    explicit GeneratorPart(halo_ctx* ctx) : ctx_(ctx) {}
    GeneratorPart(const GeneratorPart&) = delete;
    GeneratorPart& operator=(const GeneratorPart&) = delete;
    ~GeneratorPart();
    void submit(const BatchTerms& t);
    bool is_zero(BatchTerms& t, const affine_t& H);
  private:
    halo_ctx* ctx_;
    int ticket_ = -1;
};
// `check` on claims in order; a reject is thrown with *rejected_index = index_base + its claim
void check_in_order(halo_ctx* ctx, const std::vector<Query>& claims, uint64_t index_base, uint64_t* rejected_index);

// wire conversion
EvalProof proof_from_c(const halo_eval_proof& p);
void proof_to_c(const EvalProof& p, halo_eval_proof& out);

}  // namespace pcdl
}  // namespace halo
