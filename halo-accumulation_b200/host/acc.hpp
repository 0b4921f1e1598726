// host/acc.hpp -- host mirror of code/src/acc.rs (ASDL accumulation scheme).
#pragma once
#include "pcdl.hpp"

namespace halo {
namespace acc {

// acc.rs:21-28
struct Instance {
    PallasPoint C;
    uint64_t d;
    PallasScalar z, v;
    pcdl::EvalProof pi;
};
// acc.rs:54-59
struct AccumulatorHiding {
    PallasPoly h;  // degree-1 polynomial h_0
    PallasPoint U;
    PallasScalar w;
};
// acc.rs:43-51
struct Accumulator {
    PallasPoint C_bar;
    uint64_t d;
    PallasScalar z, v;
    pcdl::EvalProof pi;
    AccumulatorHiding pi_V;
};
// impl From<Accumulator> for Instance (acc.rs:121-131)
inline Instance to_instance(const Accumulator& a) { return Instance{a.C_bar, a.d, a.z, a.v, a.pi}; }

// acc.rs:61-107
struct AccumulatedHPolys {
    bool have_h0 = false;
    PallasPoly h_0;
    std::vector<pcdl::HPoly> hs;
    bool have_alpha = false;
    PallasScalar alpha;
    std::vector<PallasScalar> alphas;
    size_t alphas_capacity = 0;
    explicit AccumulatedHPolys(size_t capacity) : alphas_capacity(capacity + 1) { hs.reserve(capacity); }  // :69-76
    void set_alpha(const PallasScalar& a) {                                                                   // :79-82
        alphas = construct_powers(a, alphas_capacity);
        alpha = a;
        have_alpha = true;
    }
    PallasPoly get_poly(halo_ctx* ctx, uint32_t lg_n) const;  // :85-94, on the device
    uint64_t get_poly_resident(halo_ctx* ctx, uint32_t lg_n) const;  // same, left on the device; returns the degree
    PallasScalar eval(const PallasScalar& z) const;           // :97-106
    void serialize(Transcript& t) const;                      // #[derive(CanonicalSerialize)] (:61)
};

// acc.rs:190-220; rng draws explicit in the reference's order: h_0 (2 coefficients, :192), w (:198), open's q, w_bar
Accumulator prover(halo_ctx* ctx, uint64_t d, const std::vector<Instance>& qs, const PallasPoly& h_0, const PallasScalar& w,
                   PolyView q, const PallasScalar& w_bar);
// acc.rs:223-243
void verifier(halo_ctx* ctx, uint64_t D, const std::vector<Instance>& qs, const Accumulator& acc);
// acc.rs:245-255
void decider(halo_ctx* ctx, const Accumulator& acc);
// pcdl::check_batch over (C_bar, d, z, v, pi) of every accumulator (acc.rs:254); the reference has no batch decider
void decider_batch(halo_ctx* ctx, const std::vector<Accumulator>& accs, const PallasScalar& rho, uint64_t* rejected_index);

// Batch verifier (DESIGN.md K5c; the reference has none): k accumulation steps (qs_i, acc_i), each against D as `verifier`,
// with ONE halo_msm over all their group equations combined with the powers of the caller's rho != 0.  Accepts iff that point is
// O and every step's host checks hold.  Otherwise runs `verifier` on the steps in order and throws the first reject with
// *rejected_index = its step; if every step then accepts: HALO_EINTERNAL.  Malformed input anywhere throws HALO_EINVAL before
// any decision.
struct Step {
    const std::vector<Instance>* qs;
    const Accumulator* acc;
};
void verifier_batch(halo_ctx* ctx, uint64_t D, const std::vector<Step>& steps, const PallasScalar& rho, uint64_t* rejected_index);
// verifier_batch(steps) followed by pcdl::check_batch(claims) in one call (DESIGN.md K5d): the claims' equations follow the
// steps' with the next powers of rho, and the generator MSM of the claims runs on the device while the steps' transcripts run
// on the host.  Decisions and errors are those of the pair, a claim j counting as item k + j of the concatenated sequence
// "steps, then claims": on a reject *rejected_index = that position.
void verify_decide_batch(halo_ctx* ctx, uint64_t D, const std::vector<Step>& steps, const std::vector<pcdl::Query>& claims,
                         const PallasScalar& rho, uint64_t* rejected_index);

Instance instance_from_c(const halo_instance& q);
Accumulator accumulator_from_c(const halo_accumulator& a);
void accumulator_to_c(const Accumulator& a, halo_accumulator& out);

}  // namespace acc
}  // namespace halo
