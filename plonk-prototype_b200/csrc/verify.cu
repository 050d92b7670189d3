// verify.cu — the PLONK verifier and the BLS12-381 pairing, on the HOST (no kernels in this file).
//
// Replaces dusk-plonk 0.8.2 `Proof::verify`, `OpeningKey::batch_check` and dusk-bls12_381 0.8 `multi_miller_loop` /
// `final_exponentiation` (crates pinned at /root/reference/Cargo.toml:19-20; SURVEY.md §3.6, §8f-4).  Upstream's
// verifier is CPU code too: it is a few milliseconds of work that does not depend on the circuit size, so there is
// nothing for the GPU to do.  It lives in the library so that "proof verified" can be asserted by a user of the C ABI
// without the Rust crates; the independent checker used by the tests is the pure-Python model (oracle/plonk_model.py).
//
// pb200_verify derives the proof's pairing equation with vb::prepare_one (verify_batch.cuh) over hostf::HFr, the code
// pb200_verify_batch runs per proof on the device, so both verifiers reach their verdicts from one derivation.  The
// tower, G1 / G2 arithmetic and the pairing live in pairing_host.h.
#include <vector>

#include "../../include/pb200.h"
#include "verify_batch.cuh"

using hostf::HFp;
using hostf::HFr;
using namespace pairing;

extern "C" int pb200_opening_key_from_tau(const uint64_t tau_mont[4], uint64_t beta_h_out[24]) {
    if (!tau_mont || !beta_h_out) return PB200_ERR_ARG;
    const G2A bh = g2_mul(g2_generator(), HFr::load(tau_mont));
    if (bh.inf) return PB200_ERR_ARG;
    bh.x.a.store(beta_h_out);
    bh.x.b.store(beta_h_out + 6);
    bh.y.a.store(beta_h_out + 12);
    bh.y.b.store(beta_h_out + 18);
    return 0;
}

// e(a·G1, b·G2) == e(G1, G2)^(a·b) and ≠ 1 — the pairing's known-answer-free self check (bilinearity, non-degeneracy).
extern "C" int pb200_pairing_selftest(const uint64_t a_mont[4], const uint64_t b_mont[4], int *ok) {
    if (!a_mont || !b_mont || !ok) return PB200_ERR_ARG;
    const HFr a = HFr::load(a_mont), b = HFr::load(b_mont);
    const G1A g1 = {HFp::load(kG1x), HFp::load(kG1y), false};
    const G2A g2 = g2_generator();
    const Fp12 e = final_exponentiation(miller_loop(g1, g2));
    const Fp12 eab = final_exponentiation(miller_loop(g1_to_affine(g1_mul(g1_from_affine(g1), a)), g2_mul(g2, b)));
    const HFr ab = (a * b).from_mont();
    Fp12 p = Fp12::one();
    for (int i = 255; i >= 0; i--) {
        p = p.sqr();
        if ((ab.l[i >> 6] >> (i & 63)) & 1) p = p * e;
    }
    *ok = g2_on_curve(g2) && !(e == Fp12::one()) && p == eab;
    return 0;
}

extern "C" int pb200_verify(const uint8_t vk_commitments[15 * 48], size_t n, const uint8_t *transcript_label, size_t label_len,
                            const uint8_t proof[1040], const uint32_t *pi_gate, const uint64_t *pi_mont, size_t n_pi,
                            const uint64_t beta_h[24], int *accepted) {
    if (!vk_commitments || !proof || !beta_h || !accepted || (n_pi && (!pi_gate || !pi_mont)) || (!transcript_label && label_len))
        return PB200_ERR_ARG;
    *accepted = 0;
    G2A bh;
    if (!vb::args_ok(n, pi_gate, n_pi, beta_h, &bh)) return PB200_ERR_ARG;
    G1A vk[15], pr[vb::kProofPoints];
    uint32_t vk_identity = 0;
    for (int j = 0; j < 15; j++) {
        const int st = g1_from_bytes(vk_commitments + 48 * j, &vk[j]);
        if (st == PB200_G1_IDENTITY) vk_identity |= 1u << j;
        else if (st != PB200_G1_OK) return 0;  // malformed key ⇒ rejected, not an error
    }
    uint8_t pt_status[vb::kProofPoints];
    for (int i = 0; i < vb::kProofPoints; i++) pt_status[i] = (uint8_t)g1_from_bytes(proof + 48 * i, &pr[i]);
    std::vector<HFr> wg, pi(n_pi);
    const vb::Consts<HFr> k = vb::make_consts(n, pi_gate, n_pi, vk_identity, wg);
    for (size_t j = 0; j < n_pi; j++) pi[j] = HFr::load(pi_mont + 4 * j);
    merlin::Transcript tr(transcript_label, label_len);
    merlin::seed_transcript(tr, vk_commitments, n);
    vb::ProofOut<HFr> o;
    if (vb::prepare_one(tr, proof, pt_status, k, wg.data(), pi.data(), o) != vb::OK) return 0;

    // OpeningKey::batch_check: e(−W, βH) · e(C, H) = 1 with C = Σ coef_i·P_i + Σ e_j·B_j and W = W_z + u·W_zω
    const G1A gen = {HFp::load(kG1x), HFp::load(kG1y), false};
    G1J c = G1J::identity();
    for (int i = 0; i < vb::kProofPoints; i++) c = g1_add(c, g1_mul(g1_from_affine(pr[i]), o.coef[i]));
    for (int j = 0; j < vb::kShared; j++) c = g1_add(c, g1_mul(g1_from_affine(j == vb::GEN ? gen : vk[j]), o.e[j]));
    const G1J w = g1_add(g1_from_affine(pr[vb::P_WZ]), g1_mul(g1_from_affine(pr[vb::P_WZW]), o.u));
    const Fp12 f = miller_loop(g1_to_affine(g1_neg(w)), bh) * miller_loop(g1_to_affine(c), g2_generator());
    *accepted = final_exponentiation(f) == Fp12::one();
    return 0;
}
