// Host-emulation harness for the batched verifier's per-proof derivation (csrc/verify_batch.cuh, the code
// verify_prepare_kernel and verify_weight_kernel run), compiled for the CPU with the carry-flag primitives emulated
// (PB200_HOST_EMU), behind a C ABI for pytest.  The host-side set-up is pb200_verify_batch's (merlin::seed_transcript,
// vb::make_consts), called here as there.
#define PB200_HOST_EMU 1
#include "../../plonk-prototype_b200/csrc/g1_codec.cuh"
#include "../../plonk-prototype_b200/csrc/verify_batch.cuh"
#include <cstddef>
#include <cstring>
#include <vector>

extern "C" {
// One proof through vb::prepare_one.  Returns -1 for a malformed verifier key, else the verdict (vb::OK = 0 …).  For OK:
// coef (11 × 4 u64), e (16 × 4 u64), zu (z ‖ u, 2 × 4 u64), all Montgomery, and the 32-byte digest.
int emu_verify_prepare(const uint8_t *label, size_t label_len, const uint8_t *vk, uint64_t n, const uint8_t *proof,
                       const uint32_t *pi_gate, const uint64_t *pi_mont, size_t n_pi, uint64_t *coef, uint64_t *e, uint64_t *zu,
                       uint8_t *digest) {
    uint32_t vk_identity = 0;
    for (int j = 0; j < 15; j++) {
        G1Affine p;
        const int st = g1_decode_checked(vk + 48 * j, p);
        if (st == PB200_G1_IDENTITY) vk_identity |= 1u << j;
        else if (st != PB200_G1_OK) return -1;
    }
    uint8_t pt_status[11];
    for (int i = 0; i < 11; i++) {
        G1Affine p;
        pt_status[i] = (uint8_t)g1_decode_checked(proof + 48 * i, p);
    }
    merlin::Transcript tr(label, label_len);
    merlin::seed_transcript(tr, vk, n);
    std::vector<Fr> wg, pi(n_pi);
    const vb::Consts<Fr> kc = vb::make_consts(n, pi_gate, n_pi, vk_identity, wg);
    for (size_t j = 0; j < n_pi; j++) memcpy(pi[j].l, pi_mont + 4 * j, 32);
    vb::ProofOut<Fr> o;
    const int st = vb::prepare_one(tr, proof, pt_status, kc, wg.data(), pi.data(), o);
    if (st != vb::OK) return st;
    for (int i = 0; i < 11; i++) memcpy(coef + 4 * i, o.coef[i].l, 32);
    for (int j = 0; j < 16; j++) memcpy(e + 4 * j, o.e[j].l, 32);
    memcpy(zu, o.z.l, 32);
    memcpy(zu + 4, o.u.l, 32);
    memcpy(digest, o.digest, 32);
    return st;
}
// D = Merlin("pb200 verify_batch") over seed, n, K and the K digests; then ρ_k (Montgomery) for k < K.
void emu_verify_weights(const uint8_t seed[32], uint64_t n, uint64_t K, const uint8_t *digests, uint8_t D[32], uint64_t *rho_out) {
    merlin::Transcript dt((const uint8_t *)"pb200 verify_batch", 18);
    dt.append_message("seed", seed, 32);
    dt.append_u64("n", n);
    dt.append_u64("K", K);
    dt.append_message("digests", digests, 32 * K);
    dt.challenge_bytes("D", D, 32);
    merlin::Transcript rho_seed((const uint8_t *)"pb200 rho", 9);
    rho_seed.append_message("D", D, 32);
    for (uint64_t k = 0; k < K; k++) {
        const Fr r = vb::rho(rho_seed, k);
        memcpy(rho_out + 4 * k, r.l, 32);
    }
}
}
