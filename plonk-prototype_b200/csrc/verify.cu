// verify.cu — the PLONK verifier and the BLS12-381 pairing, on the HOST (no kernels in this file).
//
// Replaces dusk-plonk 0.8.2 `Proof::verify`, `OpeningKey::batch_check` and dusk-bls12_381 0.8 `multi_miller_loop` /
// `final_exponentiation` (crates pinned at /root/reference/Cargo.toml:19-20; SURVEY.md §3.6, §8f-4).  Upstream's
// verifier is CPU code too: it is a few milliseconds of work that does not depend on the circuit size, so there is
// nothing for the GPU to do.  It lives in the library so that "proof verified" can be asserted by a user of the C ABI
// without the Rust crates; the independent checker used by the tests is the pure-Python model (oracle/plonk_model.py).
//
// The tower, G1 / G2 arithmetic and the pairing live in pairing_host.h (shared with verify_batch.cu).
#include <algorithm>
#include <cstring>
#include <utility>
#include <vector>

#include "../../include/pb200.h"
#include "host_field.h"
#include "merlin.h"
#include "pairing_host.h"
#include "widgets.h"

using hostf::HFp;
using hostf::HFr;
using namespace pairing;

namespace {

// ------------------------------------------------------------------------------------------------ verifier
HFr fr_from_bytes(const uint8_t b[32], bool *ok) {
    HFr raw;
    for (int i = 0; i < 4; i++) {
        raw.l[i] = 0;
        for (int k = 7; k >= 0; k--) raw.l[i] = (raw.l[i] << 8) | b[8 * i + k];
    }
    if (HFr::geq_mod(raw.l)) *ok = false;
    return raw * HFr::r2();
}
}  // namespace

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
    if (n < 2 || (n & (n - 1)) || n > ((size_t)1 << 30)) return PB200_ERR_ARG;
    *accepted = 0;
    if (n_pi > 1) {  // one public input per gate, as pb200_prove requires (a duplicate would be summed here but overwritten there)
        std::vector<uint32_t> sorted(pi_gate, pi_gate + n_pi);
        std::sort(sorted.begin(), sorted.end());
        if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end()) return PB200_ERR_ARG;
    }
    enum { Q_M, Q_L, Q_R, Q_O, Q_C, Q_4, Q_ARITH, Q_RANGE, Q_LOGIC, Q_FIXED, Q_VAR, S1, S2, S3, S4 };
    G1A vk[15], pr[11];
    for (int i = 0; i < 15; i++)
        if (!g1_from_bytes(vk_commitments + 48 * i, &vk[i])) return 0;  // malformed key / proof ⇒ rejected, not an error
    for (int i = 0; i < 11; i++)
        if (!g1_from_bytes(proof + 48 * i, &pr[i])) return 0;
    enum { P_A, P_B, P_C, P_D, P_Z, P_T1, P_T2, P_T3, P_T4, P_WZ, P_WZW };
    enum { E_A, E_B, E_C, E_D, E_AN, E_BN, E_DN, E_QARITH, E_QC, E_QL, E_QR, E_S1, E_S2, E_S3, E_R, E_PERM };
    HFr ev[16];
    bool canon = true;
    for (int i = 0; i < 16; i++) ev[i] = fr_from_bytes(proof + 528 + 32 * i, &canon);
    if (!canon) return 0;
    const G2A bh = {{HFp::load(beta_h), HFp::load(beta_h + 6)}, {HFp::load(beta_h + 12), HFp::load(beta_h + 18)}, false};
    if (!g2_on_curve(bh)) return PB200_ERR_ARG;

    // transcript: verifier key, then the proof in the prover's order
    merlin::Transcript tr(transcript_label, label_len);
    {
        const char *const lab[11] = {"q_m", "q_l", "q_r", "q_o", "q_c", "q_4", "q_arith", "q_range", "q_logic", "q_variable_group_add",
                                     "q_fixed_group_add"};
        const int idx[11] = {Q_M, Q_L, Q_R, Q_O, Q_C, Q_4, Q_ARITH, Q_RANGE, Q_LOGIC, Q_VAR, Q_FIXED};
        for (int k = 0; k < 11; k++) tr.append_commitment(lab[k], vk_commitments + 48 * idx[k]);
        const char *const sl[4] = {"left_sigma", "right_sigma", "out_sigma", "fourth_sigma"};
        for (int c = 0; c < 4; c++) tr.append_commitment(sl[c], vk_commitments + 48 * (S1 + c));
        tr.circuit_domain_sep(n);
    }
    const char *const wl[4] = {"w_l", "w_r", "w_o", "w_4"};
    for (int c = 0; c < 4; c++) tr.append_commitment(wl[c], proof + 48 * c);
    const HFr beta = tr.challenge_scalar("beta");
    tr.append_scalar("beta", beta);
    const HFr gamma = tr.challenge_scalar("gamma");
    tr.append_commitment("z", proof + 48 * P_Z);
    const HFr alpha = tr.challenge_scalar("alpha");
    const HFr range_sep = tr.challenge_scalar("range separation challenge");
    const HFr logic_sep = tr.challenge_scalar("logic separation challenge");
    const HFr fixed_sep = tr.challenge_scalar("fixed base separation challenge");
    const HFr var_sep = tr.challenge_scalar("variable base separation challenge");
    const char *const tl[4] = {"t_1", "t_2", "t_3", "t_4"};
    for (int k = 0; k < 4; k++) tr.append_commitment(tl[k], proof + 48 * (P_T1 + k));
    const HFr z = tr.challenge_scalar("z");

    // domain quantities
    uint32_t log_n = 0;
    while (((size_t)1 << log_n) < n) log_n++;
    const uint64_t root32[4] = {0xb9b58d8c5f0e466aull, 0x5b1b4c801819d7ecull, 0x0af53ae352a31e64ull, 0x5bf3adda19e9b27bull};
    HFr omega = HFr::load(root32);
    for (uint32_t k = 0; k < 32 - log_n; k++) omega = omega.sqr();
    const HFr one = HFr::one(), zn = z.pow_u64(n), z_h = zn - one;
    if (z_h.is_zero() || (z - one).is_zero()) return 0;
    const HFr n_fr = HFr::from_u64(n), n_inv = n_fr.inv();
    const HFr l1 = z_h * (n_fr * (z - one)).inv();
    // PI(z) = (zⁿ − 1)/n · Σ PI_i·ωⁱ/(z − ωⁱ)
    HFr pi_eval = HFr::zero();
    for (size_t j = 0; j < n_pi; j++) {
        if (pi_gate[j] >= n) return PB200_ERR_ARG;
        const HFr wi = omega.pow_u64(pi_gate[j]), den = z - wi;
        if (den.is_zero()) return 0;
        pi_eval = pi_eval + HFr::load(pi_mont + 4 * j) * wi * den.inv();
    }
    pi_eval = pi_eval * z_h * n_inv;
    const HFr a = ev[E_A], b = ev[E_B], c = ev[E_C], d = ev[E_D];
    // quotient evaluation
    const HFr alpha2 = alpha.sqr();
    const HFr copy3 = (a + beta * ev[E_S1] + gamma) * (b + beta * ev[E_S2] + gamma) * (c + beta * ev[E_S3] + gamma);
    const HFr t_eval = (ev[E_R] + pi_eval - copy3 * (d + gamma) * ev[E_PERM] * alpha - l1 * alpha2) * z_h.inv();
    const struct { const char *label; HFr v; } order[17] = {
        {"a_eval", a}, {"b_eval", b}, {"c_eval", c}, {"d_eval", d}, {"a_next_eval", ev[E_AN]}, {"b_next_eval", ev[E_BN]},
        {"d_next_eval", ev[E_DN]}, {"left_sig_eval", ev[E_S1]}, {"right_sig_eval", ev[E_S2]}, {"out_sig_eval", ev[E_S3]},
        {"q_arith_eval", ev[E_QARITH]}, {"q_c_eval", ev[E_QC]}, {"q_l_eval", ev[E_QL]}, {"q_r_eval", ev[E_QR]},
        {"perm_eval", ev[E_PERM]}, {"t_eval", t_eval}, {"r_eval", ev[E_R]}};
    for (const auto &o : order) tr.append_scalar(o.label, o.v);

    // commitments: quotient, linearisation
    auto jac = [&](const G1A &p) { return g1_from_affine(p); };
    G1J t_comm = jac(pr[P_T1]);
    {
        HFr zp = zn;
        for (int k = 1; k < 4; k++) {
            t_comm = g1_add(t_comm, g1_mul(jac(pr[P_T1 + k]), zp));
            zp = zp * zn;
        }
    }
    G1J r_comm = G1J::identity();
    {
        const HFr qa = ev[E_QARITH];
        const HFr four = HFr::from_u64(4), kappa = range_sep.sqr();
        auto delta = [&](const HFr &f) { return f * (f - one) * (f - one - one) * (f - one - one - one); };
        HFr rg = delta(ev[E_DN] - four * a);
        rg = rg * kappa + delta(a - four * b);
        rg = rg * kappa + delta(b - four * c);
        rg = rg * kappa + delta(c - four * d);
        const HFr k1 = HFr::from_u64(7), k2 = HFr::from_u64(13), k3 = HFr::from_u64(17), bz = beta * z;
        const HFr id = (a + bz + gamma) * (b + k1 * bz + gamma) * (c + k2 * bz + gamma) * (d + k3 * bz + gamma);
        // logic / fixed-base / variable-base widgets: the same identities the prover's quotient uses, at the evaluations
        const HFr edwards_d = (HFr::from_u64(10240) * HFr::from_u64(10241).inv()).neg();
        const HFr lg = widgets::logic_term(a, ev[E_AN], b, ev[E_BN], c, d, ev[E_DN], ev[E_QC], logic_sep);
        const HFr fx = widgets::fixed_base_term(a, ev[E_AN], b, ev[E_BN], c, d, ev[E_DN], ev[E_QL], ev[E_QR], ev[E_QC], fixed_sep, edwards_d);
        const HFr vb = widgets::var_base_term(a, ev[E_AN], b, ev[E_BN], c, d, ev[E_DN], var_sep, edwards_d);
        const struct { int point; HFr s; } terms[12] = {{Q_M, a * b * qa}, {Q_L, a * qa}, {Q_R, b * qa}, {Q_O, c * qa}, {Q_4, d * qa},
                                                        {Q_C, qa}, {Q_RANGE, rg * range_sep}, {Q_LOGIC, lg}, {Q_FIXED, fx}, {Q_VAR, vb},
                                                        {-1, id * alpha + l1 * alpha2},
                                                        {S4, (copy3 * beta * ev[E_PERM] * alpha).neg()}};
        for (const auto &t : terms) r_comm = g1_add(r_comm, g1_mul(jac(t.point < 0 ? pr[P_Z] : vk[t.point]), t.s));
    }
    // the two aggregate openings
    auto flatten = [&](const std::vector<std::pair<HFr, G1J>> &parts, G1J *cm, HFr *evl) {
        const HFr v = tr.challenge_scalar("aggregate_witness");
        HFr pw = one;
        *cm = G1J::identity();
        *evl = HFr::zero();
        for (const auto &p : parts) {
            *cm = g1_add(*cm, g1_mul(p.second, pw));
            *evl = *evl + p.first * pw;
            pw = pw * v;
        }
    };
    G1J ca, cb;
    HFr ea, eb;
    flatten({{t_eval, t_comm}, {ev[E_R], r_comm}, {a, jac(pr[P_A])}, {b, jac(pr[P_B])}, {c, jac(pr[P_C])}, {d, jac(pr[P_D])},
             {ev[E_S1], jac(vk[S1])}, {ev[E_S2], jac(vk[S2])}, {ev[E_S3], jac(vk[S3])}},
            &ca, &ea);
    flatten({{ev[E_PERM], jac(pr[P_Z])}, {ev[E_AN], jac(pr[P_A])}, {ev[E_BN], jac(pr[P_B])}, {ev[E_DN], jac(pr[P_D])}}, &cb, &eb);
    tr.append_commitment("w_z", proof + 48 * P_WZ);
    tr.append_commitment("w_z_w", proof + 48 * P_WZW);
    // OpeningKey::batch_check: e(−ΣuⁱWᵢ, βH) · e(Σuⁱ(Cᵢ + zᵢWᵢ) − (Σuⁱeᵢ)G, H) = 1
    const HFr u = tr.challenge_scalar("batch");
    const G1J wz = jac(pr[P_WZ]), wzw = jac(pr[P_WZW]);
    G1J total_c = g1_add(g1_add(ca, g1_mul(wz, z)), g1_mul(g1_add(cb, g1_mul(wzw, z * omega)), u));
    const G1J total_w = g1_add(wz, g1_mul(wzw, u));
    const G1A gen = {HFp::load(kG1x), HFp::load(kG1y), false};
    total_c = g1_add(total_c, g1_neg(g1_mul(jac(gen), ea + u * eb)));
    const Fp12 f = miller_loop(g1_to_affine(g1_neg(total_w)), bh) * miller_loop(g1_to_affine(total_c), g2_generator());
    *accepted = final_exponentiation(f) == Fp12::one();
    return 0;
}
