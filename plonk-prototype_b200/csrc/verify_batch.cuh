// verify_batch.cuh — the per-proof half of the batched verifier (verify_batch.cu): one proof's Fiat–Shamir transcript,
// challenges, PI(z), t(z) and the coefficients that write its pairing equation as a linear combination of group elements.
//
// PB_HD, so verify_prepare_kernel runs it one proof per thread and the CPU host emulation (tests/host_emu/emu_verify.cpp)
// runs the same code.  It restates, scalar for scalar, what pb200_verify (verify.cu) computes before its pairing:
//
//   pb200_verify accepts  ⇔  e(−W, βH) · e(C, H) = 1  with
//   W = W_z + u·W_zω
//   C = ca + z·W_z + u·(cb + zω·W_zω) − (ea + u·eb)·G
//
// where ca, cb are the two aggregate openings (t_comm and r_comm expanded in them).  Collected per base:
//   proof points  A: v² + u·v'     B: v³ + u·v'²    C: v⁴           D: v⁵ + u·v'³    Z: v·s_z + u
//                 T1..T4: 1, zⁿ, z²ⁿ, z³ⁿ          W_z: z          W_zω: u·z·ω
//   shared bases  q_m … q_variable_group_add: v·(linearisation scalar), q_arith: 0, σ1..σ3: v⁶, v⁷, v⁸, σ4: v·s_σ4,
//                 G: −(ea + u·eb)
// with v, v' the two `aggregate_witness` challenges.  An identity point (c0 00…00, valid upstream) gets coefficient 0.
#pragma once
#include "../../include/pb200.h"
#include "field.cuh"
#include "merlin.h"
#include "widgets.h"

// Device Fr ↔ the 32-byte canonical / 64-byte wide encodings of BlsScalar, found by merlin.h's generic scalar methods.
PB_HD void scalar_to_bytes(const Fr &s, uint8_t out[32]) {
    const Fr c = s.from_mont();
    for (int i = 0; i < 8; i++)
        for (int k = 0; k < 4; k++) out[4 * i + k] = (uint8_t)(c.l[i] >> (8 * k));
}
// BlsScalar::from_bytes_wide: lo + hi·2^256 mod r.  Each half (< 2^256 < 3r) is brought below r first.
PB_HD void scalar_from_bytes_wide(const uint8_t in[64], Fr &out) {
    Fr lo, hi;
    for (int i = 0; i < 8; i++) {
        lo.l[i] = hi.l[i] = 0;
        for (int k = 3; k >= 0; k--) {
            lo.l[i] = (lo.l[i] << 8) | in[4 * i + k];
            hi.l[i] = (hi.l[i] << 8) | in[32 + 4 * i + k];
        }
    }
    lo = Fr::reduce_once(Fr::reduce_once(lo));
    hi = Fr::reduce_once(Fr::reduce_once(hi));
    const Fr r2 = Fr::r2(), r3 = r2 * r2;
    out = lo * r2 + hi * r3;
}
// 32 little-endian bytes → Montgomery form; false when the value is not below r.
PB_HD bool fr_from_bytes_checked(const uint8_t b[32], Fr &out) {
    Fr raw;
    for (int i = 0; i < 8; i++)
        raw.l[i] = (uint32_t)b[4 * i] | ((uint32_t)b[4 * i + 1] << 8) | ((uint32_t)b[4 * i + 2] << 16) | ((uint32_t)b[4 * i + 3] << 24);
    (void)cc::sub_cc(raw.l[0], FrParams::mod(0));
    for (int i = 1; i < 8; i++) (void)cc::subc_cc(raw.l[i], FrParams::mod(i));
    if (cc::subc(0, 0) == 0) return false;  // raw − r did not borrow: raw ≥ r
    out = raw.to_mont();
    return true;
}

namespace vb {

enum { P_A, P_B, P_C, P_D, P_Z, P_T1, P_T2, P_T3, P_T4, P_WZ, P_WZW };
enum { Q_M, Q_L, Q_R, Q_O, Q_C, Q_4, Q_ARITH, Q_RANGE, Q_LOGIC, Q_FIXED, Q_VAR, S1, S2, S3, S4, GEN };
enum { E_A, E_B, E_C, E_D, E_AN, E_BN, E_DN, E_QARITH, E_QC, E_QL, E_QR, E_S1, E_S2, E_S3, E_R, E_PERM };
constexpr int kProofPoints = 11, kShared = 16;  // 15 verifier-key commitments and the generator G

// Per-proof verdict before any pairing (the cases pb200_verify rejects without one).
enum { OK = 0, BAD_POINT = 1, BAD_EVAL = 2, BAD_Z = 3 };

// Everything the call shares: the domain and the circuit-independent constants, all Fr in Montgomery form.
struct Consts {
    uint64_t n;
    uint32_t n_pi;
    uint32_t vk_identity;  // bit j: verifier-key commitment j is the identity (its column of coefficients is zero)
    Fr omega, n_fr, n_inv, edwards_d;
};

struct ProofOut {
    Fr coef[kProofPoints];  // C-side coefficient of each proof point (W-side: 1 for W_z and u for W_zω, see below)
    Fr e[kShared];          // coefficient of each shared base
    Fr z, u;
    uint8_t digest[32];     // binds the whole transcript and the public inputs: input of the batch weights
};

// seed: the transcript after label, verifier key and circuit_domain_sep(n).  proof: 1040 bytes.  pt_status: the
// PB200_G1_* status of the proof's 11 points.  wg[j] = ω^{pi_gate[j]}, pi[j] = this proof's public input j.
PB_HD int prepare_one(merlin::Transcript tr, const uint8_t *proof, const uint8_t *pt_status, const Consts &k, const Fr *wg,
                      const Fr *pi, ProofOut &o) {
    for (int i = 0; i < kProofPoints; i++)
        if (pt_status[i] != PB200_G1_OK && pt_status[i] != PB200_G1_IDENTITY) return BAD_POINT;
    Fr ev[16];
    for (int i = 0; i < 16; i++)
        if (!fr_from_bytes_checked(proof + 528 + 32 * i, ev[i])) return BAD_EVAL;

    const char *const wl[4] = {"w_l", "w_r", "w_o", "w_4"};
    for (int c = 0; c < 4; c++) tr.append_commitment(wl[c], proof + 48 * c);
    const Fr beta = tr.challenge_scalar<Fr>("beta");
    tr.append_scalar("beta", beta);
    const Fr gamma = tr.challenge_scalar<Fr>("gamma");
    tr.append_commitment("z", proof + 48 * P_Z);
    const Fr alpha = tr.challenge_scalar<Fr>("alpha");
    const Fr range_sep = tr.challenge_scalar<Fr>("range separation challenge");
    const Fr logic_sep = tr.challenge_scalar<Fr>("logic separation challenge");
    const Fr fixed_sep = tr.challenge_scalar<Fr>("fixed base separation challenge");
    const Fr var_sep = tr.challenge_scalar<Fr>("variable base separation challenge");
    const char *const tl[4] = {"t_1", "t_2", "t_3", "t_4"};
    for (int c = 0; c < 4; c++) tr.append_commitment(tl[c], proof + 48 * (P_T1 + c));
    const Fr z = tr.challenge_scalar<Fr>("z");

    const Fr one = Fr::one(), zn = z.pow_u64(k.n), z_h = zn - one, zm1 = z - one;
    if (z_h.is_zero() || zm1.is_zero()) return BAD_Z;
    // Σ_j PI_j·ω^{g_j}/(z − ω^{g_j}) kept as a fraction num/den, then one inversion for 1/den, 1/z_h and 1/(n(z − 1))
    Fr num = Fr::zero(), den = one;
    for (uint32_t j = 0; j < k.n_pi; j++) {
        const Fr d = z - wg[j];
        if (d.is_zero()) return BAD_Z;
        num = num * d + pi[j] * wg[j] * den;
        den = den * d;
    }
    const Fr nzm1 = k.n_fr * zm1;
    const Fr inv = (den * z_h * nzm1).inv();
    const Fr inv_zh = inv * den * nzm1;
    const Fr l1 = z_h * (inv * den * z_h);
    const Fr pi_eval = num * (inv * z_h * nzm1) * z_h * k.n_inv;

    const Fr a = ev[E_A], b = ev[E_B], c = ev[E_C], d = ev[E_D];
    const Fr alpha2 = alpha.sqr();
    const Fr copy3 = (a + beta * ev[E_S1] + gamma) * (b + beta * ev[E_S2] + gamma) * (c + beta * ev[E_S3] + gamma);
    const Fr t_eval = (ev[E_R] + pi_eval - copy3 * (d + gamma) * ev[E_PERM] * alpha - l1 * alpha2) * inv_zh;
    const char *const olab[17] = {"a_eval", "b_eval", "c_eval", "d_eval", "a_next_eval", "b_next_eval", "d_next_eval",
                                  "left_sig_eval", "right_sig_eval", "out_sig_eval", "q_arith_eval", "q_c_eval", "q_l_eval",
                                  "q_r_eval", "perm_eval", "t_eval", "r_eval"};
    const int oidx[17] = {E_A, E_B, E_C, E_D, E_AN, E_BN, E_DN, E_S1, E_S2, E_S3, E_QARITH, E_QC, E_QL, E_QR, E_PERM, -1, E_R};
    for (int i = 0; i < 17; i++) tr.append_scalar(olab[i], oidx[i] < 0 ? t_eval : ev[oidx[i]]);

    // linearisation scalars (verify.cu's r_comm terms)
    const Fr qa = ev[E_QARITH];
    const Fr four = widgets::small<Fr>(4), kappa = range_sep.sqr();
    Fr rg = widgets::delta4(ev[E_DN] - four * a);
    rg = rg * kappa + widgets::delta4(a - four * b);
    rg = rg * kappa + widgets::delta4(b - four * c);
    rg = rg * kappa + widgets::delta4(c - four * d);
    const Fr bz = beta * z;
    const Fr id = (a + bz + gamma) * (b + widgets::small<Fr>(7) * bz + gamma) * (c + widgets::small<Fr>(13) * bz + gamma) *
                  (d + widgets::small<Fr>(17) * bz + gamma);
    const Fr lg = widgets::logic_term(a, ev[E_AN], b, ev[E_BN], c, d, ev[E_DN], ev[E_QC], logic_sep);
    const Fr fx = widgets::fixed_base_term(a, ev[E_AN], b, ev[E_BN], c, d, ev[E_DN], ev[E_QL], ev[E_QR], ev[E_QC], fixed_sep, k.edwards_d);
    const Fr vbt = widgets::var_base_term(a, ev[E_AN], b, ev[E_BN], c, d, ev[E_DN], var_sep, k.edwards_d);
    const Fr s_z = id * alpha + l1 * alpha2;
    const Fr s_s4 = (copy3 * beta * ev[E_PERM] * alpha).neg();

    const Fr v = tr.challenge_scalar<Fr>("aggregate_witness");
    const Fr v2 = tr.challenge_scalar<Fr>("aggregate_witness");
    tr.append_commitment("w_z", proof + 48 * P_WZ);
    tr.append_commitment("w_z_w", proof + 48 * P_WZW);
    const Fr u = tr.challenge_scalar<Fr>("batch");

    Fr vp[9];  // v⁰ … v⁸
    vp[0] = one;
    for (int i = 1; i < 9; i++) vp[i] = vp[i - 1] * v;
    const Fr w1 = v2, w2 = v2.sqr(), w3 = w2 * v2;
    const Fr ea = t_eval + ev[E_R] * vp[1] + a * vp[2] + b * vp[3] + c * vp[4] + d * vp[5] + ev[E_S1] * vp[6] + ev[E_S2] * vp[7] +
                  ev[E_S3] * vp[8];
    const Fr eb = ev[E_PERM] + ev[E_AN] * w1 + ev[E_BN] * w2 + ev[E_DN] * w3;

    o.coef[P_A] = vp[2] + u * w1;
    o.coef[P_B] = vp[3] + u * w2;
    o.coef[P_C] = vp[4];
    o.coef[P_D] = vp[5] + u * w3;
    o.coef[P_Z] = v * s_z + u;
    o.coef[P_T1] = one;
    o.coef[P_T2] = zn;
    o.coef[P_T3] = zn.sqr();
    o.coef[P_T4] = o.coef[P_T3] * zn;
    o.coef[P_WZ] = z;
    o.coef[P_WZW] = u * z * k.omega;
    o.e[Q_M] = v * (a * b * qa);
    o.e[Q_L] = v * (a * qa);
    o.e[Q_R] = v * (b * qa);
    o.e[Q_O] = v * (c * qa);
    o.e[Q_C] = v * qa;
    o.e[Q_4] = v * (d * qa);
    o.e[Q_ARITH] = Fr::zero();
    o.e[Q_RANGE] = v * (rg * range_sep);
    o.e[Q_LOGIC] = v * lg;
    o.e[Q_FIXED] = v * fx;
    o.e[Q_VAR] = v * vbt;
    o.e[S1] = vp[6];
    o.e[S2] = vp[7];
    o.e[S3] = vp[8];
    o.e[S4] = v * s_s4;
    o.e[GEN] = (ea + u * eb).neg();
    for (int i = 0; i < kProofPoints; i++)
        if (pt_status[i] == PB200_G1_IDENTITY) o.coef[i] = Fr::zero();
    for (int j = 0; j < 15; j++)
        if ((k.vk_identity >> j) & 1) o.e[j] = Fr::zero();
    o.z = z;
    o.u = u;
    // batch digest: the transcript so far (every commitment and evaluation of the proof) plus its public inputs
    for (uint32_t j = 0; j < k.n_pi; j++) tr.append_scalar("pi", pi[j]);
    tr.challenge_bytes("batch digest", o.digest, 32);
    return OK;
}

// ρ_k: rho_seed is Transcript("pb200 rho") after append_message("D", D); the proof index is appended and 64 bytes drawn.
PB_HD Fr rho(merlin::Transcript rho_seed, uint64_t k) {
    rho_seed.append_u64("k", k);
    return rho_seed.challenge_scalar<Fr>("rho");
}

}  // namespace vb
