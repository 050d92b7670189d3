// verify_batch.cuh — one proof's pairing equation, derived once for both verifiers: its Fiat–Shamir transcript,
// challenges, PI(z), t(z) and the coefficients that write the equation as a linear combination of group elements.
//
// prepare_one is generic over the scalar field, as widgets.h and merlin.h are: verify_prepare_kernel runs it with the
// device's Fr, one proof per thread (pb200_verify_batch, verify_batch.cu); pb200_verify (verify.cu) runs it with
// hostf::HFr; the CPU host emulation (tests/host_emu/emu_verify.cpp) runs the Fr instantiation on the host.  A proof is
// accepted iff
//
//   e(−W, βH) · e(C, H) = 1  with
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
#include "pairing_host.h"
#include "widgets.h"

#include <algorithm>
#include <vector>

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

// Everything the call shares: the domain and the circuit-independent constants, in Montgomery form.  F defaults to the
// device's Fr, so vb::Consts and vb::ProofOut without arguments name the batched verifier's types.
template <class F = Fr>
struct Consts {
    uint64_t n;
    uint32_t n_pi;
    uint32_t vk_identity;  // bit j: verifier-key commitment j is the identity (its column of coefficients is zero)
    F omega, n_fr, n_inv, edwards_d;
};

template <class F = Fr>
struct ProofOut {
    F coef[kProofPoints];  // C-side coefficient of each proof point (W-side: 1 for W_z and u for W_zω, see below)
    F e[kShared];          // coefficient of each shared base
    F z, u;
    uint8_t digest[32];    // binds the whole transcript and the public inputs: input of the batch weights
};

// seed: the transcript after label, verifier key and circuit_domain_sep(n).  proof: 1040 bytes.  pt_status: the
// PB200_G1_* status of the proof's 11 points.  wg[j] = ω^{pi_gate[j]}, pi[j] = this proof's public input j.
MERLIN_EXEC_CHECK_DISABLE
template <class F>
MERLIN_HD int prepare_one(merlin::Transcript tr, const uint8_t *proof, const uint8_t *pt_status, const Consts<F> &k, const F *wg,
                          const F *pi, ProofOut<F> &o) {
    for (int i = 0; i < kProofPoints; i++)
        if (pt_status[i] != PB200_G1_OK && pt_status[i] != PB200_G1_IDENTITY) return BAD_POINT;
    F ev[16];
    for (int i = 0; i < 16; i++)
        if (!fr_from_bytes_checked(proof + 528 + 32 * i, ev[i])) return BAD_EVAL;

    const char *const wl[4] = {"w_l", "w_r", "w_o", "w_4"};
    for (int c = 0; c < 4; c++) tr.append_commitment(wl[c], proof + 48 * c);
    const F beta = tr.challenge_scalar<F>("beta");
    tr.append_scalar("beta", beta);
    const F gamma = tr.challenge_scalar<F>("gamma");
    tr.append_commitment("z", proof + 48 * P_Z);
    const F alpha = tr.challenge_scalar<F>("alpha");
    const F range_sep = tr.challenge_scalar<F>("range separation challenge");
    const F logic_sep = tr.challenge_scalar<F>("logic separation challenge");
    const F fixed_sep = tr.challenge_scalar<F>("fixed base separation challenge");
    const F var_sep = tr.challenge_scalar<F>("variable base separation challenge");
    const char *const tl[4] = {"t_1", "t_2", "t_3", "t_4"};
    for (int c = 0; c < 4; c++) tr.append_commitment(tl[c], proof + 48 * (P_T1 + c));
    const F z = tr.challenge_scalar<F>("z");

    const F one = F::one(), zn = z.pow_u64(k.n), z_h = zn - one, zm1 = z - one;
    if (z_h.is_zero() || zm1.is_zero()) return BAD_Z;
    // Σ_j PI_j·ω^{g_j}/(z − ω^{g_j}) kept as a fraction num/den, then one inversion for 1/den, 1/z_h and 1/(n(z − 1))
    F num = F::zero(), den = one;
    for (uint32_t j = 0; j < k.n_pi; j++) {
        const F d = z - wg[j];
        if (d.is_zero()) return BAD_Z;
        num = num * d + pi[j] * wg[j] * den;
        den = den * d;
    }
    const F nzm1 = k.n_fr * zm1;
    const F inv = (den * z_h * nzm1).inv();
    const F inv_zh = inv * den * nzm1;
    const F l1 = z_h * (inv * den * z_h);
    const F pi_eval = num * (inv * z_h * nzm1) * z_h * k.n_inv;

    const F a = ev[E_A], b = ev[E_B], c = ev[E_C], d = ev[E_D];
    const F alpha2 = alpha.sqr();
    const F copy3 = (a + beta * ev[E_S1] + gamma) * (b + beta * ev[E_S2] + gamma) * (c + beta * ev[E_S3] + gamma);
    const F t_eval = (ev[E_R] + pi_eval - copy3 * (d + gamma) * ev[E_PERM] * alpha - l1 * alpha2) * inv_zh;
    const char *const olab[17] = {"a_eval", "b_eval", "c_eval", "d_eval", "a_next_eval", "b_next_eval", "d_next_eval",
                                  "left_sig_eval", "right_sig_eval", "out_sig_eval", "q_arith_eval", "q_c_eval", "q_l_eval",
                                  "q_r_eval", "perm_eval", "t_eval", "r_eval"};
    const int oidx[17] = {E_A, E_B, E_C, E_D, E_AN, E_BN, E_DN, E_S1, E_S2, E_S3, E_QARITH, E_QC, E_QL, E_QR, E_PERM, -1, E_R};
    for (int i = 0; i < 17; i++) tr.append_scalar(olab[i], oidx[i] < 0 ? t_eval : ev[oidx[i]]);

    // linearisation scalars: the coefficients of r_comm
    const F qa = ev[E_QARITH];
    const F four = widgets::small<F>(4), kappa = range_sep.sqr();
    F rg = widgets::delta4(ev[E_DN] - four * a);
    rg = rg * kappa + widgets::delta4(a - four * b);
    rg = rg * kappa + widgets::delta4(b - four * c);
    rg = rg * kappa + widgets::delta4(c - four * d);
    const F bz = beta * z;
    const F id = (a + bz + gamma) * (b + widgets::small<F>(7) * bz + gamma) * (c + widgets::small<F>(13) * bz + gamma) *
                 (d + widgets::small<F>(17) * bz + gamma);
    const F lg = widgets::logic_term(a, ev[E_AN], b, ev[E_BN], c, d, ev[E_DN], ev[E_QC], logic_sep);
    const F fx = widgets::fixed_base_term(a, ev[E_AN], b, ev[E_BN], c, d, ev[E_DN], ev[E_QL], ev[E_QR], ev[E_QC], fixed_sep, k.edwards_d);
    const F vbt = widgets::var_base_term(a, ev[E_AN], b, ev[E_BN], c, d, ev[E_DN], var_sep, k.edwards_d);
    const F s_z = id * alpha + l1 * alpha2;
    const F s_s4 = (copy3 * beta * ev[E_PERM] * alpha).neg();

    const F v = tr.challenge_scalar<F>("aggregate_witness");
    const F v2 = tr.challenge_scalar<F>("aggregate_witness");
    tr.append_commitment("w_z", proof + 48 * P_WZ);
    tr.append_commitment("w_z_w", proof + 48 * P_WZW);
    const F u = tr.challenge_scalar<F>("batch");

    F vp[9];  // v⁰ … v⁸
    vp[0] = one;
    for (int i = 1; i < 9; i++) vp[i] = vp[i - 1] * v;
    const F w1 = v2, w2 = v2.sqr(), w3 = w2 * v2;
    const F ea = t_eval + ev[E_R] * vp[1] + a * vp[2] + b * vp[3] + c * vp[4] + d * vp[5] + ev[E_S1] * vp[6] + ev[E_S2] * vp[7] +
                 ev[E_S3] * vp[8];
    const F eb = ev[E_PERM] + ev[E_AN] * w1 + ev[E_BN] * w2 + ev[E_DN] * w3;

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
    o.e[Q_ARITH] = F::zero();
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
        if (pt_status[i] == PB200_G1_IDENTITY) o.coef[i] = F::zero();
    for (int j = 0; j < 15; j++)
        if ((k.vk_identity >> j) & 1) o.e[j] = F::zero();
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

// ------------------------------------------------------------------------------------------------ host set-up
// HFr → F (HFr itself, or the device's Fr: the same 32-byte little-endian Montgomery image).
template <class F>
F from_host(const hostf::HFr &a) {
    F r;
    memcpy(r.l, a.l, 32);
    return r;
}

// The arguments both verifiers reject with PB200_ERR_ARG before they read any proof byte: n not a power of two in
// [2, 2^30], a gate in pi_gate twice (pb200_prove takes one public input per gate) or not below n, β·H not on the curve.
// *bh: beta_h (affine x.c0 ‖ x.c1 ‖ y.c0 ‖ y.c1, Montgomery) as a point.
inline bool args_ok(size_t n, const uint32_t *pi_gate, size_t n_pi, const uint64_t beta_h[24], pairing::G2A *bh) {
    using hostf::HFp;
    if (n < 2 || (n & (n - 1)) || n > ((size_t)1 << 30)) return false;
    std::vector<uint32_t> sorted(pi_gate, pi_gate + n_pi);
    std::sort(sorted.begin(), sorted.end());
    if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end() || (n_pi && sorted.back() >= n)) return false;
    *bh = {{HFp::load(beta_h), HFp::load(beta_h + 6)}, {HFp::load(beta_h + 12), HFp::load(beta_h + 18)}, false};
    return pairing::g2_on_curve(*bh);
}

// The constants of a circuit of size n (a power of two) and wg[j] = ω^{pi_gate[j]}, as F.
template <class F>
Consts<F> make_consts(uint64_t n, const uint32_t *pi_gate, size_t n_pi, uint32_t vk_identity, std::vector<F> &wg) {
    using hostf::HFr;
    uint32_t log_n = 0;
    while ((1ull << log_n) < n) log_n++;
    const HFr omega = hostf::domain_root(log_n), n_fr = HFr::from_u64(n);
    Consts<F> k;
    k.n = n;
    k.n_pi = (uint32_t)n_pi;
    k.vk_identity = vk_identity;
    k.omega = from_host<F>(omega);
    k.n_fr = from_host<F>(n_fr);
    k.n_inv = from_host<F>(n_fr.inv());
    k.edwards_d = from_host<F>((HFr::from_u64(10240) * HFr::from_u64(10241).inv()).neg());
    wg.resize(n_pi);
    for (size_t j = 0; j < n_pi; j++) wg[j] = from_host<F>(omega.pow_u64(pi_gate[j]));
    return k;
}

}  // namespace vb
