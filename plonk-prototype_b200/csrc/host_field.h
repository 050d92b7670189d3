// host_field.h — Montgomery arithmetic on the HOST for the handful of scalars a proof needs between kernels:
// transcript challenges, the linearisation coefficients, normalising the 11 commitments of a proof to their
// compressed bytes.  A few hundred field operations per proof — everything vector-sized stays on the device.
//
// Mirrors the semantics of dusk-bls12_381 0.8 `Scalar` / `Fp` (pinned at /root/reference/Cargo.toml:20; SURVEY.md §8a a1,
// a2, a9): 64-bit little-endian limbs, Montgomery form, always fully reduced, so the limb image is the one the
// device kernels and the ABI use.
#pragma once
#include <stdint.h>
#include <string.h>

namespace hostf {

typedef unsigned __int128 u128;

template <int N>
struct Params;  // N u64 limbs: modulus, −p⁻¹ mod 2^64, R² mod p

template <>
struct Params<4> {
    static constexpr uint64_t MOD[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull, 0x73eda753299d7d48ull};
    static constexpr uint64_t INV = 0xfffffffeffffffffull;
    static constexpr uint64_t R2[4] = {0xc999e990f3f29c6dull, 0x2b6cedcb87925c23ull, 0x05d314967254398full, 0x0748d9d99f59ff11ull};
};
template <>
struct Params<6> {
    static constexpr uint64_t MOD[6] = {0xb9feffffffffaaabull, 0x1eabfffeb153ffffull, 0x6730d2a0f6b0f624ull,
                                        0x64774b84f38512bfull, 0x4b1ba7b6434bacd7ull, 0x1a0111ea397fe69aull};
    static constexpr uint64_t INV = 0x89f3fffcfffcfffdull;
    static constexpr uint64_t R2[6] = {0xf4df1f341c341746ull, 0x0a76e6a609d104f1ull, 0x8de5476c4c95b6d5ull,
                                       0x67eb88a9939d83c0ull, 0x9a793e85b519952dull, 0x11988fe592cae3aaull};
};

template <int N>
struct El {
    uint64_t l[N];
    typedef Params<N> P;

    static El zero() {
        El r;
        memset(r.l, 0, sizeof(r.l));
        return r;
    }
    static El raw_u64(uint64_t v) {
        El r = zero();
        r.l[0] = v;
        return r;
    }
    static El r2() {
        El r;
        for (int i = 0; i < N; i++) r.l[i] = P::R2[i];
        return r;
    }
    static El from_u64(uint64_t v) { return raw_u64(v) * r2(); }
    static El one() { return from_u64(1); }
    static El load(const uint64_t *p) {
        El r;
        memcpy(r.l, p, sizeof(r.l));
        return r;
    }
    void store(uint64_t *p) const { memcpy(p, l, sizeof(l)); }
    bool is_zero() const {
        uint64_t o = 0;
        for (int i = 0; i < N; i++) o |= l[i];
        return o == 0;
    }
    bool operator==(const El &b) const { return memcmp(l, b.l, sizeof(l)) == 0; }
    bool operator!=(const El &b) const { return !(*this == b); }

    // a ≥ modulus ?
    static bool geq_mod(const uint64_t *a) {
        for (int i = N - 1; i >= 0; i--) {
            if (a[i] != P::MOD[i]) return a[i] > P::MOD[i];
        }
        return true;
    }
    static void sub_mod(uint64_t *a) {
        u128 borrow = 0;
        for (int i = 0; i < N; i++) {
            u128 d = (u128)a[i] - P::MOD[i] - borrow;
            a[i] = (uint64_t)d;
            borrow = (d >> 64) & 1;
        }
    }
    friend El operator+(const El &a, const El &b) {
        El r;
        u128 c = 0;
        for (int i = 0; i < N; i++) {
            c += (u128)a.l[i] + b.l[i];
            r.l[i] = (uint64_t)c;
            c >>= 64;
        }
        if (c || geq_mod(r.l)) sub_mod(r.l);
        return r;
    }
    friend El operator-(const El &a, const El &b) {
        El r;
        u128 borrow = 0;
        for (int i = 0; i < N; i++) {
            u128 d = (u128)a.l[i] - b.l[i] - borrow;
            r.l[i] = (uint64_t)d;
            borrow = (d >> 64) & 1;
        }
        if (borrow) {
            u128 c = 0;
            for (int i = 0; i < N; i++) {
                c += (u128)r.l[i] + P::MOD[i];
                r.l[i] = (uint64_t)c;
                c >>= 64;
            }
        }
        return r;
    }
    El neg() const { return zero() - *this; }
    // Montgomery product a·b·2^(−64N); operand-scanning with interleaved reduction.  Correct for a < 2^(64N), b < p.
    friend El operator*(const El &a, const El &b) {
        uint64_t t[N + 2];
        memset(t, 0, sizeof(t));
        for (int i = 0; i < N; i++) {
            u128 c = 0;
            for (int j = 0; j < N; j++) {
                c += (u128)a.l[j] * b.l[i] + t[j];
                t[j] = (uint64_t)c;
                c >>= 64;
            }
            c += t[N];
            t[N] = (uint64_t)c;
            t[N + 1] = (uint64_t)(c >> 64);
            uint64_t m = t[0] * P::INV;
            c = ((u128)m * P::MOD[0] + t[0]) >> 64;
            for (int j = 1; j < N; j++) {
                c += (u128)m * P::MOD[j] + t[j];
                t[j - 1] = (uint64_t)c;
                c >>= 64;
            }
            c += t[N];
            t[N - 1] = (uint64_t)c;
            t[N] = t[N + 1] + (uint64_t)(c >> 64);
        }
        El r;
        memcpy(r.l, t, sizeof(r.l));
        if (t[N] || geq_mod(r.l)) sub_mod(r.l);
        return r;
    }
    El sqr() const { return *this * *this; }
    El from_mont() const { return *this * raw_u64(1); }
    El pow(const uint64_t *e, int words) const {
        El r = one();
        for (int i = words * 64 - 1; i >= 0; i--) {
            r = r.sqr();
            if ((e[i >> 6] >> (i & 63)) & 1) r = r * *this;
        }
        return r;
    }
    El pow_u64(uint64_t e) const { return pow(&e, 1); }
    El inv() const {  // Fermat; 0 ↦ 0
        uint64_t e[N];
        for (int i = 0; i < N; i++) e[i] = P::MOD[i];
        e[0] -= 2;  // both moduli end in …01 / …ab: no borrow
        return pow(e, N);
    }
};
typedef El<4> HFr;
typedef El<6> HFp;

// ω_n for n = 2^log_n (log_n ≤ 32): the generator of EvaluationDomain::new(n), the root every transform of the prover uses.
inline HFr domain_root(uint32_t log_n) {
    const uint64_t root32[4] = {0xb9b58d8c5f0e466aull, 0x5b1b4c801819d7ecull, 0x0af53ae352a31e64ull, 0x5bf3adda19e9b27bull};  // ω₃₂·R
    HFr w = HFr::load(root32);
    for (uint32_t k = log_n; k < 32; k++) w = w.sqr();
    return w;
}
// BlsScalar::to_bytes: canonical value, 32 bytes little-endian.
inline void fr_to_bytes(const HFr &a, uint8_t out[32]) {
    HFr c = a.from_mont();
    for (int i = 0; i < 4; i++)
        for (int k = 0; k < 8; k++) out[8 * i + k] = (uint8_t)(c.l[i] >> (8 * k));
}
// BlsScalar::from_bytes_wide: 512-bit little-endian integer reduced mod r:  lo·R² ⊗ + hi·R³ ⊗  (⊗ = Montgomery product)
inline HFr fr_from_bytes_wide(const uint8_t in[64]) {
    HFr lo, hi;
    for (int i = 0; i < 4; i++) {
        lo.l[i] = hi.l[i] = 0;
        for (int k = 7; k >= 0; k--) {
            lo.l[i] = (lo.l[i] << 8) | in[8 * i + k];
            hi.l[i] = (hi.l[i] << 8) | in[32 + 8 * i + k];
        }
    }
    const HFr r2 = HFr::r2(), r3 = r2 * r2;
    return lo * r2 + hi * r3;
}
// 32 little-endian bytes → Montgomery form; false when the value is not below r (BlsScalar::from_bytes).
inline bool fr_from_bytes_checked(const uint8_t b[32], HFr &out) {
    HFr raw;
    for (int i = 0; i < 4; i++) {
        raw.l[i] = 0;
        for (int k = 7; k >= 0; k--) raw.l[i] = (raw.l[i] << 8) | b[8 * i + k];
    }
    if (HFr::geq_mod(raw.l)) return false;
    out = raw * HFr::r2();
    return true;
}
// G1Affine::from(G1Projective).to_bytes(): 48 bytes, zcash compressed encoding (SURVEY.md App. A.4).
// xyz: homogeneous projective X ‖ Y ‖ Z in Montgomery form (what pb200_msm_g1 returns).
inline void g1_projective_to_bytes(const uint64_t xyz[18], uint8_t out[48]) {
    HFp X = HFp::load(xyz), Y = HFp::load(xyz + 6), Z = HFp::load(xyz + 12);
    memset(out, 0, 48);
    if (Z.is_zero()) {
        out[0] = 0xc0;
        return;
    }
    HFp zi = Z.inv();
    HFp x = (X * zi).from_mont(), y = (Y * zi).from_mont();
    for (int i = 0; i < 6; i++)
        for (int k = 0; k < 8; k++) out[47 - (8 * i + k)] = (uint8_t)(x.l[i] >> (8 * k));
    // y > (p − 1)/2  ⇔  2y > p − 1  ⇔  2y ≥ p (p odd)
    uint64_t d[7];
    uint64_t c = 0;
    for (int i = 0; i < 6; i++) {
        d[i] = (y.l[i] << 1) | c;
        c = y.l[i] >> 63;
    }
    bool larger = c || HFp::geq_mod(d);
    out[0] |= 0x80 | (larger ? 0x20 : 0);
}

}  // namespace hostf
