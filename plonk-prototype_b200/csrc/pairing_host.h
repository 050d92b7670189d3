// pairing_host.h — BLS12-381 on the HOST: the Fp2 / Fp6 / Fp12 tower, G1 in Jacobian coordinates with the checked
// compressed decoder, G2 in affine coordinates, the Miller loop and the final exponentiation.  Shared by the
// single-proof verifier (verify.cu) and the batched one (verify_batch.cu), which both end in a pairing-product check.
//
// Tower: Fp2 = Fp[u]/(u² + 1), Fp6 = Fp2[v]/(v³ − ξ), Fp12 = Fp6[w]/(w² − v), ξ = u + 1.  G2 is the M-twist
// y² = x³ + 4ξ; untwisting (x, y) ↦ (x/w², y/w³) puts a line through T with slope λ evaluated at P = (xP, yP) at
// (λ·xT − yT) − λ·xP·w² + yP·w³ (scaled by w³, a factor the final exponentiation removes).  The Miller loop runs
// over |x| = 0xd201000000010000; the sign of x only conjugates the result, which does not change whether a product of
// pairings is one.  Final exponentiation: (p⁶ − 1) by conjugation and inversion, then (p⁶ + 1)/r by plain
// square-and-multiply (≈ 2000 squarings — milliseconds; no Frobenius tables to get wrong).
#pragma once
#include <stdint.h>

#include "../../include/pb200.h"
#include "host_field.h"

namespace pairing {

using hostf::HFp;
using hostf::HFr;

// ------------------------------------------------------------------------------------------------ Fp2 / Fp6 / Fp12
struct Fp2 {
    HFp a, b;  // a + b·u
    static Fp2 zero() { return {HFp::zero(), HFp::zero()}; }
    static Fp2 one() { return {HFp::one(), HFp::zero()}; }
    bool is_zero() const { return a.is_zero() && b.is_zero(); }
    bool operator==(const Fp2 &o) const { return a == o.a && b == o.b; }
    Fp2 operator+(const Fp2 &o) const { return {a + o.a, b + o.b}; }
    Fp2 operator-(const Fp2 &o) const { return {a - o.a, b - o.b}; }
    Fp2 neg() const { return {a.neg(), b.neg()}; }
    Fp2 operator*(const Fp2 &o) const {
        const HFp t0 = a * o.a, t1 = b * o.b, t2 = (a + b) * (o.a + o.b);
        return {t0 - t1, t2 - t0 - t1};
    }
    Fp2 sqr() const {
        const HFp t = a * b;
        return {(a + b) * (a - b), t + t};
    }
    Fp2 scale(const HFp &k) const { return {a * k, b * k}; }
    Fp2 mul_xi() const { return {a - b, a + b}; }  // ·(1 + u)
    Fp2 inv() const {
        const HFp t = (a.sqr() + b.sqr()).inv();
        return {a * t, (b * t).neg()};
    }
    Fp2 dbl() const { return *this + *this; }
};
struct Fp6 {
    Fp2 c0, c1, c2;  // c0 + c1·v + c2·v²
    static Fp6 zero() { return {Fp2::zero(), Fp2::zero(), Fp2::zero()}; }
    static Fp6 one() { return {Fp2::one(), Fp2::zero(), Fp2::zero()}; }
    bool operator==(const Fp6 &o) const { return c0 == o.c0 && c1 == o.c1 && c2 == o.c2; }
    Fp6 operator+(const Fp6 &o) const { return {c0 + o.c0, c1 + o.c1, c2 + o.c2}; }
    Fp6 operator-(const Fp6 &o) const { return {c0 - o.c0, c1 - o.c1, c2 - o.c2}; }
    Fp6 neg() const { return {c0.neg(), c1.neg(), c2.neg()}; }
    Fp6 operator*(const Fp6 &o) const {
        const Fp2 t0 = c0 * o.c0, t1 = c1 * o.c1, t2 = c2 * o.c2;
        const Fp2 r0 = t0 + ((c1 + c2) * (o.c1 + o.c2) - t1 - t2).mul_xi();
        const Fp2 r1 = (c0 + c1) * (o.c0 + o.c1) - t0 - t1 + t2.mul_xi();
        const Fp2 r2 = (c0 + c2) * (o.c0 + o.c2) - t0 - t2 + t1;
        return {r0, r1, r2};
    }
    Fp6 mul_v() const { return {c2.mul_xi(), c0, c1}; }
    Fp6 inv() const {
        const Fp2 t0 = c0.sqr() - (c1 * c2).mul_xi();
        const Fp2 t1 = c2.sqr().mul_xi() - c0 * c1;
        const Fp2 t2 = c1.sqr() - c0 * c2;
        const Fp2 d = (c0 * t0 + (c2 * t1 + c1 * t2).mul_xi()).inv();
        return {t0 * d, t1 * d, t2 * d};
    }
};
struct Fp12 {
    Fp6 c0, c1;  // c0 + c1·w
    static Fp12 one() { return {Fp6::one(), Fp6::zero()}; }
    bool operator==(const Fp12 &o) const { return c0 == o.c0 && c1 == o.c1; }
    Fp12 operator*(const Fp12 &o) const {
        const Fp6 t0 = c0 * o.c0, t1 = c1 * o.c1;
        return {t0 + t1.mul_v(), (c0 + c1) * (o.c0 + o.c1) - t0 - t1};
    }
    Fp12 sqr() const { return *this * *this; }
    Fp12 conj() const { return {c0, c1.neg()}; }  // the p⁶-Frobenius
    Fp12 inv() const {
        const Fp6 d = (c0 * c0 - (c1 * c1).mul_v()).inv();
        return {c0 * d, (c1 * d).neg()};
    }
};

// ------------------------------------------------------------------------------------------------ G1 (host, Jacobian)
struct G1J {
    HFp x, y, z;  // z = 0: identity
    static G1J identity() { return {HFp::zero(), HFp::one(), HFp::zero()}; }
    bool is_identity() const { return z.is_zero(); }
};
struct G1A {
    HFp x, y;
    bool inf;
};
inline G1J g1_double(const G1J &p) {
    if (p.is_identity()) return p;
    const HFp a = p.x.sqr(), b = p.y.sqr(), c = b.sqr();
    HFp d = (p.x + b).sqr() - a - c;
    d = d + d;
    const HFp e = a + a + a, f = e.sqr();
    G1J r;
    r.x = f - d - d;
    HFp c8 = c + c;
    c8 = c8 + c8;
    c8 = c8 + c8;
    r.y = e * (d - r.x) - c8;
    r.z = (p.y * p.z);
    r.z = r.z + r.z;
    return r;
}
inline G1J g1_add(const G1J &p, const G1J &q) {
    if (p.is_identity()) return q;
    if (q.is_identity()) return p;
    const HFp z1z1 = p.z.sqr(), z2z2 = q.z.sqr();
    const HFp u1 = p.x * z2z2, u2 = q.x * z1z1;
    const HFp s1 = p.y * q.z * z2z2, s2 = q.y * p.z * z1z1;
    if (u1 == u2) {
        if (s1 == s2) return g1_double(p);
        return G1J::identity();
    }
    const HFp h = u2 - u1, hh = h.sqr(), hhh = h * hh, rr = s2 - s1, v = u1 * hh;
    G1J r;
    r.x = rr.sqr() - hhh - v - v;
    r.y = rr * (v - r.x) - s1 * hhh;
    r.z = p.z * q.z * h;
    return r;
}
inline G1J g1_from_affine(const G1A &a) {
    if (a.inf) return G1J::identity();
    return {a.x, a.y, HFp::one()};
}
inline G1A g1_to_affine(const G1J &p) {
    if (p.is_identity()) return {HFp::zero(), HFp::zero(), true};
    const HFp zi = p.z.inv(), zi2 = zi.sqr();
    return {p.x * zi2, p.y * zi2 * zi, false};
}
inline G1J g1_neg(const G1J &p) { return {p.x, p.y.neg(), p.z}; }
// k·P, k a Montgomery-form scalar
inline G1J g1_mul(const G1J &p, const HFr &k_mont) {
    const HFr k = k_mont.from_mont();
    G1J acc = G1J::identity();
    for (int i = 255; i >= 0; i--) {
        acc = g1_double(acc);
        if ((k.l[i >> 6] >> (i & 63)) & 1) acc = g1_add(acc, p);
    }
    return acc;
}
const uint64_t kG1x[6] = {0x5cb38790fd530c16ull, 0x7817fc679976fff5ull, 0x154f95c7143ba1c1ull,
                          0xf0ae6acdf3d0e747ull, 0xedce6ecc21dbf440ull, 0x120177419e0bfb75ull};
const uint64_t kG1y[6] = {0xbaac93d50ce72271ull, 0x8c22631a7918fd8eull, 0xdd595f13570725ceull,
                          0x51ac582950405194ull, 0x0e1c8c3fad0059c0ull, 0x0bbc3efc5008a26aull};
const uint64_t kFrModulus[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull, 0x73eda753299d7d48ull};

// G1Affine::from_bytes (compressed): range, curve and subgroup checks as upstream.  Returns PB200_G1_* as the device
// decoder (g1_codec.cuh) does; the identity is PB200_G1_IDENTITY with *out the point at infinity.
inline int g1_from_bytes(const uint8_t b[48], G1A *out) {
    if (!(b[0] & 0x80)) return PB200_G1_BAD_FLAGS;
    if (b[0] & 0x40) {
        if (b[0] != 0xc0) return PB200_G1_BAD_FLAGS;
        for (int i = 1; i < 48; i++)
            if (b[i]) return PB200_G1_BAD_FLAGS;
        *out = {HFp::zero(), HFp::zero(), true};
        return PB200_G1_IDENTITY;
    }
    HFp raw;
    for (int i = 0; i < 6; i++) {
        raw.l[i] = 0;
        for (int k = 7; k >= 0; k--) {
            uint8_t byte = b[47 - (8 * i + k)];
            if (8 * i + k == 47) byte &= 0x1f;
            raw.l[i] = (raw.l[i] << 8) | byte;
        }
    }
    if (HFp::geq_mod(raw.l)) return PB200_G1_X_RANGE;
    const HFp x = raw * HFp::r2();
    const HFp rhs = x.sqr() * x + HFp::from_u64(4);
    static const uint64_t kSqrtExp[6] = {0xee7fbfffffffeaabull, 0x07aaffffac54ffffull, 0xd9cc34a83dac3d89ull,
                                         0xd91dd2e13ce144afull, 0x92c6e9ed90d2eb35ull, 0x0680447a8e5ff9a6ull};  // (p + 1)/4
    HFp y = rhs.pow(kSqrtExp, 6);
    if (y.sqr() != rhs) return PB200_G1_NOT_ON_CURVE;
    // choose the root the flag asks for: larger ⇔ 2y ≥ p
    const HFp yc = y.from_mont();
    uint64_t d[6], c = 0;
    for (int i = 0; i < 6; i++) {
        d[i] = (yc.l[i] << 1) | c;
        c = yc.l[i] >> 63;
    }
    const bool larger = c || HFp::geq_mod(d);
    if (larger != (bool)(b[0] & 0x20)) y = y.neg();
    *out = {x, y, false};
    // prime-order subgroup: r·P = O
    G1J acc = G1J::identity();
    const G1J p = g1_from_affine(*out);
    for (int i = 254; i >= 0; i--) {
        acc = g1_double(acc);
        if ((kFrModulus[i >> 6] >> (i & 63)) & 1) acc = g1_add(acc, p);
    }
    return acc.is_identity() ? PB200_G1_OK : PB200_G1_NOT_IN_SUBGROUP;
}

// ------------------------------------------------------------------------------------------------ G2 (affine) / pairing
struct G2A {
    Fp2 x, y;
    bool inf;
};
const uint64_t kG2[4][6] = {
    {0xf5f28fa202940a10ull, 0xb3f5fb2687b4961aull, 0xa1a893b53e2ae580ull, 0x9894999d1a3caee9ull, 0x6f67b7631863366bull, 0x058191924350bcd7ull},
    {0xa5a9c0759e23f606ull, 0xaaa0c59dbccd60c3ull, 0x3bb17e18e2867806ull, 0x1b1ab6cc8541b367ull, 0xc2b6ed0ef2158547ull, 0x11922a097360edf3ull},
    {0x4c730af860494c4aull, 0x597cfa1f5e369c5aull, 0xe7e6856caa0a635aull, 0xbbefb5e96e0d495full, 0x07d3a975f0ef25a2ull, 0x0083fd8e7e80dae5ull},
    {0xadc0fc92df64b05dull, 0x18aa270a2b1461dcull, 0x86adac6a3be4eba0ull, 0x79495c4ec93da33aull, 0xe7175850a43ccaedull, 0x0b2bc2a163de1bf2ull}};
inline G2A g2_generator() { return {{HFp::load(kG2[0]), HFp::load(kG2[1])}, {HFp::load(kG2[2]), HFp::load(kG2[3])}, false}; }
inline bool g2_on_curve(const G2A &p) {
    if (p.inf) return true;
    const Fp2 b2 = {HFp::from_u64(4), HFp::from_u64(4)};
    return p.y.sqr() == p.x.sqr() * p.x + b2;
}
inline G2A g2_add(const G2A &p, const G2A &q) {
    if (p.inf) return q;
    if (q.inf) return p;
    Fp2 lam;
    if (p.x == q.x) {
        if ((p.y + q.y).is_zero()) return {Fp2::zero(), Fp2::zero(), true};
        const Fp2 xx = p.x.sqr();
        lam = (xx + xx + xx) * p.y.dbl().inv();
    } else {
        lam = (q.y - p.y) * (q.x - p.x).inv();
    }
    const Fp2 x3 = lam.sqr() - p.x - q.x;
    return {x3, lam * (p.x - x3) - p.y, false};
}
inline G2A g2_mul(const G2A &p, const HFr &k_mont) {
    const HFr k = k_mont.from_mont();
    G2A acc = {Fp2::zero(), Fp2::zero(), true};
    for (int i = 255; i >= 0; i--) {
        acc = g2_add(acc, acc);
        if ((k.l[i >> 6] >> (i & 63)) & 1) acc = g2_add(acc, p);
    }
    return acc;
}
inline Fp12 line_eval(const G2A &t, const Fp2 &lam, const G1A &p) {
    Fp12 l;
    l.c0 = {lam * t.x - t.y, lam.scale(p.x).neg(), Fp2::zero()};  // w⁰, w² = v
    l.c1 = {Fp2::zero(), {p.y, HFp::zero()}, Fp2::zero()};         // w³ = v·w
    return l;
}
inline Fp12 miller_loop(const G1A &p, const G2A &q) {
    if (p.inf || q.inf) return Fp12::one();
    const uint64_t x_abs = 0xd201000000010000ull;
    Fp12 f = Fp12::one();
    G2A t = q;
    for (int i = 62; i >= 0; i--) {  // bits below the leading one of |x| (bit 63)
        const Fp2 xx = t.x.sqr();
        Fp2 lam = (xx + xx + xx) * t.y.dbl().inv();
        f = f.sqr() * line_eval(t, lam, p);
        t = g2_add(t, t);
        if ((x_abs >> i) & 1) {
            lam = (q.y - t.y) * (q.x - t.x).inv();
            f = f * line_eval(t, lam, p);
            t = g2_add(t, q);
        }
    }
    return f;
}
inline Fp12 final_exponentiation(const Fp12 &f) {
    static const uint64_t kHard[32] = {  // (p⁶ + 1) / r
        0x8739e1cdc0705d6aull, 0x09a5256de0381a16ull, 0x9cf0f70a61c791e2ull, 0x3a09c4497903f76eull, 0x2d7271563890f133ull,
        0x224741b36fec7760ull, 0x338259c22a12bd40ull, 0x38ee1cd4778e0de7ull, 0xc3b5ef4b188a20b0ull, 0x1d615d49e2764d7bull,
        0x816101ddd076117dull, 0xf007c01e7ebe3afcull, 0x27d7bd90935021c3ull, 0xc3b5e2f557c0b15full, 0x5e886c94c4f82384ull,
        0xee6a95db11e63f56ull, 0x2b822f514a9c4f6full, 0x12d6a874d21b73daull, 0x1304275ef499dffbull, 0x967878febcb95d1full,
        0x4744497f8b2f2922ull, 0x85a2e707f0841855ull, 0x9f0c50126c802eecull, 0xfb46e197bd2fa489ull, 0x548ce0809bc5f61aull,
        0xcf56fb1573beaa8cull, 0xad7375a3763bdf7cull, 0xe0ec9031179bdeccull, 0x6579aea83c48c1daull, 0xdbf85ae664cf5bb3ull,
        0x7b6f235c55ca7566ull, 0x000028b314877503ull};
    const Fp12 g = f.conj() * f.inv();
    Fp12 r = Fp12::one();
    for (int i = 2029; i >= 0; i--) {
        r = r.sqr();
        if ((kHard[i >> 6] >> (i & 63)) & 1) r = r * g;
    }
    return r;
}

}  // namespace pairing
