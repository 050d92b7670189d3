// g1_codec.cuh — the 48-byte compressed (zcash) encoding of BLS12-381 G1 points, checked decoding and encoding.
//
// Replaces (on the GPU) dusk-bls12_381 0.8 `G1Affine::{from_bytes, to_bytes}` (crate pinned at /root/reference/Cargo.toml:20;
// layout restated in UPSTREAM_ASSUMPTIONS.md §Serialisation), the per-point work of `CommitKey::{from_slice, to_var_bytes}`:
//   byte 0, bit 7  compressed (must be set)
//   byte 0, bit 6  identity   (then the encoding must be exactly c0 00…00)
//   byte 0, bit 5  y is the larger of the two roots: 2·y ≥ p, y canonical
//   the other 381 bits: x, big-endian, canonical (x < p)
// Decoding recovers y = (x³ + 4)^((p+1)/4) (p ≡ 3 mod 4) and accepts the point only if y² = x³ + 4 and P lies in the
// prime-order subgroup.  The subgroup test is Scott's endomorphism test (eprint 2021/1130 §6, proof of correctness in
// 2022/352), the one zkcrypto's `is_torsion_free` uses: P ∈ G1 ⇔ φ(P) = −[x²]P, φ(x, y) = (β·x, y), x = −0xd201000000010000.
// It costs two 64-bit scalar multiplications instead of one by the 255-bit r, and decides exactly what r·P = O decides.
//
// Everything is PB_HD, so the kernels (csrc/srs_io.cu) and the CPU host emulation (tests/host_emu/emu_srs.cpp) run the same
// code.  The instruction stream does not depend on the data except for the early exits of invalid points and the
// exceptional branches of the group law (reached only by points of small order): a warp of valid points does not diverge.
//
// Fp multiplications per valid point (squarings counted as multiplications): 606 in the square root (378 squarings and
// 228 multiplications: (p+1)/4 has 379 bits, 229 of them set), 2 × 637 in the two multiplications by |x| (63 doublings of
// 9 and 5 additions of 14 each), and 8 for the conversions, the curve equation and the final comparison: 1,888.
#pragma once
#include "../../include/pb200.h"
#include "g1.cuh"

namespace g1codec {

// (p + 1) / 4 as 12 little-endian u32 words; bit 378 is the top bit.
PB_HD constexpr uint32_t sqrt_exp(int i) {
    constexpr uint32_t v[12] = {0xffffeaabu, 0xee7fbfffu, 0xac54ffffu, 0x07aaffffu, 0x3dac3d89u, 0xd9cc34a8u,
                                0x3ce144afu, 0xd91dd2e1u, 0x90d2eb35u, 0x92c6e9edu, 0x8e5ff9a6u, 0x0680447au};
    return v[i];
}
// β, a primitive cube root of unity in Fp, in Montgomery form.  Of the two, β = 0x5f19672fdf76ce51ba69c6076a0f77eaddb3a93b
// e6f89688de17d813620a00022e01fffffffefffe is the one with φ(G) = −[x²]G for the generator G: with g = 2 (the smallest
// non-cube), the roots are g^((p−1)/3) and its square, and only the first satisfies the equation on G (the other gives
// φ(P) = [x⁴]P instead, since the two eigenvalues of φ on G1 are −x² and its square mod r).  tests/test_srs_io_cpu.py
// re-derives this.
PB_HD constexpr uint32_t beta_mont(int i) {
    constexpr uint32_t v[12] = {0x798a64e8u, 0x30f1361bu, 0x7ece5a2au, 0xf3b8ddabu, 0xc61577f7u, 0x16a8ca3au,
                                0x74fd029bu, 0xc26a2ff8u, 0x60701c6eu, 0x3636b766u, 0x241b6160u, 0x051ba4abu};
    return v[i];
}
constexpr uint64_t kXAbs = 0xd201000000010000ull;  // |x|, the BLS parameter; bits 63, 62, 60, 57, 48, 16

PB_HD uint32_t bswap32(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(v, 0, 0x0123);
#else
    return (v >> 24) | ((v >> 8) & 0xff00u) | ((v << 8) & 0xff0000u) | (v << 24);
#endif
}
PB_HD Fp beta() {
    Fp b;
#pragma unroll
    for (int i = 0; i < 12; i++) b.l[i] = beta_mont(i);
    return b;
}
// 2·y ≥ p for a canonical y: the larger root (y > (p − 1)/2, the lexicographic order of upstream's `lexicographically_largest`)
PB_HD bool is_larger_root(const Fp &y_canonical) {
    uint32_t d[12];
    d[0] = y_canonical.l[0] << 1;
#pragma unroll
    for (int i = 1; i < 12; i++) d[i] = (y_canonical.l[i] << 1) | (y_canonical.l[i - 1] >> 31);  // y < 2^381: no bit lost
    (void)cc::sub_cc(d[0], FpParams::mod(0));
#pragma unroll
    for (int i = 1; i < 12; i++) (void)cc::subc_cc(d[i], FpParams::mod(i));
    return cc::subc(0, 0) == 0;  // no borrow: 2y ≥ p
}
// r^((p+1)/4) by left-to-right square-and-multiply from the top bit; the exponent is a constant, so every thread takes the
// same branches.  The outer loop is unrolled (each word a compile-time constant), the inner one is not (code size).
PB_HD Fp pow_sqrt_exp(const Fp &a) {
    Fp r = a;
#pragma unroll
    for (int w = 11; w >= 0; w--) {
        const uint32_t e = sqrt_exp(w);
        const int top = w == 11 ? 25 : 31;  // word 11 is 0x0680447a: its bit 26 is the exponent's top bit, already in r
#pragma unroll 1
        for (int j = top; j >= 0; j--) {
            r = r.sqr();
            if ((e >> j) & 1) r = r * a;
        }
    }
    return r;
}
// [|x|]·P by double-and-add from the top bit, starting from P itself: 63 doublings and 5 additions.  g1_dbl / g1_add handle
// the identity and equal or opposite operands, which only points of small order reach.
PB_HD G1Xyzz mul_by_x_abs(const G1Xyzz &p) {
    G1Xyzz acc = p;
#pragma unroll 1
    for (int i = 62; i >= 0; i--) {
        acc = g1_dbl(acc);
        if ((kXAbs >> i) & 1) acc = g1_add(acc, p);
    }
    return acc;
}

}  // namespace g1codec

// φ(P) = −[x²]P for a point P on the curve: the prime-order-subgroup test.  [x²]P = [|x|]([|x|]P) in XYZZ; the comparison
// with (β·x, y) needs no inversion: β·x·ZZ = X and y·ZZZ = −Y.  [x²]P = O (P of order dividing x²) is never equal to φ(P).
PB_HD bool g1_in_subgroup(const G1Affine &p) {
    const G1Xyzz q = g1codec::mul_by_x_abs(g1codec::mul_by_x_abs(G1Xyzz::from_affine(p)));
    if (q.is_identity()) return false;
    const bool x_ok = (g1codec::beta() * p.x) * q.zz == q.x;
    const bool y_ok = (p.y * q.zzz + q.y).is_zero();
    return x_ok && y_ok;
}

// G1Affine::from_bytes on the encoding held as 12 u32 words in memory order (w[k] = bytes 4k..4k+3, little-endian loads).
// Returns PB200_G1_* (include/pb200.h); `out` (Montgomery form) is written only for PB200_G1_OK.
PB_HD int g1_decode_checked_words(const uint32_t w[12], G1Affine &out) {
    const uint32_t flags = w[0] & 0xffu;
    if (!(flags & 0x80u)) return PB200_G1_BAD_FLAGS;
    if (flags & 0x40u) {  // identity: exactly c0 00…00, and even then not representable (pb200.h conventions)
        uint32_t rest = w[0] & 0xffffff00u;
#pragma unroll
        for (int k = 1; k < 12; k++) rest |= w[k];
        return (flags == 0xc0u && rest == 0) ? PB200_G1_IDENTITY : PB200_G1_BAD_FLAGS;
    }
    Fp x;  // big-endian bytes → little-endian limbs; the flag bits are the top three bits of limb 11
#pragma unroll
    for (int j = 0; j < 12; j++) x.l[j] = g1codec::bswap32(w[11 - j]);
    x.l[11] &= 0x1fffffffu;
    (void)cc::sub_cc(x.l[0], FpParams::mod(0));
#pragma unroll
    for (int i = 1; i < 12; i++) (void)cc::subc_cc(x.l[i], FpParams::mod(i));
    if (cc::subc(0, 0) == 0) return PB200_G1_X_RANGE;  // x − p did not borrow: x ≥ p
    x = x.to_mont();
    const Fp four = Fp::one().dbl().dbl();
    const Fp rhs = x.sqr() * x + four;
    Fp y = g1codec::pow_sqrt_exp(rhs);
    if (y.sqr() != rhs) return PB200_G1_NOT_ON_CURVE;
    if (g1codec::is_larger_root(y.from_mont()) != ((flags & 0x20u) != 0)) y = y.neg();
    G1Affine p;
    p.x = x;
    p.y = y;
    if (!g1_in_subgroup(p)) return PB200_G1_NOT_IN_SUBGROUP;
    out = p;
    return PB200_G1_OK;
}
PB_HD int g1_decode_checked(const uint8_t b[48], G1Affine &out) {
    uint32_t w[12];
#pragma unroll
    for (int k = 0; k < 12; k++)
        w[k] = (uint32_t)b[4 * k] | ((uint32_t)b[4 * k + 1] << 8) | ((uint32_t)b[4 * k + 2] << 16) | ((uint32_t)b[4 * k + 3] << 24);
    return g1_decode_checked_words(w, out);
}

// G1Affine::to_bytes of a finite point (Montgomery form in, canonical bytes out), as 12 u32 words in memory order.
PB_HD void g1_encode_words(const G1Affine &p, uint32_t w[12]) {
    const Fp x = p.x.from_mont(), y = p.y.from_mont();
#pragma unroll
    for (int k = 0; k < 12; k++) w[k] = g1codec::bswap32(x.l[11 - k]);
    w[0] |= 0x80u | (g1codec::is_larger_root(y) ? 0x20u : 0u);  // byte 0 is the low byte of word 0
}
PB_HD void g1_encode(const G1Affine &p, uint8_t out[48]) {
    uint32_t w[12];
    g1_encode_words(p, w);
#pragma unroll
    for (int k = 0; k < 12; k++)
#pragma unroll
        for (int j = 0; j < 4; j++) out[4 * k + j] = (uint8_t)(w[k] >> (8 * j));
}
