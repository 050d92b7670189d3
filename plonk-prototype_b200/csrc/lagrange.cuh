// lagrange.cuh — the commit key in the Lagrange basis of the n-th roots of unity (lagrange.cu):
//
//   Q_i = [L_i(τ)]G = n⁻¹ · Σ_j ω^(−ij) · P_j      (P_j = [τ^j]G, the first n points of the monomial key)
//
// an inverse NTT over G1: radix-2 Cooley–Tukey stages on bit-reversed XYZZ points, every butterfly multiplying one point
// by its twiddle ω_m^(−j) (double-and-add over the canonical bits; twiddle 1 is skipped), then the n⁻¹ scaling and one
// normalisation to affine per point with a per-thread batch inversion.  No trapdoor is needed, so a key loaded from its
// compressed bytes gets the same table.  Commitments against it take the evaluations of a polynomial on the domain as
// scalars: Σ_i f(ω^i)·Q_i = [f(τ)]G, the same group element as the commitment to f's coefficients.
//
// PB_HD, so the kernels of lagrange.cu run it one thread per butterfly / per group of points and the CPU host emulation
// (tests/host_emu/emu_lagrange.cpp) runs the same code.
#pragma once
#include "g1.cuh"

namespace lagrange {

constexpr uint32_t kNormPer = 8;  // points per thread of the normalisation (one Fp inversion each)

PB_HD uint32_t bitrev(uint32_t i, uint32_t bits) {
    uint32_t r = 0;
    for (uint32_t b = 0; b < bits; b++) r |= ((i >> b) & 1u) << (bits - 1 - b);
    return r;
}
PB_HD G1Xyzz g1_neg(const G1Xyzz &p) {
    G1Xyzz r = p;
    r.y = p.y.neg();
    return r;
}
// k·P for a scalar k in Montgomery form: double-and-add from the top set bit of the canonical value.
PB_HD G1Xyzz g1_mul_fr(const G1Xyzz &p, const Fr &k_mont) {
    const Fr k = k_mont.from_mont();
    int top = 255;
    while (top >= 0 && !((k.l[top >> 5] >> (top & 31)) & 1)) top--;
    if (top < 0) return G1Xyzz::identity();
    G1Xyzz acc = p;
    for (int i = top - 1; i >= 0; i--) {
        acc = g1_dbl(acc);
        if ((k.l[i >> 5] >> (i & 31)) & 1) acc = g1_add(acc, p);
    }
    return acc;
}

// a[bitrev(i)] = P_i
PB_HD void load_point(const G1Affine *bases, uint32_t i, uint32_t log_n, G1Xyzz *a) {
    a[bitrev(i, log_n)] = G1Xyzz::from_affine(bases[i]);
}
// Butterfly k < n/2 of the stage that merges transforms of length `half` into length 2·half; w = ω_(2·half)^(−1).
PB_HD void butterfly(G1Xyzz *a, uint32_t half, uint32_t k, const Fr &w) {
    const uint32_t j = k & (half - 1), i0 = ((k - j) << 1) + j, i1 = i0 + half;
    const G1Xyzz u = a[i0];
    G1Xyzz t = a[i1];
    if (j) t = g1_mul_fr(t, w.pow_u32(j));
    a[i0] = g1_add(u, t);
    a[i1] = g1_add(u, g1_neg(t));
}
// Points [i0, i0 + cnt): scale by n⁻¹, write affine.  An identity result (impossible for a powers-of-τ key: L_i(τ) = 0
// needs τ on the domain) is written as zeros and raises *degenerate.
PB_HD void normalize(G1Xyzz *a, uint32_t i0, uint32_t cnt, const Fr &n_inv, G1Affine *out, uint32_t *degenerate) {
    Fp prefix[kNormPer];  // prefix[k] = Π_{j<k, not identity} ZZ_j·ZZZ_j
    Fp run = Fp::one();
    for (uint32_t k = 0; k < cnt; k++) {
        const G1Xyzz p = g1_mul_fr(a[i0 + k], n_inv);
        a[i0 + k] = p;
        prefix[k] = run;
        if (!p.is_identity()) run = run * (p.zz * p.zzz);
    }
    Fp inv = run.inv();
    for (int k = (int)cnt - 1; k >= 0; k--) {
        const G1Xyzz p = a[i0 + k];
        G1Affine r;
        if (p.is_identity()) {
            r.x = r.y = Fp::zero();
            *degenerate = 1;
        } else {
            const Fp zi = inv * prefix[k];  // 1 / (ZZ·ZZZ)
            inv = inv * (p.zz * p.zzz);
            r.x = p.x * (zi * p.zzz);
            r.y = p.y * (zi * p.zz);
        }
        out[i0 + k] = r;
    }
}

}  // namespace lagrange
