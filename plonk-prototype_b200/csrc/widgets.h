// widgets.h — the logic, fixed-base and variable-base widget identities of dusk-plonk 0.8
// (proof_system::widget::{logic, ecc::scalar_mul::fixed_base, ecc::curve_addition}; crate pinned at
// /root/reference/Cargo.toml:19, driven by the reference at /root/reference/src/zk/gadgets.rs:34-40 and circuits.rs:64).
// One generic definition over the field type F: Fr on the device (quotient_kernel, one coset point per thread, and the
// batched verifier), hostf::HFr in the prover's linearisation (plonk.cu) and in pb200_verify (both verifiers through
// verify_batch.cuh) — as upstream shares one formula between `compute_quotient_i` and `compute_linearisation`.
// F needs + − * and F::one().  Formulas restated from memory of the crate (UPSTREAM_ASSUMPTIONS.md §widgets); the logic
// polynomial and the JubJub constant are additionally pinned by mathematics (tests/test_widgets_cpu.py).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define PB_WIDGET_HD __host__ __device__ __forceinline__
#else
#define PB_WIDGET_HD inline
#endif

namespace widgets {

// small integer constant by double-and-add on one()
template <class F>
PB_WIDGET_HD F small(uint32_t v) {
    F acc = F::one(), r = F::one();
    bool have = false;
    for (uint32_t bit = 0; bit < 8; bit++) {
        if ((v >> bit) & 1u) {
            r = have ? r + acc : acc;
            have = true;
        }
        acc = acc + acc;
    }
    return r;   // v ≥ 1
}
template <class F>
PB_WIDGET_HD F quad(const F &x) {
    const F t = x + x;
    return t + t;
}
template <class F>
PB_WIDGET_HD F delta4(const F &f) {   // f(f−1)(f−2)(f−3)
    const F one = F::one();
    const F f1 = f - one, f2 = f1 - one, f3 = f2 - one;
    return (f * f1) * (f2 * f3);
}
// quads a' = a_next − 4a, b' = b_next − 4b, out d' = d_next − 4d, product w = c; q_c = −1 selects XOR, +1 AND
template <class F>
PB_WIDGET_HD F logic_term(const F &a, const F &an, const F &b, const F &bn, const F &c, const F &d, const F &dn, const F &q_c,
                          const F &sep) {
    const F kappa = sep * sep;
    const F qa = an - quad(a), qb = bn - quad(b), qd = dn - quad(d);
    const F &w = c;
    const F ab = qa + qb;
    const F c3 = small<F>(3), c9 = small<F>(9), c18 = c9 + c9, c81 = small<F>(81), c83 = small<F>(83);
    // F = w·(w·(4w − 18(a+b) + 81) + 18(a²+b²) − 81(a+b) + 83);  E = 3(a+b+d') − 2F;  B = q_c·(9d' − 3(a+b))
    F t = (quad(w) - c18 * ab + c81) * w;
    t = t + c18 * (qa * qa + qb * qb) - c81 * ab + c83;
    const F f = t * w;
    const F e = c3 * (ab + qd) - (f + f);
    const F bb = q_c * (c9 * qd - c3 * ab);
    F acc = bb + e;
    acc = acc * kappa + (w - qa * qb);
    acc = acc * kappa + delta4(qd);
    acc = acc * kappa + delta4(qb);
    acc = acc * kappa + delta4(qa);
    return acc * sep;
}
// acc (a, b) + bit·(x_β, y_β) = (a_next, b_next) on JubJub, bit = d_next − 2d ∈ {−1, 0, 1}, c = x_α·y_α;
// x_β, y_β, x_β·y_β are the row's q_l, q_r, q_c
template <class F>
PB_WIDGET_HD F fixed_base_term(const F &a, const F &an, const F &b, const F &bn, const F &c, const F &d, const F &dn, const F &q_l,
                               const F &q_r, const F &q_c, const F &sep, const F &edwards_d) {
    const F one = F::one();
    const F kappa = sep * sep;
    const F bit = dn - (d + d);
    const F bit_cons = (bit * (bit - one)) * (bit + one);
    const F y_alpha = (bit * bit) * (q_r - one) + one;
    const F x_alpha = bit * q_l;
    const F xy_cons = bit * q_c - c;
    const F t = ((c * a) * b) * edwards_d;
    const F x_cons = an + an * t - (a * y_alpha + b * x_alpha);
    const F y_cons = bn - bn * t - (b * y_alpha + a * x_alpha);
    F acc = y_cons;
    acc = acc * kappa + x_cons;
    acc = acc * kappa + xy_cons;
    acc = acc * kappa + bit_cons;
    return acc * sep;
}
// (x1, y1) = (a, b), (x2, y2) = (c, d), (x3, y3) = (a_next, b_next), x1·y2 = d_next
template <class F>
PB_WIDGET_HD F var_base_term(const F &a, const F &an, const F &b, const F &bn, const F &c, const F &d, const F &dn, const F &sep,
                             const F &edwards_d) {
    const F kappa = sep * sep;
    const F y1x2 = b * c, y1y2 = b * d, x1x2 = a * c;
    const F xy_cons = a * d - dn;
    const F t = (edwards_d * dn) * y1x2;
    const F x3_cons = dn + y1x2 - (an + an * t);
    const F y3_cons = y1y2 + x1x2 - (bn - bn * t);
    F acc = y3_cons;
    acc = acc * kappa + x3_cons;
    acc = acc * kappa + xy_cons;
    return acc * sep;
}

}  // namespace widgets
