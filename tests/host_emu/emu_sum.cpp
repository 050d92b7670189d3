// Host-emulation harness for the sum of products (Field::mul2_sum_*) and the G1 formulas that use it for Y3: the device
// templates of csrc/field.cuh and csrc/g1.cuh compiled for the CPU with the carry flag emulated (PB200_HOST_EMU).
#define PB200_HOST_EMU 1
#include "../../plonk-prototype_b200/csrc/g1.cuh"
#include <cstddef>
#include <cstring>

static bool below_2p(const Fp &v) {   // v − 2p borrows
    int64_t borrow = 0;
    for (int i = 0; i < Fp::N; i++) {
        const int64_t t = (int64_t)v.l[i] - (int64_t)Fp::mod2(i) - borrow;
        borrow = t < 0;
    }
    return borrow != 0;
}
static bool below_p(const Fp &v) { return v == v.canonical() && below_2p(v); }
static Fp ld(const uint32_t *p) { Fp r; memcpy(r.l, p, 48); return r; }
static G1Affine ld_aff(const uint32_t *p) { G1Affine a; memcpy(a.x.l, p, 48); memcpy(a.y.l, p + 12, 48); return a; }
static void st_affine(const G1Xyzz &v, uint32_t *o) {   // 24 words x‖y (Montgomery, canonical), then 1 word "is identity"
    G1Affine a;
    if (!g1_to_affine(v, a)) { memset(o, 0, 96); o[24] = 1; return; }
    memcpy(o, a.x.l, 48); memcpy(o + 12, a.y.l, 48); o[24] = 0;
}
static void check_lazy(const G1Xyzz &v) {
    if (!below_2p(v.x) || !below_2p(v.y) || !below_2p(v.zz) || !below_2p(v.zzz)) __builtin_trap();
}
static void check_canonical(const G1Xyzz &v) {
    if (!below_p(v.x) || !below_p(v.y) || !below_p(v.zz) || !below_p(v.zzz)) __builtin_trap();
}
// P as XYZZ with ZZ ≠ 1: 2P − P through g1_dbl_affine and g1_add
static G1Xyzz rescaled(const G1Affine &p) {
    G1Xyzz np = G1Xyzz::from_affine(p);
    np.y = np.y.neg();
    return g1_add(g1_dbl_affine(p), np);
}

extern "C" {
// o = mul2_sum_unreduced(a, b, c, d) as computed (lazy, traps unless < 2p); the canonical and lazy wrappers must agree with it
void emu_mul2_sum(const uint32_t *a, const uint32_t *b, const uint32_t *c, const uint32_t *d, uint32_t *o, size_t n) {
    for (size_t i = 0; i < n; i++) {
        const Fp x = ld(a + 12 * i), y = ld(b + 12 * i), z = ld(c + 12 * i), w = ld(d + 12 * i);
        const Fp r = Fp::mul2_sum_unreduced(x, y, z, w);
        if (!below_2p(r)) __builtin_trap();
        if (Fp::mul2_sum_lazy(x, y, z, w) != r || Fp::mul2_sum(x, y, z, w) != r.canonical()) __builtin_trap();
        memcpy(o + 12 * i, r.l, 48);
    }
}
void emu_neg_2p(const uint32_t *a, uint32_t *o, size_t n) {
    for (size_t i = 0; i < n; i++) memcpy(o + 12 * i, ld(a + 12 * i).neg_2p().l, 48);
}
// One chain per call over m affine points (24 words each), result as 25 words:
//   op 0: acc = identity; acc = g1_madd_lazy(acc, P_j)         (every coordinate checked < 2p after every step)
//   op 1: acc = identity; acc = g1_add(acc, P_j with ZZ ≠ 1)    (checked canonical after every step)
//   op 2: acc = identity; acc = g1_dbl(g1_add(acc, P_j with ZZ ≠ 1))
//   op 3: acc = identity; acc = g1_add(P_j with ZZ ≠ 1, acc)    (operands swapped)
//   op 4: acc = g1_dbl_affine(P_0)                              (m = 1)
void emu_g1_chain(int op, const uint32_t *pts, size_t m, uint32_t *o) {
    G1Xyzz acc = G1Xyzz::identity();
    for (size_t j = 0; j < m; j++) {
        const G1Affine p = ld_aff(pts + 24 * j);
        switch (op) {
            case 0: g1_madd_lazy(acc, p); check_lazy(acc); break;
            case 1: acc = g1_add(acc, rescaled(p)); check_canonical(acc); break;
            case 2: acc = g1_dbl(g1_add(acc, rescaled(p))); check_canonical(acc); break;
            case 3: acc = g1_add(rescaled(p), acc); check_canonical(acc); break;
            case 4: acc = g1_dbl_affine(p); check_canonical(acc); break;
            default: __builtin_trap();
        }
    }
    st_affine(op == 0 ? g1_canonical(acc) : acc, o);
}
}
