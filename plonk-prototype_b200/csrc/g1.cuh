// g1.cuh — BLS12-381 G1 (y² = x³ + 4 over Fp) group law in extended-Jacobian "XYZZ" coordinates.
//
// Replaces (on the GPU) dusk-bls12_381 0.8 `G1Projective::{add, add_mixed, double}` and
// `G1Affine::from(G1Projective)` (crate pinned at /root/reference/Cargo.toml:20; SURVEY.md §8a a10-a11).
// Upstream uses complete homogeneous-projective formulas; the result of an MSM is a group element, so
// any correct group law gives the same canonical affine output (SURVEY.md §0.2).  XYZZ is used because
// a mixed addition costs 8M + 2S against 11M+ for the complete formula.
//   x = X/ZZ, y = Y/ZZZ, ZZ³ = ZZZ²; identity ⇔ ZZ = 0.
// Exceptional cases (equal points, opposite points, identity operands) are handled by explicit
// branches — rare for random inputs, but structured prover scalars and repeated bases hit them.
#pragma once
#include "field.cuh"

struct G1Affine {  // never the identity (SURVEY.md §8b: the ABI cannot encode it)
    Fp x, y;
};
struct G1Xyzz {
    Fp x, y, zz, zzz;
    PB_HD bool is_identity() const { return zz.is_zero(); }
    PB_HD static G1Xyzz identity() {
        G1Xyzz r;
        r.x = Fp::zero();
        r.y = Fp::one();
        r.zz = Fp::zero();
        r.zzz = Fp::zero();
        return r;
    }
    PB_HD static G1Xyzz from_affine(const G1Affine &p) {
        G1Xyzz r;
        r.x = p.x;
        r.y = p.y;
        r.zz = Fp::one();
        r.zzz = Fp::one();
        return r;
    }
};

// 2·P for an affine P (mdbl-2008-s-1).  y ≠ 0 for every point of the prime-order subgroup.
PB_HD G1Xyzz g1_dbl_affine(const G1Affine &p) {
    Fp u = p.y.dbl();
    Fp v = u.sqr();
    Fp w = u * v;
    Fp s = p.x * v;
    Fp xx = p.x.sqr();
    Fp m = xx.dbl() + xx;
    G1Xyzz r;
    r.x = m.sqr() - s.dbl();
    r.y = Fp::mul2_sum(m, s - r.x, w, p.y.neg_2p());   // m·(s − x3) − w·y, one reduction
    r.zz = v;
    r.zzz = w;
    return r;
}
// 2·P (dbl-2008-s-1)
PB_HD G1Xyzz g1_dbl(const G1Xyzz &p) {
    if (p.is_identity()) return p;
    Fp u = p.y.dbl();
    Fp v = u.sqr();
    Fp w = u * v;
    Fp s = p.x * v;
    Fp xx = p.x.sqr();
    Fp m = xx.dbl() + xx;
    G1Xyzz r;
    r.x = m.sqr() - s.dbl();
    r.y = Fp::mul2_sum(m, s - r.x, w, p.y.neg_2p());   // m·(s − x3) − w·y, one reduction
    r.zz = v * p.zz;
    r.zzz = w * p.zzz;
    return r;
}
// acc += P, P affine (madd-2008-s): 8M + 2S on the common path.
PB_HD void g1_madd(G1Xyzz &acc, const G1Affine &p) {
    if (acc.is_identity()) {
        acc = G1Xyzz::from_affine(p);
        return;
    }
    Fp u2 = p.x * acc.zz;
    Fp s2 = p.y * acc.zzz;
    Fp pp_ = u2 - acc.x;
    Fp r = s2 - acc.y;
    if (pp_.is_zero()) {
        if (r.is_zero()) acc = g1_dbl_affine(p);  // same point
        else acc = G1Xyzz::identity();            // opposite points
        return;
    }
    Fp pp = pp_.sqr();
    Fp ppp = pp_ * pp;
    Fp q = acc.x * pp;
    Fp x3 = r.sqr() - ppp - q.dbl();
    acc.y = Fp::mul2_sum(r, q - x3, acc.y.neg_2p(), ppp);   // r·(q − x3) − Y1·PPP, one reduction
    acc.x = x3;
    acc.zz = acc.zz * pp;
    acc.zzz = acc.zzz * ppp;
}
// The same mixed addition on the lazy representation (field.cuh): acc's coordinates live in [0, 2p) between additions, no
// product is brought below p (Fp has three spare bits), sums and differences are taken mod 2p.  Used by the accumulation
// kernel only, which canonicalises a run's sum before it leaves the registers.  The identity is still ZZ = 0 exactly: a
// product is ≡ 0 only if a factor is, and the one factor that can be (P ≡ 0: equal or opposite points) returns early.
PB_HD void g1_madd_lazy(G1Xyzz &acc, const G1Affine &p) {
    if (acc.is_identity()) {
        acc = G1Xyzz::from_affine(p);
        return;
    }
    const Fp u2 = Fp::mul_lazy2(p.x, acc.zz), s2 = Fp::mul_lazy2(p.y, acc.zzz);
    const Fp pp_ = Fp::sub_lazy(u2, acc.x), r = Fp::sub_lazy(s2, acc.y);
    if (pp_.is_zero_lazy()) {
        if (r.is_zero_lazy()) acc = g1_dbl_affine(p);  // same point
        else acc = G1Xyzz::identity();                 // opposite points
        return;
    }
    const Fp pp = Fp::sqr_lazy(pp_), ppp = Fp::mul_lazy2(pp_, pp), q = Fp::mul_lazy2(acc.x, pp);
    const Fp x3 = Fp::sub_lazy(Fp::sub_lazy(Fp::sqr_lazy(r), ppp), Fp::add_lazy(q, q));
    acc.y = Fp::mul2_sum_lazy(r, Fp::sub_lazy(q, x3), acc.y.neg_2p(), ppp);   // r·(q − x3) − Y1·PPP, one reduction
    acc.x = x3;
    acc.zz = Fp::mul_lazy2(acc.zz, pp);
    acc.zzz = Fp::mul_lazy2(acc.zzz, ppp);
}
PB_HD G1Xyzz g1_canonical(const G1Xyzz &a) {
    G1Xyzz r;
    r.x = a.x.canonical();
    r.y = a.y.canonical();
    r.zz = a.zz.canonical();
    r.zzz = a.zzz.canonical();
    return r;
}
// a + b, both XYZZ (add-2008-s): 12M + 2S on the common path.
PB_HD G1Xyzz g1_add(const G1Xyzz &a, const G1Xyzz &b) {
    if (a.is_identity()) return b;
    if (b.is_identity()) return a;
    Fp u1 = a.x * b.zz;
    Fp u2 = b.x * a.zz;
    Fp s1 = a.y * b.zzz;
    Fp s2 = b.y * a.zzz;
    Fp pp_ = u2 - u1;
    Fp r = s2 - s1;
    if (pp_.is_zero()) {
        if (r.is_zero()) return g1_dbl(a);
        return G1Xyzz::identity();
    }
    Fp pp = pp_.sqr();
    Fp ppp = pp_ * pp;
    Fp q = u1 * pp;
    G1Xyzz o;
    o.x = r.sqr() - ppp - q.dbl();
    o.y = Fp::mul2_sum(r, q - o.x, s1.neg_2p(), ppp);   // r·(q − x3) − S1·PPP, one reduction
    o.zz = a.zz * b.zz * pp;
    o.zzz = a.zzz * b.zzz * ppp;
    return o;
}
// k·P for a small non-negative integer k (double-and-add from the top bit).
PB_HD G1Xyzz g1_mul_small(const G1Xyzz &p, uint64_t k) {
    G1Xyzz acc = G1Xyzz::identity();
    for (int i = 63; i >= 0; i--) {
        acc = g1_dbl(acc);
        if ((k >> i) & 1) acc = g1_add(acc, p);
    }
    return acc;
}
// Normalise to affine coordinates (x, y) = (X/ZZ, Y/ZZZ); returns false for the identity.
PB_HD bool g1_to_affine(const G1Xyzz &p, G1Affine &out) {
    if (p.is_identity()) return false;
    Fp t = (p.zz * p.zzz).inv();
    out.x = p.x * (t * p.zzz);
    out.y = p.y * (t * p.zz);
    return true;
}
