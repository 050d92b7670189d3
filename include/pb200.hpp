// pb200.hpp — header-only C++ host layer over the C ABI (pb200.h), shaped like the Rust API the reference is written
// against, for hosts that cannot use the Rust crates (this image has no cargo / rustc; INTEGRATION.md shows the Rust shim).
//
// Names, argument meaning and error behaviour follow dusk-plonk 0.8.2 / dusk-bls12_381 0.8 (pinned at
// /root/reference/Cargo.toml:19-20; SURVEY.md §8b, App. C):
//   BlsScalar                          dusk_bls12_381::BlsScalar (Montgomery limbs; +, −, *, neg, invert, pow, from(u64))
//   EvaluationDomain::{new_, fft, ifft, coset_fft, coset_ifft}     dusk_plonk::fft::EvaluationDomain
//   msm_variable_base(points, scalars) dusk_bls12_381::multiscalar_mul::msm_variable_base
//   PublicParameters::setup, CommitKey::commit                     dusk_plonk::commitment_scheme::kzg10
//   StandardComposer::{add_input, add, mul, mul_gate, boolean_gate, constrain_to_constant,
//                      add_witness_to_circuit_description}          the calls /root/reference/src/zk/gadgets.rs makes
//   Prover::{new_, mut_cs, preprocess, prove}, verify_proof         dusk_plonk::proof_system
// Upstream's infallible functions stay infallible here: a backend failure throws pb200::Error (the Rust shim panics) —
// there is no CPU fallback.  `EvaluationDomain::new_` throws InvalidEvalDomainSize for log2(size) ≥ 32 like upstream's Err.
#pragma once
#include <array>
#include <map>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../plonk-prototype_b200/csrc/host_field.h"
#include "pb200.h"

namespace pb200 {

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};
struct InvalidEvalDomainSize : Error {
    using Error::Error;
};

// ---- BlsScalar ------------------------------------------------------------------------------------------------
struct BlsScalar {
    hostf::HFr v;  // Montgomery form, fully reduced: the memory image of `BlsScalar.0`
    BlsScalar() : v(hostf::HFr::zero()) {}
    explicit BlsScalar(const hostf::HFr &x) : v(x) {}
    static BlsScalar zero() { return BlsScalar(); }
    static BlsScalar one() { return BlsScalar(hostf::HFr::one()); }
    static BlsScalar from(uint64_t x) { return BlsScalar(hostf::HFr::from_u64(x)); }
    static BlsScalar pow_of_2(uint64_t k) { return from(2).pow(k); }
    // `from_raw([u64; 4])`: canonical little-endian limbs → Montgomery form
    static BlsScalar from_raw(uint64_t l0, uint64_t l1, uint64_t l2, uint64_t l3) {
        hostf::HFr r = hostf::HFr::zero();
        r.l[0] = l0; r.l[1] = l1; r.l[2] = l2; r.l[3] = l3;
        return BlsScalar(r * hostf::HFr::r2());
    }
    BlsScalar operator+(const BlsScalar &o) const { return BlsScalar(v + o.v); }
    BlsScalar operator-(const BlsScalar &o) const { return BlsScalar(v - o.v); }
    BlsScalar operator*(const BlsScalar &o) const { return BlsScalar(v * o.v); }
    BlsScalar operator-() const { return BlsScalar(v.neg()); }
    bool operator==(const BlsScalar &o) const { return v == o.v; }
    bool operator!=(const BlsScalar &o) const { return v != o.v; }
    BlsScalar pow(uint64_t e) const { return BlsScalar(v.pow_u64(e)); }
    // `invert()`: (is_some, value) — zero has no inverse
    std::pair<bool, BlsScalar> invert() const { return {!v.is_zero(), BlsScalar(v.inv())}; }
    // `reduce()`: Montgomery → canonical limbs kept in the same struct (what bits_count / divn work on)
    std::array<uint64_t, 4> reduce() const {
        const hostf::HFr c = v.from_mont();
        return {c.l[0], c.l[1], c.l[2], c.l[3]};
    }
    std::array<uint8_t, 32> to_bytes() const {
        std::array<uint8_t, 32> b;
        hostf::fr_to_bytes(v, b.data());
        return b;
    }
};
static_assert(sizeof(BlsScalar) == 32, "BlsScalar is 4 × u64");

// ---- context ---------------------------------------------------------------------------------------------------
class Context {
  public:
    explicit Context(int device = 0) {
        if (pb200_init(&ctx_, device) != 0) {
            std::string msg = ctx_ ? pb200_last_error(ctx_) : "no usable sm_100 GPU";
            if (ctx_) pb200_destroy(ctx_);
            ctx_ = nullptr;
            throw Error("pb200_init failed: " + msg + " — there is no CPU fallback");
        }
    }
    ~Context() {
        if (ctx_) pb200_destroy(ctx_);
    }
    Context(const Context &) = delete;
    Context &operator=(const Context &) = delete;
    pb200_ctx *raw() const { return ctx_; }
    void check(int rc, const char *what) const {
        if (rc != 0) throw Error(std::string(what) + ": " + pb200_last_error(ctx_));
    }

  private:
    pb200_ctx *ctx_ = nullptr;
};

// ---- EvaluationDomain ------------------------------------------------------------------------------------------
class EvaluationDomain {
  public:
    static EvaluationDomain new_(Context &ctx, size_t num_coeffs) {
        uint32_t log_n = 0;
        if (pb200_domain_log_size(num_coeffs, &log_n) != 0) throw InvalidEvalDomainSize("log2(size) >= 32");
        return EvaluationDomain(ctx, log_n);
    }
    size_t size() const { return (size_t)1 << log_n_; }
    uint32_t log_size_of_group() const { return log_n_; }
    std::vector<BlsScalar> fft(const std::vector<BlsScalar> &coeffs) const { return run(coeffs, 0, 0); }
    std::vector<BlsScalar> ifft(const std::vector<BlsScalar> &evals) const { return run(evals, 1, 0); }
    std::vector<BlsScalar> coset_fft(const std::vector<BlsScalar> &coeffs) const { return run(coeffs, 0, 1); }
    std::vector<BlsScalar> coset_ifft(const std::vector<BlsScalar> &evals) const { return run(evals, 1, 1); }

  private:
    EvaluationDomain(Context &ctx, uint32_t log_n) : ctx_(&ctx), log_n_(log_n) {}
    std::vector<BlsScalar> run(std::vector<BlsScalar> v, int inverse, int coset) const {
        if (v.size() > size()) throw Error("more coefficients than the domain holds");
        v.resize(size());  // upstream zero-pads
        ctx_->check(pb200_ntt(ctx_->raw(), reinterpret_cast<uint64_t *>(v.data()), log_n_, inverse, coset), "pb200_ntt");
        return v;
    }
    Context *ctx_;
    uint32_t log_n_;
};

// ---- Polynomial / Evaluations (dusk-plonk 0.8.2 fft::{Polynomial, Evaluations}; SURVEY.md §8a a8) ------------------
// Dense coefficient form, lowest degree first, no zero coefficients at the top.  evaluate / ruffini run on the GPU
// (pb200_kzg_witness_dev: value and quotient by X − z come out of the same Ruffini pass).
class Polynomial {
  public:
    std::vector<BlsScalar> coeffs;
    static Polynomial zero() { return Polynomial(); }
    static Polynomial from_coefficients_vec(std::vector<BlsScalar> c) {
        while (!c.empty() && c.back() == BlsScalar::zero()) c.pop_back();  // truncate_leading_zeros
        Polynomial p;
        p.coeffs = std::move(c);
        return p;
    }
    static Polynomial from_coefficients_slice(const BlsScalar *c, size_t n) { return from_coefficients_vec(std::vector<BlsScalar>(c, c + n)); }
    bool is_zero() const { return coeffs.empty(); }
    size_t degree() const { return coeffs.empty() ? 0 : coeffs.size() - 1; }  // 0 for the zero polynomial, like upstream
    size_t len() const { return coeffs.size(); }
    BlsScalar evaluate(Context &ctx, const BlsScalar &point) const {
        if (is_zero()) return BlsScalar::zero();
        BlsScalar ev;
        ruffini_dev(ctx, point, nullptr, &ev);
        return ev;
    }
    // (p(X) − p(z)) / (X − z)
    Polynomial ruffini(Context &ctx, const BlsScalar &z) const {
        if (is_zero()) return zero();
        std::vector<BlsScalar> q(coeffs.size());
        BlsScalar ev;
        ruffini_dev(ctx, z, q.data(), &ev);
        q.pop_back();  // the library writes n scalars, the top one zero
        return from_coefficients_vec(std::move(q));
    }

  private:
    void ruffini_dev(Context &ctx, const BlsScalar &z, BlsScalar *quotient, BlsScalar *ev) const {
        const size_t bytes = coeffs.size() * sizeof(BlsScalar);
        void *d_p = nullptr, *d_q = nullptr;
        ctx.check(pb200_malloc(ctx.raw(), &d_p, bytes), "pb200_malloc");
        int rc = pb200_malloc(ctx.raw(), &d_q, bytes);
        if (rc == 0) rc = pb200_h2d(ctx.raw(), d_p, coeffs.data(), bytes);
        if (rc == 0) rc = pb200_kzg_witness_dev(ctx.raw(), static_cast<const uint64_t *>(d_p), coeffs.size(), z.v.l, static_cast<uint64_t *>(d_q), ev->v.l);
        if (rc == 0 && quotient) rc = pb200_d2h(ctx.raw(), quotient, d_q, bytes);
        pb200_free(ctx.raw(), d_p);
        if (d_q) pb200_free(ctx.raw(), d_q);
        ctx.check(rc, "pb200_kzg_witness_dev");
    }
};
// Values over a whole domain; interpolate() = ifft + truncate.
class Evaluations {
  public:
    std::vector<BlsScalar> evals;
    EvaluationDomain domain;
    static Evaluations from_vec_and_domain(std::vector<BlsScalar> evals, const EvaluationDomain &domain) { return Evaluations{std::move(evals), domain}; }
    Polynomial interpolate_by_ref() const { return Polynomial::from_coefficients_vec(domain.ifft(evals)); }
    Polynomial interpolate() const { return interpolate_by_ref(); }
};

// ---- G1 / MSM / KZG --------------------------------------------------------------------------------------------
struct G1Affine {
    uint64_t x[6], y[6];  // Montgomery; the identity is not representable (an SRS never holds it)
};
struct G1Projective {
    uint64_t xyz[18];  // X ‖ Y ‖ Z, not normalised (as upstream's msm_variable_base returns it)
    bool is_identity() const {
        uint64_t o = 0;
        for (int i = 12; i < 18; i++) o |= xyz[i];
        return o == 0;
    }
    // G1Affine::from(self).to_bytes(): 48-byte compressed encoding
    std::array<uint8_t, 48> to_bytes() const {
        std::array<uint8_t, 48> b;
        hostf::g1_projective_to_bytes(xyz, b.data());
        return b;
    }
};
static_assert(sizeof(G1Affine) == 96, "packed affine point");
static_assert(sizeof(G1Projective) == 144, "X ‖ Y ‖ Z");

class CommitKey {
  public:
    // CommitKey { powers_of_g }: uploaded once, resident; pre-doubled window copies for prover-size keys
    CommitKey(Context &ctx, const std::vector<G1Affine> &powers_of_g) : ctx_(&ctx) {
        ctx.check(pb200_srs_upload(ctx.raw(), reinterpret_cast<const uint64_t *>(powers_of_g.data()), powers_of_g.size(), &srs_), "pb200_srs_upload");
        if (powers_of_g.size() <= ((size_t)1 << 22)) ctx.check(pb200_srs_precompute(ctx.raw(), srs_), "pb200_srs_precompute");
    }
    // PublicParameters::setup(max_degree, rng) with the trapdoor supplied by the caller (test / benchmark parameters)
    static CommitKey setup(Context &ctx, size_t max_degree, const BlsScalar &tau) {
        pb200_srs *srs = nullptr;
        ctx.check(pb200_srs_generate(ctx.raw(), tau.v.l, max_degree + 1, &srs), "pb200_srs_generate");
        if (max_degree + 1 <= ((size_t)1 << 22)) ctx.check(pb200_srs_precompute(ctx.raw(), srs), "pb200_srs_precompute");
        return CommitKey(ctx, srs);
    }
    // CommitKey::from_slice: 48-byte compressed points, each decoded and checked on the device like G1Affine::from_bytes (flags,
    // x < p, on the curve, prime-order subgroup).  Throws Error naming the first invalid point.
    static CommitKey from_slice(Context &ctx, const std::vector<uint8_t> &bytes) {
        if (bytes.empty() || bytes.size() % 48) throw Error("CommitKey::from_slice: the length is not a positive multiple of 48");
        const size_t n = bytes.size() / 48;
        pb200_srs *srs = nullptr;
        ctx.check(pb200_srs_from_compressed(ctx.raw(), bytes.data(), n, nullptr, &srs), "pb200_srs_from_compressed");
        CommitKey ck(ctx, srs);
        if (n <= ((size_t)1 << 22)) ctx.check(pb200_srs_precompute(ctx.raw(), srs), "pb200_srs_precompute");
        return ck;
    }
    // CommitKey::to_var_bytes: the points as 48-byte compressed encodings, encoded on the device
    std::vector<uint8_t> to_var_bytes() const {
        const size_t n = pb200_srs_len(srs_);
        std::vector<uint8_t> out(48 * n);
        if (n) ctx_->check(pb200_srs_to_compressed(ctx_->raw(), srs_, 0, n, out.data()), "pb200_srs_to_compressed");
        return out;
    }
    CommitKey(CommitKey &&o) noexcept : ctx_(o.ctx_), srs_(o.srs_) { o.srs_ = nullptr; }
    CommitKey(const CommitKey &) = delete;
    ~CommitKey() {
        if (srs_) pb200_srs_free(ctx_->raw(), srs_);
    }
    size_t max_degree() const { return pb200_srs_len(srs_) - 1; }
    // commit(&Polynomial): degree check, then one MSM over powers_of_g[..len]
    G1Projective commit(const std::vector<BlsScalar> &coeffs) const {
        if (coeffs.size() > pb200_srs_len(srs_)) throw Error("PolynomialDegreeTooLarge");
        G1Projective out;
        ctx_->check(pb200_msm_g1(ctx_->raw(), srs_, 0, reinterpret_cast<const uint64_t *>(coeffs.data()), coeffs.size(), out.xyz), "pb200_msm_g1");
        return out;
    }
    G1Projective commit(const Polynomial &p) const { return commit(p.coeffs); }
    pb200_srs *raw() const { return srs_; }

  private:
    CommitKey(Context &ctx, pb200_srs *srs) : ctx_(&ctx), srs_(srs) {}
    Context *ctx_;
    pb200_srs *srs_ = nullptr;
};

// msm_variable_base(points, scalars): infallible like upstream (a backend failure throws), empty input ⇒ identity.
inline G1Projective msm_variable_base(Context &ctx, const std::vector<G1Affine> &points, const std::vector<BlsScalar> &scalars) {
    if (points.size() != scalars.size()) throw Error("points and scalars differ in length");
    G1Projective out;
    if (points.empty()) {
        ctx.check(pb200_msm_g1(ctx.raw(), nullptr, 0, nullptr, 0, out.xyz), "pb200_msm_g1");
        return out;
    }
    pb200_srs *srs = nullptr;
    ctx.check(pb200_srs_upload(ctx.raw(), reinterpret_cast<const uint64_t *>(points.data()), points.size(), &srs), "pb200_srs_upload");
    const int rc = pb200_msm_g1(ctx.raw(), srs, 0, reinterpret_cast<const uint64_t *>(scalars.data()), scalars.size(), out.xyz);
    pb200_srs_free(ctx.raw(), srs);
    ctx.check(rc, "pb200_msm_g1");
    return out;
}

// multiscalar_mul::pippenger(points, scalars): the iterator form over projective bases (Z = 0: the identity).
inline G1Projective pippenger(Context &ctx, const std::vector<G1Projective> &points, const std::vector<BlsScalar> &scalars) {
    if (points.size() != scalars.size()) throw Error("points and scalars differ in length");
    G1Projective out;
    ctx.check(pb200_pippenger_g1(ctx.raw(), reinterpret_cast<const uint64_t *>(points.data()), reinterpret_cast<const uint64_t *>(scalars.data()),
                                 points.size(), out.xyz),
              "pb200_pippenger_g1");
    return out;
}

// ---- StandardComposer ------------------------------------------------------------------------------------------
typedef uint32_t Variable;

// ---- JubJub on the host (dusk-jubjub 0.10, /root/reference/Cargo.toml:21): witness generation for the ECC gadgets ------
// −x² + y² = 1 + d·x²·y², d = −10240/10241; GENERATOR has y = 18 (x = the root of the curve equation in the prime-order
// subgroup), GENERATOR_NUMS as published — see plonk-prototype_b200/jubjub.py and tests/test_widgets_cpu.py.
namespace jubjub {
struct Affine {
    BlsScalar x, y;
};
inline BlsScalar edwards_d() { return -(BlsScalar::from(10240) * BlsScalar::from(10241).invert().second); }
inline Affine identity() { return {BlsScalar::zero(), BlsScalar::one()}; }
inline Affine generator() {
    return {BlsScalar::from_raw(0x4df7b7ffec7beacaull, 0x2e3ebb21fd6c54edull, 0xf1fbf02d0fd6cce6ull, 0x3fd2814c43ac65a6ull), BlsScalar::from(18)};
}
inline Affine generator_nums() {
    return {BlsScalar::from_raw(0x921710179df76377ull, 0x931e316a39fe4541ull, 0xbd9514c773fd4456ull, 0x5e67b8f316f414f7ull),
            BlsScalar::from_raw(0x6705b707162e3ef8ull, 0x9949ba0f82a5507aull, 0x7b162dbeeb3b34fdull, 0x43d80eb3b2f3eb1bull)};
}
inline Affine add(const Affine &p, const Affine &q) {
    const BlsScalar t = edwards_d() * p.x * q.x * p.y * q.y, one = BlsScalar::one();
    return {(p.x * q.y + p.y * q.x) * (one + t).invert().second, (p.y * q.y + p.x * q.x) * (one - t).invert().second};
}
inline Affine neg(const Affine &p) { return {-p.x, p.y}; }
inline Affine mul(Affine p, std::array<uint64_t, 4> k) {
    Affine acc = identity();
    for (int i = 0; i < 256; i++) {
        if ((k[i >> 6] >> (i & 63)) & 1) acc = add(acc, p);
        p = add(p, p);
    }
    return acc;
}
// `Fr::compute_windowed_naf(2)`: 256 digits in {−1, 0, 1}, least significant first
inline std::array<int8_t, 256> wnaf2(std::array<uint64_t, 4> k) {
    std::array<int8_t, 256> out{};
    auto is_zero = [&]() { return (k[0] | k[1] | k[2] | k[3]) == 0; };
    for (int i = 0; i < 256 && !is_zero(); i++) {
        if (k[0] & 1) {
            const int d = 2 - (int)(k[0] & 3);   // k mod 4 = 1 → +1, = 3 → −1
            out[i] = (int8_t)d;
            if (d == 1) {
                k[0] -= 1;   // k is odd: no borrow
            } else {
                for (int l = 0; l < 4 && ++k[l] == 0; l++) {}
            }
        }
        for (int l = 0; l < 4; l++) k[l] = (k[l] >> 1) | (l < 3 ? k[l + 1] << 63 : 0);
    }
    return out;
}
}  // namespace jubjub

struct Point {  // constraint_system::ecc::Point: a pair of variables
    Variable x, y;
};

class StandardComposer {
  public:
    StandardComposer() {
        zero_var_ = 0;
        zero_var_ = add_witness_to_circuit_description(BlsScalar::zero());
        add_dummy_constraints();
    }
    size_t circuit_size() const { return w_[0].size(); }
    Variable zero_var() const { return zero_var_; }
    const BlsScalar &value_of(Variable v) const { return variables_[v]; }

    Variable add_input(const BlsScalar &s) {
        variables_.push_back(s);
        return (Variable)(variables_.size() - 1);
    }
    // c = q_l·a + q_r·b + q_c + pi, constrained with q_o = −1
    Variable add(std::pair<BlsScalar, Variable> q_l_a, std::pair<BlsScalar, Variable> q_r_b, const BlsScalar &q_c, const BlsScalar *pi = nullptr) {
        BlsScalar c = q_l_a.first * variables_[q_l_a.second] + q_r_b.first * variables_[q_r_b.second] + q_c;
        if (pi) c = c + *pi;
        const Variable out = add_input(c);
        row(q_l_a.second, q_r_b.second, out, zero_var_, BlsScalar::zero(), q_l_a.first, q_r_b.first, -BlsScalar::one(), q_c, pi);
        return out;
    }
    // c = q_m·a·b + q_c + pi, constrained with q_o = −1
    Variable mul(const BlsScalar &q_m, Variable a, Variable b, const BlsScalar &q_c, const BlsScalar *pi = nullptr) {
        BlsScalar c = q_m * variables_[a] * variables_[b] + q_c;
        if (pi) c = c + *pi;
        const Variable out = add_input(c);
        row(a, b, out, zero_var_, q_m, BlsScalar::zero(), BlsScalar::zero(), -BlsScalar::one(), q_c, pi);
        return out;
    }
    void mul_gate(Variable a, Variable b, Variable c, const BlsScalar &q_m, const BlsScalar &q_o, const BlsScalar &q_c, const BlsScalar *pi = nullptr) {
        row(a, b, c, zero_var_, q_m, BlsScalar::zero(), BlsScalar::zero(), q_o, q_c, pi);
    }
    void add_gate(Variable a, Variable b, Variable c, const BlsScalar &q_l, const BlsScalar &q_r, const BlsScalar &q_o, const BlsScalar &q_c,
                  const BlsScalar *pi = nullptr) {
        row(a, b, c, zero_var_, BlsScalar::zero(), q_l, q_r, q_o, q_c, pi);
    }
    void boolean_gate(Variable a) {
        row(a, a, a, zero_var_, BlsScalar::one(), BlsScalar::zero(), BlsScalar::zero(), -BlsScalar::one(), BlsScalar::zero(), nullptr);
    }
    void constrain_to_constant(Variable a, const BlsScalar &constant, const BlsScalar *pi = nullptr) {
        row(a, a, a, zero_var_, BlsScalar::zero(), BlsScalar::one(), BlsScalar::zero(), BlsScalar::zero(), -constant, pi);
    }
    Variable add_witness_to_circuit_description(const BlsScalar &value) {
        const Variable v = add_input(value);
        constrain_to_constant(v, value, nullptr);
        return v;
    }
    void assert_equal(Variable a, Variable b) {
        row(a, b, zero_var_, zero_var_, BlsScalar::zero(), BlsScalar::one(), -BlsScalar::one(), BlsScalar::zero(), BlsScalar::zero(), nullptr);
    }
    // ---- constraint_system::ecc (call sites /root/reference/src/zk/gadgets.rs:34-40, circuits.rs:64-65) ----------------
    // 256 rows of the fixed-base widget over the 2-bit windowed NAF of the scalar (most significant digit first) plus one
    // plain row with the final accumulators; throws if the scalar is not a canonical JubJub scalar (upstream unwraps).
    Point fixed_base_scalar_mul(Variable jubjub_scalar, const jubjub::Affine &generator) {
        const int num_bits = 256;
        std::vector<jubjub::Affine> multiples(num_bits);
        multiples[num_bits - 1] = generator;   // multiples[i] = 2^(255−i)·G pairs with the i-th digit from the top
        for (int i = num_bits - 2; i >= 0; i--) multiples[i] = jubjub::add(multiples[i + 1], multiples[i + 1]);
        const std::array<uint64_t, 4> k = variables_[jubjub_scalar].reduce();
        static const uint64_t order[4] = {0xd0970e5ed6f72cb7ull, 0xa6682093ccc81082ull, 0x06673b0101343b00ull, 0x0e7db4ea6533afa9ull};
        bool below = false;
        for (int l = 3; l >= 0; l--) {
            if (k[l] != order[l]) { below = k[l] < order[l]; break; }
        }
        if (!below) throw Error("fixed_base_scalar_mul: the scalar is not a canonical JubJub scalar");
        const std::array<int8_t, 256> naf = jubjub::wnaf2(k);
        std::vector<BlsScalar> scalar_acc{BlsScalar::zero()}, xy_alphas;
        std::vector<jubjub::Affine> point_acc{jubjub::identity()};
        for (int i = 0; i < num_bits; i++) {
            const int entry = naf[num_bits - 1 - i];
            const jubjub::Affine to_add = entry == 0 ? jubjub::identity() : (entry == 1 ? multiples[i] : jubjub::neg(multiples[i]));
            BlsScalar acc = scalar_acc[i] + scalar_acc[i];
            if (entry == 1) acc = acc + BlsScalar::one();
            if (entry == -1) acc = acc - BlsScalar::one();
            scalar_acc.push_back(acc);
            point_acc.push_back(jubjub::add(point_acc[i], to_add));
            xy_alphas.push_back(to_add.x * to_add.y);
        }
        for (int i = 0; i < num_bits; i++) {
            const Variable acc_x = add_input(point_acc[i].x), acc_y = add_input(point_acc[i].y), accumulated_bit = add_input(scalar_acc[i]);
            if (i == 0) {
                constrain_to_constant(acc_x, BlsScalar::zero());
                constrain_to_constant(acc_y, BlsScalar::one());
                constrain_to_constant(accumulated_bit, BlsScalar::zero());
            }
            const Variable xy_alpha = add_input(xy_alphas[i]);
            row(acc_x, acc_y, xy_alpha, accumulated_bit, BlsScalar::zero(), multiples[i].x, multiples[i].y, BlsScalar::zero(),
                multiples[i].x * multiples[i].y, nullptr, BlsScalar::zero(), /*q_arith=*/false, Q_FIXED);
        }
        const Variable acc_x = add_input(point_acc[num_bits].x), acc_y = add_input(point_acc[num_bits].y);
        const Variable last_accumulated_bit = add_input(scalar_acc[num_bits]);
        row(acc_x, acc_y, zero_var_, last_accumulated_bit, BlsScalar::zero(), BlsScalar::zero(), BlsScalar::zero(), BlsScalar::zero(),
            BlsScalar::zero(), nullptr);   // big_add_gate with zero selectors: the "next" row of the last widget row
        assert_equal(last_accumulated_bit, jubjub_scalar);
        return {acc_x, acc_y};
    }
    Point point_addition_gate(const Point &a, const Point &b) {
        const jubjub::Affine s = jubjub::add({variables_[a.x], variables_[a.y]}, {variables_[b.x], variables_[b.y]});
        const Variable x1_y2 = add_input(variables_[a.x] * variables_[b.y]);
        const Variable x3 = add_input(s.x), y3 = add_input(s.y);
        const BlsScalar z = BlsScalar::zero();
        row(a.x, a.y, b.x, b.y, z, z, z, z, z, nullptr, z, /*q_arith=*/false, Q_VAR);
        row(x3, y3, zero_var_, x1_y2, z, z, z, z, z, nullptr, z, /*q_arith=*/false);
        return {x3, y3};
    }
    void assert_equal_public_point(const Point &p, const jubjub::Affine &public_point) {
        const BlsScalar nx = -public_point.x, ny = -public_point.y;
        constrain_to_constant(p.x, BlsScalar::zero(), &nx);
        constrain_to_constant(p.y, BlsScalar::zero(), &ny);
    }

    // column images for pb200_preprocess / pb200_prove
    pb200_circuit circuit() const {
        pb200_circuit c;
        c.n_gates = circuit_size();
        c.n_vars = variables_.size();
        for (int k = 0; k < 11; k++) c.selectors[k] = (k < 7 || used_[k]) ? reinterpret_cast<const uint64_t *>(q_[k].data()) : nullptr;
        for (int k = 0; k < 4; k++) c.wires[k] = w_[k].data();
        return c;
    }
    const std::vector<BlsScalar> &variables() const { return variables_; }
    const std::map<uint32_t, BlsScalar> &public_inputs_sparse_store() const { return pi_; }

  private:
    enum { QM, QL, QR, QO, QC, Q4, QARITH, Q_RANGE, Q_LOGIC, Q_FIXED, Q_VAR };
    // one row of all eleven selector columns; `widget` = Q_FIXED / Q_VAR sets that selector to one
    void row(Variable a, Variable b, Variable c, Variable d, const BlsScalar &q_m, const BlsScalar &q_l, const BlsScalar &q_r,
             const BlsScalar &q_o, const BlsScalar &q_c, const BlsScalar *pi, const BlsScalar &q_4 = BlsScalar::zero(), bool q_arith = true,
             int widget = -1) {
        const BlsScalar vals[7] = {q_m, q_l, q_r, q_o, q_c, q_4, q_arith ? BlsScalar::one() : BlsScalar::zero()};
        for (int k = 0; k < 7; k++) q_[k].push_back(vals[k]);
        for (int k = 7; k < 11; k++) q_[k].push_back(k == widget ? BlsScalar::one() : BlsScalar::zero());
        if (widget >= 0) used_[widget] = true;
        const Variable w[4] = {a, b, c, d};
        for (int k = 0; k < 4; k++) w_[k].push_back(w[k]);
        if (pi) pi_[(uint32_t)(w_[0].size() - 1)] = *pi;
    }
    void add_dummy_constraints() {
        const Variable six = add_input(BlsScalar::from(6)), one = add_input(BlsScalar::one()), seven = add_input(BlsScalar::from(7)),
                       m20 = add_input(-BlsScalar::from(20));
        row(six, seven, m20, one, BlsScalar::one(), BlsScalar::from(2), BlsScalar::from(3), BlsScalar::from(4), BlsScalar::from(4), nullptr,
            BlsScalar::one());
        row(m20, six, seven, zero_var_, BlsScalar::one(), BlsScalar::one(), BlsScalar::one(), BlsScalar::one(), BlsScalar::from(127), nullptr);
    }
    std::vector<BlsScalar> q_[11];
    bool used_[11] = {};
    std::vector<Variable> w_[4];
    std::vector<BlsScalar> variables_;
    std::map<uint32_t, BlsScalar> pi_;
    Variable zero_var_;
};

// ---- Prover / verify --------------------------------------------------------------------------------------------
typedef std::array<uint8_t, 1040> ProofBytes;
typedef std::array<uint8_t, 15 * 48> VerifierKeyBytes;

class Prover {
  public:
    static Prover new_(Context &ctx, const std::string &label) { return Prover(ctx, label); }
    Prover(Prover &&o) noexcept : ctx_(o.ctx_), label_(std::move(o.label_)), cs_(std::move(o.cs_)), key_(o.key_), vk_(o.vk_) { o.key_ = nullptr; }
    Prover(const Prover &) = delete;
    ~Prover() {
        if (key_) pb200_prover_key_free(ctx_->raw(), key_);
    }
    StandardComposer &mut_cs() { return cs_; }
    size_t circuit_size() const { return cs_.circuit_size(); }
    size_t padded_size() const { return pb200_prover_key_size(key_); }
    const VerifierKeyBytes &verifier_key() const { return vk_; }
    void preprocess(const CommitKey &ck) {
        if (key_) throw Error("CircuitAlreadyPreprocessed");
        const pb200_circuit c = cs_.circuit();
        ctx_->check(pb200_preprocess(ctx_->raw(), ck.raw(), &c, reinterpret_cast<const uint8_t *>(label_.data()), label_.size(), &key_, vk_.data()),
                    "pb200_preprocess");
    }
    ProofBytes prove(const CommitKey &ck) {
        if (!key_) preprocess(ck);
        std::vector<uint32_t> pos;
        std::vector<BlsScalar> val;
        for (const auto &kv : cs_.public_inputs_sparse_store()) {
            pos.push_back(kv.first);
            val.push_back(kv.second);
        }
        ProofBytes proof;
        ctx_->check(pb200_prove(ctx_->raw(), ck.raw(), key_, reinterpret_cast<const uint64_t *>(cs_.variables().data()), pos.data(),
                                reinterpret_cast<const uint64_t *>(val.data()), pos.size(), proof.data()),
                    "pb200_prove");
        return proof;
    }

  private:
    Prover(Context &ctx, const std::string &label) : ctx_(&ctx), label_(label) {}
    Context *ctx_;
    std::string label_;
    StandardComposer cs_;
    pb200_prover_key *key_ = nullptr;
    VerifierKeyBytes vk_{};
};

// circuit::verify_proof: host CPU (pairing), independent of the circuit size.  tau is the trapdoor of the test parameters.
inline bool verify_proof(const VerifierKeyBytes &vk, size_t padded_size, const std::string &label, const ProofBytes &proof,
                         const std::map<uint32_t, BlsScalar> &public_inputs, const BlsScalar &tau) {
    uint64_t beta_h[24];
    if (pb200_opening_key_from_tau(tau.v.l, beta_h) != 0) throw Error("pb200_opening_key_from_tau");
    std::vector<uint32_t> pos;
    std::vector<BlsScalar> val;
    for (const auto &kv : public_inputs) {
        pos.push_back(kv.first);
        val.push_back(kv.second);
    }
    int accepted = 0;
    if (pb200_verify(vk.data(), padded_size, reinterpret_cast<const uint8_t *>(label.data()), label.size(), proof.data(), pos.data(),
                     reinterpret_cast<const uint64_t *>(val.data()), pos.size(), beta_h, &accepted) != 0)
        throw Error("pb200_verify: bad argument");
    return accepted != 0;
}

// Many proofs of one circuit in one batched check on the GPU (pb200_verify_batch): verdict k is what verify_proof returns
// for proofs[k] with public_inputs[k].  Every proof's public inputs must sit at the same gates.  seed: 32 random bytes.
inline std::vector<bool> verify_proofs(Context &ctx, const VerifierKeyBytes &vk, size_t padded_size, const std::string &label,
                                       const std::vector<ProofBytes> &proofs, const std::vector<std::map<uint32_t, BlsScalar>> &public_inputs,
                                       const BlsScalar &tau, const std::array<uint8_t, 32> &seed) {
    if (proofs.size() != public_inputs.size() || proofs.empty()) throw Error("verify_proofs: one public-input map per proof");
    uint64_t beta_h[24];
    if (pb200_opening_key_from_tau(tau.v.l, beta_h) != 0) throw Error("pb200_opening_key_from_tau");
    std::vector<uint32_t> pos;
    for (const auto &kv : public_inputs[0]) pos.push_back(kv.first);
    std::vector<BlsScalar> val;
    std::vector<uint8_t> bytes;
    for (size_t k = 0; k < proofs.size(); k++) {
        if (public_inputs[k].size() != pos.size()) throw Error("verify_proofs: public inputs at different gates");
        size_t j = 0;
        for (const auto &kv : public_inputs[k]) {
            if (kv.first != pos[j++]) throw Error("verify_proofs: public inputs at different gates");
            val.push_back(kv.second);
        }
        bytes.insert(bytes.end(), proofs[k].begin(), proofs[k].end());
    }
    std::vector<uint8_t> accepted(proofs.size());
    int all = 0;
    ctx.check(pb200_verify_batch(ctx.raw(), vk.data(), padded_size, reinterpret_cast<const uint8_t *>(label.data()), label.size(),
                                 bytes.data(), proofs.size(), pos.data(), reinterpret_cast<const uint64_t *>(val.data()), pos.size(), beta_h,
                                 seed.data(), accepted.data(), &all),
              "pb200_verify_batch");
    return std::vector<bool>(accepted.begin(), accepted.end());
}

}  // namespace pb200
