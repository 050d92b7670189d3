// field.cuh — Montgomery prime-field arithmetic on 32-bit limbs for sm_100a.
//
// Replaces (on the GPU) the arithmetic of dusk-bls12_381 0.8's `Scalar` (Fr, 4×u64, R = 2^256) and
// `Fp` (6×u64, R = 2^384), pinned by /root/reference/Cargo.toml:20 and reached from the reference
// at /root/reference/src/zk/gadgets.rs:65-66,213,219.  The memory image is identical (little-endian
// limbs, Montgomery form, fully reduced), so 8 resp. 12 u32 limbs alias the Rust 4 resp. 6 u64.
//
// Multiplication is word-serial Montgomery (CIOS) with the partial products split into two
// accumulators — one collecting a[even]·b_i, one a[odd]·b_i one limb higher — so each row is two
// uninterrupted mad.lo.cc/madc.hi.cc carry chains (→ IMAD.WIDE.U32 with carry in SASS) and no
// carry ever has to be re-aligned.  See DESIGN.md §"Field arithmetic" for the derivation and the
// capacity argument (needs modulus < 2^(32N−1); Fr is 255 bits in 256, Fp 381 in 384).
#pragma once
#include "carry.cuh"

template <class P>
struct Field;
#if defined(PB_FIELD_NOINLINE_MUL) && defined(__CUDACC__)
template <class P>
__device__ __noinline__ Field<P> field_mul_noinline(Field<P> a, Field<P> b);  // operands travel in registers
template <class P>
__device__ __noinline__ Field<P> field_sqr_noinline(Field<P> a);
template <class P>
__device__ __noinline__ Field<P> field_mul2_sum_noinline(Field<P> a, Field<P> b, Field<P> c, Field<P> d);
#endif

template <class P>
struct Field {
    static constexpr int N = P::N;
    uint32_t l[N];

    PB_HD static Field zero() {
        Field r;
#pragma unroll
        for (int i = 0; i < N; i++) r.l[i] = 0;
        return r;
    }
    PB_HD static Field one() {  // Montgomery 1 = R mod p
        Field r;
#pragma unroll
        for (int i = 0; i < N; i++) r.l[i] = P::r1(i);
        return r;
    }
    PB_HD static Field r2() {
        Field r;
#pragma unroll
        for (int i = 0; i < N; i++) r.l[i] = P::r2(i);
        return r;
    }
    PB_HD bool is_zero() const {
        uint32_t o = 0;
#pragma unroll
        for (int i = 0; i < N; i++) o |= l[i];
        return o == 0;
    }
    PB_HD bool operator==(const Field &b) const {
        uint32_t o = 0;
#pragma unroll
        for (int i = 0; i < N; i++) o |= l[i] ^ b.l[i];
        return o == 0;
    }
    PB_HD bool operator!=(const Field &b) const { return !(*this == b); }

    // r = a − p if a ≥ p else a   (a < 2p)
    PB_HD static Field reduce_once(const Field &a) {
        Field d;
        d.l[0] = cc::sub_cc(a.l[0], P::mod(0));
#pragma unroll
        for (int i = 1; i < N; i++) d.l[i] = cc::subc_cc(a.l[i], P::mod(i));
        uint32_t borrow = cc::subc(0, 0);  // 0xffffffff when a < p
        Field r;
#pragma unroll
        for (int i = 0; i < N; i++) r.l[i] = borrow ? a.l[i] : d.l[i];
        return r;
    }
    PB_HD friend Field operator+(const Field &a, const Field &b) {
        Field s;
        s.l[0] = cc::add_cc(a.l[0], b.l[0]);
#pragma unroll
        for (int i = 1; i < N - 1; i++) s.l[i] = cc::addc_cc(a.l[i], b.l[i]);
        s.l[N - 1] = cc::addc(a.l[N - 1], b.l[N - 1]);  // a+b < 2p < 2^(32N): no carry out
        return reduce_once(s);
    }
    // d += K·p when mask ≠ 0 (K = 1, 2), limb-wise with carry.  On the device the additions are PREDICATED (N instructions)
    // instead of masking the constant first (2N): the kernels that use this are bound by dispatch slots (DESIGN.md §4).
    template <int K>
    PB_HD static constexpr uint32_t kp(int i) { return K == 1 ? P::mod(i) : mod2(i); }
    template <int K>
    PB_HD static void cond_add_kp(Field &d, uint32_t mask) {
#if defined(__CUDA_ARCH__)
        if constexpr (N == 8) {
            asm volatile(
                "{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %8, 0;\n\t"
                "@q add.cc.u32 %0, %0, %9;\n\t@q addc.cc.u32 %1, %1, %10;\n\t@q addc.cc.u32 %2, %2, %11;\n\t@q addc.cc.u32 %3, %3, %12;\n\t"
                "@q addc.cc.u32 %4, %4, %13;\n\t@q addc.cc.u32 %5, %5, %14;\n\t@q addc.cc.u32 %6, %6, %15;\n\t@q addc.u32 %7, %7, %16;\n\t}"
                : "+r"(d.l[0]), "+r"(d.l[1]), "+r"(d.l[2]), "+r"(d.l[3]), "+r"(d.l[4]), "+r"(d.l[5]), "+r"(d.l[6]), "+r"(d.l[7])
                : "r"(mask), "n"(kp<K>(0)), "n"(kp<K>(1)), "n"(kp<K>(2)), "n"(kp<K>(3)), "n"(kp<K>(4)), "n"(kp<K>(5)), "n"(kp<K>(6)), "n"(kp<K>(7)));
            return;
        } else if constexpr (N == 12) {
            asm volatile(
                "{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %12, 0;\n\t"
                "@q add.cc.u32 %0, %0, %13;\n\t@q addc.cc.u32 %1, %1, %14;\n\t@q addc.cc.u32 %2, %2, %15;\n\t@q addc.cc.u32 %3, %3, %16;\n\t"
                "@q addc.cc.u32 %4, %4, %17;\n\t@q addc.cc.u32 %5, %5, %18;\n\t@q addc.cc.u32 %6, %6, %19;\n\t@q addc.cc.u32 %7, %7, %20;\n\t"
                "@q addc.cc.u32 %8, %8, %21;\n\t@q addc.cc.u32 %9, %9, %22;\n\t@q addc.cc.u32 %10, %10, %23;\n\t@q addc.u32 %11, %11, %24;\n\t}"
                : "+r"(d.l[0]), "+r"(d.l[1]), "+r"(d.l[2]), "+r"(d.l[3]), "+r"(d.l[4]), "+r"(d.l[5]), "+r"(d.l[6]), "+r"(d.l[7]), "+r"(d.l[8]),
                  "+r"(d.l[9]), "+r"(d.l[10]), "+r"(d.l[11])
                : "r"(mask), "n"(kp<K>(0)), "n"(kp<K>(1)), "n"(kp<K>(2)), "n"(kp<K>(3)), "n"(kp<K>(4)), "n"(kp<K>(5)), "n"(kp<K>(6)), "n"(kp<K>(7)),
                  "n"(kp<K>(8)), "n"(kp<K>(9)), "n"(kp<K>(10)), "n"(kp<K>(11)));
            return;
        }
#endif
        d.l[0] = cc::add_cc(d.l[0], kp<K>(0) & mask);
#pragma unroll
        for (int i = 1; i < N - 1; i++) d.l[i] = cc::addc_cc(d.l[i], kp<K>(i) & mask);
        d.l[N - 1] = cc::addc(d.l[N - 1], kp<K>(N - 1) & mask);
    }
    PB_HD friend Field operator-(const Field &a, const Field &b) {
        Field d;
        d.l[0] = cc::sub_cc(a.l[0], b.l[0]);
#pragma unroll
        for (int i = 1; i < N; i++) d.l[i] = cc::subc_cc(a.l[i], b.l[i]);
        uint32_t mask = cc::subc(0, 0);  // all-ones when a < b
        cond_add_kp<1>(d, mask);
        return d;
    }
    PB_HD Field neg() const { return is_zero() ? *this : (zero() - *this); }
    // −x for x ≠ 0 (e.g. the y coordinate of a point of the prime-order subgroup): p − x, one subtraction chain
    PB_HD Field neg_nonzero() const {
        Field r;
        r.l[0] = cc::sub_cc(P::mod(0), l[0]);
#pragma unroll
        for (int i = 1; i < N - 1; i++) r.l[i] = cc::subc_cc(P::mod(i), l[i]);
        r.l[N - 1] = cc::subc(P::mod(N - 1), l[N - 1]);
        return r;
    }
    PB_HD Field dbl() const { return *this + *this; }

    // ---- multiplication: u64 column accumulators -------------------------------------------------
    // The running value is held as E + O·2^32 with E, O arrays of H = N/2 u64 columns: E[k] covers
    // limb positions (2k, 2k+1), O[k] positions (2k+1, 2k+2).  a[even]·b_i lands column-aligned in E,
    // a[odd]·b_i column-aligned in O, so every row is one add.cc.u64/addc.cc.u64 chain over
    // mul.wide.u32 products (→ IMAD.WIDE.U32.X).
    static constexpr int H = N / 2;

    // One Montgomery elimination step: adds m·p with m = −E[0]·p⁻¹ mod 2^32 so position 0 becomes 0.
    // p's limbs are compile-time immediates.  The E chain's carry-out (position N) is the high half
    // of O[H−1].  O's own carry-out is provably 0 (capacity argument in DESIGN.md).
    PB_HD static void redc_step(uint64_t *E, uint64_t *O) {
        if (P::LOW_LIMBS_1_FFFFFFFF) {
            // Fr: p ≡ 2^64 − 2^32 + 1 (mod 2^64), −p⁻¹ ≡ −1 (mod 2^32) ⇒ m = −e0 and the two low partial
            // products need no multiplier: m·p[0] = m (e0 + m = 2^32·nz), m·p[1] = (m−nz)·2^32 + e0,
            // with nz = (e0 ≠ 0).
            uint32_t e0 = cc::lo32(E[0]);
            uint32_t m = 0u - e0;
            (void)cc::add_cc(e0, m);
            uint32_t nz = cc::addc(0, 0);
            O[0] = cc::add_cc64(O[0], cc::pack64(e0, m - nz));
#pragma unroll
            for (int k = 1; k < H; k++) O[k] = cc::addc_cc64(O[k], cc::mul_wide(P::mod(2 * k + 1), m));
            E[0] = cc::add_cc64(cc::pack64(0, cc::hi32(E[0])), cc::pack64(0, nz));
#pragma unroll
            for (int k = 1; k < H; k++) E[k] = cc::addc_cc64(E[k], cc::mul_wide(P::mod(2 * k), m));
        } else {
            uint32_t m = cc::lo32(E[0]) * P::INV32;
            O[0] = cc::add_cc64(O[0], cc::mul_wide(P::mod(1), m));
#pragma unroll
            for (int k = 1; k < H; k++) O[k] = cc::addc_cc64(O[k], cc::mul_wide(P::mod(2 * k + 1), m));
            E[0] = cc::add_cc64(E[0], cc::mul_wide(P::mod(0), m));
#pragma unroll
            for (int k = 1; k < H; k++) E[k] = cc::addc_cc64(E[k], cc::mul_wide(P::mod(2 * k), m));
        }
        O[H - 1] = cc::pack64(cc::lo32(O[H - 1]), cc::addc(cc::hi32(O[H - 1]), 0));
    }
    // Start of round i ≥ 1.  On entry position 0 of S is zero and the value (already divided by 2^32) is
    // (S >> 32) + D·(one position down).  S's position 1 is folded into D's position 0, S is rebuilt
    // one column lower as the new odd accumulator, D becomes the new even accumulator; a·b_i is added.
    PB_HD static void shift_add_row(uint64_t *S, uint64_t *D, const uint32_t *a, uint32_t bi) {
        uint32_t d0 = cc::add_cc(cc::lo32(D[0]), cc::hi32(S[0]));  // carry → start of the odd chain
#pragma unroll
        for (int k = 0; k < H - 1; k++) S[k] = cc::addc_cc64(S[k + 1], cc::mul_wide(a[2 * k + 1], bi));
        S[H - 1] = cc::addc64(cc::mul_wide(a[N - 1], bi), 0);
        D[0] = cc::add_cc64(cc::pack64(d0, cc::hi32(D[0])), cc::mul_wide(a[0], bi));
#pragma unroll
        for (int k = 1; k < H; k++) D[k] = cc::addc_cc64(D[k], cc::mul_wide(a[2 * k], bi));
        S[H - 1] = cc::pack64(cc::lo32(S[H - 1]), cc::addc(cc::hi32(S[H - 1]), 0));
    }
    PB_HD static void round(uint64_t *S, uint64_t *D, const uint32_t *a, uint32_t bi) {
        shift_add_row(S, D, a, bi);
        redc_step(D, S);
    }
    // After the last round position 0 of B is clear: value = (B >> 32) + A  (< 2p), merged limb-wise.
    PB_HD static Field merge(const uint64_t *A, const uint64_t *B) {
        Field r;
        r.l[0] = cc::add_cc(cc::lo32(A[0]), cc::hi32(B[0]));
#pragma unroll
        for (int k = 1; k < N - 1; k++) {
            uint32_t x = (k & 1) ? cc::hi32(A[k >> 1]) : cc::lo32(A[k >> 1]);
            uint32_t y = (k & 1) ? cc::lo32(B[(k + 1) >> 1]) : cc::hi32(B[k >> 1]);
            r.l[k] = cc::addc_cc(x, y);
        }
        r.l[N - 1] = cc::addc(cc::hi32(A[H - 1]), 0);
        return r;
    }
    PB_HD static Field mul_unreduced(const Field &a, const Field &b) {   // a·b/R + (< p), not brought below p: see mul_lazy
        uint64_t A[H], B[H];
#pragma unroll
        for (int k = 0; k < H; k++) {
            A[k] = cc::mul_wide(a.l[2 * k], b.l[0]);
            B[k] = cc::mul_wide(a.l[2 * k + 1], b.l[0]);
        }
        redc_step(A, B);
#pragma unroll
        for (int i = 1; i < N - 1; i += 2) {
            round(A, B, a.l, b.l[i]);
            round(B, A, a.l, b.l[i + 1]);
        }
        round(A, B, a.l, b.l[N - 1]);
        return merge(A, B);
    }
    PB_HD static Field mul_inline(const Field &a, const Field &b) { return reduce_once(mul_unreduced(a, b)); }

    // ---- lazy representation: values in [0, 2p) (fields with a spare bit: 2p < 2^(32N)) --------------------------------
    // The Montgomery product of a CANONICAL a (< p) and any b < 2p is a·b/R + (< p) < (2p/R + 1)·p < 2p, so it needs no
    // final subtraction when the next operation accepts [0, 2p); the running value of the word-serial loop is bounded by
    // a + p < 2p as in the canonical case (b is the operand scanned limb by limb, its size does not enter).  Additions and
    // subtractions are taken mod 2p.  canonical() brings a lazy value back to [0, p).
    PB_HD static constexpr uint32_t mod2(int i) { return (P::mod(i) << 1) | (i ? (P::mod(i - 1) >> 31) : 0u); }
    PB_HD static Field mul_lazy(const Field &a_canonical, const Field &b) { return mul_unreduced(a_canonical, b); }
    PB_HD static Field add_lazy(const Field &a, const Field &b) {   // a, b < 2p → (a + b) mod 2p
        Field s;
        s.l[0] = cc::add_cc(a.l[0], b.l[0]);
#pragma unroll
        for (int i = 1; i < N - 1; i++) s.l[i] = cc::addc_cc(a.l[i], b.l[i]);
        s.l[N - 1] = cc::addc_cc(a.l[N - 1], b.l[N - 1]);
        const uint32_t carry = cc::addc(0, 0);           // 4p may not fit 32N bits (Fr has one spare bit): keep the carry-out
        Field d;
        d.l[0] = cc::sub_cc(s.l[0], mod2(0));
#pragma unroll
        for (int i = 1; i < N; i++) d.l[i] = cc::subc_cc(s.l[i], mod2(i));
        const uint32_t borrow = cc::subc(0, 0);          // all-ones when the low 32N bits are below 2p
        const bool keep = borrow != 0 && carry == 0;      // the sum is already below 2p
        Field r;
#pragma unroll
        for (int i = 0; i < N; i++) r.l[i] = keep ? s.l[i] : d.l[i];
        return r;
    }
    PB_HD static Field sub_lazy(const Field &a, const Field &b) {   // a, b < 2p → (a − b) mod 2p
        Field d;
        d.l[0] = cc::sub_cc(a.l[0], b.l[0]);
#pragma unroll
        for (int i = 1; i < N; i++) d.l[i] = cc::subc_cc(a.l[i], b.l[i]);
        const uint32_t mask = cc::subc(0, 0);
        cond_add_kp<2>(d, mask);
        return d;
    }
    PB_HD Field canonical() const { return reduce_once(*this); }   // [0, 2p) → [0, p)
    // operator*: fully inlined in the throughput kernels; translation units that define
    // PB_FIELD_NOINLINE_MUL (the latency-bound tail kernels) call one shared copy instead, which shrinks their
    // code ~10× (cold instruction fetch dominated those single-warp kernels) and their register count.
    PB_HD friend Field operator*(const Field &a, const Field &b) {
#if defined(PB_FIELD_NOINLINE_MUL) && defined(__CUDA_ARCH__)
        return field_mul_noinline(a, b);
#else
        return mul_inline(a, b);
#endif
    }
    // ---- squaring (fields with ≥ 3 spare top bits: Fp) ------------------------------------------------
    // a² = Σ_i a_i·(a_i + 2·Σ_{j>i} a_j 2^(32(j−i)))·2^(64 i): row i of the word-serial loop only needs the products
    // with j ≥ i, taken against the pre-doubled operand (78 instead of 144 products; the 144 of the interleaved
    // reduction stay).  Doubling raises the bound on the running value from 2p to 3p and on the window from
    // 2^33·p to 3·2^32·p, which still fits 32(N+1) bits because p < 2^(32N−3); two conditional subtractions finish.
    // x_j for row i: 0 (j < i) | a_i (j = i) | a_(i+1) << 1 (j = i+1) | d_j = (a_j << 1 | a_(j−1) >> 31) (j > i+1).
    PB_HD static uint64_t sqr_term(const uint32_t *a, const uint32_t *d, int i, int j) {
        if (j < i) return 0;
        if (j == i) return cc::mul_wide(a[i], a[i]);
        if (j == i + 1) return cc::mul_wide(a[j] << 1, a[i]);
        return cc::mul_wide(d[j], a[i]);
    }
    PB_HD static void round_sqr(uint64_t *S, uint64_t *D, const uint32_t *a, const uint32_t *d, int i) {
        uint32_t d0 = cc::add_cc(cc::lo32(D[0]), cc::hi32(S[0]));
#pragma unroll
        for (int k = 0; k < H - 1; k++) S[k] = cc::addc_cc64(S[k + 1], sqr_term(a, d, i, 2 * k + 1));
        S[H - 1] = cc::addc64(sqr_term(a, d, i, N - 1), 0);
        D[0] = cc::add_cc64(cc::pack64(d0, cc::hi32(D[0])), sqr_term(a, d, i, 0));
#pragma unroll
        for (int k = 1; k < H; k++) D[k] = cc::addc_cc64(D[k], sqr_term(a, d, i, 2 * k));
        S[H - 1] = cc::pack64(cc::lo32(S[H - 1]), cc::addc(cc::hi32(S[H - 1]), 0));
        redc_step(D, S);
    }
    PB_HD static Field sqr_unreduced(const Field &x) {   // x²/R + (< p), not brought below p
        const uint32_t *a = x.l;
        uint32_t d[N];
        d[0] = a[0] << 1;
#pragma unroll
        for (int j = 1; j < N; j++) d[j] = (a[j] << 1) | (a[j - 1] >> 31);  // a[N−1] >> 31 = 0: spare bits
        uint64_t A[H], B[H];
#pragma unroll
        for (int k = 0; k < H; k++) {
            A[k] = sqr_term(a, d, 0, 2 * k);
            B[k] = sqr_term(a, d, 0, 2 * k + 1);
        }
        redc_step(A, B);
#pragma unroll
        for (int i = 1; i < N - 1; i += 2) {
            round_sqr(A, B, a, d, i);
            round_sqr(B, A, a, d, i + 1);
        }
        round_sqr(A, B, a, d, N - 1);
        return merge(A, B);
    }
    PB_HD static Field sqr_inline(const Field &x) { return reduce_once(reduce_once(sqr_unreduced(x))); }  // value < 3p
    // Lazy products for fields with ≥ 3 spare bits (Fp): BOTH operands may be lazy — a·b/R + p < (4p/R + 1)·p < 2p because
    // p/R < 1/8 — and the running value a + p < 3p (2a + p < 5p in the squaring, whose operand is pre-doubled) fits 32N bits.
    PB_HD static Field mul_lazy2(const Field &a, const Field &b) { return mul_unreduced(a, b); }
    PB_HD static Field sqr_lazy(const Field &a) { return sqr_unreduced(a); }

    // ---- sum of two products, one reduction (fields with ≥ 3 spare bits: Fp) ---------------------------------------
    // (a·b + c·d)·R⁻¹ mod p in [0, 2p) for a, b, c, d ≤ 2p: row i adds a·b_i AND c·d_i to the E / O accumulators, then runs
    // ONE elimination step, so the two products share the N·(H + H + 1) wide multiplies of the reduction.  A difference
    // a·b − c·d is the sum with c replaced by neg_2p(c) (which may be exactly 2p: hence ≤ 2p, not < 2p, below).
    // Capacity, row by row.  Let U_i be the running value after row i (U_−1 = 0).  Row i forms
    //   V_i = U_(i−1) + a·b_i + c·d_i + m_i·p ≤ U_(i−1) + (2^32 − 1)·(a + c + p),   U_i = V_i / 2^32,
    // so by induction U_i < a + c + p and V_i < 2^32·(a + c + p) ≤ 2^32·5p < 2^32·2^384 = 2^(32(N+1)) since p < 2^381:
    // every state of the row fits positions 0 … N of E + O·2^32.  All terms are non-negative and every carry of a chain
    // lands at a position ≤ N, so a carry out of position N (the chains' dropped carries, the 32-bit `addc` into
    // O[H−1]'s high half) would make the state ≥ 2^(32(N+1)) — none occurs.  Per column: the top odd column O[H−1]
    // receives a[N−1]·b_i + c[N−1]·d_i + 2 carries < 2·2^30·2^32 + 2 (a, c < 2^382 ⇒ top limbs < 2^30), and its high half
    // then takes the carry out of each of the two even chains (< 2^31 + 2 < 2^32); no u64 column wraps.
    // Result: U_(N−1) = (a·b + c·d + M·p)/R with M < R, so U < (8p² + R·p)/R = 8p²/R + p < 2p because 8p < R.
    // (Fr, one spare bit, has no room for two products: the static_assert keeps it out.)
    PB_HD static void add_row(uint64_t *S, uint64_t *D, const uint32_t *c, uint32_t di) {   // S odd, D even: += c·d_i
        S[0] = cc::add_cc64(S[0], cc::mul_wide(c[1], di));
#pragma unroll
        for (int k = 1; k < H - 1; k++) S[k] = cc::addc_cc64(S[k], cc::mul_wide(c[2 * k + 1], di));
        S[H - 1] = cc::addc64(S[H - 1], cc::mul_wide(c[N - 1], di));
        D[0] = cc::add_cc64(D[0], cc::mul_wide(c[0], di));
#pragma unroll
        for (int k = 1; k < H; k++) D[k] = cc::addc_cc64(D[k], cc::mul_wide(c[2 * k], di));
        S[H - 1] = cc::pack64(cc::lo32(S[H - 1]), cc::addc(cc::hi32(S[H - 1]), 0));
    }
    PB_HD static Field mul2_sum_unreduced(const Field &a, const Field &b, const Field &c, const Field &d) {
        static_assert(P::SPARE_BITS >= 3, "two products per row need 3 spare bits (capacity argument above)");
        uint64_t A[H], B[H];
#pragma unroll
        for (int k = 0; k < H; k++) {
            A[k] = cc::mul_wide(a.l[2 * k], b.l[0]);
            B[k] = cc::mul_wide(a.l[2 * k + 1], b.l[0]);
        }
        add_row(B, A, c.l, d.l[0]);
        redc_step(A, B);
#pragma unroll
        for (int i = 1; i < N - 1; i += 2) {
            shift_add_row(A, B, a.l, b.l[i]);
            add_row(A, B, c.l, d.l[i]);
            redc_step(B, A);
            shift_add_row(B, A, a.l, b.l[i + 1]);
            add_row(B, A, c.l, d.l[i + 1]);
            redc_step(A, B);
        }
        shift_add_row(A, B, a.l, b.l[N - 1]);
        add_row(A, B, c.l, d.l[N - 1]);
        redc_step(B, A);
        return merge(A, B);
    }
    // 2p − x for x ≤ 2p, in [0, 2p]: the negated operand of a difference of products (not a lazy value: it may be 2p)
    PB_HD Field neg_2p() const {
        static_assert(P::SPARE_BITS >= 2, "2p must fit 32N bits");
        Field r;
        r.l[0] = cc::sub_cc(mod2(0), l[0]);
#pragma unroll
        for (int i = 1; i < N - 1; i++) r.l[i] = cc::subc_cc(mod2(i), l[i]);
        r.l[N - 1] = cc::subc(mod2(N - 1), l[N - 1]);
        return r;
    }
    PB_HD static Field mul2_sum_lazy(const Field &a, const Field &b, const Field &c, const Field &d) {   // in [0, 2p)
        return mul2_sum_unreduced(a, b, c, d);
    }
    PB_HD static Field mul2_sum(const Field &a, const Field &b, const Field &c, const Field &d) {        // in [0, p)
#if defined(PB_FIELD_NOINLINE_MUL) && defined(__CUDA_ARCH__)
        return field_mul2_sum_noinline(a, b, c, d);
#else
        return reduce_once(mul2_sum_unreduced(a, b, c, d));
#endif
    }
    // ≡ 0 (mod p) for a lazy value: 0 or p
    PB_HD bool is_zero_lazy() const {
        uint32_t o = 0, q = 0;
#pragma unroll
        for (int i = 0; i < N; i++) {
            o |= l[i];
            q |= l[i] ^ P::mod(i);
        }
        return o == 0 || q == 0;
    }
    PB_HD Field sqr() const {
        if (P::SPARE_BITS >= 3) {
#if defined(PB_FIELD_NOINLINE_MUL) && defined(__CUDA_ARCH__)
            return field_sqr_noinline(*this);
#else
            return sqr_inline(*this);
#endif
        }
        return *this * *this;
    }

    // Montgomery form → canonical integer (multiply by 1): N elimination rounds, no products with b.
    PB_HD Field from_mont() const {
        Field one_raw = zero();
        one_raw.l[0] = 1;
        return *this * one_raw;
    }
    PB_HD Field to_mont() const { return *this * r2(); }

    // this^e, e a plain little-endian u32 exponent of `words` words.
    PB_HD Field pow(const uint32_t *e, int words) const {
        Field r = one();
        for (int i = words * 32 - 1; i >= 0; i--) {
            r = r.sqr();
            if ((e[i >> 5] >> (i & 31)) & 1) r = r * *this;
        }
        return r;
    }
    // this^e for a 32-bit exponent, looping over the significant bits only (index-dependent powers z^j in the
    // vector kernels: ≈ log2(j) squarings instead of 64).
    PB_HD Field pow_u32(uint32_t e) const {
        if (e == 0) return one();
        int top = 31;
        while (!((e >> top) & 1)) top--;
        Field r = *this;
        for (int i = top - 1; i >= 0; i--) {
            r = r.sqr();
            if ((e >> i) & 1) r = r * *this;
        }
        return r;
    }
    PB_HD Field pow_u64(uint64_t e) const {
        uint32_t w[2] = {(uint32_t)e, (uint32_t)(e >> 32)};
        return pow(w, 2);
    }
    // Fermat inverse; 0 ↦ 0.
    PB_HD Field inv() const {
        uint32_t e[N];
        e[0] = cc::sub_cc(P::mod(0), 2);
#pragma unroll
        for (int i = 1; i < N; i++) e[i] = cc::subc_cc(P::mod(i), 0);
        return pow(e, N);
    }
};

#if defined(PB_FIELD_NOINLINE_MUL) && defined(__CUDACC__)
template <class P>
__device__ __noinline__ Field<P> field_mul_noinline(Field<P> a, Field<P> b) {
    return Field<P>::mul_inline(a, b);
}
template <class P>
__device__ __noinline__ Field<P> field_sqr_noinline(Field<P> a) {
    return Field<P>::sqr_inline(a);
}
template <class P>
__device__ __noinline__ Field<P> field_mul2_sum_noinline(Field<P> a, Field<P> b, Field<P> c, Field<P> d) {
    return Field<P>::reduce_once(Field<P>::mul2_sum_unreduced(a, b, c, d));
}
#endif

// ---------------------------------------------------------------------------------------------------
// BLS12-381 scalar field Fr (SURVEY.md Appendix A.2).  r ≡ 1 (mod 2^32) ⇒ −r⁻¹ mod 2^32 = 0xffffffff.
struct FrParams {
    static constexpr int N = 8;
    static constexpr uint32_t INV32 = 0xffffffffu;
    static constexpr bool LOW_LIMBS_1_FFFFFFFF = true;
    static constexpr int SPARE_BITS = 1;  // 255-bit modulus in 256
    PB_HD static constexpr uint32_t mod(int i) {
        constexpr uint32_t v[8] = {0x00000001u, 0xffffffffu, 0xfffe5bfeu, 0x53bda402u,
                                   0x09a1d805u, 0x3339d808u, 0x299d7d48u, 0x73eda753u};
        return v[i];
    }
    PB_HD static constexpr uint32_t r1(int i) {  // 2^256 mod r
        constexpr uint32_t v[8] = {0xfffffffeu, 0x00000001u, 0x00034802u, 0x5884b7fau,
                                   0xecbc4ff5u, 0x998c4fefu, 0xacc5056fu, 0x1824b159u};
        return v[i];
    }
    PB_HD static constexpr uint32_t r2(int i) {  // 2^512 mod r
        constexpr uint32_t v[8] = {0xf3f29c6du, 0xc999e990u, 0x87925c23u, 0x2b6cedcbu,
                                   0x7254398fu, 0x05d31496u, 0x9f59ff11u, 0x0748d9d9u};
        return v[i];
    }
};
// BLS12-381 base field Fp (SURVEY.md Appendix A.3).
struct FpParams {
    static constexpr int N = 12;
    static constexpr uint32_t INV32 = 0xfffcfffdu;
    static constexpr bool LOW_LIMBS_1_FFFFFFFF = false;
    static constexpr int SPARE_BITS = 3;  // 381-bit modulus in 384
    PB_HD static constexpr uint32_t mod(int i) {
        constexpr uint32_t v[12] = {0xffffaaabu, 0xb9feffffu, 0xb153ffffu, 0x1eabfffeu, 0xf6b0f624u, 0x6730d2a0u,
                                    0xf38512bfu, 0x64774b84u, 0x434bacd7u, 0x4b1ba7b6u, 0x397fe69au, 0x1a0111eau};
        return v[i];
    }
    PB_HD static constexpr uint32_t r1(int i) {  // 2^384 mod p
        constexpr uint32_t v[12] = {0x0002fffdu, 0x76090000u, 0xc40c0002u, 0xebf4000bu, 0x53c758bau, 0x5f489857u,
                                    0x70525745u, 0x77ce5853u, 0xa256ec6du, 0x5c071a97u, 0xfa80e493u, 0x15f65ec3u};
        return v[i];
    }
    PB_HD static constexpr uint32_t r2(int i) {  // 2^768 mod p
        constexpr uint32_t v[12] = {0x1c341746u, 0xf4df1f34u, 0x09d104f1u, 0x0a76e6a6u, 0x4c95b6d5u, 0x8de5476cu,
                                    0x939d83c0u, 0x67eb88a9u, 0xb519952du, 0x9a793e85u, 0x92cae3aau, 0x11988fe5u};
        return v[i];
    }
};
typedef Field<FrParams> Fr;
typedef Field<FpParams> Fp;
