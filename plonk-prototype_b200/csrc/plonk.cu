// plonk.cu — the PLONK prover rounds around the hot path (SURVEY.md §8f-2/3): preprocessing and the five rounds
// of dusk-plonk 0.8.2's `Prover::prove_with_preprocessed`, with every polynomial resident in HBM between rounds.
//
// Replaces (crate pinned at /root/reference/Cargo.toml:19; the reference builds its circuits against it at
// /root/reference/src/zk/gadgets.rs:28-225 and circuits.rs:51-72; SURVEY.md §3.2-3.3, App. B.3):
//   StandardComposer::preprocess_prover + VerifierKey::seed_transcript          → pb200_preprocess
//   Prover::prove_with_preprocessed (rounds 1-5), Proof::to_bytes               → pb200_prove
//   Permutation::compute_permutation_poly (grand product, batch inversion)      → perm_* kernels + Fr product scans
//   quotient_poly::compute (pointwise loop over the 4n coset)                   → quotient_kernel
//   linearisation_poly::compute, Polynomial::evaluate                           → lincomb_kernel, poly_eval_* kernels
//   CommitKey::compute_aggregate_witness                                        → lincomb_kernel + pb200_kzg_witness_dev
// The NTTs and MSMs are the library's own hot path (ntt.cu, msm.cu).  The host keeps only the Fiat–Shamir
// transcript (merlin.h) and a few dozen scalar operations per round (host_field.h).
//
// Widgets: arithmetic (q_arith·(q_m·a·b + q_l·a + q_r·b + q_o·c + q_4·d + q_c) + PI), range (q_range quad check), and —
// csrc/widgets.h — logic (XOR / AND quads), fixed-base scalar multiplication and variable-base point addition on JubJub,
// i.e. every selector column StandardComposer has.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "fr_vec.cuh"
#include "host_field.h"
#include "merlin.h"
#include "widgets.h"

using hostf::HFr;

namespace {

constexpr int kSel = 11;  // q_m q_l q_r q_o q_c q_4 q_arith q_range q_logic q_fixed_group_add q_variable_group_add
enum { Q_M, Q_L, Q_R, Q_O, Q_C, Q_4, Q_ARITH, Q_RANGE, Q_LOGIC, Q_FIXED, Q_VAR };

inline Fr to_dev(const HFr &h) {  // same memory image: 4 × u64 LE = 8 × u32 LE
    Fr r;
    memcpy(r.l, h.l, 32);
    return r;
}

// ------------------------------------------------------------------------------------------------ small kernels
// out[i] = c·g^i
__global__ void powers_kernel(Fr *out, uint32_t n, Fr c, Fr g) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    st_fr(out + i, c * g.pow_u32(i));
}
// dst[j] = j < n_src ? src[j] : 0 for `batch` vectors (dst stride n_dst, src stride n_src)
__global__ void pad_copy_kernel(Fr *dst, const Fr *src, uint32_t n_src, uint32_t n_dst) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_dst) return;
    const size_t b = blockIdx.y;
    st_fr(dst + b * n_dst + j, j < n_src ? ld_fr(src + b * n_src + j) : Fr::zero());
}
__global__ void fill_kernel(Fr *dst, uint32_t n, Fr v) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) st_fr(dst + j, v);
}
// Round 1: wire column evaluations w[col][i] = value of the variable wired to gate i (zero on the padding rows).
__global__ void gather_wires_kernel(Fr *w, const uint32_t *wires, const Fr *values, uint32_t n_gates, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t col = blockIdx.y;
    Fr v = Fr::zero();
    if (i < n_gates) v = ld_fr(values + wires[(size_t)col * n_gates + i]);
    st_fr(w + (size_t)col * n + i, v);
}
// Preprocessing: σ_col(ω^i) = K_c'·ω^i' where (c', i') is the position the permutation sends (col, i) to.
struct KFactors {
    Fr k[4];
};
__global__ void sigma_evals_kernel(Fr *sig, const uint32_t *map, const Fr *roots, uint32_t n, uint32_t log_n, KFactors ks) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t col = blockIdx.y;
    const uint32_t m = map[(size_t)col * n + i];
    st_fr(sig + (size_t)col * n + i, ks.k[m >> log_n] * ld_fr(roots + (m & (n - 1))));
}
// dense public-input vector from the sparse store
__global__ void scatter_pi_kernel(Fr *pi, const uint32_t *pos, const Fr *vals, uint32_t n_pi) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n_pi) st_fr(pi + pos[j], ld_fr(vals + j));
}

// ------------------------------------------------------------------------------------------------ Fr product scans
// Inclusive product scan over n elements, forward (REV = false: out[i] = Π_{j ≤ i} a[j]) or backward
// (REV = true: out[i] = Π_{j ≥ i} a[j]); three launches, tiles of 1024 elements (256 threads × 4), in place.
constexpr uint32_t kTile = 1024;
template <bool REV>
__device__ __forceinline__ uint32_t phys(uint32_t k, uint32_t n) {
    return REV ? n - 1 - k : k;
}
// inclusive scan across the 256 threads of a CTA (thread order = logical order)
__device__ __forceinline__ Fr block_prod_scan(Fr v, Fr *sm, Fr *total) {
    const uint32_t t = threadIdx.x;
    st_fr(sm + t, v);
    __syncthreads();
    for (uint32_t o = 1; o < 256; o <<= 1) {
        Fr left = Fr::one();
        const bool has = t >= o;
        if (has) left = ld_fr(sm + t - o);
        __syncthreads();
        if (has) v = left * v;
        st_fr(sm + t, v);
        __syncthreads();
    }
    if (total) *total = ld_fr(sm + 255);
    return v;
}
template <bool REV>
__global__ void __launch_bounds__(256) scan_tile_products_kernel(const Fr *a, uint32_t n, Fr *tile_prod) {
    __shared__ uint4 smraw[512];
    Fr *sm = reinterpret_cast<Fr *>(smraw);
    const uint32_t base = blockIdx.x * kTile + threadIdx.x * 4;
    Fr p = Fr::one();
    for (uint32_t k = 0; k < 4; k++)
        if (base + k < n) p = p * ld_fr(a + phys<REV>(base + k, n));
    Fr total;
    block_prod_scan(p, sm, &total);
    if (threadIdx.x == 0) st_fr(tile_prod + blockIdx.x, total);
}
// tile_prod[t] ← Π_{u < t} tile_prod[u] (exclusive), one CTA; the product of everything → *grand
__global__ void __launch_bounds__(256) scan_top_kernel(Fr *tile_prod, uint32_t n_tiles, Fr *grand) {
    __shared__ uint4 smraw[512];
    Fr *sm = reinterpret_cast<Fr *>(smraw);
    const uint32_t per = (n_tiles + 255) / 256;
    const uint32_t lo = min(threadIdx.x * per, n_tiles), hi = min(lo + per, n_tiles);
    Fr p = Fr::one();
    for (uint32_t i = lo; i < hi; i++) p = p * ld_fr(tile_prod + i);
    Fr total;
    block_prod_scan(p, sm, &total);
    __syncthreads();
    Fr run = threadIdx.x ? ld_fr(sm + threadIdx.x - 1) : Fr::one();
    for (uint32_t i = lo; i < hi; i++) {
        Fr v = ld_fr(tile_prod + i);
        st_fr(tile_prod + i, run);
        run = run * v;
    }
    if (threadIdx.x == 0) st_fr(grand, total);
}
template <bool REV>
__global__ void __launch_bounds__(256) scan_finish_kernel(Fr *a, uint32_t n, const Fr *tile_prod) {
    __shared__ uint4 smraw[512];
    Fr *sm = reinterpret_cast<Fr *>(smraw);
    const uint32_t base = blockIdx.x * kTile + threadIdx.x * 4;
    Fr v[4], p = Fr::one();
    for (uint32_t k = 0; k < 4; k++) {
        v[k] = (base + k < n) ? ld_fr(a + phys<REV>(base + k, n)) : Fr::one();
        p = p * v[k];
    }
    block_prod_scan(p, sm, nullptr);
    __syncthreads();
    Fr run = ld_fr(tile_prod + blockIdx.x);
    if (threadIdx.x) run = run * ld_fr(sm + threadIdx.x - 1);
    for (uint32_t k = 0; k < 4; k++) {
        run = run * v[k];
        if (base + k < n) st_fr(a + phys<REV>(base + k, n), run);
    }
}

// ------------------------------------------------------------------------------------------------ round 2
// num[i] = Π_col (w_col[i] + β·K_col·ω^i + γ),  den[i] = Π_col (w_col[i] + β·σ_col(ω^i) + γ)
__global__ void __launch_bounds__(256) perm_numden_kernel(const Fr *w, const Fr *sig, const Fr *roots, uint32_t n, Fr beta, Fr gamma,
                                                          KFactors ks, Fr *num, Fr *den) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Fr br = beta * ld_fr(roots + i);
    Fr nu = Fr::one(), de = Fr::one();
#pragma unroll
    for (int col = 0; col < 4; col++) {
        const Fr wv = ld_fr(w + (size_t)col * n + i) + gamma;
        const Fr id = col == 0 ? br : ks.k[col] * br;
        const Fr t = wv + id;
        nu = col == 0 ? t : nu * t;
        const Fr s = wv + beta * ld_fr(sig + (size_t)col * n + i);
        de = col == 0 ? s : de * s;
    }
    st_fr(num + i, nu);
    st_fr(den + i, de);
}
__global__ void fr_inv_kernel(const Fr *in, Fr *out) { st_fr(out, ld_fr(in).inv()); }
// z[0] = 1, z[k] = PN[k−1]·SD[k]·(Π den)⁻¹   (PN inclusive prefix products of num, SD inclusive suffix products of den)
__global__ void __launch_bounds__(256) perm_finish_kernel(const Fr *pn, const Fr *sd, const Fr *inv_total, uint32_t n, Fr *z) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    Fr v = Fr::one();
    if (k) v = ld_fr(pn + k - 1) * ld_fr(sd + k) * ld_fr(inv_total);
    st_fr(z + k, v);
}

// ------------------------------------------------------------------------------------------------ round 3
struct QuotArgs {
    const Fr *q[kSel];   // selector evaluations on the 4n coset (nullptr = identically zero)
    const Fr *sig;       // 4 × N4
    const Fr *lin;       // X on the coset: 7·ω_4n^i
    const Fr *w;         // a, b, c, d: 4 × N4
    const Fr *z, *pi, *l1;  // l1: L₁ on the coset (unscaled)
    Fr *out;
    uint32_t N4;
    // Sharded round 3: w, z, pi and out are this rank's row-layout shards (`count` points, wire stride `count`), the
    // shifted evaluations z(ωX), d(ωX) come from their own transforms (zw, dw) instead of index + 4, and local point
    // e = r·m + k' is global point (row0 + r) + n1·k' of the key's natural-order vectors.  dist = 0: count = N4.
    const Fr *zw, *dw;
    uint32_t dist, count, log_m, log_n1, row0;
    Fr alpha, alpha2, beta, gamma, range_sep;
    Fr logic_sep, fixed_sep, var_sep, edwards_d;   // logic / fixed-base / variable-base widgets (EXTRA instantiation only)
    Fr vh_inv[4];        // 1 / ((7ω_4n^i)^n − 1) has period 4 in i
    KFactors ks;
};
__device__ __forceinline__ Fr delta4(const Fr &f, const Fr &one) {  // f(f−1)(f−2)(f−3)
    const Fr f1 = f - one, f2 = f1 - one, f3 = f2 - one;
    return (f * f1) * (f2 * f3);
}
__device__ __forceinline__ Fr quad(const Fr &x) { return x.dbl().dbl(); }
// EXTRA: the circuit has logic / fixed-base / variable-base rows (single-GPU layout only: they read a, b at index + 4)
template <bool RANGE, bool EXTRA>
__global__ void __launch_bounds__(128) quotient_kernel(const QuotArgs A) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= A.count) return;
    const uint32_t N4 = A.N4, ws = A.count;
    const uint32_t i = A.dist ? (A.row0 + (e >> A.log_m)) + ((e & ((1u << A.log_m) - 1)) << A.log_n1) : e;
    const uint32_t enext = (e + 4) & (N4 - 1);  // dist = 0 only
    const Fr a = ld_fr(A.w + e), b = ld_fr(A.w + (size_t)ws + e), c = ld_fr(A.w + 2 * (size_t)ws + e),
             d = ld_fr(A.w + 3 * (size_t)ws + e);
    // arithmetic widget
    Fr g = Fr::zero();
    if (A.q[Q_M]) g = (a * b) * ld_fr(A.q[Q_M] + i);
    if (A.q[Q_L]) g = g + a * ld_fr(A.q[Q_L] + i);
    if (A.q[Q_R]) g = g + b * ld_fr(A.q[Q_R] + i);
    if (A.q[Q_O]) g = g + c * ld_fr(A.q[Q_O] + i);
    if (A.q[Q_4]) g = g + d * ld_fr(A.q[Q_4] + i);
    if (A.q[Q_C]) g = g + ld_fr(A.q[Q_C] + i);
    if (A.q[Q_ARITH]) g = g * ld_fr(A.q[Q_ARITH] + i);
    else g = Fr::zero();
    if (RANGE) {
        const Fr one = Fr::one();
        const Fr dn = A.dist ? ld_fr(A.dw + e) : ld_fr(A.w + 3 * (size_t)ws + enext);
        const Fr kappa = A.range_sep.sqr();
        Fr r = delta4(dn - quad(a), one);
        r = r * kappa + delta4(a - quad(b), one);
        r = r * kappa + delta4(b - quad(c), one);
        r = r * kappa + delta4(c - quad(d), one);
        g = g + (r * A.range_sep) * ld_fr(A.q[Q_RANGE] + i);
    }
    if (EXTRA) {
        const Fr an = ld_fr(A.w + enext), bn = ld_fr(A.w + (size_t)ws + enext), dn = ld_fr(A.w + 3 * (size_t)ws + enext);
        if (A.q[Q_LOGIC]) {
            const Fr ql = ld_fr(A.q[Q_LOGIC] + i);
            if (!ql.is_zero())
                g = g + ql * widgets::logic_term(a, an, b, bn, c, d, dn, A.q[Q_C] ? ld_fr(A.q[Q_C] + i) : Fr::zero(), A.logic_sep);
        }
        if (A.q[Q_FIXED]) {
            const Fr qf = ld_fr(A.q[Q_FIXED] + i);
            if (!qf.is_zero())
                g = g + qf * widgets::fixed_base_term(a, an, b, bn, c, d, dn, A.q[Q_L] ? ld_fr(A.q[Q_L] + i) : Fr::zero(),
                                                      A.q[Q_R] ? ld_fr(A.q[Q_R] + i) : Fr::zero(),
                                                      A.q[Q_C] ? ld_fr(A.q[Q_C] + i) : Fr::zero(), A.fixed_sep, A.edwards_d);
        }
        if (A.q[Q_VAR]) {
            const Fr qv = ld_fr(A.q[Q_VAR] + i);
            if (!qv.is_zero()) g = g + qv * widgets::var_base_term(a, an, b, bn, c, d, dn, A.var_sep, A.edwards_d);
        }
    }
    g = g + ld_fr(A.pi + e);
    // permutation: identity part, copy part, L1 part
    const Fr zi = ld_fr(A.z + e), zn = A.dist ? ld_fr(A.zw + e) : ld_fr(A.z + enext);
    const Fr bx = A.beta * ld_fr(A.lin + i);
    const Fr ag = a + A.gamma, bg = b + A.gamma, cg = c + A.gamma, dg = d + A.gamma;
    Fr id = (ag + bx) * (bg + A.ks.k[1] * bx);
    id = id * ((cg + A.ks.k[2] * bx) * (dg + A.ks.k[3] * bx));
    id = id * zi;
    Fr cp = (ag + A.beta * ld_fr(A.sig + i)) * (bg + A.beta * ld_fr(A.sig + (size_t)N4 + i));
    cp = cp * ((cg + A.beta * ld_fr(A.sig + 2 * (size_t)N4 + i)) * (dg + A.beta * ld_fr(A.sig + 3 * (size_t)N4 + i)));
    cp = cp * zn;
    Fr t = (id - cp) * A.alpha + ((zi - Fr::one()) * ld_fr(A.l1 + i)) * A.alpha2;
    st_fr(A.out + e, (g + t) * A.vh_inv[i & 3]);
}

// Sharded round 3: this rank's column-layout shard A[j1][c] = x[j1·m + col0 + c] (n1 × cl) of the zero-padded, coset-scaled
// polynomial x_j = p_j·gen^j (gen = 7, or 7ω for the evaluations of p(ωX)); four consecutive columns per thread.
__global__ void __launch_bounds__(256) dist_load_kernel(Fr *dst, const Fr *poly, uint32_t n, uint32_t log_m, uint32_t log_cl, uint32_t col0,
                                                        uint32_t local, Fr gen) {
    const uint32_t e0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (e0 >= local) return;
    const uint32_t j1 = e0 >> log_cl, c = e0 & ((1u << log_cl) - 1);
    const uint32_t j0 = (j1 << log_m) + col0 + c;
    Fr pw = j0 < n ? gen.pow_u32(j0) : Fr::zero();
    for (uint32_t k = 0; k < 4; k++) {
        const uint32_t j = j0 + k;
        Fr v = Fr::zero();
        if (j < n) {
            v = ld_fr(poly + j) * pw;
            pw = pw * gen;
        }
        st_fr(dst + e0 + k, v);
    }
}
// … and back: t_j ← t_j·7^{−j} on the column-layout shard after the inverse transform
__global__ void __launch_bounds__(256) dist_unscale_kernel(Fr *data, uint32_t log_m, uint32_t log_cl, uint32_t col0, uint32_t local, Fr gen_inv) {
    const uint32_t e0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (e0 >= local) return;
    const uint32_t j1 = e0 >> log_cl, c = e0 & ((1u << log_cl) - 1);
    Fr pw = gen_inv.pow_u32((j1 << log_m) + col0 + c);
    for (uint32_t k = 0; k < 4; k++) {
        st_fr(data + e0 + k, ld_fr(data + e0 + k) * pw);
        pw = pw * gen_inv;
    }
}

// ------------------------------------------------------------------------------------------------ round 4 / 5
// out[j] = Σ_k c_k·p_k[j]  (p_k zero beyond len_k)
constexpr int kMaxTerms = 12;
struct LcArgs {
    const Fr *p[kMaxTerms];
    uint32_t len[kMaxTerms];
    Fr c[kMaxTerms];
    int terms;
    uint32_t n;
    Fr *out;
};
__global__ void __launch_bounds__(256) lincomb_kernel(const LcArgs A) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= A.n) return;
    Fr acc = Fr::zero();
    for (int k = 0; k < A.terms; k++)
        if (j < A.len[k]) acc = acc + A.c[k] * ld_fr(A.p[k] + j);
    st_fr(A.out + j, acc);
}
// Polynomial::evaluate for many (polynomial, point) pairs at once.  A CTA covers 8192 coefficients: each thread
// runs Horner over 32 of them, scales by point^(first index), and the CTA tree-sums into one partial; a second
// launch adds the partials of each job.
constexpr int kMaxJobs = 20;
// (32 coefficients per thread: the x^first factor costs ≈ 30 multiplications per thread, so 8 per thread spent 4/5 of the
// kernel on it — 1.3 ms per proof at 2^20 gates)
constexpr uint32_t kEvalPerThread = 32, kEvalTile = 256 * kEvalPerThread;
struct EvalArgs {
    const Fr *p[kMaxJobs];
    uint32_t len[kMaxJobs];    // coefficients this launch covers: [off, off + len)
    uint32_t off[kMaxJobs];    // (a rank of a sharded prove evaluates its coefficient slice; the partial sums are all-gathered)
    uint32_t point[kMaxJobs];
    Fr points[2];
    Fr *partial;  // [job][tiles]
    uint32_t tiles;
};
__device__ __forceinline__ Fr block_sum(Fr v, Fr *sm) {
    const uint32_t t = threadIdx.x;
    st_fr(sm + t, v);
    __syncthreads();
    for (uint32_t o = 128; o >= 1; o >>= 1) {
        if (t < o) {
            v = v + ld_fr(sm + t + o);
            st_fr(sm + t, v);
        }
        __syncthreads();
    }
    return v;
}
__global__ void __launch_bounds__(256) poly_eval_partial_kernel(const EvalArgs A) {
    __shared__ uint4 smraw[512];
    Fr *sm = reinterpret_cast<Fr *>(smraw);
    const uint32_t job = blockIdx.y, len = A.len[job];
    if (blockIdx.x * kEvalTile >= len) {   // short job in a grid sized for the longest one: nothing to add
        if (threadIdx.x == 0) st_fr(A.partial + (size_t)job * A.tiles + blockIdx.x, Fr::zero());
        return;
    }
    const Fr *p = A.p[job] + A.off[job];
    const Fr x = A.points[A.point[job]];
    const uint32_t first = blockIdx.x * kEvalTile + threadIdx.x * kEvalPerThread;
    Fr acc = Fr::zero();
    if (first < len) {
        const uint32_t last = min(first + kEvalPerThread, len);
        acc = ld_fr(p + last - 1);
        for (uint32_t j = last - 1; j-- > first;) acc = acc * x + ld_fr(p + j);
        acc = acc * x.pow_u32(A.off[job] + first);
    }
    acc = block_sum(acc, sm);
    if (threadIdx.x == 0) st_fr(A.partial + (size_t)job * A.tiles + blockIdx.x, acc);
}
__global__ void __launch_bounds__(256) poly_eval_final_kernel(const Fr *partial, uint32_t tiles, Fr *out) {
    __shared__ uint4 smraw[512];
    Fr *sm = reinterpret_cast<Fr *>(smraw);
    const uint32_t job = blockIdx.x;
    Fr acc = Fr::zero();
    for (uint32_t t = threadIdx.x; t < tiles; t += 256) acc = acc + ld_fr(partial + (size_t)job * tiles + t);
    acc = block_sum(acc, sm);
    if (threadIdx.x == 0) st_fr(out + job, acc);
}

inline uint32_t cdiv(size_t a, uint32_t b) { return (uint32_t)((a + b - 1) / b); }

}  // namespace

// ---------------------------------------------------------------------------------------------------- prover key
struct pb200_prover_key {
    uint32_t log_n = 0;
    size_t n = 0, n_gates = 0, n_vars = 0;
    bool q_nonzero[kSel] = {};
    // device-resident (one allocation, carved)
    void *slab = nullptr;
    size_t slab_bytes = 0;
    Fr *q_poly[kSel] = {}, *q_4n[kSel] = {};
    Fr *sig_evals = nullptr, *sig_poly = nullptr, *sig_4n = nullptr;  // 4·n, 4·n, 4·4n
    Fr *roots = nullptr, *lin_4n = nullptr, *l1_4n = nullptr;  // ω^i | X on the coset | L₁ on the coset
    uint32_t *wires = nullptr;
    // Lagrange-basis commit key of this domain with its pre-doubled copies (lagrange.cu): round 1 commits the wire
    // evaluations against it.  nullptr: the wires are committed from their coefficients against the caller's key.
    pb200_srs *lagrange = nullptr;
    size_t lagrange_bytes = 0;
    // prove workspace
    Fr *values = nullptr, *w_evals = nullptr, *w_poly = nullptr, *z_poly = nullptr, *pi_poly = nullptr, *ev4 = nullptr, *t_poly = nullptr,
       *lin_poly = nullptr, *agg = nullptr, *wit = nullptr, *num = nullptr, *den = nullptr, *small = nullptr;
    uint32_t *pi_pos = nullptr;
    size_t pi_cap = 0;
    HFr vh_inv[4];
    HFr omega, omega4;
    uint8_t vk_bytes[15 * 48];
    merlin::Transcript *seeded = nullptr;
    // point-range sharding of the commitments (world = 1: none)
    pb200_shard shard = {0, 1, nullptr, nullptr, nullptr, nullptr, 0};
    size_t slice_lo = 0, slice_n = 0;  // this rank's coefficient range [slice_lo, slice_lo + slice_n)
    // peer mappings of every rank's key slab (CUDA IPC over NVLink) for the fused column-transform + exchange kernel
    void *peer_slab[8] = {};
    bool peers_open = false, peers_failed = false;
};

namespace {

struct Carver {
    char *base;
    size_t off = 0;
    explicit Carver(void *b) : base((char *)b) {}
    template <class T>
    T *take(size_t count) {
        T *p = base ? (T *)(base + off) : nullptr;
        off += (count * sizeof(T) + 255) & ~(size_t)255;
        return p;
    }
};
// `small`: 64 scalars | 2 × scan tile products | evaluation partials
inline size_t scan_tiles(size_t n) { return (n + kTile - 1) / kTile; }
inline size_t eval_tiles(size_t n4) { return (n4 + kEvalTile - 1) / kEvalTile; }

void carve(pb200_prover_key *pk, void *base, size_t *total) {
    Carver c(base);
    const size_t n = pk->n, N4 = 4 * n;
    // non-zero selectors back to back (coefficient forms, then coset evaluations) so that they transform and commit as a batch
    size_t n_sel = 0;
    for (int s = 0; s < kSel; s++) n_sel += pk->q_nonzero[s];
    Fr *qp = c.take<Fr>(n_sel * n), *q4 = c.take<Fr>(n_sel * N4);
    for (int s = 0, k = 0; s < kSel; s++) {
        if (!pk->q_nonzero[s]) continue;
        pk->q_poly[s] = qp ? qp + (size_t)k * n : nullptr;
        pk->q_4n[s] = q4 ? q4 + (size_t)k * N4 : nullptr;
        k++;
    }
    pk->sig_evals = c.take<Fr>(4 * n);
    pk->sig_poly = c.take<Fr>(4 * n);
    pk->sig_4n = c.take<Fr>(4 * N4);
    pk->roots = c.take<Fr>(n);
    pk->lin_4n = c.take<Fr>(N4);
    pk->l1_4n = c.take<Fr>(N4);
    pk->wires = c.take<uint32_t>(4 * pk->n_gates);
    pk->values = c.take<Fr>(pk->n_vars);
    pk->w_evals = c.take<Fr>(4 * n);
    pk->w_poly = c.take<Fr>(4 * n);
    pk->z_poly = c.take<Fr>(n);
    pk->pi_poly = c.take<Fr>(n);
    // a, b, c, d | z | pi on the coset; a sharded key holds 8 column shards, 8 row buffers, the local quotient and the
    // gathered coefficients of t(X) here instead
    const size_t world = pk->shard.world;
    pk->ev4 = c.take<Fr>(std::max<size_t>(6 * N4, world > 1 ? 17 * (N4 / world) + N4 + 64 : 0));
    pk->t_poly = c.take<Fr>(N4);
    pk->lin_poly = c.take<Fr>(n);
    pk->agg = c.take<Fr>(n);
    pk->wit = c.take<Fr>(2 * n);
    pk->num = c.take<Fr>(n);
    pk->den = c.take<Fr>(n);
    pk->small = c.take<Fr>(64 + 2 * scan_tiles(n) + kMaxJobs * eval_tiles(N4));
    *total = c.off;
}

int launch_scan(pb200_ctx *ctx, pb200_prover_key *pk, Fr *a, uint32_t n, bool rev, Fr *tiles, Fr *grand) {
    const uint32_t n_tiles = cdiv(n, kTile);
    if (rev) scan_tile_products_kernel<true><<<n_tiles, 256, 0, ctx->stream>>>(a, n, tiles);
    else scan_tile_products_kernel<false><<<n_tiles, 256, 0, ctx->stream>>>(a, n, tiles);
    PB_LAUNCHED(ctx);
    scan_top_kernel<<<1, 256, 0, ctx->stream>>>(tiles, n_tiles, grand);
    PB_LAUNCHED(ctx);
    if (rev) scan_finish_kernel<true><<<n_tiles, 256, 0, ctx->stream>>>(a, n, tiles);
    else scan_finish_kernel<false><<<n_tiles, 256, 0, ctx->stream>>>(a, n, tiles);
    PB_LAUNCHED(ctx);
    return 0;
}

// commit(`batch` polynomials of n coefficients, `stride` scalars apart) → 48 compressed bytes each.  Single GPU: one
// batched pass over the commit key.  Sharded: the MSM runs over this rank's coefficient slice against its slice of
// the key, the partial sums are all-gathered through the host's collective and added (pb200_g1_sum).
int commit_bytes_batch(pb200_ctx *ctx, const pb200_srs *srs, const pb200_prover_key *pk, const Fr *polys, size_t n, uint32_t batch,
                       size_t stride, uint8_t *out) {
    uint64_t xyz[18 * 16];
    PB_ARG(ctx, batch <= 16);
    if (pk->shard.world <= 1) {
        PB_TRY(pb200_msm_g1_batch_dev(ctx, srs, 0, (const uint64_t *)polys, n, batch, stride, xyz));
    } else {
        PB_ARG(ctx, n == pk->n);
        if ((pk->shard.flags & PB200_SHARD_STREAM_ORDERED) && comm_partials_buffer(ctx)) {
            // in-library NCCL: partial sums stay on the device — MSM → all-gather → one add kernel → one D2H
            bool handled = false;
            PB_TRY(msm_batch_to_dev(ctx, srs, 0, (const uint64_t *)(polys + pk->slice_lo), pk->slice_n, batch, stride, comm_partials_buffer(ctx),
                                    &handled));
            if (handled) {
                PB_TRY(comm_sum_partials(ctx, batch, xyz));
                for (uint32_t j = 0; j < batch; j++) hostf::g1_projective_to_bytes(xyz + 18 * j, out + 48 * j);
                return 0;
            }
        }
        PB_TRY(pb200_msm_g1_batch_dev(ctx, srs, 0, (const uint64_t *)(polys + pk->slice_lo), pk->slice_n, batch, stride, xyz));
        const uint32_t world = pk->shard.world;
        std::vector<uint64_t> all((size_t)world * batch * 18), one((size_t)world * 18);
        if (pk->shard.allgather(pk->shard.user, xyz, all.data(), (size_t)batch * 144) != 0)
            return pb_fail(ctx, PB200_ERR_ARG, "sharded commit", "the all-gather callback failed", __FILE__, __LINE__);
        for (uint32_t j = 0; j < batch; j++) {
            for (uint32_t r = 0; r < world; r++) memcpy(&one[(size_t)r * 18], &all[((size_t)r * batch + j) * 18], 144);
            PB_TRY(pb200_g1_sum(ctx, one.data(), world, xyz + 18 * j));
        }
    }
    for (uint32_t j = 0; j < batch; j++) hostf::g1_projective_to_bytes(xyz + 18 * j, out + 48 * j);
    return 0;
}
int commit_bytes(pb200_ctx *ctx, const pb200_srs *srs, const pb200_prover_key *pk, const Fr *poly, size_t n, uint8_t out[48]) {
    return commit_bytes_batch(ctx, srs, pk, poly, n, 1, n, out);
}

int coset_extend(pb200_ctx *ctx, Fr *dst, const Fr *src, uint32_t n, uint32_t log_n4, uint32_t batch) {
    const uint32_t N4 = 1u << log_n4;
    pad_copy_kernel<<<dim3(cdiv(N4, 256), batch), 256, 0, ctx->stream>>>(dst, src, n, N4);
    PB_LAUNCHED(ctx);
    return pb200_ntt_batch_dev(ctx, (uint64_t *)dst, log_n4, batch, 0, 1);
}

// Σ over the ranks of `count` scalars each rank computed from its slice (evaluation partial sums): one host all-gather
// (count × 32 bytes per rank) and `world` exact field additions — every rank derives the same values.  world = 1: a copy.
int sum_over_ranks(pb200_ctx *ctx, const pb200_prover_key *pk, const uint64_t *mine, int count, HFr *out) {
    const uint32_t world = pk->shard.world;
    if (world <= 1) {
        for (int k = 0; k < count; k++) out[k] = HFr::load(mine + 4 * k);
        return 0;
    }
    std::vector<uint64_t> send(mine, mine + 4 * (size_t)count), all((size_t)world * 4 * count);
    if (pk->shard.allgather(pk->shard.user, send.data(), all.data(), (size_t)count * 32) != 0)
        return pb_fail(ctx, PB200_ERR_ARG, "sharded evaluation", "the all-gather callback failed", __FILE__, __LINE__);
    for (int k = 0; k < count; k++) {
        HFr acc = HFr::zero();
        for (uint32_t r = 0; r < world; r++) acc = acc + HFr::load(&all[((size_t)r * count + k) * 4]);
        out[k] = acc;
    }
    return 0;
}

struct RoundClock {
    pb200_ctx *ctx;
    std::chrono::steady_clock::time_point t0;
    explicit RoundClock(pb200_ctx *c) : ctx(c), t0(std::chrono::steady_clock::now()) {}
    void lap(const char *name) {
        if (!ctx->profile) return;
        cudaStreamSynchronize(ctx->stream);
        auto t1 = std::chrono::steady_clock::now();
        const float ms = std::chrono::duration<float, std::milli>(t1 - t0).count();
        ctx->prof_ms[name] = ms;
        ctx->prof_sum[name] += ms;
        ctx->prof_cnt[name]++;
        t0 = t1;
    }
};

}  // namespace

extern "C" void pb200_prover_key_free(pb200_ctx *ctx, pb200_prover_key *pk) {
    if (!pk) return;
    if (ctx) cudaSetDevice(ctx->device);
    for (uint32_t h = 0; h < 8; h++)
        if (pk->peer_slab[h] && h != pk->shard.rank) cudaIpcCloseMemHandle(pk->peer_slab[h]);
    cudaFree(pk->slab);
    cudaFree(pk->pi_pos);
    pb200_srs_free(ctx, pk->lagrange);
    delete pk->seeded;
    delete pk;
}
extern "C" size_t pb200_prover_key_size(const pb200_prover_key *pk) { return pk ? pk->n : 0; }
extern "C" size_t pb200_prover_key_bytes(const pb200_prover_key *pk) { return pk ? pk->slab_bytes + pk->lagrange_bytes : 0; }

extern "C" int pb200_preprocess(pb200_ctx *ctx, const pb200_srs *srs, const pb200_circuit *circuit, const uint8_t *transcript_label,
                                size_t label_len, pb200_prover_key **out, uint8_t vk_commitments[15 * 48]) {
    return pb200_preprocess_sharded(ctx, srs, circuit, transcript_label, label_len, nullptr, out, vk_commitments);
}
extern "C" int pb200_preprocess_sharded(pb200_ctx *ctx, const pb200_srs *srs, const pb200_circuit *circuit,
                                        const uint8_t *transcript_label, size_t label_len, const pb200_shard *shard,
                                        pb200_prover_key **out, uint8_t vk_commitments[15 * 48]) {
    if (!ctx) return PB200_ERR_ARG;
    const uint32_t world = shard ? shard->world : 1;
    PB_ARG(ctx, world >= 1 && (world & (world - 1)) == 0 && (world == 1 || (shard->allgather != nullptr && shard->rank < world)));
    PB_ARG(ctx, srs != nullptr && circuit != nullptr && out != nullptr && (transcript_label != nullptr || label_len == 0));
    PB_ARG(ctx, circuit->n_gates >= 1 && circuit->n_vars >= 1 && circuit->n_vars < ((size_t)1 << 32));
    for (int c = 0; c < 4; c++) PB_ARG(ctx, circuit->wires[c] != nullptr);
    uint32_t log_n = 0;
    PB_TRY(pb200_domain_log_size(circuit->n_gates, &log_n));
    PB_ARG(ctx, log_n <= 26);  // 4n domain (2^28 scalars = 8 GiB per vector) and the 2-bit column tag of the permutation map
    const size_t n = (size_t)1 << log_n, N4 = 4 * n, ng = circuit->n_gates;
    PB_ARG(ctx, world <= n && pb200_srs_len(srs) >= n / world);
    PB_CUDA(ctx, cudaSetDevice(ctx->device));

    pb200_prover_key *pk = new pb200_prover_key();
    if (world > 1) pk->shard = *shard;
    pk->slice_n = n / world;
    pk->slice_lo = (size_t)pk->shard.rank * pk->slice_n;
    pk->log_n = log_n;
    pk->n = n;
    pk->n_gates = ng;
    pk->n_vars = circuit->n_vars;
    auto fail = [&](int rc) {
        pb200_prover_key_free(ctx, pk);
        return rc;
    };
    // which selector columns are not identically zero
    for (int s = 0; s < kSel; s++) {
        const uint64_t *col = circuit->selectors[s];
        bool nz = false;
        if (col)
            for (size_t i = 0; i < 4 * ng && !nz; i++) nz = col[i] != 0;
        pk->q_nonzero[s] = nz;
    }
    // permutation: position (col, i) ↦ next occurrence of the same variable, cyclically, in gate order then l, r, o, 4
    std::vector<uint32_t> map(4 * n);
    {
        const uint32_t none = 0xffffffffu;
        std::vector<uint32_t> first(circuit->n_vars, none), last(circuit->n_vars, none);
        for (uint32_t c = 0; c < 4; c++)
            for (size_t i = 0; i < n; i++) map[c * n + i] = (uint32_t)((c << log_n) | i);
        for (size_t i = 0; i < ng; i++)
            for (uint32_t c = 0; c < 4; c++) {
                const uint32_t v = circuit->wires[c][i];
                if (v >= circuit->n_vars) {
                    pb_fail(ctx, PB200_ERR_ARG, "bad circuit", "wire refers to an unallocated variable", __FILE__, __LINE__);
                    return fail(PB200_ERR_ARG);
                }
                const uint32_t here = (uint32_t)((c << log_n) | i);
                if (last[v] == none) first[v] = here;
                else map[(size_t)(last[v] >> log_n) * n + (last[v] & (n - 1))] = here;
                last[v] = here;
            }
        for (size_t v = 0; v < circuit->n_vars; v++)
            if (last[v] != none) map[(size_t)(last[v] >> log_n) * n + (last[v] & (n - 1))] = first[v];
    }
    carve(pk, nullptr, &pk->slab_bytes);
    cudaError_t e = cudaMalloc(&pk->slab, pk->slab_bytes);
    if (e != cudaSuccess) {
        pb_fail(ctx, PB200_ERR_CUDA, "prover key allocation", cudaGetErrorString(e), __FILE__, __LINE__);
        return fail(PB200_ERR_CUDA);
    }
    size_t dummy;
    carve(pk, pk->slab, &dummy);
    cudaStream_t st = ctx->stream;
#define PK_CUDA(call)                                                                                         \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess) {                                                                             \
            pb_fail(ctx, PB200_ERR_CUDA, #call, cudaGetErrorString(e__), __FILE__, __LINE__);                 \
            return fail(PB200_ERR_CUDA);                                                                      \
        }                                                                                                     \
    } while (0)
#define PK_TRY(expr)                    \
    do {                                \
        int rc__ = (expr);              \
        if (rc__) return fail(rc__);    \
    } while (0)
#define PK_LAUNCHED()                                                                                         \
    do {                                                                                                      \
        ctx->launches++;                                                                                      \
        PK_CUDA(cudaGetLastError());                                                                          \
    } while (0)

    // domain constants on the host
    {
        const HFr w4 = hostf::domain_root(log_n + 2);
        pk->omega = hostf::domain_root(log_n);
        pk->omega4 = w4;
        // 1 / ((7·ω_4n^i)^n − 1), i mod 4:  7^n · (ω_4n^n)^i − 1
        const HFr g = HFr::from_u64(7), gn = g.pow_u64(n), i4 = w4.pow_u64(n), one = HFr::one();
        HFr cur = gn;
        for (int k = 0; k < 4; k++) {
            pk->vh_inv[k] = (cur - one).inv();
            cur = cur * i4;
        }
    }
    KFactors ks;
    ks.k[0] = to_dev(HFr::one());
    ks.k[1] = to_dev(HFr::from_u64(7));
    ks.k[2] = to_dev(HFr::from_u64(13));
    ks.k[3] = to_dev(HFr::from_u64(17));

    // wires, permutation map (staged in the t_poly workspace), roots of unity, σ evaluations
    for (int c = 0; c < 4; c++)
        PK_CUDA(cudaMemcpyAsync(pk->wires + (size_t)c * ng, circuit->wires[c], ng * 4, cudaMemcpyHostToDevice, st));
    uint32_t *map_dev = (uint32_t *)pk->t_poly;
    PK_CUDA(cudaMemcpyAsync(map_dev, map.data(), 4 * n * 4, cudaMemcpyHostToDevice, st));
    powers_kernel<<<cdiv(n, 256), 256, 0, st>>>(pk->roots, (uint32_t)n, to_dev(HFr::one()), to_dev(pk->omega));
    PK_LAUNCHED();
    powers_kernel<<<cdiv(N4, 256), 256, 0, st>>>(pk->lin_4n, (uint32_t)N4, to_dev(HFr::from_u64(7)), to_dev(pk->omega4));
    PK_LAUNCHED();
    sigma_evals_kernel<<<dim3(cdiv(n, 256), 4), 256, 0, st>>>(pk->sig_evals, map_dev, pk->roots, (uint32_t)n, log_n, ks);
    PK_LAUNCHED();
    PK_CUDA(cudaStreamSynchronize(st));  // `map` (pageable) must outlive its copy

    // selector and σ polynomials: interpolate, commit, extend to the 4n coset
    uint8_t *vk = pk->vk_bytes;
    {
        int first = -1;
        uint32_t n_sel = 0;
        for (int s = 0; s < kSel; s++) {
            uint8_t *dst = vk + 48 * s;
            memset(dst, 0, 48);
            dst[0] = 0xc0;  // commitment to the zero polynomial: the identity
            if (!pk->q_nonzero[s]) continue;
            if (first < 0) first = s;
            n_sel++;
            PK_CUDA(cudaMemsetAsync(pk->q_poly[s], 0, n * sizeof(Fr), st));
            PK_CUDA(cudaMemcpyAsync(pk->q_poly[s], circuit->selectors[s], ng * sizeof(Fr), cudaMemcpyHostToDevice, st));
        }
        if (n_sel) {
            uint8_t packed[kSel * 48];
            PK_TRY(pb200_ntt_batch_dev(ctx, (uint64_t *)pk->q_poly[first], log_n, n_sel, 1, 0));
            PK_TRY(commit_bytes_batch(ctx, srs, pk, pk->q_poly[first], n, n_sel, n, packed));
            PK_TRY(coset_extend(ctx, pk->q_4n[first], pk->q_poly[first], (uint32_t)n, log_n + 2, n_sel));
            for (int s = 0, k = 0; s < kSel; s++)
                if (pk->q_nonzero[s]) memcpy(vk + 48 * s, packed + 48 * k++, 48);
        }
    }
    PK_CUDA(cudaMemcpyAsync(pk->sig_poly, pk->sig_evals, 4 * n * sizeof(Fr), cudaMemcpyDeviceToDevice, st));
    PK_TRY(pb200_ntt_batch_dev(ctx, (uint64_t *)pk->sig_poly, log_n, 4, 1, 0));
    PK_TRY(commit_bytes_batch(ctx, srs, pk, pk->sig_poly, n, 4, n, vk + 48 * kSel));
    PK_TRY(coset_extend(ctx, pk->sig_4n, pk->sig_poly, (uint32_t)n, log_n + 2, 4));
    // L₁ on the coset (its n coefficients are all 1/n): circuit-independent, so the prover only scales it by α²
    fill_kernel<<<cdiv(n, 256), 256, 0, st>>>(pk->lin_poly, (uint32_t)n, to_dev(HFr::from_u64(n).inv()));
    PK_LAUNCHED();
    PK_TRY(coset_extend(ctx, pk->l1_4n, pk->lin_poly, (uint32_t)n, log_n + 2, 1));
    PK_CUDA(cudaStreamSynchronize(st));

    // Lagrange-basis key for round 1: one GPU, a commit key with pre-doubled copies (the batched MSM needs them) and a
    // domain whose copies fit (n ≤ 2^22, like pb200_srs_precompute).  PB200_LAGRANGE_COMMIT=0 keeps the monomial path.
    const char *lag_env = getenv("PB200_LAGRANGE_COMMIT");
    if (world == 1 && log_n <= 22 && srs->pre != nullptr && !(lag_env && strcmp(lag_env, "0") == 0)) {
        bool degenerate = false;  // some L_i(τ) = 0: not a powers-of-τ key; the monomial path still commits correctly
        PK_TRY(lagrange_srs_build(ctx, srs, log_n, &pk->lagrange, &degenerate));
        if (pk->lagrange) {
            PK_TRY(pb200_srs_precompute(ctx, pk->lagrange));
            pk->lagrange_bytes = n * 96 * (1 + pk->lagrange->W_pre);  // affine points + their pre-doubled copies
        }
    }

    // Transcript::new(label) seeded with the verifier key
    pk->seeded = new merlin::Transcript(transcript_label, label_len);
    merlin::seed_transcript(*pk->seeded, vk, n);
    if (vk_commitments) memcpy(vk_commitments, vk, sizeof(pk->vk_bytes));
    *out = pk;
    return 0;
#undef PK_CUDA
#undef PK_TRY
#undef PK_LAUNCHED
}

static int prove_impl(pb200_ctx *ctx, const pb200_srs *srs, pb200_prover_key *pk, const uint64_t *values_mont, bool values_on_device,
                      const uint32_t *pi_gate, const uint64_t *pi_mont, size_t n_pi, uint8_t proof_out[1040]);
extern "C" int pb200_prove(pb200_ctx *ctx, const pb200_srs *srs, pb200_prover_key *pk, const uint64_t *values_mont,
                           const uint32_t *pi_gate, const uint64_t *pi_mont, size_t n_pi, uint8_t proof_out[1040]) {
    return prove_impl(ctx, srs, pk, values_mont, false, pi_gate, pi_mont, n_pi, proof_out);
}
extern "C" int pb200_prove_dev(pb200_ctx *ctx, const pb200_srs *srs, pb200_prover_key *pk, const uint64_t *values_mont_dev,
                               const uint32_t *pi_gate, const uint64_t *pi_mont, size_t n_pi, uint8_t proof_out[1040]) {
    return prove_impl(ctx, srs, pk, values_mont_dev, true, pi_gate, pi_mont, n_pi, proof_out);
}
static int prove_impl(pb200_ctx *ctx, const pb200_srs *srs, pb200_prover_key *pk, const uint64_t *values_mont, bool values_on_device,
                      const uint32_t *pi_gate, const uint64_t *pi_mont, size_t n_pi, uint8_t proof_out[1040]) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, srs != nullptr && pk != nullptr && values_mont != nullptr && proof_out != nullptr);
    PB_ARG(ctx, n_pi == 0 || (pi_gate != nullptr && pi_mont != nullptr));
    PB_ARG(ctx, pb200_srs_len(srs) >= pk->slice_n);
    for (size_t j = 0; j < n_pi; j++) PB_ARG(ctx, pi_gate[j] < pk->n);
    if (n_pi > 1) {  // a gate carries one public input: duplicates would race in the scatter and disagree with the verifier's sum
        std::vector<uint32_t> sorted(pi_gate, pi_gate + n_pi);
        std::sort(sorted.begin(), sorted.end());
        PB_ARG(ctx, std::adjacent_find(sorted.begin(), sorted.end()) == sorted.end());
    }
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t n = pk->n, N4 = 4 * n;
    const uint32_t n32 = (uint32_t)n, log_n = pk->log_n;
    RoundClock clk(ctx);
    merlin::Transcript tr = *pk->seeded;  // dusk clones the preprocessed transcript for every proof
    uint8_t *P = proof_out;
    KFactors ks;
    ks.k[0] = to_dev(HFr::one());
    ks.k[1] = to_dev(HFr::from_u64(7));
    ks.k[2] = to_dev(HFr::from_u64(13));
    ks.k[3] = to_dev(HFr::from_u64(17));
    Fr *scal = pk->small;                  // 64 device scalars
    Fr *tilesA = pk->small + 64, *tilesB = tilesA + scan_tiles(n), *partial = tilesB + scan_tiles(n);

    // ---- round 1: wire polynomials --------------------------------------------------------------------------------
    const Fr *values_dev = (const Fr *)values_mont;
    if (!values_on_device) {
        PB_CUDA(ctx, cudaMemcpyAsync(pk->values, values_mont, pk->n_vars * sizeof(Fr), cudaMemcpyHostToDevice, st));
        values_dev = pk->values;
    }
    gather_wires_kernel<<<dim3(cdiv(n, 256), 4), 256, 0, st>>>(pk->w_evals, pk->wires, values_dev, (uint32_t)pk->n_gates, n32);
    PB_LAUNCHED(ctx);
    PB_CUDA(ctx, cudaMemcpyAsync(pk->w_poly, pk->w_evals, 4 * n * sizeof(Fr), cudaMemcpyDeviceToDevice, st));
    PB_TRY(pb200_ntt_batch_dev(ctx, (uint64_t *)pk->w_poly, log_n, 4, 1, 0));
    const char *const w_label[4] = {"w_l", "w_r", "w_o", "w_4"};
    // Σ_i w(ω^i)·[L_i(τ)]G = [w(τ)]G: the evaluations are mostly zero or small (d is zero off a few rows, padding rows
    // are zero), and a zero or small scalar costs no or one MSM entry where its coefficient form costs 13
    if (pk->lagrange) PB_TRY(commit_bytes_batch(ctx, pk->lagrange, pk, pk->w_evals, n, 4, n, P));
    else PB_TRY(commit_bytes_batch(ctx, srs, pk, pk->w_poly, n, 4, n, P));
    for (int c = 0; c < 4; c++) tr.append_commitment(w_label[c], P + 48 * c);
    clk.lap("prove.round1");

    // ---- round 2: permutation polynomial ------------------------------------------------------------------------------
    const HFr beta = tr.challenge_scalar("beta");
    tr.append_scalar("beta", beta);
    const HFr gamma = tr.challenge_scalar("gamma");
    perm_numden_kernel<<<cdiv(n, 256), 256, 0, st>>>(pk->w_evals, pk->sig_evals, pk->roots, n32, to_dev(beta), to_dev(gamma), ks, pk->num,
                                                    pk->den);
    PB_LAUNCHED(ctx);
    PB_TRY(launch_scan(ctx, pk, pk->num, n32, false, tilesA, scal + 0));
    PB_TRY(launch_scan(ctx, pk, pk->den, n32, true, tilesB, scal + 1));
    fr_inv_kernel<<<1, 1, 0, st>>>(scal + 1, scal + 2);
    PB_LAUNCHED(ctx);
    perm_finish_kernel<<<cdiv(n, 256), 256, 0, st>>>(pk->num, pk->den, scal + 2, n32, pk->z_poly);
    PB_LAUNCHED(ctx);
    PB_TRY(pb200_ntt_dev(ctx, (uint64_t *)pk->z_poly, log_n, 1, 0));
    PB_TRY(commit_bytes(ctx, srs, pk, pk->z_poly, n, P + 48 * 4));
    tr.append_commitment("z", P + 48 * 4);
    clk.lap("prove.round2");

    // ---- round 3: quotient polynomial ------------------------------------------------------------------------------------
    const HFr alpha = tr.challenge_scalar("alpha");
    const HFr range_sep = tr.challenge_scalar("range separation challenge");
    const HFr logic_sep = tr.challenge_scalar("logic separation challenge");
    const HFr fixed_sep = tr.challenge_scalar("fixed base separation challenge");
    const HFr var_sep = tr.challenge_scalar("variable base separation challenge");
    const HFr edwards_d = (HFr::from_u64(10240) * HFr::from_u64(10241).inv()).neg();   // JubJub: −x² + y² = 1 + d·x²y²
    // dense public inputs → pi_poly
    PB_CUDA(ctx, cudaMemsetAsync(pk->pi_poly, 0, n * sizeof(Fr), st));
    if (n_pi) {
        if (pk->pi_cap < n_pi) {
            cudaFree(pk->pi_pos);
            pk->pi_pos = nullptr;
            pk->pi_cap = 0;
            PB_CUDA(ctx, cudaMalloc((void **)&pk->pi_pos, n_pi * (4 + sizeof(Fr)) + 32));
            pk->pi_cap = n_pi;
        }
        Fr *pi_vals = (Fr *)((char *)pk->pi_pos + ((n_pi * 4 + 31) & ~(size_t)31));
        PB_CUDA(ctx, cudaMemcpyAsync(pk->pi_pos, pi_gate, n_pi * 4, cudaMemcpyHostToDevice, st));
        PB_CUDA(ctx, cudaMemcpyAsync(pi_vals, pi_mont, n_pi * sizeof(Fr), cudaMemcpyHostToDevice, st));
        scatter_pi_kernel<<<cdiv(n_pi, 256), 256, 0, st>>>(pk->pi_poly, pk->pi_pos, pi_vals, (uint32_t)n_pi);
        PB_LAUNCHED(ctx);
        PB_TRY(pb200_ntt_dev(ctx, (uint64_t *)pk->pi_poly, log_n, 1, 0));
    }
    QuotArgs A;
    for (int s = 0; s < kSel; s++) A.q[s] = pk->q_4n[s];
    A.sig = pk->sig_4n;
    A.lin = pk->lin_4n;
    A.l1 = pk->l1_4n;
    A.N4 = (uint32_t)N4;
    A.alpha = to_dev(alpha);
    A.alpha2 = to_dev(alpha.sqr());
    A.beta = to_dev(beta);
    A.gamma = to_dev(gamma);
    A.range_sep = to_dev(range_sep);
    A.logic_sep = to_dev(logic_sep);
    A.fixed_sep = to_dev(fixed_sep);
    A.var_sep = to_dev(var_sep);
    A.edwards_d = to_dev(edwards_d);
    for (int k = 0; k < 4; k++) A.vh_inv[k] = to_dev(pk->vh_inv[k]);
    A.ks = ks;
    A.zw = A.dw = nullptr;
    A.dist = A.log_m = A.log_n1 = A.row0 = 0;
    const bool range = pk->q_nonzero[Q_RANGE];
    const bool extra = pk->q_nonzero[Q_LOGIC] || pk->q_nonzero[Q_FIXED] || pk->q_nonzero[Q_VAR];
    const uint32_t world = pk->shard.world, log_n4 = log_n + 2;
    uint32_t log_g = 0;
    while ((1u << log_g) < world) log_g++;
    // (the sharded layout transforms z(ωX) and d(ωX) only: circuits with ECC / logic rows keep round 3 replicated)
    const bool dist3 = world > 1 && pk->shard.alltoall_dev && pk->shard.allgather_dev && log_n4 >= 8 + log_g + 2 && !extra;
    if (!dist3) {
        // coset evaluations on 4n: a, b, c, d | z | pi   (L₁ is kept from preprocessing)
        Fr *w4 = pk->ev4, *z4 = pk->ev4 + 4 * N4, *pi4 = z4 + N4;
        PB_TRY(coset_extend(ctx, w4, pk->w_poly, n32, log_n4, 4));
        PB_TRY(coset_extend(ctx, z4, pk->z_poly, n32, log_n4, 1));
        PB_TRY(coset_extend(ctx, pi4, pk->pi_poly, n32, log_n4, 1));
        A.w = w4;
        A.z = z4;
        A.pi = pi4;
        A.out = pk->t_poly;
        A.count = (uint32_t)N4;
        if (extra) {
            if (range) quotient_kernel<true, true><<<cdiv(N4, 128), 128, 0, st>>>(A);
            else quotient_kernel<false, true><<<cdiv(N4, 128), 128, 0, st>>>(A);
        } else {
            if (range) quotient_kernel<true, false><<<cdiv(N4, 128), 128, 0, st>>>(A);
            else quotient_kernel<false, false><<<cdiv(N4, 128), 128, 0, st>>>(A);
        }
        PB_LAUNCHED(ctx);
        PB_TRY(pb200_ntt_dev(ctx, (uint64_t *)pk->t_poly, log_n4, 1, 1));
    } else {
        // Sharded four-step transforms (SURVEY.md §8e): N4 = n1 × m, this rank owns cl = m / world columns of the
        // coefficient side and rl = n1 / world rows of the evaluation side; one all-to-all per transform.
        const uint32_t log_n1 = 8, log_m = log_n4 - log_n1, log_cl = log_m - log_g, log_rl = log_n1 - log_g;
        const uint32_t rank = pk->shard.rank, cl = 1u << log_cl, rl = 1u << log_rl, col0 = rank << log_cl;
        const size_t local = N4 >> log_g, peer_bytes = (local >> log_g) * sizeof(Fr);
        const HFr seven = HFr::from_u64(7);
        Fr *cols = pk->ev4;                   // column-layout shards (sources of the fused kernel): 8 × `local` scalars
        Fr *shard = pk->ev4 + 8 * local;      // row-layout shards a b c d | z | pi | z(ωX) | d(ωX)
        Fr *t_loc = pk->ev4 + 16 * local;     // this rank's quotient evaluations / coefficients
        Fr *gathered = pk->ev4 + 17 * local;  // all ranks' coefficient shards (N4 scalars)
        Fr *tmp = pk->t_poly;                 // exchange buffer of the NCCL path
        struct { const Fr *poly; HFr gen; } src[8] = {{pk->w_poly, seven}, {pk->w_poly + n, seven}, {pk->w_poly + 2 * n, seven},
                                                      {pk->w_poly + 3 * n, seven}, {pk->z_poly, seven}, {pk->pi_poly, seven},
                                                      {pk->z_poly, seven * pk->omega}, {pk->w_poly + 3 * n, seven * pk->omega}};
        const int n_src = range ? 8 : 7;
        // in-library NCCL (pb200_preprocess_comm): collectives are enqueued on `st` itself — no host synchronisation anywhere
        const bool ordered = (pk->shard.flags & PB200_SHARD_STREAM_ORDERED) != 0;
        auto exchange = [&](Fr *send, Fr *recv) -> int {
            if (!ordered) PB_CUDA(ctx, cudaStreamSynchronize(st));
            if (pk->shard.alltoall_dev(pk->shard.user, send, recv, peer_bytes) != 0)
                return ordered ? PB200_ERR_CUDA : pb_fail(ctx, PB200_ERR_ARG, "sharded transform", "the all-to-all callback failed", __FILE__, __LINE__);
            return 0;
        };
        auto barrier = [&]() -> int {  // every rank's stream has drained: a one-byte all-gather through the host collective
            if (ordered) return comm_stream_barrier(ctx);   // … or, stream-ordered, a one-word NCCL all-gather on `st`
            PB_CUDA(ctx, cudaStreamSynchronize(st));
            uint8_t one_byte = 1, all[8];
            if (pk->shard.allgather(pk->shard.user, &one_byte, all, 1) != 0)
                return pb_fail(ctx, PB200_ERR_ARG, "sharded transform", "the all-gather callback failed", __FILE__, __LINE__);
            return 0;
        };
        // Peer mappings of all key slabs, once per key: the forward exchange is then the column kernel's own store
        // (pb200_ntt_columns_scatter_dev writes every output into the owner's row buffer over NVLink).  The keys have the
        // same layout on every rank (same circuit), so a peer's buffer is its slab base plus this rank's offset.
        static const bool force_nccl = getenv("PB200_ROUND3_NCCL") != nullptr;  // measurement switch
        if (!pk->peers_open && !pk->peers_failed && !force_nccl && world <= 8) {
            cudaIpcMemHandle_t mine;
            std::vector<cudaIpcMemHandle_t> all(world);
            bool ok = cudaIpcGetMemHandle(&mine, pk->slab) == cudaSuccess;
            uint8_t flag = ok ? 1 : 0;
            if (!ok) memset(&mine, 0, sizeof(mine));
            if (pk->shard.allgather(pk->shard.user, &mine, all.data(), sizeof(mine)) != 0)
                return pb_fail(ctx, PB200_ERR_ARG, "sharded transform", "the all-gather callback failed", __FILE__, __LINE__);
            for (uint32_t h = 0; h < world && ok; h++) {
                if (h == rank) pk->peer_slab[h] = pk->slab;
                else ok = cudaIpcOpenMemHandle(&pk->peer_slab[h], all[h], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
            }
            flag = ok ? 1 : 0;
            uint8_t flags[8];
            if (pk->shard.allgather(pk->shard.user, &flag, flags, 1) != 0)
                return pb_fail(ctx, PB200_ERR_ARG, "sharded transform", "the all-gather callback failed", __FILE__, __LINE__);
            for (uint32_t h = 0; h < world; h++) ok = ok && flags[h];
            (void)cudaGetLastError();
            pk->peers_open = ok;        // all ranks or none: otherwise fall back to the NCCL all-to-all everywhere
            pk->peers_failed = !ok;
        }
        const bool fused = pk->peers_open && !force_nccl;
        if (fused) PB_TRY(barrier());  // nobody is still reading the row buffers of an earlier use
        for (int k = 0; k < n_src; k++) {
            Fr *col = cols + (size_t)k * local, *row = shard + (size_t)k * local;
            dist_load_kernel<<<cdiv(local / 4, 256), 256, 0, st>>>(col, src[k].poly, n32, log_m, log_cl, col0, (uint32_t)local, to_dev(src[k].gen));
            PB_LAUNCHED(ctx);
            if (fused) {
                void *peer_rows[8];
                const size_t off = (size_t)((char *)row - (char *)pk->slab);
                for (uint32_t h = 0; h < world; h++) peer_rows[h] = (char *)pk->peer_slab[h] + off;
                PB_TRY(pb200_ntt_columns_scatter_dev(ctx, (uint64_t *)col, log_n4, log_n1, log_cl, col0, world, peer_rows));
            } else {
                PB_TRY(pb200_ntt_columns_dev(ctx, (uint64_t *)col, log_n4, log_n1, log_cl, col0, 0));
                PB_TRY(exchange(col, tmp));                                                              // block h (rl × cl) → rank h
                PB_TRY(pb200_block_transpose_dev(ctx, (uint64_t *)row, (const uint64_t *)tmp, world, rl, cl));  // → rl rows of length m
            }
        }
        if (fused) PB_TRY(barrier());  // every rank has finished storing into every row buffer
        PB_TRY(pb200_ntt_batch_dev(ctx, (uint64_t *)shard, log_m, (uint32_t)n_src * rl, 0, 0));       // all rows of all shards at once
        A.w = shard;
        A.z = shard + 4 * local;
        A.pi = shard + 5 * local;
        A.zw = shard + 6 * local;
        A.dw = shard + 7 * local;
        A.out = t_loc;
        A.dist = 1;
        A.count = (uint32_t)local;
        A.log_m = log_m;
        A.log_n1 = log_n1;
        A.row0 = rank << log_rl;
        if (range) quotient_kernel<true, false><<<cdiv(local, 128), 128, 0, st>>>(A);
        else quotient_kernel<false, false><<<cdiv(local, 128), 128, 0, st>>>(A);
        PB_LAUNCHED(ctx);
        // inverse: rows → regroup → all-to-all → columns (with n⁻¹ and the twiddles) → coset unscale
        PB_TRY(pb200_ntt_batch_dev(ctx, (uint64_t *)t_loc, log_m, rl, 1, 0));
        PB_TRY(pb200_block_transpose_dev(ctx, (uint64_t *)tmp, (const uint64_t *)t_loc, rl, world, cl));
        PB_TRY(exchange(tmp, t_loc));
        PB_TRY(pb200_ntt_columns_dev(ctx, (uint64_t *)t_loc, log_n4, log_n1, log_cl, col0, 1));
        dist_unscale_kernel<<<cdiv(local / 4, 256), 256, 0, st>>>(t_loc, log_m, log_cl, col0, (uint32_t)local, to_dev(seven.inv()));
        PB_LAUNCHED(ctx);
        // every rank needs all of t(X) for rounds 4-5: all-gather the column shards, then back to natural order
        if (!ordered) PB_CUDA(ctx, cudaStreamSynchronize(st));
        if (pk->shard.allgather_dev(pk->shard.user, t_loc, gathered, local * sizeof(Fr)) != 0)
            return ordered ? PB200_ERR_CUDA : pb_fail(ctx, PB200_ERR_ARG, "sharded transform", "the device all-gather callback failed", __FILE__, __LINE__);
        PB_TRY(pb200_block_transpose_dev(ctx, (uint64_t *)pk->t_poly, (const uint64_t *)gathered, world, 1u << log_n1, cl));
    }
    const char *const t_label[4] = {"t_1", "t_2", "t_3", "t_4"};
    PB_TRY(commit_bytes_batch(ctx, srs, pk, pk->t_poly, n, 4, n, P + 48 * 5));
    for (int k = 0; k < 4; k++) tr.append_commitment(t_label[k], P + 48 * (5 + k));
    clk.lap("prove.round3");

    // ---- round 4: evaluations and the linearisation polynomial -------------------------------------------------------------
    const HFr z = tr.challenge_scalar("z");
    const HFr zw = z * pk->omega;
    enum { E_A, E_B, E_C, E_D, E_AN, E_BN, E_DN, E_S1, E_S2, E_S3, E_QARITH, E_QC, E_QL, E_QR, E_PERM, E_T, E_COUNT };
    HFr ev[E_COUNT + 1];
    {
        EvalArgs A;
        int j = 0;
        auto job = [&](const Fr *p, size_t len, int point) {   // sharded: this rank's coefficient slice of every polynomial
            A.p[j] = p;
            A.len[j] = p ? (uint32_t)(len / world) : 0;
            A.off[j] = p ? (uint32_t)(pk->shard.rank * (len / world)) : 0;
            A.point[j] = point;
            j++;
        };
        for (int c = 0; c < 4; c++) job(pk->w_poly + (size_t)c * n, n, 0);
        job(pk->w_poly, n, 1);
        job(pk->w_poly + n, n, 1);
        job(pk->w_poly + 3 * n, n, 1);
        for (int c = 0; c < 3; c++) job(pk->sig_poly + (size_t)c * n, n, 0);
        job(pk->q_poly[Q_ARITH], n, 0);
        job(pk->q_poly[Q_C], n, 0);
        job(pk->q_poly[Q_L], n, 0);
        job(pk->q_poly[Q_R], n, 0);
        job(pk->z_poly, n, 1);
        job(pk->t_poly, N4, 0);
        A.points[0] = to_dev(z);
        A.points[1] = to_dev(zw);
        A.partial = partial;
        A.tiles = cdiv(N4 / world, kEvalTile);
        poly_eval_partial_kernel<<<dim3(A.tiles, j), 256, 0, st>>>(A);
        PB_LAUNCHED(ctx);
        poly_eval_final_kernel<<<j, 256, 0, st>>>(partial, A.tiles, scal + 8);
        PB_LAUNCHED(ctx);
        PB_CUDA(ctx, cudaMemcpyAsync(ctx->pinned, scal + 8, E_COUNT * sizeof(Fr), cudaMemcpyDeviceToHost, st));
        PB_CUDA(ctx, cudaStreamSynchronize(st));
        PB_TRY(sum_over_ranks(ctx, pk, (const uint64_t *)ctx->pinned, E_COUNT, ev));
    }
    const HFr one = HFr::one();
    const HFr zn = z.pow_u64(n);
    const HFr z_h = zn - one;
    const HFr l1 = z_h * (HFr::from_u64(n) * (z - one)).inv();
    HFr lin_z, lin_s4;
    {
        const HFr k1 = HFr::from_u64(7), k2 = HFr::from_u64(13), k3 = HFr::from_u64(17), bz = beta * z;
        const HFr id = (ev[E_A] + bz + gamma) * (ev[E_B] + k1 * bz + gamma) * (ev[E_C] + k2 * bz + gamma) * (ev[E_D] + k3 * bz + gamma);
        lin_z = id * alpha + l1 * alpha.sqr();
        lin_s4 = ((ev[E_A] + beta * ev[E_S1] + gamma) * (ev[E_B] + beta * ev[E_S2] + gamma) * (ev[E_C] + beta * ev[E_S3] + gamma) * beta *
                  ev[E_PERM] * alpha)
                     .neg();
    }
    {
        LcArgs A;
        int k = 0;
        auto term = [&](const Fr *p, const HFr &c) {
            if (!p) return;
            A.p[k] = p;
            A.len[k] = n32;
            A.c[k] = to_dev(c);
            k++;
        };
        const HFr qa = ev[E_QARITH];
        term(pk->q_poly[Q_M], ev[E_A] * ev[E_B] * qa);
        term(pk->q_poly[Q_L], ev[E_A] * qa);
        term(pk->q_poly[Q_R], ev[E_B] * qa);
        term(pk->q_poly[Q_O], ev[E_C] * qa);
        term(pk->q_poly[Q_4], ev[E_D] * qa);
        term(pk->q_poly[Q_C], qa);
        if (pk->q_nonzero[Q_RANGE]) {
            const HFr four = HFr::from_u64(4), kappa = range_sep.sqr();
            auto delta = [&](const HFr &f) { return f * (f - one) * (f - one - one) * (f - one - one - one); };
            HFr r = delta(ev[E_DN] - four * ev[E_A]);
            r = r * kappa + delta(ev[E_A] - four * ev[E_B]);
            r = r * kappa + delta(ev[E_B] - four * ev[E_C]);
            r = r * kappa + delta(ev[E_C] - four * ev[E_D]);
            term(pk->q_poly[Q_RANGE], r * range_sep);
        }
        if (pk->q_nonzero[Q_LOGIC])
            term(pk->q_poly[Q_LOGIC], widgets::logic_term(ev[E_A], ev[E_AN], ev[E_B], ev[E_BN], ev[E_C], ev[E_D], ev[E_DN], ev[E_QC], logic_sep));
        if (pk->q_nonzero[Q_FIXED])
            term(pk->q_poly[Q_FIXED], widgets::fixed_base_term(ev[E_A], ev[E_AN], ev[E_B], ev[E_BN], ev[E_C], ev[E_D], ev[E_DN], ev[E_QL],
                                                               ev[E_QR], ev[E_QC], fixed_sep, edwards_d));
        if (pk->q_nonzero[Q_VAR])
            term(pk->q_poly[Q_VAR], widgets::var_base_term(ev[E_A], ev[E_AN], ev[E_B], ev[E_BN], ev[E_C], ev[E_D], ev[E_DN], var_sep, edwards_d));
        term(pk->z_poly, lin_z);
        term(pk->sig_poly + 3 * n, lin_s4);
        A.terms = k;
        A.n = n32;
        A.out = pk->lin_poly;
        lincomb_kernel<<<cdiv(n, 256), 256, 0, st>>>(A);
        PB_LAUNCHED(ctx);
    }
    {
        EvalArgs A;
        A.p[0] = pk->lin_poly;
        A.len[0] = n32 / world;
        A.off[0] = pk->shard.rank * (n32 / world);
        A.point[0] = 0;
        A.points[0] = to_dev(z);
        A.points[1] = to_dev(zw);
        A.partial = partial;
        A.tiles = cdiv(n / world, kEvalTile);
        poly_eval_partial_kernel<<<dim3(A.tiles, 1), 256, 0, st>>>(A);
        PB_LAUNCHED(ctx);
        poly_eval_final_kernel<<<1, 256, 0, st>>>(partial, A.tiles, scal + 8);
        PB_LAUNCHED(ctx);
        PB_CUDA(ctx, cudaMemcpyAsync(ctx->pinned, scal + 8, sizeof(Fr), cudaMemcpyDeviceToHost, st));
        PB_CUDA(ctx, cudaStreamSynchronize(st));
        PB_TRY(sum_over_ranks(ctx, pk, (const uint64_t *)ctx->pinned, 1, &ev[E_COUNT]));  // r(z)
    }
    {
        const struct { const char *label; int idx; } order[17] = {
            {"a_eval", E_A}, {"b_eval", E_B}, {"c_eval", E_C}, {"d_eval", E_D}, {"a_next_eval", E_AN}, {"b_next_eval", E_BN},
            {"d_next_eval", E_DN}, {"left_sig_eval", E_S1}, {"right_sig_eval", E_S2}, {"out_sig_eval", E_S3},
            {"q_arith_eval", E_QARITH}, {"q_c_eval", E_QC}, {"q_l_eval", E_QL}, {"q_r_eval", E_QR}, {"perm_eval", E_PERM},
            {"t_eval", E_T}, {"r_eval", E_COUNT}};
        for (const auto &o : order) tr.append_scalar(o.label, ev[o.idx]);
        // ProofEvaluations::to_bytes order
        const int bytes_order[16] = {E_A, E_B, E_C, E_D, E_AN, E_BN, E_DN, E_QARITH, E_QC, E_QL, E_QR, E_S1, E_S2, E_S3, E_COUNT, E_PERM};
        for (int k = 0; k < 16; k++) hostf::fr_to_bytes(ev[bytes_order[k]], P + 528 + 32 * k);
    }
    clk.lap("prove.round4");

    // ---- round 5: opening witnesses ---------------------------------------------------------------------------------
    for (int which = 0; which < 2; which++) {
        const HFr v = tr.challenge_scalar("aggregate_witness");
        LcArgs A;
        int k = 0;
        HFr pw = one;
        auto term = [&](const Fr *p, const HFr &c) {
            A.p[k] = p;
            A.len[k] = n32;
            A.c[k] = to_dev(c);
            k++;
        };
        if (which == 0) {
            // quotient opening polynomial t_1 + z^n·t_2 + z^2n·t_3 + z^3n·t_4, then r, a, b, c, d, σ1, σ2, σ3
            HFr zp = one;
            for (int j = 0; j < 4; j++) {
                term(pk->t_poly + (size_t)j * n, zp);
                zp = zp * zn;
            }
            const Fr *rest[8] = {pk->lin_poly, pk->w_poly, pk->w_poly + n, pk->w_poly + 2 * n, pk->w_poly + 3 * n,
                                 pk->sig_poly, pk->sig_poly + n, pk->sig_poly + 2 * n};
            for (int j = 0; j < 8; j++) {
                pw = pw * v;
                term(rest[j], pw);
            }
        } else {
            const Fr *polys[4] = {pk->z_poly, pk->w_poly, pk->w_poly + n, pk->w_poly + 3 * n};
            for (int j = 0; j < 4; j++) {
                term(polys[j], pw);
                pw = pw * v;
            }
        }
        A.terms = k;
        uint64_t point[4], unused[4];
        (which == 0 ? z : zw).store(point);
        const bool z_zero = (point[0] | point[1] | point[2] | point[3]) == 0;
        if (world > 1 && !z_zero && kzg_witness_slice_work_scalars((uint32_t)pk->slice_n) <= n / 2) {
            // Sharded: this rank only needs its coefficient slice of the witness (its share of the commitment).  Linear
            // combination over the slice, local suffix scan, and the totals of the later slices (32 bytes per rank) as carry.
            const uint32_t lo = (uint32_t)pk->slice_lo, cnt = (uint32_t)pk->slice_n;
            for (int t = 0; t < k; t++) {
                A.p[t] += lo;
                A.len[t] = cnt;
            }
            A.n = cnt;
            A.out = pk->agg + lo;
            lincomb_kernel<<<cdiv(cnt, 256), 256, 0, st>>>(A);
            PB_LAUNCHED(ctx);
            Fr *q_slice = pk->wit + (size_t)which * n + lo;
            uint64_t *work = (uint64_t *)(pk->num + (size_t)which * (n / 2));   // round-2 scratch, free by now: ≥ 5 + cnt/1024 scalars
            uint64_t mine[4];
            PB_TRY(kzg_witness_slice_phase1(ctx, (const uint64_t *)(pk->agg + lo), lo, cnt, point, (uint64_t *)q_slice, work, mine));
            std::vector<uint64_t> all((size_t)world * 4);
            if (pk->shard.allgather(pk->shard.user, mine, all.data(), 32) != 0)
                return pb_fail(ctx, PB200_ERR_ARG, "sharded witness", "the all-gather callback failed", __FILE__, __LINE__);
            HFr later = HFr::zero();
            for (uint32_t r = pk->shard.rank + 1; r < world; r++) later = later + HFr::load(&all[(size_t)r * 4]);
            uint64_t carry[4];
            later.store(carry);
            PB_TRY(kzg_witness_slice_phase2(ctx, lo, cnt, (uint64_t *)q_slice, work, carry));
            continue;
        }
        A.n = n32;
        A.out = pk->agg;
        lincomb_kernel<<<cdiv(n, 256), 256, 0, st>>>(A);
        PB_LAUNCHED(ctx);
        PB_TRY(pb200_kzg_witness_dev(ctx, (const uint64_t *)pk->agg, n, point, (uint64_t *)(pk->wit + (size_t)which * n), unused));
    }
    // the second challenge is squeezed before either witness is committed, so both commitments are one batched MSM
    PB_TRY(commit_bytes_batch(ctx, srs, pk, pk->wit, n, 2, n, P + 48 * 9));
    clk.lap("prove.round5");
    return 0;
}

extern "C" int pb200_transcript_selftest(const char *label, const char *msg_label, const uint8_t *msg, size_t msg_len,
                                         const char *challenge_label, uint8_t *out, size_t out_len) {
    if (!label || !msg_label || !challenge_label || !out || (!msg && msg_len)) return PB200_ERR_ARG;
    merlin::Transcript t((const uint8_t *)label, strlen(label));
    t.append_message(msg_label, msg, msg_len);
    t.challenge_bytes(challenge_label, out, out_len);
    return 0;
}

// ---- synthetic workload (bench / tests): the circuit of plonk-prototype_b200/synth.py, assembled on the host in C++ so
// that 2^24 gates take a second instead of a minute.  Same rows, same witness.
extern "C" int pb200_synthetic_circuit(size_t n_gates, uint64_t seed, uint32_t n_pub, uint64_t *const selectors7[7], uint32_t *const wires[4],
                                       uint64_t *values_mont, size_t n_vars_capacity, size_t *n_vars_out, uint32_t *pi_gate,
                                       uint64_t *pi_mont) {
    if (!selectors7 || !wires || !values_mont || !n_vars_out || n_gates < 8 + (size_t)n_pub || n_pub < 1) return PB200_ERR_ARG;
    if (n_pub > 1 && (!pi_gate || !pi_mont)) return PB200_ERR_ARG;
    // SplitMix64 → uniform scalars by rejection (SURVEY.md §8d)
    uint64_t st = seed;
    auto next64 = [&]() {
        uint64_t z = (st += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    };
    HFr consts[4];
    for (int k = 0; k < 4;) {
        HFr v;
        for (int i = 0; i < 4; i++) v.l[i] = next64();
        v.l[3] &= 0x7fffffffffffffffull;
        if (!HFr::geq_mod(v.l)) consts[k++] = v * HFr::r2();
    }
    const size_t steps = (n_gates - n_pub - 3) / 2, n_bool = n_gates - n_pub - 3 - 2 * steps;
    const size_t n_vars = 6 + 2 * steps + (n_pub - 1);
    *n_vars_out = n_vars;
    if (n_vars > n_vars_capacity) return PB200_ERR_ARG;
    enum { M, L, R, O, C, F, A };
    for (int k = 0; k < 7; k++) memset(selectors7[k], 0, n_gates * 32);
    for (int c = 0; c < 4; c++) memset(wires[c], 0, n_gates * 4);
    const HFr one = HFr::one(), minus_one = one.neg();
    auto setq = [&](int col, size_t row, const HFr &v) { v.store(selectors7[col] + 4 * row); };
    auto setw = [&](size_t row, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
        wires[0][row] = a; wires[1][row] = b; wires[2][row] = c; wires[3][row] = d;
    };
    for (size_t i = 0; i < n_gates; i++) setq(A, i, one);
    HFr *vals = (HFr *)values_mont;
    vals[0] = HFr::zero();
    vals[1] = HFr::from_u64(6);
    vals[2] = one;
    vals[3] = HFr::from_u64(7);
    vals[4] = HFr::from_u64(20).neg();
    vals[5] = consts[0];
    setq(L, 0, one);
    setw(1, 1, 3, 4, 2);
    setq(M, 1, one); setq(L, 1, HFr::from_u64(2)); setq(R, 1, HFr::from_u64(3)); setq(O, 1, HFr::from_u64(4));
    setq(C, 1, HFr::from_u64(4)); setq(F, 1, one);
    setw(2, 4, 1, 3, 0);
    setq(M, 2, one); setq(L, 2, one); setq(R, 2, one); setq(O, 2, one); setq(C, 2, HFr::from_u64(127));
    HFr x = consts[0], c = consts[1];
    for (size_t k = 0; k < steps; k++) {
        const uint32_t xv = (uint32_t)(5 + 2 * k), sq = xv + 1, xn = xv + 2;
        const size_t r_mul = 3 + 2 * k, r_add = r_mul + 1;
        const HFr s = x * x;
        x = s + x + c;
        vals[sq] = s;
        vals[xn] = x;
        setw(r_mul, xv, xv, sq, 0);
        setq(M, r_mul, one); setq(O, r_mul, minus_one);
        setw(r_add, sq, xv, xn, 0);
        setq(L, r_add, one); setq(R, r_add, one); setq(O, r_add, minus_one); setq(C, r_add, c);
        c = c + one;
    }
    const uint32_t x_var = (uint32_t)(5 + 2 * steps);
    for (size_t r = 3 + 2 * steps; r < 3 + 2 * steps + n_bool; r++) { setq(M, r, one); setq(O, r, minus_one); }
    for (uint32_t j = 0; j < n_pub; j++) {
        const size_t row = n_gates - n_pub + j;
        uint32_t var = x_var;
        HFr v = x;
        if (j > 0) {
            var = (uint32_t)(6 + 2 * steps + (j - 1));
            vals[var] = consts[2];
            v = consts[2];
        }
        setw(row, var, var, var, 0);
        setq(L, row, one);
        pi_gate[j] = (uint32_t)row;
        v.neg().store(pi_mont + 4 * j);
    }
    return 0;
}
