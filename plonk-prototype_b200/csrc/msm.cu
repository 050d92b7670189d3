// msm.cu — variable-base multi-scalar multiplication over BLS12-381 G1 for sm_100a.
//
// Replaces dusk-bls12_381 0.8 `multiscalar_mul::msm_variable_base(&[G1Affine], &[Scalar]) -> G1Projective`
// (crate pinned at /root/reference/Cargo.toml:20; upstream algorithm restated in SURVEY.md App. B.1 and
// oracle/oracle.c).  The result is a group element, so it is compared after normalisation to affine.
//
// Pipeline (DESIGN.md §MSM) — everything stays on the device, no host round trip until the result:
//   1. count    scalars → canonical → signed c-bit digits; histogram of (window, |digit|) buckets
//   2. scan     exclusive prefix sum of the histogram → bucket offsets
//   3. scatter  (bucket id, point index | sign) entries, grouped by bucket           ("sort by bucket")
//   4. accumulate  segmented reduction over the entry list: every thread owns a fixed-length segment
//                  (perfect balance whatever the digit distribution), sums runs of equal bucket id with
//                  mixed XYZZ+affine additions, writes complete runs to their bucket and emits ≤ 2
//                  boundary partials; partials are reduced by the same scheme, level by level
//   5. reduce   Σ_b b·B_b per window as chunked running sums, then a per-window tree sum
//   6. combine  Horner over the windows (c doublings each), normalise to affine
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "msm_common.cuh"

namespace {

// --------------------------------------------------------------------------------- digit recoding
// Signed-digit decomposition of a canonical 255-bit scalar into W digits of c bits:
// digit ∈ [−2^(c−1), 2^(c−1)]; the top window is never recoded (W·c ≥ 256 leaves it a spare bit).
template <class F>
__device__ __forceinline__ void for_each_digit(const Fr &canon, uint32_t c, uint32_t W, F &&f) {
    const uint32_t half = 1u << (c - 1), mask = (1u << c) - 1;
    uint32_t carry = 0;
    for (uint32_t w = 0; w < W; w++) {
        const uint32_t bit = w * c, limb = bit >> 5, off = bit & 31;
        uint64_t v = canon.l[limb];
        if (limb + 1 < 8) v |= (uint64_t)canon.l[limb + 1] << 32;
        uint32_t raw = ((uint32_t)(v >> off) & mask) + carry;
        uint32_t sign = 0;
        carry = 0;
        if (w + 1 < W && raw > half) {
            raw = (1u << c) - raw;
            sign = 1;
            carry = 1;
        }
        if (raw) f(w, raw, sign);
    }
}

// blockIdx.y = scalar vector of a batched call (pre-doubled path): vector j reads scalars + j·stride and owns bucket set j.
__global__ void __launch_bounds__(256) msm_count_kernel(const uint64_t *scalars, MsmCfg cfg, uint32_t *count) {
    const uint32_t set = blockIdx.y << cfg.nb_log;
    scalars += 4 * (size_t)blockIdx.y * cfg.scalar_stride;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < cfg.n; i += (size_t)gridDim.x * blockDim.x) {
        Fr s = load_fr(scalars, i).from_mont();
        for_each_digit(s, cfg.c, cfg.W, [&](uint32_t w, uint32_t mag, uint32_t) {
            atomicAdd(&count[(cfg.pre_stride ? set : (w << cfg.nb_log)) + mag - 1], 1u);
        });
    }
}
// `shift` = 0: entries go straight to their bucket's slot range (cursor = per-bucket offsets).
// `shift` > 0: first level of the two-level scatter used once the entry list outgrows L2 — the cursor array is per
// *coarse bin* (2^shift buckets, ≈ 32 Ki entries) and entries are only grouped by bin.  All CTAs share one write
// frontier per bin, so the open lines (bins × 128 B) stay in L2 and reach DRAM complete: ncu shows 6.65 GB written
// for 6.44 GB of entries at 2^26, against one 32-byte sector per 8-byte entry for the single-level scatter.
// (Reserving per-CTA runs from shared-memory histograms was tried: fewer global atomics, but the open set becomes
// in-flight-entries × 8 B ≈ 465 MB ≫ L2 and DRAM traffic triples — 74 ms instead of 42 ms — so it was dropped.)
__global__ void __launch_bounds__(256) msm_scatter_kernel(const uint64_t *scalars, MsmCfg cfg, uint32_t *cursor, uint2 *entries,
                                                          uint32_t shift) {
    const uint32_t set = blockIdx.y << cfg.nb_log;
    scalars += 4 * (size_t)blockIdx.y * cfg.scalar_stride;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < cfg.n; i += (size_t)gridDim.x * blockDim.x) {
        Fr s = load_fr(scalars, i).from_mont();
        for_each_digit(s, cfg.c, cfg.W, [&](uint32_t w, uint32_t mag, uint32_t sign) {
            const uint32_t gb = (cfg.pre_stride ? set : (w << cfg.nb_log)) + mag - 1;
            const uint32_t pos = atomicAdd(&cursor[gb >> shift], 1u);
            entries[pos] = make_uint2(gb, (uint32_t)(w * cfg.pre_stride + i) | (sign << 31));
        });
    }
}
// coarse[b] = offsets[b << shift]: where each coarse bin starts in the entry list
__global__ void msm_coarse_init_kernel(const uint32_t *offsets, uint32_t *coarse, uint32_t n_coarse, uint32_t shift) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < n_coarse) coarse[b] = offsets[b << shift];
}
// Second level: walk the bin-grouped list in order; each entry moves to its bucket's slot.  CTAs that run at the
// same time cover a few neighbouring bins, so the scattered 8-byte writes stay inside an L2-resident window.
// Both levels are bound by global atomics with return (~45-50 G/s on B200).
__global__ void __launch_bounds__(256) msm_fine_scatter_kernel(const uint2 *__restrict__ grouped, const uint32_t *__restrict__ n_entries_ptr,
                                                               uint32_t *cursor, uint2 *entries) {
    const uint32_t M = *n_entries_ptr;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const uint2 e = grouped[i];
    const uint32_t pos = atomicAdd(&cursor[e.x], 1u);
    entries[pos] = e;
}

// ------------------------------------------------------------------------------------------- scan
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t *block_total) {
    __shared__ uint32_t warp_sums[32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc += t;
    }
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t ws = warp_sums[lane];
        uint32_t winc = ws;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= (uint32_t)o) winc += t;
        }
        warp_sums[lane] = winc - ws;  // exclusive
        if (lane == 31 && block_total) *block_total = winc;
    }
    __syncthreads();
    uint32_t r = inc - v + warp_sums[warp];
    __syncthreads();
    return r;
}
__global__ void __launch_bounds__(kScanThreads) scan_block_sums_kernel(const uint32_t *in, uint32_t n, uint32_t *block_sums) {
    __shared__ uint32_t total;
    const uint32_t base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
    uint32_t s = 0;
#pragma unroll
    for (uint32_t k = 0; k < kScanItems; k++)
        if (base + k < n) s += in[base + k];
    block_exclusive_scan(s, &total);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}
__global__ void __launch_bounds__(kScanThreads) scan_top_kernel(uint32_t *block_sums, uint32_t nblocks, uint32_t *total_out) {
    __shared__ uint32_t total;
    const uint32_t per = (nblocks + kScanThreads - 1) / kScanThreads;
    const uint32_t lo = threadIdx.x * per, hi = min(lo + per, nblocks);
    uint32_t s = 0;
    for (uint32_t i = lo; i < hi; i++) s += block_sums[i];
    uint32_t ex = block_exclusive_scan(s, &total);
    for (uint32_t i = lo; i < hi; i++) {
        uint32_t v = block_sums[i];
        block_sums[i] = ex;
        ex += v;
    }
    if (threadIdx.x == 0) *total_out = total;
}
__global__ void __launch_bounds__(kScanThreads) scan_apply_kernel(const uint32_t *in, uint32_t n, const uint32_t *block_sums, uint32_t *out) {
    const uint32_t base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
    uint32_t v[kScanItems], s = 0;
#pragma unroll
    for (uint32_t k = 0; k < kScanItems; k++) {
        v[k] = (base + k < n) ? in[base + k] : 0;
        s += v[k];
    }
    uint32_t ex = block_exclusive_scan(s, nullptr) + block_sums[blockIdx.x];
#pragma unroll
    for (uint32_t k = 0; k < kScanItems; k++) {
        if (base + k < n) out[base + k] = ex;
        ex += v[k];
    }
}

// Level 1: entries (bucket id, point index | sign) → buckets / partial slots, mixed additions.
__device__ __forceinline__ void msm_accumulate_body(const G1Affine *__restrict__ bases, const uint2 *__restrict__ entries,
                                                    const uint32_t *__restrict__ n_entries_ptr, uint32_t L, G1Xyzz *buckets,
                                                    uint32_t *out_gb, G1Xyzz *out_pt, uint32_t *n_out_ptr) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t M = *n_entries_ptr;
    if (t == 0) *n_out_ptr = 2 * ((M + L - 1) / L);
    const uint64_t start64 = (uint64_t)t * L;
    if (start64 >= M) return;
    const uint32_t start = (uint32_t)start64, end = (uint32_t)min((uint64_t)M, start64 + L);
    const uint32_t prev = start > 0 ? entries[start - 1].x : kInvalid;
    const uint32_t next = end < M ? entries[end].x : kInvalid;
    RunSink sink{buckets, out_gb, out_pt, t, kInvalid, kInvalid};

    uint2 e = entries[start];
    uint32_t cur = e.x;
    bool tl = (prev == cur);
    G1Xyzz acc = G1Xyzz::identity();
    for (uint32_t i = start; i < end; i++) {
        G1Affine pt = load_affine(bases, e.y);
        const uint32_t gb = e.x;
        if (i + 1 < end) {
            e = entries[i + 1];
            // pull the next base towards L2/L1 while this addition runs
            const char *np = reinterpret_cast<const char *>(bases + (e.y & 0x7fffffffu));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(np));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(np + 64));
        }
        if (gb != cur) {
            sink.flush(cur, g1_canonical(acc), tl, false);
            cur = gb;
            tl = false;
            acc = G1Xyzz::identity();
        }
        g1_madd_lazy(acc, pt);   // coordinates stay in [0, 2p) while the run's sum lives in registers (g1.cuh)
    }
    sink.flush(cur, g1_canonical(acc), tl, next == cur);
    sink.finish();
}
__global__ void __launch_bounds__(128) msm_accumulate_kernel(const G1Affine *__restrict__ bases, const uint2 *__restrict__ entries,
                                                             const uint32_t *__restrict__ n_entries_ptr, uint32_t L, G1Xyzz *buckets,
                                                             uint32_t *out_gb, G1Xyzz *out_pt, uint32_t *n_out_ptr) {
    msm_accumulate_body(bases, entries, n_entries_ptr, L, buckets, out_gb, out_pt, n_out_ptr);
}
// Window width with pre-doubled copies: one shared bucket set, so only W·n additions + one reduction of 2^(c−1) buckets.
uint32_t choose_window_pre(size_t n) {
    uint32_t best_c = 8;
    double best = 1e300;
    for (uint32_t c = 8; c <= 23; c++) {
        const double W = (256 + c - 1) / c;
        const double cost = W * (double)n + 3.0 * (double)(1u << (c - 1));
        if (cost <= best) { best = cost; best_c = c; }
    }
    return best_c;
}

// Window width minimising W·(n + 3·2^(c−1)): n·W mixed additions plus ≈ 3 addition-equivalents per bucket
// for the running-sum reduction.
uint32_t choose_window(size_t n) {
    uint32_t best_c = 4;
    double best = 1e300;
    for (uint32_t c = 4; c <= 23; c++) {
        const double W = (256 + c - 1) / c;
        const double cost = W * ((double)n + 3.0 * (double)(1u << (c - 1)));
        if (cost <= best) { best = cost; best_c = c; }
    }
    return best_c;
}
uint32_t floor_pow2(uint64_t v) {
    uint32_t p = 1;
    while (((uint64_t)p << 1) <= v) p <<= 1;
    return p;
}

}  // namespace

int msm_module_init(pb200_ctx *) { return 0; }

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// One piece (n < 2^27) of an MSM; bases / scalars on the device.
// batch > 1 (pre-doubled path only): `batch` scalar vectors, `scalar_stride` scalars apart, against the same bases;
// result_dev then receives `batch` records of 36 words.
static int msm_piece(pb200_ctx *ctx, const G1Affine *bases, const uint64_t *scalars, uint32_t n, int first, int last,
                     G1Xyzz *running_total, uint32_t *result_dev, uint32_t pre_c, uint32_t pre_stride, uint32_t batch = 1,
                     uint32_t scalar_stride = 0) {
    PB_ARG(ctx, batch >= 1 && (batch == 1 || (pre_stride && first && last)));
    MsmCfg cfg;
    cfg.batch = batch;
    cfg.scalar_stride = scalar_stride;
    cfg.n = n;
    cfg.c = pre_stride ? pre_c : choose_window(n);
    cfg.W = (256 + cfg.c - 1) / cfg.c;
    cfg.nb_log = cfg.c - 1;
    cfg.pre_stride = pre_stride;
    const uint64_t m0 = (uint64_t)n * cfg.W * batch;  // upper bound on entries
    PB_ARG(ctx, m0 < (1ull << 32));
    cfg.L1 = std::min<uint32_t>(128, std::max<uint32_t>(8, floor_pow2(m0 / 262144 + 1)));
    {   // every thread of the accumulation does the same work, so a partly filled last wave is pure loss (prover-size calls
        // ran 11.24 waves: 6 %): shorten the segments until the grid is a whole number of waves (2 CTAs of 128 threads per SM)
        const uint64_t wave = (uint64_t)ctx->sm_count * 2 * 128;
        const uint64_t waves = (m0 + wave * cfg.L1 - 1) / (wave * cfg.L1);
        cfg.L1 = std::max<uint32_t>(8, (uint32_t)((m0 + wave * waves - 1) / (wave * waves)));
    }
    cfg.L2 = 16;
    const uint32_t n_win = pre_stride ? batch : cfg.W;   // bucket sets (windows to reduce / combine)
    const uint32_t TB = n_win << cfg.nb_log;          // total buckets
    {   // Chunk size K of the bucket reduction (one thread per K consecutive buckets: 2K running-sum additions plus one small
        // scalar multiple of ≈ 22 addition-equivalents for the chunk's offset).  The kernel runs 2 CTAs of 128 threads per SM
        // (255 registers), every thread does the same work, so the time is (number of waves) × (work per thread): choose the K
        // that minimises it — larger K amortises the scalar multiple, smaller K fills the machine, and a partly filled last
        // wave costs a whole one.  (Measured, profiles/msm_tail_scaling_r02.json: the old fixed rule — ≥ 64 Ki threads — ran
        // 2^19 buckets as 2 waves of K = 8 where one wave of K = 16 does the same work in 2/3 of the time.)
        const uint32_t slots = (uint32_t)ctx->sm_count * 2;
        double best = 1e300;
        uint32_t best_k = 3;
        for (uint32_t k_log = 2; k_log <= 8 && k_log <= cfg.nb_log; k_log++) {
            const uint64_t ctas = (((uint64_t)TB >> k_log) + 127) / 128;
            const uint64_t waves = (ctas + slots - 1) / slots;
            const double cost = (double)waves * (2.0 * (double)(1u << k_log) + 22.0);
            if (cost < best) { best = cost; best_k = k_log; }
        }
        if (const char *v = getenv("PB200_MSM_REDUCE_K_LOG")) best_k = std::min<uint32_t>((uint32_t)atoi(v), cfg.nb_log);  // tests / tuning
        cfg.K_log = best_k;
    }
    const uint32_t n_chunks = TB >> cfg.K_log, chunks_per_window = n_chunks / n_win;

    // level bounds
    std::vector<uint32_t> lvl_threads, lvl_slots;
    lvl_threads.push_back((uint32_t)((m0 + cfg.L1 - 1) / cfg.L1));
    lvl_slots.push_back(2 * lvl_threads[0]);
    while (lvl_slots.back() > 32) {
        uint32_t thr = (lvl_slots.back() + cfg.L2 - 1) / cfg.L2;
        lvl_threads.push_back(thr);
        lvl_slots.push_back(2 * thr);
    }
    const uint32_t n_scan_blocks = (TB + kScanTile - 1) / kScanTile;

    // workspace carve-up
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_count = carve((size_t)TB * 4), o_cursor = carve((size_t)TB * 4), o_bsum = carve((size_t)n_scan_blocks * 4);
    const size_t o_meta = carve(64 * 4);
    const size_t o_entries = carve((size_t)m0 * 8);
    // two-level scatter once the entry list outgrows L2: coarse bins of ~32 Ki entries, never crossing a window
    uint32_t coarse_shift = 0;
    size_t two_level_min = (size_t)1 << 30;
    if (const char *v = getenv("PB200_MSM_TWO_LEVEL_MIN_BYTES")) two_level_min = (size_t)atoll(v);  // tests force the path at small sizes
    if (m0 * 8 > two_level_min) {
        const double per_bucket = std::max(1.0, (double)m0 / (double)TB);
        while (coarse_shift < cfg.nb_log && per_bucket * (double)(2u << coarse_shift) <= 32768.0) coarse_shift++;
    }
    const uint32_t n_coarse = coarse_shift ? (TB >> coarse_shift) : 0;
    const size_t o_grouped = carve(coarse_shift ? (size_t)m0 * 8 : 0), o_coarse = carve((size_t)n_coarse * 4);
    const size_t o_buckets = carve((size_t)TB * sizeof(G1Xyzz));
    const size_t slotsA = lvl_slots[0], slotsB = lvl_slots.size() > 1 ? lvl_slots[1] : 2;
    const size_t o_gbA = carve(slotsA * 4), o_ptA = carve(slotsA * sizeof(G1Xyzz));
    const size_t o_gbB = carve(slotsB * 4), o_ptB = carve(slotsB * sizeof(G1Xyzz));
    const size_t o_chunks = carve((size_t)n_chunks * sizeof(G1Xyzz)), o_wsum = carve((size_t)n_win * sizeof(G1Xyzz));
    // two-stage window sum when a window has many chunk sums: ≤ 4 items per thread in the first stage
    const uint32_t sum_parts = std::min<uint32_t>(256, (chunks_per_window + 511) / 512);
    const size_t o_psum = carve((size_t)n_win * sum_parts * sizeof(G1Xyzz));
    PB_TRY(pb_ensure(ctx, &ctx->msm_ws, &ctx->msm_ws_bytes, off));
    char *ws = (char *)ctx->msm_ws;
    uint32_t *count = (uint32_t *)(ws + o_count), *cursor = (uint32_t *)(ws + o_cursor), *bsum = (uint32_t *)(ws + o_bsum);
    uint32_t *meta = (uint32_t *)(ws + o_meta);  // [0] = #entries, [1+k] = #slots produced by level k
    uint2 *entries = (uint2 *)(ws + o_entries), *grouped = (uint2 *)(ws + o_grouped);
    uint32_t *coarse = (uint32_t *)(ws + o_coarse);
    G1Xyzz *buckets = (G1Xyzz *)(ws + o_buckets);
    uint32_t *gbA = (uint32_t *)(ws + o_gbA), *gbB = (uint32_t *)(ws + o_gbB);
    G1Xyzz *ptA = (G1Xyzz *)(ws + o_ptA), *ptB = (G1Xyzz *)(ws + o_ptB);
    G1Xyzz *chunks = (G1Xyzz *)(ws + o_chunks), *wsum = (G1Xyzz *)(ws + o_wsum), *psum = (G1Xyzz *)(ws + o_psum);
    cudaStream_t st = ctx->stream;

    PbTimer t_sort(ctx, "msm.sort");
    PB_CUDA(ctx, cudaMemsetAsync(count, 0, (size_t)TB * 4, st));
    const uint32_t sgrid = std::min<uint32_t>((n + 255) / 256, ctx->sm_count * 16);
    msm_count_kernel<<<dim3(sgrid, batch), 256, 0, st>>>(scalars, cfg, count);
    PB_LAUNCHED(ctx);
    scan_block_sums_kernel<<<n_scan_blocks, kScanThreads, 0, st>>>(count, TB, bsum);
    PB_LAUNCHED(ctx);
    scan_top_kernel<<<1, kScanThreads, 0, st>>>(bsum, n_scan_blocks, meta + 0);
    PB_LAUNCHED(ctx);
    scan_apply_kernel<<<n_scan_blocks, kScanThreads, 0, st>>>(count, TB, bsum, cursor);
    PB_LAUNCHED(ctx);
    if (coarse_shift) {
        msm_coarse_init_kernel<<<(n_coarse + 255) / 256, 256, 0, st>>>(cursor, coarse, n_coarse, coarse_shift);
        PB_LAUNCHED(ctx);
        msm_scatter_kernel<<<dim3(sgrid, batch), 256, 0, st>>>(scalars, cfg, coarse, grouped, coarse_shift);
        PB_LAUNCHED(ctx);
        msm_fine_scatter_kernel<<<(uint32_t)((m0 + 255) / 256), 256, 0, st>>>(grouped, meta + 0, cursor, entries);
    } else {
        msm_scatter_kernel<<<dim3(sgrid, batch), 256, 0, st>>>(scalars, cfg, cursor, entries, 0);
    }
    PB_LAUNCHED(ctx);
    t_sort.stop();

    PbTimer t_acc(ctx, "msm.accumulate");
    // 168 registers let three CTAs share an SM; two measured faster (profiles/pipe_model_experiments_r02.txt §5), and the grid is
    // sized in whole waves of two: 80 KiB of (unused) dynamic shared memory per CTA keeps it at two.  PB200_MSM_ACC_CTAS=3 lifts it.
    static const bool acc_three = getenv("PB200_MSM_ACC_CTAS") && atoi(getenv("PB200_MSM_ACC_CTAS")) == 3;
    const size_t acc_smem = acc_three ? 0 : 80 * 1024;
    static bool acc_attr = false;
    if (!acc_attr) {
        PB_CUDA(ctx, cudaFuncSetAttribute(msm_accumulate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
        acc_attr = true;
    }
    msm_accumulate_kernel<<<(lvl_threads[0] + 127) / 128, 128, acc_smem, st>>>(bases, entries, meta + 0, cfg.L1, buckets, gbA, ptA, meta + 1);
    PB_LAUNCHED(ctx);
    t_acc.stop();
    PbTimer t_fix(ctx, "msm.partials");
    {
        uint32_t *in_gb = gbA, *out_gb = gbB;
        G1Xyzz *in_pt = ptA, *out_pt = ptB;
        for (size_t k = 1; k < lvl_threads.size(); k++) {
            PB_TRY(tail_accumulate_slots(ctx, lvl_threads[k], in_gb, in_pt, meta + k, cfg.L2, buckets, out_gb, out_pt, meta + k + 1));
            std::swap(in_gb, out_gb);
            std::swap(in_pt, out_pt);
        }
        // whatever is left (≤ 32 slots) is finished by one thread: no neighbours, so every run is complete
        PB_TRY(tail_accumulate_slots(ctx, 1, in_gb, in_pt, meta + lvl_threads.size(), 0x7fffffffu, buckets, out_gb, out_pt,
                                     meta + lvl_threads.size() + 1));
    }
    t_fix.stop();

    PbTimer t_red(ctx, "msm.reduce");
    MsmCfg rcfg = cfg;
    rcfg.W = n_win;
    PB_TRY(tail_reduce_chunks(ctx, n_chunks, buckets, count, rcfg, chunks));
    if (sum_parts > 1) {
        PB_TRY(tail_sum(ctx, n_win, sum_parts, chunks, chunks_per_window, psum));
        PB_TRY(tail_sum(ctx, n_win, 1, psum, sum_parts, wsum));
    } else {
        PB_TRY(tail_sum(ctx, n_win, 1, chunks, chunks_per_window, wsum));
    }
    if (batch > 1 || (pre_stride && running_total == nullptr)) PB_TRY(tail_batch_results(ctx, wsum, batch, result_dev));
    else PB_TRY(tail_combine(ctx, wsum, rcfg, running_total, first, last, result_dev));
    t_red.stop();
    if (ctx->profile) {
        PB_CUDA(ctx, cudaStreamSynchronize(st));
        t_sort.collect();
        t_acc.collect();
        t_fix.collect();
        t_red.collect();
    }
    return 0;
}

static int msm_run(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, const uint64_t *scalars_dev, size_t n, uint64_t *out_host,
                   uint32_t batch = 1, size_t scalar_stride = 0) {
    if (batch > 1) {
        // one pass over the shared bases when the pre-doubled copies are usable, otherwise one MSM after the other
        const bool pre_ok = srs != nullptr && srs->pre != nullptr && n * 16 >= srs->n && (uint64_t)srs->W_pre * srs->n < (1ull << 31) &&
                            (uint64_t)n * srs->W_pre * batch < (1ull << 32) && n <= ((size_t)1 << 26) && n > 0;
        if (!pre_ok) {
            for (uint32_t j = 0; j < batch; j++) PB_TRY(msm_run(ctx, srs, offset, scalars_dev + 4 * j * scalar_stride, n, out_host + 18 * j));
            return 0;
        }
        PB_ARG(ctx, offset <= srs->n && n <= srs->n - offset && scalars_dev != nullptr && batch <= 64);
        PB_CUDA(ctx, cudaSetDevice(ctx->device));
        const G1Affine *bases = reinterpret_cast<const G1Affine *>(srs->pre) + offset;
        void *small = nullptr;
        PB_CUDA(ctx, cudaMallocAsync(&small, (size_t)batch * 36 * 4, ctx->stream));
        PbTimer t_total(ctx, "msm.total");
        int rc = msm_piece(ctx, bases, scalars_dev, (uint32_t)n, 1, 1, nullptr, (uint32_t *)small, srs->c_pre, (uint32_t)srs->n, batch,
                           (uint32_t)scalar_stride);
        t_total.stop();
        cudaError_t e = cudaSuccess;
        if (rc == 0) e = cudaMemcpyAsync(ctx->pinned, small, (size_t)batch * 36 * 4, cudaMemcpyDeviceToHost, ctx->stream);
        cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
        cudaFreeAsync(small, ctx->stream);
        if (rc) return rc;
        if (e != cudaSuccess || e2 != cudaSuccess)
            return pb_fail(ctx, PB200_ERR_CUDA, "batched msm", cudaGetErrorString(e != cudaSuccess ? e : e2), __FILE__, __LINE__);
        t_total.collect();
        memcpy(out_host, ctx->pinned, (size_t)batch * 36 * 4);
        return 0;
    }
    // identity for the empty sum
    if (n == 0) {
        memset(out_host, 0, 18 * 8);
        const uint64_t r1[6] = {0x760900000002fffdull, 0xebf4000bc40c0002ull, 0x5f48985753c758baull,
                                0x77ce585370525745ull, 0x5c071a97a256ec6dull, 0x15f65ec3fa80e493ull};
        memcpy(out_host + 6, r1, 48);
        return 0;
    }
    PB_ARG(ctx, srs != nullptr && srs->dev != nullptr);
    PB_ARG(ctx, offset <= srs->n && n <= srs->n - offset);
    PB_ARG(ctx, scalars_dev != nullptr);
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    const G1Affine *bases = reinterpret_cast<const G1Affine *>(srs->dev) + offset;
    // pre-doubled copies pay off unless the call touches a small fraction of the SRS (the bucket count is sized for it)
    const bool use_pre = srs->pre != nullptr && n * 16 >= srs->n && (uint64_t)srs->W_pre * srs->n < (1ull << 31);
    if (use_pre) bases = reinterpret_cast<const G1Affine *>(srs->pre) + offset;
    void *small = nullptr;  // running total (XYZZ) + result (36 words)
    PB_CUDA(ctx, cudaMallocAsync(&small, sizeof(G1Xyzz) + 36 * 4, ctx->stream));
    G1Xyzz *running = (G1Xyzz *)small;
    uint32_t *result = (uint32_t *)((char *)small + sizeof(G1Xyzz));
    PbTimer t_total(ctx, "msm.total");
    const size_t piece = (size_t)1 << 26;
    int rc = 0;
    for (size_t done = 0; done < n && rc == 0; done += piece) {
        const uint32_t m = (uint32_t)std::min(piece, n - done);
        rc = msm_piece(ctx, bases + done, scalars_dev + 4 * done, m, done == 0, done + m == n, running, result,
                       use_pre ? srs->c_pre : 0, use_pre ? (uint32_t)srs->n : 0);
    }
    t_total.stop();
    cudaError_t e = cudaSuccess;
    if (rc == 0) e = cudaMemcpyAsync(ctx->pinned, result, 36 * 4, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    cudaFreeAsync(small, ctx->stream);
    if (rc) return rc;
    if (e != cudaSuccess) return pb_fail(ctx, PB200_ERR_CUDA, "msm result copy", cudaGetErrorString(e), __FILE__, __LINE__);
    if (e2 != cudaSuccess) return pb_fail(ctx, PB200_ERR_CUDA, "msm sync", cudaGetErrorString(e2), __FILE__, __LINE__);
    t_total.collect();
    memcpy(out_host, ctx->pinned, 36 * 4);
    return 0;
}

// Batched MSM over pre-doubled bases whose `batch` results (36 words each: projective X ‖ Y ‖ Z) stay in device memory, stream-
// ordered, no host synchronisation — for the sharded prover, which all-gathers and adds the ranks' partial sums on the device
// before anything returns to the host.  *handled = false (and nothing launched) when the pre-doubled path does not apply.
int msm_batch_to_dev(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, const uint64_t *scalars_dev, size_t n, uint32_t batch,
                     size_t scalar_stride, uint32_t *result_dev, bool *handled) {
    *handled = false;
    const bool pre_ok = srs != nullptr && srs->pre != nullptr && n > 0 && n * 16 >= srs->n && (uint64_t)srs->W_pre * srs->n < (1ull << 31) &&
                        (uint64_t)n * srs->W_pre * batch < (1ull << 32) && n <= ((size_t)1 << 26) && batch >= 1 && batch <= 64 &&
                        offset <= srs->n && n <= srs->n - offset && (batch == 1 || scalar_stride >= n);
    if (!pre_ok) return 0;
    *handled = true;
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    const G1Affine *bases = reinterpret_cast<const G1Affine *>(srs->pre) + offset;
    return msm_piece(ctx, bases, scalars_dev, (uint32_t)n, 1, 1, nullptr, result_dev, srs->c_pre, (uint32_t)srs->n, batch, (uint32_t)scalar_stride);
}

extern "C" int pb200_srs_upload(pb200_ctx *ctx, const uint64_t *xy_mont_host, size_t n_points, pb200_srs **out) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, out != nullptr && (xy_mont_host != nullptr || n_points == 0));
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    void *dev = nullptr;
    PB_CUDA(ctx, cudaMalloc(&dev, std::max<size_t>(n_points, 1) * 96));
    if (n_points) {
        cudaError_t e = cudaMemcpyAsync(dev, xy_mont_host, n_points * 96, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) {
            cudaFree(dev);
            return pb_fail(ctx, PB200_ERR_CUDA, "srs upload", cudaGetErrorString(e), __FILE__, __LINE__);
        }
    }
    pb200_srs *s = new pb200_srs();
    s->dev = (const uint64_t *)dev;
    s->n = n_points;
    s->owned = true;
    *out = s;
    return 0;
}
extern "C" int pb200_srs_wrap_dev(pb200_ctx *ctx, const uint64_t *xy_mont_dev, size_t n_points, pb200_srs **out) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, out != nullptr && xy_mont_dev != nullptr);
    pb200_srs *s = new pb200_srs();
    s->dev = xy_mont_dev;
    s->n = n_points;
    s->owned = false;
    *out = s;
    return 0;
}
extern "C" int pb200_srs_precompute(pb200_ctx *ctx, pb200_srs *srs) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, srs != nullptr && srs->dev != nullptr);
    PB_ARG(ctx, srs->n >= 1 && srs->n <= ((size_t)1 << 22));
    if (srs->pre) return 0;
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t c = choose_window_pre(srs->n), W = (256 + c - 1) / c;
    void *pre = nullptr;
    PB_CUDA(ctx, cudaMalloc(&pre, (size_t)W * srs->n * sizeof(G1Affine)));
    int rc = tail_precompute(ctx, reinterpret_cast<const G1Affine *>(srs->dev), (uint32_t)srs->n, c, W, (G1Affine *)pre);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (rc != 0 || e != cudaSuccess) {
        cudaFree(pre);
        return rc ? rc : pb_fail(ctx, PB200_ERR_CUDA, "srs precompute", cudaGetErrorString(e), __FILE__, __LINE__);
    }
    srs->pre = pre;
    srs->c_pre = c;
    srs->W_pre = W;
    return 0;
}
extern "C" void pb200_srs_free(pb200_ctx *ctx, pb200_srs *srs) {
    if (!srs) return;
    if (srs->pre) {
        if (ctx) cudaStreamSynchronize(ctx->stream);
        cudaFree(srs->pre);
    }
    if (srs->owned && srs->dev) {
        if (ctx) cudaStreamSynchronize(ctx->stream);
        cudaFree((void *)srs->dev);
    }
    delete srs;
}
extern "C" size_t pb200_srs_len(const pb200_srs *srs) { return srs ? srs->n : 0; }
extern "C" uint32_t pb200_msm_window_bits(size_t n) { return choose_window(std::min<size_t>(n, (size_t)1 << 26)); }

extern "C" int pb200_msm_g1_dev(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, const uint64_t *scalars_mont_dev, size_t n,
                                uint64_t out_xyz_mont[18]) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, out_xyz_mont != nullptr);
    return msm_run(ctx, srs, offset, scalars_mont_dev, n, out_xyz_mont);
}
extern "C" int pb200_msm_g1_batch_dev(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, const uint64_t *scalars_mont_dev, size_t n,
                                      uint32_t batch, size_t scalar_stride, uint64_t *out_xyz_mont) {
    if (!ctx || !out_xyz_mont) return PB200_ERR_ARG;
    PB_ARG(ctx, batch >= 1 && batch <= 64 && (batch == 1 || scalar_stride >= n) && scalar_stride < ((size_t)1 << 32));
    return msm_run(ctx, srs, offset, scalars_mont_dev, n, out_xyz_mont, batch, scalar_stride);
}
extern "C" int pb200_msm_g1(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, const uint64_t *scalars_mont_host, size_t n,
                            uint64_t out_xyz_mont[18]) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, out_xyz_mont != nullptr);
    if (n == 0) return msm_run(ctx, srs, offset, nullptr, 0, out_xyz_mont);
    PB_ARG(ctx, scalars_mont_host != nullptr);
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    PB_TRY(pb_ensure(ctx, &ctx->stage, &ctx->stage_bytes, n * 32));
    PB_CUDA(ctx, cudaMemcpyAsync(ctx->stage, scalars_mont_host, n * 32, cudaMemcpyHostToDevice, ctx->stream));
    return msm_run(ctx, srs, offset, (const uint64_t *)ctx->stage, n, out_xyz_mont);
}
// multiscalar_mul::pippenger(points: Iterator<G1Projective>, scalars: Iterator<Scalar>): the bases arrive in projective
// coordinates; they are normalised on the device (one inversion per eight points) and summed by the same pipeline.
extern "C" int pb200_pippenger_g1(pb200_ctx *ctx, const uint64_t *points_xyz_mont_host, const uint64_t *scalars_mont_host, size_t n,
                                  uint64_t out_xyz_mont[18]) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, out_xyz_mont != nullptr);
    if (n == 0) return msm_run(ctx, nullptr, 0, nullptr, 0, out_xyz_mont);
    PB_ARG(ctx, points_xyz_mont_host != nullptr && scalars_mont_host != nullptr && n < ((size_t)1 << 32));
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    void *dev = nullptr;   // [n × 144 B projective][n × 32 B scalars in][n × 96 B affine][n × 32 B scalars out]
    PB_CUDA(ctx, cudaMalloc(&dev, n * (144 + 32 + 96 + 32)));
    uint8_t *base = (uint8_t *)dev;
    uint32_t *xyz = (uint32_t *)base;
    uint64_t *sc_in = (uint64_t *)(base + n * 144), *sc_out = (uint64_t *)(base + n * (144 + 32 + 96));
    G1Affine *aff = (G1Affine *)(base + n * (144 + 32));
    int rc = 0;
    cudaError_t e = cudaMemcpyAsync(xyz, points_xyz_mont_host, n * 144, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(sc_in, scalars_mont_host, n * 32, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) rc = tail_g1_normalize(ctx, xyz, sc_in, n, aff, sc_out);
    if (e == cudaSuccess && rc == 0) {
        pb200_srs tmp;
        tmp.dev = (const uint64_t *)aff;
        tmp.n = n;
        rc = msm_run(ctx, &tmp, 0, sc_out, n, out_xyz_mont);
    }
    cudaStreamSynchronize(ctx->stream);
    cudaFree(dev);
    if (e != cudaSuccess) return pb_fail(ctx, PB200_ERR_CUDA, "pippenger", cudaGetErrorString(e), __FILE__, __LINE__);
    return rc;
}
extern "C" int pb200_g1_sum(pb200_ctx *ctx, const uint64_t *points_xyz_mont_host, size_t count, uint64_t out_xyz_mont[18]) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, out_xyz_mont != nullptr && (points_xyz_mont_host != nullptr || count == 0) && count <= 4096);
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    void *dev = nullptr;
    PB_CUDA(ctx, cudaMallocAsync(&dev, (count + 1) * 144, ctx->stream));
    uint32_t *pts = (uint32_t *)dev, *res = pts + 36 * count;
    cudaError_t e = cudaSuccess;
    if (count) e = cudaMemcpyAsync(pts, points_xyz_mont_host, count * 144, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && tail_g1_sum(ctx, pts, (uint32_t)count, res) != 0) e = cudaErrorLaunchFailure;
    if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->pinned, res, 144, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    cudaFreeAsync(dev, ctx->stream);
    if (e != cudaSuccess) return pb_fail(ctx, PB200_ERR_CUDA, "g1_sum", cudaGetErrorString(e), __FILE__, __LINE__);
    if (e2 != cudaSuccess) return pb_fail(ctx, PB200_ERR_CUDA, "g1_sum sync", cudaGetErrorString(e2), __FILE__, __LINE__);
    memcpy(out_xyz_mont, ctx->pinned, 144);
    return 0;
}
extern "C" int pb200_synthetic_bases_dev(pb200_ctx *ctx, uint64_t *xy_mont_dev, size_t n, uint64_t a, uint64_t d) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, xy_mont_dev != nullptr || n == 0);
    if (n == 0) return 0;
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    PB_TRY(tail_synthetic_bases(ctx, (G1Affine *)xy_mont_dev, n, a, d));
    PB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
