// ntt_tma.cuh — the TMA-staged NTT pass kernel (included by ntt.cu).
//
// Same transform as ntt_pass_kernel (one pass of the four-step decomposition, DESIGN.md §4.2), re-laid for Blackwell's
// copy engine and 128-bit shared-memory accesses:
//   * tiles are 2^S points × 4 columns; shared memory holds them element-major, one 128-byte row per x (4 scalars of
//     32 B), with the 16-byte chunks of a row XOR-swizzled by (x mod 8) — exactly CU_TENSOR_MAP_SWIZZLE_128B, so the tile
//     of a strided pass is loaded by ONE cp.async.bulk.tensor.2d (UTMALDG) per 256 rows and every tile is written back
//     by cp.async.bulk.tensor.2d stores (UTMASTG): no LDG/STG and no address arithmetic in the instruction stream;
//   * every butterfly round reads / writes a scalar as two LDS.128 / STS.128 (the planar layout of the first kernel
//     needed eight 32-bit accesses); with the swizzle a quarter-warp's eight 16-byte accesses fall into eight different
//     bank groups in the staging loop, every round with b_lo ≥ 1 and the final write-back (only the last round's load is 2-way);
//   * the butterfly twiddles of all rounds are staged into shared memory by one cp.async.bulk (UBLKCP) from a compact
//     per-round image built with the plan, so the rounds issue no global loads at all;
//   * between the passes of a transform the scalars stay in the lazy range [0, 2r) (field.cuh): sums and differences are taken
//     mod 2r and the product by a canonical twiddle needs no final subtraction — 17 instructions fewer per multiplication on a
//     kernel bound by dispatch slots; the last pass stores canonical values;
//   * the bit reversal and the inter-pass twiddle / coset factor are applied in registers after the last round, the
//     results go to shared memory at their output row, and one elected thread issues the tensor store.
// Used for transforms of 2^12 … 2^26 points (two passes up to 2^18, three above; S ∈ 6…9) whose plan has single-lookup tables;
// everything else (2^27 and up, plans built after the table budget ran out), and the peer-store variant of the sharded
// transform, stays on ntt_pass_kernel.
#pragma once
// (ntt.cu includes <cuda.h> and defines Fr, g_load, g_store, bfly, bfly1 before including this file inside its namespace)

namespace tma {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a transfer that never completes (bad descriptor) traps instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    for (uint32_t spin = 0; !mbar_try_wait(bar, parity); spin++)
        if (spin > (1u << 24)) __trap();
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
                 "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tensor_g2s_2d(uint32_t dst, const CUtensorMap *map, uint32_t c0, uint32_t c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tensor_s2g_2d(const CUtensorMap *map, uint32_t src, uint32_t c0, uint32_t c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
                 "r"(src), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4 &v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// Read-only global load the compiler must leave where it is written (volatile): used to issue table loads a whole
// multiplication ahead of their use — plain C++ loads were scheduled right in front of the consuming multiply, and the ncu
// of the first version showed the full L2 / DRAM latency of each of the eight inter-pass twiddles as long-scoreboard stall.
__device__ __forceinline__ Fr ldg_fr_pinned(const Fr *p) {
    Fr r;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.l[0]), "=r"(r.l[1]), "=r"(r.l[2]), "=r"(r.l[3]) : "l"(p));
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4+16];" : "=r"(r.l[4]), "=r"(r.l[5]), "=r"(r.l[6]), "=r"(r.l[7]) : "l"(p));
    return r;
}
// byte offset of the low half of scalar (x, c) inside the tile; the high half is at offset ^ 16
__device__ __forceinline__ uint32_t tile_off(uint32_t x, uint32_t c) { return (x << 7) + ((((c << 1)) ^ (x & 7u)) << 4); }
__device__ __forceinline__ Fr lds_fr(uint32_t addr) {
    const uint4 a = lds128(addr), b = lds128(addr ^ 16u);
    Fr r;
    r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
    r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
    return r;
}
__device__ __forceinline__ void sts_fr(uint32_t addr, const Fr &v) {
    sts128(addr, make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]));
    sts128(addr ^ 16u, make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]));
}

// Butterflies on the lazy representation [0, 2r) (field.cuh): the product by the canonical twiddle needs no final subtraction.
__device__ __forceinline__ void bfly_lz(Fr &a, Fr &b, const Fr &w) {
    const Fr s = Fr::add_lazy(a, b), d = Fr::sub_lazy(a, b);
    a = s;
    b = Fr::mul_lazy(w, d);
}
__device__ __forceinline__ void bfly1_lz(Fr &a, Fr &b) {
    const Fr s = Fr::add_lazy(a, b);
    b = Fr::sub_lazy(a, b);
    a = s;
}

}  // namespace tma

struct NttPassTma {
    uint32_t S;           // log2 of the sub-transform length, 6 … 9
    uint32_t type;        // 0: strided sub-transform (columns contiguous) | 1: contiguous rows, output transposed
    uint32_t ncol_log;    // type 0: log2(columns per row block)
    uint32_t nrows_log;   // type 1: log2(number of rows) = log n − S
    uint32_t n1_log;      // type 1: log2 of the first-pass length (row ↔ natural-index digit swap of the 3-pass plan)
    uint32_t load_mode;   // 0 none | 2 × l_full[natural input index]                           (type 0, coset_fft)
    uint32_t store_mode;  // 0 none | 4 × s_full[(k << ncol_log) + col] (type 0) | 5 × s_full[natural output index] (type 1)
    uint32_t batch_log;   // vectors of a batch are 2^batch_log scalars apart (blockIdx.y)
    uint32_t last;        // last pass of the transform: results leave in canonical form (between passes they stay in [0, 2r))
    uint32_t tw_bytes;    // size of the twiddle image
    const Fr *tw_img;     // per-round compact butterfly twiddles (ntt_tw_image_kernel)
    const Fr *l_full, *s_full;
};

// Twiddle image of a 2^S-point sub-transform: for every radix-8 round on bits [b_lo, b_lo+2], from the top down,
//   [(e << b_lo) + v]            e < 4 : ω^(((e << b_lo) | v) << (S−3−b_lo))      first stage
//   [(4 << b_lo) + (e << b_lo) + v] e < 2 : ω^(((e << b_lo) | v) << (S−2−b_lo))   second stage
//   [(6 << b_lo) + v]                  : ω^(v << (S−1−b_lo))                      third stage
// (v < 2^b_lo), then ω₈, ω₈², ω₈³ for the last round.  tw[j] = ω_{2^S}^j, j < 2^(S−1).
__host__ __device__ inline uint32_t ntt_tw_image_entries(uint32_t S) {
    uint32_t n = 3;
    for (int b_top = (int)S - 1; b_top >= 3; b_top -= 3) n += 7u << (b_top - 2);
    return n;
}
__global__ void ntt_tw_image_kernel(Fr *img, const Fr *tw, uint32_t S) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t off = 0;
    for (int b_top = (int)S - 1; b_top >= 3; b_top -= 3) {
        const uint32_t b_lo = (uint32_t)b_top - 2, cnt = 7u << b_lo;
        if (i < off + cnt) {
            const uint32_t j = i - off, blk = j >> b_lo, v = j & ((1u << b_lo) - 1);
            uint32_t src;
            if (blk < 4) src = ((blk << b_lo) | v) << (S - 3 - b_lo);
            else if (blk < 6) src = (((blk - 4) << b_lo) | v) << (S - 2 - b_lo);
            else src = v << (S - 1 - b_lo);
            g_store(img + i, g_load(tw + src));
            return;
        }
        off += cnt;
    }
    if (i < off + 3) g_store(img + i, g_load(tw + ((i - off + 1) << (S - 3))));
}

// One pass.  blockDim.x = 2^(S−1) threads, 8 points per thread per round; dynamic shared memory: 1 KiB alignment slack,
// the tile (2^(S+7) bytes), the twiddle image, one mbarrier.
template <int S, int THREADS_PER_SM>
__global__ void __launch_bounds__(1 << (S - 1), THREADS_PER_SM >> (S - 1))
ntt_pass_tma_kernel(const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_out, const Fr *__restrict__ in,
                    const NttPassTma p) {
    extern __shared__ uint8_t smem_raw[];
    constexpr uint32_t T = 1u << (S + 2), TILE_BYTES = T * 32u, NTHR = 1u << (S - 1);
    constexpr uint32_t BOX_ROWS = S > 8 ? 256u : (1u << S), N_BOX = (1u << S) / BOX_ROWS;
    const uint32_t tile = (tma::smem_u32(smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B atoms are 1 KiB
    const uint32_t twb = tile + TILE_BYTES;
    const uint32_t bar = twb + ((p.tw_bytes + 15u) & ~15u);
    const uint32_t tid = threadIdx.x, c = tid & 3u, tx = tid >> 2;
    const uint32_t b = blockIdx.y;

    uint32_t col0 = 0, row_base = 0, rowrev0 = 0;
    uint64_t in_base = 0;   // type 0: element index of tile point (x = 0, c = 0) inside this vector
    if (p.type == 0) {
        const uint32_t bpr_log = p.ncol_log - 2;
        const uint32_t R = blockIdx.x >> bpr_log;
        col0 = (blockIdx.x & ((1u << bpr_log) - 1)) << 2;
        in_base = ((uint64_t)R << (S + p.ncol_log)) + col0;
        row_base = (b << (p.batch_log - p.ncol_log)) + (R << S);   // row of the [rows][2^ncol_log] view of the whole batch
    } else {
        rowrev0 = blockIdx.x << 2;
    }
    if (tid == 0) {
        tma::mbar_init(bar, 1);
        tma::fence_mbar_init();
    }
    __syncthreads();
    if (tid == 0) {
        tma::mbar_expect_tx(bar, p.tw_bytes + (p.type == 0 ? TILE_BYTES : 0u));
        tma::bulk_g2s(twb, p.tw_img, p.tw_bytes, bar);
        if (p.type == 0) {
#pragma unroll
            for (uint32_t k = 0; k < N_BOX; k++)
                tma::tensor_g2s_2d(tile + k * BOX_ROWS * 128u, &map_in, col0 * 4u, row_base + k * BOX_ROWS, bar);
        }
    }
    if (p.type == 1) {
        // rows are contiguous in global memory but the tile is point-major: stage through registers (coalesced 128-bit loads)
        const Fr *src = in + ((uint64_t)b << p.batch_log);
        const uint32_t n2_log = p.nrows_log - p.n1_log;
#pragma unroll
        for (uint32_t i = tid; i < T; i += NTHR) {   // T / NTHR = 8 iterations, fully unrolled: sixteen 128-bit loads in flight
            const uint32_t x = i & ((1u << S) - 1), cc = i >> S;
            const uint32_t rr = rowrev0 + cc;
            const uint32_t row = ((rr & ((1u << p.n1_log) - 1)) << n2_log) + (rr >> p.n1_log);
            tma::sts_fr(tile + tma::tile_off(x, cc), g_load(src + (((uint64_t)row << S) + x)));
        }
    }
    // The last round's thread ↔ row assignment is bit-reversed (rows (brev(tx) << 3) | e), so that the output rows k a
    // quarter-warp writes differ in their LOW bits and the write-back to the tile is bank-conflict free (ncu, first version:
    // 25 % of the shared wavefronts were conflicts, half of them from that store).  k = brev_S(x) = (brev3(e) << (S−3)) | tx.
    const uint32_t tx_rev = __brev(tx) >> (32 - (S - 3));
    if (p.store_mode) {
        // the inter-pass twiddles / coset factors this thread multiplies by at the very end come from a table as long as the
        // vector (DRAM): start pulling them towards L2 now, the butterflies hide the latency
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const uint32_t e_rev = ((e & 1) << 2) | (e & 2) | ((e >> 2) & 1);
            const uint32_t k = (e_rev << (S - 3)) | tx;
            const uint64_t idx = p.store_mode == 4 ? (((uint64_t)k << p.ncol_log) + col0 + c) : ((uint64_t)(rowrev0 + c) + ((uint64_t)k << p.nrows_log));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(p.s_full + idx));
        }
    }
    tma::mbar_wait(bar, 0);
    __syncthreads();
    if (p.load_mode == 2) {   // coset_fft: a_j ← a_j·7^j on the way in (one multiplier instance, its own sweep over the tile)
        const Fr *lf = p.l_full + in_base;
        Fr f_next = tma::ldg_fr_pinned(lf + (((uint64_t)(tid >> 2) << p.ncol_log) + (tid & 3u)));
#pragma unroll 1
        for (uint32_t i = tid; i < T; i += NTHR) {
            const uint32_t x = i >> 2, cc = i & 3u;
            const uint32_t off = tile + tma::tile_off(x, cc);
            const Fr f = f_next;
            const uint32_t i2 = min(i + NTHR, T - 1);   // the factor of the next iteration travels during this multiply
            f_next = tma::ldg_fr_pinned(lf + (((uint64_t)(i2 >> 2) << p.ncol_log) + (i2 & 3u)));
            tma::sts_fr(off, Fr::mul_lazy(f, tma::lds_fr(off)));
        }
        __syncthreads();
    }

    Fr a[8];
    int b_top = S - 1;
    uint32_t tw_off = twb;
    while (b_top >= 3) {
        const uint32_t b_lo = (uint32_t)b_top - 2;
        const uint32_t v = tx & ((1u << b_lo) - 1), u = tx >> b_lo;
        const uint32_t xbase = (u << (b_lo + 3)) | v;
#pragma unroll
        for (int e = 0; e < 8; e++) a[e] = tma::lds_fr(tile + tma::tile_off(xbase | ((uint32_t)e << b_lo), c));
        {
#pragma unroll
            for (int e = 0; e < 4; e++) tma::bfly_lz(a[e], a[e + 4], tma::lds_fr(tw_off + ((((uint32_t)e << b_lo) + v) << 5)));
            const uint32_t s2 = tw_off + ((4u << b_lo) << 5);
#pragma unroll
            for (int e = 0; e < 2; e++) {
                const Fr w = tma::lds_fr(s2 + ((((uint32_t)e << b_lo) + v) << 5));
                tma::bfly_lz(a[e], a[e + 2], w);
                tma::bfly_lz(a[e + 4], a[e + 6], w);
            }
            const Fr w3 = tma::lds_fr(tw_off + (((6u << b_lo) + v) << 5));
#pragma unroll
            for (int e = 0; e < 8; e += 2) tma::bfly_lz(a[e], a[e + 1], w3);
        }
#pragma unroll
        for (int e = 0; e < 8; e++) tma::sts_fr(tile + tma::tile_off(xbase | ((uint32_t)e << b_lo), c), a[e]);
        __syncthreads();
        tw_off += (7u << b_lo) << 5;
        b_top -= 3;
    }
    // last round on bits [0, 2]: twiddles are ω₈^k
#pragma unroll
    for (int e = 0; e < 8; e++) a[e] = tma::lds_fr(tile + tma::tile_off((tx_rev << 3) | (uint32_t)e, c));
    __syncthreads();   // every thread has read its rows: they may now be overwritten with outputs of other rows
    // Output row of a[e] and the address of its inter-pass twiddle / coset factor.  The factors come from a table as long as
    // the vector (L2 at best, DRAM on the first pass): PF of them are always in flight — the first PF are requested here, before
    // the last round's butterflies, the others PF − 1 multiplications before their use.
    constexpr int PF = THREADS_PER_SM >= 512 ? 2 : 4;
    const uint32_t k_hi = tx;   // k = brev_S((tx_rev << 3) | e) = (brev3(e) << (S−3)) | brev_{S−3}(tx_rev) = … | tx
    auto out_row = [&](int e) -> uint32_t {
        const uint32_t e_rev = ((e & 1) << 2) | (e & 2) | ((e >> 2) & 1);
        return (e_rev << (S - 3)) | k_hi;
    };
    auto factor_at = [&](int e) -> const Fr * {   // 4: inter-pass twiddle full[(k << ncol_log) + col] | 5: coset factor full[natural output index]
        const uint32_t k = out_row(e);
        const uint64_t idx = p.store_mode == 4 ? (((uint64_t)k << p.ncol_log) + col0 + c)
                                               : ((uint64_t)(rowrev0 + c) + ((uint64_t)k << p.nrows_log));
        return p.s_full + idx;
    };
    constexpr bool EARLY = !(S == 6 && THREADS_PER_SM >= 512);   // (that one variant would spill four registers)
    Fr f[PF];
    if (EARLY && p.store_mode) {
#pragma unroll
        for (int e = 0; e < PF; e++) f[e] = tma::ldg_fr_pinned(factor_at(e));
    }
    if (b_top >= 2) {
        tma::bfly1_lz(a[0], a[4]);
#pragma unroll
        for (int e = 1; e < 4; e++) tma::bfly_lz(a[e], a[e + 4], tma::lds_fr(tw_off + ((uint32_t)(e - 1) << 5)));
    }
    if (b_top >= 1) {
        const Fr w4 = tma::lds_fr(tw_off + 32u);
        tma::bfly1_lz(a[0], a[2]);
        tma::bfly1_lz(a[4], a[6]);
        tma::bfly_lz(a[1], a[3], w4);
        tma::bfly_lz(a[5], a[7], w4);
    }
#pragma unroll
    for (int e = 0; e < 8; e += 2) tma::bfly1_lz(a[e], a[e + 1]);
    // bit reversal + factor in registers, then to the tile at the OUTPUT row k
    if (p.store_mode) {
        if (!EARLY) {
#pragma unroll
            for (int e = 0; e < PF; e++) f[e] = tma::ldg_fr_pinned(factor_at(e));
        }
#pragma unroll
        for (int e = 0; e < 8; e++) {
            Fr val = Fr::mul_lazy(f[e % PF], a[e]);
            if (e + PF < 8) f[e % PF] = tma::ldg_fr_pinned(factor_at(e + PF));
            if (p.last) val = val.canonical();
            tma::sts_fr(tile + tma::tile_off(out_row(e), c), val);
        }
    } else {
#pragma unroll
        for (int e = 0; e < 8; e++) tma::sts_fr(tile + tma::tile_off(out_row(e), c), p.last ? a[e].canonical() : a[e]);
    }
    tma::fence_proxy_async();   // generic-proxy writes above → visible to the async proxy (the tensor store)
    __syncthreads();
    if (tid == 0) {
#pragma unroll
        for (uint32_t k = 0; k < N_BOX; k++) {
            if (p.type == 0) tma::tensor_s2g_2d(&map_out, tile + k * BOX_ROWS * 128u, col0 * 4u, row_base + k * BOX_ROWS);
            else tma::tensor_s2g_2d(&map_out, tile + k * BOX_ROWS * 128u, rowrev0 * 4u, (b << S) + k * BOX_ROWS);
        }
        tma::bulk_commit();
        tma::bulk_wait_read0();   // shared memory must stay valid until the copy engine has read it
    }
}

// ---- host side: tensor maps (cuTensorMapEncodeTiled through the runtime's driver entry point: no -lcuda) ------------------
typedef CUresult (*PbEncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                    const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);
static PbEncodeTiledFn pb_encode_tiled() {
    static PbEncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (PbEncodeTiledFn)p;
    }
    return fn;
}
// A [rows][cols] matrix of 32-byte scalars seen as u64 elements; box = 4 scalars (128 B) × box_rows rows, SWIZZLE_128B.
static int pb_make_tile_map(pb200_ctx *ctx, CUtensorMap *map, const void *base, uint64_t cols, uint64_t rows, uint32_t box_rows) {
    PbEncodeTiledFn enc = pb_encode_tiled();
    if (!enc) return pb_fail(ctx, PB200_ERR_CUDA, "tensor map", "cuTensorMapEncodeTiled is not available from this driver", __FILE__, __LINE__);
    const cuuint64_t gdim[2] = {cols * 4, rows};
    const cuuint64_t gstride[1] = {cols * 32};
    const cuuint32_t box[2] = {16, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, const_cast<void *>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        char msg[64];
        snprintf(msg, sizeof(msg), "cuTensorMapEncodeTiled failed (%d)", (int)r);
        return pb_fail(ctx, PB200_ERR_CUDA, "tensor map", msg, __FILE__, __LINE__);
    }
    return 0;
}
