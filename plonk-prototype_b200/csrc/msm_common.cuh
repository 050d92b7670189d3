// msm_common.cuh — declarations shared by msm.cu (throughput kernels, multiplier inlined) and msm_tail.cu
// (latency-bound tail kernels, compiled with the shared non-inlined multiplier).
#pragma once
#include "common.cuh"
#include "g1.cuh"

constexpr uint32_t kInvalid = 0xffffffffu;
constexpr uint32_t kScanItems = 4, kScanThreads = 1024, kScanTile = kScanItems * kScanThreads;

struct MsmCfg {
    uint32_t n;       // points in this piece (< 2^27)
    uint32_t c;       // window bits
    uint32_t W;       // windows = ceil(256 / c)
    uint32_t nb_log;  // log2 buckets per window = c − 1
    uint32_t L1, L2;  // segment length at level 1 / higher levels
    uint32_t K_log;   // log2 buckets per reduction chunk
    uint32_t pre_stride;  // 0, or the SRS length when pre-doubled copies are used: window w reads base w·stride + i
                          // and every window shares the bucket set of window 0
    uint32_t batch;          // pre-doubled path only: number of scalar vectors summed over the same bases in one pass
                             // (blockIdx.y of the count / scatter kernels); vector j owns bucket set j
    uint32_t scalar_stride;  // distance between consecutive scalar vectors, in scalars
};

// ------------------------------------------------------------------------------------------ loads
__device__ __forceinline__ Fr load_fr(const uint64_t *scalars, size_t i) {
    const uint4 *q = reinterpret_cast<const uint4 *>(scalars + 4 * i);
    uint4 a = q[0], b = q[1];
    Fr r;
    r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
    r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
    return r;
}
__device__ __forceinline__ void load_fp2(const uint4 *q, Fp &a, Fp &b) {
    uint4 v0 = q[0], v1 = q[1], v2 = q[2], v3 = q[3], v4 = q[4], v5 = q[5];
    a.l[0] = v0.x; a.l[1] = v0.y; a.l[2] = v0.z; a.l[3] = v0.w; a.l[4] = v1.x; a.l[5] = v1.y;
    a.l[6] = v1.z; a.l[7] = v1.w; a.l[8] = v2.x; a.l[9] = v2.y; a.l[10] = v2.z; a.l[11] = v2.w;
    b.l[0] = v3.x; b.l[1] = v3.y; b.l[2] = v3.z; b.l[3] = v3.w; b.l[4] = v4.x; b.l[5] = v4.y;
    b.l[6] = v4.z; b.l[7] = v4.w; b.l[8] = v5.x; b.l[9] = v5.y; b.l[10] = v5.z; b.l[11] = v5.w;
}
__device__ __forceinline__ void store_fp2(uint4 *q, const Fp &a, const Fp &b) {
    q[0] = make_uint4(a.l[0], a.l[1], a.l[2], a.l[3]);
    q[1] = make_uint4(a.l[4], a.l[5], a.l[6], a.l[7]);
    q[2] = make_uint4(a.l[8], a.l[9], a.l[10], a.l[11]);
    q[3] = make_uint4(b.l[0], b.l[1], b.l[2], b.l[3]);
    q[4] = make_uint4(b.l[4], b.l[5], b.l[6], b.l[7]);
    q[5] = make_uint4(b.l[8], b.l[9], b.l[10], b.l[11]);
}
__device__ __forceinline__ G1Affine load_affine(const G1Affine *bases, uint32_t idx_sign) {
    G1Affine p;
    load_fp2(reinterpret_cast<const uint4 *>(bases + (idx_sign & 0x7fffffffu)), p.x, p.y);
    if (idx_sign >> 31) p.y = p.y.neg_nonzero();   // y ≠ 0 on the prime-order subgroup
    return p;
}
__device__ __forceinline__ G1Xyzz load_xyzz(const G1Xyzz *p) {
    G1Xyzz r;
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    load_fp2(q, r.x, r.y);
    load_fp2(q + 6, r.zz, r.zzz);
    return r;
}
__device__ __forceinline__ void store_xyzz(G1Xyzz *p, const G1Xyzz &v) {
    uint4 *q = reinterpret_cast<uint4 *>(p);
    store_fp2(q, v.x, v.y);
    store_fp2(q + 6, v.zz, v.zzz);
}


// ---- tail-kernel launchers (msm_tail.cu) ----------------------------------------------------------
int tail_accumulate_slots(pb200_ctx *ctx, uint32_t grid_threads, const uint32_t *in_gb, const G1Xyzz *in_pt, const uint32_t *n_in_ptr,
                          uint32_t L, G1Xyzz *buckets, uint32_t *out_gb, G1Xyzz *out_pt, uint32_t *n_out_ptr);
int tail_reduce_chunks(pb200_ctx *ctx, uint32_t n_chunks, const G1Xyzz *buckets, const uint32_t *count, MsmCfg cfg, G1Xyzz *chunk_sums);
int tail_sum(pb200_ctx *ctx, uint32_t groups, uint32_t parts, const G1Xyzz *in, uint32_t items_per_group, G1Xyzz *out);
int tail_combine(pb200_ctx *ctx, const G1Xyzz *window_sums, MsmCfg cfg, G1Xyzz *running_total, int first_piece, int last_piece,
                 uint32_t *result);
int tail_batch_results(pb200_ctx *ctx, const G1Xyzz *set_sums, uint32_t batch, uint32_t *results);
int tail_g1_sum(pb200_ctx *ctx, const uint32_t *pts, uint32_t count, uint32_t *result);
int tail_g1_sum_batch(pb200_ctx *ctx, const uint32_t *pts, uint32_t count, uint32_t batch, uint32_t *results);
int tail_g1_normalize(pb200_ctx *ctx, const uint32_t *xyz, const uint64_t *scalars_in, uint64_t n, G1Affine *out, uint64_t *scalars_out);
int tail_precompute(pb200_ctx *ctx, const G1Affine *bases, uint32_t n, uint32_t c, uint32_t W, G1Affine *pre);
int tail_synthetic_bases(pb200_ctx *ctx, G1Affine *out, uint64_t n, uint64_t a, uint64_t d);

// ---- checked compressed-point decoder (srs_io.cu): G1Affine::from_bytes, one thread per point, 128 threads per block
__global__ void g1_decompress_kernel(const uint4 *__restrict__ enc, uint32_t n, G1Affine *__restrict__ out, uint8_t *__restrict__ status,
                                     uint32_t *first_bad);

// ------------------------------------------------------------------------------------ accumulate
// Output rule shared by every level.  A run that lies strictly inside its segment is complete and
// goes to its bucket.  A run that touches the left (right) segment boundary *and* continues in the
// neighbouring segment is a partial: left-touching partials go to the head slot, right-touching
// ones to the tail slot; a run touching both sides stores its sum in the head slot and the identity
// in the tail slot, so all partials of one bucket stay contiguous in slot order (no holes inside).
struct RunSink {
    G1Xyzz *buckets;
    uint32_t *out_gb;
    G1Xyzz *out_pt;
    uint32_t t;
    uint32_t head_gb, tail_gb;
    __device__ __forceinline__ void flush(uint32_t gb, const G1Xyzz &acc, bool tl, bool tr) {
        if (!tl && !tr) {
            store_xyzz(buckets + gb, acc);
        } else if (tl) {
            head_gb = gb;
            store_xyzz(out_pt + 2 * (size_t)t, acc);
            if (tr) {
                tail_gb = gb;
                store_xyzz(out_pt + 2 * (size_t)t + 1, G1Xyzz::identity());
            }
        } else {
            tail_gb = gb;
            store_xyzz(out_pt + 2 * (size_t)t + 1, acc);
        }
    }
    __device__ __forceinline__ void finish() {
        out_gb[2 * (size_t)t] = head_gb;
        out_gb[2 * (size_t)t + 1] = tail_gb;
    }
};

