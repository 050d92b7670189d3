// srs_io.cu — commit keys in the checked compressed format: dusk-plonk 0.8.2 `CommitKey::{from_slice, to_var_bytes}`
// (crate pinned at /root/reference/Cargo.toml:19), one point per thread with the codec of g1_codec.cuh.
//
// Loading is compute-bound (≈ 1,900 Fp multiplications per point: square root and subgroup test), storing is memory-bound
// (two conversions out of Montgomery form per point).  Both entry points stage the 48-byte encodings in one device buffer,
// copy with cudaMemcpyAsync on the context stream, launch one kernel and synchronise once.
#include <cstring>

#include "g1_codec.cuh"
#include "msm_common.cuh"

// One thread per point: three 16-byte loads, decode + checks, one 96-byte store of the packed affine point.  An invalid
// point is an ordinary result: its status is written and its index folded into *first_bad; the thread returns normally.
// Also launched by the batched verifier (verify_batch.cu) on the points of its proofs and verifier key.
__global__ void __launch_bounds__(128) g1_decompress_kernel(const uint4 *__restrict__ enc, uint32_t n, G1Affine *__restrict__ out,
                                                            uint8_t *__restrict__ status, uint32_t *first_bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint4 a = enc[3 * (size_t)i], b = enc[3 * (size_t)i + 1], c = enc[3 * (size_t)i + 2];
    const uint32_t w[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
    G1Affine p;
    const int st = g1_decode_checked_words(w, p);
    status[i] = (uint8_t)st;
    if (st == PB200_G1_OK) {
        store_fp2(reinterpret_cast<uint4 *>(out + i), p.x, p.y);
    } else {
        atomicMin(first_bad, i);
    }
}

namespace {

// One thread per point: one 96-byte load, two conversions out of Montgomery form, three 16-byte stores.
__global__ void __launch_bounds__(256) g1_compress_kernel(const G1Affine *__restrict__ pts, uint32_t n, uint4 *__restrict__ enc) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    G1Affine p;
    load_fp2(reinterpret_cast<const uint4 *>(pts + i), p.x, p.y);
    uint32_t w[12];
    g1_encode_words(p, w);
    enc[3 * (size_t)i] = make_uint4(w[0], w[1], w[2], w[3]);
    enc[3 * (size_t)i + 1] = make_uint4(w[4], w[5], w[6], w[7]);
    enc[3 * (size_t)i + 2] = make_uint4(w[8], w[9], w[10], w[11]);
}

const char *g1_status_name(int st) {
    switch (st) {
        case PB200_G1_BAD_FLAGS: return "bad flag bits (PB200_G1_BAD_FLAGS)";
        case PB200_G1_X_RANGE: return "x is not below p (PB200_G1_X_RANGE)";
        case PB200_G1_NOT_ON_CURVE: return "not on the curve (PB200_G1_NOT_ON_CURVE)";
        case PB200_G1_NOT_IN_SUBGROUP: return "not in the prime-order subgroup (PB200_G1_NOT_IN_SUBGROUP)";
        case PB200_G1_IDENTITY: return "the identity, which a commit key cannot hold (PB200_G1_IDENTITY)";
        default: return "unknown status";
    }
}

}  // namespace

extern "C" int pb200_srs_from_compressed(pb200_ctx *ctx, const uint8_t *bytes_host, size_t n_points, uint8_t *status_host,
                                         pb200_srs **out) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, bytes_host != nullptr && out != nullptr && n_points >= 1 && n_points < ((size_t)1 << 31));
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t enc_bytes = 48 * n_points;
    // staging: encodings (48·n) | first invalid index (16 B slot) | per-point status (n)
    void *pts = nullptr, *stage = nullptr;
    PB_CUDA(ctx, cudaMalloc(&pts, n_points * sizeof(G1Affine)));
    cudaError_t e = cudaMalloc(&stage, enc_bytes + 16 + n_points);
    uint32_t *first_bad = (uint32_t *)((uint8_t *)stage + enc_bytes);
    uint8_t *status = (uint8_t *)stage + enc_bytes + 16;
    const uint32_t n = (uint32_t)n_points;
    if (e == cudaSuccess) e = cudaMemcpyAsync(stage, bytes_host, enc_bytes, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(first_bad, 0xff, 4, ctx->stream);
    PbTimer t(ctx, "srs.decompress");  // started after the copy is enqueued: it times the kernel alone
    if (e == cudaSuccess) {
        g1_decompress_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>((const uint4 *)stage, n, (G1Affine *)pts, status, first_bad);
        ctx->launches++;
        e = cudaGetLastError();
        t.stop();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->pinned, first_bad, 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && status_host) e = cudaMemcpyAsync(status_host, status, n_points, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) t.collect();
    uint32_t bad = 0xffffffffu;
    uint8_t why = 0;
    if (e == cudaSuccess) {
        memcpy(&bad, ctx->pinned, 4);
        if (bad != 0xffffffffu) {
            e = cudaMemcpyAsync(ctx->pinned, status + bad, 1, cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
            if (e == cudaSuccess) why = *(const uint8_t *)ctx->pinned;
        }
    }
    cudaFree(stage);
    if (e != cudaSuccess) {
        cudaFree(pts);
        return pb_fail(ctx, PB200_ERR_CUDA, "srs from compressed", cudaGetErrorString(e), __FILE__, __LINE__);
    }
    if (bad != 0xffffffffu) {
        cudaFree(pts);
        char msg[160];
        snprintf(msg, sizeof(msg), "point %u of %zu: %s", bad, n_points, g1_status_name(why));
        return pb_fail(ctx, PB200_ERR_ARG, "invalid compressed G1 point", msg, __FILE__, __LINE__);
    }
    pb200_srs *s = new pb200_srs();
    s->dev = (const uint64_t *)pts;
    s->n = n_points;
    s->owned = true;
    *out = s;
    return 0;
}

extern "C" int pb200_srs_to_compressed(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, size_t n, uint8_t *bytes_host) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, srs != nullptr && srs->dev != nullptr && bytes_host != nullptr && n >= 1 && n < ((size_t)1 << 31));
    PB_ARG(ctx, offset <= srs->n && n <= srs->n - offset);
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    void *stage = nullptr;
    PB_CUDA(ctx, cudaMalloc(&stage, 48 * n));
    cudaError_t e;
    {
        PbTimer t(ctx, "srs.compress");
        g1_compress_kernel<<<(uint32_t)((n + 255) / 256), 256, 0, ctx->stream>>>(reinterpret_cast<const G1Affine *>(srs->dev) + offset,
                                                                                (uint32_t)n, (uint4 *)stage);
        ctx->launches++;
        e = cudaGetLastError();
        t.stop();
        if (e == cudaSuccess) e = cudaMemcpyAsync(bytes_host, stage, 48 * n, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e == cudaSuccess) t.collect();
    }
    cudaFree(stage);
    if (e != cudaSuccess) return pb_fail(ctx, PB200_ERR_CUDA, "srs to compressed", cudaGetErrorString(e), __FILE__, __LINE__);
    return 0;
}
