// lagrange.cu — builds the Lagrange-basis commit key Q_i = [L_i(τ)]G from a monomial key (lagrange.cuh has the
// algorithm).  The prover commits its wire polynomials against it from their evaluations (plonk.cu, round 1): zero and
// small evaluations have few or no non-zero MSM digits, which the coefficients of the same polynomial do not.
// One launch per radix-2 stage; every thread runs long serial chains of group operations, so the kernels use the shared,
// non-inlined field multiplier as the MSM tail kernels do.
#define PB_FIELD_NOINLINE_MUL 1
#include "common.cuh"
#include "host_field.h"
#include "lagrange.cuh"

namespace {

__global__ void __launch_bounds__(128) lagrange_load_kernel(const G1Affine *__restrict__ bases, uint32_t log_n, G1Xyzz *a) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (1u << log_n)) lagrange::load_point(bases, i, log_n, a);
}
__global__ void __launch_bounds__(128) lagrange_stage_kernel(G1Xyzz *a, uint32_t n, uint32_t half, Fr w) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n / 2) lagrange::butterfly(a, half, k, w);
}
__global__ void __launch_bounds__(128) lagrange_normalize_kernel(G1Xyzz *a, uint32_t n, Fr n_inv, G1Affine *out, uint32_t *degenerate) {
    const uint32_t i0 = (blockIdx.x * blockDim.x + threadIdx.x) * lagrange::kNormPer;
    if (i0 < n) lagrange::normalize(a, i0, min(lagrange::kNormPer, n - i0), n_inv, out, degenerate);
}

inline Fr to_dev(const hostf::HFr &h) {
    Fr r;
    memcpy(r.l, h.l, 32);
    return r;
}

}  // namespace

int lagrange_srs_build(pb200_ctx *ctx, const pb200_srs *srs, uint32_t log_n, pb200_srs **out, bool *degenerate) {
    *out = nullptr;
    *degenerate = false;
    PB_ARG(ctx, srs != nullptr && srs->dev != nullptr && log_n <= 26 && ((size_t)1 << log_n) <= srs->n);
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = 1u << log_n;
    cudaStream_t st = ctx->stream;
    void *work = nullptr, *pts = nullptr;  // work: n XYZZ points + the degenerate flag
    PB_CUDA(ctx, cudaMalloc(&work, (size_t)n * sizeof(G1Xyzz) + 256));
    cudaError_t e = cudaMalloc(&pts, (size_t)n * sizeof(G1Affine));
    G1Xyzz *a = (G1Xyzz *)work;
    uint32_t *flag = (uint32_t *)((char *)work + (size_t)n * sizeof(G1Xyzz));
    uint32_t flag_host = 0;
    if (e == cudaSuccess) e = cudaMemsetAsync(flag, 0, 4, st);
    if (e == cudaSuccess) {
        lagrange_load_kernel<<<(n + 127) / 128, 128, 0, st>>>((const G1Affine *)srs->dev, log_n, a);
        ctx->launches++;
        e = cudaGetLastError();
    }
    const hostf::HFr w_inv = hostf::domain_root(log_n).inv();
    for (uint32_t half = 1; half < n && e == cudaSuccess; half <<= 1) {
        // ω_(2·half)^(−1) = (ω_n^(−1))^(n / (2·half))
        lagrange_stage_kernel<<<(n / 2 + 127) / 128, 128, 0, st>>>(a, n, half, to_dev(w_inv.pow_u64(n / (2 * half))));
        ctx->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) {
        const uint32_t threads = (n + lagrange::kNormPer - 1) / lagrange::kNormPer;
        lagrange_normalize_kernel<<<(threads + 127) / 128, 128, 0, st>>>(a, n, to_dev(hostf::HFr::from_u64(n).inv()), (G1Affine *)pts, flag);
        ctx->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&flag_host, flag, 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(work);
    if (e != cudaSuccess || flag_host) {
        cudaFree(pts);
        if (e != cudaSuccess) return pb_fail(ctx, PB200_ERR_CUDA, "lagrange commit key", cudaGetErrorString(e), __FILE__, __LINE__);
        *degenerate = true;
        return 0;
    }
    pb200_srs *s = new pb200_srs();
    s->dev = (const uint64_t *)pts;
    s->n = n;
    s->owned = true;
    *out = s;
    return 0;
}

extern "C" int pb200_srs_lagrange(pb200_ctx *ctx, const pb200_srs *srs, uint32_t log_n, pb200_srs **out) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, out != nullptr);
    bool degenerate = false;
    PB_TRY(lagrange_srs_build(ctx, srs, log_n, out, &degenerate));
    if (degenerate) return pb_fail(ctx, PB200_ERR_ARG, "lagrange commit key", "a Lagrange point is the identity: the key is not powers of tau",
                                   __FILE__, __LINE__);
    return 0;
}
