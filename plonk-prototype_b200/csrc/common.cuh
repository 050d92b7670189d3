// common.cuh — context object, error plumbing and launch bookkeeping shared by the .cu files.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/pb200.h"

struct NttPlan;     // ntt.cu
struct pb200_comm;  // comm.cu: NCCL communicator of a multi-GPU context (nullptr = single GPU)

struct pb200_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    uint64_t launches = 0;
    bool profile = false;
    std::map<std::string, float> prof_ms;    // most recent duration per timer name
    std::map<std::string, float> prof_sum;   // Σ of every collected duration since pb200_profile_reset
    std::map<std::string, uint32_t> prof_cnt;
    // NTT state
    std::map<uint32_t, NttPlan *> ntt_plans;  // key: log_n | inverse << 8 | coset << 9
    void *ntt_scratch = nullptr;
    size_t ntt_scratch_bytes = 0;
    // MSM workspace (grown on demand, reused across calls)
    void *msm_ws = nullptr;
    size_t msm_ws_bytes = 0;
    void *stage = nullptr;   // device staging for the host-buffer entry points (scalars / NTT vector)
    size_t stage_bytes = 0;
    void *pinned = nullptr;  // small pinned staging block for results
    size_t pinned_bytes = 0;
    pb200_comm *comm = nullptr;
};

struct pb200_srs {
    const uint64_t *dev = nullptr;
    size_t n = 0;
    bool owned = false;
    // optional pre-doubled copies: pre[w·n + i] = 2^(c_pre·w)·P_i (affine), w < W_pre   (pb200_srs_precompute)
    void *pre = nullptr;
    uint32_t c_pre = 0, W_pre = 0;
};

inline int pb_fail(pb200_ctx *ctx, int code, const char *what, const char *detail, const char *file, int line) {
    if (ctx) {
        char buf[512];
        snprintf(buf, sizeof(buf), "%s: %s (%s:%d)", what, detail ? detail : "", file, line);
        ctx->err = buf;
    }
    return code;
}
#define PB_CUDA(ctx, call)                                                                          \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) return pb_fail(ctx, PB200_ERR_CUDA, #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)
#define PB_ARG(ctx, cond)                                                                           \
    do {                                                                                            \
        if (!(cond)) return pb_fail(ctx, PB200_ERR_ARG, "bad argument", #cond, __FILE__, __LINE__); \
    } while (0)
#define PB_TRY(expr)            \
    do {                        \
        int rc__ = (expr);      \
        if (rc__) return rc__;  \
    } while (0)
// After a kernel launch: count it and surface launch-configuration errors.
#define PB_LAUNCHED(ctx)                                                                            \
    do {                                                                                            \
        (ctx)->launches++;                                                                          \
        cudaError_t e__ = cudaGetLastError();                                                       \
        if (e__ != cudaSuccess) return pb_fail(ctx, PB200_ERR_CUDA, "kernel launch", cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

// Scoped CUDA-event timer feeding pb200_profile_ms (only when profiling is on).
struct PbTimer {
    pb200_ctx *ctx;
    const char *name;
    cudaEvent_t a = nullptr, b = nullptr;
    PbTimer(pb200_ctx *c, const char *n) : ctx(c), name(n) {
        if (ctx->profile) {
            cudaEventCreate(&a);
            cudaEventCreate(&b);
            cudaEventRecord(a, ctx->stream);
        }
    }
    void stop() {
        if (a && b) cudaEventRecord(b, ctx->stream);
    }
    // Call after the stream has been synchronised.
    void collect() {
        if (a && b) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, a, b) == cudaSuccess) {
                ctx->prof_ms[name] = ms;
                ctx->prof_sum[name] += ms;
                ctx->prof_cnt[name]++;
            }
            cudaEventDestroy(a);
            cudaEventDestroy(b);
            a = b = nullptr;
        }
    }
    ~PbTimer() {
        if (a) cudaEventDestroy(a);
        if (b) cudaEventDestroy(b);
    }
};

int pb_ensure(pb200_ctx *ctx, void **buf, size_t *have, size_t need);  // api.cu
int comm_allgather_host(pb200_ctx *ctx, const void *send, void *recv, size_t bytes);  // comm.cu
int comm_stream_barrier(pb200_ctx *ctx);                                              // comm.cu
// Σ over ranks of `batch` projective points each rank holds in comm_partials_buffer(): all-gather + add on the device, one D2H
uint32_t *comm_partials_buffer(pb200_ctx *ctx);                                       // comm.cu
int comm_sum_partials(pb200_ctx *ctx, uint32_t batch, uint64_t *out_xyz_host);        // comm.cu
// msm.cu: batched MSM over pre-doubled bases with the results left in device memory (36 words each)
struct pb200_srs;
int msm_batch_to_dev(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, const uint64_t *scalars_dev, size_t n, uint32_t batch,
                     size_t scalar_stride, uint32_t *result_dev, bool *handled);
int tail_g1_sum_batch(pb200_ctx *ctx, const uint32_t *pts, uint32_t count, uint32_t batch, uint32_t *results);  // msm_tail.cu
// kzg.cu: a rank's coefficient slice of the Ruffini witness (two phases around a 32-byte all-gather)
int kzg_witness_slice_phase1(pb200_ctx *ctx, const uint64_t *poly_slice_dev, uint32_t lo, uint32_t cnt, const uint64_t z_mont[4],
                             uint64_t *q_slice_dev, uint64_t *work_dev, uint64_t slice_total_out[4]);
int kzg_witness_slice_phase2(pb200_ctx *ctx, uint32_t lo, uint32_t cnt, uint64_t *q_slice_dev, uint64_t *work_dev,
                             const uint64_t later_slices_total[4]);
size_t kzg_witness_slice_work_scalars(uint32_t cnt);
// lagrange.cu: Lagrange-basis key [L_i(τ)]G, i < 2^log_n, from the first 2^log_n points of `srs` (owned, no pre-doubled
// copies).  *degenerate (and *out = nullptr, return 0) when some point is the identity, i.e. `srs` is not powers of τ.
int lagrange_srs_build(pb200_ctx *ctx, const pb200_srs *srs, uint32_t log_n, pb200_srs **out, bool *degenerate);
