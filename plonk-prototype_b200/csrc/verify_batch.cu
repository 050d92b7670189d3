// verify_batch.cu — many proofs of one circuit in one batched pairing check (pb200_verify_batch).
//
// pb200_verify (verify.cu) ends every proof k in e(−W_k, βH)·e(C_k, H) = 1, where W_k and C_k are linear combinations of
// the proof's 11 points and of 16 bases every proof shares (15 verifier-key commitments and G) with scalars that come from
// the proof's transcript alone (verify_batch.cuh).  With random weights ρ_k the K equations become one:
//
//     e(−Σ ρ_k W_k, βH) · e(Σ ρ_k C_k, H) = 1
//
// which is two MSMs over the proofs' points (C and W side, one pipeline pass each), one 16-point MSM over the shared bases
// with the column sums Σ ρ_k e_{k,j}, and one pairing check on the host.  If it fails, bisection over contiguous proof
// ranges (the same ρ_k; a range's shared-base scalars are its own column sums) finds the invalid proofs.
//
// Device work, in order on the context stream:
//   1. g1_decompress_kernel (srs_io.cu, unchanged) over the 11·K proof points and the 15 verifier-key points;
//   2. verify_prepare_kernel, one thread per proof: evaluations, transcript, challenges, PI(z), t(z), coefficients, digest;
//   3. (host) D = Merlin("pb200 verify_batch") over the seed, n, K and every digest;
//   4. verify_weight_kernel, one thread per proof: ρ_k, the two MSM scalar vectors, placeholder bases for identity slots;
//   5. verify_colsum_kernel: shared-base scalars over a proof range; then the MSMs (msm.cu) and the pairing (host).
#include <algorithm>
#include <chrono>
#include <cstring>
#include <vector>

#include "msm_common.cuh"
#include "pairing_host.h"
#include "verify_batch.cuh"

using hostf::HFp;
using hostf::HFr;

namespace {

constexpr int kPts = vb::kProofPoints, kSh = vb::kShared;

// One thread per proof.  Writes the proof's C-side coefficients (kPts), shared-base coefficients (kSh), u_k, its digest
// and its verdict; a rejected proof writes its verdict only.
__global__ void __launch_bounds__(128) verify_prepare_kernel(const merlin::Transcript seed, const uint8_t *__restrict__ proofs,
                                                             const uint8_t *__restrict__ pt_status, const vb::Consts k,
                                                             const Fr *__restrict__ wg, const Fr *__restrict__ pi, uint32_t K,
                                                             Fr *__restrict__ coef, Fr *__restrict__ ecoef, Fr *__restrict__ u_out,
                                                             uint8_t *__restrict__ digest, uint8_t *__restrict__ verdict) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= K) return;
    vb::ProofOut o;
    const int st = vb::prepare_one(seed, proofs + 1040 * (size_t)p, pt_status + kPts * (size_t)p, k, wg, pi + (size_t)k.n_pi * p, o);
    verdict[p] = (uint8_t)st;
    if (st != vb::OK) {
        for (int i = 0; i < 32; i++) digest[32 * (size_t)p + i] = 0;
        return;
    }
    for (int i = 0; i < kPts; i++) coef[kPts * (size_t)p + i] = o.coef[i];
    for (int j = 0; j < kSh; j++) ecoef[kSh * (size_t)p + j] = o.e[j];
    u_out[p] = o.u;
    for (int i = 0; i < 32; i++) digest[32 * (size_t)p + i] = o.digest[i];
}

// One thread per proof: ρ_k and the scalar vectors.  scal[0 .. kPts·K) is the C side (ρ·coef), scal[kPts·K .. 2·kPts·K) the
// W side (ρ at W_z, ρ·u at W_zω); ecoef is scaled by ρ in place.  Rows of rejected proofs and identity slots are zero, and
// every slot whose point did not decode gets G (shared slot 15) as its base so that the MSM only ever reads valid points.
__global__ void __launch_bounds__(128) verify_weight_kernel(const merlin::Transcript rho_seed, uint32_t K, const uint8_t *__restrict__ verdict,
                                                            const uint8_t *__restrict__ pt_status, const Fr *__restrict__ coef,
                                                            Fr *__restrict__ ecoef, const Fr *__restrict__ u_in, Fr *__restrict__ scal,
                                                            G1Affine *__restrict__ pts) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= K) return;
    const bool ok = verdict[p] == vb::OK;
    const Fr r = ok ? vb::rho(rho_seed, p) : Fr::zero();
    const Fr ru = ok ? r * u_in[p] : Fr::zero();
    Fr *sc = scal + kPts * (size_t)p, *sw = scal + kPts * ((size_t)K + p);
    for (int i = 0; i < kPts; i++) {
        const bool live = ok && pt_status[kPts * (size_t)p + i] == PB200_G1_OK;
        sc[i] = live ? r * coef[kPts * (size_t)p + i] : Fr::zero();
        sw[i] = live && i == vb::P_WZ ? r : live && i == vb::P_WZW ? ru : Fr::zero();
        if (pt_status[kPts * (size_t)p + i] != PB200_G1_OK) pts[kPts * (size_t)p + i] = pts[kPts * (size_t)K + vb::GEN];
    }
    for (int j = 0; j < kSh; j++) ecoef[kSh * (size_t)p + j] = ok ? r * ecoef[kSh * (size_t)p + j] : Fr::zero();
}

// Σ_{p ∈ [lo, hi)} ecoef[p][j] for the kSh columns: one block per column.
constexpr int kSumThreads = 256;
__global__ void __launch_bounds__(kSumThreads) verify_colsum_kernel(const Fr *__restrict__ ecoef, uint32_t lo, uint32_t hi, Fr *__restrict__ out) {
    __shared__ Fr part[kSumThreads];
    const int j = blockIdx.x;
    Fr acc = Fr::zero();
    for (uint32_t p = lo + threadIdx.x; p < hi; p += kSumThreads) acc = acc + ecoef[kSh * (size_t)p + j];
    part[threadIdx.x] = acc;
    __syncthreads();
    for (int s = kSumThreads / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) part[threadIdx.x] = part[threadIdx.x] + part[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[j] = part[0];
}

void profile_add(pb200_ctx *ctx, const char *name, float ms) {
    if (!ctx->profile) return;
    ctx->prof_ms[name] = ms;
    ctx->prof_sum[name] += ms;
    ctx->prof_cnt[name]++;
}

// MSM result (homogeneous X ‖ Y ‖ Z) → Jacobian (X·Z, Y·Z², Z)
pairing::G1J jac_from_homogeneous(const uint64_t xyz[18]) {
    const HFp X = HFp::load(xyz), Y = HFp::load(xyz + 6), Z = HFp::load(xyz + 12);
    if (Z.is_zero()) return pairing::G1J::identity();
    return {X * Z, Y * Z.sqr(), Z};
}

// Device buffers of one call, carved out of a single allocation.
struct Bufs {
    void *base = nullptr;
    uint8_t *proofs, *enc, *pt_status, *digest, *verdict;
    G1Affine *pts;  // kPts·K proof points, then kSh shared bases (15 vk + G)
    Fr *wg, *pi, *coef, *ecoef, *u, *scal, *sums;
    uint32_t *first_bad;
};
size_t carve(Bufs &b, size_t K, size_t n_pi, bool assign) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t at = off;
        off = (off + bytes + 255) & ~(size_t)255;
        return (uint8_t *)b.base + at;
    };
    uint8_t *p[14];
    p[0] = take(1040 * K);
    p[1] = take(48 * (kPts * K + 15));
    p[2] = take(kPts * K + 15);
    p[3] = take(32 * K);
    p[4] = take(K);
    p[5] = take(96 * (kPts * K + kSh));
    p[6] = take(32 * (n_pi ? n_pi : 1));
    p[7] = take(32 * (n_pi ? n_pi * K : 1));
    p[8] = take(32 * kPts * K);
    p[9] = take(32 * kSh * K);
    p[10] = take(32 * K);
    p[11] = take(32 * 2 * kPts * K);
    p[12] = take(32 * kSh);
    p[13] = take(4);
    if (assign) {
        b.proofs = p[0], b.enc = p[1], b.pt_status = p[2], b.digest = p[3], b.verdict = p[4];
        b.pts = (G1Affine *)p[5], b.wg = (Fr *)p[6], b.pi = (Fr *)p[7], b.coef = (Fr *)p[8], b.ecoef = (Fr *)p[9];
        b.u = (Fr *)p[10], b.scal = (Fr *)p[11], b.sums = (Fr *)p[12], b.first_bad = (uint32_t *)p[13];
    }
    return off;
}

// The batched check over proofs [lo, hi): two MSMs over their points, one over the shared bases, one pairing product.
struct Checker {
    pb200_ctx *ctx;
    const Bufs &b;
    size_t K;
    pb200_srs *srs_pts, *srs_shared;
    pairing::G2A bh;
    float msm_ms = 0;
    int checks = 0;

    int msm_timed(int (*fn)(pb200_ctx *, const pb200_srs *, size_t, const uint64_t *, size_t, uint32_t, size_t, uint64_t *),
                  const pb200_srs *s, size_t off, const uint64_t *sc, size_t n, uint32_t batch, size_t stride, uint64_t *out) {
        if (!ctx->profile) return fn(ctx, s, off, sc, n, batch, stride, out);
        cudaEvent_t a, e;
        cudaEventCreate(&a);
        cudaEventCreate(&e);
        cudaEventRecord(a, ctx->stream);
        const int rc = fn(ctx, s, off, sc, n, batch, stride, out);  // blocks: the result is on the host
        cudaEventRecord(e, ctx->stream);
        float ms = 0;
        if (rc == 0 && cudaEventSynchronize(e) == cudaSuccess && cudaEventElapsedTime(&ms, a, e) == cudaSuccess) msm_ms += ms;
        cudaEventDestroy(a);
        cudaEventDestroy(e);
        return rc;
    }
    // *pass = 1 iff e(−W, βH)·e(C, H) = 1 over the range
    int check(uint32_t lo, uint32_t hi, bool *pass) {
        verify_colsum_kernel<<<kSh, kSumThreads, 0, ctx->stream>>>(b.ecoef, lo, hi, b.sums);
        PB_LAUNCHED(ctx);
        uint64_t cw[36], sh[18];
        PB_TRY(msm_timed(pb200_msm_g1_batch_dev, srs_pts, (size_t)kPts * lo, (const uint64_t *)(b.scal + (size_t)kPts * lo),
                         (size_t)kPts * (hi - lo), 2, kPts * K, cw));
        PB_TRY(msm_timed(pb200_msm_g1_batch_dev, srs_shared, 0, (const uint64_t *)b.sums, kSh, 1, kSh, sh));
        const auto t0 = std::chrono::steady_clock::now();
        const pairing::G1J c = pairing::g1_add(jac_from_homogeneous(cw), jac_from_homogeneous(sh));
        const pairing::G1J w = jac_from_homogeneous(cw + 18);
        const pairing::Fp12 f = pairing::miller_loop(pairing::g1_to_affine(pairing::g1_neg(w)), bh) *
                                pairing::miller_loop(pairing::g1_to_affine(c), pairing::g2_generator());
        *pass = pairing::final_exponentiation(f) == pairing::Fp12::one();
        profile_add(ctx, "verify.pairing", std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count());
        checks++;
        return 0;
    }
};

// Bisection over [lo, hi) once the range is known to fail (or not yet checked: known_fail = false).  A passing range
// accepts its surviving proofs; a failing range with one survivor rejects it.  If the left half passes, the right half
// fails (its product is the parent's), so it is not checked again.
int bisect(Checker &ck, const std::vector<uint32_t> &surv_prefix, const std::vector<uint8_t> &alive, uint32_t lo, uint32_t hi,
           bool known_fail, uint8_t *accepted) {
    const uint32_t s = surv_prefix[hi] - surv_prefix[lo];
    if (s == 0) return 0;
    if (!known_fail) {
        bool pass = false;
        PB_TRY(ck.check(lo, hi, &pass));
        if (pass) {
            for (uint32_t p = lo; p < hi; p++) accepted[p] = alive[p];
            return 0;
        }
    }
    if (s == 1) return 0;
    const uint32_t mid = lo + (hi - lo) / 2;
    const uint32_t sl = surv_prefix[mid] - surv_prefix[lo], sr = surv_prefix[hi] - surv_prefix[mid];
    if (sl == 0) return bisect(ck, surv_prefix, alive, mid, hi, true, accepted);
    if (sr == 0) return bisect(ck, surv_prefix, alive, lo, mid, true, accepted);
    bool left_pass = false;
    PB_TRY(ck.check(lo, mid, &left_pass));
    if (left_pass) {
        for (uint32_t p = lo; p < mid; p++) accepted[p] = alive[p];
    } else {
        PB_TRY(bisect(ck, surv_prefix, alive, lo, mid, true, accepted));
    }
    return bisect(ck, surv_prefix, alive, mid, hi, left_pass, accepted);
}

HFr host_omega(size_t n) {
    uint32_t log_n = 0;
    while (((size_t)1 << log_n) < n) log_n++;
    const uint64_t root32[4] = {0xb9b58d8c5f0e466aull, 0x5b1b4c801819d7ecull, 0x0af53ae352a31e64ull, 0x5bf3adda19e9b27bull};
    HFr omega = HFr::load(root32);
    for (uint32_t k = 0; k < 32 - log_n; k++) omega = omega.sqr();
    return omega;
}
Fr to_dev(const HFr &a) {
    Fr r;
    memcpy(r.l, a.l, 32);
    return r;
}

int run(pb200_ctx *ctx, Bufs &b, const uint8_t *vk_commitments, size_t n, const uint8_t *label, size_t label_len, const uint8_t *proofs,
        size_t K, const uint32_t *pi_gate, const uint64_t *pi_mont, size_t n_pi, const pairing::G2A &bh, const uint8_t seed[32],
        uint8_t *accepted, int *all_accepted) {
    cudaStream_t st = ctx->stream;
    const uint32_t n_pts = (uint32_t)(kPts * K + 15);
    // 1. decode every point
    PB_CUDA(ctx, cudaMemcpyAsync(b.proofs, proofs, 1040 * K, cudaMemcpyHostToDevice, st));
    PB_CUDA(ctx, cudaMemcpy2DAsync(b.enc, 48 * kPts, b.proofs, 1040, 48 * kPts, K, cudaMemcpyDeviceToDevice, st));
    PB_CUDA(ctx, cudaMemcpyAsync(b.enc + 48 * kPts * K, vk_commitments, 15 * 48, cudaMemcpyHostToDevice, st));
    PB_CUDA(ctx, cudaMemsetAsync(b.first_bad, 0xff, 4, st));
    uint64_t gen[12];
    memcpy(gen, pairing::kG1x, 48);
    memcpy(gen + 6, pairing::kG1y, 48);
    PB_CUDA(ctx, cudaMemcpyAsync(b.pts + kPts * K + vb::GEN, gen, 96, cudaMemcpyHostToDevice, st));
    {
        PbTimer t(ctx, "verify.decompress");
        g1_decompress_kernel<<<(n_pts + 127) / 128, 128, 0, st>>>((const uint4 *)b.enc, n_pts, b.pts, b.pt_status, b.first_bad);
        PB_LAUNCHED(ctx);
        t.stop();
        uint8_t vk_st[15];
        PB_CUDA(ctx, cudaMemcpyAsync(vk_st, b.pt_status + kPts * K, 15, cudaMemcpyDeviceToHost, st));
        PB_CUDA(ctx, cudaStreamSynchronize(st));
        t.collect();
        uint32_t vk_identity = 0;
        for (int j = 0; j < 15; j++) {
            if (vk_st[j] == PB200_G1_IDENTITY) vk_identity |= 1u << j;
            else if (vk_st[j] != PB200_G1_OK) return 0;  // malformed verifier key: every proof is rejected, as pb200_verify does
        }
        for (int j = 0; j < 15; j++)
            if ((vk_identity >> j) & 1) PB_CUDA(ctx, cudaMemcpyAsync(b.pts + kPts * K + j, gen, 96, cudaMemcpyHostToDevice, st));

        // 2. per-proof derivation
        merlin::Transcript tr(label, label_len);
        {
            enum { Q_M, Q_L, Q_R, Q_O, Q_C, Q_4, Q_ARITH, Q_RANGE, Q_LOGIC, Q_FIXED, Q_VAR, S1 };
            const char *const lab[11] = {"q_m", "q_l", "q_r", "q_o", "q_c", "q_4", "q_arith", "q_range", "q_logic", "q_variable_group_add",
                                         "q_fixed_group_add"};
            const int idx[11] = {Q_M, Q_L, Q_R, Q_O, Q_C, Q_4, Q_ARITH, Q_RANGE, Q_LOGIC, Q_VAR, Q_FIXED};
            for (int q = 0; q < 11; q++) tr.append_commitment(lab[q], vk_commitments + 48 * idx[q]);
            const char *const sl[4] = {"left_sigma", "right_sigma", "out_sigma", "fourth_sigma"};
            for (int c = 0; c < 4; c++) tr.append_commitment(sl[c], vk_commitments + 48 * (S1 + c));
            tr.circuit_domain_sep(n);
        }
        vb::Consts kc;
        const HFr omega = host_omega(n), n_fr = HFr::from_u64(n);
        kc.n = n;
        kc.n_pi = (uint32_t)n_pi;
        kc.vk_identity = vk_identity;
        kc.omega = to_dev(omega);
        kc.n_fr = to_dev(n_fr);
        kc.n_inv = to_dev(n_fr.inv());
        kc.edwards_d = to_dev((HFr::from_u64(10240) * HFr::from_u64(10241).inv()).neg());
        std::vector<uint64_t> wg(4 * (n_pi ? n_pi : 1));
        for (size_t j = 0; j < n_pi; j++) omega.pow_u64(pi_gate[j]).store(&wg[4 * j]);
        if (n_pi) {
            PB_CUDA(ctx, cudaMemcpyAsync(b.wg, wg.data(), 32 * n_pi, cudaMemcpyHostToDevice, st));
            PB_CUDA(ctx, cudaMemcpyAsync(b.pi, pi_mont, 32 * n_pi * K, cudaMemcpyHostToDevice, st));
        }
        PbTimer tp(ctx, "verify.prepare");
        verify_prepare_kernel<<<(uint32_t)((K + 127) / 128), 128, 0, st>>>(tr, b.proofs, b.pt_status, kc, b.wg, b.pi, (uint32_t)K, b.coef,
                                                                          b.ecoef, b.u, b.digest, b.verdict);
        PB_LAUNCHED(ctx);
        tp.stop();
        std::vector<uint8_t> digests(32 * K), verdict(K);
        PB_CUDA(ctx, cudaMemcpyAsync(digests.data(), b.digest, 32 * K, cudaMemcpyDeviceToHost, st));
        PB_CUDA(ctx, cudaMemcpyAsync(verdict.data(), b.verdict, K, cudaMemcpyDeviceToHost, st));
        PB_CUDA(ctx, cudaStreamSynchronize(st));
        tp.collect();

        // 3. the batch digest D and the weight transcript
        merlin::Transcript dt((const uint8_t *)"pb200 verify_batch", 18);
        dt.append_message("seed", seed, 32);
        dt.append_u64("n", n);
        dt.append_u64("K", K);
        dt.append_message("digests", digests.data(), 32 * K);
        uint8_t D[32];
        dt.challenge_bytes("D", D, 32);
        merlin::Transcript rho_seed((const uint8_t *)"pb200 rho", 9);
        rho_seed.append_message("D", D, 32);

        // 4. weights and scalar vectors
        PbTimer tw(ctx, "verify.weight");
        verify_weight_kernel<<<(uint32_t)((K + 127) / 128), 128, 0, st>>>(rho_seed, (uint32_t)K, b.verdict, b.pt_status, b.coef, b.ecoef,
                                                                         b.u, b.scal, b.pts);
        PB_LAUNCHED(ctx);
        tw.stop();
        PB_CUDA(ctx, cudaStreamSynchronize(st));
        tw.collect();

        // 5. the combined check, then bisection if it fails
        std::vector<uint8_t> alive(K);
        std::vector<uint32_t> prefix(K + 1, 0);
        for (size_t p = 0; p < K; p++) {
            alive[p] = verdict[p] == vb::OK;
            prefix[p + 1] = prefix[p] + alive[p];
        }
        pb200_srs *srs_pts = nullptr, *srs_shared = nullptr;
        PB_TRY(pb200_srs_wrap_dev(ctx, (const uint64_t *)b.pts, kPts * K, &srs_pts));
        const int rc_w = pb200_srs_wrap_dev(ctx, (const uint64_t *)(b.pts + kPts * K), kSh, &srs_shared);
        Checker ck{ctx, b, K, srs_pts, srs_shared, bh};
        int rc = rc_w ? rc_w : bisect(ck, prefix, alive, 0, (uint32_t)K, false, accepted);
        pb200_srs_free(ctx, srs_pts);
        if (srs_shared) pb200_srs_free(ctx, srs_shared);
        if (rc) return rc;
        profile_add(ctx, "verify.msm", ck.msm_ms);
    }
    int all = 1;
    for (size_t p = 0; p < K; p++) all &= accepted[p];
    *all_accepted = all;
    return 0;
}

}  // namespace

extern "C" int pb200_verify_batch(pb200_ctx *ctx, const uint8_t vk_commitments[15 * 48], size_t n, const uint8_t *transcript_label,
                                  size_t label_len, const uint8_t *proofs, size_t n_proofs, const uint32_t *pi_gate, const uint64_t *pi_mont,
                                  size_t n_pi, const uint64_t beta_h[24], const uint8_t seed[32], uint8_t *accepted, int *all_accepted) {
    if (!ctx) return PB200_ERR_ARG;
    PB_ARG(ctx, vk_commitments && proofs && beta_h && seed && accepted && all_accepted);
    PB_ARG(ctx, !n_pi || (pi_gate && pi_mont));
    PB_ARG(ctx, transcript_label || !label_len);
    PB_ARG(ctx, n >= 2 && !(n & (n - 1)) && n <= ((size_t)1 << 30));
    PB_ARG(ctx, n_proofs >= 1 && n_proofs <= ((size_t)1 << 20));
    if (n_pi > 1) {
        std::vector<uint32_t> sorted(pi_gate, pi_gate + n_pi);
        std::sort(sorted.begin(), sorted.end());
        PB_ARG(ctx, std::adjacent_find(sorted.begin(), sorted.end()) == sorted.end());
    }
    for (size_t j = 0; j < n_pi; j++) PB_ARG(ctx, pi_gate[j] < n);
    const pairing::G2A bh = {{HFp::load(beta_h), HFp::load(beta_h + 6)}, {HFp::load(beta_h + 12), HFp::load(beta_h + 18)}, false};
    PB_ARG(ctx, pairing::g2_on_curve(bh));
    memset(accepted, 0, n_proofs);
    *all_accepted = 0;
    PB_CUDA(ctx, cudaSetDevice(ctx->device));
    Bufs b;
    PB_CUDA(ctx, cudaMalloc(&b.base, carve(b, n_proofs, n_pi, false)));
    carve(b, n_proofs, n_pi, true);
    const int rc = run(ctx, b, vk_commitments, n, transcript_label, label_len, proofs, n_proofs, pi_gate, pi_mont, n_pi, bh, seed,
                       accepted, all_accepted);
    if (rc) {
        cudaStreamSynchronize(ctx->stream);  // nothing of this call may still be in flight when its buffers go
        memset(accepted, 0, n_proofs);
        *all_accepted = 0;
    }
    cudaFree(b.base);
    return rc;
}
