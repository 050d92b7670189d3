/* pb200.h — C ABI of the B200-native MSM / NTT prover backend.
 *
 * The reference (/root/reference, Manta-Network/Plonk-Prototype) has no FFI or plugin interface of its
 * own: its hot path lives in two functions of crates pinned by /root/reference/Cargo.toml:19-20
 *   - dusk_bls12_381::multiscalar_mul::msm_variable_base(&[G1Affine], &[Scalar]) -> G1Projective
 *   - dusk_plonk::fft::EvaluationDomain::{new, fft, ifft, coset_fft, coset_ifft}
 * (SURVEY.md §8a rows a3-a7, a12; §8b).  The entry points below are what a `-sys` crate patched into
 * those two functions would bind; INTEGRATION.md shows the Rust side.  Every entry point cites the
 * upstream function it replaces.
 *
 * Conventions (SURVEY.md §8b)
 *   - Scalars: 4 × u64 little-endian limbs, Montgomery form (a·2^256 mod r), fully reduced — the
 *     memory image of `Scalar.0` / `BlsScalar.0`.
 *   - Points: packed affine x[6] ‖ y[6] u64 limbs, Montgomery form (a·2^384 mod p), 96 bytes.  The
 *     identity is not encodable; callers drop identity bases (an SRS never holds one).
 *   - MSM result: homogeneous projective X ‖ Y ‖ Z (18 × u64, Montgomery) — the fields of `G1Projective`.
 *     As with upstream's msm_variable_base the representative is NOT normalised (Z is an arbitrary non-zero
 *     value for a finite point; the identity is (0, R, 0)); `G1Affine::from` / `to_bytes` on the caller's side
 *     yield the canonical bytes, and only those are compared for parity.
 *   - All functions return 0 on success, non-zero on failure (pb200_last_error has the text).  No
 *     exception, abort or CPU fallback ever crosses this boundary; a missing GPU is an error.
 *   - A context is bound to one CUDA device and one stream and is not thread-safe.
 */
#ifndef PB200_H
#define PB200_H
#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define PB200_API __attribute__((visibility("default")))
#else
#define PB200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pb200_ctx pb200_ctx;
typedef struct pb200_srs pb200_srs;

enum {
    PB200_OK = 0,
    PB200_ERR_ARG = 1,      /* bad argument (null pointer, log_n >= 32, range outside the SRS …) */
    PB200_ERR_CUDA = 2,     /* a CUDA runtime call or kernel failed */
    PB200_ERR_NO_DEVICE = 3 /* no usable sm_100 device */
};

/* ---- context ---------------------------------------------------------------------------------- */
PB200_API int pb200_init(pb200_ctx **out, int device_id);
PB200_API void pb200_destroy(pb200_ctx *ctx);
PB200_API const char *pb200_last_error(const pb200_ctx *ctx);
/* The CUDA stream (cudaStream_t) every call of this context is ordered on. */
PB200_API void *pb200_stream(pb200_ctx *ctx);
PB200_API int pb200_sync(pb200_ctx *ctx);

/* ---- device buffers (for callers that keep polynomials resident between calls) ---------------- */
PB200_API int pb200_malloc(pb200_ctx *ctx, void **dev_ptr, size_t bytes);
PB200_API int pb200_free(pb200_ctx *ctx, void *dev_ptr);
PB200_API int pb200_h2d(pb200_ctx *ctx, void *dev_dst, const void *host_src, size_t bytes);
PB200_API int pb200_d2h(pb200_ctx *ctx, void *host_dst, const void *dev_src, size_t bytes);

/* ---- NTT: dusk_plonk::fft::EvaluationDomain (SURVEY.md §8a a3-a7, App. B.2) ------------------- */
/* EvaluationDomain::new(num_coeffs): size = next power of two, error when log2(size) >= 32.
 * Writes log2(size) to *log_n. */
PB200_API int pb200_domain_log_size(size_t num_coeffs, uint32_t *log_n);
/* EvaluationDomain::{fft_in_place, ifft_in_place, coset_fft_in_place, coset_ifft_in_place} on a HOST
 * vector of exactly 2^log_n scalars (the Rust shim zero-pads shorter inputs as upstream does).
 *   inverse = 0, coset = 0 : fft          out[i] = Σ_j a_j ω^{ij}
 *   inverse = 1, coset = 0 : ifft         ω → ω⁻¹, then × n⁻¹
 *   inverse = 0, coset = 1 : coset_fft    a_j ← a_j·7^j, then fft
 *   inverse = 1, coset = 1 : coset_ifft   ifft, then a_j ← a_j·7^{-j}
 * Natural order in, natural order out.  Blocks until the result is in `data`. */
PB200_API int pb200_ntt(pb200_ctx *ctx, uint64_t *data_host, uint32_t log_n, int inverse, int coset);
/* Same transform on a DEVICE-resident vector, in place, ordered on the context stream (no sync). */
PB200_API int pb200_ntt_dev(pb200_ctx *ctx, uint64_t *data_dev, uint32_t log_n, int inverse, int coset);

/* `batch` independent transforms of 2^log_n scalars each, stored back to back in one device buffer, one launch per
 * pass for the whole batch (the prover transforms several wire polynomials per round; the sharded transform runs
 * its rows through this). */
PB200_API int pb200_ntt_batch_dev(pb200_ctx *ctx, uint64_t *data_dev, uint32_t log_n, uint32_t batch, int inverse, int coset);
/* Building blocks of the sharded four-step transform for domains ≥ 2^24 spread over G GPUs (SURVEY.md §8e): one
 * process per GPU owns a column range of the n1 × (n / n1) view; the host layer (plonk-prototype_b200/dist_ntt.py,
 * or the Rust shim with NCCL) runs  columns → all-to-all → block transpose → rows (pb200_ntt_dev per row).
 * pb200_ntt_columns_dev: in-place length-2^log_n1 (i)NTT down every column of the local 2^log_n1 × 2^log_cols
 * row-major matrix holding global columns [col_offset, col_offset + 2^log_cols), fused with the inter-step twiddle
 * ω_n^{±col·k} of the 2^log_n transform (forward: after the columns; inverse: before them, plus the 2^-log_n1 scale). */
PB200_API int pb200_ntt_columns_dev(pb200_ctx *ctx, uint64_t *data_dev, uint32_t log_n, uint32_t log_n1, uint32_t log_cols,
                                    uint32_t col_offset, int inverse);
/* Fused compute + exchange (forward direction): the same column step, but every output is stored straight into the
 * row-layout buffer of the rank that owns its row — peer memory over NVLink / NVSwitch — so the all-to-all and the
 * block transpose ARE the kernel's store and overlap its arithmetic tile by tile.  peer_row_bufs[h] is rank h's
 * receive buffer of (2^log_n1 / world) rows × (2^log_n / 2^log_n1) scalars (its own for h = this rank); remote ones
 * come from pb200_ipc_open.  The caller barriers all ranks before reading its buffer. */
PB200_API int pb200_ntt_columns_scatter_dev(pb200_ctx *ctx, uint64_t *data_dev, uint32_t log_n, uint32_t log_n1, uint32_t log_cols,
                                            uint32_t col_offset, uint32_t world, void *const *peer_row_bufs);
/* CUDA IPC plumbing for one-process-per-GPU hosts: export a pb200_malloc'ed buffer / map a peer's buffer. */
PB200_API int pb200_ipc_export(pb200_ctx *ctx, void *dev_ptr, unsigned char handle_out[64]);
PB200_API int pb200_ipc_open(pb200_ctx *ctx, const unsigned char handle[64], void **dev_ptr_out);
PB200_API int pb200_ipc_close(pb200_ctx *ctx, void *dev_ptr);
/* dst[(r·blocks + b)·cols + c] = src[(b·rows + r)·cols + c] on 32-byte scalars: regroups what an all-to-all delivered. */
PB200_API int pb200_block_transpose_dev(pb200_ctx *ctx, uint64_t *dst_dev, const uint64_t *src_dev, uint32_t blocks,
                                        uint32_t rows, uint32_t cols);

/* ---- MSM: dusk_bls12_381::multiscalar_mul::msm_variable_base (SURVEY.md §8a a12, App. B.1) ---- */
/* Upload bases once (CommitKey::powers_of_g); they stay resident for every later commit. */
PB200_API int pb200_srs_upload(pb200_ctx *ctx, const uint64_t *xy_mont_host, size_t n_points, pb200_srs **out);
/* Wrap bases that are already on the device (n_points × 96 B, not copied, not freed by srs_free). */
PB200_API int pb200_srs_wrap_dev(pb200_ctx *ctx, const uint64_t *xy_mont_dev, size_t n_points, pb200_srs **out);
/* Optional, once per SRS of at most 2^22 points: store the pre-doubled copies 2^(c·w)·P_i of every base so that
 * all Pippenger windows share one bucket set — no per-window reduction and no Horner pass, which is what bounds
 * prover-size (2^16…2^22) MSMs.  Costs W ≈ 12-13 times the SRS memory; results are unchanged. */
PB200_API int pb200_srs_precompute(pb200_ctx *ctx, pb200_srs *srs);
/* The commit key in the Lagrange basis of the domain of n = 2^log_n points: *out holds Q_i = [L_i(τ)]G = n⁻¹·Σ_j ω^(−ij)·P_j,
 * i < n, computed on the device from the first n points of `srs` (an inverse NTT over G1: no trapdoor needed), so that
 * Σ_i f(ω^i)·Q_i is the commitment to the polynomial f of degree < n from its evaluations.  log_n ≤ 26, n ≤ pb200_srs_len.
 * A key that is not powers of τ can give an identity point: PB200_ERR_ARG, nothing allocated.  Free with pb200_srs_free.
 * pb200_preprocess builds one for its domain itself (see there). */
PB200_API int pb200_srs_lagrange(pb200_ctx *ctx, const pb200_srs *srs, uint32_t log_n, pb200_srs **out);
PB200_API void pb200_srs_free(pb200_ctx *ctx, pb200_srs *srs);
PB200_API size_t pb200_srs_len(const pb200_srs *srs);
/* msm_variable_base(&points[offset .. offset + n], scalars): Σ scalars[i]·points[offset + i].
 * Scalars on the HOST; n = 0 or all-zero scalars give the identity.  Blocks; result on the host. */
PB200_API int pb200_msm_g1(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, const uint64_t *scalars_mont_host, size_t n,
                 uint64_t out_xyz_mont[18]);
/* Same with scalars already on the DEVICE (n × 32 B).  Blocks; result on the host. */
PB200_API int pb200_msm_g1_dev(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, const uint64_t *scalars_mont_dev, size_t n,
                     uint64_t out_xyz_mont[18]);
/* `batch` MSMs over the SAME bases in one pass — the shape of a prover round (four wire commitments, four quotient
 * parts, two opening witnesses): scalar vector j starts at scalars_mont_dev + 4·j·scalar_stride (scalar_stride ≥ n, in
 * scalars) and out_xyz_mont receives batch × 18 u64.  With pre-doubled copies (pb200_srs_precompute) every vector gets
 * its own bucket set and the sort, accumulation and reduction run once for all of them; otherwise the calls are made
 * one after the other.  Blocks; results on the host. */
PB200_API int pb200_msm_g1_batch_dev(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, const uint64_t *scalars_mont_dev, size_t n,
                                     uint32_t batch, size_t scalar_stride, uint64_t *out_xyz_mont);
/* dusk_bls12_381::multiscalar_mul::pippenger(points: impl Iterator<Item = G1Projective>, scalars: impl Iterator<Item =
 * Scalar>) -> G1Projective — the iterator form next to msm_variable_base in the same upstream file (crate pinned at
 * /root/reference/Cargo.toml:20; SURVEY.md §8a a13; no caller in the reference or in dusk-plonk's prover).  Bases in
 * homogeneous projective coordinates, n × (X ‖ Y ‖ Z) = n × 18 u64 Montgomery words on the HOST, Z = 0 for the identity;
 * scalars n × 4 u64 Montgomery.  The bases are normalised on the device (one inversion per eight points) and summed by the
 * same pipeline as pb200_msm_g1; the group element returned is the one upstream computes.  Blocks; result on the host. */
PB200_API int pb200_pippenger_g1(pb200_ctx *ctx, const uint64_t *points_xyz_mont_host, const uint64_t *scalars_mont_host, size_t n,
                                 uint64_t out_xyz_mont[18]);
/* Sum of `count` projective points (each X ‖ Y ‖ Z, 18 × u64 Montgomery, HOST memory) — the combine step after
 * a point-range-sharded MSM (SURVEY.md §8e): every rank's partial result is gathered and added here.
 * Output as for pb200_msm_g1. */
PB200_API int pb200_g1_sum(pb200_ctx *ctx, const uint64_t *points_xyz_mont_host, size_t count, uint64_t out_xyz_mont[18]);
/* Pippenger window width used for n points (exposed for the benches' work model). */
PB200_API uint32_t pb200_msm_window_bits(size_t n);

/* ---- KZG10 layer above the MSM: dusk_plonk::commitment_scheme::kzg10 (SURVEY.md §2.2 D5, §8f-1) ---------------- */
/* PublicParameters::setup: powers_of_g[i] = τ^i·G for i < n_points, generated on the device and resident (τ given
 * in Montgomery form, non-zero; the G2 side of the parameters belongs to the host verifier). */
PB200_API int pb200_srs_generate(pb200_ctx *ctx, const uint64_t tau_mont[4], size_t n_points, pb200_srs **out);
/* The slice powers_of_g[first .. first + n_points) of the same parameters: what one rank of a point-range-sharded
 * prover holds (SURVEY.md §8e). */
PB200_API int pb200_srs_generate_range(pb200_ctx *ctx, const uint64_t tau_mont[4], size_t first, size_t n_points, pb200_srs **out);
/* Device address of an SRS's packed affine points (n × 96 B), e.g. to serialise the CommitKey. */
PB200_API const uint64_t *pb200_srs_dev_ptr(const pb200_srs *srs);
/* Per-point result of G1Affine::from_bytes on a 48-byte compressed (zcash) encoding. */
enum {
    PB200_G1_OK = 0,
    PB200_G1_BAD_FLAGS = 1,       /* bit 7 clear, or bit 6 (identity) set on anything but c0 00…00 */
    PB200_G1_X_RANGE = 2,         /* x ≥ p */
    PB200_G1_NOT_ON_CURVE = 3,    /* x³ + 4 is not a square */
    PB200_G1_NOT_IN_SUBGROUP = 4, /* on the curve, outside the prime-order subgroup */
    PB200_G1_IDENTITY = 5         /* the canonical identity encoding: valid upstream, not representable here */
};
/* CommitKey::from_slice over a whole key (G1Affine::from_bytes per point): n_points 48-byte compressed encodings on the HOST
 * are decoded and checked on the device (flags, x < p, on the curve, prime-order subgroup) and kept resident as an SRS in the
 * layout of pb200_srs_upload.  Any invalid point: PB200_ERR_ARG, pb200_last_error names the first invalid index and its
 * reason, *out is left untouched and nothing stays allocated.  status_host (optional, n_points bytes): PB200_G1_* per point.
 * The identity encoding is rejected (PB200_G1_IDENTITY): the ABI cannot hold it and a commit key never contains it.
 * 1 ≤ n_points < 2^31.  A rank of a point-range-sharded prover loads its slice powers_of_g[first .. first + n) by passing
 * bytes_host + 48·first and n: the encoding has no prefix, so no other entry point is needed.  Blocks. */
PB200_API int pb200_srs_from_compressed(pb200_ctx *ctx, const uint8_t *bytes_host, size_t n_points, uint8_t *status_host,
                                        pb200_srs **out);
/* CommitKey::to_var_bytes: points [offset, offset + n) of an SRS as 48-byte compressed encodings, 48·n bytes on the HOST.
 * 1 ≤ n < 2^31 and the range must lie inside the SRS.  Blocks. */
PB200_API int pb200_srs_to_compressed(pb200_ctx *ctx, const pb200_srs *srs, size_t offset, size_t n, uint8_t *bytes_host);
/* CommitKey::compute_single_witness: p(z) and q(X) = (p(X) − p(z)) / (X − z) for a device-resident polynomial of
 * n coefficients (Ruffini's rule as scale → Fr suffix scan → scale).  quotient_dev receives n scalars (the top one
 * is zero).  Blocks; p(z) is returned on the host. */
PB200_API int pb200_kzg_witness_dev(pb200_ctx *ctx, const uint64_t *poly_dev, size_t n, const uint64_t z_mont[4],
                                    uint64_t *quotient_dev, uint64_t eval_mont_out[4]);
/* One Horner step over whole polynomials, acc[j] ← acc[j]·c + poly[j] (poly zero-padded to n_acc): the
 * random-linear-combination Σ vⁱ·pᵢ of CommitKey::compute_aggregate_witness. */
PB200_API int pb200_fr_horner_step_dev(pb200_ctx *ctx, uint64_t *acc_dev, size_t n_acc, const uint64_t *poly_dev, size_t n_poly,
                                       const uint64_t c_mont[4]);

/* ---- PLONK prover rounds above the hot path: dusk_plonk::proof_system::Prover (SURVEY.md §3.2-3.3, §8f-2/3) --------- */
typedef struct pb200_prover_key pb200_prover_key;
/* The constraint system as StandardComposer holds it after circuit synthesis (the reference's gadgets,
 * /root/reference/src/zk/gadgets.rs:28-225, only append rows to these vectors):  n_gates rows; 11 selector columns in
 * the order q_m q_l q_r q_o q_c q_4 q_arith q_range q_logic q_fixed_group_add q_variable_group_add, each n_gates
 * Montgomery scalars (NULL = all zero); 4 wire columns w_l w_r w_o w_4 holding the `Variable` index of each row. */
typedef struct pb200_circuit {
    size_t n_gates;
    size_t n_vars;
    const uint64_t *selectors[11];
    const uint32_t *wires[4];
} pb200_circuit;
/* Prover::preprocess: pads to n = next power of two, interpolates and commits the 11 selector and 4 permutation
 * polynomials (15 iNTT + 15 MSM), extends them to the 4n coset (15 coset NTTs), and seeds Transcript::new(label) with
 * the verifier key.  Everything stays resident in HBM behind the returned handle.  vk_commitments (optional) receives
 * the 15 compressed commitments in the column order above followed by left/right/out/fourth sigma.
 * Widgets: arithmetic, range, logic, fixed-base scalar multiplication and variable-base point addition on JubJub (all
 * eleven selector columns of StandardComposer).
 * On one GPU, with n ≤ 2^22 and a commit key that has pre-doubled copies (pb200_srs_precompute), the key also holds the
 * Lagrange-basis key of its domain (pb200_srs_lagrange) with its own pre-doubled copies — (W + 1)·n·96 bytes, 1.3 GiB at
 * n = 2^20 — and pb200_prove commits the wire polynomials from their evaluations, whose zero and small values cost almost
 * nothing in the MSM.  The proof bytes are the same.  Environment PB200_LAGRANGE_COMMIT=0, read here, leaves it out. */
PB200_API int pb200_preprocess(pb200_ctx *ctx, const pb200_srs *srs, const pb200_circuit *circuit, const uint8_t *transcript_label,
                               size_t label_len, pb200_prover_key **out, uint8_t vk_commitments[15 * 48]);
PB200_API void pb200_prover_key_free(pb200_ctx *ctx, pb200_prover_key *pk);
PB200_API size_t pb200_prover_key_size(const pb200_prover_key *pk);  /* padded circuit size n */
PB200_API size_t pb200_prover_key_bytes(const pb200_prover_key *pk); /* device memory held */
/* Point-range-sharded proving over `world` GPUs, one process per GPU (SURVEY.md §8e; BASELINE.json configs[4]): every
 * commitment of preprocessing and of the five rounds is an MSM over this rank's slice of the commit key
 * (powers_of_g[rank·n/world .. (rank+1)·n/world), see pb200_srs_generate_range) against the matching coefficient slice;
 * the `world` partial sums (144 bytes each) are exchanged through `allgather` — the host's NCCL / gloo all-gather —
 * and added, so every rank derives the same transcript challenges and returns the same proof.  NTTs and pointwise
 * kernels run replicated on every rank (they are ~15 % of a single-GPU prove).  The callback receives `bytes` bytes in
 * `send` and must fill `recv` with world × bytes, rank-major; non-zero return aborts the call. */
typedef int (*pb200_allgather_fn)(void *user, const void *send, void *recv, size_t bytes);
/* Optional device-memory collectives (NCCL over NVLink).  When both are given, round 3 — seven coset transforms of 4n
 * points, the quotient kernel and the inverse transform — is sharded too: four-step transforms with this rank owning a
 * column range of the coefficient side and a row range of the evaluation side (one all-to-all each, as in
 * pb200_ntt_columns_dev), the quotient evaluated on the local rows, and one all-gather of t(X)'s coefficient shards.
 * With up to 8 ranks on one NVLink domain the forward exchange is not a collective at all: the keys' device memory is
 * mapped into every peer with CUDA IPC (handles travel through `allgather`) and pb200_ntt_columns_scatter_dev stores each
 * output straight into its owner's row buffer — transfer and transpose overlap the column arithmetic tile by tile; only the
 * inverse transform and the final all-gather use the callbacks below.  Free sharded keys on all ranks together.
 * alltoall_dev: block h (bytes_per_peer bytes) of send_dev goes to rank h, block b of recv_dev comes from rank b.
 * allgather_dev: recv_dev = world × bytes, rank-major.  Both must have completed when they return. */
typedef int (*pb200_alltoall_dev_fn)(void *user, const void *send_dev, void *recv_dev, size_t bytes_per_peer);
typedef int (*pb200_allgather_dev_fn)(void *user, const void *send_dev, void *recv_dev, size_t bytes);
typedef struct pb200_shard {
    uint32_t rank, world;
    pb200_allgather_fn allgather;
    void *user;
    pb200_alltoall_dev_fn alltoall_dev;   /* may be NULL: NTTs and the quotient kernel then run replicated */
    pb200_allgather_dev_fn allgather_dev; /* may be NULL */
    uint32_t flags;                       /* PB200_SHARD_* */
} pb200_shard;
/* The device collectives are enqueued on the context's own stream (pb200_stream): the library then neither synchronises
 * the stream before calling them nor assumes they have completed on return, and uses a stream-ordered collective as its
 * cross-rank barrier.  Set by pb200_preprocess_comm; host-language callbacks that run on another stream leave it clear. */
#define PB200_SHARD_STREAM_ORDERED 1u
/* As pb200_preprocess, with `srs` holding this rank's slice.  The shard description is kept in the key: pb200_prove on a
 * sharded key must be given the same slice and is collective over all ranks. */
PB200_API int pb200_preprocess_sharded(pb200_ctx *ctx, const pb200_srs *srs_slice, const pb200_circuit *circuit,
                                       const uint8_t *transcript_label, size_t label_len, const pb200_shard *shard,
                                       pb200_prover_key **out, uint8_t vk_commitments[15 * 48]);
/* ---- multi-GPU communicator inside the library (SURVEY.md §8b, §8e): one process per GPU, NCCL over NVLink / NVSwitch.
 * Rank 0 obtains a 128-byte id (ncclUniqueId) and the host distributes it by any means; every rank then binds a
 * communicator to its context.  All collectives below run on the context's stream.  NCCL is resolved at run time
 * (libnccl.so.2 — the copy the host process already loaded, or the system's): PB200_ERR_NO_DEVICE when it cannot be. */
PB200_API int pb200_comm_unique_id(unsigned char id_out[128]);
PB200_API int pb200_comm_init(pb200_ctx *ctx, const unsigned char id[128], uint32_t rank, uint32_t world);
PB200_API int pb200_comm_destroy(pb200_ctx *ctx);
PB200_API int pb200_comm_info(const pb200_ctx *ctx, uint32_t *rank, uint32_t *world);
/* recv_dev = world × bytes, rank-major | block h of send_dev → rank h, block b of recv_dev ← rank b.  Stream-ordered. */
PB200_API int pb200_allgather_dev(pb200_ctx *ctx, const void *send_dev, void *recv_dev, size_t bytes);
PB200_API int pb200_alltoall_dev(pb200_ctx *ctx, const void *send_dev, void *recv_dev, size_t bytes_per_peer);
/* msm_variable_base over a point-range-sharded commit key (SURVEY.md §8e): this rank's slice against its scalars, the
 * 144-byte partial results all-gathered and summed; every rank receives the total.  Blocks; result on the host. */
PB200_API int pb200_msm_g1_sharded_dev(pb200_ctx *ctx, const pb200_srs *srs_slice, size_t offset, const uint64_t *scalars_mont_dev, size_t n,
                                       uint64_t out_xyz_mont[18]);
/* EvaluationDomain::fft / ifft of ONE 2^log_n vector sharded over the communicator's ranks (SURVEY.md §8e, domains ≥ 2^24):
 * four-step, n = n1·m with n1 = 2^8.  Forward: `data` holds this rank's column-layout shard A[j1][c] = x[j1·m + rank·m/G + c]
 * and receives its row-layout shard B[r][k'] = X[(rank·n1/G + r) + n1·k']; inverse: the way back (with n⁻¹).  `tmp`: a
 * second buffer of 2^log_n / G scalars.  One all-to-all; stream-ordered, no host synchronisation. */
PB200_API int pb200_ntt_sharded_dev(pb200_ctx *ctx, uint64_t *data_dev, uint64_t *tmp_dev, uint32_t log_n, int inverse);
/* pb200_preprocess_sharded with the context's communicator supplying every collective (no host callbacks). */
PB200_API int pb200_preprocess_comm(pb200_ctx *ctx, const pb200_srs *srs_slice, const pb200_circuit *circuit, const uint8_t *transcript_label,
                                    size_t label_len, pb200_prover_key **out, uint8_t vk_commitments[15 * 48]);

/* Prover::prove_with_preprocessed + Proof::to_bytes: the witness is the value of every variable (n_vars Montgomery
 * scalars, host), the public inputs a sparse (gate index, value) list.  Rounds 1-5 run on the device with the
 * polynomials resident between rounds; the host hashes the transcript.  proof_out: 11 compressed G1 + 16 scalars.
 * With profiling on, pb200_profile_ms knows "prove.round1" … "prove.round5" (host wall-clock per round). */
PB200_API int pb200_prove(pb200_ctx *ctx, const pb200_srs *srs, pb200_prover_key *pk, const uint64_t *values_mont,
                          const uint32_t *pi_gate, const uint64_t *pi_mont, size_t n_pi, uint8_t proof_out[1040]);
/* The same with the witness already in DEVICE memory (n_vars × 32 B, e.g. produced by a GPU witness generator or
 * uploaded once with pb200_h2d): no bulk host→device copy inside the call.  Public inputs and the proof stay on the
 * host (a few hundred bytes).  A gate index may appear at most once in pi_gate (both entry points; PB200_ERR_ARG). */
PB200_API int pb200_prove_dev(pb200_ctx *ctx, const pb200_srs *srs, pb200_prover_key *pk, const uint64_t *values_mont_dev,
                              const uint32_t *pi_gate, const uint64_t *pi_mont, size_t n_pi, uint8_t proof_out[1040]);
/* ---- verifier (host CPU, as upstream's): dusk_plonk Proof::verify + OpeningKey::batch_check + the BLS12-381 pairing of
 * dusk_bls12_381 (SURVEY.md §3.6, §8f-4).  No context and no GPU: the work is milliseconds and independent of n. ------- */
/* vk_commitments: the 15 compressed commitments pb200_preprocess returns; n: padded circuit size; public inputs as for
 * pb200_prove; beta_h: the opening key's β·H ∈ G2, affine x.c0 ‖ x.c1 ‖ y.c0 ‖ y.c1 (4 × 6 u64, Montgomery).
 * Returns 0 with *accepted = 1 / 0 (a malformed proof is a rejection, not an error); PB200_ERR_ARG for a null pointer, n not
 * a power of two in [2, 2^30], a duplicate pi_gate, pi_gate[j] ≥ n or β·H not on the curve — all checked before any proof
 * byte is looked at, so a bad argument is reported whatever the proof holds. */
PB200_API int pb200_verify(const uint8_t vk_commitments[15 * 48], size_t n, const uint8_t *transcript_label, size_t label_len,
                           const uint8_t proof[1040], const uint32_t *pi_gate, const uint64_t *pi_mont, size_t n_pi,
                           const uint64_t beta_h[24], int *accepted);
/* Many proofs of ONE circuit in one batched check on the GPU (dusk-plonk 0.8 has no multi-proof API; this is the
 * standard random-linear-combination batch of Proof::verify).  One verifier key, label and padded size n as for
 * pb200_verify; proofs: n_proofs × 1040 bytes back to back; pi_gate (n_pi entries) is shared by every proof and
 * pi_mont holds n_proofs × n_pi × 4 u64 Montgomery values, proof-major.
 *   accepted[k] (out, n_proofs bytes) = what pb200_verify returns for proof k with its public inputs: a valid proof is
 *   never rejected; an invalid one is accepted with probability about 1/r per pairing check.  *all_accepted = 1 iff
 *   every accepted[k] is 1.  Verdicts are deterministic for a given seed (32 bytes; callers draw it at random).
 * Errors: PB200_ERR_ARG for a null pointer (seed included), n not a power of two in [2, 2^30], a duplicate pi_gate,
 *   pi_gate[j] ≥ n, β·H not on the curve, n_proofs = 0 or n_proofs > 2^20 — all checked before any proof is looked at.
 *   A malformed verifier key rejects every proof (not an error).  A proof with a point that fails G1Affine::from_bytes, an
 *   evaluation ≥ r, z_H(z) = 0, z = 1 or z = ω^g for a public-input gate g is rejected and left out of the combination.
 *   The identity encoding c0 00…00 is a valid proof point and contributes zero.  Nothing stays allocated on return.
 * Algorithm: each proof's equation e(−W_k, βH)·e(C_k, H) = 1 has C_k, W_k linear in its 11 points and in 16 shared
 *   bases (the 15 key commitments and G), with scalars from its own transcript (derived on the device, one thread per
 *   proof).  Weights: per proof, after the transcript's challenge u, its public inputs are appended ("pi", one scalar
 *   each) and 32 bytes drawn ("batch digest") = d_k; on the host D = Merlin("pb200 verify_batch") absorbing seed, n,
 *   n_proofs and d_0‖…‖d_{K−1} ("seed", "n", "K", "digests"; challenge "D"); ρ_k = Merlin("pb200 rho") absorbing D ("D")
 *   and k ("k"), challenge scalar "rho".  Then e(−Σρ_kW_k, βH)·e(Σρ_kC_k, H) = 1 is one pairing check on the host over
 *   two MSMs on the device.  If it fails, bisection over contiguous proof ranges (same ρ_k) finds the invalid proofs:
 *   an all-valid batch costs exactly one pairing check, b invalid proofs at most about 1 + 2·b·⌈log2 K⌉.
 * With profiling on, pb200_profile_sum_ms knows "verify.decompress", "verify.prepare", "verify.weight" (kernel time),
 *   "verify.msm" (device time of the call's MSMs) and "verify.pairing" (host wall clock, one sample per pairing check).
 * Blocks. */
PB200_API int pb200_verify_batch(pb200_ctx *ctx, const uint8_t vk_commitments[15 * 48], size_t n, const uint8_t *transcript_label,
                                 size_t label_len, const uint8_t *proofs, size_t n_proofs, const uint32_t *pi_gate, const uint64_t *pi_mont,
                                 size_t n_pi, const uint64_t beta_h[24], const uint8_t seed[32], uint8_t *accepted, int *all_accepted);
/* β·H for parameters generated from a known trapdoor (pb200_srs_generate): the G2 half of PublicParameters::setup. */
PB200_API int pb200_opening_key_from_tau(const uint64_t tau_mont[4], uint64_t beta_h_out[24]);
/* Pairing self-check without a known-answer table: e(a·G1, b·G2) = e(G1, G2)^(ab) ≠ 1. */
PB200_API int pb200_pairing_selftest(const uint64_t a_mont[4], const uint64_t b_mont[4], int *ok);
/* merlin::Transcript known-answer hook: Transcript::new(label); append_message(msg_label, msg); challenge_bytes(ch_label). */
PB200_API int pb200_transcript_selftest(const char *label, const char *msg_label, const uint8_t *msg, size_t msg_len,
                                        const char *challenge_label, uint8_t *out, size_t out_len);

/* ---- synthetic workloads & measurement helpers (bench.py / tests; SURVEY.md §8d) -------------- */
/* bases[i] = (a + i·d)·G, packed affine Montgomery, written to a device buffer of n × 96 B. */
PB200_API int pb200_synthetic_bases_dev(pb200_ctx *ctx, uint64_t *xy_mont_dev, size_t n, uint64_t a, uint64_t d);
/* The synthetic arithmetic circuit of SURVEY.md §8d (chain x ← x·x + x + c from mul / add rows, boolean padding, n_pub
 * public-input rows) written into caller-allocated column images: selectors7 = q_m q_l q_r q_o q_c q_4 q_arith (n_gates × 4
 * u64 each), wires (n_gates u32 each), values (n_vars × 4 u64; n_vars = 6 + 2·⌊(n_gates − n_pub − 3)/2⌋ + n_pub − 1),
 * pi_gate / pi_mont (n_pub entries).  Host-side helper for benches and tests; no GPU involved. */
PB200_API int pb200_synthetic_circuit(size_t n_gates, uint64_t seed, uint32_t n_pub, uint64_t *const selectors7[7], uint32_t *const wires[4],
                                      uint64_t *values_mont, size_t n_vars_capacity, size_t *n_vars_out, uint32_t *pi_gate,
                                      uint64_t *pi_mont);
/* Per-kernel device time of the most recent MSM / NTT call, from CUDA events on the context stream.
 * Known names: "msm.accumulate", "msm.sort", "msm.reduce", "msm.total", "ntt.total", and "srs.decompress" / "srs.compress"
 * (the kernels of pb200_srs_from_compressed / pb200_srs_to_compressed).
 * Profiling must have been switched on before that call. */
PB200_API int pb200_profile_enable(pb200_ctx *ctx, int on);
PB200_API int pb200_profile_ms(pb200_ctx *ctx, const char *name, float *ms);
/* Every collected duration is also accumulated per name: pb200_profile_sum_ms returns the sum (and, optionally, the
 * number of samples) since the last pb200_profile_reset — e.g. the total msm_accumulate_kernel time of one pb200_prove,
 * which makes 11 MSM calls.  An unknown name reads as 0 ms / 0 samples. */
PB200_API int pb200_profile_reset(pb200_ctx *ctx);
PB200_API int pb200_profile_sum_ms(pb200_ctx *ctx, const char *name, float *ms, uint32_t *count);
/* Number of kernels this library has launched on the context since init (bench.py's gpu_launches). */
PB200_API uint64_t pb200_launch_count(const pb200_ctx *ctx);
/* Integer-pipe microbenchmark: sustained IMAD.WIDE.U32.X (32×32+64 with carry) lane-operations per second
 * over the whole chip — the denominator of the MSM / NTT integer rooflines (DESIGN.md).  The second output
 * is that rate expressed as an SM clock assuming 32 lane-ops/clk/SM (the measured issue rate). */
PB200_API int pb200_imad_peak(pb200_ctx *ctx, double *wide_lane_ops_per_s, double *sm_clock_mhz_est);

#ifdef __cplusplus
}
#endif
#endif /* PB200_H */
