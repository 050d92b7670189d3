// merlin.h — Merlin transcripts (STROBE-128 over Keccak-f[1600]) with dusk-plonk's TranscriptProtocol helpers.
//
// Replaces the `merlin` crate (transitive dependency of dusk-plonk 0.8.2, /root/reference/Cargo.toml:19) and
// dusk-plonk's `transcript.rs` (SURVEY.md §8f-3, App. B.3) on the host: Fiat–Shamir challenges are a few hundred
// bytes of hashing per proof and stay on the CPU.  Pinned by Merlin's own known-answer vector
// (tests/test_prover_cpu.py): protocol "test protocol", message ("some label", "some data"), 32 challenge bytes
// d5a21972d0d5fe32…efcf0615.
//
// The same code runs on the device (csrc/verify_batch.cu derives every proof's challenges in its own thread): everything
// is MERLIN_HD, the constant tables are constexpr functions both sides can read, and the scalar conversions are generic
// over the field type — found by argument-dependent lookup as scalar_to_bytes(s, out) / scalar_from_bytes_wide(in, out),
// defined for hostf::HFr below and for the device's Fr in verify_batch.cuh.
#pragma once
#include <stdint.h>
#include <string.h>

#include "host_field.h"

#if defined(__CUDACC__)
#define MERLIN_HD __host__ __device__ __forceinline__
#define MERLIN_EXEC_CHECK_DISABLE _Pragma("nv_exec_check_disable")
#define MERLIN_UNROLL(n) _Pragma(#n)
#else
#define MERLIN_HD inline
#define MERLIN_EXEC_CHECK_DISABLE
#define MERLIN_UNROLL(n)
#endif

namespace hostf {
inline void scalar_to_bytes(const HFr &s, uint8_t out[32]) { fr_to_bytes(s, out); }
inline void scalar_from_bytes_wide(const uint8_t in[64], HFr &out) { out = fr_from_bytes_wide(in); }
}  // namespace hostf

namespace merlin {

MERLIN_HD uint64_t rotl64(uint64_t v, int n) { return n ? (v << n) | (v >> (64 - n)) : v; }

MERLIN_HD constexpr uint64_t keccak_rc(int i) {
    constexpr uint64_t RC[24] = {
        0x0000000000000001ull, 0x0000000000008082ull, 0x800000000000808aull, 0x8000000080008000ull, 0x000000000000808bull,
        0x0000000080000001ull, 0x8000000080008081ull, 0x8000000000008009ull, 0x000000000000008aull, 0x0000000000000088ull,
        0x0000000080008009ull, 0x000000008000000aull, 0x000000008000808bull, 0x800000000000008bull, 0x8000000000008089ull,
        0x8000000000008003ull, 0x8000000000008002ull, 0x8000000000000080ull, 0x000000000000800aull, 0x800000008000000aull,
        0x8000000080008081ull, 0x8000000000008080ull, 0x0000000080000001ull, 0x8000000080008008ull};
    return RC[i];
}
// ρ offsets and π destinations walked along the single 24-cycle of π starting at lane 1
MERLIN_HD constexpr int keccak_rho(int i) {
    constexpr int RHO[24] = {1, 3, 6, 10, 15, 21, 28, 36, 45, 55, 2, 14, 27, 41, 56, 8, 25, 43, 62, 18, 39, 61, 20, 44};
    return RHO[i];
}
MERLIN_HD constexpr int keccak_pi(int i) {
    constexpr int PI[24] = {10, 7, 11, 17, 18, 3, 5, 16, 8, 21, 24, 4, 15, 23, 19, 13, 12, 2, 20, 14, 22, 9, 6, 1};
    return PI[i];
}

// The loops inside a round are unrolled so that every lane index is a constant (the state stays in registers on the
// device); the 24 rounds are not (code size).
MERLIN_HD void keccak_f1600(uint64_t s[25]) {
MERLIN_UNROLL(unroll 1)
    for (int round = 0; round < 24; round++) {
        uint64_t c[5];
MERLIN_UNROLL(unroll)
        for (int x = 0; x < 5; x++) c[x] = s[x] ^ s[x + 5] ^ s[x + 10] ^ s[x + 15] ^ s[x + 20];
MERLIN_UNROLL(unroll)
        for (int x = 0; x < 5; x++) {
            uint64_t d = c[(x + 4) % 5] ^ rotl64(c[(x + 1) % 5], 1);
MERLIN_UNROLL(unroll)
            for (int y = 0; y < 25; y += 5) s[y + x] ^= d;
        }
        uint64_t cur = s[1];
MERLIN_UNROLL(unroll)
        for (int i = 0; i < 24; i++) {
            uint64_t nxt = s[keccak_pi(i)];
            s[keccak_pi(i)] = rotl64(cur, keccak_rho(i));
            cur = nxt;
        }
MERLIN_UNROLL(unroll)
        for (int y = 0; y < 25; y += 5) {
            uint64_t row[5];
MERLIN_UNROLL(unroll)
            for (int x = 0; x < 5; x++) row[x] = s[y + x];
MERLIN_UNROLL(unroll)
            for (int x = 0; x < 5; x++) s[y + x] = row[x] ^ (~row[(x + 1) % 5] & row[(x + 2) % 5]);
        }
        s[0] ^= keccak_rc(round);
    }
}
MERLIN_HD size_t cstr_len(const char *s) {
    size_t n = 0;
    while (s[n]) n++;
    return n;
}

class Strobe128 {
  public:
    MERLIN_HD explicit Strobe128(const char *protocol) {
        memset(st_, 0, sizeof(st_));
        const uint8_t head[6] = {1, kRate + 2, 1, 0, 1, 96};
        memcpy(st_, head, 6);
        memcpy(st_ + 6, "STROBEv1.0.2", 12);
        permute();
        meta_ad((const uint8_t *)protocol, cstr_len(protocol), false);
    }
    MERLIN_HD void meta_ad(const uint8_t *d, size_t n, bool more) {
        begin_op(kM | kA, more);
        absorb(d, n);
    }
    MERLIN_HD void ad(const uint8_t *d, size_t n, bool more) {
        begin_op(kA, more);
        absorb(d, n);
    }
    MERLIN_HD void prf(uint8_t *out, size_t n) {
        begin_op(kI | kA | kC, false);
        for (size_t i = 0; i < n; i++) {
            out[i] = st_[pos_];
            st_[pos_] = 0;
            if (++pos_ == kRate) run_f();
        }
    }

  private:
    static constexpr uint8_t kRate = 166;
    static constexpr uint8_t kI = 1, kA = 2, kC = 4, kT = 8, kM = 16, kK = 32;
    uint8_t st_[200];
    uint8_t pos_ = 0, pos_begin_ = 0, cur_flags_ = 0;

    MERLIN_HD void permute() {  // little-endian host (x86-64 / aarch64): the byte state aliases the 25 lanes
        uint64_t lanes[25];
        memcpy(lanes, st_, 200);
        keccak_f1600(lanes);
        memcpy(st_, lanes, 200);
    }
    MERLIN_HD void run_f() {
        st_[pos_] ^= pos_begin_;
        st_[pos_ + 1] ^= 0x04;
        st_[kRate + 1] ^= 0x80;
        permute();
        pos_ = 0;
        pos_begin_ = 0;
    }
    MERLIN_HD void absorb(const uint8_t *d, size_t n) {
        for (size_t i = 0; i < n; i++) {
            st_[pos_] ^= d[i];
            if (++pos_ == kRate) run_f();
        }
    }
    MERLIN_HD void begin_op(uint8_t flags, bool more) {
        if (more) return;  // continuation of the current operation (same flags by construction)
        const uint8_t old_begin = pos_begin_;
        pos_begin_ = pos_ + 1;
        cur_flags_ = flags;
        const uint8_t hdr[2] = {old_begin, flags};
        absorb(hdr, 2);
        if ((flags & (kC | kK)) && pos_ != 0) run_f();
    }
};

class Transcript {
  public:
    MERLIN_HD Transcript(const uint8_t *label, size_t n) : strobe_("Merlin v1.0") { append_message("dom-sep", label, n); }
    MERLIN_HD void append_message(const char *label, const uint8_t *msg, size_t n) {
        uint8_t len[4] = {(uint8_t)n, (uint8_t)(n >> 8), (uint8_t)(n >> 16), (uint8_t)(n >> 24)};
        strobe_.meta_ad((const uint8_t *)label, cstr_len(label), false);
        strobe_.meta_ad(len, 4, true);
        strobe_.ad(msg, n, false);
    }
    MERLIN_HD void append_u64(const char *label, uint64_t v) {
        uint8_t b[8];
        for (int k = 0; k < 8; k++) b[k] = (uint8_t)(v >> (8 * k));
        append_message(label, b, 8);
    }
    MERLIN_HD void challenge_bytes(const char *label, uint8_t *out, size_t n) {
        uint8_t len[4] = {(uint8_t)n, (uint8_t)(n >> 8), (uint8_t)(n >> 16), (uint8_t)(n >> 24)};
        strobe_.meta_ad((const uint8_t *)label, cstr_len(label), false);
        strobe_.meta_ad(len, 4, true);
        strobe_.prf(out, n);
    }
    // ---- dusk-plonk TranscriptProtocol
    MERLIN_HD void append_commitment(const char *label, const uint8_t compressed[48]) { append_message(label, compressed, 48); }
    // F is hostf::HFr on the host and the device's Fr in kernels: the conversion each one calls lives on its own side.
    MERLIN_EXEC_CHECK_DISABLE
    template <class F>
    MERLIN_HD void append_scalar(const char *label, const F &s) {
        uint8_t b[32];
        scalar_to_bytes(s, b);
        append_message(label, b, 32);
    }
    MERLIN_EXEC_CHECK_DISABLE
    template <class F = hostf::HFr>
    MERLIN_HD F challenge_scalar(const char *label) {
        uint8_t b[64];
        challenge_bytes(label, b, 64);
        F r;
        scalar_from_bytes_wide(b, r);
        return r;
    }
    MERLIN_HD void circuit_domain_sep(uint64_t n) {
        append_message("dom-sep", (const uint8_t *)"circuit_size", 12);
        append_u64("n", n);
    }

  private:
    Strobe128 strobe_;
};

// VerifierKey::seed_transcript.  vk: the 15 compressed commitments in the library's order (q_m q_l q_r q_o q_c q_4
// q_arith q_range q_logic q_fixed_group_add q_variable_group_add σ1 σ2 σ3 σ4); upstream absorbs the variable-base selector
// before the fixed-base one (SURVEY.md App. B.3).  The prover and both verifiers seed their transcripts here.
inline void seed_transcript(Transcript &tr, const uint8_t vk[15 * 48], uint64_t n) {
    const char *const label[11] = {"q_m", "q_l", "q_r", "q_o", "q_c", "q_4", "q_arith", "q_range", "q_logic", "q_variable_group_add",
                                   "q_fixed_group_add"};
    const int idx[11] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 10, 9};
    for (int k = 0; k < 11; k++) tr.append_commitment(label[k], vk + 48 * idx[k]);
    const char *const sigma[4] = {"left_sigma", "right_sigma", "out_sigma", "fourth_sigma"};
    for (int c = 0; c < 4; c++) tr.append_commitment(sigma[c], vk + 48 * (11 + c));
    tr.circuit_domain_sep(n);
}

}  // namespace merlin
