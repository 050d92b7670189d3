// Host-emulation harness for the Lagrange-basis commit key (csrc/lagrange.cuh, the code lagrange_load_kernel,
// lagrange_stage_kernel and lagrange_normalize_kernel run), compiled for the CPU with the carry-flag primitives emulated
// (PB200_HOST_EMU), behind a C ABI for pytest.  The launch sequence and its constants mirror lagrange_srs_build
// (csrc/lagrange.cu): one thread index at a time instead of one thread each.
#define PB200_HOST_EMU 1
#include "../../plonk-prototype_b200/csrc/host_field.h"
#include "../../plonk-prototype_b200/csrc/lagrange.cuh"
#include <cstring>
#include <vector>

namespace {
Fr to_fr(const hostf::HFr &a) {
    Fr r;
    memcpy(r.l, a.l, 32);
    return r;
}
}  // namespace

extern "C" {
// 2^log_n affine points (24 u32 Montgomery each: x ‖ y) → their Lagrange-basis key in the same layout.
// Returns 1 when a point came out as the identity (written as zeros), else 0.
int emu_lagrange(const uint32_t *bases_xy, uint32_t log_n, uint32_t *out_xy) {
    const uint32_t n = 1u << log_n;
    std::vector<G1Affine> in(n), out(n);
    std::vector<G1Xyzz> a(n);
    memcpy(in.data(), bases_xy, (size_t)n * 96);
    for (uint32_t i = 0; i < n; i++) lagrange::load_point(in.data(), i, log_n, a.data());
    const hostf::HFr w_inv = hostf::domain_root(log_n).inv();
    for (uint32_t half = 1; half < n; half <<= 1) {
        const Fr w = to_fr(w_inv.pow_u64(n / (2 * half)));
        for (uint32_t k = 0; k < n / 2; k++) lagrange::butterfly(a.data(), half, k, w);
    }
    uint32_t degenerate = 0;
    const Fr n_inv = to_fr(hostf::HFr::from_u64(n).inv());
    for (uint32_t i0 = 0; i0 < n; i0 += lagrange::kNormPer)
        lagrange::normalize(a.data(), i0, n - i0 < lagrange::kNormPer ? n - i0 : lagrange::kNormPer, n_inv, out.data(), &degenerate);
    memcpy(out_xy, out.data(), (size_t)n * 96);
    return (int)degenerate;
}
}
