// Host-emulation harness for the compressed-point codec (csrc/g1_codec.cuh): the decoder and encoder the srs_io kernels
// inline, compiled for the CPU with the carry-flag primitives emulated (PB200_HOST_EMU), behind a C ABI for pytest.
#define PB200_HOST_EMU 1
#include "../../plonk-prototype_b200/csrc/g1_codec.cuh"
#include <cstddef>
#include <cstring>

extern "C" {
// n encodings of 48 bytes → status per point and, for PB200_G1_OK, the packed affine point (x ‖ y, 24 u32 Montgomery);
// the point of an invalid encoding is left zero.
void emu_g1_decode(const uint8_t *bytes, size_t n, uint32_t *out_xy, uint8_t *status) {
    for (size_t i = 0; i < n; i++) {
        G1Affine p;
        const int st = g1_decode_checked(bytes + 48 * i, p);
        status[i] = (uint8_t)st;
        if (st == PB200_G1_OK) {
            memcpy(out_xy + 24 * i, p.x.l, 48);
            memcpy(out_xy + 24 * i + 12, p.y.l, 48);
        } else {
            memset(out_xy + 24 * i, 0, 96);
        }
    }
}
// n packed affine points (24 u32 Montgomery each) → 48-byte encodings.
void emu_g1_encode(const uint32_t *xy, size_t n, uint8_t *out) {
    for (size_t i = 0; i < n; i++) {
        G1Affine p;
        memcpy(p.x.l, xy + 24 * i, 48);
        memcpy(p.y.l, xy + 24 * i + 12, 48);
        g1_encode(p, out + 48 * i);
    }
}
// n packed affine points on the curve → 1 if the endomorphism test puts them in the prime-order subgroup.
void emu_g1_in_subgroup(const uint32_t *xy, size_t n, uint8_t *out) {
    for (size_t i = 0; i < n; i++) {
        G1Affine p;
        memcpy(p.x.l, xy + 24 * i, 48);
        memcpy(p.y.l, xy + 24 * i + 12, 48);
        out[i] = g1_in_subgroup(p);
    }
}
// β (Montgomery, 12 u32) and [|x|]·P (affine, Montgomery; returns 0 for the identity) of the subgroup test.
void emu_g1_beta(uint32_t *out) { const Fp b = g1codec::beta(); memcpy(out, b.l, 48); }
int emu_g1_mul_by_x_abs(const uint32_t *xy, uint32_t *out_xy) {
    G1Affine p, r;
    memcpy(p.x.l, xy, 48);
    memcpy(p.y.l, xy + 12, 48);
    if (!g1_to_affine(g1codec::mul_by_x_abs(G1Xyzz::from_affine(p)), r)) return 0;
    memcpy(out_xy, r.x.l, 48);
    memcpy(out_xy + 12, r.y.l, 48);
    return 1;
}
}
