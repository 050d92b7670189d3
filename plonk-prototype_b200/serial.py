"""Byte (de)serialisation of the KZG10 parameters, host side: dusk-plonk 0.8.2 `commitment_scheme::kzg10::{CommitKey,
OpeningKey, PublicParameters}::{to_raw_bytes, from_slice_unchecked, to_var_bytes}` (crate pinned at
/root/reference/Cargo.toml:19; SURVEY.md §2.2 D5, §5 "checkpoint / resume", §8f-1) — the reference never calls them, a
host that caches a generated SRS on disk does.

**Unpinned** like the rest of the upstream surface (UPSTREAM_ASSUMPTIONS.md §Serialisation): the layouts below are restated
from memory of the crates —
  * `G1Affine::to_raw_bytes` (dusk-bls12_381): 97 bytes = x ‖ y as 2 × 6 little-endian u64 limbs in MONTGOMERY form (the
    memory image) ‖ one infinity byte;  `G1Affine::to_bytes`: the 48-byte compressed encoding (`msm.g1_to_bytes`);
  * `CommitKey::to_raw_bytes`: u64 LE point count ‖ the points' raw bytes;  `to_var_bytes`: the points compressed, no prefix;
  * `OpeningKey::to_bytes`: g (48, compressed G1) ‖ h (96, compressed G2) ‖ β·h (96) = 240 bytes;
  * `PublicParameters::to_raw_bytes` / `to_var_bytes`: the opening key, then the commit key.
The commit key's points never pass through Python integers: the raw form is a numpy reshape of the device image, the compressed
form is encoded and decoded (with every check of `G1Affine::from_bytes`) on the GPU (`pb200_srs_{to,from}_compressed`).  The
opening key's two G2 points do (compression needs canonical coordinates and a square root on the way back) — cold, three
points per SRS."""
import numpy as np

from . import _native

P = 0x1A0111EA397FE69A4B1BA7B6434BACD764774B84F38512BF6730D2A0F6B0F6241EABFFFEB153FFFFB9FEFFFFFFFFAAAB
R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
_R_INV = pow(1 << 384, -1, P)
G1_RAW_SIZE, G1_SIZE, G2_SIZE, OPENING_KEY_SIZE = 97, 48, 96, 240
# the generators' compressed encodings (zcash format; SURVEY.md App. A.3-A.4)
G1_GENERATOR_BYTES = bytes.fromhex("97f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb")
G2_GENERATOR_BYTES = bytes.fromhex(
    "93e02b6052719f607dacd3a088274f65596bd0d09920b61ab5da61bbdc7f5049334cf11213945d57e5ac7d055d042b7e"
    "024aa2b2f08f0a91260805272dc51051c6e47ad4fa403b02b4510b647ae3d1770bac0326a805bbefd48056c8c121bdb8")


# ---- Fp2 = Fp[u]/(u² + 1), pairs (c0, c1) of canonical integers ------------------------------------------------------
def _fp2_mul(a, b):
    return ((a[0] * b[0] - a[1] * b[1]) % P, (a[0] * b[1] + a[1] * b[0]) % P)


def _fp2_pow(a, e):
    r = (1, 0)
    while e:
        if e & 1:
            r = _fp2_mul(r, a)
        a = _fp2_mul(a, a)
        e >>= 1
    return r


def _fp2_sqrt(a):
    """A square root in Fp2 (p ≡ 3 mod 4), or None."""
    if a == (0, 0):
        return (0, 0)
    a1 = _fp2_pow(a, (P - 3) // 4)
    alpha = _fp2_mul(_fp2_mul(a1, a1), a)
    x0 = _fp2_mul(a1, a)
    if alpha == (P - 1, 0):
        x = ((-x0[1]) % P, x0[0])                       # u·x0
    else:
        b = _fp2_pow(((1 + alpha[0]) % P, alpha[1]), (P - 1) // 2)
        x = _fp2_mul(b, x0)
    return x if _fp2_mul(x, x) == a else None


def _limbs_to_int_mont(l6):
    return sum(int(v) << (64 * i) for i, v in enumerate(l6)) * _R_INV % P


def _int_to_limbs_mont(v):
    v = v * (1 << 384) % P
    return [(v >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(6)]


def g2_to_bytes(xy24):
    """`G2Affine::to_bytes`: x.c1 ‖ x.c0 big-endian; bit 7 compressed, bit 5 = y lexicographically larger (c1 first)."""
    v = np.asarray(xy24, dtype=np.uint64).reshape(4, 6)
    x0, x1, y0, y1 = (_limbs_to_int_mont(v[k]) for k in range(4))
    b = bytearray(x1.to_bytes(48, "big") + x0.to_bytes(48, "big"))
    larger = y1 > (P - 1) // 2 if y1 else y0 > (P - 1) // 2
    b[0] |= 0x80 | (0x20 if larger else 0)
    return bytes(b)


def g2_from_bytes(b):
    """Inverse of g2_to_bytes for a finite compressed point → 24 u64 (x.c0 ‖ x.c1 ‖ y.c0 ‖ y.c1, Montgomery)."""
    assert len(b) == 96 and b[0] & 0x80 and not b[0] & 0x40, "a finite compressed G2 point"
    sign = bool(b[0] & 0x20)
    x1 = int.from_bytes(bytes([b[0] & 0x1F]) + b[1:48], "big")
    x0 = int.from_bytes(b[48:], "big")
    assert x0 < P and x1 < P
    x = (x0, x1)
    rhs = _fp2_mul(_fp2_mul(x, x), x)
    rhs = ((rhs[0] + 4) % P, (rhs[1] + 4) % P)          # y² = x³ + 4(u + 1)
    y = _fp2_sqrt(rhs)
    assert y is not None, "not on the curve"
    larger = y[1] > (P - 1) // 2 if y[1] else y[0] > (P - 1) // 2
    if larger != sign:
        y = ((-y[0]) % P, (-y[1]) % P)
    return np.array(_int_to_limbs_mont(x[0]) + _int_to_limbs_mont(x[1]) + _int_to_limbs_mont(y[0]) + _int_to_limbs_mont(y[1]), dtype=np.uint64)


def _fp2_inv(a):
    t = pow((a[0] * a[0] + a[1] * a[1]) % P, -1, P)
    return (a[0] * t % P, (-a[1]) * t % P)


def _g2_add(p, q):
    """Affine addition on the twist over Fp2; None is the identity."""
    if p is None:
        return q
    if q is None:
        return p
    if p[0] == q[0]:
        if ((p[1][0] + q[1][0]) % P, (p[1][1] + q[1][1]) % P) == (0, 0):
            return None
        xx = _fp2_mul(p[0], p[0])
        lam = _fp2_mul((3 * xx[0] % P, 3 * xx[1] % P), _fp2_inv((2 * p[1][0] % P, 2 * p[1][1] % P)))
    else:
        lam = _fp2_mul(((q[1][0] - p[1][0]) % P, (q[1][1] - p[1][1]) % P), _fp2_inv(((q[0][0] - p[0][0]) % P, (q[0][1] - p[0][1]) % P)))
    ll = _fp2_mul(lam, lam)
    x3 = ((ll[0] - p[0][0] - q[0][0]) % P, (ll[1] - p[0][1] - q[0][1]) % P)
    t = _fp2_mul(lam, ((p[0][0] - x3[0]) % P, (p[0][1] - x3[1]) % P))
    return (x3, ((t[0] - p[1][0]) % P, (t[1] - p[1][1]) % P))


def g2_from_bytes_checked(b):
    """`G2Affine::from_bytes` with every check: flags, x.c0 and x.c1 < p, on the twist, and r·Q = O (the order-r subgroup;
    double-and-add over Fp2 on Python integers — cold, one point).  The identity is rejected: an opening key's β·H never is.
    → 24 u64 (x.c0 ‖ x.c1 ‖ y.c0 ‖ y.c1, Montgomery); ValueError on anything invalid."""
    if len(b) != G2_SIZE or not b[0] & 0x80:
        raise ValueError("G2 point: not a 96-byte compressed encoding")
    if b[0] & 0x40:
        raise ValueError("G2 point: the identity")
    x1 = int.from_bytes(bytes([b[0] & 0x1F]) + b[1:48], "big")
    x0 = int.from_bytes(b[48:], "big")
    if x0 >= P or x1 >= P:
        raise ValueError("G2 point: x is not below p")
    x = (x0, x1)
    rhs = _fp2_mul(_fp2_mul(x, x), x)
    y = _fp2_sqrt(((rhs[0] + 4) % P, (rhs[1] + 4) % P))
    if y is None:
        raise ValueError("G2 point: not on the curve")
    larger = y[1] > (P - 1) // 2 if y[1] else y[0] > (P - 1) // 2
    if larger != bool(b[0] & 0x20):
        y = ((-y[0]) % P, (-y[1]) % P)
    acc, add, k = None, (x, y), R
    while k:
        if k & 1:
            acc = _g2_add(acc, add)
        add = _g2_add(add, add)
        k >>= 1
    if acc is not None:
        raise ValueError("G2 point: not in the prime-order subgroup")
    return np.array(_int_to_limbs_mont(x[0]) + _int_to_limbs_mont(x[1]) + _int_to_limbs_mont(y[0]) + _int_to_limbs_mont(y[1]), dtype=np.uint64)


def opening_key_to_bytes(beta_h):
    """`OpeningKey::to_bytes` for the opening key (G, H, β·H) of a trapdoor-generated SRS (`_native.opening_key_from_tau`)."""
    return G1_GENERATOR_BYTES + G2_GENERATOR_BYTES + g2_to_bytes(beta_h)


def opening_key_from_bytes(b):
    """→ β·H as the 24 u64 `verify` takes.  g and h must be the generators (dusk's `setup` never produces anything else)."""
    assert len(b) == OPENING_KEY_SIZE
    if b[:48] != G1_GENERATOR_BYTES or b[48:144] != G2_GENERATOR_BYTES:
        raise ValueError("opening key over other generators than the BLS12-381 ones")
    return g2_from_bytes(b[144:])


def opening_key_from_bytes_checked(b):
    """The opening key of `PublicParameters::from_slice`: as opening_key_from_bytes, and β·H must be a valid point of G2
    (g2_from_bytes_checked).  ValueError on anything invalid."""
    if len(b) != OPENING_KEY_SIZE:
        raise ValueError("opening key: %d bytes, expected %d" % (len(b), OPENING_KEY_SIZE))
    if b[:48] != G1_GENERATOR_BYTES or b[48:144] != G2_GENERATOR_BYTES:
        raise ValueError("opening key over other generators than the BLS12-381 ones")
    return g2_from_bytes_checked(bytes(b[144:]))


# ---- commit key ---------------------------------------------------------------------------------------------------------
def commit_key_to_raw_bytes(ctx, srs):
    """`CommitKey::to_raw_bytes` of a device-resident SRS: one D2H copy and a numpy reshape."""
    n = _native.lib().pb200_srs_len(srs)
    pts = np.empty((n, 96), np.uint8)
    if n:
        ctx.d2h(pts, ctx.srs_dev_ptr(srs))
    raw = np.zeros((n, G1_RAW_SIZE), np.uint8)           # the infinity byte stays 0: an SRS never holds the identity
    raw[:, :96] = pts
    return int(n).to_bytes(8, "little") + raw.tobytes()


def commit_key_from_slice_unchecked(ctx, b, precompute=True):
    """`CommitKey::from_slice_unchecked` → an SRS handle resident on the GPU (no curve / subgroup checks, like upstream)."""
    n = int.from_bytes(b[:8], "little")
    if len(b) != 8 + n * G1_RAW_SIZE:
        raise ValueError("CommitKey: %d bytes for %d points" % (len(b), n))
    raw = np.frombuffer(b, dtype=np.uint8, offset=8).reshape(n, G1_RAW_SIZE)
    if raw[:, 96].any():
        raise ValueError("CommitKey holds the point at infinity")
    pts = np.ascontiguousarray(raw[:, :96]).view(np.uint64).reshape(n, 12)
    srs = ctx.srs_upload(pts)
    if precompute and 1 <= n <= (1 << 22):
        ctx.srs_precompute(srs)
    return srs


def commit_key_to_var_bytes(ctx, srs):
    """`CommitKey::to_var_bytes`: the points compressed (48 bytes each, no prefix), encoded on the GPU."""
    n = _native.lib().pb200_srs_len(srs)
    return ctx.srs_to_compressed(srs) if n else b""


def commit_key_from_slice(ctx, b, precompute=True):
    """`CommitKey::from_slice` → an SRS handle resident on the GPU.  Every point is decoded and checked on the device as
    `G1Affine::from_bytes` does (flags, x < p, on the curve, prime-order subgroup); ValueError names the first invalid one.
    Keys of up to 2^22 points also get their pre-doubled window copies, as commit_key_from_slice_unchecked."""
    b = bytes(b)
    if not b or len(b) % G1_SIZE:
        raise ValueError("CommitKey: %d bytes is not a positive multiple of %d" % (len(b), G1_SIZE))
    srs = ctx.srs_from_compressed(b)
    n = len(b) // G1_SIZE
    if precompute and n <= (1 << 22):
        try:
            ctx.srs_precompute(srs)
        except Exception:
            ctx.srs_free(srs)
            raise
    return srs
