"""CPU tests of the compressed G1 codec the srs_io kernels run (csrc/g1_codec.cuh: G1Affine::from_bytes with the
endomorphism subgroup test, G1Affine::to_bytes).  The same C++ is compiled for the host with the carry-flag primitives emulated
(PB200_HOST_EMU, tests/host_emu/emu_srs.cpp) and compared with the CPU reference decoder (tests/srs_io_ref.c: square root,
then r·P = O), which is itself cross-checked against the pure-Python model.  Also the checked opening-key decoder of
plonk-prototype_b200/serial.py, which needs no GPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import model
import srs_io_ref as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host_emu", "emu_srs.cpp")
X_ABS = 0xD201000000010000


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_srs") / "emu_srs.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-o", out])
    return ctypes.CDLL(out)


@pytest.fixture(scope="module")
def corpus(oracle):
    return ref.corpus()


def _vp(a):
    return ctypes.c_void_p(a.ctypes.data)


def emu_decode(lib, data):
    buf = np.frombuffer(bytes(data), dtype=np.uint8)
    n = buf.size // 48
    st = np.zeros(n, np.uint8)
    xy = np.zeros((n, 12), np.uint64)
    lib.emu_g1_decode(_vp(buf), ctypes.c_size_t(n), _vp(xy), _vp(st))
    return st, xy


def emu_encode(lib, xy):
    xy = np.ascontiguousarray(xy, dtype=np.uint64).reshape(-1, 12)
    out = np.zeros(48 * xy.shape[0], np.uint8)
    lib.emu_g1_encode(_vp(xy), ctypes.c_size_t(xy.shape[0]), _vp(out))
    return out.tobytes()


def _mont_int(limbs):
    return model.fp_from_mont(sum(int(v) << (64 * i) for i, v in enumerate(np.asarray(limbs).reshape(-1))))


def test_reference_decoder_matches_model(corpus):
    """The C reference (upstream's algorithm) and the Python model agree on every encoding of the corpus, status and point."""
    data, labels = corpus
    st, xy = ref.g1_from_bytes_checked(data, threads=4)
    assert list(st) == labels
    for i in range(len(labels)):
        ms, pt = ref.model_decode(data[48 * i:48 * i + 48])
        assert ms == labels[i], i
        if ms == ref.OK:
            assert (_mont_int(xy[i, :6]), _mont_int(xy[i, 6:])) == pt, i


def test_device_decoder_matches_reference(emu, corpus):
    """g1_decode_checked: per-point status and decoded limbs equal the reference's; the encoding with bit 5 flipped decodes
    to −P."""
    data, labels = corpus
    st, xy = emu_decode(emu, data)
    rst, rxy = ref.g1_from_bytes_checked(data, threads=4)
    assert list(st) == list(rst) == labels
    assert (xy == rxy).all()
    ok = [i for i, s in enumerate(labels) if s == ref.OK]
    assert len(ok) >= 64
    for i in ok[::2]:                                     # pairs (P, P with bit 5 flipped)
        x0, y0 = _mont_int(xy[i, :6]), _mont_int(xy[i, 6:])
        x1, y1 = _mont_int(xy[i + 1, :6]), _mont_int(xy[i + 1, 6:])
        assert x0 == x1 and y1 == (model.P - y0) % model.P and y0 != 0


def test_device_decoder_rejects_each_kind(emu):
    """One hand-built encoding per reject reason, named, so a failure says which check broke."""
    g = model.g1_compress(model.G1_GEN)
    cases = {
        "bit 7 clear": (bytes([g[0] & 0x7F]) + g[1:], ref.BAD_FLAGS),
        "identity": (bytes([0xC0]) + bytes(47), ref.IDENTITY),
        "identity with bit 5": (bytes([0xE0]) + bytes(47), ref.BAD_FLAGS),
        "identity with a low byte": (bytes([0xC0]) + bytes(46) + b"\x01", ref.BAD_FLAGS),
        "x = p": (ref._enc_x(model.P, 0x80), ref.X_RANGE),
        "G with x + p": (ref._enc_x(model.GX + model.P, 0x80 | (g[0] & 0x20)), ref.X_RANGE) if model.GX + model.P < 1 << 381 else None,
        "x = 1 (x³ + 4 = 5, not a square)": (ref._enc_x(1, 0x80), ref.NOT_ON_CURVE),
        "(0, 2)": (model.g1_compress((0, 2)), ref.NOT_IN_SUBGROUP),
        "G + (0, 2)": (model.g1_compress(model.g1_add(model.G1_GEN, (0, 2))), ref.NOT_IN_SUBGROUP),
        "G": (g, ref.OK),
    }
    assert not ref._is_square(5, model.P)
    for name, case in cases.items():
        if case is None:
            continue
        st, _ = emu_decode(emu, case[0])
        assert st[0] == case[1], name


def test_encoder_matches_model(emu, oracle):
    """g1_encode gives the bytes of model.g1_compress (and of the reference encoder) for both roots of y."""
    tau = oracle.fr_to_mont(oracle.ints_to_limbs([0x51CE], 4))
    pts = np.concatenate([oracle.srs_setup(tau, 24), oracle.synthetic_bases(24)])
    neg = pts.copy()
    neg[:, 6:] = oracle.fp_sub(np.zeros((pts.shape[0], 6), np.uint64), pts[:, 6:])
    pts = np.concatenate([pts, neg])
    got = emu_encode(emu, pts)
    assert got == ref.g1_to_bytes(pts)
    want = b"".join(model.g1_compress((_mont_int(p[:6]), _mont_int(p[6:]))) for p in pts)
    assert got == want
    larger = [got[48 * i] & 0x20 for i in range(pts.shape[0])]
    assert any(larger) and not all(larger)
    st, xy = emu_decode(emu, got)                       # and back
    assert (st == 0).all() and (xy == pts).all()


def test_endomorphism_constant(emu, oracle):
    """β is a primitive cube root of unity in Fp, and the one for which φ(G) = −[x²]G; [|x|]·G of the device ladder is the
    model's."""
    b32 = np.zeros(12, np.uint32)
    emu.emu_g1_beta(_vp(b32))
    beta = _mont_int(b32.view(np.uint64))
    P = model.P
    assert beta != 1 and pow(beta, 3, P) == 1
    assert (beta * model.GX % P, model.GY) == model.g1_neg(model.g1_mul(model.G1_GEN, X_ABS * X_ABS))
    other = beta * beta % P                               # the other root is not the eigenvalue −x² of φ
    assert (other * model.GX % P, model.GY) != model.g1_neg(model.g1_mul(model.G1_GEN, X_ABS * X_ABS))
    g = oracle.g1_generator()
    out = np.zeros(12, np.uint64)
    assert emu.emu_g1_mul_by_x_abs(_vp(g), _vp(out)) == 1
    assert (_mont_int(out[:6]), _mont_int(out[6:])) == model.g1_mul(model.G1_GEN, X_ABS)


def test_endomorphism_test_decides_like_r_times_p(emu, oracle):
    """g1_in_subgroup on points on the curve: true on G1, false on P + T for T of order 3 and on random curve points — the
    decision of r·P = O."""
    P = model.P
    pts = [model.g1_mul(model.G1_GEN, k) for k in (1, 2, 3, X_ABS, model.R - 1)]
    off = [model.g1_add(p, t) for p in pts for t in ((0, 2), (0, P - 2))] + [(0, 2)]
    g = model.splitmix64_stream(77)
    while len(off) < 20:
        x = next(g) % P
        if ref._is_square(x ** 3 + 4, P):
            off.append((x, pow(x ** 3 + 4, (P + 1) // 4, P)))
    for q in off:
        assert q is not None and model.g1_on_curve(q)
    xy = np.array([[(model.fp_to_mont(c) >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for c in q for i in range(6)] for q in pts + off],
                  dtype=np.uint64)
    got = np.zeros(len(pts) + len(off), np.uint8)
    emu.emu_g1_in_subgroup(_vp(xy), ctypes.c_size_t(xy.shape[0]), _vp(got))
    assert list(got) == [1] * len(pts) + [0] * len(off)


# ---- the checked opening key (serial.py; host only) -----------------------------------------------------------------------
def _serial():
    import plonk_prototype_b200 as pb
    return pb.serial


def test_opening_key_checked_accepts_and_rejects():
    """`PublicParameters::from_slice`'s opening key: β·H must decode, lie on the twist and in the order-r subgroup of G2."""
    import plonk_prototype_b200 as pb
    serial = _serial()
    if not os.path.exists(pb.LIB_PATH):
        pytest.skip("libpb200.so is not built")
    beta_h = pb._native.opening_key_from_tau(pb.scalars_to_mont([0x7A05]))
    good = serial.opening_key_to_bytes(beta_h)
    assert (serial.opening_key_from_bytes_checked(good) == beta_h).all()
    for bad in (good[:-1], good[:144] + bytes([0xC0]) + bytes(95), good[:144] + bytes([good[144] & 0x7F]) + good[145:],
                good[:144] + ref.g2_off_subgroup_bytes(), good[:200] + bytes([good[200] ^ 1]) + good[201:],
                good[:100] + bytes([good[100] ^ 1]) + good[101:]):
        with pytest.raises(ValueError):
            serial.opening_key_from_bytes_checked(bad)
