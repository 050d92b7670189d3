"""ctypes loader for tests/srs_io_ref.c, the CPU reference of the compressed G1 codec (TEST INFRASTRUCTURE).

Used by tests/test_srs_io_cpu.py, tests/test_srs_io_gpu.py and scripts/srs_io_bench.py (its labelled CPU baseline).  The
shared library is compiled on first use into the temporary directory, keyed by the sources' contents, so the checkout is
never written to."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
SRC = os.path.join(_HERE, "srs_io_ref.c")
_DEPS = [SRC] + [os.path.join(_ROOT, "oracle", f) for f in ("oracle.c", "plonk_oracle.inc", "mont.h", "mont_asm.h")]
_LIB = None

OK, BAD_FLAGS, X_RANGE, NOT_ON_CURVE, NOT_IN_SUBGROUP, IDENTITY = range(6)   # PB200_G1_* (include/pb200.h)


def lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha256()
        for d in _DEPS:
            with open(d, "rb") as f:
                h.update(f.read())
        so = os.path.join(tempfile.gettempdir(), "pb200_srs_io_ref_%d_%s.so" % (os.getuid(), h.hexdigest()[:16]))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-madx", "-fPIC", "-fvisibility=hidden", "-Wall",
                                   "-Wno-unused-function", "-shared", "-o", tmp, SRC, "-lpthread"])
            os.replace(tmp, so)
        _LIB = ctypes.CDLL(so)
    return _LIB


def g1_from_bytes_checked(data, threads=1):
    """`G1Affine::from_bytes` (square root, r·P = O) over n 48-byte encodings → (status uint8 (n,), points (n, 12) uint64
    packed affine Montgomery, zero rows where the status is not OK)."""
    buf = np.frombuffer(bytes(data), dtype=np.uint8)
    assert buf.size % 48 == 0
    n = buf.size // 48
    st = np.zeros(n, np.uint8)
    xy = np.zeros((n, 12), np.uint64)
    lib().orc_g1_from_bytes_checked(ctypes.c_void_p(buf.ctypes.data), ctypes.c_size_t(n), ctypes.c_void_p(xy.ctypes.data),
                                    ctypes.c_void_p(st.ctypes.data), ctypes.c_int(threads))
    return st, xy


def g1_to_bytes(xy, threads=1):
    """`G1Affine::to_bytes` of (n, 12) packed affine Montgomery points → 48·n bytes."""
    xy = np.ascontiguousarray(xy, dtype=np.uint64).reshape(-1, 12)
    out = np.zeros(48 * xy.shape[0], np.uint8)
    lib().orc_g1_to_bytes(ctypes.c_void_p(xy.ctypes.data), ctypes.c_size_t(xy.shape[0]), ctypes.c_void_p(out.ctypes.data),
                          ctypes.c_int(threads))
    return out.tobytes()


# ---- the test corpus: valid points, every reject reason, and the edge cases between them -----------------------------------
def _enc_x(x, flags):
    b = bytearray(int(x).to_bytes(48, "big"))
    b[0] |= flags
    return bytes(b)


def _is_square(v, P):
    return v % P == 0 or pow(v, (P - 1) // 2, P) == 1


def corpus(n_valid=16, seed=0x5EB5):
    """→ (48·n bytes, list of n labels).  The label is the status the encoding must get (PB200_G1_*).

    valid: τ^i·G and synthetic bases (a + i·d)·G, each as encoded and with bit 5 flipped (which encodes −P);
    flag errors: bit 7 clear, malformed identities (a non-zero byte after c0, bit 5 or an x bit set next to bit 6);
    the canonical identity c0 00…00; non-canonical x (a valid x plus p, still below 2^381; x = p; x = 2^381 − 1);
    x with x³ + 4 not a square; on-curve points outside G1: P + (0, 2) ((0, ±2) is 3-torsion) and points from random x."""
    import model
    import pyoracle as O
    P = model.P
    g = model.splitmix64_stream(seed)

    def rand_x():
        while True:
            v = sum(next(g) << (64 * i) for i in range(6)) & ((1 << 381) - 1)
            if v < P:
                return v

    out, labels = [], []

    def add(b, st):
        assert len(b) == 48
        out.append(bytes(b))
        labels.append(st)

    tau = O.fr_to_mont(O.ints_to_limbs([0x7A05ED], 4))
    valid = np.concatenate([O.srs_setup(tau, n_valid), O.synthetic_bases(n_valid)])
    venc = g1_to_bytes(valid)
    vints = []
    for i in range(valid.shape[0]):
        b = venc[48 * i:48 * i + 48]
        add(b, OK)
        add(bytes([b[0] ^ 0x20]) + b[1:], OK)                         # −P
        xy = O.fp_from_mont(valid[i].reshape(2, 6))
        vints.append((O.limbs_to_int(xy[0]), O.limbs_to_int(xy[1])))
    b0 = venc[:48]
    for k in range(4):                                               # bit 7 clear
        b = venc[48 * k:48 * k + 48]
        add(bytes([b[0] & 0x7F]) + b[1:], BAD_FLAGS)
    add(bytes([0x40]) + bytes(47), BAD_FLAGS)                        # identity bit without the compression bit
    add(bytes([0xC0]) + bytes(47), IDENTITY)                         # the canonical identity
    for pos in (1, 23, 47):                                          # malformed identities
        b = bytearray([0xC0]) + bytearray(47)
        b[pos] = 0x01
        add(b, BAD_FLAGS)
    add(bytes([0xE0]) + bytes(47), BAD_FLAGS)                        # bit 5 on the identity
    add(bytes([0xC1]) + bytes(47), BAD_FLAGS)                        # an x bit on the identity
    add(bytes([b0[0] | 0x40]) + b0[1:], BAD_FLAGS)                   # identity bit on a valid point
    small = [(x, y) for x, y in vints if x + P < (1 << 381)]         # non-canonical x: x + p with the same flags
    assert small, "no valid point with x < 2^381 − p in the sample"
    for x, y in small[:4]:
        add(_enc_x(x + P, 0x80 | (0x20 if y > (P - 1) // 2 else 0)), X_RANGE)
    add(_enc_x(P, 0x80), X_RANGE)
    add(_enc_x((1 << 381) - 1, 0x80), X_RANGE)
    add(_enc_x((1 << 381) - 1, 0xA0), X_RANGE)
    k = 0
    while k < 8:                                                     # x³ + 4 not a square
        x = rand_x()
        if not _is_square(x ** 3 + 4, P):
            add(_enc_x(x, 0x80 | (0x20 if k & 1 else 0)), NOT_ON_CURVE)
            k += 1
    for x, y in vints[:6]:                                           # P + (0, 2): on the curve, order 3r
        for t in ((0, 2), (0, P - 2)):
            q = model.g1_add((x, y), t)
            add(model.g1_compress(q), NOT_IN_SUBGROUP)
    for t in ((0, 2), (0, P - 2)):                                   # the 3-torsion points themselves
        add(model.g1_compress(t), NOT_IN_SUBGROUP)
    k = 0
    while k < 8:                                                     # random x on the curve: outside G1 but with probability 1/h
        x = rand_x()
        if _is_square(x ** 3 + 4, P):
            add(_enc_x(x, 0x80 | (0x20 if k & 1 else 0)), NOT_IN_SUBGROUP)
            k += 1
    return b"".join(out), labels


def model_decode(b):
    """The same decision from the pure-Python model (plonk_model.bytes_to_g1, then r·P = O by double-and-add on integers):
    → (status, (x, y) canonical or None)."""
    import model
    import plonk_model as pm
    try:
        pt = pm.bytes_to_g1(b)
    except ValueError as e:
        msg = str(e)
        if "range" in msg:
            return X_RANGE, None
        if "curve" in msg:
            return NOT_ON_CURVE, None
        return BAD_FLAGS, None
    if pt is None:
        return IDENTITY, None
    acc, add, k = None, pt, model.R                                  # model.g1_mul reduces k mod r: multiply by r by hand
    while k:
        if k & 1:
            acc = model.g1_add(acc, add)
        add = model.g1_add(add, add)
        k >>= 1
    return (OK, pt) if acc is None else (NOT_IN_SUBGROUP, None)


def g2_off_subgroup_bytes():
    """A compressed point of the twist y² = x³ + 4(u + 1) outside G2: the first x = (k, 1) with a square right-hand side (the
    cofactor of G2 is ~2^381, so such a point lies in G2 with negligible probability; the decoders' r·Q check decides)."""
    import model
    P = model.P

    def mul(a, b):
        return ((a[0] * b[0] - a[1] * b[1]) % P, (a[0] * b[1] + a[1] * b[0]) % P)

    def power(a, e):
        r = (1, 0)
        while e:
            if e & 1:
                r = mul(r, a)
            a = mul(a, a)
            e >>= 1
        return r

    for k in range(1, 1000):
        x = (k, 1)
        xx = mul(mul(x, x), x)
        rhs = ((xx[0] + 4) % P, (xx[1] + 4) % P)
        if power(rhs, (P * P - 1) // 2) == (1, 0):                   # a square in Fp2 (Euler's criterion)
            b = bytearray(x[1].to_bytes(48, "big") + x[0].to_bytes(48, "big"))
            b[0] |= 0x80
            return bytes(b)
    raise AssertionError("no point of the twist found")
