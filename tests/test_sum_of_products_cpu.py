"""The Fp sum of products with one Montgomery reduction (Field::mul2_sum_*, csrc/field.cuh) and the G1 formulas that compute
Y3 with it (csrc/g1.cuh), run under host emulation (the device templates compiled for the CPU with the carry flag
emulated) against Python integers and the model's group law.  The harness traps when a lazy result leaves [0, 2p) or a
canonical one leaves [0, p)."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "plonk-prototype_b200", "csrc")
SRC = os.path.join(ROOT, "tests", "host_emu", "emu_sum.cpp")
P = model.P
RINV = pow(1 << 384, -1, P)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_sum") / "emu_sum.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-o", out])
    return ctypes.CDLL(out)


def _limbs(vals):
    return np.array([[(v >> (32 * i)) & 0xFFFFFFFF for i in range(12)] for v in vals], np.uint32).reshape(-1, 12)


def _ints(arr):
    return [sum(int(w) << (32 * i) for i, w in enumerate(row)) for row in arr]


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _mul2_sum(lib, a, b, c, d):
    A, B, C, D = (_limbs(v) for v in (a, b, c, d))
    o = np.empty_like(A)
    lib.emu_mul2_sum(_ptr(A), _ptr(B), _ptr(C), _ptr(D), _ptr(o), ctypes.c_size_t(len(a)))
    return _ints(o)


def _check(lib, a, b, c, d):
    got = _mul2_sum(lib, a, b, c, d)
    for v, x, y, z, w in zip(got, a, b, c, d):
        assert v < 2 * P
        assert v % P == (x * y + z * w) * RINV % P


def test_random_operands_in_lazy_range(emu):
    rng = random.Random(0x5A11)
    n = 3000
    a, b, c, d = ([rng.randrange(2 * P + 1) for _ in range(n)] for _ in range(4))
    _check(emu, a, b, c, d)


def test_corner_operands_in_every_position(emu):
    corners = [0, 1, P - 1, P, 2 * P - 1, 2 * P]
    rng = random.Random(0xC0E)
    quads = []
    for pos in range(4):                          # one argument runs over the corners, the others random or corners too
        for v in corners:
            for _ in range(8):
                q = [rng.randrange(2 * P + 1) for _ in range(4)]
                q[pos] = v
                quads.append(q)
    quads += [[w, x, y, z] for w in corners for x in corners for y in corners for z in corners]   # 6^4 all-corner quads
    a, b, c, d = (list(t) for t in zip(*quads))
    _check(emu, a, b, c, d)


def test_sums_that_are_multiples_of_p(emu):
    """a·b + c·d ≡ 0: the result must be 0 or p, the two lazy representatives of zero."""
    rng = random.Random(0x0FF)
    a, b, c, d = [], [], [], []
    for _ in range(500):
        x, y, z = (rng.randrange(1, P) for _ in range(3))
        w = (-x * y * pow(z, -1, P)) % P                         # z·w ≡ −x·y
        for dx, dw in ((0, 0), (P, 0), (0, P), (P, P)):       # canonical and lifted representatives
            a.append(x + dx)
            b.append(y)
            c.append(z)
            d.append(w + dw)
    got = _mul2_sum(emu, a, b, c, d)
    assert all(v in (0, P) for v in got)
    _check(emu, a, b, c, d)


def test_difference_through_neg_2p(emu):
    """x·y − z·w as x·y + neg_2p(z)·w, with z at the ends of [0, 2p] (neg_2p(0) = 2p is an operand the proof allows)."""
    rng = random.Random(0xD1F)
    zs = [0, 1, P - 1, P, 2 * P - 1, 2 * P] + [rng.randrange(2 * P + 1) for _ in range(300)]
    Z = _limbs(zs)
    nz = np.empty_like(Z)
    emu.emu_neg_2p(_ptr(Z), _ptr(nz), ctypes.c_size_t(len(zs)))
    assert _ints(nz) == [2 * P - z for z in zs]
    x, y, w = ([rng.randrange(2 * P) for _ in zs] for _ in range(3))
    got = _mul2_sum(emu, x, y, _ints(nz), w)
    assert [v % P for v in got] == [(a * b - c * d) * RINV % P for a, b, c, d in zip(x, y, zs, w)]


def test_fr_cannot_instantiate_the_sum(tmp_path):
    """Fr has one spare bit: two products per row would overflow the accumulator, so the template refuses it."""
    src = tmp_path / "fr_sum.cpp"
    src.write_text('#define PB200_HOST_EMU 1\n#include "%s"\nFr f(const Fr &a) { return Fr::mul2_sum_unreduced(a, a, a, a); }\n'
                   % os.path.join(CSRC, "field.cuh"))
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", str(src)], capture_output=True, text=True)
    assert r.returncode != 0 and "3 spare bits" in r.stderr


# ---- G1 formulas with Y3 from the sum of products ----------------------------------------------------------------------
def _pts(points):
    out = np.zeros((len(points), 24), np.uint32)
    for i, (x, y) in enumerate(points):
        out[i, :12] = _limbs([model.fp_to_mont(x)])[0]
        out[i, 12:] = _limbs([model.fp_to_mont(y)])[0]
    return out


def _chain(lib, op, points):
    pts = _pts(points)
    o = np.zeros(25, np.uint32)
    lib.emu_g1_chain(op, _ptr(pts), ctypes.c_size_t(len(points)), _ptr(o))
    if o[24]:
        return None
    x, y = _ints(o[:24].reshape(2, 12))
    return model.fp_from_mont(x), model.fp_from_mont(y)


def _sequences():
    """Point sequences that reach every branch: identity accumulator, equal points and opposite points, both while the
    accumulator still has ZZ = 1 and after it has been through general additions."""
    B = model.synthetic_bases(8)
    neg = model.g1_neg
    seqs = [[B[0], B[1], B[2], B[3], B[4]]]
    seqs.append([B[0], B[0], B[1]])                           # equal at ZZ = 1 → doubling
    seqs.append([B[0], neg(B[0]), B[1], B[2]])                # opposite at ZZ = 1 → identity, then from the identity
    s = model.g1_add(model.g1_add(B[2], B[3]), B[4])
    seqs.append([B[2], B[3], B[4], s, B[5]])                  # equal after general additions
    seqs.append([B[2], B[3], B[4], neg(s), B[6], B[6]])       # opposite after general additions
    seqs.append([B[7]] * 9)                                   # repeated base: doubling, then equal-x … cases of k·P
    seqs.append([B[1], neg(B[1]), neg(B[1]), B[1], B[1]])
    return seqs


def _fold(seq, dbl_each=False):
    acc = None
    for p in seq:
        acc = model.g1_add(acc, p)
        if dbl_each:
            acc = model.g1_add(acc, acc)
    return acc


@pytest.mark.parametrize("op", [0, 1, 3])
def test_additions_match_model(emu, op):
    """op 0: g1_madd_lazy (lazy coordinates), 1 / 3: g1_add with either operand order (canonical coordinates)."""
    for seq in _sequences():
        assert _chain(emu, op, seq) == _fold(seq), seq


def test_doublings_match_model(emu):
    for seq in _sequences():
        assert _chain(emu, 2, seq) == _fold(seq, dbl_each=True), seq
    for p in model.synthetic_bases(16):
        assert _chain(emu, 4, [p]) == model.g1_add(p, p)
