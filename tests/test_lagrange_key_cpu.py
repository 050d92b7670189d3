"""CPU test of the Lagrange-basis commit key (csrc/lagrange.cuh: the G1 inverse NTT the lagrange_* kernels run), compiled
for the host with the carry-flag primitives emulated (PB200_HOST_EMU, tests/host_emu/emu_lagrange.cpp).

A key P_j = s_j·G with known s_j must become Q_i = (n⁻¹·Σ_j ω^(−ij)·s_j)·G, checked with the model's G1 arithmetic for a
trapdoor key (s_j = τ^j, where the sum is the closed form L_i(τ) = ω^i·(τ^n − 1) / (n·(τ − ω^i))) and for the synthetic
family s_j = a + j·d of model.synthetic_bases.  A τ on the domain makes all but one L_i(τ) zero: the harness must report it."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host_emu", "emu_lagrange.cpp")
TAU = 0x1234_5678_9ABC_DEF0_0FED_CBA9_8765_4321


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_lagrange") / "emu_lagrange.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-o", out])
    return ctypes.CDLL(out)


def _pack(points):
    return np.array([model.to_limbs(model.fp_to_mont(x), 6) + model.to_limbs(model.fp_to_mont(y), 6) for x, y in points], dtype=np.uint64)


def _unpack(rows):
    return [(model.fp_from_mont(model.from_limbs(r[:6])), model.fp_from_mont(model.from_limbs(r[6:]))) for r in rows]


def emu_lagrange(lib, points, log_n):
    bases = _pack(points)
    out = np.zeros_like(bases)
    deg = lib.emu_lagrange(ctypes.c_void_p(bases.ctypes.data), ctypes.c_uint32(log_n), ctypes.c_void_p(out.ctypes.data))
    return deg, out


def lagrange_scalars(s, log_n):
    n = 1 << log_n
    d = model.domain(n)
    w_inv, n_inv = d["group_gen_inv"], d["size_inv"]
    return [n_inv * sum(pow(w_inv, i * j, model.R) * s[j] for j in range(n)) % model.R for i in range(n)]


@pytest.mark.parametrize("log_n", range(1, 7))
def test_trapdoor_key(emu, log_n):
    n = 1 << log_n
    s = [pow(TAU, j, model.R) for j in range(n)]
    deg, out = emu_lagrange(emu, [model.g1_mul(model.G1_GEN, v) for v in s], log_n)
    assert deg == 0
    w = model.domain(n)["group_gen"]
    closed = [pow(w, i, model.R) * (pow(TAU, n, model.R) - 1) * pow(n * (TAU - pow(w, i, model.R)), -1, model.R) % model.R for i in range(n)]
    assert closed == lagrange_scalars(s, log_n)
    assert _unpack(out) == [model.g1_mul(model.G1_GEN, v) for v in closed]


@pytest.mark.parametrize("log_n", range(1, 7))
def test_synthetic_key(emu, log_n):
    n = 1 << log_n
    a, d = 0xB2000001, 0x9E3779B1
    deg, out = emu_lagrange(emu, model.synthetic_bases(n, a, d), log_n)
    assert deg == 0
    assert _unpack(out) == [model.g1_mul(model.G1_GEN, v) for v in lagrange_scalars([a + j * d for j in range(n)], log_n)]


def test_tau_on_the_domain_is_reported(emu):
    log_n = 3
    n = 1 << log_n
    tau = pow(model.domain(n)["group_gen"], 5, model.R)
    deg, out = emu_lagrange(emu, [model.g1_mul(model.G1_GEN, pow(tau, j, model.R)) for j in range(n)], log_n)
    assert deg == 1
    got = _unpack(out)
    assert got[5] == model.G1_GEN                     # L_5(ω^5) = 1
    assert all(got[i] == (0, 0) for i in range(n) if i != 5)
