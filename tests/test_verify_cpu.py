"""CPU tests of pb200_verify (csrc/verify.cu, host only): its verdict equals the model verifier's (oracle/plonk_model.py)
on the golden proofs, on a proof with an identity commitment and on every tampering of them, and a bad argument is
reported as PB200_ERR_ARG before any byte of the proof is looked at."""
import ctypes
import os
import sys

import numpy as np
import pytest

import plonk_model as pm

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_verify_batch_cpu import golden_cases, identity_case, tampered, vk_from_bytes  # noqa: E402,F401

PB200_ERR_ARG = 1


def raw_verify(case, gates=None, beta_h=None):
    """pb200_verify's return code and verdict; gates / beta_h replace the case's own."""
    import plonk_prototype_b200 as pb
    from plonk_prototype_b200 import _native
    _, tau, label, vkb, n, proof, pi = case
    items = sorted(pi.items())
    g = np.ascontiguousarray(gates if gates is not None else [k for k, _ in items], dtype=np.uint32)
    piv = pb.scalars_to_mont([v for _, v in items])
    bh = beta_h if beta_h is not None else pb.opening_key_from_tau(pb.scalars_to_mont([tau]))
    vk, pr = np.frombuffer(vkb, np.uint8).copy(), np.frombuffer(proof, np.uint8).copy()
    ok = ctypes.c_int(-1)
    P = _native._ptr
    rc = _native.lib().pb200_verify(P(vk), n, label, len(label), P(pr), P(g), P(piv), g.size, P(bh), ctypes.byref(ok))
    return rc, ok.value


def assert_same_verdicts(case):
    for c in [case] + tampered(case):
        name, tau, label, vkb, n, proof, pi = c
        expected = pm.verify(vk_from_bytes(vkb, n), proof, pi, pm.opening_key(tau), label)
        assert raw_verify(c) == (0, int(expected)), name


@pytest.mark.parametrize("idx", [0, 1, 2])
def test_verdicts_match_model_on_golden_proofs_and_tampering(idx):
    case = golden_cases()[idx]
    assert raw_verify(case) == (0, 1)
    assert_same_verdicts(case)


def test_verdicts_match_model_with_identity_commitment(identity_case):
    assert raw_verify(identity_case) == (0, 1)
    assert_same_verdicts(identity_case)


def test_argument_errors_come_before_the_proof():
    import plonk_prototype_b200 as pb
    case = golden_cases()[0]
    _, tau, label, vkb, n, proof, pi = case
    gates = sorted(pi)
    bad_flags, bad_eval = bytearray(proof), bytearray(proof)
    bad_flags[48 * 2] &= 0x7F
    bad_eval[528:560] = b"\xff" * 32
    off_curve = pb.opening_key_from_tau(pb.scalars_to_mont([tau])).copy()
    off_curve[0] ^= 1
    for bad in (bad_flags, bad_eval):
        malformed = case[:5] + (bytes(bad),) + case[6:]
        assert raw_verify(malformed) == (0, 0)
        for g in ([n] + gates[1:], gates[:-1] + [n + 5]):   # an out-of-range gate first or last
            assert raw_verify(malformed, gates=g)[0] == PB200_ERR_ARG, g
        assert raw_verify(malformed, beta_h=off_curve)[0] == PB200_ERR_ARG
