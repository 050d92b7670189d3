"""CPU tests of the batched verifier's per-proof derivation (csrc/verify_batch.cuh: the code verify_prepare_kernel and
verify_weight_kernel run), compiled for the host with the carry-flag primitives emulated (PB200_HOST_EMU,
tests/host_emu/emu_verify.cpp).

With a known trapdoor τ the pairing equation e(−W, τH)·e(C, H) = 1 is the G1 equation C = τ·W.  For every case the
emulated coefficients are applied to the proof's points with the model's G1 arithmetic, and C = τ·W must hold exactly
when the model verifier (oracle/plonk_model.py) accepts.  The emulated z and u must be the model transcript's, and the
batch weights ρ_k restated with the model's Merlin transcript must equal the emulated ones."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import model
import plonk_model as pm
from helpers import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host_emu", "emu_verify.cpp")
IDENTITY = bytes([0xC0]) + bytes(47)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_verify") / "emu_verify.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-o", out])
    return ctypes.CDLL(out)


def _vp(a):
    return ctypes.c_void_p(a.ctypes.data)


def _mont(v):
    return np.array(model.to_limbs(model.fr_to_mont(v % model.R), 4), dtype=np.uint64)


def _unmont(limbs):
    return model.fr_from_mont(model.from_limbs([int(x) for x in limbs]))


def emu_prepare(lib, label, vkb, n, proof, pi):
    items = sorted(pi.items())
    gates = np.asarray([g for g, _ in items] or [0], dtype=np.uint32)
    vals = np.stack([_mont(v) for _, v in items]) if items else np.zeros((1, 4), np.uint64)
    lab = np.frombuffer(bytes(label) + b"\0", dtype=np.uint8).copy()
    vk = np.frombuffer(bytes(vkb), dtype=np.uint8).copy()
    pr = np.frombuffer(bytes(proof), dtype=np.uint8).copy()
    coef, e, zu = np.zeros((11, 4), np.uint64), np.zeros((16, 4), np.uint64), np.zeros((2, 4), np.uint64)
    dig = np.zeros(32, np.uint8)
    st = lib.emu_verify_prepare(_vp(lab), ctypes.c_size_t(len(label)), _vp(vk), ctypes.c_uint64(n), _vp(pr), _vp(gates), _vp(vals),
                                ctypes.c_size_t(len(items)), _vp(coef), _vp(e), _vp(zu), _vp(dig))
    return st, [_unmont(c) for c in coef], [_unmont(c) for c in e], _unmont(zu[0]), _unmont(zu[1]), dig.tobytes()


def emu_weights(lib, seed, n, digests):
    K = len(digests) // 32
    d = np.frombuffer(digests, dtype=np.uint8).copy()
    s = np.frombuffer(seed, dtype=np.uint8).copy()
    D = np.zeros(32, np.uint8)
    rho = np.zeros((K, 4), np.uint64)
    lib.emu_verify_weights(_vp(s), ctypes.c_uint64(n), ctypes.c_uint64(K), _vp(d), _vp(D), _vp(rho))
    return D.tobytes(), [_unmont(r) for r in rho]


def model_z_u(vk, proof, pi, label):
    """z and u of Proof::verify's transcript, restated with the model (no group arithmetic)."""
    pr = pm.proof_from_bytes(proof)
    t = pm.Transcript(label)
    pm.seed_transcript(t, vk)
    n = vk["n"]
    d = pm.domain(n)
    ev = pr["evals"]
    for i, lab in enumerate((b"w_l", b"w_r", b"w_o", b"w_4")):
        t.append_message(lab, proof[48 * i:48 * i + 48])
    beta = t.challenge_scalar(b"beta")
    t.append_scalar(b"beta", beta)
    gamma = t.challenge_scalar(b"gamma")
    t.append_message(b"z", proof[192:240])
    alpha = t.challenge_scalar(b"alpha")
    seps = [t.challenge_scalar(lab) for lab in (b"range separation challenge", b"logic separation challenge",
                                                b"fixed base separation challenge", b"variable base separation challenge")]
    for i, lab in enumerate((b"t_1", b"t_2", b"t_3", b"t_4")):
        t.append_message(lab, proof[240 + 48 * i:288 + 48 * i])
    z = t.challenge_scalar(b"z")
    R = model.R
    lin = pm.linearisation_terms(ev, alpha, beta, gamma, seps, z, d)
    z_h, l1 = lin["z_h"], lin["l1"]
    w = d["group_gen"]
    pi_eval = 0
    for i, v in pi.items():
        wi = pow(w, i, R)
        pi_eval = (pi_eval + v * wi % R * pow((z - wi) % R, -1, R)) % R
    pi_eval = pi_eval * z_h % R * d["size_inv"] % R
    a, b, c, dd = ev["a_eval"], ev["b_eval"], ev["c_eval"], ev["d_eval"]
    bprod = ((a + beta * ev["left_sigma_eval"] + gamma) * (b + beta * ev["right_sigma_eval"] + gamma) % R
             * (c + beta * ev["out_sigma_eval"] + gamma) % R * ((dd + gamma) * ev["perm_eval"] % R * alpha % R)) % R
    t_eval = (ev["lin_poly_eval"] + pi_eval - bprod - l1 * alpha * alpha) % R * pow(z_h, -1, R) % R
    for lab, key in pm.EVAL_TRANSCRIPT_ORDER:
        t.append_scalar(lab, t_eval if key == "t_eval" else ev[key])
    t.challenge_scalar(b"aggregate_witness")
    t.challenge_scalar(b"aggregate_witness")
    t.append_message(b"w_z", proof[432:480])
    t.append_message(b"w_z_w", proof[480:528])
    return z, t.challenge_scalar(b"batch"), t


def vk_from_bytes(vkb, n):
    pts = [pm.bytes_to_g1(vkb[48 * i:48 * i + 48]) for i in range(15)]
    return {"n": n, "q": dict(zip(pm.SELECTORS, pts[:11])), "sigma": pts[11:]}


def combined(coef, e, u, vkb, proof):
    """(C, W) of the proof's pairing equation from the emulated coefficients."""
    pts = [pm.bytes_to_g1(proof[48 * i:48 * i + 48]) for i in range(11)]
    shared = [pm.bytes_to_g1(vkb[48 * j:48 * j + 48]) for j in range(15)] + [model.G1_GEN]
    C = model.msm_naive(pts + shared, coef + e)
    W = model.g1_add(pts[9], model.g1_mul(pts[10], u))
    return C, W


# ------------------------------------------------------------------------------------------------ the cases
def golden_cases():
    g = load_golden("plonk_kat.json")
    tau, label = int(g["tau"], 16), g["label"].encode()
    out = []
    for case in g["cases"]:
        pi = {int(k): int(v, 16) for k, v in case["pi"].items()}
        out.append((case["name"], tau, label, bytes.fromhex(case["vk"]), case["n"], bytes.fromhex(case["proof"]), pi))
    return out


def identity_circuit():
    """A circuit without dummy rows whose fourth wire is identically zero: its proof commits to the zero polynomial."""
    comp = pm.Composer(with_dummy=False)
    x, y = comp.add_input(5), comp.add_input(7)
    for k in range(10):
        x = comp.add((1, x), (1, y), k, 0)
    p = comp.mul(1, x, y, 0, 0)
    comp.constrain_to_constant(p, 0, -comp.values[p])
    assert comp.check() and comp.n == 13
    return comp


@pytest.fixture(scope="module")
def identity_case():
    comp = identity_circuit()
    n = pm.domain(comp.n)["size"]
    tau, label = 0x1D3A7, b"identity commitment"
    ck = pm.srs_setup(tau, n)
    pk, vk, tr = pm.preprocess(comp, ck, label)
    _, proof = pm.prove(comp, pk, ck, tr)
    vkb = b"".join(model.g1_compress(vk["q"][k]) for k in pm.SELECTORS) + b"".join(model.g1_compress(s) for s in vk["sigma"])
    return ("identity", tau, label, vkb, n, proof, dict(comp.pi))


def tampered(case):
    name, tau, label, vkb, n, proof, pi = case
    out = []

    def edit(tag, f, **kw):
        b = bytearray(proof)
        f(b)
        out.append((name + "/" + tag, tau, kw.get("label", label), vkb, n, bytes(b), kw.get("pi", pi)))

    edit("eval_canonical", lambda b: b.__setitem__(528 + 5, b[528 + 5] ^ 0x10))
    edit("eval_ge_r", lambda b: b.__setitem__(slice(528 + 32, 528 + 64), b"\xff" * 32))
    edit("point_byte", lambda b: b.__setitem__(48 * 4 + 20, b[48 * 4 + 20] ^ 0x01))
    edit("bad_flags", lambda b: b.__setitem__(48 * 2, b[48 * 2] & 0x7F))
    edit("identity_for_point", lambda b: b.__setitem__(slice(48 * 5, 48 * 6), IDENTITY))
    edit("swap_openings", lambda b: b.__setitem__(slice(432, 528), proof[480:528] + proof[432:480]))
    k = next(iter(pi))
    edit("wrong_pi", lambda b: None, pi={**pi, k: (pi[k] + 1) % model.R})
    edit("label", lambda b: None, label=b"another label")
    return out


def check_case(emu, case):
    name, tau, label, vkb, n, proof, pi = case
    vk = vk_from_bytes(vkb, n)
    accepted = pm.verify(vk, proof, pi, pm.opening_key(tau), label)
    st, coef, e, z, u, _ = emu_prepare(emu, label, vkb, n, proof, pi)
    if st != 0:
        assert not accepted, name
        return st
    mz, mu, _ = model_z_u(vk, proof, pi, label)
    assert (z, u) == (mz, mu), name
    C, W = combined(coef, e, u, vkb, proof)
    assert (C == model.g1_mul(W, tau)) == accepted, name
    return accepted


@pytest.mark.parametrize("idx", [0, 1, 2])
def test_golden_proofs_and_tampering(emu, idx):
    case = golden_cases()[idx]
    assert check_case(emu, case) is True
    verdicts = {c[0].split("/")[1]: check_case(emu, c) for c in tampered(case)}
    assert verdicts["eval_ge_r"] == 2                      # rejected before any pairing: evaluation not below r
    assert verdicts["point_byte"] == 1 and verdicts["bad_flags"] == 1
    assert all(v is False for k, v in verdicts.items() if k not in ("eval_ge_r", "point_byte", "bad_flags")), verdicts


def test_identity_commitment_is_a_zero_term(emu, identity_case):
    name, tau, label, vkb, n, proof, pi = identity_case
    assert IDENTITY in [proof[48 * i:48 * i + 48] for i in range(11)]
    assert check_case(emu, identity_case) is True
    for c in tampered(identity_case):
        assert check_case(emu, c) is not True, c[0]


def test_weights_restated_with_model_transcript(emu):
    cases = golden_cases()
    digests = b""
    for _, tau, label, vkb, n, proof, pi in cases:
        st, _, _, _, _, dig = emu_prepare(emu, label, vkb, n, proof, pi)
        assert st == 0
        # the digest: the proof's transcript after u, its public inputs appended
        _, _, t = model_z_u(vk_from_bytes(vkb, n), proof, pi, label)
        for g in sorted(pi):
            t.append_scalar(b"pi", pi[g])
        assert t.challenge_bytes(b"batch digest", 32) == dig
        digests += dig
    for seed in (bytes(32), bytes(range(32)), b"\xa5" * 32):
        D, rho = emu_weights(emu, seed, 16, digests)
        t = pm.Transcript(b"pb200 verify_batch")
        t.append_message(b"seed", seed)
        t.append_u64(b"n", 16)
        t.append_u64(b"K", 3)
        t.append_message(b"digests", digests)
        assert t.challenge_bytes(b"D", 32) == D
        rt = pm.Transcript(b"pb200 rho")
        rt.append_message(b"D", D)
        for k in range(3):
            tk = rt.clone()
            tk.append_u64(b"k", k)
            assert tk.challenge_scalar(b"rho") == rho[k]
        assert len(set(rho)) == 3
