"""GPU tests of pb200_verify_batch (csrc/verify_batch.cu): every verdict of a batch equals pb200_verify's on that proof,
an all-valid batch costs exactly one pairing check, bisection finds the invalid proofs, and the weights bind the public
inputs (a pair of proofs whose errors cancel in an unweighted sum is rejected)."""
import ctypes
import os
import sys

import numpy as np
import pytest

import model
import plonk_model as pm

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_verify_batch_cpu import IDENTITY, identity_circuit, model_z_u, vk_from_bytes  # noqa: E402

pytestmark = pytest.mark.gpu

LABEL = b"pb200 batch verify"
TAU = 0xBA7C4
N_GATES = 1000


def synthetic_circuit_x0(n_gates, x0, seed=0xB47C, n_pub=2):
    """pm.synthetic_circuit with the chain's starting value x0 as a parameter: the circuit (every selector and wire) does
    not depend on x0, the witness and the public inputs do."""
    from model import random_fr
    comp = pm.Composer()
    consts = random_fr(seed, 4)
    x = comp.add_input(x0)
    k = 0
    while comp.n + 2 <= n_gates - n_pub:
        sq = comp.mul(1, x, x, 0, 0)
        x = comp.add((1, sq), (1, x), (consts[1] + k) % model.R, 0)
        k += 1
    while comp.n < n_gates - n_pub:
        comp.boolean_gate(comp.zero_var)
    for j in range(n_pub):
        v = comp.values[x] if j == 0 else consts[2]
        var = x if j == 0 else comp.add_input(v)
        comp.constrain_to_constant(var, 0, -v)
    assert comp.n == n_gates and comp.check()
    return comp


def mont(vals):
    import plonk_prototype_b200 as pb
    return pb.scalars_to_mont([v % model.R for v in vals])


def columns(comp):
    sel = [mont(comp.q[k]) if any(comp.q[k]) else None for k in pm.SELECTORS]
    return sel, [np.asarray(w, dtype=np.uint32) for w in comp.w]


class Supply:
    pass


@pytest.fixture(scope="module")
def supply(ctx, oracle):
    """64 valid proofs of one circuit (distinct witnesses and public inputs), a proof of another circuit, a proof under
    another label, and a proof containing the identity commitment, with everything needed to verify them."""
    import plonk_prototype_b200 as pb
    s = Supply()
    comps = [synthetic_circuit_x0(N_GATES, 3 + 7 * i) for i in range(64)]
    s.n = pm.domain(N_GATES)["size"]
    pp = pb.PublicParameters(s.n - 1, TAU, ctx)
    s.beta_h = pp.beta_h
    sel, wires = columns(comps[0])
    pk, s.vk = ctx.preprocess(pp.srs, sel, wires, len(comps[0].values), LABEL)
    s.gates = np.asarray(sorted(comps[0].pi), dtype=np.uint32)
    s.pis = [{g: c.pi[g] for g in sorted(c.pi)} for c in comps]
    s.proofs = [ctx.prove(pp.srs, pk, mont(c.values), s.gates, mont([c.pi[g] for g in s.gates])) for c in comps]
    ctx.prover_key_free(pk)
    pk2, _ = ctx.preprocess(pp.srs, sel, wires, len(comps[0].values), b"another label")
    s.other_label = ctx.prove(pp.srs, pk2, mont(comps[0].values), s.gates, mont([comps[0].pi[g] for g in s.gates]))
    ctx.prover_key_free(pk2)
    other = pm.synthetic_circuit(N_GATES, seed=0x0C1C)
    osel, owires = columns(other)
    pk3, _ = ctx.preprocess(pp.srs, osel, owires, len(other.values), LABEL)
    og = np.asarray(sorted(other.pi), dtype=np.uint32)
    assert (og == s.gates).all()
    s.other_circuit = ctx.prove(pp.srs, pk3, mont(other.values), og, mont([other.pi[g] for g in og]))
    ctx.prover_key_free(pk3)
    # the identity-commitment proof, with its own key
    ic = identity_circuit()
    s.id_n = pm.domain(ic.n)["size"]
    isel, iwires = columns(ic)
    pk4, s.id_vk = ctx.preprocess(pp.srs, isel, iwires, len(ic.values), LABEL)
    s.id_gates = np.asarray(sorted(ic.pi), dtype=np.uint32)
    s.id_pi = {g: ic.pi[g] for g in s.id_gates}
    s.id_proof = ctx.prove(pp.srs, pk4, mont(ic.values), s.id_gates, mont([ic.pi[g] for g in s.id_gates]))
    ctx.prover_key_free(pk4)
    pp.close()
    return s


def pi_array(pis, gates):
    return np.stack([mont([pi[int(g)] for g in gates]) for pi in pis]) if len(gates) else np.zeros((len(pis), 0, 4), np.uint64)


def single(s, proof, pi, vk=None, n=None, gates=None, beta_h=None):
    import plonk_prototype_b200 as pb
    gates = s.gates if gates is None else gates
    return pb.verify(vk or s.vk, n or s.n, LABEL, proof, gates, mont([pi[int(g)] for g in gates]), s.beta_h if beta_h is None else beta_h)


def batch(ctx, s, proofs, pis, seed=b"\x01" * 32, vk=None, n=None, gates=None, beta_h=None):
    """(verdicts, number of pairing checks) of one pb200_verify_batch call."""
    gates = s.gates if gates is None else gates
    ctx.profile_enable(True)
    ctx.profile_reset()
    got = ctx.verify_batch(vk or s.vk, n or s.n, LABEL, proofs, gates, pi_array(pis, gates), s.beta_h if beta_h is None else beta_h, seed)
    checks = ctx.profile_sum_ms("verify.pairing")[1]
    ctx.profile_enable(False)
    return got, checks


def tampers(s):
    """(name, proof bytes, public inputs) of every tamper class, each built from a valid proof."""
    import srs_io_ref as ref
    data, labels = ref.corpus()
    outside = next(data[48 * i:48 * i + 48] for i, st in enumerate(labels) if st == ref.NOT_IN_SUBGROUP)
    p, pi = s.proofs[5], s.pis[5]

    def ed(f):
        b = bytearray(p)
        f(b)
        return bytes(b)

    g0 = int(s.gates[0])
    return [
        ("eval_canonical", ed(lambda b: b.__setitem__(528 + 5, b[528 + 5] ^ 0x10)), pi),
        ("eval_ge_r", ed(lambda b: b.__setitem__(slice(528 + 32, 528 + 64), b"\xff" * 32)), pi),
        ("point_byte", ed(lambda b: b.__setitem__(48 * 4 + 20, b[48 * 4 + 20] ^ 0x01)), pi),
        ("bad_flags", ed(lambda b: b.__setitem__(48 * 2, b[48 * 2] & 0x7F)), pi),
        ("not_in_g1", ed(lambda b: b.__setitem__(slice(48 * 1, 48 * 2), outside)), pi),
        ("identity_for_point", ed(lambda b: b.__setitem__(slice(48 * 6, 48 * 7), IDENTITY)), pi),
        ("wrong_pi", p, {**pi, g0: (pi[g0] + 1) % model.R}),
        ("other_label", s.other_label, s.pis[0]),
        ("other_circuit", s.other_circuit, s.pis[0]),
        ("swap_openings", ed(lambda b: b.__setitem__(slice(432, 528), p[480:528] + p[432:480])), pi),
        ("mixed_proofs", s.proofs[7][:528] + s.proofs[8][528:], s.pis[7]),
    ]


@pytest.mark.parametrize("K", [1, 2, 3, 64, 4096, 16384])
def test_all_valid_batch_is_one_pairing_check(ctx, supply, K):
    s = supply
    idx = [k % 64 for k in range(K)]
    got, checks = batch(ctx, s, [s.proofs[i] for i in idx], [s.pis[i] for i in idx])
    assert got.all() and got.size == K
    assert checks == 1
    if K <= 3:
        assert all(single(s, s.proofs[i], s.pis[i]) for i in idx)


@pytest.mark.parametrize("K", [64, 4096])
def test_mixed_batch_matches_single_verifier(ctx, supply, K):
    s = supply
    bad = tampers(s)
    proofs = [s.proofs[k % 64] for k in range(K)]
    pis = [s.pis[k % 64] for k in range(K)]
    mid = K // 2
    spots = [0, K - 1, mid, mid + 1, mid - 1, 3, K // 4, K // 4 + 1, 3 * K // 4, K - 2, 9]
    assert len(set(spots)) == len(bad)
    want = [True] * K
    for pos, (name, p, pi) in zip(spots, bad):
        proofs[pos], pis[pos] = p, pi
        want[pos] = single(s, p, pi)
        assert want[pos] is False, name
    got, checks = batch(ctx, s, proofs, pis)
    assert list(got) == want
    b = len(bad)
    assert checks <= 1 + 2 * b * int(np.ceil(np.log2(K)))


def test_cancelling_pair_is_rejected(ctx, supply):
    """Proofs a and b with the public input at gate g shifted by δ_a and δ_b = −δ_a·(z_b − ω^g)/(z_a − ω^g): each is invalid
    and their unweighted sum is the identity.  The weights bind the public inputs, so both are rejected."""
    s = supply
    R = model.R
    vk = vk_from_bytes(s.vk, s.n)
    g = int(s.gates[1])
    wg = pow(pm.domain(s.n)["group_gen"], g, R)
    a, b = 10, 11
    za = model_z_u(vk, s.proofs[a], s.pis[a], LABEL)[0]
    zb = model_z_u(vk, s.proofs[b], s.pis[b], LABEL)[0]
    da = 12345
    db = (-da * (zb - wg) * pow(za - wg, -1, R)) % R
    pa = {**s.pis[a], g: (s.pis[a][g] + da) % R}
    pb_ = {**s.pis[b], g: (s.pis[b][g] + db) % R}
    assert not single(s, s.proofs[a], pa) and not single(s, s.proofs[b], pb_)
    proofs = [s.proofs[k] for k in range(64)]
    pis = list(s.pis)
    pis[a], pis[b] = pa, pb_
    for seed in (bytes(32), b"\x42" * 32, bytes(range(32))):
        got, _ = batch(ctx, s, proofs, pis, seed=seed)
        assert [k for k in range(64) if not got[k]] == [a, b]


@pytest.mark.parametrize("b", [1, 2, 17])
def test_bisection_finds_invalid_proofs(ctx, supply, b):
    s = supply
    K = 4096
    rng = np.random.default_rng(0xB15EC + b)
    bad_pos = sorted(rng.choice(K, size=b, replace=False).tolist())
    proofs = [s.proofs[k % 64] for k in range(K)]
    pis = [s.pis[k % 64] for k in range(K)]
    for pos in bad_pos:
        p = bytearray(proofs[pos])
        p[528 + 5] ^= 0x10                                  # a_eval changed, still canonical: only the pairing can tell
        proofs[pos] = bytes(p)
    got, checks = batch(ctx, s, proofs, pis)
    assert [k for k in range(K) if not got[k]] == bad_pos
    assert checks <= 1 + 2 * b * 12


def test_identity_commitment_proof(ctx, supply):
    s = supply
    assert IDENTITY in [s.id_proof[48 * i:48 * i + 48] for i in range(11)]
    assert single(s, s.id_proof, s.id_pi, vk=s.id_vk, n=s.id_n, gates=s.id_gates)
    got, checks = batch(ctx, s, [s.id_proof], [s.id_pi], vk=s.id_vk, n=s.id_n, gates=s.id_gates)
    assert list(got) == [True] and checks == 1
    bad = bytearray(s.id_proof)
    bad[528 + 5] ^= 0x10
    got, _ = batch(ctx, s, [s.id_proof, bytes(bad), s.id_proof], [s.id_pi] * 3, vk=s.id_vk, n=s.id_n, gates=s.id_gates)
    assert list(got) == [True, False, True]


def test_whole_batch_cases(ctx, supply):
    import plonk_prototype_b200 as pb
    s = supply
    proofs, pis = s.proofs[:16], s.pis[:16]
    vk = bytearray(s.vk)
    vk[48 * 3] &= 0x7F                                       # q_o: bad flags
    assert not single(s, proofs[0], pis[0], vk=bytes(vk))
    got, checks = batch(ctx, s, proofs, pis, vk=bytes(vk))
    assert not got.any() and checks == 0
    other_bh = pb.opening_key_from_tau(mont([TAU + 1]))
    assert not single(s, proofs[0], pis[0], beta_h=other_bh)
    got, _ = batch(ctx, s, proofs, pis, beta_h=other_bh)
    assert not got.any()
    mixed = list(proofs)
    mixed[4] = tampers(s)[0][1]
    g1, _ = batch(ctx, s, mixed, pis, seed=b"\x07" * 32)
    g2, _ = batch(ctx, s, mixed, pis, seed=b"\x08" * 32)
    assert list(g1) == list(g2) == [k != 4 for k in range(16)]


def test_argument_errors(ctx, supply):
    import plonk_prototype_b200 as pb
    L = pb._native.lib()
    s = supply
    K = 2
    vk = np.frombuffer(s.vk, np.uint8).copy()
    pr = np.frombuffer(s.proofs[0] + s.proofs[1], np.uint8).copy()
    gates = s.gates.copy()
    piv = pi_array(s.pis[:2], gates)
    bh = np.ascontiguousarray(s.beta_h, dtype=np.uint64)
    seed = np.zeros(32, np.uint8)
    acc = np.zeros(K, np.uint8)
    allok = ctypes.c_int(7)
    P = pb._native._ptr

    def call(vk=P(vk), n=s.n, label=LABEL, pr=P(pr), k=K, gates=P(gates), piv=P(piv), n_pi=gates.size, bh=P(bh), seed=P(seed), acc=P(acc)):
        return L.pb200_verify_batch(ctx._h, vk, n, label, len(label) if label else 0, pr, k, gates, piv, n_pi, bh, seed, acc, ctypes.byref(allok))

    assert call() == 0 and allok.value == 1 and list(acc) == [1, 1]
    for kw in ({"vk": None}, {"pr": None}, {"bh": None}, {"seed": None}, {"acc": None}, {"gates": None}, {"piv": None},
               {"n": 0}, {"n": 1}, {"n": 3 * 1024}, {"n": 1 << 31}, {"k": 0}, {"k": (1 << 20) + 1}):
        assert call(**kw) == 1, kw
    dup = np.asarray([gates[0], gates[0]], np.uint32)
    assert call(gates=P(dup)) == 1
    big = np.asarray([gates[0], s.n], np.uint32)
    assert call(gates=P(big)) == 1
    bad_bh = bh.copy()
    bad_bh[0] ^= 1
    assert call(bh=P(bad_bh)) == 1


def test_device_memory_is_released(ctx, supply):
    import torch
    s = supply
    proofs = [s.proofs[k % 64] for k in range(4096)]
    pis = [s.pis[k % 64] for k in range(4096)]
    batch(ctx, s, proofs, pis)                               # warm-up: the MSM workspace of this size stays with the context
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    for i in range(10):
        got, _ = batch(ctx, s, proofs, pis, seed=bytes([i]) * 32)
        assert got.all()
    torch.cuda.synchronize()
    free1 = torch.cuda.mem_get_info(0)[0]
    assert abs(free1 - free0) < (32 << 20), (free0, free1)   # the device is shared: allow for other processes' noise


def test_python_wrappers_agree_with_raw_call(ctx, supply):
    import plonk_prototype_b200 as pb
    s = supply
    proofs = list(s.proofs[:8])
    proofs[2] = tampers(s)[0][1]
    piv = pi_array(s.pis[:8], s.gates)
    a = pb.verify_batch(ctx, s.vk, s.n, LABEL, proofs, s.gates, piv, s.beta_h, seed=b"\x33" * 32)
    b = ctx.verify_batch(s.vk, s.n, LABEL, b"".join(proofs), s.gates, piv, s.beta_h, seed=b"\x33" * 32)
    c = pb.verify_batch(ctx, s.vk, s.n, LABEL, proofs, s.gates, piv, s.beta_h)   # random seed
    L = pb._native.lib()
    acc = np.zeros(8, np.uint8)
    allok = ctypes.c_int(7)
    P = pb._native._ptr
    pr = np.frombuffer(b"".join(proofs), np.uint8).copy()
    seed = np.frombuffer(b"\x33" * 32, np.uint8).copy()
    assert L.pb200_verify_batch(ctx._h, P(np.frombuffer(s.vk, np.uint8).copy()), s.n, LABEL, len(LABEL), P(pr), 8, P(s.gates), P(piv),
                                s.gates.size, P(np.ascontiguousarray(s.beta_h, dtype=np.uint64)), P(seed), P(acc), ctypes.byref(allok)) == 0
    assert allok.value == 0
    assert list(a) == list(b) == list(c) == [bool(x) for x in acc] == [k != 2 for k in range(8)]
