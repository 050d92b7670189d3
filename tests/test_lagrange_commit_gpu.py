"""GPU tests of the Lagrange-basis commit key (csrc/lagrange.cu) and of the round-1 commitments the prover makes against it
(csrc/plonk.cu): key points against closed forms, commitments from evaluations against commitments from coefficients,
byte-identical proofs with PB200_LAGRANGE_COMMIT on and off, the fallbacks, and the key's device memory."""
import os

import numpy as np
import pytest

import model

pytestmark = pytest.mark.gpu

TAU = 0x5EED_1A6_0000_0000_0000_0000_0000_0000_0000_0001
A_SYN, D_SYN = 0xB2000001, 0x9E3779B1
G_ROW = None


def mont(vals):
    import plonk_prototype_b200 as pb
    return pb.scalars_to_mont(vals)


def times_g(oracle, s):
    """s·G as canonical affine (x, y) by the C checker."""
    global G_ROW
    if G_ROW is None:
        G_ROW = oracle.g1_generator().reshape(1, 12)
    return oracle.g1_proj_to_affine_canonical(oracle.msm_naive(G_ROW, mont([s % model.R])))


def key_points(ctx, srs, n, idx):
    host = np.zeros((n, 12), np.uint64)
    ctx.d2h(host, ctx.srs_dev_ptr(srs))
    return [(model.fp_from_mont(model.from_limbs(host[i, :6])), model.fp_from_mont(model.from_limbs(host[i, 6:]))) for i in idx]


def lagrange_at_tau(tau, n, i):
    w = pow(model.domain(n)["group_gen"], i, model.R)
    return w * (pow(tau, n, model.R) - 1) * pow(n * (tau - w), -1, model.R) % model.R


def lagrange_synthetic(n, i):
    """n⁻¹·Σ_j ω^(−ij)·(a + j·d): Σ_j x^j = 0 and Σ_j j·x^j = n / (x − 1) for x = ω^(−i) ≠ 1."""
    if i == 0:
        return (A_SYN + D_SYN * (n - 1) * pow(2, -1, model.R)) % model.R
    x = pow(model.domain(n)["group_gen_inv"], i, model.R)
    return D_SYN * pow(x - 1, -1, model.R) % model.R


def indices(log_n):
    n = 1 << log_n
    if log_n <= 12:
        return list(range(n))
    rng = np.random.default_rng(log_n)
    return sorted({0, 1, n // 2, n - 1} | set(int(v) for v in rng.integers(0, n, 60)))


@pytest.mark.parametrize("log_n", list(range(1, 13)) + [16, 20])
def test_trapdoor_key_points(ctx, oracle, log_n):
    n = 1 << log_n
    srs = ctx.srs_generate(mont([TAU]), n)
    lag = ctx.srs_lagrange(srs, log_n)
    try:
        idx = indices(log_n)
        assert key_points(ctx, lag, n, idx) == [times_g(oracle, lagrange_at_tau(TAU, n, i)) for i in idx]
    finally:
        ctx.srs_free(lag)
        ctx.srs_free(srs)


@pytest.mark.parametrize("log_n", list(range(1, 13)) + [16, 20])
def test_synthetic_key_points(ctx, oracle, log_n):
    n = 1 << log_n
    dev = ctx.malloc(n * 96)
    ctx.synthetic_bases_dev(dev, n, A_SYN, D_SYN)
    srs = ctx.srs_wrap_dev(dev, n)
    lag = ctx.srs_lagrange(srs, log_n)
    try:
        idx = indices(log_n)
        assert key_points(ctx, lag, n, idx) == [times_g(oracle, lagrange_synthetic(n, i)) for i in idx]
    finally:
        ctx.srs_free(lag)
        ctx.srs_free(srs)
        ctx.free(dev)


def test_key_from_more_points_and_tau_on_the_domain(ctx, oracle):
    import plonk_prototype_b200 as pb
    srs = ctx.srs_generate(mont([TAU]), 100)
    lag = ctx.srs_lagrange(srs, 6)                       # the first 64 of 100 points
    assert key_points(ctx, lag, 64, [0, 5, 63]) == [times_g(oracle, lagrange_at_tau(TAU, 64, i)) for i in (0, 5, 63)]
    ctx.srs_free(lag)
    with pytest.raises(pb.Pb200Error):
        ctx.srs_lagrange(srs, 7)                         # more points than the key has
    ctx.srs_free(srs)
    srs = ctx.srs_generate(mont([pow(model.domain(8)["group_gen"], 3, model.R)]), 8)
    with pytest.raises(pb.Pb200Error, match="identity"):
        ctx.srs_lagrange(srs, 3)
    ctx.srs_free(srs)


def _vectors(n, seed):
    rng = np.random.default_rng(seed)
    dense = [int(v) for v in rng.integers(0, 2**62, n)]
    dense = [(v * 0x9E3779B97F4A7C15 * (i + 1) ** 5) % model.R for i, v in enumerate(dense)]
    one = [0] * n
    one[n // 3] = (0xABCDEF << 200) + 17
    small = [int(v) for v in rng.integers(0, 2, n)]
    small[::7] = [int(v) for v in rng.integers(0, 1 << 19, len(small[::7]))]
    half = [v if i % 2 else 0 for i, v in enumerate(dense)]
    return {"dense": dense, "zero": [0] * n, "one": one, "small": small, "half": half}


@pytest.mark.parametrize("log_n", [10, 16, 20])
def test_commit_from_evaluations_equals_commit_from_coefficients(ctx, log_n):
    import plonk_prototype_b200 as pb
    n = 1 << log_n
    pp = pb.PublicParameters(n - 1, TAU, ctx)
    lag = ctx.srs_lagrange(pp.srs, log_n)
    ctx.srs_precompute(lag)
    vec = _vectors(n, log_n)
    cases = [[k] for k in ("dense", "zero", "one", "small")] + [["dense", "zero", "one", "small"], ["half", "small", "one", "dense"]]
    ev_dev, co_dev = ctx.malloc(4 * n * 32), ctx.malloc(4 * n * 32)
    try:
        for names in cases:
            evals = np.concatenate([mont(vec[k]) for k in names]).reshape(-1, 4)
            ctx.h2d(ev_dev, evals)
            ctx.h2d(co_dev, evals)
            ctx.ntt_batch_dev(co_dev, log_n, len(names), inverse=True)
            b = len(names)
            got = ctx.msm_batch_dev(lag, ev_dev, n, b, n)
            want = ctx.msm_batch_dev(pp.srs, co_dev, n, b, n)
            got, want = np.asarray(got).reshape(b, 18), np.asarray(want).reshape(b, 18)
            for j in range(b):
                assert pb.g1_to_bytes(got[j]) == pb.g1_to_bytes(want[j]), (names, j)
            if names == ["zero"]:
                assert pb.g1_to_bytes(got[0]) == bytes([0xC0]) + bytes(47)
    finally:
        ctx.free(ev_dev)
        ctx.free(co_dev)
        ctx.srs_free(lag)
        pp.close()


def _with_switch(value, fn):
    old = os.environ.get("PB200_LAGRANGE_COMMIT")
    os.environ["PB200_LAGRANGE_COMMIT"] = value
    try:
        return fn()
    finally:
        if old is None:
            del os.environ["PB200_LAGRANGE_COMMIT"]
        else:
            os.environ["PB200_LAGRANGE_COMMIT"] = old


def _prove(ctx, srs, sel, wires, values, pos, piv, label):
    pk, vk = ctx.preprocess(srs, sel, wires, values.shape[0], label)
    try:
        return ctx.prove(srs, pk, values, pos, piv), vk, ctx.prover_key_bytes(pk)
    finally:
        ctx.prover_key_free(pk)


def _on_off(ctx, srs, sel, wires, values, pos, piv, label):
    on = _with_switch("1", lambda: _prove(ctx, srs, sel, wires, values, pos, piv, label))
    off = _with_switch("0", lambda: _prove(ctx, srs, sel, wires, values, pos, piv, label))
    return on, off


@pytest.mark.parametrize("log_n", [12, 16, 20])
def test_synthetic_proofs_identical_with_switch_on_and_off(ctx, log_n):
    import plonk_prototype_b200 as pb
    from plonk_prototype_b200.synth import synthetic_circuit_columns
    n = 1 << log_n
    sel, wires, values, pos, piv = synthetic_circuit_columns(n)
    pp = pb.PublicParameters(n - 1, TAU, ctx)
    try:
        (p1, vk1, b1), (p0, vk0, b0) = _on_off(ctx, pp.srs, sel, wires, values, pos, piv, b"lagrange")
    finally:
        pp.close()
    assert p1 == p0 and vk1 == vk0
    w_pre = -(-256 // 20) if log_n == 20 else None
    assert b1 > b0                                                       # the Lagrange key was built …
    if w_pre:
        assert b1 - b0 == (w_pre + 1) * n * 96                           # … with its pre-doubled copies (c = 20 at 2^20)
    assert pb.verify(vk1, n, b"lagrange", p1, pos, piv, pp.beta_h)


def _gadget(which):
    import plonk_prototype_b200 as pb
    G, jj = pb.gadgets, pb.jubjub
    cs = pb.StandardComposer()
    if which == "commitment_gadget":
        value, blinder = 0x1234567890ABCDEF, 0xFEDCBA9876543210FEDCBA
        point = G.commitment_gadget(cs, cs.add_input(value), cs.add_input(blinder))
        cs.assert_equal_public_point(point, jj.add(jj.mul(jj.GENERATOR, value), jj.mul(jj.GENERATOR_NUMS, blinder)))
    elif which == "prove_ownership":
        sk = 0x0A11CE5EC2E7
        G.MockCircuit(None, private_key=cs.add_input(sk), public_key=jj.mul(jj.GENERATOR, sk)).prove_ownership(cs)
    else:
        a, b = 0x9E3779B97F4A7C15, 0xBF58476D1CE4E5B9
        x = cs.xor_gate(cs.add_input(a), cs.add_input(b), 64)
        y = cs.and_gate(cs.add_input(a), cs.add_input(b), 64)
        cs.constrain_to_constant(x, 0, -(a ^ b))
        cs.constrain_to_constant(y, a & b, None)
    return cs


@pytest.mark.parametrize("which", ["commitment_gadget", "prove_ownership", "logic"])
def test_gadget_proofs_identical_with_switch_on_and_off(ctx, which):
    import plonk_prototype_b200 as pb
    cs = _gadget(which)
    n = 1
    while n < cs.n:
        n *= 2
    pis = sorted(cs.public_inputs_sparse_store.items())
    pos = np.asarray([p for p, _ in pis], dtype=np.uint32)
    piv = mont([v for _, v in pis]) if pis else np.zeros((0, 4), np.uint64)
    pp = pb.PublicParameters(n - 1, 0xECC0, ctx)
    try:
        (p1, vk1, b1), (p0, vk0, b0) = _on_off(ctx, pp.srs, cs.selector_columns(), cs.wire_columns(), mont(cs.variables), pos, piv,
                                               which.encode())
    finally:
        pp.close()
    assert b1 > b0
    assert p1 == p0 and vk1 == vk0
    assert pb.verify(vk1, n, which.encode(), p1, pos, piv, pp.beta_h)


def test_fallbacks_keep_the_monomial_path(ctx):
    """No pre-doubled copies, or a point-range-sharded key: no Lagrange key is built (same device memory either way)."""
    import plonk_prototype_b200 as pb
    from plonk_prototype_b200.synth import synthetic_circuit_columns
    n = 1 << 12
    sel, wires, values, pos, piv = synthetic_circuit_columns(n)
    pp = pb.PublicParameters(n - 1, TAU, ctx, precompute=False)
    try:
        (p1, _, b1), (p0, _, b0) = _on_off(ctx, pp.srs, sel, wires, values, pos, piv, b"fallback")
    finally:
        pp.close()
    assert b1 == b0 and p1 == p0
    # a sharded key (rank 0 of 2, the all-gather played by this process): the commit key slice has pre-doubled copies
    srs = ctx.srs_generate(mont([TAU]), n // 2)
    ctx.srs_precompute(srs)

    def key_bytes():
        pk, _ = ctx.preprocess(srs, sel, wires, values.shape[0], b"fallback", shard=(0, 2, lambda send: bytes(send) * 2))
        try:
            return ctx.prover_key_bytes(pk)
        finally:
            ctx.prover_key_free(pk)
    try:
        assert _with_switch("1", key_bytes) == _with_switch("0", key_bytes)
    finally:
        ctx.srs_free(srs)


def test_device_memory_returns_after_key_free(ctx):
    import torch
    import plonk_prototype_b200 as pb
    from plonk_prototype_b200.synth import synthetic_circuit_columns
    n = 1 << 16
    sel, wires, values, pos, piv = synthetic_circuit_columns(n)
    pp = pb.PublicParameters(n - 1, TAU, ctx)
    try:
        _with_switch("1", lambda: _prove(ctx, pp.srs, sel, wires, values, pos, piv, b"mem"))  # grow the workspaces once
        ctx.sync()
        free0 = torch.cuda.mem_get_info(ctx.device)[0]
        pk, _ = _with_switch("1", lambda: ctx.preprocess(pp.srs, sel, wires, values.shape[0], b"mem"))
        ctx.sync()
        held = ctx.prover_key_bytes(pk)
        assert free0 - torch.cuda.mem_get_info(ctx.device)[0] >= held - (8 << 20)
        ctx.prover_key_free(pk)
        ctx.sync()
        assert abs(torch.cuda.mem_get_info(ctx.device)[0] - free0) <= (16 << 20)
    finally:
        pp.close()
