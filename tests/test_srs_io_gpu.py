"""GPU tests of the checked compressed commit-key format (csrc/srs_io.cu through pb200_srs_{from,to}_compressed):
`CommitKey::{from_slice, to_var_bytes}` and `PublicParameters::{from_slice, to_var_bytes}` against the CPU reference decoder
(tests/srs_io_ref.c, upstream's algorithm), bit for bit."""
import numpy as np
import pytest

import srs_io_ref as ref

pytestmark = pytest.mark.gpu

TAU = 0x7A05ED


def _pb():
    import plonk_prototype_b200 as pb
    return pb


def _device_image(ctx, srs):
    n = _pb()._native.lib().pb200_srs_len(srs)
    out = np.empty((n, 12), np.uint64)
    ctx.d2h(out, ctx.srs_dev_ptr(srs))
    return out


@pytest.mark.parametrize("log_n", [10, 16, 20])
def test_round_trip(ctx, oracle, log_n):
    """Generated key → to_compressed (every byte equal to the reference encoder's) → from_compressed (the device image again,
    96 bytes per point) → a commitment over the reloaded key equal to one over the generated key."""
    pb = _pb()
    n = 1 << log_n
    srs = ctx.srs_generate(pb.scalars_to_mont([TAU]), n)
    srs2 = None
    try:
        img = _device_image(ctx, srs)
        enc = ctx.srs_to_compressed(srs)
        assert len(enc) == 48 * n and enc == ref.g1_to_bytes(img, threads=16)
        assert ctx.srs_to_compressed(srs, 5, 3) == enc[48 * 5:48 * 8]
        launches = ctx.launch_count()
        status = np.full(n, 0xFF, np.uint8)
        srs2 = ctx.srs_from_compressed(enc, status_out=status)
        assert ctx.launch_count() == launches + 1 and (status == 0).all()
        assert (_device_image(ctx, srs2) == img).all()
        coeffs = oracle.fr_to_mont(oracle.random_fr(0x5E + log_n, min(n, 1 << 16)))
        assert pb.g1_to_bytes(ctx.msm(srs2, coeffs)) == pb.g1_to_bytes(ctx.msm(srs, coeffs))
    finally:
        ctx.srs_free(srs)
        if srs2 is not None:
            ctx.srs_free(srs2)


def test_corpus_status_matches_reference(ctx, oracle):
    """Every valid point and every kind of invalid one (tests/srs_io_ref.corpus): per-point status equal to the reference's;
    the call fails, naming the first invalid index."""
    data, labels = ref.corpus()
    rst, _ = ref.g1_from_bytes_checked(data, threads=8)
    assert list(rst) == labels
    status = np.full(len(labels), 0xFF, np.uint8)
    with pytest.raises(ValueError, match="point %d of %d" % (labels.index(ref.BAD_FLAGS), len(labels))):
        ctx.srs_from_compressed(data, status_out=status)
    assert list(status) == labels
    ok = [i for i, s in enumerate(labels) if s == ref.OK]     # the valid part alone loads, with the reference's limbs
    sub = b"".join(data[48 * i:48 * i + 48] for i in ok)
    srs = ctx.srs_from_compressed(sub)
    try:
        _, rxy = ref.g1_from_bytes_checked(sub)
        assert (_device_image(ctx, srs) == rxy).all()
    finally:
        ctx.srs_free(srs)


@pytest.mark.parametrize("kind", ["not_in_subgroup", "not_on_curve", "bad_flags"])
def test_one_bad_point_in_a_large_key(ctx, oracle, kind):
    """One invalid point at a chosen index among 2^20 valid ones: PB200_ERR_ARG, a message naming the index and the reason, no
    SRS returned — and the context still works (one more MSM)."""
    import model
    pb = _pb()
    n, bad = 1 << 20, 777_777
    srs = ctx.srs_generate(pb.scalars_to_mont([TAU]), n)
    try:
        enc = bytearray(ctx.srs_to_compressed(srs))
        if kind == "not_in_subgroup":
            rec, reason = model.g1_compress(model.g1_add(model.G1_GEN, (0, 2))), "prime-order subgroup"
        elif kind == "not_on_curve":
            rec, reason = ref._enc_x(1, 0x80), "not on the curve"
        else:
            rec, reason = bytes([enc[48 * bad] & 0x7F]) + bytes(enc[48 * bad + 1:48 * bad + 48]), "flag"
        enc[48 * bad:48 * bad + 48] = rec
        status = np.zeros(n, np.uint8)
        with pytest.raises(ValueError) as ei:
            ctx.srs_from_compressed(bytes(enc), status_out=status)
        assert ("point %d of %d" % (bad, n)) in str(ei.value) and reason in str(ei.value)
        assert np.count_nonzero(status) == 1 and status[bad] != 0
        coeffs = oracle.fr_to_mont(oracle.random_fr(0xBAD, 1 << 12))
        got = ctx.msm(srs, coeffs)
        want = oracle.msm_variable_base(_device_image(ctx, srs)[:1 << 12], coeffs, threads=8)
        assert oracle.g1_proj_to_affine_canonical(got) == oracle.g1_proj_to_affine_canonical(want)
    finally:
        ctx.srs_free(srs)


def test_public_parameters_var_bytes_prove(ctx):
    """PublicParameters.to_var_bytes → from_slice, then preprocess, prove and verify a small circuit: the proof and the
    verifier key equal those made with the original parameters, and the reloaded opening key verifies it."""
    pb = _pb()
    from plonk_prototype_b200.synth import synthetic_circuit_columns
    sel, wires, values, pi_pos, pi_vals = synthetic_circuit_columns(1000)
    pp = pb.PublicParameters(1023, 0x5EED, ctx)
    pp2 = None
    try:
        data = pp.to_var_bytes()
        assert len(data) == 240 + 48 * 1024
        pp2 = pb.PublicParameters.from_slice(data, ctx)
        assert pp2.n_points == 1024 and (pp2.beta_h == pp.beta_h).all()
        proofs = []
        for p in (pp, pp2):
            pk, vk = ctx.preprocess(p.srs, sel, wires, values.shape[0], b"srs io")
            try:
                proofs.append((ctx.prove(p.srs, pk, values, pi_pos, pi_vals), vk, ctx.prover_key_size(pk)))
            finally:
                ctx.prover_key_free(pk)
        assert proofs[0] == proofs[1]
        proof, vk, n = proofs[1]
        assert pb._native.verify(vk, n, b"srs io", proof, pi_pos, pi_vals, pp2.beta_h)
        with pytest.raises(ValueError):                       # a truncated commit key
            pb.PublicParameters.from_slice(data[:-1], ctx)
    finally:
        pp.close()
        if pp2 is not None:
            pp2.close()


def test_public_parameters_from_slice_rejects_bad_opening_key(ctx):
    """A tampered β·H — on the twist but outside the order-r subgroup — is rejected by from_slice, before the commit key is
    loaded."""
    pb = _pb()
    pp = pb.PublicParameters(63, 0x5EED, ctx, precompute=False)
    try:
        data = pp.to_var_bytes()
        bad = data[:144] + ref.g2_off_subgroup_bytes() + data[240:]
        with pytest.raises(ValueError, match="subgroup"):
            pb.PublicParameters.from_slice(bad, ctx)
    finally:
        pp.close()
