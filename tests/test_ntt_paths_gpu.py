"""Every code path of `ntt_run` (csrc/ntt.cu) against an exact reference.

`ntt_run` picks the kernel and the plan of a transform from its size, from environment switches and from how much of the
context's 16 GiB twiddle-table budget earlier plans have used:
  * 2^12 … 2^26 by default: `ntt_pass_tma_kernel` with single-lookup tables (two passes up to 2^18, three above, S ∈ 6…9);
  * 2^27: the same plan shape on `ntt_pass_kernel` with two-level tables (single-lookup tables stop at 2^26);
  * 2^28 and up, and PB200_NTT_PLAN=legacy: the legacy plan (tiles ≤ 2^11) on `ntt_pass_kernel`;
  * PB200_NTT_FULL_TABLE_MAX_LOG=0, or a plan built after the budget ran out: `ntt_pass_kernel` with two-level tables
    (store_mode 2/3, load_mode 1), possibly mixed with single-lookup tables for the parts that still fit;
  * PB200_NTT_TMA_REGS=168 / PB200_NTT_KERNEL=legacy (read once per process): the 384-thread TMA build / `ntt_pass_kernel`
    on the default plans.  These run in child processes started from this file (`python test_ntt_paths_gpu.py MODE`).

References: the C oracle for whole vectors, and two closed forms that cost nothing at any size — `sparse_reference` (a
handful of nonzero inputs, any chosen outputs) and `constant_reference` (every input equal).  All comparisons are
bit-exact.  Inputs are raw limbs below r used as Montgomery representations; every variant is linear, so the raw limbs
of the output are the transform of the raw limbs of the input and the references work on plain integers.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if __name__ == "__main__":  # child process: the import paths conftest.py sets up for the suite
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))

import model  # noqa: E402

gpu = pytest.mark.gpu
VARIANTS = (("fft", 0, 0), ("ifft", 1, 0), ("coset_fft", 0, 1), ("coset_ifft", 1, 1))
THREADS = os.cpu_count() or 8
R_MINUS_1 = np.array(model.to_limbs(model.R - 1, 4), np.uint64)


# ----------------------------------------------------------------------------- references on plain integers
def sparse_reference(log_n, terms, inverse, coset, indices):
    """Outputs at `indices` of the transform of x with x[j] = v for (j, v) in `terms` and 0 elsewhere (g = 7, ω = ω_n):
    fft Σ v ω^{ij} | ifft n⁻¹ Σ v ω^{−ij} | coset_fft Σ v g^j ω^{ij} | coset_ifft n⁻¹ g^{−i} Σ v ω^{−ij}."""
    n = 1 << log_n
    d = model.domain(n)
    w = d["group_gen_inv"] if inverse else d["group_gen"]
    out = []
    for i in indices:
        acc = 0
        for j, v in terms:
            t = v * pow(w, (i * j) % n, model.R)
            if coset and not inverse:
                t = t * pow(model.GENERATOR, j, model.R)
            acc += t
        if inverse:
            acc = acc * d["size_inv"]
            if coset:
                acc = acc * pow(d["generator_inv"], i, model.R)
        out.append(acc % model.R)
    return out


def constant_reference(log_n, c, inverse, coset, indices):
    """Outputs at `indices` of the transform of the constant vector x[j] = c: Σ_j ω^{ij} = n·[i = 0], so fft gives c·n at 0,
    ifft and coset_ifft give c at 0, all three 0 elsewhere; coset_fft gives c·(g^n − 1)/(g·ω^i − 1) everywhere."""
    n = 1 << log_n
    if coset and not inverse:
        w = model.domain(n)["group_gen"]
        gn1 = pow(model.GENERATOR, n, model.R) - 1
        return [c * gn1 * pow(model.GENERATOR * pow(w, i, model.R) - 1, -1, model.R) % model.R for i in indices]
    at0 = c if inverse else c * n % model.R
    return [at0 if i == 0 else 0 for i in indices]


def sparse_terms(log_n, seed, k=6):
    """k distinct positions (0, 1, n − 1, n/2 + 3 and pseudo-random ones) with random values, one of them r − 1."""
    n = 1 << log_n
    pos = []
    g = model.splitmix64_stream(seed)
    for j in [0, 1, n - 1, n // 2 + 3] + [next(g) % n for _ in range(4 * k)]:
        if j < n and j not in pos:
            pos.append(j)
    pos = pos[:k]
    vals = model.random_fr(seed, len(pos))
    vals[-1] = model.R - 1
    return list(zip(pos, vals))


def sample_indices(log_n, count=64):
    n = 1 << log_n
    idx = [0, 1, 2, 3, n // 3, n // 2 - 1, n // 2, n // 2 + 1, n - 2, n - 1]
    g = model.splitmix64_stream(0x1D5 + log_n)
    while len(idx) < count:
        idx.append(next(g) % n)
    return sorted(set(i for i in idx if 0 <= i < n))


def near_r(log_n, seed):
    """Values r − 1 − e with e < 2^16 (r − 1 ends in 32 zero bits: no borrow out of the low limb)."""
    n = 1 << log_n
    x = np.repeat(R_MINUS_1.reshape(1, 4), n, axis=0)
    e = np.frombuffer(np.random.default_rng(seed).bytes(2 * n), dtype=np.uint16).astype(np.uint64)
    x[:, 0] -= e
    return x


def all_r_minus_1(log_n):
    return np.repeat(R_MINUS_1.reshape(1, 4), 1 << log_n, axis=0)


def test_sparse_and_constant_references_match_oracle(oracle):
    """The closed forms against the C oracle, every output index, all four variants, 2^1 … 2^14."""
    for log_n in range(1, 15):
        n = 1 << log_n
        terms = sparse_terms(log_n, 0x5BA + log_n)
        x = np.zeros((n, 4), np.uint64)
        for j, v in terms:
            x[j] = model.to_limbs(v, 4)
        c = model.R - 1 - 12345
        xc = np.repeat(np.array(model.to_limbs(c, 4), np.uint64).reshape(1, 4), n, axis=0)
        for name, inv, cos in VARIANTS:
            want = sparse_reference(log_n, terms, inv, cos, range(n))
            got = oracle.ntt(x, inv, cos, threads=4)
            assert [model.from_limbs(r) for r in got] == want, (log_n, name, "sparse")
            want = constant_reference(log_n, c, inv, cos, range(n))
            got = oracle.ntt(xc, inv, cos, threads=4)
            assert [model.from_limbs(r) for r in got] == want, (log_n, name, "constant")


# ----------------------------------------------------------------------------- device helpers
_ZERO_CHUNK = None


def dev_zero(ctx, d, n):
    """Zero n scalars at device address d (uploads of one 64 MiB zero block)."""
    global _ZERO_CHUNK
    if _ZERO_CHUNK is None:
        _ZERO_CHUNK = np.zeros((1 << 21, 4), np.uint64)
    step = _ZERO_CHUNK.shape[0]
    for off in range(0, n, step):
        ctx.h2d(d + 32 * off, _ZERO_CHUNK[:min(step, n - off)])


def dev_put(ctx, d, j, v):
    ctx.h2d(d + 32 * j, np.array(model.to_limbs(v, 4), np.uint64))


def dev_get(ctx, d, indices):
    buf = np.empty(4, np.uint64)
    out = []
    for i in indices:
        ctx.d2h(buf, d + 32 * i)
        out.append(model.from_limbs(buf))
    return out


def run_dev(ctx, x, log_n, inverse, coset, batch=1):
    d = ctx.malloc(x.nbytes)
    try:
        ctx.h2d(d, x)
        if batch == 1:
            ctx.ntt_dev(d, log_n, inverse, coset)
        else:
            ctx.ntt_batch_dev(d, log_n, batch, inverse, coset)
        got = np.empty_like(x)
        ctx.d2h(got, d)
    finally:
        ctx.free(d)
    return got


def assert_same(got, want, what):
    bad = np.flatnonzero((got != want).any(axis=1))
    assert bad.size == 0, "%s: %d wrong outputs, first bad index %d" % (what, bad.size, bad[0])


def assert_sparse_and_constant(ctx, d, log_n, name, inverse, coset, seed):
    """One device buffer of 2^log_n scalars: the sparse input and the all-(r − 1) input, checked at ~64 outputs."""
    n = 1 << log_n
    idx = sample_indices(log_n)
    terms = sparse_terms(log_n, seed)
    dev_zero(ctx, d, n)
    for j, v in terms:
        dev_put(ctx, d, j, v)
    ctx.ntt_dev(d, log_n, inverse, coset)
    got, want = dev_get(ctx, d, idx), sparse_reference(log_n, terms, inverse, coset, idx)
    bad = [i for i, a, b in zip(idx, got, want) if a != b]
    assert not bad, "L=%d %s sparse: first bad index %d" % (log_n, name, bad[0])
    dev_fill_r_minus_1(ctx, d, n)
    ctx.ntt_dev(d, log_n, inverse, coset)
    got, want = dev_get(ctx, d, idx), constant_reference(log_n, model.R - 1, inverse, coset, idx)
    bad = [i for i, a, b in zip(idx, got, want) if a != b]
    assert not bad, "L=%d %s all r-1: first bad index %d" % (log_n, name, bad[0])


def dev_fill_r_minus_1(ctx, d, n):
    block = all_r_minus_1(21)
    for off in range(0, n, block.shape[0]):
        ctx.h2d(d + 32 * off, block[:min(block.shape[0], n - off)])


@pytest.fixture
def fresh_ctx():
    """A context of its own: an empty plan cache, so the whole 16 GiB table budget is available and the plan is the
    default one whatever ran before."""
    import plonk_prototype_b200 as pb
    c = pb.Context(0)
    yield c
    c.close()


# ----------------------------------------------------------------------------- default path
@gpu
@pytest.mark.parametrize("log_n,variants", [(19, (0, 1, 2, 3)), (21, (0, 1, 2, 3)), (22, (1, 2)), (23, (1, 2)), (25, (0, 3))],
                         ids=["19-all", "21-all", "22-ifft+coset_fft", "23-ifft+coset_fft", "25-fft+coset_ifft"])
def test_default_geometries_full_vector(fresh_ctx, oracle, log_n, variants):
    """Three-pass TMA plans S = (7,6,6) at 2^19 (the only plan with S = 6 in the middle pass), (7,7,7) at 2^21, (8,7,7) /
    (8,8,7) at 2^22 / 2^23, (9,8,8) at 2^25: every output against the oracle."""
    x = oracle.random_fr(0xDA7A0000 + log_n, 1 << log_n)
    for v in variants:
        name, inv, cos = VARIANTS[v]
        assert_same(run_dev(fresh_ctx, x, log_n, inv, cos), oracle.ntt(x, inv, cos, threads=THREADS), (log_n, name))


@gpu
@pytest.mark.parametrize("log_n", [12, 13, 15, 17, 18, 19, 21])
def test_edge_vectors_every_geometry(fresh_ctx, oracle, log_n):
    """All-(r − 1) and values just below r: the largest values the lazy [0, 2r) range between TMA passes has to carry."""
    for kind, x in (("all_r_minus_1", all_r_minus_1(log_n)), ("near_r", near_r(log_n, 0xED6E + log_n))):
        for name, inv, cos in VARIANTS:
            assert_same(run_dev(fresh_ctx, x, log_n, inv, cos), oracle.ntt(x, inv, cos, threads=THREADS), (log_n, kind, name))


@gpu
@pytest.mark.parametrize("log_n", [24, 25, 26, 27, 28])
def test_sparse_and_constant_inputs_large(fresh_ctx, log_n):
    """All four variants at ~64 outputs on a sparse input and on the all-(r − 1) input; 2^27 and 2^28 run ntt_pass_kernel
    (two-level tables, legacy plan at 2^28)."""
    d = fresh_ctx.malloc(32 << log_n)
    try:
        for name, inv, cos in VARIANTS:
            assert_sparse_and_constant(fresh_ctx, d, log_n, name, inv, cos, 0x5BA0 + log_n)
    finally:
        fresh_ctx.free(d)


@gpu
def test_2e27_full_vector(fresh_ctx, oracle):
    """2^27 (4 GiB): fft and coset_ifft, every output against the oracle."""
    log_n = 27
    x = oracle.random_fr(0xDA7A0000 + log_n, 1 << log_n)
    for name, inv, cos in (VARIANTS[0], VARIANTS[3]):
        got = run_dev(fresh_ctx, x, log_n, inv, cos)
        want = oracle.ntt(x, inv, cos, threads=THREADS)
        assert_same(got, want, (log_n, name))
        del got, want


@gpu
def test_2e28_round_trip(fresh_ctx, oracle):
    """2^28 (8 GiB, 8 GiB of scratch): fft → ifft → coset_fft → coset_ifft returns the random input exactly."""
    log_n, chunk = 28, 1 << 22
    n = 1 << log_n
    d = fresh_ctx.malloc(32 * n)
    try:
        for k in range(n // chunk):
            fresh_ctx.h2d(d + 32 * k * chunk, oracle.random_fr(0x28000 + k, chunk))
        for name, inv, cos in VARIANTS:
            fresh_ctx.ntt_dev(d, log_n, inv, cos)
        got = np.empty((chunk, 4), np.uint64)
        for k in range(n // chunk):
            fresh_ctx.d2h(got, d + 32 * k * chunk)
            assert_same(got, oracle.random_fr(0x28000 + k, chunk), ("round trip 2^28, chunk", k))
    finally:
        fresh_ctx.free(d)


@gpu
@pytest.mark.parametrize("log_n,batch,variants", [(19, 3, (0, 1, 2, 3)), (20, 3, (0, 1, 2, 3)), (22, 4, (2,))],
                         ids=["19x3-all", "20x3-all", "22x4-coset_fft"])
def test_batched_against_oracle(fresh_ctx, oracle, log_n, batch, variants):
    """Batched transforms at three-pass sizes (the prover's coset extension and its batch-of-4 inverse transforms),
    vector by vector against the oracle."""
    n = 1 << log_n
    x = oracle.random_fr(0xBA7C0000 + log_n, n * batch)
    x[n:2 * n] = near_r(log_n, log_n)        # a vector of large values rides along
    for v in variants:
        name, inv, cos = VARIANTS[v]
        got = run_dev(fresh_ctx, x, log_n, inv, cos, batch)
        for b in range(batch):
            assert_same(got[b * n:(b + 1) * n], oracle.ntt(x[b * n:(b + 1) * n], inv, cos, threads=THREADS), (log_n, name, b))


@gpu
def test_batched_2e26_coset_fft_matches_single(fresh_ctx, oracle):
    log_n, batch = 26, 2
    n = 1 << log_n
    x = oracle.random_fr(0xBA7C0000 + log_n, n * batch)
    got = run_dev(fresh_ctx, x, log_n, 0, 1, batch)
    for b in range(batch):
        assert_same(got[b * n:(b + 1) * n], run_dev(fresh_ctx, np.ascontiguousarray(x[b * n:(b + 1) * n]), log_n, 0, 1), b)


# ----------------------------------------------------------------------------- per-plan switches
PLAN_SWITCHES = (("PB200_NTT_FULL_TABLE_MAX_LOG", "0"), ("PB200_NTT_PLAN", "legacy"))


@gpu
@pytest.mark.parametrize("log_n,batch", [(12, 1), (13, 1), (18, 1), (19, 1), (22, 1), (23, 1), (25, 1), (13, 3)])
def test_plan_switches(oracle, monkeypatch, log_n, batch):
    """PB200_NTT_FULL_TABLE_MAX_LOG=0 (TMA-shaped plans with two-level tables on ntt_pass_kernel) and PB200_NTT_PLAN=legacy
    (the legacy 2- and 3-pass shapes at testable sizes).  Both are read when a plan is built: one fresh context each."""
    import plonk_prototype_b200 as pb
    n = 1 << log_n
    x = oracle.random_fr(0x5A170000 + log_n, n * batch)
    if batch > 1:
        x[n:2 * n] = near_r(log_n, log_n)
    ctxs = {}
    try:
        for var, val in PLAN_SWITCHES:
            ctxs[var] = pb.Context(0)
        for name, inv, cos in VARIANTS:
            want = np.concatenate([oracle.ntt(x[b * n:(b + 1) * n], inv, cos, threads=THREADS) for b in range(batch)])
            for var, val in PLAN_SWITCHES:
                monkeypatch.setenv(var, val)
                got = run_dev(ctxs[var], x, log_n, inv, cos, batch)
                monkeypatch.delenv(var)
                assert_same(got, want, (var, val, log_n, name))
    finally:
        for c in ctxs.values():
            c.close()


# ----------------------------------------------------------------------------- table budget exhausted
def fill_table_budget(ctx, d):
    """Build plans until the context's 16 GiB table budget is nearly used, on the 2 GiB buffer d (contents irrelevant).
    Tables per plan: 32·n for pass 0, 32·n/2^S0 for pass 1, 32·n for a coset factor.  2^26 fft, ifft, coset_ifft:
    2052 + 2052 + 4100 MiB; 2^25: 1026 + 1026 + 2050 MiB; 12306 MiB in all, 4078 MiB left."""
    for log_n in (26, 25):
        for inv, cos in ((0, 0), (1, 0), (1, 1)):
            ctx.ntt_dev(d, log_n, inv, cos)
    ctx.sync()


# After fill_table_budget, in this order (the plans that follow and what of them still fits):
#   2^26 coset_fft:  pass-0 table (2048 MiB) fits, coset table (2048) does not → load_mode 1 next to store_mode 4 (2026 left);
#   2^24 fft, ifft:  514 MiB each (998 left);
#   2^24 coset_ifft: pass-0 and pass-1 tables fit, the coset table (512) does not → last pass store_mode 3 (484 left);
#   2^24 coset_fft:  pass-0 (512) and coset tables do not fit, pass 1 (2) does → store_mode 2 and load_mode 1.
BUDGET_STEPS = ((26, 0, 1, True), (24, 0, 0, False), (24, 1, 0, False), (24, 1, 1, True), (24, 0, 1, True))


@gpu
def test_table_budget_fallback(fresh_ctx, oracle):
    """Plans built after the table budget ran out (the mixed cases included) against the oracle at full length."""
    ctx = fresh_ctx
    d = ctx.malloc(32 << 26)
    try:
        dev_zero(ctx, d, 1 << 26)
        fill_table_budget(ctx, d)
        for log_n, inv, cos, check in BUDGET_STEPS:
            x = oracle.random_fr(0xB0D6E700 + 4 * log_n + 2 * inv + cos, 1 << log_n)
            ctx.h2d(d, x)
            ctx.ntt_dev(d, log_n, inv, cos)
            if check:
                got = np.empty_like(x)
                ctx.d2h(got, d)
                assert_same(got, oracle.ntt(x, inv, cos, threads=THREADS), ("budget", log_n, inv, cos))
    finally:
        ctx.free(d)


# ----------------------------------------------------------------------------- switches read once per process
CHILD_TIMEOUT_S = 1800


def run_child(mode, env_extra, done_marker):
    env = dict(os.environ)
    for k in list(env):
        if k.startswith("PB200_"):
            del env[k]
    env.update(env_extra)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), mode], env=env, timeout=CHILD_TIMEOUT_S, cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, "child %s %s failed (%d):\n%s" % (mode, env_extra, r.returncode, r.stdout[-6000:])
    assert done_marker in r.stdout, r.stdout[-3000:]


@gpu
@pytest.mark.parametrize("var,val,mode", [("PB200_NTT_TMA_REGS", "168", "ntt"), ("PB200_NTT_KERNEL", "legacy", "ntt"),
                                          ("PB200_MSM_ACC_CTAS", "3", "msm")])
def test_process_switches(var, val, mode):
    """Switches read once per process (`static` in ntt_launch_tma, ntt_run and the MSM accumulate launch): the default
    path's checks in a child process started with the switch set."""
    run_child(mode, {var: val}, "L=%d ok" % CHILD_NTT_LOGS[-1] if mode == "ntt" else "msm ok")


@gpu
@pytest.mark.parametrize("config", ["default", "tma_regs_168", "kernel_legacy"])
def test_kernel_that_ran(config):
    """torch.profiler's kernel names show which NTT kernel each configuration above actually executes."""
    env = {"default": {}, "tma_regs_168": {"PB200_NTT_TMA_REGS": "168"}, "kernel_legacy": {"PB200_NTT_KERNEL": "legacy"}}[config]
    run_child("kernels-" + config, env, "kernels ok")


# ----------------------------------------------------------------------------- child processes
CHILD_NTT_LOGS = (12, 13, 15, 17, 18, 19, 21, 24, 26)


def child_ntt(pyoracle, pb):
    """The default path's geometries: S = 6…9 in both pass types, load / store modes 2, 4, 5, and a batch."""
    for log_n in CHILD_NTT_LOGS:
        n = 1 << log_n
        x = pyoracle.random_fr(0xC41D0000 + log_n, n)
        full = (0, 1, 2, 3) if log_n <= 24 else (2,)        # 2^26: the coset_fft plan (S = 9 in both strided passes) in full
        wants = {v: pyoracle.ntt(x, VARIANTS[v][1], VARIANTS[v][2], threads=THREADS) for v in full}
        ctx = pb.Context(0)                                  # (the first device call: everything above runs on the CPU)
        try:
            for v in full:
                name, inv, cos = VARIANTS[v]
                got = run_dev(ctx, x, log_n, inv, cos)
                bad = np.flatnonzero((got != wants[v]).any(axis=1))
                if bad.size:
                    sys.exit("FAIL L=%d %s first bad index %d" % (log_n, name, bad[0]))
            if log_n >= 24:
                d = ctx.malloc(32 << log_n)
                try:
                    for name, inv, cos in VARIANTS:
                        assert_sparse_and_constant(ctx, d, log_n, name, inv, cos, 0xC41D + log_n)
                finally:
                    ctx.free(d)
            if log_n == 19:
                xb = pyoracle.random_fr(0xC41DBA7C, 3 * n)
                for name, inv, cos in VARIANTS:
                    got = run_dev(ctx, xb, log_n, inv, cos, 3)
                    for b in range(3):
                        want = pyoracle.ntt(xb[b * n:(b + 1) * n], inv, cos, threads=THREADS)
                        bad = np.flatnonzero((got[b * n:(b + 1) * n] != want).any(axis=1))
                        if bad.size:
                            sys.exit("FAIL L=%d batch %d %s first bad index %d" % (log_n, b, name, bad[0]))
        finally:
            ctx.close()
        print("L=%d ok" % log_n, flush=True)


def child_msm(pyoracle, pb):
    import test_msm_gpu as T
    ctx = pb.Context(0)
    try:
        T.test_random_matches_oracle(ctx, pyoracle, 1 << 16)
        T.test_adversarial_scalar_sets(ctx, pyoracle)
        for n in (300, 4096, 1 << 15):
            T.test_precomputed_srs_gives_identical_results(ctx, pyoracle, n)
    finally:
        ctx.close()
    print("msm ok", flush=True)


def _classify(names):
    """{'plain'} / {('tma', S, threads_per_sm)} for the NTT pass kernels among the profiled kernel names."""
    kinds = set()
    for s in names:
        m = re.search(r"ntt_pass_tma_kernel(?:<(\d+), ?(\d+)>|ILi(\d+)ELi(\d+)E)", s)
        if m:
            g = [int(t) for t in m.groups() if t is not None]
            kinds.add(("tma", g[0], g[1]))
        elif "ntt_pass_kernel" in s:
            kinds.add("plain")
    return kinds


def _ran(ctx, fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        ctx.sync()
    return _classify(e.name for e in prof.events())


def tma_pass_sizes(log_n):
    """S of every pass of the default plan (ntt_build_plan): two passes up to 2^18, three above."""
    if log_n <= 18:
        return [(log_n + 1) // 2, log_n // 2]
    s0 = (log_n + 2) // 3
    s1 = (log_n - s0 + 1) // 2
    return [s0, s1, log_n - s0 - s1]


def child_kernels(config, pb):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]):
        pass                                                 # CUPTI is up before the library creates its context
    tma_threads = 384 if config == "tma_regs_168" else 512

    def expect(kinds, want, what):
        if kinds != want:
            sys.exit("FAIL %s: ran %s, expected %s" % (what, sorted(map(str, kinds)), sorted(map(str, want))))

    for log_n in range(12, 29):                              # a context per size: every plan gets its tables
        ctx = pb.Context(0)
        d = ctx.malloc(32 << log_n)
        try:
            dev_zero(ctx, d, 1 << log_n)
            for name, inv, cos in VARIANTS:
                if log_n >= 27 or config == "kernel_legacy":
                    want = {"plain"}
                else:
                    want = {("tma", s, tma_threads) for s in tma_pass_sizes(log_n)}
                expect(_ran(ctx, lambda: ctx.ntt_dev(d, log_n, inv, cos)), want, "L=%d %s" % (log_n, name))
        finally:
            ctx.free(d)
            ctx.close()
    if config != "default":
        print("kernels ok", flush=True)
        return
    for var, val in PLAN_SWITCHES:
        os.environ[var] = val
        ctx = pb.Context(0)
        d = ctx.malloc(32 << 19)
        try:
            for log_n in (13, 19):
                for name, inv, cos in VARIANTS:
                    expect(_ran(ctx, lambda: ctx.ntt_dev(d, log_n, inv, cos)), {"plain"}, "%s=%s L=%d %s" % (var, val, log_n, name))
        finally:
            ctx.free(d)
            ctx.close()
            del os.environ[var]
    ctx = pb.Context(0)
    d = ctx.malloc(32 << 26)
    try:
        dev_zero(ctx, d, 1 << 26)
        fill_table_budget(ctx, d)
        for log_n, inv, cos, fallback in BUDGET_STEPS:
            want = {"plain"} if fallback else {("tma", s, 512) for s in tma_pass_sizes(log_n)}
            expect(_ran(ctx, lambda: ctx.ntt_dev(d, log_n, inv, cos)), want, "budget step L=%d inverse=%d coset=%d" % (log_n, inv, cos))
    finally:
        ctx.free(d)
        ctx.close()
    print("kernels ok", flush=True)


def child_main(argv):
    modes = ("ntt", "msm", "kernels-default", "kernels-tma_regs_168", "kernels-kernel_legacy")
    if len(argv) != 1 or argv[0] not in modes:
        sys.exit("usage: %s {%s}" % (os.path.basename(__file__), "|".join(modes)))
    import pyoracle
    pyoracle.build()
    import plonk_prototype_b200 as pb
    if argv[0] == "ntt":
        child_ntt(pyoracle, pb)
    elif argv[0] == "msm":
        child_msm(pyoracle, pb)
    else:
        child_kernels(argv[0][len("kernels-"):], pb)


if __name__ == "__main__":
    child_main(sys.argv[1:])
