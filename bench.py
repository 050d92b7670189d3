#!/usr/bin/env python
"""bench.py — headline measurement of the PLONK-prover hot path (DESIGN.md §6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--log-gates L] [--dump-outputs DIR]

--steps K is the number of timed steps of the headline and of the MSM, NTT and large-prove context objects.
--dump-outputs DIR writes the proof of the last timed step to DIR/proof.npy; the inputs are seeded, so two builds run
with the same arguments can be compared output for output.

Headline (BASELINE.json `metric`, first item; configs[3]): **PLONK prove time at 2^20 gates** — one step = one proof
of the synthetic arithmetic circuit (mul / add chain, boolean padding, 2 public inputs; SURVEY.md §8d): 11 G1 MSMs of
2^20 points, 10 NTTs of 2^20, 8 coset NTTs of 2^22 and the pointwise kernels, witness in → 1040-byte proof out.
    value  = ms per proof with the witness already resident in HBM (pb200_prove_dev; CUDA events on the library's stream)
    e2e    = ms per proof through pb200_prove with the witness in pinned HOST memory (H2D + proof D2H inside the timing)
Both arms (`--impl ours`, `--impl reference`) run the SAME circuit at the SAME size, so the driver's ratio is a
same-config number: the reference arm is the C restatement of the upstream prover (oracle/, all host cores — the Rust
reference cannot be built here, SURVEY.md §0.3).  In our arm the CPU prove is run once on the GPU's own SRS and its
proof bytes are compared with the GPU proof (`parity.byte_identical_with_cpu_port`), and the pairing verifier must
accept it.
The same JSON line carries, as context objects: `roofline` (msm_accumulate_kernel inside the timed proves against the
live IMAD.WIDE peak), `msm` (standalone 2^26-point G1 MSM, BASELINE.json configs[1]: throughput, e2e, integer roofline,
closed-form check), `ntt` (2^24 forward NTT, configs[2]: Melem/s, HBM and integer fractions), `prove_2e24` (the
2^24-gate circuit of configs[4] on one GPU) and `cpu_baseline`.

N > 1 (torchrun; STRONG scaling — the problem sizes are BASELINE.json's, split over the ranks): the headline is the
same 2^20-gate proof with every commitment sharded by point range and round 3 as sharded four-step transforms; the
line adds `msm` (ONE 2^26-point MSM split over N), `ntt_sharded` (one 2^26-point NTT over N) and `prove_sharded_2e24`
(configs[4]) with in-run equality against the single-GPU proof.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the checkout may be read-only: leave no __pycache__ in it

R_MOD = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
FR_MONT_R = (1 << 256) % R_MOD
A0, D0 = 0xB2000001, 0x9E3779B1
LABEL = b"pb200-bench"
N_PUB = 2
DTYPE = "u32 limbs (Fr 8x32, Fp 12x32)"


# ------------------------------------------------------------------------------------------ inputs
def splitmix64_block(seed, start, count):
    """Outputs start … start+count−1 of SplitMix64(seed) — the state is a counter, so this vectorises."""
    with np.errstate(over="ignore"):
        k = np.arange(start + 1, start + count + 1, dtype=np.uint64)
        z = np.uint64(seed) + k * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def random_fr_limbs(seed, n, out=None):
    """n values uniform in [0, r) as (n, 4) uint64 limbs; identical stream to oracle/model random_fr."""
    r_limbs = [(R_MOD >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(4)]
    res = out if out is not None else np.empty((n, 4), np.uint64)
    filled, cand = 0, 0
    chunk = 1 << 22
    while filled < n:
        raw = splitmix64_block(seed, 4 * cand, 4 * chunk).reshape(chunk, 4)
        cand += chunk
        raw[:, 3] &= np.uint64(0x7FFFFFFFFFFFFFFF)
        lt = np.zeros(chunk, bool)
        eq = np.ones(chunk, bool)
        for i in (3, 2, 1, 0):
            lt |= eq & (raw[:, i] < np.uint64(r_limbs[i]))
            eq &= raw[:, i] == np.uint64(r_limbs[i])
        ok = raw[lt]
        take = min(n - filled, ok.shape[0])
        res[filled:filled + take] = ok[:take]
        filled += take
    return res


def closed_form_scalar(scalars_mont, a, d):
    """k with Σ sᵢ·Pᵢ = k·G for Pᵢ = (a + i·d)·G (exact; 16-bit partial dot products)."""
    s = np.ascontiguousarray(scalars_mont, dtype=np.uint64).reshape(-1, 4)
    n = s.shape[0]
    k = np.uint64(a) + np.arange(n, dtype=np.uint64) * np.uint64(d)
    s16 = s.view(np.uint16).reshape(n, 16)
    k16 = k.view(np.uint16).reshape(n, 4).astype(np.uint64)
    total = 0
    for i in range(16):
        col = s16[:, i].astype(np.uint64)
        for j in range(4):
            total += int(np.dot(col, k16[:, j])) << (16 * (i + j))
    return total * pow(FR_MONT_R, -1, R_MOD) % R_MOD


MSM_CHUNKS = 8  # the global scalar vector of the MSM bench is 8 seeded chunks, so any rank count ≤ 8 splits the SAME problem


def msm_scalar_slice(log_total, rank, world, out):
    """This rank's contiguous slice of the global 2^log_total scalar vector (chunk c has its own SplitMix64 seed)."""
    per_chunk = (1 << log_total) // MSM_CHUNKS
    chunks = MSM_CHUNKS // world
    for k in range(chunks):
        c = rank * chunks + k
        random_fr_limbs(0xB2000000 + log_total + 1000 * c, per_chunk, out=out[k * per_chunk:(k + 1) * per_chunk])
    return out


def msm_shard_base(rank, n):
    """Point-range sharding (SURVEY.md §8e): rank r owns global indices [r·n, (r+1)·n) of the synthetic SRS, i.e. bases
    (a_r + i·d)·G with a_r = A0 + r·n·D0."""
    return A0 + rank * n * D0


def gather_partials(dist, local_u64x18, world, device):
    """All-gather of the ranks' 144-byte partial results (as int64) — the only collective on the MSM path."""
    import torch
    mine = torch.from_numpy(np.ascontiguousarray(local_u64x18).view(np.int64).copy()).to(device)
    bufs = [torch.zeros(18, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(bufs, mine)
    return torch.stack(bufs).cpu().numpy().view(np.uint64)


def oracle():
    """The CPU checker (oracle/): cpu_baseline legs, result verification and the reference arm only."""
    p = os.path.join(ROOT, "oracle")
    if p not in sys.path:
        sys.path.insert(0, p)
    import pyoracle
    return pyoracle


def headline_config(L, world):
    """Identical in both arms (same-config comparison)."""
    cfg = {"workload": "PLONK prove of the synthetic arithmetic circuit, 2^%d gates (BASELINE.json configs[3]): "
                       "11 KZG commitments (G1 MSM), wire / permutation / quotient NTTs, 1040-byte proof" % L,
           "log_gates": L, "public_inputs": N_PUB, "circuit": "x <- x*x + x + c chain of mul/add rows, boolean padding (SURVEY.md §8d)",
           "l2": "inputs larger than L2: prover key + workspace %.1f GiB, 126 MB L2" % (129.0 * 32 * (1 << L) / 2**30),
           "n_gpus": world}
    return cfg


def headline_metric(L):
    return "PLONK prove time (BLS12-381 / KZG10, synthetic arithmetic circuit, 2^%d gates)" % L


def dump_outputs(out_dir, proof):
    """The 1040 proof bytes (11 compressed G1 commitments, then 16 scalar evaluations) as float64, which holds every
    byte value exactly."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "proof.npy"), np.frombuffer(proof, dtype=np.uint8).astype(np.float64))


# ---------------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                                       "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons, pw = [], [], set(), []
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        loaded = [c for c, p in zip(sm, pw) if p > 0.5 * max(pw)] if pw else sm
        return {"sm_mhz": statistics.median(loaded) if loaded else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------- reference arm
def cpu_prove(log_gates, threads, reps=None, srs=None, circuit=None):
    """The C restatement of dusk-plonk 0.8's prover (oracle/plonk_oracle.inc: same NTT / MSM call list; window-parallel
    MSM and parallel FFT / quotient loop as the rayon build) on the synthetic circuit.  → (proof, vk, preprocess s, prove s | [s…]).
    Without `srs` the commit key is the synthetic family (a + i·d)·G — prover cost does not depend on which points it holds."""
    O = oracle()
    n = 1 << log_gates
    sel, wires, values, pi_pos, pi_vals = circuit if circuit is not None else O.synthetic_circuit_columns(n, n_pub=N_PUB)
    if srs is None:
        srs = O.synthetic_bases(n)
    return O.plonk_prove(sel, wires, values, pi_pos, pi_vals, srs, LABEL, threads=threads, reps=reps)


def run_reference(args, rank, world):
    """`--impl reference`: the CPU prover alone, on the same circuit and size as our arm, all host threads.  Never imports
    the product package (the circuit generator is the checker's own, oracle/plonk_oracle.inc)."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    L = args.log_gates
    budget = float(os.environ.get("PB200_REF_BUDGET_S", "780"))
    t_start = time.perf_counter()
    # calibrate on 2^16 gates (also the warm-up: pages in the library and the thread pool; CPU code has no other warm state).
    # Linear extrapolation is conservative: the per-gate cost of the CPU prover falls with the size (Pippenger windows grow).
    cal_log = min(L, 16)
    _, _, cal_pre, cal_prove = cpu_prove(cal_log, cores)
    for _ in range(max(args.warmup - 1, 0)):
        cpu_prove(min(L, 12), cores)
    scale = float(1 << (L - cal_log))
    sample_log = L
    while sample_log > 12 and (cal_pre + args.steps * cal_prove) * scale * 2.0 ** (sample_log - L) > budget - (time.perf_counter() - t_start):
        sample_log -= 1
    proof, _, t_pre, t_steps = cpu_prove(sample_log, cores, reps=args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, proof)
    ms = 1e3 * sum(t_steps) / len(t_steps)
    same = sample_log == L
    sample = ("each step = one full prove_with_preprocessed of the SAME 2^%d-gate circuit (C restatement of dusk-plonk 0.8, oracle/plonk_oracle.inc), "
              "%d threads; preprocess once (%.1f s, untimed); warm-up on a 2^%d-gate circuit of the same family" % (sample_log, cores, t_pre, cal_log))
    if not same:
        sample = ("BOUNDED SAMPLE: 2^%d gates instead of 2^%d (projected full-size run exceeds the %d s budget on %d cores); value is the "
                  "measured 2^%d time, NOT extrapolated — " % (sample_log, L, budget, cores, sample_log)) + sample
    line = {
        "impl": "reference", "metric": headline_metric(L), "value": ms, "unit": "ms", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64 limbs (CPU, mulx/adcx/adox)", "data": "synthetic", "config": headline_config(L, args.gpus),
        "same_config": same, "sample_log_gates": sample_log, "steps_ms": [round(1e3 * t, 1) for t in t_steps],
        "cpu_baseline": {"value": ms, "unit": "ms", "cores": cores, "kind": "port", "sample": sample, "preprocess_ms": 1e3 * t_pre},
        "e2e": {"value": ms, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "proof_sha256_16": __import__("hashlib").sha256(proof).hexdigest()[:16],
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------- our arm
class ProveSetup:
    """Circuit, commit key, preprocessed prover key, witness in pinned host memory and in HBM."""

    def __init__(self, ctx, L, torch, shard=None, dist=None, device=None, lib_collectives=True):
        import plonk_prototype_b200 as pb
        from plonk_prototype_b200.synth import synthetic_circuit_columns
        self.ctx, self.L, self.n = ctx, L, 1 << L
        self.tau = 0xB2000000 + L
        self.circuit = synthetic_circuit_columns(self.n, n_pub=N_PUB)
        sel, wires, values, self.pi_pos, self.pi_vals = self.circuit
        pinned = torch.empty(values.shape, dtype=torch.int64, pin_memory=True)
        pinned.numpy().view(np.uint64)[:] = values
        self._pinned = pinned
        self.values = pinned.numpy().view(np.uint64)
        t0 = time.perf_counter()
        if shard is None:
            self.pp = pb.PublicParameters(self.n - 1, self.tau, ctx)
            self.pk, self.vk = ctx.preprocess(self.pp.srs, sel, wires, values.shape[0], LABEL)
        else:
            rank, world = shard
            self.pp = pb.ShardedParameters(self.n, self.tau, rank, world, ctx)
            if lib_collectives:   # every collective is the library's own NCCL call on its stream (pb200_comm)
                self.pk, self.vk = ctx.preprocess_comm(self.pp.srs, sel, wires, values.shape[0], LABEL)
            else:                 # host-language callbacks (torch.distributed), as a Python host without pb200_comm would
                self.pk, self.vk = ctx.preprocess(self.pp.srs, sel, wires, values.shape[0], LABEL,
                                                  shard=(rank, world, pb.torch_allgather(dist, device)) + pb.torch_device_collectives(dist, device))
        ctx.sync()
        self.setup_ms = 1e3 * (time.perf_counter() - t0)
        self.values_dev = ctx.malloc(values.nbytes)
        ctx.h2d(self.values_dev, self.values)

    def prove_dev(self):
        return self.ctx.prove_dev(self.pp.srs, self.pk, self.values_dev, self.pi_pos, self.pi_vals)

    def prove_host(self):
        return self.ctx.prove(self.pp.srs, self.pk, self.values, self.pi_pos, self.pi_vals)

    def verify(self, proof):
        import plonk_prototype_b200 as pb
        beta_h = pb.opening_key_from_tau(pb.scalars_to_mont([self.tau]))
        return pb.verify(self.vk, self.n, LABEL, proof, self.pi_pos, self.pi_vals, beta_h)

    def close(self):
        self.ctx.free(self.values_dev)
        self.ctx.prover_key_free(self.pk)
        self.pp.close()


def msm_model_imad(n):
    """SURVEY.md §8d work model of one MSM of n points, in IMAD.WIDE lane-ops: N·⌈256/(log₂N−4)⌉·10 Fp mul·300."""
    L = max(n.bit_length() - 1, 5)
    return float(n) * (-(-256 // max(L - 4, 1))) * 10 * 300.0


def timed_proves(setup, args, torch, stream, dist=None, device=None):
    """W warm-up + K timed proofs, twice: witness resident in HBM (CUDA events on the library's stream, profiling on so
    the per-kernel sums of exactly these K steps are known) and witness in pinned host memory (wall clock)."""
    ctx = setup.ctx

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    proofs = set()
    sampler = ClockSampler(ctx.device)   # started before the warm-up: nvidia-smi needs a moment, and a sharded step is milliseconds
    time.sleep(0.5)
    for _ in range(args.warmup):
        proofs.add(setup.prove_dev())
    ctx.profile_enable(True)
    ctx.profile_reset()
    barrier()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    torch.cuda.cudart().cudaProfilerStart()   # `ncu --profile-from-start off` then lists exactly the launches of the timed steps
    e0.record(stream)
    for _ in range(args.steps):
        last_proof = setup.prove_dev()
        proofs.add(last_proof)
    e1.record(stream)
    barrier()
    torch.cuda.cudart().cudaProfilerStop()
    wall_dev_ms = 1e3 * (time.perf_counter() - t0) / args.steps
    launches = ctx.launch_count() - l0
    dev_ms = e0.elapsed_time(e1) / args.steps
    sums = {k: ctx.profile_sum_ms(k) for k in ("msm.accumulate", "msm.sort", "msm.partials", "msm.reduce", "msm.total", "ntt.total")}
    rounds = {"round%d" % k: ctx.profile_sum_ms("prove.round%d" % k)[0] / args.steps for k in range(1, 6)}
    ctx.profile_enable(False)
    if args.steps * wall_dev_ms < 400.0:    # keep the sampler over a few more (untimed) steps so that it sees the GPU under load
        for _ in range(int(400.0 / max(wall_dev_ms, 1.0)) + 1):
            setup.prove_dev()
    clocks = sampler.stop()
    for _ in range(min(args.warmup, 2)):
        proofs.add(setup.prove_host())
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        proofs.add(setup.prove_host())
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / args.steps
    if dist is not None:
        t = torch.tensor([dev_ms, e2e_ms, wall_dev_ms] + [rounds["round%d" % k] for k in range(1, 6)], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        v = t.tolist()
        dev_ms, e2e_ms, wall_dev_ms = v[:3]
        rounds = {"round%d" % k: v[2 + k] for k in range(1, 6)}
    return {"dev_ms": dev_ms, "e2e_ms": e2e_ms, "wall_dev_ms": wall_dev_ms, "proofs": proofs, "launches": int(launches), "clocks": clocks,
            "sums": sums, "rounds_ms": {k: round(v, 3) for k, v in rounds.items()}, "last_proof": last_proof}


def prove_roofline(setup, timed, args, imad_peak, n_per_msm):
    """msm_accumulate_kernel inside the K timed proofs (the dominant kernel of a prove) against the live IMAD.WIDE peak."""
    acc_ms, acc_launches = timed["sums"]["msm.accumulate"]
    acc_per_step = acc_ms / args.steps
    alg = 11 * msm_model_imad(n_per_msm)   # 11 commitments per proof: 4 wires, z, 4 quotient parts, 2 opening witnesses
    return {
        "bound": "imad", "kernel": "msm_accumulate_kernel", "achieved": alg / (acc_per_step * 1e-3) / 1e12, "peak": imad_peak / 1e12,
        "unit": "T IMAD.WIDE.U32 lane-op/s", "frac": alg / (acc_per_step * 1e-3) / imad_peak,
        # dram__bytes_read.sum + dram__bytes_write.sum per accumulate launch inside a 2^20-gate prove on one GPU, ncu --set full
        # (profiles/ncu_prove_r02_summary.txt: 11.1 GB for a batch-of-4 launch, 2.87 GB for a single one; 4 launches = 11 MSMs per
        # proof ⇒ ≈ 7.7 GB per launch on average, against ≈ 3.9 GB algorithmic — 8-byte entries + 96-byte base gathers)
        "traffic": 7.7e9 if (n_per_msm == 1 << 20) else None,
        "kernel_ms_per_step": acc_per_step, "launches_per_step": acc_launches / args.steps,
        "avg_launch_ms": acc_ms / max(acc_launches, 1), "share_of_step": acc_per_step / timed["dev_ms"],
        "peak_source": "pb200_imad_peak: IMAD.WIDE.U32.X carry-chain microbenchmark run in this process (MEASURED_PEAKS.json holds no integer peak)",
        "model": "per proof 11 MSMs x N*ceil(256/(log2N-4))*10 Fp mul*300 IMAD.WIDE with N = %d (SURVEY.md §8d, unchanged; the kernel runs wider "
                 "windows over pre-doubled bases, so the fraction may exceed 1: fewer additions than the model's window count)" % n_per_msm,
        "measured": "CUDA events around every msm_accumulate_kernel launch of the K timed proofs (library stream), summed",
        "phases_ms_per_step": {"msm.sort": timed["sums"]["msm.sort"][0] / args.steps, "msm.accumulate": acc_per_step,
                               "msm.partials": timed["sums"]["msm.partials"][0] / args.steps,
                               "msm.reduce": timed["sums"]["msm.reduce"][0] / args.steps, "ntt": timed["sums"]["ntt.total"][0] / args.steps},
    }


def run_ours(args, rank, world, local_rank):
    import torch
    import plonk_prototype_b200 as pb

    dist = None
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=device)
    ctx = pb.Context(local_rank)  # raises without a B200: there is no fallback
    stream = torch.cuda.ExternalStream(ctx.stream, device=device)
    L = args.log_gates
    cores = os.cpu_count() or 1
    imad_peak, _ = ctx.imad_peak()

    lib_coll = args.collectives == "lib"
    if world > 1 and lib_coll:
        ctx.comm_init_from_torch(dist)   # torch.distributed only carries the 128-byte NCCL id
    setup = ProveSetup(ctx, L, torch, shard=(rank, world) if world > 1 else None, dist=dist, device=device, lib_collectives=lib_coll)
    timed = timed_proves(setup, args, torch, stream, dist, device)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, timed["last_proof"])
    proof = next(iter(timed["proofs"]))
    parity = {"deterministic": len(timed["proofs"]) == 1, "verifier_accepts": bool(setup.verify(proof)) if rank == 0 else None}
    extra = {}
    n_per_msm = (1 << L) // world
    if rank == 0:
        extra["roofline"] = prove_roofline(setup, timed, args, imad_peak, n_per_msm)

    if world == 1:
        # ---- CPU baseline = parity check: the C restatement proves the same circuit on the GPU's own commit key; bytes must match
        if not args.skip_cpu:
            est = lambda lg: 4.8 * (1 << (lg - 16)) * 8.0 / min(cores, 20)  # noqa: E731  (2^16: 4.8 s on 8 threads, measured)
            cl = L
            while cl > 12 and est(cl) > 60.0:
                cl -= 1
            gpu_same = None
            if cl == L:
                srs_host = np.zeros((1 << L, 12), np.uint64)
                ctx.d2h(srs_host, ctx.srs_dev_ptr(setup.pp.srs))
                cpu_proof, cpu_vk, t_pre, t_prove = cpu_prove(L, cores, srs=srs_host, circuit=setup.circuit)
                del srs_host
                parity["byte_identical_with_cpu_port"] = bool(cpu_proof == proof and cpu_vk == setup.vk)
                parity["compared_at_log_gates"] = L
            else:  # few host cores: bounded sample, with the GPU prove of that size beside it
                gpu_same, t_pre, t_prove, ok = gpu_prove_ms_and_check(ctx, cl, torch, cores)
                parity["byte_identical_with_cpu_port"] = bool(ok)
                parity["compared_at_log_gates"] = cl
            if parity["byte_identical_with_cpu_port"] is False:
                raise SystemExit("GPU proof differs from the CPU restatement — refusing to report a number")
            _, _, _, t1 = cpu_prove(14, 1)
            g14 = gpu_prove_ms(ctx, 14, torch)
            extra["cpu_baseline"] = {
                "value": 1e3 * t_prove, "unit": "ms", "cores": cores, "kind": "port", "log_gates": cl, "preprocess_ms": 1e3 * t_pre,
                "gpu_ms_same_size": gpu_same if cl != L else timed["e2e_ms"],
                "single_thread": {"log_gates": 14, "cpu_ms": 1e3 * t1, "gpu_ms": g14,
                                  "note": "1 thread = what /root/reference/Cargo.toml:19 builds (dusk-plonk without `std`: no rayon)"},
                "sample": "one prove_with_preprocessed of the same synthetic circuit at 2^%d gates by the C restatement of dusk-plonk 0.8 "
                          "(oracle/plonk_oracle.inc), %d threads, on the GPU run's own SRS (proof bytes compared with the GPU proof); "
                          "the Rust reference is not buildable here (no cargo, crates not vendored)" % (cl, cores)}
        parity["note"] = "parity unpinned against the Rust crates (not on disk); oracle = C restatement + independent Python model"
        if not args.skip_large:
            setup_bytes = ctx.prover_key_bytes(setup.pk)
            setup.close()
            setup = None
            extra["msm"] = bench_msm(ctx, stream, args, torch, imad_peak, None, 0, 1, device)
            extra["ntt"] = bench_ntt(ctx, stream, args, imad_peak, torch)
            if args.large_log_gates > L:
                extra["prove_2e%d" % args.large_log_gates] = bench_prove_large(ctx, args, torch, stream)
            extra["prover_key_gib"] = setup_bytes / 2**30
    else:
        # every rank also proves alone (one GPU, full commit key): the sharded proof must be the same bytes
        single = ProveSetup(ctx, L, torch)
        p1 = single.prove_host()
        same = torch.tensor([1 if (p1 == proof and single.vk == setup.vk) else 0], device=device)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        parity["equals_single_gpu_proof"] = bool(int(same))
        single.close()
        if not bool(int(same)):
            raise SystemExit("sharded proof differs from the single-GPU proof — refusing to report a number")
        setup.close()
        setup = None
        if not args.skip_large:
            m = bench_msm(ctx, stream, args, torch, imad_peak, dist, rank, world, device)
            s = bench_ntt_sharded(ctx, dist, rank, world, args, torch)
            big = bench_prove_large(ctx, args, torch, stream, dist, rank, world, device) if args.large_log_gates > L else None
            if rank == 0:
                extra["msm"], extra["ntt_sharded"] = m, s
                if big is not None:
                    extra["prove_sharded_2e%d" % args.large_log_gates] = big

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except (OSError, ValueError):
            pass
        n_vars_bytes = int((6 + 2 * (((1 << L) - N_PUB - 3) // 2) + N_PUB - 1) * 32)
        line = {
            "metric": headline_metric(L), "value": timed["dev_ms"], "unit": "ms", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": timed["dev_ms"], "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE,
            "data": "synthetic", "config": headline_config(L, world),
            "e2e": {"value": timed["e2e_ms"], "unit": "ms", "ms_per_step": timed["e2e_ms"],
                    "h2d_bytes_per_step": n_vars_bytes + N_PUB * 36, "d2h_bytes_per_step": 1040,
                    "note": "pb200_prove: witness (value of every variable) from pinned host memory, proof bytes to the host; the commit key "
                            "and prover key are resident, as CommitKey / ProverKey are across dusk-plonk proofs"},
            "gpu_launches": timed["launches"], "clocks": timed["clocks"], "parity": parity, "rounds_ms": timed["rounds_ms"],
            "wall_ms_per_step": timed["wall_dev_ms"], "hbm_peak_gbs": peaks.get("hbm_gbs"),
            "sharding": ("commitments by point range (commit-key slice per rank, 144-byte partial sums all-gathered); round 3 as sharded "
                         "four-step transforms (peer stores over NVLink + one all-to-all back); rounds 1, 2, 4, 5 replicated; collectives: "
                         + ("NCCL inside libpb200.so on the library's stream (pb200_comm)" if lib_coll else "torch.distributed callbacks")) if world > 1 else "single GPU",
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if setup is not None:
        setup.close()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


def gpu_prove_ms(ctx, L, torch):
    s = ProveSetup(ctx, L, torch)
    for _ in range(2):
        s.prove_host()
    t = []
    for _ in range(3):
        t0 = time.perf_counter()
        s.prove_host()
        t.append(1e3 * (time.perf_counter() - t0))
    s.close()
    return sum(t) / len(t)


def gpu_prove_ms_and_check(ctx, L, torch, cores):
    """GPU prove at a reduced size next to the CPU restatement on the same SRS (hosts with few cores)."""
    s = ProveSetup(ctx, L, torch)
    proof = s.prove_host()
    t = []
    for _ in range(3):
        t0 = time.perf_counter()
        s.prove_host()
        t.append(1e3 * (time.perf_counter() - t0))
    srs_host = np.zeros((1 << L, 12), np.uint64)
    ctx.d2h(srs_host, ctx.srs_dev_ptr(s.pp.srs))
    cpu_proof, cpu_vk, t_pre, t_prove = cpu_prove(L, cores, srs=srs_host, circuit=s.circuit)
    ok = cpu_proof == proof and cpu_vk == s.vk
    s.close()
    return sum(t) / len(t), t_pre, t_prove, ok


# ------------------------------------------------------------------------------------------- MSM
def bench_msm(ctx, stream, args, torch, imad_peak, dist, rank, world, device):
    """BASELINE.json configs[1], largest size: ONE G1 MSM of 2^26 points.  N = 1: the whole MSM on one GPU.  N > 1: the same
    MSM split by point range (rank r holds bases / scalars [r·2^26/N, (r+1)·2^26/N)), the 144-byte partial results
    all-gathered over NCCL and summed on rank 0 (strong scaling).  Result checked against the closed form Σ sᵢ(a + i·d)·G."""
    import plonk_prototype_b200 as pb
    LT = args.msm_log_n
    n = (1 << LT) // world
    a_rank = msm_shard_base(rank, n)
    bases = ctx.malloc(n * 96)
    ctx.synthetic_bases_dev(bases, n, a_rank, D0)
    srs = ctx.srs_wrap_dev(bases, n)
    pinned = torch.empty((n, 4), dtype=torch.int64, pin_memory=True)
    s_host = pinned.numpy().view(np.uint64)
    msm_scalar_slice(LT, rank, world, s_host)
    s_dev = ctx.malloc(n * 32)
    ctx.h2d(s_dev, s_host)
    steps = args.steps

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    def combine(out):
        if dist is None:
            return out
        parts = gather_partials(dist, out, world, device)  # 144 B per rank over NVLink: the only collective on the MSM path
        if rank == 0:
            return ctx.g1_sum(parts)
        return out

    res = combine(ctx.msm_dev(srs, s_dev, n))
    k_local = closed_form_scalar(s_host, a_rank, D0)
    if dist is not None:
        ks = [None] * world
        dist.all_gather_object(ks, k_local)
        k_total = sum(ks) % R_MOD
    else:
        k_total = k_local
    verified = None
    if rank == 0:
        O = oracle()  # checker only (result verification), never the measured path
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import model
        verified = bool(O.g1_proj_to_affine_canonical(res) == model.g1_mul(model.G1_GEN, k_total))
        if not verified:
            raise SystemExit("MSM result does not match the closed form — refusing to report a number")
    for _ in range(3):
        combine(ctx.msm_dev(srs, s_dev, n))
    ctx.profile_enable(True)
    ctx.profile_reset()
    barrier()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        combine(ctx.msm_dev(srs, s_dev, n))
    e1.record(stream)
    barrier()
    launches = (ctx.launch_count() - l0) // steps
    dev_ms = e0.elapsed_time(e1) / steps
    ph = {k: ctx.profile_sum_ms("msm." + k)[0] / steps for k in ("sort", "accumulate", "partials", "reduce")}
    ctx.profile_enable(False)
    for _ in range(2):
        combine(ctx.msm(srs, s_host))
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        combine(ctx.msm(srs, s_host))
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / steps
    if dist is not None:
        t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms = t.tolist()
    total = n * world
    alg = msm_model_imad(n)   # per GPU: what one rank's accumulate launch processes
    out = {
        "metric": "G1 MSM throughput, ONE 2^%d-point MSM over %d GPU%s (BASELINE.json configs[1])" % (LT, world, "s" if world > 1 else ""),
        "value": total / (dev_ms * 1e-3) / 1e6, "unit": "Mpts/s", "ms": dev_ms, "scaling": "strong", "points_total": total, "points_per_gpu": n,
        "steps": steps, "window_bits": int(pb._native.lib().pb200_msm_window_bits(n)), "kernels_per_msm": int(launches), "result_verified": verified,
        "e2e": {"value": total / (e2e_ms * 1e-3) / 1e6, "unit": "Mpts/s", "ms": e2e_ms, "h2d_bytes_per_step": n * 32, "d2h_bytes_per_step": 144,
                "note": "pb200_msm_g1: scalars from pinned host memory, result on the host; bases are the resident SRS"},
        "roofline": {"bound": "imad", "kernel": "msm_accumulate_kernel", "achieved": alg / (ph["accumulate"] * 1e-3) / 1e12, "peak": imad_peak / 1e12,
                     "unit": "T IMAD.WIDE.U32 lane-op/s", "frac": alg / (ph["accumulate"] * 1e-3) / imad_peak,
                     "whole_msm_frac": alg / (dev_ms * 1e-3) / imad_peak, "kernel_ms": ph["accumulate"], "share_of_step": ph["accumulate"] / dev_ms,
                     "traffic": 167.0e9 if (LT == 26 and world == 1) else None,
                     "traffic_note": "dram bytes read+written by one accumulate launch at 2^26, ncu --set full (profiles/ncu_full_r01_summary.txt); ~84 GB algorithmic",
                     "model": "N*ceil(256/(log2N-4))*10 Fp mul*300 IMAD.WIDE per rank (SURVEY.md §8d)", "phases_ms": ph},
    }
    if world == 1 and not args.skip_cpu:
        O = oracle()
        cores = os.cpu_count() or 1
        sl = min(LT, args.cpu_sample_log)
        pts = O.synthetic_bases(1 << sl)
        sc = random_fr_limbs(0xB2000000 + LT, 1 << sl)
        t0 = time.perf_counter()
        O.msm_variable_base(pts, sc, threads=cores)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": (1 << sl) / dt / 1e6, "unit": "Mpts/s", "cores": cores, "kind": "port",
                               "sample": "msm_variable_base restatement (oracle/oracle.c, SURVEY App. B.1) on 2^%d distinct points, %d threads over "
                                         "windows: %.2f s (a 2^%d CPU MSM would take minutes)" % (sl, cores, dt, LT)}
    ctx.srs_free(srs)
    ctx.free(bases)
    ctx.free(s_dev)
    return out


# ------------------------------------------------------------------------------------------- NTT
def bench_ntt_sharded(ctx, dist, rank, world, args, torch):
    """Sharded four-step NTT (SURVEY.md §8e) of ONE 2^L vector over all ranks: column pass + exchange + batched rows.
    Strong scaling by nature (the domain is fixed); verified by a sharded ifft(fft(x)) = x round trip here and against the
    single-GPU transform in tests/test_multi_gpu.py."""
    import plonk_prototype_b200 as pb
    L = args.ntt_dist_log_n
    be = pb.GpuBackend(ctx, dist, torch)
    dom = pb.DistributedDomain(L, rank, world, be)
    spec = dom.spec
    shard = random_fr_limbs(0xF1F00000 + L + 1000 * rank, spec.local)
    buf = torch.from_numpy(shard.view(np.int64).reshape(-1).copy()).cuda()
    tmp = torch.empty_like(buf)
    torch.cuda.synchronize()   # `buf` was filled on torch's stream
    dom.fft(buf, tmp)
    dom.ifft(buf, tmp)
    ctx.sync(); torch.cuda.synchronize()
    ok = bool((buf.cpu().numpy().view(np.uint64).reshape(-1, 4) == shard).all())
    for _ in range(3):
        dom.fft(buf, tmp)
    dist.barrier(); ctx.sync(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = args.steps
    e0.record(be.stream)
    for _ in range(reps):
        dom.fft(buf, tmp)
    e1.record(be.stream)
    ctx.sync(); torch.cuda.synchronize(); dist.barrier()
    nccl_ms = e0.elapsed_time(e1) / reps
    # fused variant: the column kernel stores straight into the peers' row buffers (CUDA IPC over NVLink); wall clock
    # per transform including the cross-rank barrier, median of 10, input restored between repetitions
    peers = pb.PeerBuffers(ctx, dist, rank, world, spec.local)
    col = torch.from_numpy(shard.view(np.int64).reshape(-1).copy()).cuda()
    work = torch.empty_like(col)
    ts = []
    for i in range(13):
        work.copy_(col); torch.cuda.synchronize(); dist.barrier()
        t0 = time.perf_counter()
        dom.fft_fused(work, peers)
        ctx.sync()
        if i >= 3:
            ts.append((time.perf_counter() - t0) * 1e3)
    fused_ms = sorted(ts)[len(ts) // 2]
    buf.copy_(col)
    torch.cuda.synchronize()   # the copy runs on torch's stream, the transform on the library's
    dom.fft(buf, tmp)
    ctx.sync(); torch.cuda.synchronize()
    fused_out = np.empty((spec.local, 4), np.uint64)
    ctx.d2h(fused_out, peers.mine.ptr)
    same = bool((fused_out == buf.cpu().numpy().view(np.uint64).reshape(-1, 4)).all())
    peers.close()
    # the same transform driven entirely by the library (pb200_ntt_sharded_dev: NCCL all-to-all on the library's stream)
    lib_ms, lib_same = float("inf"), True
    if args.collectives == "lib":
        d_data, d_tmp = ctx.malloc(spec.local * 32), ctx.malloc(spec.local * 32)
        ctx.h2d(d_data, shard)
        ctx.ntt_sharded_dev(d_data, d_tmp, L, False)
        lib_out = np.empty((spec.local, 4), np.uint64)
        ctx.d2h(lib_out, d_data)
        lib_same = bool((lib_out == fused_out).all())
        for _ in range(3):
            ctx.ntt_sharded_dev(d_data, d_tmp, L, False)
        dist.barrier(); ctx.sync()
        e0.record(be.stream)
        for _ in range(reps):
            ctx.ntt_sharded_dev(d_data, d_tmp, L, False)
        e1.record(be.stream)
        ctx.sync(); dist.barrier()
        lib_ms = e0.elapsed_time(e1) / reps
        ctx.free(d_data); ctx.free(d_tmp)
    t = torch.tensor([nccl_ms, fused_ms, 0.0 if (ok and same and lib_same) else 1.0, lib_ms], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    nccl_ms, fused_ms, bad, lib_ms = t.tolist()
    ms = min(nccl_ms, fused_ms, lib_ms)
    return {"metric": "sharded four-step NTT, 2^%d points over %d GPUs (forward)" % (L, world), "ms": ms,
            "value": (1 << L) / (ms * 1e-3) / 1e6, "unit": "Melem/s", "scaling": "strong", "n1": spec.n1,
            "fused_peer_store_ms": fused_ms, "nccl_all_to_all_ms": nccl_ms, "library_nccl_ms": lib_ms if lib_ms != float("inf") else None,
            "exchange_bytes_per_gpu": spec.local * 32 * (world - 1) // world,
            "verified": bad == 0.0, "roundtrip_ok": ok, "fused_equals_nccl": same,
            "note": "fused: column kernel writes the owners' row buffers over NVLink peer memory, wall clock incl. the cross-rank barrier; "
                    "nccl: column kernel + all_to_all_single + transpose kernel, CUDA events"}


def bench_ntt(ctx, stream, args, imad_peak, torch):
    """BASELINE.json configs[2]: forward NTT of 2^24 scalars, device-resident and host-to-host, against both rooflines."""
    L = args.ntt_log_n
    n = 1 << L
    pinned = torch.empty((n, 4), dtype=torch.int64, pin_memory=True)
    x = pinned.numpy().view(np.uint64)
    random_fr_limbs(0xF1F00000 + L, n, out=x)
    keep = x.copy()
    d = ctx.malloc(n * 32)
    ctx.h2d(d, x)
    ctx.ntt_dev(d, L, 0, 0)
    ctx.ntt_dev(d, L, 1, 0)
    back = np.empty_like(keep)
    ctx.d2h(back, d)
    ok = bool((back == keep).all())
    for _ in range(max(args.warmup, 3)):
        ctx.ntt_dev(d, L, 0, 0)
    ctx.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = args.steps
    l0 = ctx.launch_count()
    e0.record(stream)
    for _ in range(reps):
        ctx.ntt_dev(d, L, 0, 0)
    e1.record(stream)
    ctx.sync()
    ms = e0.elapsed_time(e1) / reps
    launches = (ctx.launch_count() - l0) // reps
    ctx.ntt(x, L, 0, 0)
    t0 = time.perf_counter()
    for _ in range(3):
        ctx.ntt(x, L, 0, 0)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / 3
    ctx.free(d)
    alg_bytes_moved = 64.0 * n * launches                # what this build moves: 32 B read + 32 B write per element per pass
    alg_bytes_survey = 64.0 * n * (-(-L // 12))          # SURVEY.md §8d model
    alg_imad = (n / 2) * L * 136.0                       # SURVEY §8d: 272 lo/hi lane-ops = 136 IMAD.WIDE per Fr mul
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    hbm = peaks.get("hbm_gbs", 6650.0)
    out = {
        "metric": "NTT throughput (BLS12-381 Fr, 2^%d, forward, device-resident)" % L,
        "value": n / (ms * 1e-3) / 1e6, "unit": "Melem/s", "ms": ms, "kernels_per_transform": int(launches), "roundtrip_verified": ok,
        "e2e": {"value": n / (e2e_ms * 1e-3) / 1e6, "unit": "Melem/s", "ms": e2e_ms, "h2d_bytes_per_step": n * 32, "d2h_bytes_per_step": n * 32},
        "roofline": {"bound": "hbm", "achieved": alg_bytes_survey / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                     "frac": alg_bytes_survey / (ms * 1e-3) / 1e9 / hbm, "traffic": None,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                     "model": "64 B * n * ceil(log2 n / 12) (SURVEY.md §8d); this build moves 64 B * n * %d" % launches,
                     "moved_bytes_frac": alg_bytes_moved / (ms * 1e-3) / 1e9 / hbm},
        "roofline_imad": {"bound": "imad", "achieved": alg_imad / (ms * 1e-3) / 1e12, "peak": imad_peak / 1e12,
                          "unit": "T IMAD.WIDE.U32 lane-op/s", "frac": alg_imad / (ms * 1e-3) / imad_peak,
                          "model": "(n/2)*log2(n) Fr mul * 136 IMAD.WIDE (SURVEY.md §8d) — the roofline that binds a 255-bit field"},
    }
    if not args.skip_cpu:
        cores = os.cpu_count() or 1
        cpu_log = min(L, 22)
        O = oracle()
        xs = random_fr_limbs(0xF1F00000 + L, 1 << cpu_log)
        t0 = time.perf_counter()
        O.ntt(xs, 0, 0, cores)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": (1 << cpu_log) / dt / 1e6, "unit": "Melem/s", "cores": cores, "kind": "port",
                               "sample": "best_fft/parallel_fft restatement (oracle/oracle.c) on 2^%d, %d threads: %.2f s" % (cpu_log, cores, dt)}
    return out


# ------------------------------------------------------------------------------ 2^24-gate circuit
def bench_prove_large(ctx, args, torch, stream, dist=None, rank=0, world=1, device=None):
    """BASELINE.json configs[4]: the 2^24-gate synthetic circuit.  N = 1: one GPU (57 GiB prover key) — the baseline of the
    scaling curve.  N > 1: sharded prove; afterwards rank 0 proves the same circuit alone and the bytes must be equal."""
    L = args.large_log_gates
    s = ProveSetup(ctx, L, torch, shard=(rank, world) if world > 1 else None, dist=dist, device=device, lib_collectives=args.collectives == "lib")
    proofs = {s.prove_host() for _ in range(2)}
    reps = args.steps
    ctx.profile_enable(True)
    ctx.profile_reset()
    t = []
    for _ in range(reps):
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        proofs.add(s.prove_host())
        dt = time.perf_counter() - t0
        if dist is not None:
            x = torch.tensor([dt], device=device, dtype=torch.float64)
            dist.all_reduce(x, op=dist.ReduceOp.MAX)
            dt = float(x)
        t.append(1e3 * dt)
    rounds = [ctx.profile_sum_ms("prove.round%d" % k)[0] / reps for k in range(1, 6)]
    ctx.profile_enable(False)
    if dist is not None:
        x = torch.tensor(rounds, device=device, dtype=torch.float64)
        dist.all_reduce(x, op=dist.ReduceOp.MAX)
        rounds = x.tolist()
    proof = next(iter(proofs))
    out = {"metric": "PLONK prove, synthetic arithmetic circuit, 2^%d gates, %d GPU%s (BASELINE.json configs[4])" % (L, world, "s" if world > 1 else ""),
           "value": sum(t) / len(t), "unit": "ms", "min_ms": min(t), "steps": reps, "higher_is_better": False, "scaling": "strong",
           "setup_ms": s.setup_ms, "rounds_ms": {"round%d" % (k + 1): round(v, 2) for k, v in enumerate(rounds)},
           "deterministic": len(proofs) == 1, "prover_key_gib_per_gpu": ctx.prover_key_bytes(s.pk) / 2**30,
           "e2e": {"value": sum(t) / len(t), "unit": "ms", "h2d_bytes_per_step": int(s.values.nbytes), "d2h_bytes_per_step": 1040}}
    vk = s.vk
    if rank == 0:
        out["verifier_accepts"] = bool(s.verify(proof))
    s.close()
    if world > 1 and not args.skip_single_check:
        # rank 0 alone, full commit key (the other ranks wait at the barrier): byte equality with the sharded proof
        if rank == 0:
            one = ProveSetup(ctx, L, torch)
            p1 = one.prove_host()
            t0 = time.perf_counter()
            one.prove_host()
            out["single_gpu_ms"] = 1e3 * (time.perf_counter() - t0)
            out["equals_single_gpu_proof"] = bool(p1 == proof and one.vk == vk)
            one.close()
        dist.barrier()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-gates", type=int, default=20, help="log2 of the gate count of the headline PLONK prove")
    ap.add_argument("--large-log-gates", type=int, default=24, help="log2 of the gate count of the configs[4] prove (context object)")
    ap.add_argument("--msm-log-n", type=int, default=26, help="log2 of the TOTAL point count of the MSM context object")
    ap.add_argument("--ntt-log-n", type=int, default=24)
    ap.add_argument("--ntt-dist-log-n", type=int, default=26, help="log2 of the sharded NTT domain (N > 1 only)")
    ap.add_argument("--cpu-sample-log", type=int, default=20, help="log2 of the CPU MSM baseline's bounded sample")
    ap.add_argument("--skip-large", action="store_true", help="headline only: no MSM / NTT / 2^24-gate context objects")
    ap.add_argument("--skip-cpu", action="store_true", help="no CPU baseline legs (and no CPU byte-parity check)")
    ap.add_argument("--skip-single-check", action="store_true", help="N > 1: skip rank 0's single-GPU 2^24 proof")
    ap.add_argument("--collectives", default="lib", choices=["lib", "torch"],
                    help="N > 1: NCCL inside the library (pb200_comm) or torch.distributed callbacks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the proof of the last timed step to DIR/proof.npy (float64 bytes)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)
    if world not in (1, 2, 4, 8):
        raise SystemExit("sharded prove needs a power-of-two rank count ≤ 8")
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
