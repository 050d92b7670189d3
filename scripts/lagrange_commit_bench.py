"""Cost of the Lagrange-basis commit key (pb200_srs_lagrange) and what it saves in the batched MSM.

- Key build at 2^12 … 2^22 points (powers-of-τ key generated on the device): wall clock of pb200_srs_lagrange (one
  call, synchronised) and of the pre-doubled copies the prover key adds to it, and the device bytes of both.
- Per-phase MSM times (pb200_profile_sum_ms of msm.sort / msm.accumulate / msm.partials / msm.reduce) at 2^20 points for
  one batch of four scalar vectors against the pre-doubled key: dense, half zero, and a single non-zero scalar per vector.
- Registers, stack and spills of the lagrange_* kernels from the ptxas log the build leaves in csrc/build/.

    python scripts/lagrange_commit_bench.py [--out profiles/lagrange_commit_r05.json] [--reps 5] [--max-log 22]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import plonk_prototype_b200 as pb  # noqa: E402

TAU = 0xB2000014
PHASES = ["msm.sort", "msm.accumulate", "msm.partials", "msm.reduce", "msm.total"]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [v.strip() for v in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def ptxas_info():
    log = os.path.join(ROOT, "plonk-prototype_b200", "csrc", "build", "lagrange.ptxas.log")
    out, name = {}, None
    for line in open(log):
        m = re.search(r"Compiling entry function .*(lagrange_(?:load|stage|normalize)_kernel)", line)
        if m:
            name = m.group(1)
            continue
        if name is None:
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and "stack_bytes" not in out.get(name, {}):   # the entry's own frame, not its callees'
            out.setdefault(name, {}).update(stack_bytes=int(m.group(1)), spill_store_bytes=int(m.group(2)), spill_load_bytes=int(m.group(3)))
        m = re.search(r"Used (\d+) registers", line)
        if m:
            out.setdefault(name, {})["registers"] = int(m.group(1))
    return out


def key_build(ctx, log_n):
    n = 1 << log_n
    srs = ctx.srs_generate(pb.scalars_to_mont([TAU]), n)
    ctx.sync()
    t0 = time.perf_counter()
    lag = ctx.srs_lagrange(srs, log_n)
    t1 = time.perf_counter()
    ctx.srs_precompute(lag)
    ctx.sync()
    t2 = time.perf_counter()
    W = -(-256 // _window_pre(n))
    ctx.srs_free(lag)
    ctx.srs_free(srs)
    return {"log_n": log_n, "lagrange_s": t1 - t0, "precompute_s": t2 - t1, "lagrange_bytes": n * 96,
            "pre_doubled_bytes": W * n * 96, "prover_key_adds_bytes": (W + 1) * n * 96,
            "twiddle_multiplications": (n // 2) * log_n - (n - 1) + n}


def _window_pre(n):
    """msm.cu choose_window_pre: c minimising W·n + 3·2^(c−1)."""
    best, best_c = None, 8
    for c in range(8, 24):
        cost = -(-256 // c) * n + 3.0 * (1 << (c - 1))
        if best is None or cost <= best:
            best, best_c = cost, c
    return best_c


def msm_phases(ctx, log_n, reps):
    n = 1 << log_n
    pp = pb.PublicParameters(n - 1, TAU, ctx)
    lag = ctx.srs_lagrange(pp.srs, log_n)
    ctx.srs_precompute(lag)
    rng = np.random.default_rng(5)
    dense = rng.integers(0, 2**63, size=(4 * n, 4), dtype=np.uint64)
    dense[:, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)          # < r, Montgomery images of arbitrary scalars
    half = dense.copy()
    half[::2] = 0
    single = np.zeros_like(dense)
    single[n // 3::n] = dense[n // 3::n]
    dev = ctx.malloc(dense.nbytes)
    out = {}
    for name, v in (("dense", dense), ("half_zero", half), ("single_nonzero", single)):
        ctx.h2d(dev, v)
        for _ in range(2):
            ctx.msm_batch_dev(lag, dev, n, 4, n)
        ctx.profile_enable(True)
        ctx.profile_reset()
        t0 = time.perf_counter()
        for _ in range(reps):
            ctx.msm_batch_dev(lag, dev, n, 4, n)
        wall = (time.perf_counter() - t0) / reps
        out[name] = {"wall_ms": 1e3 * wall, **{p: ctx.profile_sum_ms(p)[0] / reps for p in PHASES}}
        ctx.profile_enable(False)
    ctx.free(dev)
    ctx.srs_free(lag)
    pp.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "lagrange_commit_r05.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--max-log", type=int, default=22)
    args = ap.parse_args()
    ctx = pb.Context(0)
    key_build(ctx, 10)  # module load / first launches
    res = {"gpu": gpu_info(), "ptxas": ptxas_info(),
           "key_build": [key_build(ctx, L) for L in range(12, args.max_log + 1)],
           "msm_batch4_2e20_ms": msm_phases(ctx, 20, args.reps),
           "note": "key build: one synchronised call each, wall clock; MSM: batch of 4 vectors of 2^20 scalars against the pre-doubled "
                   "Lagrange key, CUDA-event phase times averaged over --reps calls after 2 warm-ups"}
    ctx.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["key_build"][-1]), json.dumps(res["msm_batch4_2e20_ms"]))


if __name__ == "__main__":
    main()
