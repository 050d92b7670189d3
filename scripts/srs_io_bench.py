"""Load and store rates of commit keys in the checked compressed format (pb200_srs_from_compressed / pb200_srs_to_compressed,
csrc/srs_io.cu) at 2^16 … 2^26 points, with a labelled CPU baseline.

Per size: a key τ^i·G is generated on the device, stored (to_compressed) and loaded back (from_compressed) `--reps` times.
Reported per direction: the blocking call on the host clock (copies included) and the kernel alone (CUDA events,
"srs.decompress" / "srs.compress"), as points/s; for the load also the Fp-multiplication rate, from the counted
multiplications per valid point (1,888: csrc/g1_codec.cuh).  The reloaded key is compared with the generated one at every
size up to 2^22 (its compressed bytes again; the tests compare the device images themselves).

CPU baseline: the reference decoder (tests/srs_io_ref.c: square root, then r·P = O — upstream's algorithm) on every host
thread over a 2^16-point sample, extrapolated linearly to each size and labelled as such.

    python scripts/srs_io_bench.py --out srs_io.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.dont_write_bytecode = True

FP_MULS_PER_POINT = 1888   # csrc/g1_codec.cuh: 606 (square root) + 2 × 637 (two multiplications by |x|) + 8


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power, clock = (s.strip() for s in out[0].split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers stay valid without it, but say so
        return {"name": "unknown (%s)" % e}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logs", default="16,20,22,24,26")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import plonk_prototype_b200 as pb
    import srs_io_ref as ref

    ctx = pb.Context(0)
    ctx.profile_enable(True)
    tau = pb.scalars_to_mont([0x7A05ED])
    warm = ctx.srs_generate(tau, 1 << 10)                       # module load, first launches
    ctx.srs_free(ctx.srs_from_compressed(ctx.srs_to_compressed(warm)))
    ctx.srs_free(warm)

    rows, sample = [], None
    for log_n in (int(s) for s in a.logs.split(",")):
        n = 1 << log_n
        srs = ctx.srs_generate(tau, n)
        st_host, st_kern, ld_host, ld_kern = [], [], [], []
        enc = None
        for _ in range(a.reps):
            t0 = time.perf_counter()
            enc = ctx.srs_to_compressed(srs)
            st_host.append(time.perf_counter() - t0)
            st_kern.append(ctx.profile_ms("srs.compress") * 1e-3)
        if sample is None:
            sample = enc[:48 << 16]
        for rep in range(a.reps):
            t0 = time.perf_counter()
            srs2 = ctx.srs_from_compressed(enc)
            ld_host.append(time.perf_counter() - t0)
            ld_kern.append(ctx.profile_ms("srs.decompress") * 1e-3)
            if rep == 0 and log_n <= 22:
                assert ctx.srs_to_compressed(srs2) == enc, "reloaded key differs at 2^%d" % log_n
            ctx.srs_free(srs2)
        ctx.srs_free(srs)
        del enc
        med = statistics.median
        rows.append({
            "log_n": log_n, "points": n, "reps": a.reps,
            "store_call_s": med(st_host), "store_kernel_s": med(st_kern),
            "store_call_points_per_s": n / med(st_host), "store_kernel_points_per_s": n / med(st_kern),
            "store_kernel_GB_per_s": 144 * n / med(st_kern) / 1e9,       # 96 B read + 48 B written per point
            "load_call_s": med(ld_host), "load_kernel_s": med(ld_kern),
            "load_call_points_per_s": n / med(ld_host), "load_kernel_points_per_s": n / med(ld_kern),
            "load_kernel_fp_mul_per_s": FP_MULS_PER_POINT * n / med(ld_kern),
            "load_kernel_s_all": ld_kern, "store_kernel_s_all": st_kern,
        })
        print(json.dumps(rows[-1]), flush=True)

    threads = os.cpu_count() or 1
    ref.lib()
    t0 = time.perf_counter()
    st, _ = ref.g1_from_bytes_checked(sample, threads=threads)
    cpu_s = time.perf_counter() - t0
    assert (st == 0).all()
    m = len(sample) // 48
    cpu = {"what": "CPU reference decoder (square root, then r·P = O), %d host threads, %d-point sample; other sizes "
                   "EXTRAPOLATED linearly from it, not measured" % (threads, m),
           "sample_points": m, "sample_s": cpu_s, "points_per_s": m / cpu_s,
           "extrapolated_load_s": {str(r["log_n"]): r["points"] * cpu_s / m for r in rows}}
    res = {"card": card(), "fp_muls_per_point": FP_MULS_PER_POINT, "sizes": rows, "cpu_baseline": cpu,
           "launches": ctx.launch_count()}
    print(json.dumps(cpu))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
