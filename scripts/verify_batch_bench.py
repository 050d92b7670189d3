"""Batched verification rates (pb200_verify_batch) against the single-proof host verifier (pb200_verify).

64 distinct proofs of one ~2^10-gate synthetic circuit (the chain's starting value varies, so every proof has its own
witness and public inputs) are repeated to K ∈ {1, 16, 256, 4096, 16384, 65536}; every K is warmed up, then timed over
--reps calls.  Also one K = 4096 batch with 17 invalid proofs (bisection), and pb200_verify on a 32-proof sample on the
same host.  Records call wall clock, per-phase times (pb200_profile_sum_ms over one profiled call), the number of
pairing checks, proofs/s, the GPU name and power limit and the host thread count.

    python scripts/verify_batch_bench.py [--out profiles/verify_batch_r04.json] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import model  # noqa: E402
import plonk_model as pm  # noqa: E402
import plonk_prototype_b200 as pb  # noqa: E402

LABEL = b"pb200 verify_batch bench"
TAU = 0xBE7C4
PHASES = ["verify.decompress", "verify.prepare", "verify.weight", "verify.msm", "verify.pairing"]


def circuit(x0, n_gates=1000, seed=0xB47C, n_pub=2):
    comp = pm.Composer()
    consts = model.random_fr(seed, 4)
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
    return comp


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [v.strip() for v in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "verify_batch_r04.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sizes", default="1,16,256,4096,16384,65536")
    args = ap.parse_args()

    ctx = pb.Context(0)
    comps = [circuit(3 + 7 * i) for i in range(64)]
    n = pm.domain(comps[0].n)["size"]
    pp = pb.PublicParameters(n - 1, TAU, ctx)
    sel = [pb.scalars_to_mont(comps[0].q[k]) if any(comps[0].q[k]) else None for k in pm.SELECTORS]
    wires = [np.asarray(w, dtype=np.uint32) for w in comps[0].w]
    pk, vk = ctx.preprocess(pp.srs, sel, wires, len(comps[0].values), LABEL)
    gates = np.asarray(sorted(comps[0].pi), dtype=np.uint32)
    pis = [pb.scalars_to_mont([c.pi[int(g)] for g in gates]) for c in comps]
    proofs = [ctx.prove(pp.srs, pk, pb.scalars_to_mont(c.values), gates, pis[i]) for i, c in enumerate(comps)]
    ctx.prover_key_free(pk)

    def inputs(K):
        return b"".join(proofs[k % 64] for k in range(K)), np.stack([pis[k % 64] for k in range(K)])

    def run(K, blob, piv, reps):
        ctx.verify_batch(vk, n, LABEL, blob, gates, piv, pp.beta_h, seed=b"\x11" * 32)   # warm-up
        ctx.profile_enable(True)
        ctx.profile_reset()
        got = ctx.verify_batch(vk, n, LABEL, blob, gates, piv, pp.beta_h, seed=b"\x12" * 32)
        phases = {}
        for p in PHASES:
            ms, cnt = ctx.profile_sum_ms(p)
            phases[p] = {"ms": round(ms, 4), "samples": cnt}
        ctx.profile_enable(False)
        walls = []
        for r in range(reps):
            t0 = time.perf_counter()
            ctx.verify_batch(vk, n, LABEL, blob, gates, piv, pp.beta_h, seed=bytes([r]) * 32)
            walls.append(time.perf_counter() - t0)
        wall = min(walls)
        return got, {"K": K, "call_wall_s_min": round(wall, 6), "call_wall_s_all": [round(w, 6) for w in walls],
                     "proofs_per_s": round(K / wall, 1), "us_per_proof": round(1e6 * wall / K, 3), "profiled_call": phases}

    rows = []
    for K in [int(v) for v in args.sizes.split(",")]:
        blob, piv = inputs(K)
        got, row = run(K, blob, piv, args.reps)
        assert got.all(), K
        rows.append(row)
        print(json.dumps(row), flush=True)

    # one K = 4096 batch with 17 invalid proofs
    K = 4096
    rng = np.random.default_rng(0x17)
    bad = sorted(rng.choice(K, size=17, replace=False).tolist())
    ps = [proofs[k % 64] for k in range(K)]
    for b in bad:
        p = bytearray(ps[b])
        p[528 + 5] ^= 0x10
        ps[b] = bytes(p)
    got, bis = run(K, b"".join(ps), inputs(K)[1], 1)
    assert [k for k in range(K) if not got[k]] == bad
    bis["invalid"] = 17
    print(json.dumps(bis), flush=True)

    # pb200_verify on the same host, 32 proofs
    t0 = time.perf_counter()
    for i in range(32):
        assert pb.verify(vk, n, LABEL, proofs[i], gates, pis[i], pp.beta_h)
    single_s = (time.perf_counter() - t0) / 32
    per_4096 = next(r for r in rows if r["K"] == 4096)["call_wall_s_min"] / 4096 if any(r["K"] == 4096 for r in rows) else None
    out = {
        "what": "pb200_verify_batch on one GPU vs pb200_verify on one host thread; 64 distinct proofs of one 1000-gate circuit "
                "(n = %d, 2 public inputs) repeated to K; call wall clock is the best of %d calls after a warm-up" % (n, args.reps),
        "gpu": gpu_info(),
        "host_threads": os.cpu_count(),
        "batch": rows,
        "batch_17_invalid_of_4096": bis,
        "pb200_verify_single_proof_s": round(single_s, 6),
        "speedup_per_proof_at_4096": round(single_s / per_4096, 1) if per_4096 else None,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "host_threads", "pb200_verify_single_proof_s", "speedup_per_proof_at_4096")}))
    pp.close()
    ctx.close()


if __name__ == "__main__":
    main()
