"""CPU tests of bench.py's host logic: the reference arm runs the checker only (it must never load the product
library), reports the circuit it actually proved, and the checker's circuit generator is the product's, row for row."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_oracle_synthetic_circuit_equals_product_helpers(oracle):
    from plonk_prototype_b200.synth import synthetic_circuit_columns, synthetic_circuit_columns_py
    for n_gates, n_pub in ((12, 2), (1000, 2), (5001, 3), (4096, 1)):
        a = oracle.synthetic_circuit_columns(n_gates, 0x5EED, n_pub)
        for b in (synthetic_circuit_columns(n_gates, 0x5EED, n_pub), synthetic_circuit_columns_py(n_gates, 0x5EED, n_pub)):
            for k in range(11):
                assert (a[0][k] is None) == (b[0][k] is None), k
                if a[0][k] is not None:
                    assert (a[0][k] == b[0][k]).all(), k
            for k in range(4):
                assert (a[1][k] == b[1][k]).all()
            assert (a[2] == b[2]).all() and (a[3] == b[3]).all() and (a[4] == b[4]).all()


def test_reference_arm_runs_without_the_product_library(tmp_path):
    code = ("import sys, runpy\n"
            "sys.argv = ['bench.py', '--impl', 'reference', '--log-gates', '10', '--steps', '2', '--warmup', '1', '--dump-outputs', %r]\n"
            "runpy.run_path(%r, run_name='__main__')\n"
            "assert not any(m.startswith('plonk_prototype_b200') for m in sys.modules), 'product package imported'\n"
            "assert 'libpb200' not in open('/proc/self/maps').read(), 'product library mapped'\n" % (str(tmp_path), os.path.join(ROOT, "bench.py")))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "ms" and line["higher_is_better"] is False
    assert line["steps"] == 2 and len(line["steps_ms"]) == 2 and line["same_config"] is True
    assert line["config"]["log_gates"] == 10 and line["sample_log_gates"] == 10
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    proof = np.load(tmp_path / "proof.npy")
    assert proof.dtype == np.float64 and proof.shape == (1040,)
    assert hashlib.sha256(proof.astype(np.uint8).tobytes()).hexdigest()[:16] == line["proof_sha256_16"]


def test_reference_arm_bounds_its_sample_and_says_so():
    env = dict(os.environ, PB200_REF_BUDGET_S="3")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--log-gates", "16", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["same_config"] is False and line["sample_log_gates"] < 16 and "BOUNDED SAMPLE" in line["cpu_baseline"]["sample"]
    assert line["config"]["log_gates"] == 16


def test_both_arms_share_config_and_metric():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.headline_config(20, 1) == bench.headline_config(20, 1)
    assert "2^20" in bench.headline_metric(20)
    # the global MSM scalar vector is the same problem for every rank count
    full = np.empty((1 << 10, 4), np.uint64)
    bench.msm_scalar_slice(10, 0, 1, full)
    for world in (2, 4, 8):
        parts = [bench.msm_scalar_slice(10, r, world, np.empty(((1 << 10) // world, 4), np.uint64)) for r in range(world)]
        assert (np.concatenate(parts) == full).all()
