"""bench.py's reference arm runs on the host cores only, so its JSON line can be checked here: the keys and meanings the
driver's contract asks for (the GPU arm prints the same line plus roofline / clocks; it is checked on the GPU box)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["unit"] == "pool-evals/s" and d["higher_is_better"] is True and d["scaling"] == "strong"
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert "workload" in d["config"] and "1000000 constant-product pools" in d["config"]["workload"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    e = d["e2e"]
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0 and e["value"] > 0
    assert e["status"] == "optimal" and d["time_to_1e-6_gap"]["rel_gap"] <= 1e-6
    assert "oracle_solve_pairs" in e["what"]            # the CPU arm's solve is the oracle's own C loop, not product code


def test_bench_b200_arm_is_syntactically_sound_and_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "20", "--warmup", "5"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "needs a CUDA device" in (out.stderr + out.stdout)


@pytest.mark.gpu
def test_b200_arm_times_exactly_the_steps_asked_and_dumps_its_last_step(tmp_path):
    """70 steps = one replay of the 64-step graph + a 6-step tail graph; the dumped outputs are what the 70th step
    returned, i.e. the oracle's evaluation of that step's pool instance and prices"""
    import bench
    from cfmm_routing_code_b200 import instances as I
    from oracle import c_oracle as CO
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "70", "--warmup", "1", "--no-cpu",
                          "--no-e2e", "--no-configs", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 70
    k = (70 - 1) % bench.n_instances(bench.M_POOLS)               # the instance and prices of the last step (N = 1)
    s = I.synth_const_product(bench.M_POOLS, bench.N_TOKENS, seed=3 + 100 * (k % 8))
    nu = s["prices"] * np.exp(0.01 * np.random.default_rng(k).standard_normal(bench.N_TOKENS))
    psi, arb = CO.eval_pairs(s["idx"], s["reserves"], s["gamma"], bench.N_TOKENS, nu)
    got_psi, got_arb = np.load(tmp_path / "psi.npy"), np.load(tmp_path / "arb.npy")
    assert got_psi.dtype == np.float64 and got_psi.shape == (bench.N_TOKENS,) and got_arb.shape == (1,)
    np.testing.assert_allclose(got_psi, psi, rtol=0, atol=1e-9 * np.abs(psi).max())
    assert abs(got_arb[0] - arb) <= 1e-9 * abs(arb)
