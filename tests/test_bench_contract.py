"""bench.py contract checks: the reference arm prints exactly one JSON line with the documented keys (stdout is
machine-read), the CLI exposes the documented switches, and (GPU) --dump-outputs writes what the timed path computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "dsa_inputs_prioritized_per_sec" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_cli_switches():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--workload", "--shard", "--no-cpu", "--dump-outputs"):
        assert flag in out.stdout, flag


@pytest.mark.gpu
def test_dump_outputs_are_the_dsa_results_of_the_c2_inputs(tmp_path):
    """--dump-outputs: after K timed steps the C2 results a DSA caller receives, one float64 entry per test input in
    input order, equal bit for bit to the C oracle on sampled inputs."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-c5",
                          "--no-others", "--no-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                         timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2, lines
    import bench
    from oracle import c_oracle, np_oracle

    names = ("dist_a", "dist_b", "dsa", "winner_index")
    assert sorted(os.listdir(tmp_path)) == [f"{n}.npy" for n in names]
    got = {n: np.load(os.path.join(tmp_path, f"{n}.npy")) for n in names}
    xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(**bench.C2)
    for v in got.values():
        assert v.dtype == np.float64 and v.shape == (xte.shape[0],)
    assert sum(v.nbytes for v in got.values()) <= 64 << 20
    sel = np.sort(np.random.default_rng(0).choice(xte.shape[0], 64, replace=False))
    want = c_oracle.dsa(xtr, ytr, xte[sel], pte[sel])
    assert np.array_equal(got["dist_a"][sel], want["dist_a"]) and np.array_equal(got["dist_b"][sel], want["dist_b"])
    assert np.array_equal(got["winner_index"][sel], want["idx_a"]) and np.array_equal(got["dsa"][sel], want["dsa"])
