"""bench.py's contract: the reference arm (`--impl reference`: the CPU port of the path on the host cores, one JSON line
with the base keys, `impl`, `cpu_baseline`, `e2e`), the refusal to run the product arm without a CUDA device (no CPU
fallback), argument checks, and (gpu) `--dump-outputs`: the keys of the last timed step as .npy files."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line(oracle_b):
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0"], cwd=ROOT,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "placements/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "C2" in d["config"]["workload"]


def test_reference_arm_other_ranks_exit_quietly(oracle_b):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], cwd=ROOT,
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_product_arm_needs_a_gpu():
    # every device hidden, so the refusal is checked on a machine with a GPU too
    out = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--warmup", "3"], cwd=ROOT, capture_output=True, text=True,
                         timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode != 0 and "no CPU path" in (out.stderr + out.stdout)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]])
def test_bad_arguments_are_refused(argv):
    out = subprocess.run([sys.executable, "bench.py"] + argv, cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and out.stdout == "" and "error:" in out.stderr
    assert not os.path.exists(os.path.join(ROOT, "unused"))


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_keys(tmp_path, oracle_b):
    """--dump-outputs holds the keys of the timed steps (same digest as the JSON line), unpacked losslessly, and they are
    the oracle's answer; --steps sets the number of timed steps."""
    from kubegpu_b200 import synth
    out = subprocess.run([sys.executable, "bench.py", "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-variants",
                          "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2
    f = {n: np.load(tmp_path / (n + ".npy")) for n in ("cost", "node_id", "gpu_mask")}
    assert all(a.dtype == np.float64 and a.shape == (d["config"]["pods"],) for a in f.values())
    keys = (f["cost"].astype(np.uint64) << np.uint64(40)) | (f["node_id"].astype(np.uint64) << np.uint64(8)) | f["gpu_mask"].astype(np.uint64)
    assert hashlib.sha256(keys.tobytes()).hexdigest()[:12] == d["keys_sha256_12"]
    topo, free, pods = synth.gen_c2(d["config"]["nodes"], d["config"]["pods"])
    S = 256
    assert (keys[:S] == oracle_b.score_batch(topo, free, pods[:S], fast=True, nthreads=8)).all()
