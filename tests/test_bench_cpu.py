"""bench.py contract on CPU: the reference arm (`--impl reference`) runs without a GPU (it times the oracle port) and
prints ONE JSON line with the contract's keys; the product arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--meshlets", "20000", "--width", "640",
                          "--height", "360", "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "meshlet_instances_culled_per_s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and d["vs_baseline"] is None and "workload" in d["config"]


def test_reference_arm_dumps_the_last_timed_frame(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--meshlets", "20000", "--width", "640",
                          "--height", "360", "--steps", "3", "--warmup", "1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 3
    assert sorted(os.listdir(tmp_path)) == ["counters.npy", "depth.npy", "vis32.npy", "visible_meshlet_instances.npy"]
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert got["vis32"].dtype == np.float64 and got["depth"].dtype == np.float32 and got["vis32"].shape == got["depth"].shape == (360, 640)
    assert got["visible_meshlet_instances"].dtype == np.float64 and got["counters"].dtype == np.float64
    total, early, late, triangles = got["counters"]
    ids = got["visible_meshlet_instances"]
    assert len(ids) == early + late > 0 and total >= len(ids) and triangles > 0
    assert np.all(np.diff(ids) > 0) and ids[-1] < total  # sorted, distinct meshlet-instance indices
    assert (got["vis32"] != 0xFFFFFFFF).any() and np.all(got["vis32"] == np.floor(got["vis32"]))
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True,
                         text=True, timeout=120)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                         text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_product_arm_needs_a_gpu():
    try:
        import torch

        if torch.cuda.is_available():
            return
    except Exception:
        pass
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
