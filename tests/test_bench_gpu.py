"""bench.py --dump-outputs on the GPU: the files hold the last timed frame, equal to what the CPU reference arm computes for
the same arguments (both arms bring the visibility mask to the same steady state before the frame they dump)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--meshlets", "20000", "--width", "640", "--height", "360", "--steps", "3", "--warmup", "4"]


def _bench(out_dir, *extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + ARGS + list(extra) + ["--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(out_dir / f) for f in os.listdir(out_dir)}


def test_dump_outputs_equal_the_reference_arm(tmp_path):
    d, got = _bench(tmp_path / "ours", "--no-e2e", "--no-cpu")
    _, want = _bench(tmp_path / "reference", "--impl", "reference")
    assert d["steps"] == 3
    pf = d["per_frame"]
    np.testing.assert_array_equal(got["counters"], [pf["meshlet_instances"], pf["early_survivors"], pf["late_survivors"],
                                                    pf["triangles_rasterised"]])
    assert sorted(got) == sorted(want)
    for name in ("vis32", "visible_meshlet_instances", "counters"):
        assert got[name].dtype == want[name].dtype == np.float64
        np.testing.assert_array_equal(got[name], want[name], err_msg=name)
    assert got["depth"].dtype == want["depth"].dtype == np.float32
    np.testing.assert_array_equal(got["depth"].view(np.uint32), want["depth"].view(np.uint32))
