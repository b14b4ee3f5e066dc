"""bench.py --dump-outputs: the last timed step's results as float32 .npy files, identical inputs from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out_dir, cwd, steps=2):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--batch", "2", "--steps", str(steps), "--warmup", "1", "--no-e2e",
           "--no-cpu-baseline", "--no-side", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    a, b, c = tmp_path / "a", tmp_path / "b", tmp_path / "c"
    res = run_bench(a, tmp_path)
    assert res["steps"] == 2
    files = sorted(os.listdir(a))
    assert files == sorted(["dpoints.npy", "world.npy", "sampled.npy", "vertices.npy", "sum_texture_subset.npy",
                            "softor_texture_subset.npy"])
    assert sum(os.path.getsize(a / f) for f in files) <= 64 << 20
    got = {f: np.load(a / f) for f in files}
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in got.values())
    assert got["dpoints.npy"].shape == (4096, 2) and np.abs(got["dpoints.npy"]).max() > 0
    w = got["world.npy"]
    assert w.shape[0] == 2 and w.shape[2:] == (4, 4) and got["vertices.npy"].shape == (2, 100_000, 3)
    assert got["sum_texture_subset.npy"].shape == got["softor_texture_subset.npy"].shape == (1 << 20,)
    run_bench(b, tmp_path)
    for f in files:                       # same inputs; accumulation order of the splat kernels may differ in the last bits
        ref = np.load(b / f)
        np.testing.assert_allclose(got[f], ref, rtol=1e-5, atol=1e-6 * max(float(np.abs(ref).max()), 1.0), err_msg=f)
    # one more timed step: the first timed step is the same as above, the last one randomises other scene samples
    assert run_bench(c, tmp_path, steps=3)["steps"] == 3
    assert not np.array_equal(np.load(c / "world.npy"), got["world.npy"])
    ref = np.load(c / "dpoints.npy")            # same pattern and upstream gradients: the same pattern gradient
    np.testing.assert_allclose(got["dpoints.npy"], ref, rtol=1e-5, atol=1e-6 * float(np.abs(ref).max()))
