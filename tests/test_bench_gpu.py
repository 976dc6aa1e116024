"""bench.py on the GPU at a reduced size: --dump-outputs writes the film and ray counts of the last timed step, the same
arguments give the same outputs, --steps sets the number of timed steps, and nothing is written into the tree."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

SMALL = ["--gpus", "1", "--warmup", "3", "--xres", "96", "--yres", "54", "--spp", "4", "--no-cpu-baseline"]


def tree_files():
    return sorted((os.path.join(d, f), os.path.getsize(os.path.join(d, f))) for d, dirs, files in os.walk(ROOT)
                  for f in files if "__pycache__" not in d and ".pytest_cache" not in d)


def run_bench(*args):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + SMALL + list(args), stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, res.stdout
    return json.loads(lines[0])


def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    before = tree_files()
    a = run_bench("--tris", "20000", "--steps", "2", "--dump-outputs", str(tmp_path / "a"))
    b = run_bench("--tris", "20000", "--steps", "5", "--dump-outputs", str(tmp_path / "b"))
    k = run_bench("--workload", "killeroo", "--spp", "2", "--steps", "1", "--dump-outputs", str(tmp_path / "k"))
    assert tree_files() == before, "bench.py must not write into the tree"
    assert (a["steps"], b["steps"], k["steps"]) == (2, 5, 1)
    for d in ("a", "b", "k"):
        assert sorted(os.listdir(tmp_path / d)) == ["film.npy", "ray_counts.npy"]
    fa, fb, fk = (np.load(tmp_path / d / "film.npy") for d in ("a", "b", "k"))
    ca, cb, ck = (np.load(tmp_path / d / "ray_counts.npy") for d in ("a", "b", "k"))
    assert fa.dtype == np.float32 and fa.shape == (54, 96, 4) and ca.dtype == np.float64
    n = 96 * 54 * 4
    # one frame's samples (every step clears the film), not a sum over the steps
    assert n <= fa[..., 3].sum() <= 1.02 * n and ca[0] == n and ca[1] > 0
    assert np.array_equal(fa[..., 3], fb[..., 3]) and np.allclose(fa, fb, rtol=1e-5, atol=1e-5) and np.array_equal(ca, cb)
    assert fk.shape == (54, 96, 4) and ck[0] == 96 * 54 * 2 and fk[..., :3].sum() > 0
