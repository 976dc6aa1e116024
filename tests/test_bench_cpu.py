"""bench.py's reference arm (--impl reference) runs on the host alone: its JSON line is checked here at a reduced size."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def test_reference_arm_prints_the_contract_line():
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3",
           "--tris", "20000", "--xres", "96", "--yres", "54", "--spp", "4", "--ref-seconds", "0.3"]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300, cwd=ROOT)
    assert res.returncode == 0, res.stderr
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "Msamples/sec" and d["unit"] == "Msamples/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] >= 3 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic" and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_dump_of_a_film_beyond_the_limit_is_a_seeded_sample(tmp_path):
    """--dump-outputs stays within 64 MB: a larger film is written as a fixed sample of its pixels plus their indices."""
    import numpy as np

    import bench
    from pbrt_v3_b200 import Stats
    h, w = 2400, 2000                                            # 76.8 MB of rgbw
    film = np.arange(h * w * 4, dtype=np.float32).reshape(h, w, 4)
    st = Stats(camera_rays=h * w, regular_rays=7, shadow_rays=3)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), film, st)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["film.npy", "film_pixel_index.npy", "ray_counts.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    sample, index = np.load(tmp_path / "a" / "film.npy"), np.load(tmp_path / "a" / "film_pixel_index.npy")
    assert sample.dtype == np.float32 and index.dtype == np.float64 and len(sample) == len(index) > 1000000
    assert (np.diff(index) > 0).all() and np.array_equal(sample, film.reshape(-1, 4)[index.astype(np.int64)])
    assert np.array_equal(index, np.load(tmp_path / "b" / "film_pixel_index.npy"))
    assert np.load(tmp_path / "a" / "ray_counts.npy").tolist() == [h * w, 7, 3]


def test_reference_arm_under_torchrun_prints_once():
    """Launched like the driver launches N > 1: rank 0 alone runs the reference and prints; the other ranks exit 0."""
    import socket
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
           "--warmup", "3", "--tris", "20000", "--xres", "96", "--yres", "54", "--spp", "4", "--ref-seconds", "0.3"]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0
