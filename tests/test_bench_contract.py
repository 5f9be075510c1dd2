"""bench.py's contract: the reference arm (the CPU restatement of the reference on the host cores) prints one JSON line
with the agreed keys, the GPU arm fails loudly without a device instead of measuring anything else, and
--dump-outputs writes the frame of the last timed step, the same frame for the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import HAS_GPU, ROOT, get_scene


def test_reference_arm_prints_the_agreed_line():
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--config", "random_spheres", "--steps", "1", "--warmup", "3"],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "Mpaths/s" and d["unit"] == "Mpaths/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] >= 3 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["dtype"] == "f32" and "workload" in d["config"] and "random_spheres_demo 400x225" in d["config"]["workload"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == os.cpu_count() and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_runs_on_rank_zero_only():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--config", "random_spheres", "--steps", "1"],
                       capture_output=True, text=True, cwd=ROOT, timeout=300, env=env)
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith("{")]


@pytest.mark.skipif(HAS_GPU, reason="a GPU is present")
def test_gpu_arm_fails_loudly_without_a_device():
    r = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--warmup", "3", "--no-cpu-baseline"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]  # no number of any kind


def run_and_dump(out_dir, *args):
    r = subprocess.run([sys.executable, "bench.py", "--config", "random_spheres", "--dump-outputs", str(out_dir), *args],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    assert sorted(os.listdir(out_dir)) == ["frame.npy"]
    return json.loads(lines[0]), np.load(os.path.join(out_dir, "frame.npy"))


def test_reference_arm_dumps_the_same_last_frame_twice(tmp_path):
    (d1, a), (_, b) = (run_and_dump(tmp_path / run, "--impl", "reference", "--steps", "2") for run in ("a", "b"))
    assert d1["steps"] == 2
    assert a.dtype == np.float32 and a.shape == (225, 400, 3) and a.mean() > 0
    assert np.array_equal(a, b)


def test_dump_of_a_large_frame_is_a_fixed_sample_within_the_limit(tmp_path):
    import bench
    frame = np.random.default_rng(1).random((2160, 3840, 3), dtype=np.float32)  # stress_1m's frame: 99.5 MB
    bench.dump_frame(str(tmp_path), frame)
    assert sorted(os.listdir(tmp_path)) == ["frame_sample.npy", "frame_sample_pixels.npy"]
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= bench.DUMP_LIMIT
    sample, pixels = np.load(tmp_path / "frame_sample.npy"), np.load(tmp_path / "frame_sample_pixels.npy")
    assert sample.dtype == np.float32 and pixels.dtype == np.float64 and len(np.unique(pixels)) == len(sample) == 1 << 20
    assert np.array_equal(sample, frame.reshape(-1, 3)[pixels.astype(np.int64)])
    again = tmp_path / "again"
    bench.dump_frame(str(again), frame)
    assert np.array_equal(np.load(again / "frame_sample_pixels.npy"), pixels)


@pytest.mark.gpu
def test_gpu_arm_dumps_the_frame_of_its_last_timed_step(vb, ctx, tmp_path):
    flags = ("--steps", "3", "--no-cpu-baseline", "--no-other-configs")
    (d1, a), (d2, b) = (run_and_dump(tmp_path / run, *flags) for run in ("a", "b"))
    assert d1["steps"] == d2["steps"] == 3 and d1["n_gpus"] == 1
    assert a.dtype == np.float32 and a.shape == (225, 400, 3) and np.array_equal(a, b)
    scene, cam = get_scene(vb, "random_spheres_demo")
    ctx.upload(scene)
    last, _, _ = ctx.render(cam, vb.render_params(400, 225, 16, 50, seed=3))  # timed step k renders with seed k
    assert np.allclose(a, last, rtol=1e-5, atol=1e-7)
