"""bench.py's JSON contract, checked on the CPU through the reference arm (the oracle port on a tiny crop)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tree_files():
    return {os.path.join(d, f) for d, dirs, files in os.walk(ROOT) if ".git" not in d.split(os.sep) for f in dirs + files}


def test_reference_arm_prints_one_contract_line(mm, oracle):
    before = _tree_files()
    env = {k: v for k, v in os.environ.items() if k != "PYTHONDONTWRITEBYTECODE"}
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-crop", "512"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr
    # the tree may be read-only: the native oracle build goes to a temporary directory, no bytecode caches
    assert sorted(_tree_files() - before) == []
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"].startswith("Mrays/s") and d["config"]["workload"].startswith("32x32 Kruskal maze")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "f32"


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                         text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_keeps_small_frames_whole_and_samples_large_ones(tmp_path, monkeypatch):
    """--dump-outputs: float32 .npy files within the byte budget; a frame over it becomes the same seeded pixel sample on
    every run, with the pixels' flat indices beside it."""
    sys.path.insert(0, ROOT)
    import bench

    small = np.arange(6 * 5 * 4, dtype=np.float64).reshape(6, 5, 4)
    bench.dump_outputs(str(tmp_path / "small"), {"frame": small})
    got = np.load(tmp_path / "small" / "frame.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small)
    monkeypatch.setattr(bench, "DUMP_BYTES", 40_000)
    big = np.random.default_rng(1).random((64, 64, 4), dtype=np.float32)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"frame": big})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["frame.npy", "frame_index.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 40_000
    px, idx = np.load(tmp_path / "a" / "frame.npy"), np.load(tmp_path / "a" / "frame_index.npy")
    assert px.dtype == np.float32 and idx.dtype == np.float64 and len(px) == len(idx) > 1000
    assert np.array_equal(px, big.reshape(-1, 4)[idx.astype(np.int64)])
    for f in files:
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes()


def _bench(args, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--no-cpu-baseline", "--no-extras",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_frame(mm, noise, scenes, tmp_path):
    """--steps sets the timed steps and --dump-outputs writes what the last one computed: timed step i renders the frame
    at time warmup + i, so the dump equals a fresh render at time warmup + steps - 1."""
    d = _bench(["--steps", "3", "--warmup", "2", "--width", "128", "--height", "64"], tmp_path / "cfg2")
    assert d["steps"] == 3 and d["warmup"] == 2
    r = mm.Renderer(0)
    r.upload_scene(scenes(32), noise)
    u = mm.default_uniform(32, 128, 64, 4, time=2 + 3 - 1)
    want = r.render(u, mm.full_frame_params(u, spp=16, bounce_limit=8), mm.gen_chunks(128, 64, 4))[0]
    r.close()
    assert np.load(tmp_path / "cfg2" / "frame.npy").tobytes() == want.tobytes()
    # fly-throughs: a step is a frame; the dump is the last frame read back
    d = _bench(["--workload", "cfg5", "--steps", "3", "--warmup", "1", "--width", "64", "--height", "64"], tmp_path / "cfg5")
    assert d["steps"] == 3 and d["warmup"] == 1 and d["gpu_launches"] == 6
    frame = np.load(tmp_path / "cfg5" / "frame.npy")
    assert frame.shape == (64, 64, 4) and frame.dtype == np.float32 and (frame[..., 3] == 1).all() and frame[..., :3].max() > 0
