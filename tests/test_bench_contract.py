"""bench.py's output contract on CPU: the reference arm prints exactly ONE line on stdout, a JSON object with the keys the driver
reads; everything else (library chatter, progress) goes to stderr.  (The rtb200 arm needs a GPU: tests/test_gpu_*.)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, RTB_BENCH_CPU_SECONDS="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert set(d["config"]) == {"workload", "width", "height", "spp"}


def test_reference_arm_other_ranks_exit_quietly():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"))
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_steps_and_dump_arguments_are_checked(tmp_path):
    # no step count is silently replaced; the reference arm's row sample is sized by timing, so it has no reproducible output
    for extra in (["--steps", "0"], ["--impl", "reference", "--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120, cwd=tmp_path)
        assert p.returncode == 2 and p.stdout == "" and list(tmp_path.iterdir()) == [], extra


def test_dump_of_a_large_frame_is_a_fixed_sample(tmp_path):
    # the N > 1 frame (3840x2160) is over the 64 MB budget in float32: the same seeded pixel sample on every run
    import numpy as np

    import bench

    frame = np.random.default_rng(1).integers(0, 256, (2160, 3840, 3), dtype=np.uint8)
    for d in ("a", "b"):
        bench.dump_frame(str(tmp_path / d), frame)
    assert sorted(os.listdir(tmp_path / "a")) == ["frame_pixels.npy", "frame_sample.npy"]
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 << 20
    idx, px = np.load(tmp_path / "a" / "frame_pixels.npy"), np.load(tmp_path / "a" / "frame_sample.npy")
    assert idx.dtype == np.float64 and px.dtype == np.float32 and px.shape == (idx.size, 3)
    assert (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < 3840 * 2160
    assert np.array_equal(px, frame.reshape(-1, 3)[idx.astype(np.int64)])
    assert np.array_equal(idx, np.load(tmp_path / "b" / "frame_pixels.npy"))
    small = frame[:1080, :1920]
    bench.dump_frame(str(tmp_path / "c"), small)
    assert sorted(os.listdir(tmp_path / "c")) == ["frame.npy"]
    assert np.array_equal(np.load(tmp_path / "c" / "frame.npy"), small.astype(np.float32))


import pytest


@pytest.mark.gpu
def test_rtb200_arm_line_has_the_contract_keys():
    # a reduced-spp run (debug flag, invalid as a bench number) is enough to check the SHAPE of the line the driver parses
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3", "--spp", "8", "--no-configs", "--no-cpu-baseline"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "e2e", "gpu_launches", "clocks", "roofline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 3 and d["value"] > 0 and d["gpu_launches"] > 0
    assert d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    r = d["roofline"]
    assert r["bound"] == "issue" and 0 < r["frac"] < 1 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
    assert set(d["config"]) >= {"workload", "width", "height", "spp"}


@pytest.mark.gpu
def test_rtb200_arm_dumps_the_last_timed_frame(gpu_scene, tmp_path):
    # timed step i renders seed 1000 + warmup + i; the dump is the last one's RGB8 frame, untiled into scan-line order
    import numpy as np

    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--spp", "8", "--no-configs", "--no-cpu-baseline",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout)["steps"] == 2
    assert os.listdir(out) == ["frame.npy"]
    got = np.load(out / "frame.npy")
    assert got.dtype == np.float32 and got.shape == (1080, 1920, 3)
    want = gpu_scene("flying_unicorn").render(1920, 1080, 8, seed=1000 + 1 + 1)
    assert np.abs(got - want).max() <= 1
