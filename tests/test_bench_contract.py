"""CPU: the reference arm of bench.py prints exactly one JSON line with the contract's keys (the B200 arm needs a
GPU; its line is checked by tests/test_bench_gpu.py)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["impl"] == "reference" and d["metric"] == "sr_frames_per_s_4x_1080p_out" and d["unit"] == "frames/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["extrapolated"] is True and 0 < d["frame_fraction_measured"] < 1 and d["cpu_baseline"]["extrapolated"] is True
    import bench
    assert d["config"]["workload"] == bench.WORKLOAD            # both arms print the same workload string


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bad_arguments_are_refused(argv, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True,
                       timeout=120, cwd=tmp_path)
    assert r.returncode == 2 and r.stdout == "" and "error" in r.stderr
    assert not os.path.exists(tmp_path / "out")


def test_dump_frames_samples_the_same_pixels_of_every_frame_past_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    frames = torch.randint(0, 256, (3, 40, 50, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(0))
    bench.dump_frames(str(tmp_path / "all"), frames)
    assert np.array_equal(np.load(tmp_path / "all" / "frames.npy"), frames.float().numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 3 * 40 * 50 * 3 * 4 // 2)
    bench.dump_frames(str(tmp_path / "sample"), frames)
    assert sorted(os.listdir(tmp_path / "sample")) == ["frames_sample.npy", "frames_sample_pixels.npy"]
    sample, pix = np.load(tmp_path / "sample" / "frames_sample.npy"), np.load(tmp_path / "sample" / "frames_sample_pixels.npy")
    assert sample.dtype == np.float32 and pix.dtype == np.float64 and sample.nbytes + pix.nbytes <= bench.DUMP_LIMIT_BYTES
    assert sample.shape == (3, pix.size, 3) and pix.size > 0 and np.unique(pix).size == pix.size
    assert np.array_equal(sample, frames.float().numpy().reshape(3, -1, 3)[:, pix.astype(np.int64)])


@pytest.mark.gpu
def test_b200_arm_prints_one_contract_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-cpu-baseline",
                        "--no-extras", "--dump-outputs", str(tmp_path / "dump")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert (REQUIRED - {"cpu_baseline"}) <= set(d)
    assert d["gpu_launches"] > 0 and d["dtype"] == "bf16" and d["n_gpus"] == 1 and d["steps"] == 2
    import numpy as np
    assert os.listdir(tmp_path / "dump") == ["frames.npy"]
    frames = np.load(tmp_path / "dump" / "frames.npy")
    assert frames.dtype == np.float32 and frames.shape == (1, 1080, 1920, 3)
    assert np.array_equal(frames, np.round(frames)) and 0 <= frames.min() and frames.max() <= 255 and frames.std() > 1
    import bench
    assert d["config"]["workload"] == bench.WORKLOAD
    roof = d["roofline"]
    # SURVEY.md 8(d): the conv stack is bounded by the tensor cores; the HBM engineering view is a secondary key
    assert roof["bound"] == "tensor" and roof["unit"] == "TFLOP/s" and 0 < roof["frac"] <= 1.2 and roof["peak"] > 0
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-6
    assert 0 < roof["hbm_view"]["frac"] <= 1.2 and roof["hbm_view"]["unit"] == "GB/s"
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] > 0
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
