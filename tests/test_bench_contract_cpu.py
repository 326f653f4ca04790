"""CPU test of bench.py's reference arm (the one leg of the bench that needs no GPU): it runs, prints ONE JSON
line with the contract's keys, and its `config` object is exactly the one the B200 arm prints for the same
workload and N (the driver compares the two)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line(built):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "shaded_gpixels_per_s" and d["unit"] == "Gpixels/s"
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["cpu"]
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.make_config("views1080_tex", bench.WORKLOADS["views1080_tex"]["views"], 1)
    assert "configs[4]" in d["config"]["workload"] and d["config"]["views_per_step_per_gpu"] == 512


def test_other_ranks_of_the_reference_arm_exit_quietly(built):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_raster_stage_split_labels():
    """roofline.raster_kernels_ms_per_step names the kernels the stage really ran: the one-kernel opaque stage,
    the visibility + resolve pair, or the one raster kernel of a pass with blended primitives."""
    sys.path.insert(0, ROOT)
    import bench
    assert bench.kernel_split((4.0, 0.0), 2, 2, True) == {"raster_opaque_kernel<true>": 2.0}
    assert bench.kernel_split((4.0, 2.0), 2, 1, True) == {"raster_opaque_kernel<false>": 2.0, "resolve_kernel": 1.0}
    assert bench.kernel_split((4.0, 0.0), 2, 0, True) == {"raster_tex_kernel": 2.0}
    assert bench.kernel_split((4.0, 0.0), 0, 0, False) == {"raster_kernel": 4.0}
    assert bench.stage_label(2, True).startswith("raster_opaque_kernel<true>") and bench.stage_label(0, False) == "raster_kernel"


@pytest.mark.parametrize("n_frames,w,h", [(512, 1920, 1080), (1000, 64, 48), (1, 3840, 2160)])
def test_dump_outputs_is_a_fixed_bounded_sample(tmp_path, n_frames, w, h):
    """--dump-outputs: float32 files under 64 MB in all, the same sample on every run, and every sampled value is
    the pixel it claims to be (frame f's pixel i holds colour f * w * h + i and depth i, so both can be decoded)."""
    sys.path.insert(0, ROOT)
    import bench
    idx = np.arange(w * h, dtype=np.uint32).reshape(h, w)

    def read_frame(f):
        return idx + np.uint32(f * w * h), idx.astype(np.float32)

    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), "wl", read_frame, n_frames, w, h)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["wl_color_crop.npy", "wl_color_sample.npy", "wl_depth_crop.npy", "wl_depth_sample.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    out = {}
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float32 and np.array_equal(a, b)
        out[n[3:-4]] = a
    col = out["color_sample"].astype(np.uint8).view(np.uint32)[..., 0].astype(np.int64)
    frames, pix = np.divmod(col, w * h)
    assert np.array_equal(pix, out["depth_sample"].astype(np.int64))
    assert np.all(pix == pix[0]) and np.all(np.diff(pix[0]) > 0)  # the same pixels of every frame
    assert np.all(frames == frames[:, :1]) and np.all(np.diff(frames[:, 0]) > 0) and frames[-1, 0] < n_frames
    assert len(frames) == min(n_frames, bench.DUMP_FRAMES)
    crop = out["color_crop"].astype(np.uint8).view(np.uint32)[..., 0].astype(np.int64)
    assert crop.shape == (min(h, bench.DUMP_CROP), min(w, bench.DUMP_CROP))
    assert np.all(crop // (w * h) == frames[-1, 0]) and np.array_equal(crop % (w * h), out["depth_crop"].astype(np.int64))


def test_gpu_arm_fails_loudly_without_a_device(built):
    """No CPU fallback: on a box without a GPU the B200 arm must not print a line."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu-baseline",
                          "--no-others"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0
    assert not [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
