"""bench.py --dump-outputs: what the timed path computed in its last step, written so that two builds can be compared output for
output (whole frame when small, the same seeded pixel sample on every run when large, at most 64 MB in all)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def _sizes(d):
    return {f: os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_of_a_large_frame_is_a_fixed_sample(tmp_path):
    import torch
    ny, nx = 2160, 3840
    fb = torch.arange(ny * nx * 3, dtype=torch.float32).reshape(ny, nx, 3)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), fb, 7.0, 9.0)
    a, b = tmp_path / "a", tmp_path / "b"
    assert sorted(_sizes(a)) == ["frame_sample.npy", "frame_sample_pixels.npy", "ray_counts.npy"]
    assert sum(_sizes(a).values()) <= 64 << 20
    for f in _sizes(a):
        assert np.array_equal(np.load(a / f), np.load(b / f)), f
    pix, sample = np.load(a / "frame_sample_pixels.npy"), np.load(a / "frame_sample.npy")
    assert pix.dtype == np.float64 and sample.dtype == np.float32 and sample.shape == (bench.DUMP_SAMPLE_PIXELS, 3)
    assert np.array_equal(sample, fb.reshape(-1, 3).numpy()[pix.astype(np.int64)])
    assert np.load(a / "ray_counts.npy").tolist() == [7.0, 9.0]


def test_dump_of_a_small_frame_is_the_frame(tmp_path):
    import torch
    fb = torch.rand((800, 1200, 3), generator=torch.Generator().manual_seed(1))
    bench.dump_outputs(str(tmp_path), fb, 1.0, 2.0)
    assert sorted(_sizes(tmp_path)) == ["frame.npy", "ray_counts.npy"]
    assert np.array_equal(np.load(tmp_path / "frame.npy"), fb.numpy())


@pytest.mark.gpu
def test_bench_dumps_the_frame_of_its_last_step(pkg, golden_dir, tmp_path):
    """BASELINE config 2 through bench.py: the dumped frame is the reference CUDA build's 8-bit image, every sample traced."""
    out = tmp_path / "dump"
    subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--config", "C2",
                    "--no-cpu-baseline", "--dump-outputs", str(out)], check=True, stdout=subprocess.DEVNULL, cwd=str(tmp_path))
    frame = np.load(out / "frame.npy")
    gold = np.load(os.path.join(golden_dir, "ref_cuda", "C2_1200x800x10_u8.npz"))["rgb"]
    assert frame.dtype == np.float32 and np.array_equal(pkg.quantise(frame), gold)
    rays, paths = np.load(out / "ray_counts.npy")
    assert paths == 1200 * 800 * 10 and rays >= paths
