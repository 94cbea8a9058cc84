"""bench.py --dump-outputs: file names and dtypes, the whole frame when it is small, and a fixed pixel sample within
64 MiB when it is not."""
import os

import numpy as np

import bench


def _frame(h, w):
    return (np.arange(h * w * 3, dtype=np.float64) * 0.5).astype(np.float32).reshape(h, w, 3)


def test_small_frame_is_written_whole(tmp_path):
    img = _frame(48, 64)
    counts = np.array([3, 7], np.int32)
    bench.dump_outputs(str(tmp_path), {"counts": counts, "pos": np.ones(4, np.float32)}, img)
    assert sorted(os.listdir(tmp_path)) == ["counts.npy", "image.npy", "pos.npy"]
    got = np.load(tmp_path / "image.npy")
    assert got.dtype == np.float32 and np.array_equal(got, img)
    c = np.load(tmp_path / "counts.npy")
    assert c.dtype == np.float64 and np.array_equal(c, counts)
    assert np.load(tmp_path / "pos.npy").dtype == np.float32


def test_large_frame_is_a_fixed_sample_within_64_mib(tmp_path):
    h, w = 1440, 1500  # more pixels than bench.DUMP_PIXELS
    img = _frame(h, w)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {}, img)
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= 64 << 20
    idx = np.load(tmp_path / "a" / "image_pixels.npy")
    assert idx.dtype == np.float64 and idx.shape == (bench.DUMP_PIXELS,) and np.all(np.diff(idx) > 0)
    got = np.load(tmp_path / "a" / "image.npy")
    assert np.array_equal(got, img.reshape(-1, 3)[idx.astype(np.int64)])
    for f in ("image.npy", "image_pixels.npy"):
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes()
