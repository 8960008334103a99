"""bench.py --dump-outputs: the file format, without a GPU (the arrays are built here in the layout the device path returns)."""
import os

import numpy as np

import bench


def _dets(nf, cap, seed):
    rng = np.random.default_rng(seed)
    d = rng.integers(0, 2000, size=(nf, cap, 4), dtype=np.int32)
    d[..., 3] = rng.uniform(-5.0, 20.0, size=(nf, cap)).astype(np.float32).view(np.int32)
    return d, rng.integers(0, cap + 3, size=nf, dtype=np.int32)


def test_dump_writes_float32_slots_up_to_the_count(tmp_path):
    d, c = _dets(5, 8, 0)
    c[:] = [0, 3, 8, 11, 1]                      # 11 > cap: the frame's count is kept, every slot is filled
    bench.dump_outputs(str(tmp_path), d, c)
    assert sorted(os.listdir(tmp_path)) == ["counts.npy", "detections.npy", "frame_index.npy"]
    det = np.load(tmp_path / "detections.npy")
    assert det.dtype == np.float32 and det.shape == (5, 8, 4)
    assert np.array_equal(np.load(tmp_path / "counts.npy"), c.astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "frame_index.npy"), np.arange(5, dtype=np.float32))
    for f, n in enumerate(np.minimum(c, 8)):
        assert np.array_equal(det[f, :n, :3], d[f, :n, :3].astype(np.float32))
        assert det[f, :n, 3].tobytes() == d[f, :n, 3].tobytes()          # the score's float32 bits, unchanged
        assert not det[f, n:].any()


def test_dump_samples_a_fixed_set_of_frames_above_the_size_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 10 * (16 * 16 + 8))
    d, c = _dets(40, 16, 1)
    bench.dump_outputs(str(tmp_path / "a"), d, c)
    bench.dump_outputs(str(tmp_path / "b"), d, c)
    idx = np.load(tmp_path / "a" / "frame_index.npy").astype(np.int64)
    assert len(idx) == 10 and len(set(idx)) == 10 and (np.diff(idx) > 0).all()
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in os.listdir(tmp_path / "a")) <= 10 * (16 * 16 + 8) + 3 * 128   # + .npy headers
    for name in ("counts", "detections", "frame_index"):
        assert np.load(tmp_path / "a" / f"{name}.npy").tobytes() == np.load(tmp_path / "b" / f"{name}.npy").tobytes()
    assert np.array_equal(np.load(tmp_path / "a" / "counts.npy"), c[idx].astype(np.float32))
