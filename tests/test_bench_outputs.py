"""bench.py --dump-outputs: what the last timed step returned, as float32 .npy files within the size cap."""
import os

import numpy as np
import torch

import bench


def _result(B, seed=0):
    g = torch.Generator().manual_seed(seed)
    return {"scale_crop": torch.rand(B, 1, generator=g), "center": torch.rand(B, 2, generator=g),
            "keypoint_coord3d": torch.rand(B, 21, 3, generator=g),
            "keypoints_uv": torch.randint(0, 320, (B, 21, 2), dtype=torch.int32, generator=g), "hand_scoremap": None}


def test_dump_writes_every_returned_array_as_float32(tmp_path):
    r = _result(32)
    bench.dump_outputs(str(tmp_path), r)
    assert sorted(os.listdir(tmp_path)) == ["center.npy", "keypoint_coord3d.npy", "keypoints_uv.npy", "scale_crop.npy"]
    for k in ("scale_crop", "center", "keypoint_coord3d", "keypoints_uv"):
        a = np.load(tmp_path / (k + ".npy"))
        assert a.dtype == np.float32
        np.testing.assert_array_equal(a, r[k].numpy())


def test_dump_above_the_cap_keeps_one_seeded_sample_of_images(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 2 << 20)
    r = _result(8192)                                   # 432 B per image: 3.4 MB
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), r)
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= 2 << 20
    rows = np.load(tmp_path / "a" / "sample_rows.npy")
    assert rows.dtype == np.float64 and 0 < len(rows) < 8192 and np.all(np.diff(rows) > 0)
    np.testing.assert_array_equal(rows, np.load(tmp_path / "b" / "sample_rows.npy"))
    idx = rows.astype(np.int64)
    for k in ("center", "keypoint_coord3d", "keypoints_uv"):
        np.testing.assert_array_equal(np.load(tmp_path / "a" / (k + ".npy")), r[k].numpy()[idx])
