"""GPU parity of the dataset readers' forward generators (SURVEY.md 8(f) row 4) -- h3d_rhd_reader_items, h3d_stb_reader_items,
h3d_gaussian_scoremap, h3d_canonical_trafo and the BinaryDbReader / BinaryDbReaderSTB mirrors -- against the CPU oracle
(oracle/reader_oracle.py) and against the vectors produced by the reference's unmodified reader classes
(tests/golden/golden_reference_reader.npz).  Selection logic and integer items exact; float items 1e-6 (device expf / atanf vs
numpy: a few ulp)."""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import synth_records as SR  # noqa: E402
from make_golden_reference_reader import sub_step  # noqa: E402
from oracle import reader_oracle as R  # noqa: E402

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(HERE, "golden", "golden_reference_reader.npz"))
BIG = ("image", "image_crop", "scoremap", "hand_parts", "hand_mask")


def _np(t):
    return t.detach().cpu().numpy()


def _check(d, ref, keys, i, atol=2e-6):
    for k in keys:
        v, r = _np(d[k])[i], np.asarray(ref[k])
        if r.dtype == bool or np.issubdtype(r.dtype, np.integer):
            np.testing.assert_array_equal(v.astype(r.dtype), r, err_msg=k)
        else:
            np.testing.assert_allclose(v, r, atol=atol, rtol=2e-6, err_msg=k)


def _write(tmp_path, name, recs):
    p = tmp_path / name
    p.write_bytes(b"".join(recs))
    return str(p)


RHD_KEYS = ["keypoint_xyz", "keypoint_uv", "keypoint_vis", "hand_side", "keypoint_xyz21", "keypoint_scale", "keypoint_xyz21_normed", "keypoint_vis21",
            "keypoint_uv21", "cam_mat", "image", "hand_parts", "hand_mask", "scoremap"]


@pytest.mark.parametrize("cfg", ["rhd_crop", "rhd_full", "rhd_scaled"])
def test_rhd_reader_mirror(tmp_path, cfg):
    from hand3d_b200.data.BinaryDbReader import BinaryDbReader
    recs = SR.rhd_records(4)
    kw = {"rhd_crop": dict(hand_crop=True, use_wrist_coord=False), "rhd_full": dict(use_wrist_coord=False),
          "rhd_scaled": dict(use_wrist_coord=True, scale_to_size=True)}[cfg]
    rd = BinaryDbReader(mode="evaluation", shuffle=False, batch_size=4, path_to_db=_write(tmp_path, "rhd.bin", recs), **kw)
    d = rd.get()
    torch.cuda.synchronize()
    for i in range(4):
        ref = R.rhd_items(recs[i], **kw)
        keys = [k for k in ref if k in d and k not in ("keypoint_xyz21_local", "keypoint_xyz21_can", "rot_mat")]
        assert set(keys) >= (set(RHD_KEYS) & set(ref)), (sorted(ref), sorted(d))
        _check(d, ref, keys, i)
        if "rot_mat" in ref:     # canonical frame: atanf / sinf / cosf chains on device
            np.testing.assert_allclose(_np(d["keypoint_xyz21_can"])[i], ref["keypoint_xyz21_can"], atol=2e-5)
            np.testing.assert_allclose(_np(d["rot_mat"])[i], ref["rot_mat"], atol=2e-5)
        if cfg == "rhd_crop":
            np.testing.assert_array_equal(_np(d["image_crop"])[i], ref["image_crop"])          # crop: bit-exact given centre / scale
            np.testing.assert_array_equal(_np(d["crop_scale"])[i], ref["crop_scale"])
        # ... and against the reference-generated vectors directly
        pre = "%s/%d" % (cfg, i)
        for k in ("hand_side", "keypoint_xyz21", "keypoint_uv21", "keypoint_vis21", "keypoint_scale", "crop_scale"):
            if pre + "/" + k in G.files:
                np.testing.assert_allclose(_np(d[k])[i].astype(np.float64), G[pre + "/" + k].astype(np.float64), atol=2e-6, rtol=2e-6, err_msg=k)
        if pre + "/scoremap/shape" in G.files:
            sm = _np(d["scoremap"])[i]
            s = sub_step("scoremap")
            np.testing.assert_allclose(sm[::s, ::s], G["%s/scoremap/sub%d" % (pre, s)], atol=2e-6)
            np.testing.assert_allclose(sm.astype(np.float64).sum(), G[pre + "/scoremap/sums"][0], rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("wrist", [False, True])
def test_stb_reader_mirror(tmp_path, wrist):
    from hand3d_b200.data.BinaryDbReader import BinaryDbReaderSTB
    recs = SR.stb_records(2)
    rd = BinaryDbReaderSTB(mode="evaluation", shuffle=False, batch_size=2, use_wrist_coord=wrist, path_to_db=_write(tmp_path, "stb.bin", recs),
                           with_scoremap=True)
    d = rd.get()
    torch.cuda.synchronize()
    for i in range(2):
        ref = R.stb_items(recs[i], use_wrist_coord=wrist)
        _check(d, ref, ["keypoint_xyz21", "keypoint_vis21", "keypoint_uv21", "image", "cam_mat", "hand_side", "keypoint_scale", "keypoint_xyz21_normed",
                        "scoremap"], i)
        np.testing.assert_allclose(_np(d["keypoint_xyz21_can"])[i], ref["keypoint_xyz21_can"], atol=2e-5)
        np.testing.assert_allclose(_np(d["rot_mat"])[i], ref["rot_mat"], atol=2e-5)
        pre = "stb_%s/%d" % ("wrist" if wrist else "palm", i)
        np.testing.assert_allclose(_np(d["keypoint_xyz21"])[i], G[pre + "/keypoint_xyz21"], atol=1e-7)
        np.testing.assert_array_equal(_np(d["keypoint_vis21"])[i], G[pre + "/keypoint_vis21"])


def test_gaussian_scoremap_edges():
    """key-points on the border rows / columns and invalid ones contribute nothing; coordinates are truncated toward zero"""
    from hand3d_b200 import runtime
    ctx = runtime.default_context()
    hw = np.array([[[0.9, 10.0], [1.0, 1.0], [254.99, 254.2], [255.0, 100.0], [100.7, -0.5], [128.5, 64.25], [30.0, 255.0]]], np.float32)
    valid = np.array([[1, 1, 1, 1, 1, 0, 1]], np.uint8)
    hw = np.concatenate([hw, hw[:, :1].repeat(1, 1)], 1)[:, :8]          # N = 8 (W * N multiple of 4)
    valid = np.concatenate([valid, valid[:, :1]], 1)
    out = _np(ctx.gaussian_scoremap(torch.from_numpy(hw).cuda(), (256, 256), 25.0, torch.from_numpy(valid).cuda()))[0]
    ref = R.create_multiple_gaussian_map(hw[0], (256, 256), 25.0, valid[0])
    np.testing.assert_allclose(out, ref, atol=2e-6)
    assert out[..., 0].max() == 0 and out[..., 3].max() == 0 and out[..., 4].max() == 0 and out[..., 5].max() == 0 and out[..., 6].max() == 0
    assert out[1, 1, 1] == 1.0 and out[254, 254, 2] == 1.0


def test_canonical_trafo_random():
    from hand3d_b200 import runtime
    ctx = runtime.default_context()
    rng = np.random.default_rng(5)
    xyz = rng.normal(size=(16, 21, 3)).astype(np.float32)
    right = (rng.uniform(size=16) > 0.5)
    can, rot, inv = ctx.canonical_trafo(torch.from_numpy(xyz).cuda(), torch.from_numpy(right).cuda())
    for b in range(16):
        c, r = R.canonical_trafo(xyz[b])
        np.testing.assert_allclose(_np(can)[b], R.flip_right_hand(c, right[b]), atol=3e-5)
        np.testing.assert_allclose(_np(rot)[b], r, atol=3e-5)
        np.testing.assert_allclose(_np(inv)[b] @ _np(rot)[b], np.eye(3), atol=3e-6)
    # the defining properties (utils/canonical_trafo.py:97-136): root at the origin, key-point 12 on the +y axis, key-point 20 in the z = 0 plane with x > 0
    c = _np(can)
    assert np.abs(c[:, 0]).max() < 1e-6 and np.abs(c[:, 12, [0, 2]]).max() < 1e-5 and np.abs(c[:, 20, 2]).max() < 1e-5
