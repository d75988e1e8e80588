"""oracle/reader_oracle.py (restatement of the dataset readers' derived items, SURVEY.md 8(f) row 4) against vectors produced by
the reference's UNMODIFIED reader classes (tests/golden/make_golden_reference_reader.py): exact for the integer / selection logic,
1e-6 for the float arithmetic (numpy float32 on both sides; the stand-in evaluates op by op like TF)."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import synth_records as SR  # noqa: E402
from make_golden_reference_reader import sub_step  # noqa: E402
from oracle import reader_oracle as R  # noqa: E402

G = np.load(os.path.join(HERE, "golden", "golden_reference_reader.npz"))
BIG = ("image", "image_crop", "scoremap", "hand_parts", "hand_mask")


def golden_items(prefix):
    names = sorted({k[len(prefix) + 1:].split("/")[0] for k in G.files if k.startswith(prefix + "/")})
    return names


def check(prefix, d, atol=1e-6):
    names = golden_items(prefix)
    assert names, prefix
    for k in names:
        assert k in d, "oracle does not produce %s" % k
        v = np.asarray(d[k])
        if k in BIG:
            assert list(v.shape) == list(G["%s/%s/shape" % (prefix, k)]), k
            s = sub_step(k)
            np.testing.assert_allclose(v[::s, ::s], G["%s/%s/sub%d" % (prefix, k, s)], atol=atol, rtol=0, err_msg=k)
            sums = np.array([v.astype(np.float64).sum(), np.square(v.astype(np.float64)).sum()])
            np.testing.assert_allclose(sums, G["%s/%s/sums" % (prefix, k)], rtol=1e-7, atol=1e-6, err_msg=k)
        else:
            g = G["%s/%s" % (prefix, k)]
            assert v.shape == g.shape, (k, v.shape, g.shape)
            if g.dtype == bool or np.issubdtype(g.dtype, np.integer):
                np.testing.assert_array_equal(v, g, err_msg=k)
            else:
                np.testing.assert_allclose(v, g, atol=atol, rtol=1e-6, err_msg=k)
    return names


@pytest.mark.parametrize("i", range(4))
def test_rhd_reader_hand_crop(i):
    """eval3d.py:50 / eval2d_gt_cropped.py:37 configuration: palm coordinates, dominant hand, GT crop, score-map targets."""
    names = check("rhd_crop/%d" % i, R.rhd_items(SR.rhd_records(4)[i], use_wrist_coord=False, hand_crop=True))
    assert {"scoremap", "image_crop", "crop_scale", "hand_side", "keypoint_xyz21", "keypoint_scale", "keypoint_uv21", "cam_mat",
            "keypoint_xyz21_can", "rot_mat", "keypoint_xyz21_local"} <= set(names)


@pytest.mark.parametrize("i", range(4))
def test_rhd_reader_full_image(i):
    check("rhd_full/%d" % i, R.rhd_items(SR.rhd_records(4)[i], use_wrist_coord=False, hand_crop=False))


@pytest.mark.parametrize("i", range(4))
def test_rhd_reader_scale_to_size(i):
    """eval2d.py:43: wrist coordinates, image and key-points scaled to 240 x 320; everything else dropped."""
    names = check("rhd_scaled/%d" % i, R.rhd_items(SR.rhd_records(4)[i], use_wrist_coord=True, scale_to_size=True))
    assert sorted(names) == ["image", "keypoint_uv21", "keypoint_vis21"]


@pytest.mark.parametrize("i", range(2))
@pytest.mark.parametrize("wrist", [False, True])
def test_stb_reader(i, wrist):
    check("stb_%s/%d" % ("wrist" if wrist else "palm", i), R.stb_items(SR.stb_records(2)[i], use_wrist_coord=wrist))


def test_records_cover_the_branches():
    sides = [tuple(G["rhd_crop/%d/hand_side" % i]) for i in range(4)]
    assert (1.0, 0.0) in sides and (0.0, 1.0) in sides                        # left- and right-dominant records
    assert not G["rhd_crop/2/keypoint_vis21"].any() and float(G["rhd_crop/2/crop_scale"]) == pytest.approx(256 / 50.0)
    assert float(G["rhd_crop/2/scoremap/sums"][0]) == 0.0                        # no valid key-point -> empty score map
