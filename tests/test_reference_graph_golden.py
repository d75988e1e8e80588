"""Pins the GRAPH restatement of the oracle (and, on the GPU, the CUDA path) to tensors produced by the reference's own code.

`tests/golden/golden_reference_graph.npz` was produced by tests/golden/make_golden_reference_graph.py: the UNMODIFIED
nets/ColorHandPose3DNetwork.py, nets/PosePriorNetwork.py, utils/general.py and utils/relative_trafo.py of the reference, imported
from /root/reference and executed function by function over an eager numpy stand-in for `tensorflow` (oracle/tf1_eager.py).  The
structure of the computation (layers, names, strides, concat order, mask growing, crop arithmetic, Rodrigues / flip, kinematic
chain, tuple orders) therefore comes from the reference source; the heavy ops underneath are the oracle's restatement of the TF 1.3
kernels, so op-level semantics remain pinned by tests/test_oracle_kat.py only."""
import os
import sys

import numpy as np
import pytest

from hand3d_b200 import arch
from hand3d_b200 import weights as Wt
from oracle import hand3d_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
G = np.load(os.path.join(HERE, "golden", "golden_reference_graph.npz"))
sys.path.insert(0, os.path.join(HERE, "golden"))
TOL = 2e-5      # conv + bias_add as two ops (reference) vs one fused op (oracle): last-bit differences through 30 layers


@pytest.fixture(scope="module")
def wd():
    return Wt.synthetic_weights(0, seg_shift=0.15)


@pytest.fixture(scope="module")
def oracle_inference(wd):
    return O.inference(G["image"], G["hand_side"], wd)


def test_fixture_inputs_are_reproducible():
    np.testing.assert_array_equal(Wt.synthetic_blob_images(2, 48, 64, seed=41), G["image"])


def test_reference_requests_exactly_the_variables_of_the_layer_tables():
    """tf.get_variable calls made by the reference while building inference(): names and count match hand3d_b200/arch.py."""
    ours = sorted(arch.variable_shapes().keys()) if hasattr(arch, "variable_shapes") else None
    assert ours is not None
    assert list(G["variables_requested"]) == ours and len(ours) == 134


def test_oracle_inference_matches_reference_graph(oracle_inference):
    hand_scoremap, image_crop, scale_crop, center, kp_scoremap, coord3d = oracle_inference
    np.testing.assert_allclose(hand_scoremap, G["inf_hand_scoremap"], rtol=0, atol=TOL)
    np.testing.assert_array_equal(center, G["inf_center"])
    np.testing.assert_array_equal(scale_crop, G["inf_scale_crop"])
    np.testing.assert_array_equal(image_crop[:, ::8, ::8, :], G["inf_image_crop_s"])
    np.testing.assert_allclose([image_crop.astype(np.float64).sum(), np.abs(image_crop).astype(np.float64).sum()], G["inf_image_crop_sum"], rtol=1e-12)
    np.testing.assert_allclose(kp_scoremap[:, 3::16, 5::16, :], G["inf_kp_scoremap_s"], rtol=0, atol=TOL)
    np.testing.assert_allclose(coord3d, G["inf_coord3d"], rtol=0, atol=TOL)
    uv = np.stack([O.detect_keypoints(kp_scoremap[b]) for b in (0, 1)])
    np.testing.assert_array_equal(uv, G["inf_kp_uv"])
    assert bool(G["inf2d_tuple_ok"].all()) and float(G["det_hand_scoremap_max_abs_diff_vs_inference"]) == 0.0


def test_oracle_mask_stages_match_reference_graph(oracle_inference):
    hand_scoremap = oracle_inference[0]
    for literal in (True, False):
        mask = O.single_obj_scoremap(hand_scoremap, literal=literal)
        np.testing.assert_array_equal(mask[..., 0].sum(2), G["st_mask_rows"])
        np.testing.assert_array_equal(mask[..., 0].sum(1), G["st_mask_cols"])
    center, bb, size = O.calc_center_bb(O.single_obj_scoremap(hand_scoremap))
    np.testing.assert_array_equal(center, G["st_center"]); np.testing.assert_array_equal(bb, G["st_bb"])
    np.testing.assert_array_equal(size, G["st_crop_size"])
    fg, _ = O.seg_fg_det(hand_scoremap)
    np.testing.assert_array_equal(O.find_max_location(fg), G["st_max_loc"])
    ce, _, se = O.calc_center_bb(np.zeros((1, 16, 24, 1), np.float32))
    np.testing.assert_array_equal(ce, G["st_empty_center"]); np.testing.assert_array_equal(se, G["st_empty_size"])


def test_oracle_posenet_and_lifting_match_reference_graph(oracle_inference, wd):
    image_crop = oracle_inference[1]
    s = O.inference_pose2d(image_crop, wd)
    assert len(s) == 3
    np.testing.assert_allclose(s[0][:, ::2, ::2, :], G["pose_s0_s"], rtol=0, atol=TOL)
    np.testing.assert_allclose(s[2], G["pose_s2"], rtol=0, atol=TOL)
    can = O.inference_pose3d_can(G["pose_s2"], G["hand_side"], wd)
    np.testing.assert_allclose(can, G["lift_can"], rtol=0, atol=TOL)
    ux, uy, uz = O.rotation_estimation(G["pose_s2"], G["hand_side"], wd)
    np.testing.assert_allclose(O.get_rot_mat(ux, uy, uz), G["lift_rot"], rtol=0, atol=TOL)


@pytest.mark.parametrize("variant", ["direct", "bottleneck", "local", "local_w_xyz_loss", "proposed"])
def test_oracle_pose_prior_variants_match_reference_graph(variant, wd):
    from make_golden_reference_graph import prior_scoremap
    w = Wt.synthetic_weights(0, bottleneck=True) if variant == "bottleneck" else wd
    normed, c3, R = O.pose_prior_inference(prior_scoremap(), G["hand_side"], w, variant)
    np.testing.assert_allclose(normed, G["prior_%s_normed" % variant], rtol=0, atol=5e-5)
    np.testing.assert_allclose(c3, G["prior_%s_coord3d" % variant], rtol=0, atol=TOL)
    assert (R is not None) == bool(G["prior_%s_has_R" % variant])
    if R is not None:
        np.testing.assert_allclose(R, G["prior_%s_R" % variant], rtol=0, atol=TOL)


def test_oracle_relative_trafo_matches_reference_graph():
    np.testing.assert_allclose(O.bone_rel_trafo(G["coords_xyz"]), G["rel_fwd"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(O.bone_rel_trafo_inv(G["coords_rel"]), G["rel_inv"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(G["rel_roundtrip"], G["coords_xyz"], rtol=0, atol=1e-4)      # the reference's own round trip


# ------------------------------------------------------------------------------------------- CUDA path (GPU)
@pytest.mark.gpu
@pytest.mark.parametrize("prec,tol", [("fp32_ffma", 2e-4), ("bf16x3", 1e-3), ("fp16x3", 1e-3)])
def test_cuda_path_matches_reference_graph(prec, tol, wd):
    """Stage-wise against the reference-graph tensors (teacher-forced inputs), plus the key-points of the whole pipeline."""
    import torch
    from hand3d_b200 import runtime
    ctx = runtime.default_context()
    ctx.load_weights(wd)
    ctx.set_precision(prec)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    try:
        seg = ctx.handsegnet(dev(G["image"])).cpu().numpy()
        assert np.abs(seg - G["inf_hand_scoremap"]).max() < tol
        r = ctx.seg_postprocess(dev(G["inf_hand_scoremap"]))                      # discrete stages on the reference's logits: exact
        np.testing.assert_array_equal(r["center"].cpu().numpy(), G["inf_center"])
        np.testing.assert_array_equal(r["scale_crop"].cpu().numpy(), G["inf_scale_crop"])
        np.testing.assert_array_equal(r["crop_size"].cpu().numpy(), G["st_crop_size"])
        np.testing.assert_array_equal(r["max_loc"].cpu().numpy(), G["st_max_loc"])
        m = r["hand_mask"].cpu().numpy().astype(np.int64)
        np.testing.assert_array_equal(m.sum(2), G["st_mask_rows"].astype(np.int64))
        crop = ctx.crop_image_from_xy(dev(G["image"]), r["center"], 256, r["scale_crop"])
        np.testing.assert_array_equal(crop.cpu().numpy()[:, ::8, ::8, :], G["inf_image_crop_s"])
        s = [t.cpu().numpy() for t in ctx.posenet(crop)]
        assert np.abs(s[2] - G["pose_s2"]).max() < tol and np.abs(s[0][:, ::2, ::2, :] - G["pose_s0_s"]).max() < tol
        out, can, R = ctx.lifting(dev(G["pose_s2"]), dev(G["hand_side"]), "proposed")
        assert np.abs(can.cpu().numpy() - G["lift_can"]).max() < tol and np.abs(R.cpu().numpy() - G["lift_rot"]).max() < tol
        full = ctx.pipeline(dev(G["image"]), dev(G["hand_side"]), True, force_center=dev(G["inf_center"]), force_scale=dev(G["inf_scale_crop"]))
        assert np.abs(full["keypoint_coord3d"].cpu().numpy() - G["inf_coord3d"]).max() < tol
        assert np.abs(full["keypoints_scoremap"].cpu().numpy()[:, 3::16, 5::16, :] - G["inf_kp_scoremap_s"]).max() < tol
        agree = (full["keypoints_uv"].cpu().numpy() == G["inf_kp_uv"].astype(np.int32)).all(axis=2).mean()
        assert agree >= 0.95, agree                                               # arg-max of near-tied maps may move under 1e-5 .. 1e-4 noise
    finally:
        ctx.set_precision("bf16x3")
        ctx.load_weights(Wt.synthetic_weights(0))
