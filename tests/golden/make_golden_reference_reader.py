"""Golden vectors of the dataset readers' derived items, produced by running the reference's UNMODIFIED reader classes
(data/BinaryDbReader.py, data/BinaryDbReaderSTB.py, with utils/canonical_trafo.py, utils/relative_trafo.py, utils/general.py
underneath -- all imported from /root/reference) over the eager TF stand-in (oracle/tf1_eager.py) on seeded synthetic records
(tests/golden/synth_records.py) written to the file names the readers insist on.

Pins oracle/reader_oracle.py (and through it the CUDA generators of SURVEY.md 8(f) row 4) to the reference SOURCE: palm / wrist
substitution, dominant-hand rule, 21-key-point subsets, root-relative normalisation, GT hand-crop arithmetic, intrinsics update,
create_multiple_gaussian_map, scale_to_size, convert_kp, canonical_trafo.  The heavy TF ops underneath (crop_and_resize, legacy
resize) are oracle/tf1_ops.py, pinned separately by tests/test_tf_published_vectors.py.

    python tests/golden/make_golden_reference_reader.py       # only where /root/reference exists; ~1 minute of CPU
Large tensors (image, image_crop, scoremap) are stored as a sub-sampled copy plus float64 sum / sum of squares.  Score maps
take every 16th pixel (their Gaussians have sigma = 25 px), the others every 8th, which keeps the file well under 1 MB.
"""
import os
import sys
import tempfile
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("H3D_REFERENCE", "/root/reference")
OUT = os.path.join(HERE, "golden_reference_reader.npz")
sys.path.insert(0, HERE)
import synth_records as SR  # noqa: E402


def setup_imports():
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or ".") not in (ROOT,)]
    sys.path.insert(0, REF)
    sys.path.append(ROOT)
    import oracle.tf1_eager as tfe
    py = types.ModuleType("tensorflow.python")
    py.pywrap_tensorflow = types.ModuleType("tensorflow.python.pywrap_tensorflow")
    tfe.python = py
    sys.modules["tensorflow"] = tfe
    sys.modules["tensorflow.python"] = py
    sys.modules["tensorflow.python.pywrap_tensorflow"] = py.pywrap_tensorflow
    for pkg in ("nets", "utils", "data"):
        m = types.ModuleType(pkg)
        m.__path__ = [os.path.join(REF, pkg)]
        sys.modules[pkg] = m
    import data.BinaryDbReader as rhd
    import data.BinaryDbReaderSTB as stb
    for m in (rhd, stb):
        assert os.path.abspath(m.__file__).startswith(os.path.abspath(REF)), m.__file__
    return tfe, rhd, stb


BIG = ("image", "image_crop", "scoremap", "hand_parts", "hand_mask")


def sub_step(k):
    return 16 if k == "scoremap" else 8


def pack(prefix, d, out):
    for k, v in d.items():
        v = np.squeeze(np.asarray(v), 0)                  # batch_join adds the batch dimension of 1
        if k in BIG:
            s = sub_step(k)
            out["%s/%s/sub%d" % (prefix, k, s)] = np.ascontiguousarray(v[::s, ::s])
            out["%s/%s/sums" % (prefix, k)] = np.array([v.astype(np.float64).sum(), np.square(v.astype(np.float64)).sum()])
            out["%s/%s/shape" % (prefix, k)] = np.array(v.shape)
        else:
            out["%s/%s" % (prefix, k)] = v


def main():
    tf, rhd, stb = setup_imports()
    out = {}
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            os.makedirs("data/bin"); os.makedirs("data/stb")
            recs = SR.rhd_records(4)
            with open("data/bin/rhd_evaluation.bin", "wb") as f:
                f.write(b"".join(recs))
            srecs = SR.stb_records(2)
            with open("data/stb/stb_eval.bin", "wb") as f:
                f.write(b"".join(srecs))
            # the three reader configurations the evaluation drivers use
            configs = {
                "rhd_crop": dict(mode="evaluation", shuffle=False, hand_crop=True, use_wrist_coord=False),          # eval3d.py:50, eval2d_gt_cropped.py:37
                "rhd_full": dict(mode="evaluation", shuffle=False, use_wrist_coord=False),                          # eval_full.py:44
                "rhd_scaled": dict(mode="evaluation", shuffle=False, use_wrist_coord=True, scale_to_size=True),      # eval2d.py:43
            }
            for name, kw in configs.items():
                tf.reset_readers()
                for i in range(len(recs)):
                    pack("%s/%d" % (name, i), rhd.BinaryDbReader(**kw).get(), out)
            for name, kw in {"stb_palm": dict(mode="evaluation", shuffle=False, use_wrist_coord=False),                 # eval_full.py:45
                             "stb_wrist": dict(mode="evaluation", shuffle=False, use_wrist_coord=True)}.items():
                tf.reset_readers()
                for i in range(len(srecs)):
                    pack("%s/%d" % (name, i), stb.BinaryDbReaderSTB(**kw).get(), out)
        finally:
            os.chdir(cwd)
    np.savez_compressed(OUT, **out)
    print("wrote %s: %d arrays, %.1f KB" % (OUT, len(out), os.path.getsize(OUT) / 1024))


if __name__ == "__main__":
    main()
