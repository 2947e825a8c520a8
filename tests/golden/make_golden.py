"""Regenerates the committed golden fixtures from the oracle (cv2 is used only to decode the PNG).  The
fixtures let the -m gpu tests compare the CUDA path with known outputs even where cv2 / the oracle's
dependencies differ, and pin the oracle against regressions.

  python tests/golden/make_golden.py
  python tests/golden/make_golden.py --reference-topology <SIVO checkout>   # reference_topology.json only
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cv2  # noqa: E402

from oracle import orb_oracle as O, segnet_oracle as S  # noqa: E402
from sivo_b200.synth import bgr_to_gray, stereo_frame  # noqa: E402


def orb_record(gray, nfeatures):
    r = O.extract(gray, O.ExtractorParams(nfeatures=nfeatures))
    return dict(keypoints=r.keypoints.astype(np.float32), descriptors=r.descriptors,
                level_counts=np.array(r.level_counts, np.int32),
                cand_counts=np.array([len(c[0]) for c in r.candidates], np.int32))


def layer_signature(net):
    """What test_host.py compares of each layer: wiring, shapes and the sampling / normalisation parameters."""
    return [[ly.name, ly.type, list(ly.bottoms), list(ly.tops), ly.num_output, ly.kernel, ly.pad, ly.local_size, ly.alpha,
             ly.beta, ly.dropout_ratio, ly.sample_weights_test, ly.weight_filler] for ly in net.layers]


REFERENCE_PROTOTXTS = {"basic": "config/bayesian_segnet/basic/kitti/bayesian_segnet_basic_kitti.prototxt",
                       "standard": "config/bayesian_segnet/standard/kitti/bayesian_segnet_kitti.prototxt"}


def reference_topology(ref_root):
    """Layer signatures of the original SIVO project's two KITTI prototxts, one layer per line."""
    from sivo_b200.prototxt import load_net
    parts = []
    for kind, rel in REFERENCE_PROTOTXTS.items():
        net = load_net(open(os.path.join(ref_root, rel)).read())
        layers = ",\n    ".join(json.dumps(s) for s in layer_signature(net))
        parts.append(f'"{kind}": {{"source": {json.dumps(rel)}, "input_dims": {json.dumps(net.input_dims)}, "layers": [\n    {layers}]}}')
    with open(os.path.join(HERE, "reference_topology.json"), "w") as f:
        f.write("{" + ",\n".join(parts) + "}\n")


def main():
    if len(sys.argv) == 3 and sys.argv[1] == "--reference-topology":
        reference_topology(sys.argv[2])
        print("reference_topology.json written")
        return
    img = cv2.imread(os.path.join(HERE, "kitti_000000_1242x375.png"))
    gray = np.ascontiguousarray(bgr_to_gray(img)[11:11 + 352, 109:109 + 1024])
    assert np.array_equal(bgr_to_gray(img), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))
    np.savez_compressed(os.path.join(HERE, "orb_kitti_2000.npz"), **orb_record(gray, 2000))
    np.savez_compressed(os.path.join(HERE, "orb_kitti_1000.npz"), **orb_record(gray, 1000))
    left, _ = stereo_frame(0)
    g0 = np.ascontiguousarray(bgr_to_gray(left)[11:11 + 352, 109:109 + 1024])
    np.savez_compressed(os.path.join(HERE, "orb_synth0_2000.npz"), **orb_record(g0, 2000))
    # small SegNets on a crop of the fixture, fp32 and fp16-operand models
    import tempfile
    from conftest import make_model
    with tempfile.TemporaryDirectory() as tmp:
        out = {}
        crop = np.ascontiguousarray(img[100:100 + 64, 300:300 + 128])
        for kind, kw in (("basic", dict(T=3, H=64, W=128)), ("standard", dict(T=2, H=64, W=128, widths=(64, 64, 64, 64, 64)))):
            net, w, _, _ = make_model(tmp, kind, seed=0, **kw)
            for prec in ("fp32", "fp16"):
                c, f, e = S.segment_image(net, w, crop, seed=1234, frame=0, precision=prec)
                out[f"{kind}_{prec}_classes"] = c
                out[f"{kind}_{prec}_confidence"] = f
                out[f"{kind}_{prec}_entropy"] = e
        np.savez_compressed(os.path.join(HERE, "segnet_small.npz"), **out)
    print("golden fixtures written")


if __name__ == "__main__":
    main()
