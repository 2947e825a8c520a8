"""CPU-only checks of the drop-in boundary: the C-ABI library loads, exports every declared symbol,
mirrors the reference's constructor error behaviour, and its host logic (prototxt / caffemodel readers,
quad tree) agrees with the Python twins and the oracle.  No compute call needs a GPU here."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import make_model
from sivo_b200 import _lib as L
from sivo_b200 import BayesianSegNet, BayesianSegNetParams, distribute_octtree
from sivo_b200.caffemodel import read_caffemodel, synth_weights
from sivo_b200.prototxt import load_net, blob_shapes, param_shapes


def test_library_exports_every_declared_symbol():
    syms = L.declared_symbols()
    assert len(syms) >= 25
    lib = L.lib()
    for s in syms:
        assert hasattr(lib, s), s
    assert b"sm_100a" in lib.sivo_version()


def test_ctor_throws_like_the_reference(model_dir):
    # tests/test_bayesian_segnet.cpp:138-150 (std::invalid_argument on empty paths)
    with pytest.raises(ValueError, match="model_file"):
        BayesianSegNet(BayesianSegNetParams("", "weights.caffemodel"))
    with pytest.raises(ValueError, match="weights_file"):
        BayesianSegNet(BayesianSegNetParams("model.prototxt", ""))
    # batch (= T) must be > 1 (bayesian_segnet.cpp:67-70)
    _, _, proto, model = make_model(model_dir, "basic", T=1, H=32, W=64, width=8)
    with pytest.raises(ValueError, match="batch size greater than 1"):
        BayesianSegNet(BayesianSegNetParams(proto, model))


def test_error_codes(model_dir, tmp_path):
    _, _, proto, model = make_model(model_dir, "basic", T=2, H=32, W=64, width=8)
    with pytest.raises(L.SivoError) as e:
        BayesianSegNet(BayesianSegNetParams(str(tmp_path / "nope.prototxt"), model))
    assert e.value.code == L.ENOENT
    stub = tmp_path / "stub.caffemodel"
    stub.write_text("version https://git-lfs.github.com/spec/v1\noid sha256:b2b0\nsize 5670476\n")
    with pytest.raises(L.SivoError) as e:
        BayesianSegNet(BayesianSegNetParams(proto, str(stub)))
    assert e.value.code == L.EFORMAT and "LFS" in str(e.value)
    bad = tmp_path / "bad.prototxt"
    bad.write_text(open(proto).read().replace('type: "LRN"', 'type: "InnerProduct"'))
    with pytest.raises(L.SivoError) as e:
        BayesianSegNet(BayesianSegNetParams(str(bad), model))
    assert e.value.code == L.EFORMAT


def test_blank_sample_dim_is_accepted_by_the_parser():
    text = ('name: "x"\ninput: "data"\ninput_shape {\n  dim: # SET SAMPLE SIZE HERE\n  dim: 3\n  dim: 32\n  dim: 64\n}\n'
            'layer { name: "c" type: "Convolution" bottom: "data" top: "c" convolution_param { num_output: 15 kernel_size: 1 } }\n'
            'layer { name: "prob" type: "Softmax" bottom: "c" top: "prob" }\n')
    net = load_net(text)
    assert net.input_dims == [None, 3, 32, 64]
    assert load_net(text, T=4).T == 4


def test_generated_prototxts_match_reference_topology():
    """Against the layer signatures of the original project's two KITTI prototxts, stored in
    tests/golden/reference_topology.json (tests/golden/make_golden.py --reference-topology)."""
    import json
    from conftest import GOLDEN, ROOT
    ref = json.load(open(os.path.join(GOLDEN, "reference_topology.json")))

    def sig(n):
        return [[l.name, l.type, list(l.bottoms), list(l.tops), l.num_output, l.kernel, l.pad, l.local_size, l.alpha,
                 l.beta, l.dropout_ratio, l.sample_weights_test, l.weight_filler] for l in n.layers]
    for mine, theirs in (("bayesian_segnet_basic.prototxt", "basic"), ("bayesian_segnet.prototxt", "standard")):
        a = load_net(open(os.path.join(ROOT, "configs", mine)).read())
        assert len(ref[theirs]["layers"]) > 20
        assert sig(a) == ref[theirs]["layers"]
        assert a.input_dims[1:] == ref[theirs]["input_dims"][1:] == [3, 352, 1024]


def test_flop_table_matches_survey():
    # SURVEY 8d: Basic 247.11 GF / sample (52.00 shared prefix), Standard 445.96 GF (134.12 shared)
    import gen_prototxt
    for text, total, prefix in ((gen_prototxt.basic(), 247.11, 52.00), (gen_prototxt.standard(), 445.96, 134.12)):
        net = load_net(text)
        shapes = blob_shapes(net)
        tot = pre = 0.0
        seen_drop = False
        for ly in net.layers:
            if ly.type == "Dropout":
                seen_drop = True
            if ly.type == "Convolution":
                cin = shapes[ly.bottoms[0]][0]
                c, h, w = shapes[ly.tops[0]]
                f = 2.0 * cin * ly.kernel ** 2 * c * h * w / 1e9
                tot += f
                if not seen_drop:
                    pre += f
        assert abs(tot - total) < 0.01 and abs(pre - prefix) < 0.01


def test_caffemodel_round_trip(model_dir):
    net, w, proto, model = make_model(model_dir, "standard", T=2, H=32, W=64, widths=(8, 8, 8, 8, 8))
    back = read_caffemodel(model)
    assert set(back) == set(w)
    for k in w:
        for a, b in zip(w[k], back[k]):
            assert a.shape == b.shape and np.array_equal(a, b)
    assert param_shapes(net)["conv1_1"] == [(8, 3, 3, 3), (8,)]
    assert param_shapes(net)["conv1_1_bn"] == [(1, 8, 1, 1), (1, 8, 1, 1)]


def test_quad_tree_matches_oracle():
    from oracle import orb_oracle as O
    rng = np.random.default_rng(0)
    for trial in range(20):
        n = int(rng.integers(1, 3000))
        w, h = int(rng.integers(100, 1000)), int(rng.integers(60, 330))
        xs = rng.integers(0, w, n).astype(np.float32)
        ys = rng.integers(0, h, n).astype(np.float32)
        rs = rng.integers(7, 120, n).astype(np.float32)  # many response ties
        tgt = int(rng.integers(1, 500))
        a = O.distribute_octtree(xs, ys, rs, 16, 16 + w, 16, 16 + h, tgt)
        b = distribute_octtree(xs, ys, rs, 16, 16 + w, 16, 16 + h, tgt)
        assert list(a) == b.tolist()
        assert len(b) <= max(tgt + 3, 1) or len(b) <= n


def test_bn_absorber_follows_the_reference_script(tmp_path):
    """8(f)-3: BN-absorber.py restated (W' = W * gamma, b' = b * gamma + beta in float64, BN blobs zeroed, BN layers dropped);
    the merged net computes the same probabilities as the BN net (fp32 rounding of W * gamma only), and the tool's files load."""
    import torch
    from conftest import make_model
    from oracle import segnet_oracle as S
    from sivo_b200 import bn_absorb
    from sivo_b200.caffemodel import read_caffemodel
    from sivo_b200.prototxt import load_net
    from sivo_b200.synth import stereo_frame
    net, w, proto, model = make_model(tmp_path, "standard", T=2, H=32, W=64, widths=(8, 8, 16, 16, 16))
    text = open(proto).read()
    new_text, new_w = bn_absorb.absorb(text, w)
    bn_names = [l.name for l in net.layers if l.type == "BN"]
    assert bn_names and all(n not in [l.name for l in load_net(new_text).layers] for n in bn_names)
    assert len(load_net(new_text).layers) == len(net.layers) - len(bn_names)
    # the literal per-feature-map loop of the script (:78-84)
    for i, layer in enumerate(net.layers):
        if layer.type != "BN":
            continue
        conv = net.layers[i - 1].name
        weight = np.array(w[conv][0], dtype=np.double)
        bias = np.array(w[conv][1], dtype=np.double).reshape(-1)
        gamma, beta = w[layer.name][0].reshape(-1), w[layer.name][1].reshape(-1)
        for j in range(weight.shape[0]):
            assert np.array_equal(new_w[conv][0][j], (weight[j] * gamma.item(j)).astype(np.float32))
            assert new_w[conv][1].reshape(-1)[j] == np.float32(bias[j] * gamma.item(j) + beta.item(j))
        assert not new_w[layer.name][0].any() and not new_w[layer.name][1].any()
    left, _ = stereo_frame(1, w=64, h=32)
    p0 = S.forward(net, w, left, seed=3, frame=0)
    p1 = S.forward(load_net(new_text), new_w, left, seed=3, frame=0)
    assert np.abs(p0 - p1).max() < 2e-4
    # command-line form writes the two files the script writes, and they read back
    bn_absorb.main(["--model", proto, "--weights", model, "--out_dir", str(tmp_path / "merged")])
    back = read_caffemodel(str(tmp_path / "merged" / "bn_conv_merged_weights.caffemodel"))
    assert all(np.array_equal(back[k][0], new_w[k][0]) for k in new_w)
    assert open(tmp_path / "merged" / "bn_conv_merged_model.prototxt").read() == new_text


def test_caffemodel_reader_survives_damaged_files(model_dir, tmp_path):
    """8(f)-3 loader hardening: truncated, bit-flipped and random .caffemodel bytes come back as an error code through the C-ABI
    (never a crash, never a silent success with the wrong shapes).  Without a GPU a file that still parses ends at the first
    CUDA call (ECUDA); with one, at the layer / shape check (EFORMAT)."""
    _, _, proto, model = make_model(model_dir, "basic", T=2, H=32, W=64, width=8)
    raw = open(model, "rb").read()
    rng = np.random.default_rng(0)
    cases = [raw[:cut] for cut in (1, 7, len(raw) // 3, len(raw) // 2, len(raw) - 1)]
    for _ in range(24):
        b = bytearray(raw)
        for _ in range(8):
            b[int(rng.integers(0, min(len(b), 4000)))] = int(rng.integers(0, 256))
        cases.append(bytes(b))
    cases.append(bytes(rng.integers(0, 256, 5000, dtype=np.uint8)))
    p = tmp_path / "damaged.caffemodel"
    import torch
    for data in cases:
        p.write_bytes(data)
        try:
            BayesianSegNet(BayesianSegNetParams(proto, str(p)))
            survived = True
        except L.SivoError as e:
            survived = False
            assert e.code in (L.EFORMAT, L.ECUDA, L.EINVAL), e
        # a damaged file may only load if the damage left every blob intact in size (a flipped weight byte)
        assert not survived or (torch.cuda.is_available() and len(data) == len(raw))


def test_record_maps_are_writable_in_place():
    """bench.py (N > 1) lets SegNet write classes / confidence / entropy straight into the packed record: the two f32 maps must
    sit on 16-byte boundaries and the regions must not overlap, for the full-size frame and for odd keypoint capacities."""
    from sivo_b200 import record
    for hw, cap in ((352 * 1024, 2096), (32 * 64, 17), (8, 1)):
        o = record.offsets(hw, cap)
        assert o["confidence"] % 16 == 0 and o["entropy"] % 4 == 0 and o["kp_left"] % 4 == 0
        assert o["classes"] >= record.HEADER and o["classes"] + hw <= o["confidence"]
        assert o["confidence"] + 4 * hw <= o["entropy"] and o["entropy"] + 4 * hw <= o["kp_left"]
        assert o["desc_right"] + cap * 32 <= record.record_bytes(hw, cap) and record.record_bytes(hw, cap) % 256 == 0
    assert record.record_bytes(352 * 1024, 2024) < 3.6e6  # SURVEY 8e: ~3.5 MB per rank
