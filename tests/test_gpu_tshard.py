"""-m gpu: sample shards (latency mode of SURVEY 8e).  A shard handle computes a contiguous range of the T Monte-Carlo samples
with the dropout masks an unsharded handle draws for them and leaves the per-pixel double sums of their softmax
probabilities; finalize turns the sums of all T samples into the three maps.

Run one after another into one buffer, the shards of [0, T) perform exactly the unsharded reduction's sequence of double
additions, so the maps are bitwise those of one handle.  That also needs each sample's logits not to depend on the batch the
convolutions were planned for: row-block and tile choices move a pixel to another CTA but keep its accumulation order.  The
NCCL reduce adds the shards' sums in another order, which moves the results by a few ulp (test 5 and tools/tshard_check.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import make_model
from sivo_b200 import BayesianSegNet, BayesianSegNetParams
from sivo_b200 import _lib as L
from sivo_b200.orb import KP_DTYPE
from sivo_b200.synth import stereo_frame

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = {"strict": dict(precision="fp32", engine="tcgen05"), "fast": dict(precision="fp16", engine="auto")}


@pytest.fixture(autouse=True)
def side_stream():
    """Every test runs on one torch stream, so the handles' calls and torch's own work are ordered on it: stream 0 (torch's
    default) would make each handle use its own stream, and shards writing one buffer would race."""
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        yield s
    torch.cuda.synchronize()


def _p(a):
    import ctypes
    return a.ctypes.data_as(ctypes.c_void_p)


def _logits(T, H, W, seed=3):
    rng = np.random.default_rng(seed)
    logits = rng.normal(0, 3, size=(T, 15, H, W)).astype(np.float32)
    logits[:, :, 0, 0] = 0.0           # exact 15-way tie -> class 0
    logits[:, 3, 0, 1] = 200.0         # saturated softmax -> p = 0 elsewhere -> 0 log 0 := 0
    logits[:, :, 0, 2] = -120.0        # probabilities that underflow in the mean
    logits[:, 5, 0, 2] = 0.0
    return logits


def _finalize(sums, T, H, W):
    cls, conf, ent = np.empty((H, W), np.uint8), np.empty((H, W), np.float64), np.empty((H, W), np.float64)
    L.check(L.lib().sivo_dbg_mc_finalize(0, _p(sums), T, 15, H, W, _p(cls), _p(conf), _p(ent)))
    return cls, conf, ent


def test_partial_and_finalize_equal_the_one_pass_reduction_bitwise():
    T, H, W = 6, 9, 33
    logits = _logits(T, H, W)
    cls, conf, ent = np.empty((H, W), np.uint8), np.empty((H, W), np.float64), np.empty((H, W), np.float64)
    L.check(L.lib().sivo_dbg_mc_reduce(0, _p(logits), T, 15, H, W, _p(cls), _p(conf), _p(ent)))
    sums = np.full((15, H, W), np.nan)
    L.check(L.lib().sivo_dbg_mc_partial(0, _p(logits), T, 15, H, W, 0, _p(sums)))  # accumulate = 0 ignores what is there
    got = _finalize(sums, T, H, W)
    assert np.array_equal(got[0], cls) and np.array_equal(got[1], conf) and np.array_equal(got[2], ent)
    assert cls[0, 0] == 0 and cls[0, 1] == 3 and ent[0, 1] == 0.0
    for k in range(1, T):
        part = np.zeros((15, H, W))
        L.check(L.lib().sivo_dbg_mc_partial(0, _p(np.ascontiguousarray(logits[:k])), k, 15, H, W, 0, _p(part)))
        L.check(L.lib().sivo_dbg_mc_partial(0, _p(np.ascontiguousarray(logits[k:])), T - k, 15, H, W, 1, _p(part)))
        assert np.array_equal(part, sums), k
        got = _finalize(part, T, H, W)
        assert np.array_equal(got[0], cls) and np.array_equal(got[1], conf) and np.array_equal(got[2], ent), k


def _dropout_tops(net):
    return [ly.tops[0] for ly in net.layers if ly.type == "Dropout" and ly.sample_weights_test]


@pytest.mark.parametrize("kind,kw", [("basic", dict(T=6, H=64, W=128)), ("standard", dict(T=6, H=64, W=128, widths=(64, 64, 64, 64, 64)))])
def test_shard_draws_the_masks_of_its_global_samples(model_dir, kitti_bgr, kind, kw):
    net, _, proto, model = make_model(model_dir, kind, seed=0, **kw)
    img = np.ascontiguousarray(kitti_bgr[100:164, 300:428])
    blobs = []
    for samples in (None, (2, 2)):
        seg = BayesianSegNet(BayesianSegNetParams(proto, model), seed=1234, keep_blobs=True, samples=samples)
        seg.set_frame(4)
        d_bgr = torch.from_numpy(img).cuda()
        if samples is None:
            seg.segmentImage(img)
        else:
            sums = torch.empty((seg.n_classes, seg.height * seg.width), dtype=torch.float64, device="cuda")
            seg.run_device_partial(d_bgr.data_ptr(), sums.data_ptr(), False, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
        names = _dropout_tops(net)
        assert names
        blobs.append({n: seg.blob(n) for n in names})
    for n, full in blobs[0].items():
        assert full.shape[0] == 6 and blobs[1][n].shape[0] == 2, n
        assert np.array_equal(full[2:4], blobs[1][n]), n
        assert not np.array_equal(full[0:2], blobs[1][n]), n


def _device_frame(i, H, W):
    left, _ = stereo_frame(i)
    y0, x0 = (left.shape[0] - H) // 2, (left.shape[1] - W) // 2
    return torch.from_numpy(np.ascontiguousarray(left[y0:y0 + H, x0:x0 + W])).cuda()


def _maps(hw):
    return (torch.empty(hw, dtype=torch.uint8, device="cuda"), torch.empty(hw, dtype=torch.float64, device="cuda"),
            torch.empty(hw, dtype=torch.float64, device="cuda"), torch.empty(hw, dtype=torch.float32, device="cuda"),
            torch.empty(hw, dtype=torch.float32, device="cuda"))


def _unsharded(proto, model, T, mode, d_bgr, frame, seed=1234):
    seg = BayesianSegNet(BayesianSegNetParams(proto, model), seed=seed, T=T, **MODES[mode])
    out = _maps(seg.height * seg.width)
    seg.set_frame(frame)
    seg.run_device_maps(d_bgr.data_ptr(), *(t.data_ptr() for t in out), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    seg.maps = out  # semantic_keys reads the handle's last maps where they are
    return seg, [t.cpu().numpy() for t in out]


def _sequential_shards(proto, model, T, mode, ranges, d_bgr, frame, seed=1234):
    stream = torch.cuda.current_stream().cuda_stream
    shards = [BayesianSegNet(BayesianSegNetParams(proto, model), seed=seed, T=T, samples=r, **MODES[mode]) for r in ranges]
    hw = shards[0].height * shards[0].width
    sums = torch.full((shards[0].n_classes, hw), float("nan"), dtype=torch.float64, device="cuda")
    for i, sh in enumerate(shards):
        sh.set_frame(frame)
        sh.run_device_partial(d_bgr.data_ptr(), sums.data_ptr(), i > 0, stream)
    out = _maps(hw)
    shards[-1].finalize_device(sums.data_ptr(), *(t.data_ptr() for t in out), stream=stream)
    torch.cuda.synchronize()
    shards[-1].maps = out
    return shards, sums, [t.cpu().numpy() for t in out]


def _assert_maps_equal(got, want):
    for name, a, b in zip(("classes", "confidence", "entropy", "confidence_f32", "entropy_f32"), got, want):
        assert np.array_equal(a, b), (name, int((a != b).sum()))


@pytest.mark.parametrize("mode", ["fast", "strict"])
def test_sequential_shards_equal_one_handle_basic_full_size(tmp_path, mode):
    from bench import NET_H, NET_W, model_files
    _, proto, model, _ = model_files("basic", 6, str(tmp_path))
    d_bgr = _device_frame(2, NET_H, NET_W)
    _, want = _unsharded(proto, model, 6, mode, d_bgr, 11)
    shards, _, got = _sequential_shards(proto, model, 6, mode, [(0, 2), (2, 3), (5, 1)], d_bgr, 11)
    assert all(sh.T == 6 for sh in shards)
    _assert_maps_equal(got, want)


def test_sequential_shards_equal_one_handle_standard_T12(model_dir):
    _, _, proto, model = make_model(model_dir, "standard", T=12, H=128, W=384)
    d_bgr = _device_frame(1, 128, 384)
    _, want = _unsharded(proto, model, 12, "fast", d_bgr, 5)
    _, _, got = _sequential_shards(proto, model, 12, "fast", [(0, 3), (3, 3), (6, 3), (9, 3)], d_bgr, 5)
    _assert_maps_equal(got, want)


def test_reduction_order_moves_results_by_rounding_only(model_dir):
    """What the NCCL reduce does: each shard's sums in its own buffer, added in another order."""
    _, _, proto, model = make_model(model_dir, "standard", T=12, H=128, W=384)
    d_bgr = _device_frame(3, 128, 384)
    stream = torch.cuda.current_stream().cuda_stream
    _, want = _unsharded(proto, model, 12, "fast", d_bgr, 8)
    parts = []
    for r in [(0, 3), (3, 3), (6, 3), (9, 3)]:
        sh = BayesianSegNet(BayesianSegNetParams(proto, model), seed=1234, T=12, samples=r)
        s = torch.empty((sh.n_classes, sh.height * sh.width), dtype=torch.float64, device="cuda")
        sh.set_frame(8)
        sh.run_device_partial(d_bgr.data_ptr(), s.data_ptr(), False, stream)
        parts.append(s)
    total = (parts[3] + parts[2]) + (parts[1] + parts[0])
    out = _maps(sh.height * sh.width)
    sh.finalize_device(total.data_ptr(), *(t.data_ptr() for t in out), stream=stream)
    torch.cuda.synchronize()
    got = [t.cpu().numpy() for t in out]
    assert np.abs(got[1] - want[1]).max() <= 1e-12 and np.abs(got[2] - want[2]).max() <= 1e-12
    top2 = torch.topk(total / 12, 2, dim=0).values.cpu().numpy()
    differ = got[0] != want[0]
    assert np.all((top2[0] - top2[1])[differ] < 1e-12), int(differ.sum())


def test_semantic_keys_refusals_and_the_whole_range_shard(model_dir, kitti_bgr):
    _, _, proto, model = make_model(model_dir, "basic", T=6, H=64, W=128)
    img = np.ascontiguousarray(kitti_bgr[100:164, 300:428])
    d_bgr = torch.from_numpy(img).cuda()
    stream = torch.cuda.current_stream().cuda_stream
    full, want = _unsharded(proto, model, 6, "fast", d_bgr, 3)
    shards, _, got = _sequential_shards(proto, model, 6, "fast", [(0, 4), (4, 2)], d_bgr, 3)
    _assert_maps_equal(got, want)
    rng = np.random.default_rng(0)
    kps = np.zeros(300, KP_DTYPE)
    kps["x"] = rng.uniform(-2, 130, 300)
    kps["y"] = rng.uniform(-2, 66, 300)
    a, b = full.semantic_keys(kps), shards[-1].semantic_keys(kps)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    # whole-frame calls on a partial shard: their mean would be over the wrong sample count
    part = shards[0]
    hw = part.height * part.width
    o = _maps(hw)
    with pytest.raises(L.SivoError, match=r"samples \[0, 4\) of T = 6"):
        part.segmentImage(img)
    with pytest.raises(L.SivoError):
        part.run_device(d_bgr.data_ptr(), o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), stream)
    with pytest.raises(L.SivoError):
        part.run_device_maps(d_bgr.data_ptr(), *(t.data_ptr() for t in o), stream)
    # a shard [0, T) is a normal handle
    whole = BayesianSegNet(BayesianSegNetParams(proto, model), seed=1234, T=6, samples=(0, 6))
    plain = BayesianSegNet(BayesianSegNetParams(proto, model), seed=1234, T=6)
    for seg in (whole, plain):
        seg.set_frame(3)
    r0, r1 = whole.segmentImage(img), plain.segmentImage(img)
    assert all(np.array_equal(x, y) for x, y in zip(r0, r1))
    assert np.array_equal(r1[0].reshape(-1), want[0]) and np.array_equal(r1[2].reshape(-1), want[2])


def test_nccl_t_sharded_maps_match_one_handle():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = min(n, 4)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                        "--master-port", "29613", os.path.join(ROOT, "tools", "tshard_check.py")], capture_output=True, text=True, timeout=900)
    print(r.stdout[-3000:])
    assert r.returncode == 0 and "TSHARD OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
