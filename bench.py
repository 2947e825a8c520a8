#!/usr/bin/env python
"""Headline benchmark: frames/sec of the SIVO perception front-end -- Bayesian SegNet(T) on the left image plus
the ORB extractor on the left and right images -- on synthetic 1242x375 stereo frames (centre-cropped to the
net's 1024x352 like System::TrackStereo does), N x B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model basic|standard] [--T 6] [--dump-outputs DIR]

One "step" = one stereo frame through both operators.  `value` times the operators with the cropped inputs
already resident in HBM; `e2e` times the reference-facing calls (segmentImage / operator()) on HOST buffers,
host<->device copies included, left/right ORB on two threads as Frame.cc:126-129 does.  N > 1 shards frames
one per rank (weak scaling) and all-gathers a packed per-frame record over NCCL each step.
`--impl reference` times the CPU restatement of the reference path (oracle/) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

CROP_X, CROP_Y, NET_W, NET_H = 109, 11, 1024, 352
BASELINE_PUBLISHED = None  # BASELINE.md holds no published number for this metric
DUMP_BYTES = 64 << 20  # --dump-outputs writes at most this much


def count_arg(minimum):
    def parse(text):
        v = int(text)
        if v < minimum:
            raise argparse.ArgumentTypeError(f"must be at least {minimum}")
        return v
    return parse


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=count_arg(1), default=30, help="timed steps")
    ap.add_argument("--warmup", type=count_arg(0), default=5, help="untimed steps before them")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="basic", choices=["basic", "standard"])
    ap.add_argument("--T", type=int, default=0, help="MC samples (default 6 basic / 12 standard; 6 standard for N>1)")
    ap.add_argument("--nfeatures", type=int, default=2000)
    ap.add_argument("--engine", default="auto", choices=["auto", "simt", "tcgen05"])
    ap.add_argument("--precision", default="fp16", choices=["fp16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-budget-seconds", type=float, default=1200.0,
                    help="--impl reference: full frames per step if (warmup + steps) of them fit this budget, else bounded samples")
    ap.add_argument("--sustain-seconds", type=float, default=3.0,
                    help="extra sustained leg on rank 0 (N=1): frames back to back for this long, own clock samples (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's frame) to DIR/<name>.npy; see dump_outputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def model_files(kind, T, cache_dir):
    """Prototxt + seeded synthetic caffemodel (the reference's weights are Git-LFS stubs; SURVEY 8d)."""
    import gen_prototxt
    from sivo_b200.caffemodel import shipped_scales, write_synth_model
    from sivo_b200.prototxt import load_net
    os.makedirs(cache_dir, exist_ok=True)
    text = getattr(gen_prototxt, kind)(T=T)
    proto = os.path.join(cache_dir, f"{kind}_T{T}.prototxt")
    model = os.path.join(cache_dir, f"{kind}_seed0_calibrated.caffemodel")
    with open(proto, "w") as f:
        f.write(text)
    net = load_net(text)
    weights = None
    if not os.path.exists(model):
        weights = write_synth_model(net, model, 0, shipped_scales(kind))  # calibrated: O(1) activations, unsaturated softmax
    return net, proto, model, weights


def frames(n, start=0):
    from sivo_b200.synth import bgr_to_gray, stereo_frame
    out = []
    for i in range(n):
        left, right = stereo_frame(start + i)
        gl = np.ascontiguousarray(bgr_to_gray(left)[CROP_Y:CROP_Y + NET_H, CROP_X:CROP_X + NET_W])
        gr = np.ascontiguousarray(bgr_to_gray(right)[CROP_Y:CROP_Y + NET_H, CROP_X:CROP_X + NET_W])
        out.append((left, gl, gr))
    return out


def dump_outputs(out_dir, rec, conf, ent):
    """Writes one timed step's results as out_dir/<name>.npy, in float32 or float64, so that two builds can be compared output
    for output: `classes`, `confidence` and `entropy` (SegNet's [H, W] maps, the latter two in double), `record_confidence` and
    `record_entropy` (the single-precision copies written into the packed record), and per image (`_left`, `_right`)
    `keypoints` [n, 7] (x, y, size, angle, response, octave, class_id) and `descriptors` [n, 32] (one byte per column).
    `rec` is the step's unpacked record (sivo_b200/record.py).  Should the keypoints take the files past DUMP_BYTES, each image
    keeps a fixed, seeded sample of its keypoint rows, in keypoint order."""
    out = {"classes": rec["classes"].astype(np.float32), "confidence": conf, "entropy": ent,
           "record_confidence": rec["confidence"].astype(np.float32), "record_entropy": rec["entropy"].astype(np.float32)}
    max_rows = (DUMP_BYTES - sum(a.nbytes for a in out.values())) // (2 * 4 * (7 + 32))
    for side in ("left", "right"):
        kp, desc = rec["kp_" + side], rec["desc_" + side]
        rows = np.arange(len(kp))
        if len(rows) > max_rows:
            rows = np.sort(np.random.default_rng(0).choice(len(kp), max_rows, replace=False))
        out["keypoints_" + side] = np.stack([kp[f][rows].astype(np.float32) for f in kp.dtype.names], axis=1).reshape(-1, 7)
        out["descriptors_" + side] = desc[rows].astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML from a thread every 2 ms
    (the timed regions last tens of milliseconds, too short for `nvidia-smi -lms`), nvidia-smi as the fallback."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index = index
        self.sm, self.mask, self.max_mhz, self.power = [], 0, None, []
        self.stop_flag = threading.Event()
        self.thread = None
        self.nvml = None

    def _handle(self):
        import pynvml
        pynvml.nvmlInit()
        self.nvml = pynvml
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            return pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            return pynvml.nvmlDeviceGetHandleByIndex(self.index)

    def _loop(self, h):
        nv = self.nvml
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.mask |= int(reasons(h))
                self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1e3)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            h = self._handle()
            self.max_mhz = float(self.nvml.nvmlDeviceGetMaxClockInfo(h, self.nvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._loop, args=(h,), daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None

    def stop(self):
        if self.thread:
            self.stop_flag.set()
            self.thread.join(timeout=2)
        if not self.sm:  # NVML unavailable: one nvidia-smi query (not under load -- says so)
            try:
                q = "clocks.sm,clocks.max.sm"
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=10).stdout.strip().split(",")
                return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "reasons": [], "samples": 0, "source": "nvidia-smi after the run"}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_min_mhz": float(min(self.sm)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in self.REASONS.items() if self.mask & b), "samples": len(self.sm),
                "power_w_median": float(np.median(self.power)) if self.power else None, "source": "nvml, 2 ms period, value + e2e regions"}


def cpu_reference_frame(net, weights, left_bgr, gl, gr, nfeatures, threads):
    """One frame of the CPU restatement of the reference path: SegNet(T) (torch fp32, all host threads) then
    the OpenCV-composed ORB extractor on two threads (Frame.cc:125-129 order)."""
    from oracle import orb_cv2, segnet_oracle as S
    t0 = time.perf_counter()
    S.segment_image(net, weights, left_bgr, seed=1234, frame=0, precision="fp32", threads=threads)
    t1 = time.perf_counter()
    th = [threading.Thread(target=orb_cv2.extract, args=(g, nfeatures)) for g in (gl, gr)]
    [t.start() for t in th]
    [t.join() for t in th]
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def load_weights(net, model):
    from sivo_b200.caffemodel import read_caffemodel
    return read_caffemodel(model)


def conv_flops(net):
    """(shared, per_sample) algorithmic convolution flops of a net: 2 Cin k^2 Cout H W per layer, split at the first sampling
    Dropout (everything upstream is sample-invariant; SURVEY 8d: Basic 52.00 + T 195.11 GF, Standard 134.12 + T 311.84 GF)."""
    from sivo_b200.prototxt import blob_shapes
    shapes = blob_shapes(net)
    shared = per = 0.0
    sampled = False
    for ly in net.layers:
        if ly.type == "Dropout" and ly.sample_weights_test:
            sampled = True
        if ly.type == "Convolution":
            cin = shapes[ly.bottoms[0]][0]
            cout, ho, wo = shapes[ly.tops[0]]
            f = 2.0 * cin * ly.kernel * ly.kernel * cout * ho * wo
            if sampled:
                per += f
            else:
                shared += f
    return shared, per


def run_reference(args, rank, world):
    """Reference arm: the CPU restatement of the reference path (the reference itself cannot be built here, DESIGN.md §2) on all
    host cores, same workload as the GPU arm.  Every step is ONE FULL FRAME -- SegNet(T) at full resolution, then the two
    extractor calls on two threads (Frame.cc:125-129 order) -- as long as (warmup + steps) such frames fit --ref-budget-seconds
    (a frame costs 10-15 s on a 128-core host; the driver's 25 frames take ~6 min).  Only if they do not, a step becomes a bounded
    sample: the same network at full resolution with T_S = 2 Monte-Carlo samples instead of T, scaled by this host's measured
    full-frame / sample time ratio (one untimed calibration), plus the two full extractor calls; `sample` says which.
    Exactly --steps timed steps after --warmup untimed ones."""
    if rank != 0:
        return
    import gen_prototxt
    from sivo_b200.prototxt import load_net
    T = args.T or (6 if args.model == "basic" else (12 if world == 1 else 6))  # the GPU arm's rule: configs[1] / [2] / [3]
    models = tempfile.TemporaryDirectory(prefix="sivo_b200_models_")
    net, proto, model, weights = model_files(args.model, T, models.name)
    weights = weights or load_weights(net, model)
    cores = os.cpu_count() or 1
    fr = frames(1)
    t0 = time.perf_counter()
    cpu_reference_frame(net, weights, fr[0][0], fr[0][1], fr[0][2], args.nfeatures, cores)  # untimed: warms the thread pool / allocator
    first = time.perf_counter() - t0
    n_total = args.warmup + args.steps
    times = []
    if first * n_total <= args.ref_budget_seconds:
        for i in range(n_total):
            a, b = cpu_reference_frame(net, weights, fr[0][0], fr[0][1], fr[0][2], args.nfeatures, cores)
            if i >= args.warmup:
                times.append(a + b)
        sample = (f"per step: 1 full frame -- SegNet {args.model} T={T} at 1024x352 (torch-CPU fp32 restatement, {cores} threads) + "
                  f"ORB({args.nfeatures}) x2 (cv2 composition, two threads); no sampling, no scaling")
    else:
        T_S = 2
        sample_net = load_net(getattr(gen_prototxt, args.model)(T=T_S))
        shared, per = conv_flops(net)
        flop_ratio = (shared + T * per) / (shared + T_S * per)
        cpu_reference_frame(sample_net, weights, fr[0][0], fr[0][1], fr[0][2], args.nfeatures, cores)
        samp_a, _ = cpu_reference_frame(sample_net, weights, fr[0][0], fr[0][1], fr[0][2], args.nfeatures, cores)
        full_a, _ = cpu_reference_frame(net, weights, fr[0][0], fr[0][1], fr[0][2], args.nfeatures, cores)
        scale = full_a / samp_a
        for i in range(n_total):
            a, b = cpu_reference_frame(sample_net, weights, fr[0][0], fr[0][1], fr[0][2], args.nfeatures, cores)
            if i >= args.warmup:
                times.append(a * scale + b)
        sample = (f"per step: SegNet {args.model} at full resolution with T={T_S} of {T} samples (a full frame took {first:.1f} s: "
                  f"{n_total} of them exceed the {args.ref_budget_seconds:.0f} s budget), time scaled by {scale:.3f} = this host's measured "
                  f"full-frame / sample SegNet time ({full_a:.2f} s / {samp_a:.2f} s, one untimed calibration; flop ratio {flop_ratio:.3f}), "
                  f"+ ORB({args.nfeatures}) x2 on the full images (cv2 composition, two threads)")
    ms = 1e3 * float(np.mean(times))
    fps = 1e3 / ms
    line = {"impl": "reference", "metric": "frames/sec SegNet(T)+ORB", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": len(times), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, T),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(args, T):
    return {"workload": f"Bayesian SegNet {args.model.capitalize()} T={T} + ORB({args.nfeatures}) x2, synthetic 1242x375 stereo "
                        f"(centre-cropped to 1024x352), one frame per GPU",
            "model": args.model, "T": T, "nfeatures": args.nfeatures, "engine": args.engine, "precision": args.precision,
            "l2": "inputs+activations per frame (>300 MB) exceed the 126 MB L2; distinct frame each step",
            "calls": "value: run_device (graph replay) + the two extractors on two host threads, inputs resident in HBM.  "
                     "e2e: the reference's call order -- segmentImage(host image) returns, THEN the two ORBextractor calls on two "
                     "threads (src/orbslam/Frame.cc:125-129), page-locked caller buffers; e2e_variants holds the same with the three "
                     "calls issued concurrently (one-line Frame.cc change, INTEGRATION.md) and with pageable caller buffers.  "
                     "N > 1: every step also shares the frame's packed record (classes u8 + f32 maps + keypoints, 3.5 MB) with all "
                     "ranks by one NCCL all-gather -- in `value` written on the device and gathered under the next frame, in `e2e` "
                     "the maps stay on the device (set_record_outputs), header + keypoints go back up, the gather is pipelined one frame"}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    from sivo_b200 import BayesianSegNet, BayesianSegNetParams, ORBextractor

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # Run the host side next to the GPU: bind this process (and the threads it starts) to the CPUs NVML names for the device, so
    # that the pinned buffers and the threads that touch them sit on the GPU's NUMA node.  Undone before the CPU baseline.
    all_cpus = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            h_nv = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)).encode())
        except Exception:
            h_nv = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        pynvml.nvmlDeviceSetCpuAffinity(h_nv)
    except Exception:
        pass
    if world > 1:
        # The gather overlaps the next frame's convolutions, whose grids are sized to the 148 SMs (conv_decode1: 288 CTAs = two
        # waves of 144).  A default NCCL all-gather takes a dozen SMs and would push them into a third wave, so keep it to a
        # few channels: 3.5 MB per rank needs little bandwidth (measured at N=2 with the earlier 6.4 MB record: 8 channels 1278 fps,
        # 2: 1425, 1: 1443).
        # measured with the 3.5 MB record (profiles/r2_scaling.md): N=8 2 channels 9972 frames/s, 4 channels 10396 (N=1 1324)
        nch = "1" if world <= 2 else ("2" if world <= 4 else "4")
        os.environ.setdefault("NCCL_MAX_NCHANNELS", nch)
        os.environ.setdefault("NCCL_MAX_CTAS", nch)
        dist.init_process_group("nccl", device_id=dev)
    T = args.T or (6 if args.model == "basic" else (12 if world == 1 else 6))
    # every rank writes its own copy of the seeded model into a directory of its own, removed at exit: nothing is shared
    # with other runs or users, and the source tree may be read-only
    models = tempfile.TemporaryDirectory(prefix="sivo_b200_models_")
    net, proto, model, weights = model_files(args.model, T, models.name)

    seg = BayesianSegNet(BayesianSegNetParams(proto, model), device=local_rank, seed=1234, precision=args.precision,
                         engine=args.engine)
    orb_l = ORBextractor(args.nfeatures, 1.2, 8, 20, 7, device=local_rank)
    orb_r = ORBextractor(args.nfeatures, 1.2, 8, 20, 7, device=local_rank)
    n_frames = 8
    fr = frames(n_frames, start=rank * n_frames)
    hw = NET_H * NET_W
    # ---- device-resident inputs for `value`
    d_bgr = [torch.from_numpy(np.ascontiguousarray(f[0][CROP_Y:CROP_Y + NET_H, CROP_X:CROP_X + NET_W])).to(dev) for f in fr]
    d_gl = [torch.from_numpy(f[1]).to(dev) for f in fr]
    d_gr = [torch.from_numpy(f[2]).to(dev) for f in fr]
    d_cls = torch.empty(hw, dtype=torch.uint8, device=dev)
    d_conf = torch.empty(hw, dtype=torch.float64, device=dev)
    d_ent = torch.empty(hw, dtype=torch.float64, device=dev)
    # packed per-frame record for the N>1 all-gather (sivo_b200/record.py)
    from sivo_b200 import record
    kp_cap = args.nfeatures + 4 * 8 + 64
    rec_bytes = record.record_bytes(hw, kp_cap)
    offs = record.offsets(hw, kp_cap)
    o_cls, o_conf, o_ent, o_kp = offs["classes"], offs["confidence"], offs["entropy"], offs["kp_left"]
    # double-buffered: the gather of frame i runs on a side stream under the convolutions of frame i+1.  SegNet writes its
    # three maps straight into the record (no device-to-device packing copies).
    NBUF = 3  # records in flight: frame i reuses the buffers of frame i-3, so a late gather (a late peer) has two frames of slack
    d_rec = [torch.zeros(rec_bytes, dtype=torch.uint8, device=dev) for _ in range(NBUF)]
    d_all = [torch.empty(rec_bytes * world, dtype=torch.uint8, device=dev) for _ in range(NBUF)] if world > 1 else None
    h_rec_t = [torch.zeros(rec_bytes, dtype=torch.uint8).pin_memory() for _ in range(NBUF)]
    h_rec = [t.numpy() for t in h_rec_t]
    stream = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(dev)  # joins a frame's three producers; carries the all-gather at N > 1
    ev_side = [torch.cuda.Event() for _ in range(NBUF)]
    ev_seg = [torch.cuda.Event() for _ in range(NBUF)]
    side_used = [False] * NBUF

    prof = {"segnet_launch": 0.0, "orb": 0.0, "pack": 0.0, "gather": 0.0}

    # two persistent host threads for the extractor calls (the reference starts two std::threads per frame, Frame.cc:126-129;
    # a Python thread start costs more than the C++ one, so the bench keeps them alive)
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=2)

    frame_ids = torch.arange(0, 1 << 16, dtype=torch.int64).pin_memory()  # header word 0 of the record, by frame index
    o_dl, o_kr, o_dr = offs["desc_left"], offs["kp_right"], offs["desc_right"]
    use_async_orb = orb_l.has_device_tree() and orb_r.has_device_tree() and orb_l.capacity() <= kp_cap

    JOIN_ON_MAIN = os.environ.get("SIVO_BENCH_JOIN", "main") != "side"  # where a frame's extractors are joined (see device_step)

    def device_step(i):
        """One frame with everything resident in HBM and nothing synchronous on the host: SegNet (one graph launch) writes its three
        maps, the two extractors (asynchronous form, device quad tree) their keypoints / descriptors / counts, all straight into the
        frame's packed record; at N > 1 the record is all-gathered on a side stream under the next frame's work."""
        j = i % n_frames
        t0 = time.perf_counter()
        k = i % NBUF
        base = d_rec[k].data_ptr()
        # Stream graph of frame i (record k = i mod NBUF):
        #   main : wait side[k] (frame i-NBUF's record fully consumed) -> SegNet(i) -> wait orb_l, orb_r -> seg[k]
        #   orb_l, orb_r (the handles' own streams, highest priority): wait side[k] -> extractor(i)
        #   side : wait seg[k] -> [all-gather of record k] -> side[k]
        # The extractors start with the frame, i.e. under SegNet's small early launches that leave SMs idle, and the main stream
        # waits for them before the next frame: measured (profiles/r2_notes.md), letting SegNet run ahead instead (joining the
        # extractors on the side stream, SIVO_BENCH_JOIN=side) starves their 13 short dependent kernels behind 0.2 ms CTAs.
        if side_used[k]:
            stream.wait_event(ev_side[k])
            if use_async_orb:
                orb_l.wait_event(ev_side[k].cuda_event)
                orb_r.wait_event(ev_side[k].cuda_event)
        # classes + the record's f32 maps straight into the record; the operator's double maps stay in d_conf / d_ent
        seg.run_device_maps(d_bgr[j].data_ptr(), base + o_cls, d_conf.data_ptr(), d_ent.data_ptr(), base + o_conf, base + o_ent, stream.cuda_stream)
        t1 = time.perf_counter()
        out = None
        if use_async_orb:
            orb_l.enqueue_device(d_gl[j].data_ptr(), NET_H, NET_W, NET_W, base + o_kp, base + o_dl, base + 8)
            orb_r.enqueue_device(d_gr[j].data_ptr(), NET_H, NET_W, NET_W, base + o_kr, base + o_dr, base + 16)
            d_rec[k][:8].view(torch.int64).copy_(frame_ids[(rank * 4096 + i) & 0xFFFF:][:1], non_blocking=True)
            if JOIN_ON_MAIN:
                orb_l.stream_wait(stream.cuda_stream)
                orb_r.stream_wait(stream.cuda_stream)
            t2 = t3 = time.perf_counter()
        else:  # host quad tree (nfeatures beyond the device tree's capacity): blocking extractor calls, host-packed record
            fr_ = pool.submit(orb_r.run_device_input, d_gr[j].data_ptr(), NET_H, NET_W, NET_W)
            out = [orb_l.run_device_input(d_gl[j].data_ptr(), NET_H, NET_W, NET_W), None]
            out[1] = fr_.result()
            t2 = time.perf_counter()
            if side_used[k]:
                ev_seg[k].synchronize()  # the upload that last read this pinned buffer (NBUF frames ago) has been consumed
            record.pack_host_part(h_rec[k], hw, kp_cap, rank * 100000 + i, out[0][0], out[0][1], out[1][0], out[1][1])
            t3 = time.perf_counter()
            d_rec[k][:record.HEADER].copy_(h_rec_t[k][:record.HEADER], non_blocking=True)
            d_rec[k][o_kp:].copy_(h_rec_t[k][o_kp:], non_blocking=True)
        ev_seg[k].record(stream)
        with torch.cuda.stream(side):
            side.wait_event(ev_seg[k])
            if use_async_orb and not JOIN_ON_MAIN:
                orb_l.stream_wait(side.cuda_stream)
                orb_r.stream_wait(side.cuda_stream)
            if world > 1:
                dist.all_gather_into_tensor(d_all[k], d_rec[k])
            ev_side[k].record(side)
        side_used[k] = True
        t4 = time.perf_counter()
        prof["segnet_launch"] += t1 - t0
        prof["orb"] += t2 - t1
        prof["pack"] += t3 - t2
        prof["gather"] += t4 - t3
        kp = (i - 1) % NBUF
        if (i & 3) == 3 and side_used[kp]:
            # bounded run-ahead: nothing above waits for the GPU, so without this the host would queue the whole run at once.
            # Waiting for the PREVIOUS frame keeps one frame queued behind the one that is running (no bubble)
            ev_side[kp].synchronize()
        return out

    # e2e buffers: page-locked host memory, as the contract asks (inputs from pinned memory; the results land in
    # caller-owned buffers the way the C++ shim's Eigen matrices / cv::Mat level buffers would)
    def pinned_like(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t, t.numpy()
    keep = []
    h_fr = []
    for (left, gl, gr) in fr:
        items = [pinned_like(x) for x in (left, gl, gr)]
        keep.append(items)
        h_fr.append(tuple(it[1] for it in items))
    out_t = [torch.empty((NET_H, NET_W), dtype=torch.uint8).pin_memory(), torch.empty((NET_H, NET_W), dtype=torch.float64).pin_memory(),
             torch.empty((NET_H, NET_W), dtype=torch.float64).pin_memory()]
    out_np = tuple(t.numpy() for t in out_t)
    pyr_t = [[torch.empty(shp, dtype=torch.uint8).pin_memory() for shp in orb_l.level_shapes(NET_H, NET_W)] for _ in range(2)]
    pyr_np = [[t.numpy() for t in lst] for lst in pyr_t]

    # pageable twins of the e2e buffers: what the untouched shim hands over (Eigen / cv::Mat storage, integration/src)
    h_fr_pageable = [tuple(np.array(a, copy=True) for a in f) for f in h_fr]
    out_pageable = tuple(np.empty_like(a) for a in out_np)
    pyr_pageable = [[np.empty_like(a) for a in lst] for lst in pyr_np]

    ev_e2e = [torch.cuda.Event() for _ in range(NBUF)]
    ev_up = [torch.cuda.Event() for _ in range(NBUF)]
    e2e_used = [False] * NBUF

    def host_step(i, order="reference", pinned=True):
        """One frame through the reference-facing calls on HOST buffers; each call is synchronous for its caller (host image in,
        host results out, copies inside).  order "reference": segmentImage returns before the two extractor threads start
        (src/orbslam/Frame.cc:125-129); "concurrent": the three independent calls are issued together."""
        j = i % n_frames
        left, gl, gr = (h_fr if pinned else h_fr_pageable)[j]
        outs, pyr = (out_np, pyr_np) if pinned else (out_pageable, pyr_pageable)
        if world > 1:
            # N > 1: the frame's record is shared with every rank (SURVEY 8e).  segmentImage leaves the record's maps (classes + f32
            # confidence / entropy) on the device next to the host results, so only the header and the keypoints go back up.
            k = i % NBUF
            if e2e_used[k]:
                ev_e2e[k].synchronize()  # record k's previous gather (NBUF frames ago) has read d_rec[k] / the upload has read h_rec[k]
            base = d_rec[k].data_ptr()
            seg.set_record_outputs(base + o_cls, base + o_conf, base + o_ent)
        if order == "reference":
            res = seg.segmentImage(left, out=outs)
            fl_ = pool.submit(orb_l, gl, None, want_pyramid=True, pyramid_buffers=pyr[0])
            fr_ = pool.submit(orb_r, gr, None, want_pyramid=True, pyramid_buffers=pyr[1])
        else:
            fl_ = pool.submit(orb_l, gl, None, want_pyramid=True, pyramid_buffers=pyr[0])
            fr_ = pool.submit(orb_r, gr, None, want_pyramid=True, pyramid_buffers=pyr[1])
            res = seg.segmentImage(left, out=outs)
        out = [fl_.result(), fr_.result()]
        if world > 1:
            record.pack_host_part(h_rec[k], hw, kp_cap, rank * 100000 + i, out[0][0], out[0][1], out[1][0], out[1][1])
            d_rec[k][:record.HEADER].copy_(h_rec_t[k][:record.HEADER], non_blocking=True)
            d_rec[k][o_kp:].copy_(h_rec_t[k][o_kp:], non_blocking=True)
            ev_up[k].record(stream)
            # the all-gather of frame i runs on the side stream under frame i+1's calls; frame i-1's must have landed before this
            # step returns (one frame of pipelining; the timed region ends with a device synchronize, so the last one is inside it)
            with torch.cuda.stream(side):
                side.wait_event(ev_up[k])
                dist.all_gather_into_tensor(d_all[k], d_rec[k])
                ev_e2e[k].record(side)
            e2e_used[k] = True
            kp = (i - 1) % NBUF
            if e2e_used[kp] and kp != k:
                ev_e2e[kp].synchronize()
        return res, out

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- value: inputs resident in HBM
    # set-up, not a step: the library captures one CUDA graph per (input, output, stream) pointer set the caller uses; touch every
    # input buffer of the rotation once so that no capture falls into the timed region whatever --warmup is
    for i in range(n_frames * NBUF):  # every (input buffer, record buffer) pair of the rotation: i mod n_frames x i mod NBUF
        device_step(i)
    for i in range(args.warmup):
        device_step(i)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # before the barrier: NVML start-up takes milliseconds, and a rank that enters the timed region late stalls
                         # every other rank's first all-gathers (measured at N=4: one 8 ms bubble in a 20-step region)
    import gc
    gc.collect()
    gc.disable()  # a collection pause inside a 20-ms timed region would be a visible fraction of it
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    t0 = time.perf_counter()
    launches = 0
    step_t = [time.perf_counter()]
    for i in range(args.steps):
        device_step(args.warmup + i)
        launches += seg.last_timing()["launches"] + orb_l.last_timing()["launches"] + orb_r.last_timing()["launches"]
        step_t.append(time.perf_counter())
    step_ms = 1e3 * np.diff(step_t)  # host-side issue time of each step (the last steps' GPU work drains before `elapsed` is read)
    e1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    gc.enable()
    if use_async_orb and (orb_l.device_status() or orb_r.device_status()):
        raise SystemExit("a pyramid level exceeded the device quad tree's capacity: the asynchronous records are not valid")
    if args.dump_outputs and rank == 0:
        # the last timed step's record and double maps, read before the legs below run device_step again
        last = record.unpack(d_rec[(args.warmup + args.steps - 1) % NBUF].cpu().numpy(), NET_H, NET_W, kp_cap)
        dump_outputs(args.dump_outputs, last, d_conf.cpu().numpy().reshape(NET_H, NET_W), d_ent.cpu().numpy().reshape(NET_H, NET_W))
    prof_value = dict(prof)  # the sustained leg and the e2e variants call device_step / the extractors again
    dev_ms = e0.elapsed_time(e1)
    elapsed = max(wall, dev_ms / 1e3)  # the ORB streams are the library's own; wall brackets everything (synced both sides)
    # ---- e2e: host buffers through the operator calls, three call patterns (the first is the headline)
    e2e_times = {}
    E2E_REPEATS = 3  # each measurement is exactly --steps frames; the median of three damps host-thread scheduling jitter
    for name, order, pinned in (("reference_order_pinned", "reference", True), ("concurrent_pinned", "concurrent", True),
                                ("reference_order_pageable", "reference", False)):
        for i in range(max(2, args.warmup // 2)):
            host_step(i, order, pinned)
        reps = []
        for _ in range(E2E_REPEATS):
            barrier()
            t0 = time.perf_counter()
            for i in range(args.steps):
                res, out = host_step(args.warmup + i, order, pinned)
            barrier()
            reps.append(time.perf_counter() - t0)
        e2e_times[name] = float(np.median(reps))
    e2e_elapsed = e2e_times["reference_order_pinned"]
    seg.set_record_outputs()
    clocks = sampler.stop() if rank == 0 else None
    n_kp = len(out[0][0]) + len(out[1][0])
    # per step, counted from the copies the three calls make: the cropped colour image and the two gray images go up; the three maps,
    # per extractor (count + status, the keypoint and descriptor capacity) and the 8 bordered pyramid levels come down
    pyr_bytes = 2 * sum((int(round(NET_H / 1.2 ** l)) + 38) * (int(round(NET_W / 1.2 ** l)) + 38 + 15) for l in range(8))
    if orb_l.has_device_tree():
        h2d = hw * 3 + 2 * hw
        d2h = hw * 17 + 2 * (8 + orb_l.capacity() * 60) + pyr_bytes
    else:  # host quad tree: candidates down, selected keypoints up
        h2d = hw * 3 + 2 * hw + n_kp * 8
        d2h = hw * 17 + n_kp * 36 + 2 * (32768 * 4 + 9 * 4) + pyr_bytes
    if world > 1:
        h2d += record.HEADER + 2 * kp_cap * 60  # the record's header and keypoint / descriptor blocks go back up for the gather
        names = sorted(e2e_times)
        tt = torch.tensor([elapsed] + [e2e_times[n] for n in names], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        elapsed = float(tt[0])
        e2e_times = {n: float(v) for n, v in zip(names, tt[1:])}
        e2e_elapsed = e2e_times["reference_order_pinned"]

    # ---- roofline of the dominant kernel: per-op CUDA events on the launching stream (profiling pass)
    roof = None
    cpu_base = None
    if rank == 0:
        seg.set_profiling(True)
        conv_ms, tot_ms, per_op = [], [], []
        for i in range(min(args.steps, 10)):
            seg.run_device(d_bgr[i % n_frames].data_ptr(), d_cls.data_ptr(), d_conf.data_ptr(), d_ent.data_ptr(), stream.cuda_stream)
            tm = seg.last_timing()
            conv_ms.append(tm["conv_ms"])
            tot_ms.append(tm["total_ms"])
            per_op.append(seg.op_timings())
        seg.set_profiling(False)
        # dominant kernel = the launch that EXECUTES the most multiply-adds (ties: the longer one).  Executed == algorithmic
        # except for the composed conv_decode1 x classifier layer (one 64 -> 16 convolution: 217 GF for the reference's 872) and
        # the split-operand fp32 mode (3 MMAs per product); the roofline counts what runs, the algorithmic figure rides along
        names = [o[0] for o in per_op[0]]
        op_alg = [o[2] for o in per_op[0]]
        op_flops = seg.op_flops_executed()
        op_ms = np.mean([[o[1] for o in run] for run in per_op], axis=0)
        dom = int(np.lexsort((op_ms, op_flops))[-1])
        fl = seg.flops()
        fl["exec"] = float(sum(op_flops))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        # the kernel is timed alone, by CUDA events, in a pass of <= 10 frames (milliseconds): burst regime -> the burst peak
        peak = peaks.get("bf16_tflops") or 1650.0
        which = "measured burst (MEASURED_PEAKS.json bf16_tflops): kernel timed alone in a <=10-frame pass" if peaks.get("bf16_tflops") \
            else "fallback 1.65 PF burst (B200_PROFILING.md)"
        peak_sus = peaks.get("bf16_tflops_sustained") or 1400.0
        ach = op_flops[dom] / (op_ms[dom] * 1e-3) / 1e12
        ach_all = fl["exec"] / (np.mean(conv_ms) * 1e-3) / 1e12
        traffic = None
        for tf in ("r2_traffic.json", "r1_traffic.json"):  # dram bytes of that kernel from the committed `ncu --set full` capture
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", tf)))
                traffic = tj.get(args.model, {}).get("dram_bytes_per_launch")
                if traffic:
                    break
            except Exception:
                pass
        # ---- sustained leg: >= --sustain-seconds of back-to-back work with its own clock samples, against the SUSTAINED peak
        sustained = None
        if args.sustain_seconds > 0 and world == 1:
            sustained = {}
            for leg in ("segnet_only", "full_step"):
                sm = ClockSampler(local_rank)
                sm.start()
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                n_done = 0
                while time.perf_counter() - t0 < args.sustain_seconds:
                    for _ in range(50):
                        if leg == "segnet_only":
                            seg.run_device(d_bgr[n_done % n_frames].data_ptr(), d_cls.data_ptr(), d_conf.data_ptr(), d_ent.data_ptr(), stream.cuda_stream)
                        else:
                            device_step(n_done)
                        n_done += 1
                    if leg == "segnet_only":
                        torch.cuda.synchronize(dev)  # bounded queue depth; the GPU is re-fed within microseconds
                torch.cuda.synchronize(dev)
                dt = time.perf_counter() - t0
                tf_s = fl["exec"] * n_done / dt / 1e12
                sustained[leg] = {"seconds": round(dt, 3), "frames": n_done, "frames_per_s": n_done / dt, "ms_per_frame": 1e3 * dt / n_done,
                                  "conv_tflops_executed": tf_s, "frac_of_sustained_peak": tf_s / peak_sus,
                                  "conv_tflops_algorithmic": fl["dedup"] * n_done / dt / 1e12, "clocks": sm.stop()}
            sustained["peak"] = peak_sus
            sustained["peak_source"] = "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks.get("bf16_tflops_sustained") else "fallback 1.4 PF"
            sustained["note"] = "conv_tflops_executed = executed conv FLOPs per frame x frames / wall seconds of the whole leg (non-conv kernels and, in full_step, the extractors included)"
        roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic,
                "kernel": f"tcgen05 convolution launch '{names[dom]}'", "peak_source": which,
                "kernel_ms": float(op_ms[dom]), "kernel_gflop": op_flops[dom] / 1e9, "kernel_gflop_algorithmic": op_alg[dom] / 1e9,
                "flops_counted": "executed multiply-adds x 2 (see kernel_gflop_algorithmic / algorithmic_gflop_per_frame for the reference's operation count)",
                "all_conv_launches": {"achieved": ach_all, "frac": ach_all / peak, "ms_per_frame": float(np.mean(conv_ms)),
                                      "gflop_per_frame": fl["exec"] / 1e9, "algorithmic_tflops": fl["dedup"] / (np.mean(conv_ms) * 1e-3) / 1e12},
                "conv_ms_per_frame": float(np.mean(conv_ms)), "segnet_ms_per_frame": float(np.mean(tot_ms)),
                "algorithmic_gflop_per_frame": fl["dedup"] / 1e9, "executed_gflop_per_frame": fl["exec"] / 1e9, "naive_gflop_per_frame": fl["naive"] / 1e9,
                "launch_ms": {n: round(float(m), 4) for n, m in zip(names, op_ms)},
                "launch_gflop": {n: round(f / 1e9, 2) for n, f in zip(names, op_flops)}, "sustained": sustained}
        if not args.no_cpu_baseline and world == 1:
            if all_cpus:  # the baseline gets every host core again (all threads of the process, incl. any OpenMP workers)
                try:
                    for tid in os.listdir("/proc/self/task"):
                        os.sched_setaffinity(int(tid), all_cpus)
                except Exception:
                    os.sched_setaffinity(0, all_cpus)
            w = weights or load_weights(net, model)
            cores = os.cpu_count() or 1
            a, b = cpu_reference_frame(net, w, fr[0][0], fr[0][1], fr[0][2], args.nfeatures, cores)
            cpu_base = {"value": 1.0 / (a + b), "unit": "frames/s", "cores": cores, "kind": "port",
                        "sample": f"1 full frame: SegNet {args.model} T={T} torch-CPU fp32 restatement ({a:.2f} s) + ORB({args.nfeatures}) x2 cv2 composition ({b:.2f} s)"}
    if rank == 0:
        total_frames = args.steps * world
        fps = total_frames / elapsed
        line = {"metric": "frames/sec SegNet(T)+ORB", "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f16" if args.precision == "fp16" else "f32", "data": "synthetic",
                "config": workload_config(args, T), "clocks": clocks,
                "e2e": {"value": total_frames / e2e_elapsed, "unit": "frames/s", "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(d2h), "calls": "reference order (segmentImage, then the two extractor threads), page-locked buffers"},
                "e2e_variants": {n: {"value": total_frames / t, "unit": "frames/s", "ms_per_step": 1e3 * t / args.steps} for n, t in e2e_times.items()},
                "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu_base,
                "host_ms_per_step": {k: round(1e3 * v / (args.steps + args.warmup + n_frames * NBUF), 3) for k, v in prof_value.items()},
                "orb_last_call": {"left": orb_l.last_timing(), "right": orb_r.last_timing()},
                "host_issue_ms_per_step": {"min": float(step_ms.min()), "median": float(np.median(step_ms)), "max": float(step_ms.max()),
                                           "argmax": int(step_ms.argmax()), "all": [round(float(v), 3) for v in step_ms]},
                "keypoints_last_frame": int(n_kp)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
