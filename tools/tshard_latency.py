"""Per-frame latency of the T-sharded SegNet (latency mode of SURVEY 8e) against one unsharded handle, on rank 0.

    python tools/tshard_latency.py --model standard --T 12 --precision fp16               # N = 1
    python -m torch.distributed.run --nproc-per-node N tools/tshard_latency.py ...          # N ranks, one GPU each

Input and outputs stay on the device.  A frame's latency is the host clock from before the broadcast of the cropped image to
after a device synchronize on the finalized maps; the unsharded figure is the same clock around run_device_maps + synchronize
of a plain handle on the same frame, and the two alternate frame by frame.  Stage times are CUDA events on the calling
stream: broadcast, partial (the median on each rank, then the maximum over ranks), reduce, finalize.  Frames are the seeded
synthetic frames of bench.py.  Prints one JSON line; writes nothing."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def power_limit_w(index):
    """The enforced board power limit of GPU `index`, read (not set) through NVML or nvidia-smi."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        return nv.nvmlDeviceGetEnforcedPowerLimit(nv.nvmlDeviceGetHandleByIndex(index)) / 1e3
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        return float(out)
    except Exception:
        return None


def pct(xs):
    a = np.asarray(xs, dtype=np.float64)
    return {"median": float(np.median(a)), "p10": float(np.percentile(a, 10)), "p90": float(np.percentile(a, 90))}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--model", choices=["basic", "standard"], default="standard")
    ap.add_argument("--T", type=int, default=12)
    ap.add_argument("--precision", choices=["fp16", "fp32"], default="fp16", help="fp16: fast mode; fp32: strict mode (tcgen05 split operands)")
    ap.add_argument("--frames", type=int, default=200, help="timed frames (each also timed unsharded)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic frames, cycled")
    args = ap.parse_args()
    if args.frames < 1 or args.warmup < 0:
        ap.error("--frames must be at least 1 and --warmup at least 0")

    import torch
    import torch.distributed as dist
    from bench import CROP_X, CROP_Y, NET_H, NET_W, frames, model_files
    from sivo_b200 import BayesianSegNet, BayesianSegNetParams
    from sivo_b200.tshard import TShardedSegNet, shard_ranges
    distributed = "WORLD_SIZE" in os.environ
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if distributed:
        dist.init_process_group("nccl", device_id=dev)
    rank = dist.get_rank() if distributed else 0
    world = dist.get_world_size() if distributed else 1
    engine = "tcgen05" if args.precision == "fp32" else "auto"
    models = tempfile.TemporaryDirectory(prefix="sivo_b200_models_")
    _, proto, model, _ = model_files(args.model, args.T, models.name)
    params = BayesianSegNetParams(proto, model)
    ts = TShardedSegNet(params, args.T, device=local, seed=1234, precision=args.precision, engine=engine)
    hw = NET_H * NET_W
    stream = torch.cuda.current_stream(dev)
    imgs = [torch.from_numpy(np.ascontiguousarray(f[0][CROP_Y:CROP_Y + NET_H, CROP_X:CROP_X + NET_W])).to(dev)
            for f in frames(args.distinct)] if rank == 0 else [None] * args.distinct
    cls, conf, ent = (torch.empty(hw, dtype=d, device=dev) for d in (torch.uint8, torch.float64, torch.float64))
    conf32, ent32 = (torch.empty(hw, dtype=torch.float32, device=dev) for _ in range(2))
    one = BayesianSegNet(params, device=local, seed=1234, T=args.T, precision=args.precision, engine=engine) if rank == 0 else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    lat, base, stages = [], [], {"broadcast": [], "partial": [], "reduce": [], "finalize": []}

    def sharded(i, timed):
        ts.set_frame(i)
        t0 = time.perf_counter()
        ts.segment_device(imgs[i % args.distinct], cls, conf, ent, conf32, ent32, events=ev if timed else None)
        torch.cuda.synchronize(dev)
        t1 = time.perf_counter()
        if not timed:
            return
        stages["partial"].append(ev[1].elapsed_time(ev[2]))
        if rank == 0:
            lat.append((t1 - t0) * 1e3)
            stages["broadcast"].append(ev[0].elapsed_time(ev[1]))
            stages["reduce"].append(ev[2].elapsed_time(ev[3]))
            stages["finalize"].append(ev[3].elapsed_time(ev[4]))

    def unsharded(i, timed):
        if rank != 0:
            return
        one.set_frame(i)
        t0 = time.perf_counter()
        one.run_device_maps(imgs[i % args.distinct].data_ptr(), cls.data_ptr(), conf.data_ptr(), ent.data_ptr(), conf32.data_ptr(),
                            ent32.data_ptr(), stream.cuda_stream)
        torch.cuda.synchronize(dev)
        if timed:
            base.append((time.perf_counter() - t0) * 1e3)

    for i in range(args.warmup + args.frames):
        timed = i >= args.warmup
        if i % 2:  # alternate which of the two runs first
            unsharded(i, timed)
            sharded(i, timed)
        else:
            sharded(i, timed)
            unsharded(i, timed)
    partial_max = float(np.median(stages["partial"]))
    if distributed:
        t = torch.tensor([partial_max], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        partial_max = float(t.item())
    if rank == 0:
        shards = [list(r) for r in shard_ranges(args.T, world)]
        line = {"metric": "tshard_latency_ms", "model": args.model, "T": args.T, "precision": args.precision,
                "mode": "strict" if args.precision == "fp32" else "fast", "N": world, "shards": shards,
                "geometry": [NET_W, NET_H], "frames": args.frames, "warmup": args.warmup,
                "sharded": pct(lat), "unsharded": pct(base),
                "speedup_median": float(np.median(base) / np.median(lat)),
                "stages_ms_median": {"broadcast": float(np.median(stages["broadcast"])), "partial_max_over_ranks": partial_max,
                                     "reduce": float(np.median(stages["reduce"])), "finalize": float(np.median(stages["finalize"]))},
                "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(local),
                "clock": "host perf_counter, broadcast to synchronize on the finalized maps"}
        print(json.dumps(line))
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
