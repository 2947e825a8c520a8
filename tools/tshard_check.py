"""T-sharded SegNet on real devices (latency mode of SURVEY 8e), launched by tests/test_gpu_tshard.py under torch.distributed.run:
every rank runs its contiguous range of the T Monte-Carlo samples of the same frame, one NCCL reduce adds the per-pixel
probability sums on rank 0, and rank 0 finalizes the maps and compares them with its own unsharded run of that frame.  The
reduce adds the shards in its own order, so confidence and entropy may move by rounding (<= 1e-12) and a class may differ only
where the top two mean probabilities are closer than that.  Cases: Basic T=6 at 1024x352 and Standard T=12 at 128x384."""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import torch.distributed as dist
    from bench import NET_H, NET_W, frames, model_files
    from conftest import make_model
    from sivo_b200 import BayesianSegNet, BayesianSegNetParams
    from sivo_b200.tshard import TShardedSegNet
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    models = tempfile.TemporaryDirectory(prefix="sivo_b200_models_")  # this rank's own copy of the seeded models
    cases = []
    _, proto, model, _ = model_files("basic", 6, models.name)
    cases.append(("basic_T6_1024x352", proto, model, 6, NET_H, NET_W))
    _, _, proto, model = make_model(models.name, "standard", T=12, H=128, W=384)
    cases.append(("standard_T12_128x384", proto, model, 12, 128, 384))
    ok = True
    for name, proto, model, T, H, W in cases:
        left = frames(1, start=4)[0][0]
        y0, x0 = (left.shape[0] - H) // 2, (left.shape[1] - W) // 2
        d_bgr = torch.from_numpy(np.ascontiguousarray(left[y0:y0 + H, x0:x0 + W])).to(dev)
        ts = TShardedSegNet(BayesianSegNetParams(proto, model), T, device=local, seed=1234)
        for frame in (7, 8):
            ts.set_frame(frame)
            res = ts.segment_device(d_bgr if rank == 0 else None)
            torch.cuda.synchronize(dev)
            if rank != 0:
                continue
            cls, conf, ent = (t.cpu().numpy() for t in res)
            top2 = torch.topk(ts.sums / T, 2, dim=0).values.cpu().numpy()
            one = BayesianSegNet(BayesianSegNetParams(proto, model), device=local, seed=1234, T=T)
            one.set_frame(frame)
            hw = H * W
            w_cls = torch.empty(hw, dtype=torch.uint8, device=dev)
            w_conf, w_ent = (torch.empty(hw, dtype=torch.float64, device=dev) for _ in range(2))
            one.run_device(d_bgr.data_ptr(), w_cls.data_ptr(), w_conf.data_ptr(), w_ent.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
            torch.cuda.synchronize(dev)
            wc, wf, we = w_cls.cpu().numpy(), w_conf.cpu().numpy(), w_ent.cpu().numpy()
            d_conf, d_ent = float(np.abs(conf - wf).max()), float(np.abs(ent - we).max())
            differ = cls != wc
            same = d_conf <= 1e-12 and d_ent <= 1e-12 and bool(np.all((top2[0] - top2[1])[differ] < 1e-12))
            print(f"{name} frame {frame}, {world} ranks: |d conf| {d_conf:.1e}, "
                  f"|d entropy| {d_ent:.1e}, {int(differ.sum())} tie classes, {'OK' if same else 'MISMATCH'}")
            ok = ok and same
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("TSHARD OK" if int(flag) == 1 else "TSHARD FAILED")
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if int(flag) == 1 else 1)


if __name__ == "__main__":
    main()
