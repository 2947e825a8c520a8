"""Multi-GPU data path check (SURVEY 8e), launched by tests/test_gpu_multirank.py under torch.distributed.run: every rank runs
SegNet + the two extractors on ITS frame with everything resident on the device (the bench's N > 1 step: maps, keypoints,
descriptors and counts written straight into the packed record), one NCCL all-gather moves the records, and rank 0 checks every
rank's slice of the gathered buffer against its own recomputation of that rank's frame (same seed, same frame counter ->
bit-identical maps; ORB is deterministic)."""
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
    from bench import CROP_X, CROP_Y, NET_H, NET_W, frames, model_files
    from sivo_b200 import BayesianSegNet, BayesianSegNetParams, ORBextractor, record
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    T = 2
    models = tempfile.TemporaryDirectory(prefix="sivo_b200_models_")  # this rank's own copy of the seeded model
    net, proto, model, _ = model_files("basic", T, models.name)
    hw = NET_H * NET_W
    nfeat = 1000

    def run_frame(r, seg, orb_l, orb_r):
        """The device-resident step of bench.py for frame r; returns the packed record (device tensor)."""
        left, gl, gr = frames(1, start=r)[0]
        kp_cap = orb_l.capacity()
        offs = record.offsets(hw, kp_cap)
        rec = torch.zeros(record.record_bytes(hw, kp_cap), dtype=torch.uint8, device=dev)
        d_bgr = torch.from_numpy(np.ascontiguousarray(left[CROP_Y:CROP_Y + NET_H, CROP_X:CROP_X + NET_W])).to(dev)
        d_gl, d_gr = torch.from_numpy(gl).to(dev), torch.from_numpy(gr).to(dev)
        stream = torch.cuda.current_stream(dev)
        base = rec.data_ptr()
        seg.set_frame(100 + r)
        d_conf, d_ent = torch.empty(hw, dtype=torch.float64, device=dev), torch.empty(hw, dtype=torch.float64, device=dev)
        seg.run_device_maps(d_bgr.data_ptr(), base + offs["classes"], d_conf.data_ptr(), d_ent.data_ptr(), base + offs["confidence"],
                            base + offs["entropy"], stream.cuda_stream)
        orb_l.enqueue_device(d_gl.data_ptr(), NET_H, NET_W, NET_W, base + offs["kp_left"], base + offs["desc_left"], base + 8)
        orb_r.enqueue_device(d_gr.data_ptr(), NET_H, NET_W, NET_W, base + offs["kp_right"], base + offs["desc_right"], base + 16)
        rec[:8].view(torch.int64).fill_(1000 + r)
        orb_l.stream_wait(stream.cuda_stream)
        orb_r.stream_wait(stream.cuda_stream)
        torch.cuda.synchronize(dev)
        assert orb_l.device_status() == 0 and orb_r.device_status() == 0
        # the record's f32 maps are the rounded double maps
        u = record.unpack(rec.cpu().numpy(), NET_H, NET_W, kp_cap)
        assert np.array_equal(u["confidence"].reshape(-1), d_conf.cpu().numpy().astype(np.float32))
        assert np.array_equal(u["entropy"].reshape(-1), d_ent.cpu().numpy().astype(np.float32))
        return rec, kp_cap

    def run_frame_host(r, seg, orb_l, orb_r):
        """The same record built the way bench.py's N > 1 e2e step does: the operator calls on host buffers, segmentImage leaving
        the record's maps on the device, header + keypoints packed on the host and uploaded."""
        left, gl, gr = frames(1, start=r)[0]
        kp_cap = orb_l.capacity()
        offs = record.offsets(hw, kp_cap)
        rec = torch.zeros(record.record_bytes(hw, kp_cap), dtype=torch.uint8, device=dev)
        base = rec.data_ptr()
        seg.set_record_outputs(base + offs["classes"], base + offs["confidence"], base + offs["entropy"])
        seg.set_frame(100 + r)
        seg.segmentImage(left)
        seg.set_record_outputs()
        (kl, dl), (kr, dr) = orb_l(gl, None)[:2], orb_r(gr, None)[:2]
        h = np.zeros(rec.numel(), np.uint8)
        record.pack_host_part(h, hw, kp_cap, 1000 + r, kl, dl, kr, dr)
        ht = torch.from_numpy(h)
        rec[:record.HEADER].copy_(ht[:record.HEADER])
        rec[offs["kp_left"]:].copy_(ht[offs["kp_left"]:])
        torch.cuda.synchronize(dev)
        return rec

    seg = BayesianSegNet(BayesianSegNetParams(proto, model), device=local, seed=1234, T=T)
    orb_l, orb_r = ORBextractor(nfeat, 1.2, 8, 20, 7, device=local), ORBextractor(nfeat, 1.2, 8, 20, 7, device=local)
    rec, kp_cap = run_frame(rank, seg, orb_l, orb_r)
    gathered = torch.empty(rec.numel() * world, dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(gathered, rec)
    torch.cuda.synchronize(dev)
    ok = True
    if rank == 0:
        g = gathered.cpu().numpy().reshape(world, -1)
        for r in range(world):
            mine, _ = run_frame(r, seg, orb_l, orb_r)
            a, b = record.unpack(g[r], NET_H, NET_W, kp_cap), record.unpack(mine.cpu().numpy(), NET_H, NET_W, kp_cap)
            same = a["frame_id"] == 1000 + r and all(np.array_equal(a[k], b[k]) for k in ("classes", "confidence", "entropy", "desc_left", "desc_right")) \
                and a["kp_left"].tobytes() == b["kp_left"].tobytes() and a["kp_right"].tobytes() == b["kp_right"].tobytes() \
                and len(a["kp_left"]) > 300 and len(a["kp_right"]) > 300
            # ... and the record the host-call (e2e) path builds for the same frame is the same bytes where both define them
            c = record.unpack(run_frame_host(r, seg, orb_l, orb_r).cpu().numpy(), NET_H, NET_W, kp_cap)
            same = same and all(np.array_equal(a[k], c[k]) for k in ("classes", "confidence", "entropy", "desc_left", "desc_right")) \
                and a["kp_left"].tobytes() == c["kp_left"].tobytes() and a["kp_right"].tobytes() == c["kp_right"].tobytes() and c["frame_id"] == 1000 + r
            print(f"rank {r}: frame_id {a['frame_id']}, {len(a['kp_left'])}+{len(a['kp_right'])} keypoints, record {'OK' if same else 'MISMATCH'}")
            ok = ok and same
        # the records of different ranks really are different frames
        ok = ok and not np.array_equal(g[0], g[world - 1])
        print("MULTIRANK OK" if ok else "MULTIRANK FAILED")
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
