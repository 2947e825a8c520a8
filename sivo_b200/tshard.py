"""Latency mode of the multi-GPU path (SURVEY 8e): one frame's T Monte-Carlo dropout samples split across the ranks of a
torch.distributed NCCL group.  Every rank runs the sample-invariant prefix and its own contiguous range of samples
(BayesianSegNet(samples=...)), which leaves the per-pixel double sums of its softmax probabilities on its device; one
`dist.reduce` adds the sums on the root, and the root computes classes, confidence and entropy from them.  The frame-sharded
path (bench.py, tools/multirank_check.py) puts one frame on each GPU instead, which adds throughput but not latency.

The collective stays in Python; the library has no NCCL dependency."""
from __future__ import annotations

from typing import Optional

from .segnet import BayesianSegNet, BayesianSegNetParams


def shard_ranges(T: int, G: int) -> list:
    """G contiguous (first, count) ranges that cover [0, T) in order; counts differ by at most one, larger ones first."""
    if G < 1 or G > T:
        raise ValueError(f"cannot split T = {T} samples into {G} non-empty shards")
    base, extra = divmod(T, G)
    out, first = [], 0
    for g in range(G):
        count = base + (1 if g < extra else 0)
        out.append((first, count))
        first += count
    return out


class TShardedSegNet:
    """One rank of a T-sharded SegNet.  Every rank of `group` (default: the initialised process group, or none: a single
    rank) constructs one (same model, seed, T and precision) and calls segment_device once per frame, in the same order; the
    frame counters stay in lockstep because every rank runs one partial per frame.  Results appear on the group's rank 0 (the
    root).  Each rank recomputes the sample-invariant prefix: broadcasting its activations would not shorten the critical path."""

    def __init__(self, params: BayesianSegNetParams, T: int, device: int, seed: int = 1234, precision: str = "fp16",
                 engine: str = "auto", group=None):
        import torch
        import torch.distributed as dist
        self._dist, self._torch = dist, torch
        self.group = group
        if dist.is_available() and dist.is_initialized():
            self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
            self.root = dist.get_global_rank(group, 0) if group is not None else 0
        else:  # no process group: one rank holding all T samples
            self.rank, self.world, self.root = 0, 1, 0
        self.is_root = self.rank == 0
        self.samples = shard_ranges(T, self.world)[self.rank]
        self.seg = BayesianSegNet(params, device=device, seed=seed, T=T, precision=precision, engine=engine, samples=self.samples)
        self.T, self.width, self.height, self.n_classes = self.seg.T, self.seg.width, self.seg.height, self.seg.n_classes
        self.device = torch.device("cuda", device)
        hw = self.width * self.height
        self.sums = torch.empty((self.n_classes, hw), dtype=torch.float64, device=self.device)
        self._bgr = torch.empty((self.height, self.width, 3), dtype=torch.uint8, device=self.device)
        # the frame's work runs on one stream of its own, ordered after the caller's current stream and before what the caller
        # issues next (the library would take stream 0, torch's default stream, as "the handle's own stream")
        self.stream = torch.cuda.Stream(self.device)
        torch.cuda.synchronize(self.device)

    def set_frame(self, frame: int):
        """Sets the dropout frame counter; call it on every rank with the same value."""
        self.seg.set_frame(frame)

    def semantic_keys(self, kps, max_static_class: int = 8):
        """On the root: BayesianSegNet.semantic_keys on the last finalized maps."""
        return self.seg.semantic_keys(kps, max_static_class)

    def segment_device(self, bgr=None, classes=None, conf=None, ent=None, conf32=None, ent32=None, events: Optional[list] = None):
        """One frame.  bgr: on the root, the cropped height x width x 3 uint8 image on this rank's device (ignored elsewhere).
        The outputs (device tensors of H*W elements; allocated when None) are written on the root, which gets
        (classes, conf, ent); other ranks get None.  `events`: five CUDA events recorded on the current stream before the
        broadcast and after the broadcast, the partial, the reduce and the finalize (the last two only on the root); the work
        is ordered after everything issued on the caller's current stream and before what it issues next."""
        torch = self._torch
        if self.is_root and (bgr is None or tuple(bgr.shape) != (self.height, self.width, 3) or bgr.dtype != torch.uint8
                             or bgr.device != self.device):
            raise ValueError(f"segment_device: the root needs a {self.height}x{self.width}x3 uint8 image on {self.device}")
        caller = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(caller)
        with torch.cuda.stream(self.stream):
            out = self._frame(bgr, classes, conf, ent, conf32, ent32, events)
        caller.wait_stream(self.stream)
        return out

    def _frame(self, bgr, classes, conf, ent, conf32, ent32, events):
        torch, dist = self._torch, self._dist
        stream = self.stream
        hw = self.width * self.height
        buf = self._bgr
        if self.is_root:
            if bgr.is_contiguous():
                buf = bgr
            else:
                buf.copy_(bgr)
        if events:
            events[0].record(stream)
        if self.world > 1:
            dist.broadcast(buf, self.root, group=self.group)
        if events:
            events[1].record(stream)
        self.seg.run_device_partial(buf.data_ptr(), self.sums.data_ptr(), False, stream.cuda_stream)
        if events:
            events[2].record(stream)
        if self.world > 1:
            dist.reduce(self.sums, self.root, op=dist.ReduceOp.SUM, group=self.group)
        if not self.is_root:
            return None
        if events:
            events[3].record(stream)
        if classes is None:
            classes = torch.empty(hw, dtype=torch.uint8, device=self.device)
        if conf is None:
            conf = torch.empty(hw, dtype=torch.float64, device=self.device)
        if ent is None:
            ent = torch.empty(hw, dtype=torch.float64, device=self.device)
        ptr = lambda t: 0 if t is None else t.data_ptr()
        self.seg.finalize_device(self.sums.data_ptr(), ptr(classes), ptr(conf), ptr(ent), ptr(conf32), ptr(ent32), stream.cuda_stream)
        if events:
            events[4].record(stream)
        return classes, conf, ent
