"""Python mirror of `SIVO::BayesianSegNet` (include/bayesian_segnet/bayesian_segnet.hpp:108-170) over the
C-ABI: same names, argument meaning and error behaviour, so the parity tests read like the reference's
tests/test_bayesian_segnet.cpp."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _lib as L


@dataclass
class BayesianSegNetParams:
    """bayesian_segnet.hpp:85-105."""
    model_file: str = ""
    weights_file: str = ""
    use_gpu: bool = True  # kept for signature parity; this backend is GPU only


class BayesianSegNet:
    def __init__(self, params: BayesianSegNetParams, device: int = 0, seed: int = 1234, T: int = 0,
                 precision: str = "fp16", engine: str = "auto", keep_blobs: bool = False, samples: Optional[tuple] = None):
        """samples = (first, count): a sample shard that computes Monte-Carlo samples [first, first + count) of T with the
        dropout masks an unsharded handle draws for them (run_device_partial / finalize_device; segmentImage and run_device
        refuse unless the shard covers all T samples)."""
        self._h = C.c_void_p()
        opt = L.SegnetOptions(device=device, T=T, seed=seed,
                              precision={"fp16": L.PRECISION_FP16, "fp32": L.PRECISION_FP32}[precision],
                              engine={"auto": L.ENGINE_AUTO, "simt": L.ENGINE_SIMT, "tcgen05": L.ENGINE_TCGEN05}[engine],
                              keep_blobs=int(keep_blobs), reserved=0)
        if samples is None:
            rc = L.lib().sivo_segnet_create_ex(params.model_file.encode(), params.weights_file.encode(), C.byref(opt),
                                               C.byref(self._h))
        else:
            first, count = (int(v) for v in samples)
            rc = L.lib().sivo_segnet_create_shard(params.model_file.encode(), params.weights_file.encode(), C.byref(opt),
                                                  first, count, C.byref(self._h))
        if rc == L.EINVAL:  # the reference throws std::invalid_argument (bayesian_segnet.cpp:66,68,82,86)
            raise ValueError(L.lib().sivo_last_error().decode())
        L.check(rc)
        w, h, t, nc = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        L.check(L.lib().sivo_segnet_geometry(self._h, C.byref(w), C.byref(h), C.byref(t), C.byref(nc)))
        self.width, self.height, self.T, self.n_classes = w.value, h.value, t.value, nc.value
        self.samples = (0, self.T) if samples is None else (first, count)

    def __del__(self):
        if getattr(self, "_h", None) and self._h.value and L is not None and getattr(L, "lib", None):
            try:
                L.lib().sivo_segnet_destroy(self._h)
            except Exception:  # interpreter shutdown: module globals may already be gone
                pass
            self._h = C.c_void_p()

    def getInputGeometry(self):
        return (self.width, self.height)  # cv::Size(width, height)

    def set_frame(self, frame: int):
        L.check(L.lib().sivo_segnet_set_frame(self._h, C.c_uint64(frame)))

    def set_profiling(self, on: bool):
        L.check(L.lib().sivo_segnet_set_profiling(self._h, int(on)))

    def segmentImage(self, image: np.ndarray, out=None):
        """image: HxWx3 u8 BGR.  Returns (classes u8 [H,W], confidence f64 [H,W], entropy f64 [H,W]).
        `out` = (classes, confidence, entropy) reuses caller buffers (like the Eigen matrices the C++ shim resizes
        once); page-locked buffers receive the device copies directly."""
        if image.dtype != np.uint8 or image.ndim != 3 or image.shape[2] != 3:
            raise ValueError("segmentImage expects an HxWx3 uint8 BGR image")
        if image.strides[2] != 1 or image.strides[1] != 3:
            image = np.ascontiguousarray(image)
        if out is not None:
            classes, conf, ent = out
            assert classes.shape == conf.shape == ent.shape == (self.height, self.width)
            assert classes.dtype == np.uint8 and conf.dtype == np.float64 and ent.dtype == np.float64
            assert classes.flags.c_contiguous and conf.flags.c_contiguous and ent.flags.c_contiguous
        else:
            classes = np.empty((self.height, self.width), np.uint8)
            conf = np.empty((self.height, self.width), np.float64)
            ent = np.empty((self.height, self.width), np.float64)
        L.check(L.lib().sivo_segnet_run(self._h, image.ctypes.data_as(C.c_void_p), image.shape[0], image.shape[1],
                                        C.c_size_t(image.strides[0]), classes.ctypes.data_as(C.c_void_p),
                                        conf.ctypes.data_as(C.c_void_p), ent.ctypes.data_as(C.c_void_p)))
        return classes, conf, ent

    def segment_on_device(self, image: np.ndarray):
        """segmentImage without the read-back: the three maps stay on the device for semantic_keys()."""
        if image.dtype != np.uint8 or image.ndim != 3 or image.shape[2] != 3:
            raise ValueError("segmentImage expects an HxWx3 uint8 BGR image")
        if image.strides[2] != 1 or image.strides[1] != 3:
            image = np.ascontiguousarray(image)
        L.check(L.lib().sivo_segnet_run(self._h, image.ctypes.data_as(C.c_void_p), image.shape[0], image.shape[1],
                                        C.c_size_t(image.strides[0]), None, None, None))

    def semantic_keys(self, kps: np.ndarray, max_static_class: int = 8):
        """Frame::SelectSemanticKeys (Frame.cc:177-203) + per-keypoint map reads on the device-resident result of the last
        run.  kps: structured array (orb.KP_DTYPE).  Returns (classes u8 [n], confidence f64 [n], entropy f64 [n], keep int32 [m]):
        keep = indices whose class <= max_static_class (Classes::TERRAIN), in keypoint order."""
        kps = np.ascontiguousarray(kps)
        if kps.dtype.itemsize != 28:
            raise ValueError("keypoints must be the 28-byte sivo_keypoint records")
        n = len(kps)
        cls = np.empty(n, np.uint8)
        conf = np.empty(n, np.float64)
        ent = np.empty(n, np.float64)
        keep = np.empty(max(n, 1), np.int32)
        m = C.c_int(0)
        L.check(L.lib().sivo_segnet_semantic_keys(self._h, kps.ctypes.data_as(C.c_void_p), n, int(max_static_class),
                                                  cls.ctypes.data_as(C.c_void_p), conf.ctypes.data_as(C.c_void_p),
                                                  ent.ctypes.data_as(C.c_void_p), keep.ctypes.data_as(C.c_void_p), C.byref(m)))
        return cls, conf, ent, keep[:m.value].copy()

    def run_device(self, bgr_ptr: int, classes_ptr: int, conf_ptr: int, ent_ptr: int, stream: int = 0):
        L.check(L.lib().sivo_segnet_run_device(self._h, C.c_void_p(bgr_ptr), C.c_void_p(classes_ptr), C.c_void_p(conf_ptr),
                                               C.c_void_p(ent_ptr), C.c_void_p(stream)))

    def set_record_outputs(self, classes_ptr: int = 0, conf32_ptr: int = 0, ent32_ptr: int = 0):
        """segmentImage additionally leaves classes + f32 maps at these device addresses (a packed multi-GPU record); 0s: off."""
        L.check(L.lib().sivo_segnet_set_record_outputs(self._h, C.c_void_p(classes_ptr), C.c_void_p(conf32_ptr), C.c_void_p(ent32_ptr)))

    def run_device_maps(self, bgr_ptr: int, classes_ptr: int, conf_ptr: int, ent_ptr: int, conf32_ptr: int, ent32_ptr: int, stream: int = 0):
        """run_device plus single-precision copies of the two maps (the packed multi-GPU record's layout); any pointer may be 0."""
        L.check(L.lib().sivo_segnet_run_device_maps(self._h, C.c_void_p(bgr_ptr), C.c_void_p(classes_ptr), C.c_void_p(conf_ptr),
                                                    C.c_void_p(ent_ptr), C.c_void_p(conf32_ptr), C.c_void_p(ent32_ptr), C.c_void_p(stream)))

    def run_device_partial(self, bgr_ptr: int, sum_ptr: int, accumulate: bool = False, stream: int = 0):
        """This handle's samples of one frame: sum_ptr (n_classes x H*W doubles) receives (accumulate: gains) the per-pixel
        sums of their softmax probabilities.  Advances the frame counter."""
        L.check(L.lib().sivo_segnet_run_device_partial(self._h, C.c_void_p(bgr_ptr), C.c_void_p(sum_ptr), int(bool(accumulate)),
                                                       C.c_void_p(stream)))

    def finalize_device(self, sum_ptr: int, classes_ptr: int, conf_ptr: int, ent_ptr: int, conf32_ptr: int = 0, ent32_ptr: int = 0,
                        stream: int = 0):
        """classes / confidence / entropy (+ f32 copies) from the probability sums of all T samples; any output may be 0.
        The maps become the result semantic_keys reads."""
        L.check(L.lib().sivo_segnet_finalize_device(self._h, C.c_void_p(sum_ptr), C.c_void_p(classes_ptr), C.c_void_p(conf_ptr),
                                                    C.c_void_p(ent_ptr), C.c_void_p(conf32_ptr), C.c_void_p(ent32_ptr),
                                                    C.c_void_p(stream)))

    def blob(self, name: str) -> np.ndarray:
        n, c, h, w = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        L.check(L.lib().sivo_segnet_blob(self._h, name.encode(), None, C.c_size_t(0), C.byref(n), C.byref(c), C.byref(h), C.byref(w)))
        out = np.empty((n.value, c.value, h.value, w.value), np.float32)
        L.check(L.lib().sivo_segnet_blob(self._h, name.encode(), out.ctypes.data_as(C.c_void_p), C.c_size_t(out.size),
                                         None, None, None, None))
        return out

    def op_flops_executed(self):
        """Executed conv flops per launch (== algorithmic except for the composed classifier and the split-operand mode)."""
        n = C.c_int()
        L.check(L.lib().sivo_segnet_op_timing(self._h, -1, None, 0, None, None, C.byref(n)))
        out = []
        for i in range(n.value):
            fl = C.c_double()
            L.check(L.lib().sivo_segnet_op_flops_executed(self._h, i, C.byref(fl)))
            out.append(fl.value)
        return out

    def op_timings(self):
        """[(layer names, ms in the last profiled run, algorithmic conv flops)] per launch of the op list."""
        n = C.c_int()
        L.check(L.lib().sivo_segnet_op_timing(self._h, -1, None, 0, None, None, C.byref(n)))
        out = []
        for i in range(n.value):
            buf = C.create_string_buffer(256)
            ms, fl = C.c_float(), C.c_double()
            L.check(L.lib().sivo_segnet_op_timing(self._h, i, buf, 256, C.byref(ms), C.byref(fl), None))
            out.append((buf.value.decode(), ms.value, fl.value))
        return out

    def last_timing(self):
        a, b, c, d, n = C.c_float(), C.c_float(), C.c_float(), C.c_float(), C.c_int()
        L.check(L.lib().sivo_segnet_last_timing(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d), C.byref(n)))
        return {"conv_ms": a.value, "other_ms": b.value, "reduce_ms": c.value, "total_ms": d.value, "launches": n.value}

    def flops(self):
        a, b = C.c_double(), C.c_double()
        L.check(L.lib().sivo_segnet_flops(self._h, C.byref(a), C.byref(b)))
        return {"dedup": a.value, "naive": b.value}
