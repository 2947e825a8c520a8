// Launch wrappers of the SegNet layer kernels.  Activations are NHWC ("pixel-major": the channel
// vector of one pixel is contiguous) in half (default) or float (strict mode); `cs` is the channel
// stride in elements (4 for the 3-channel input, 16 for the 15 logits, C otherwise).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace sivo {

enum class DType : int { F16 = 0, F32 = 1 };
inline size_t dtype_size(DType t) { return t == DType::F16 ? 2 : 4; }

struct TensorView {
  void* p = nullptr;
  int n = 0, c = 0, h = 0, w = 0, cs = 0;
  DType dt = DType::F16;
  size_t elems() const { return static_cast<size_t>(n) * h * w * cs; }
  size_t bytes() const { return elems() * dtype_size(dt); }
};

struct ConvParams {
  TensorView in, out;
  const float* w_simt = nullptr;   // [k*k][cin_p][cout_p] float
  const float* bias = nullptr;     // [cout_p]
  const float* bn_scale = nullptr; // [cout_p] or null
  const float* bn_shift = nullptr;
  int k = 0, pad = 0, cin_p = 0, cout_p = 0;
  int relu = 0;
  float slope = 0.f;
};

// What changes from frame to frame, in device memory, so that ONE captured CUDA graph serves every call: the dropout frame
// counter and the caller's image / result pointers.  run_device() overwrites it by value (k_set_frame_args, outside the graph);
// the kernels that touch caller memory (input conversion, MC reduction) read their pointers from it.
struct FrameArgs {
  uint64_t frame;        // first member: DropoutParams::frame_dev points here
  const uint8_t* bgr;
  uint8_t* classes;
  double* conf;
  double* ent;
  float* conf32;         // optional single-precision copies of the two maps (the packed multi-GPU record carries those)
  float* ent32;
  double* prob_sum;      // partial runs (sample shards): [C][H*W] per-pixel sums of this handle's softmax probabilities
  int accumulate;        // 0: the partial run overwrites prob_sum, 1: adds to it
};

struct DropoutParams {
  uint64_t seed = 0;
  const uint64_t* frame_dev = nullptr;  // device scalar, so a captured graph replays with a new frame
  int layer = 0;
  int sample0 = 0;  // global index of the handle's first Monte-Carlo sample (sample shards); the keep bits use sample0 + n
};

// `args` != nullptr: the image / result pointers are read from *args on the device instead of the by-value arguments
void launch_input_u8(const uint8_t* bgr_hwc, TensorView out, cudaStream_t s, const FrameArgs* args = nullptr);
void launch_lrn(TensorView in, TensorView out, int size, float alpha, float beta, float k, cudaStream_t s);
void launch_conv_simt(const ConvParams& p, cudaStream_t s);
// 4-channel input -> K*blk-channel tap-expanded tensor (see k_expand_taps)
void launch_expand_taps(TensorView in, TensorView out, int K, int blk, cudaStream_t s);
// [N][H][W][4] half -> zero-padded [N][H][W + 8][8] half (3 zero pixels left, 5 right, channels 4..7 zero)
void launch_dropout_unpool(TensorView in, int T, const uint8_t* mask, int mask_n, TensorView out, const DropoutParams& d, float scale,
                           cudaStream_t s);
// per-keypoint gather from the three result maps (Frame.cc:181-186 indexing); out-of-map keypoints get (255, 0, 0)
void launch_keypoint_lookup(const sivo_keypoint* kps, int n, const uint8_t* classes, const double* conf, const double* ent, int H, int W,
                            uint8_t* out_class, double* out_conf, double* out_ent, cudaStream_t s);
void launch_pad8(TensorView in, TensorView out, cudaStream_t s);
// the three steps input_u8 -> lrn -> pad8 in one pass (same arithmetic, so the same half values)
void launch_input_lrn_pad8(const uint8_t* bgr, TensorView out, int size, float alpha, float beta, float k, cudaStream_t s,
                           const FrameArgs* args = nullptr);
// float [px][C] -> half [px][hi C | lo C] (split-operand fp32 mode of the tensor-core convolution)
void launch_split_hilo(TensorView in, void* out_half, cudaStream_t s);
// *dst = v on stream s, the value passed as a kernel argument
void launch_set_frame_args(FrameArgs* dst, const FrameArgs& v, cudaStream_t s);
void launch_pool(TensorView in, TensorView out, uint8_t* mask, cudaStream_t s);
// mask_n: batch of the mask tensor (1 when the pool ran in the sample-invariant prefix)
void launch_unpool(TensorView in, const uint8_t* mask, int mask_n, TensorView out, cudaStream_t s);
// in.n may be 1 (broadcast to out.n samples)
void launch_dropout(TensorView in, TensorView out, const DropoutParams& d, float scale, cudaStream_t s);
// logits: float [T, H, W, 16]
// pix0 / npix restrict the pass to pixels [pix0, pix0 + npix) (npix < 0: all of them)
void launch_mc_reduce(const float* logits, int T, int C, int cs, int hw, uint8_t* classes, double* conf,
                      double* entropy, cudaStream_t s, int pix0 = 0, int npix = -1, const FrameArgs* args = nullptr);
// The reduction split in two for sample shards.  partial: prob_sum[c * hw + p] (+)= sum over the n samples of `logits` (float
// [n, H, W, 16]) of the softmax probabilities, in double and in sample order (accumulate = 0 starts from 0).  finalize: the
// three maps (and optional f32 copies) from the sums of all T samples.  Partial over [0, T) + finalize is bitwise
// launch_mc_reduce.  `args` != nullptr: prob_sum / accumulate (partial) or the map pointers (finalize) come from *args.
void launch_mc_partial(const float* logits, int n, int C, int cs, int hw, double* prob_sum, int accumulate, cudaStream_t s,
                       const FrameArgs* args = nullptr);
void launch_mc_finalize(const double* prob_sum, int T, int C, int hw, uint8_t* classes, double* conf, double* entropy, float* conf32,
                        float* ent32, cudaStream_t s);
void launch_dropout_bits(uint64_t seed, const uint64_t* frame_dev, int layer, int T, int C, int H, int W,
                         uint8_t* keep_nchw, cudaStream_t s);
// layout converters for the test hooks (float NCHW host order <-> NHWC activation)
void launch_nchw_to_act(const float* src, TensorView dst, cudaStream_t s);
void launch_act_to_nchw(TensorView src, float* dst, cudaStream_t s);
void launch_mask_to_nchw(const uint8_t* mask, int n, int c, int ho, int wo, int* dst, cudaStream_t s);
void launch_mask_from_nchw(const int* src, int n, int c, int ho, int wo, uint8_t* mask, cudaStream_t s);

}  // namespace sivo
