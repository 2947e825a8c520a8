// Bayesian SegNet executor: prototxt + caffemodel -> a static list of device ops over NHWC tensors.
// Host-side twin of `SIVO::BayesianSegNet` (src/bayesian_segnet/bayesian_segnet.cpp).
#pragma once
#include <cuda_fp16.h>

#include <map>
#include <memory>
#include <string>
#include <vector>

#include "caffemodel.h"
#include "common.h"
#include "prototxt.h"
#include "segnet_kernels.h"

namespace sivo {

struct ConvTcPlan;  // conv_tc.cu

struct Tensor {
  std::string name;
  TensorView v;
  DevBuf buf;
  bool is_mask = false;  // u8 2-bit argmax codes, dims = pooled dims
  bool elided = false;   // a fusion consumes this blob in registers: it is never written (blob() refuses to read it)
};

struct Op {
  enum Kind { Input, LRN, Expand, InputPad8, DropoutUnpool, Conv, Pool, Unpool, Dropout, Reduce } kind = Input;
  std::string layer;
  int in = -1, in2 = -1, out = -1, out2 = -1;
  // LRN
  int lrn_size = 5;
  float lrn_alpha = 1.f, lrn_beta = 0.75f, lrn_k = 1.f;
  // Conv
  int k = 0, pad = 0, cin = 0, cout = 0, cin_p = 0, cout_p = 0;
  std::vector<float> h_w_raw;  // the caffemodel's (cout, cin, k, k) floats, unrounded (composed-classifier experiment)
  std::vector<float> h_bias, h_bn_scale, h_bn_shift, h_w;  // host copies (the tensor-core kernels take them as kernel parameters)
  int fold_kw = 0;                  // > 0: KxK conv over 3 channels run as a Kx1 conv over the window-folded padded input (conv_tc.cu)
  int expand_k = 0, expand_blk = 0;  // > 0: a KxK conv over 3 channels run as a 1x1 conv over the tap-expanded input
  bool relu = false, has_bn = false;
  float slope = 0.f;
  DevBuf w_simt, w_tc, w_tc_pair, bias, bn_scale, bn_shift;  // w_tc_pair: [kw][kh][cout][cin] half for the paired-tap kernel
  // split-operand fp32 mode (precision fp32 on the tcgen05 engine): x = hi + lo and w * 2^s = hi + lo in half, and
  // x * w ~= (x_hi w_hi + x_hi w_lo + x_lo w_hi) * 2^-s accumulated in fp32 -- three MMAs per tap, ~2^-22 relative per product.
  // w_tc holds [tap][cout_p][3 cin_p] = per 64-channel chunk [W_hi | W_lo | W_hi]; a_split the [hi Cin | lo Cin] planes of the input.
  bool split = false;
  float acc_scale = 1.f;
  DevBuf a_split;
  std::shared_ptr<ConvTcPlan> tc;
  bool use_tc = false;
  // batch the tensor-core plan picks its kernel variant for (0: the input's own).  A sample shard plans its per-sample layers
  // for all T samples, so that each sample's accumulation order -- and hence its logits -- is the unsharded handle's
  int plan_n = 0;
  double flops = 0;       // algorithmic (the reference's operation count), for this op's batch
  double flops_exec = 0;  // what the launch executes: differs for the composed classifier (0.25x) and the split-operand mode (3x)
  // Dropout
  int drop_layer = 0;
  float drop_scale = 2.f;
};

class SegNet {
 public:
  // n_samples < 0: all T samples.  Otherwise the handle computes samples [first_sample, first_sample + n_samples) of T (a
  // sample shard): the op list after the first sampling Dropout has batch n_samples, and its dropout keys use the global index
  SegNet(const std::string& prototxt, const std::string& caffemodel, const sivo_segnet_options& opt, int first_sample = 0,
         int n_samples = -1);
  ~SegNet();
  int width() const { return W_; }
  int height() const { return H_; }
  int T() const { return T_; }
  int first_sample() const { return s0_; }
  int n_samples() const { return n_; }
  int classes() const { return n_classes_; }
  void set_frame(uint64_t f) { frame_ = f; }
  void run_host(const uint8_t* bgr, int rows, int cols, size_t stride, uint8_t* classes, double* conf, double* ent);
  // segmentImage (run_host) additionally leaves the classes and f32 copies of the two maps at these device addresses, complete
  // when it returns (all NULL: off)
  void set_record_outputs(uint8_t* classes_dev, float* conf32_dev, float* ent32_dev) {
    rec_classes_ = classes_dev; rec_conf32_ = conf32_dev; rec_ent32_ = ent32_dev;
  }
  // conf32 / ent32 (optional): single-precision copies of the two maps, e.g. straight into the packed multi-GPU record
  void run_device(const uint8_t* bgr_dev, uint8_t* classes_dev, double* conf_dev, double* ent_dev, cudaStream_t s, float* conf32_dev = nullptr,
                  float* ent32_dev = nullptr);
  // sample shards: the op list with the MC reduction replaced by the per-pixel double sums of this handle's softmax
  // probabilities, prob_sum[c * H*W + p] (accumulate: add to what is there); advances the frame counter like run_device
  void run_device_partial(const uint8_t* bgr_dev, double* prob_sum_dev, int accumulate, cudaStream_t s);
  // the maps from the summed probabilities of all T samples; they become the last result (semantic_keys)
  void finalize_device(const double* prob_sum_dev, uint8_t* classes_dev, double* conf_dev, double* ent_dev, float* conf32_dev,
                       float* ent32_dev, cudaStream_t s);
  void semantic_keys(const sivo_keypoint* kps, int n, int max_static_class, uint8_t* kp_class, double* kp_conf, double* kp_entropy,
                     int* keep_idx, int* n_keep);
  void blob(const std::string& name, float* out, size_t cap, int* n, int* c, int* h, int* w);
  void set_profiling(bool on) { profiling_ = on; }
  float conv_ms = 0, other_ms = 0, reduce_ms = 0, total_ms = 0;
  std::vector<float> op_ms;  // per launch of the last profiled run, in launch order
  size_t n_ops() const { return ops_.size(); }
  const Op& op_at(size_t i) const { return ops_[i]; }
  int launches = 0;
  double flops_dedup = 0, flops_naive = 0;

 private:
  int add_tensor(const std::string& name, int n, int c, int h, int w, int cs, DType dt, bool mask = false);
  void build(const NetSpec& net, const WeightMap& weights);
  void prepare_conv(Op& op, const std::vector<Blob>& conv_blobs, const std::vector<Blob>* bn_blobs);
  void enqueue(const uint8_t* bgr_dev, uint8_t* classes_dev, double* conf_dev, double* ent_dev, cudaStream_t s, bool timed);
  void run_frame(const FrameArgs& fa, cudaStream_t s);
  void require_whole(const char* what) const;  // refuses whole-frame calls on a shard that holds only part of the T samples

  sivo_segnet_options opt_;
  int device_ = 0, T_ = 0, H_ = 0, W_ = 0, n_classes_ = 0;
  int s0_ = 0, n_ = 0;  // this handle's samples [s0_, s0_ + n_) of T_ (n_ == T_ unless it is a sample shard)
  DType act_ = DType::F16;
  uint64_t frame_ = 0;
  bool profiling_ = false;
  std::vector<std::unique_ptr<Tensor>> tensors_;
  std::map<std::string, int> by_name_;
  std::vector<Op> ops_;
  std::vector<Op> fused_;  // ops folded into a neighbour's epilogue; kept alive for their weight buffers
  cudaStream_t stream_ = nullptr;
  DevBuf d_bgr_, d_classes_, d_conf_, d_ent_, d_frame_;
  PinnedBuf h_in_, h_classes_, h_conf_, h_ent_;
  // where the last run left its maps on the device, and the stream it ran on (semantic_keys reads them)
  const uint8_t* last_classes_ = nullptr;
  const double* last_conf_ = nullptr;
  const double* last_ent_ = nullptr;
  cudaStream_t last_stream_ = nullptr;
  DevBuf d_kp_, d_kp_out_;
  PinnedBuf h_kp_, h_kp_out_;
  std::vector<cudaEvent_t> events_;
  // the op list captured once as a CUDA graph (one launch per frame); re-captured if the buffers or the stream change
  // captured op lists, one per (input, outputs, stream) pointer set the caller has used; most recently used first
  struct GraphEntry { const void* key[5]; cudaGraphExec_t exec; };
  std::vector<GraphEntry> graphs_;
  static constexpr size_t kMaxGraphs = 32;
  bool graph_ok_ = true;
  // segmentImage read-back overlap: the MC reduction runs in row bands and each band's slices of the three maps start their
  // device-to-host copy on a second stream while the next band is reduced
  bool skip_reduce_ = false;      // set by run_host around run_device: the op list stops before the Reduce op
  bool partial_ = false;          // set by run_device_partial: the Reduce op writes the probability sums (FrameArgs::prob_sum)
  cudaStream_t copy_stream_ = nullptr;
  std::vector<cudaEvent_t> band_ev_;
  // device-resident copies run_host leaves for a packed multi-GPU record (set_record_outputs)
  uint8_t* rec_classes_ = nullptr;
  float* rec_conf32_ = nullptr;
  float* rec_ent32_ = nullptr;
};

// conv_tc.cu -- tcgen05 implicit-GEMM convolution
bool conv_tc_supported(const Op& op, const TensorView& in, const TensorView& out);
std::shared_ptr<ConvTcPlan> conv_tc_plan(const Op& op, const TensorView& in, const TensorView& out, const void* w_tc);
void conv_tc_launch(const ConvTcPlan& plan, const Op& op, cudaStream_t s);
// fuses the sampling Dropout that follows the convolution in place into its epilogue; batch image i is sample sample0 + i
void conv_tc_set_dropout(ConvTcPlan& plan, uint64_t seed, const uint64_t* frame_dev, int layer, int sample0, float scale);
// fuses the max-unpool (Upsample) that consumes the convolution's output into its epilogue; `out_2h_2w` is the
// unpooled tensor the convolution then writes instead of its own output
void conv_tc_set_unpool(ConvTcPlan& plan, const uint8_t* mask, int mask_n, void* out_2h_2w);
// fuses the 2x2/2 max pool (+ argmax mask) that consumes the convolution's output into its epilogue
bool conv_tc_can_fuse_pool(const ConvTcPlan& plan);
void conv_tc_set_pool(ConvTcPlan& plan, void* pooled, uint8_t* mask);
// fuses a following 1x1 convolution to <= 16 float logits (the layer feeding Softmax) into the epilogue
bool conv_tc_can_fuse_classifier(const ConvTcPlan& plan);
// host-side weight layout of the split-operand fp32 mode: [tap][cout_p][3 cin_p] half + the accumulator scale 2^-s
std::vector<__half> conv_tc_split_weights(const float* w_cout_cin_k_k, int cout, int cin, int K, int cout_p, int cin_p, float* acc_scale);
// host-side weight layout of the paired-tap kernel (64 -> 64 channels)
std::vector<__half> conv_tc_pair_weights(const float* w_cout_cin_k_k, int K);
// Experimental (SIVO_B200_COMPOSE=1): conv (64 -> 64, 7x7, no BN / ReLU) followed by the 1x1 classifier run as ONE 64 -> 16
// convolution with composed weights; logits come straight from the accumulators.  wc = [n_cls][64], bc = [n_cls] (host).
bool conv_tc_can_compose_classifier(const ConvTcPlan& plan);
void conv_tc_set_composed_classifier(ConvTcPlan& plan, const Op& conv, const float* wc, const float* bc, int n_cls, float* logits);
void conv_tc_set_classifier(ConvTcPlan& plan, const float* w_cin_by_cout, int stride, const float* bias, int n_bias, float* logits);  // host pointers

}  // namespace sivo
