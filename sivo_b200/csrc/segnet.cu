// Host side of the Bayesian SegNet operator: builds the op list from the prototxt (fusing the in-place
// BN / ReLU followers into their convolution, running everything upstream of the first sampling Dropout
// once instead of T times) and executes it on one stream.
#include "segnet.h"

#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

namespace sivo {

namespace {
int round_up(int a, int b) { return (a + b - 1) / b * b; }
float through_half(float x) { return __half2float(__float2half_rn(x)); }
}  // namespace

int SegNet::add_tensor(const std::string& name, int n, int c, int h, int w, int cs, DType dt, bool mask) {
  auto t = std::make_unique<Tensor>();
  t->name = name;
  t->v.n = n; t->v.c = c; t->v.h = h; t->v.w = w; t->v.cs = cs; t->v.dt = dt;
  t->is_mask = mask;
  size_t bytes = mask ? static_cast<size_t>(n) * h * w * cs : t->v.bytes();
  t->buf.alloc(bytes);
  t->v.p = t->buf.p;
  tensors_.push_back(std::move(t));
  int id = static_cast<int>(tensors_.size()) - 1;
  by_name_[name] = id;
  return id;
}

void SegNet::prepare_conv(Op& op, const std::vector<Blob>& cb, const std::vector<Blob>* bn) {
  // K is the layer's kernel size; a tap-expanded layer (expand_k > 0) stores it as one tap over expand_k*blk channels
  const int K = op.expand_k ? op.expand_k : op.k, cin = (op.expand_k || op.fold_kw) ? 3 : op.cin, cout = op.cout;
  const int taps = op.expand_k ? 1 : op.fold_kw ? K : K * K;
  auto slot = [&](int t, int ci, int& tap, int& cidx) {
    if (op.expand_k) { tap = 0; cidx = (t / K) * op.expand_blk + (t % K) * 4 + ci; }
    // tap row kh; "channel" = window pixel * 8 + c.  The window of output pixel x starts at image pixel x - 3, tap column
    // kw reads image pixel x + kw - (K-1)/2, i.e. window pixel kw + 3 - (K-1)/2
    else if (op.fold_kw) { tap = t / K; cidx = (t % K + 3 - (K - 1) / 2) * 8 + ci; }
    else { tap = t; cidx = ci; }
  };
  if (cb.empty() || cb[0].shape.size() != 4 || cb[0].shape[0] != cout || cb[0].shape[1] != cin || cb[0].shape[2] != K ||
      cb[0].shape[3] != K)
    fail(SIVO_EFORMAT, "layer '%s': weight blob shape does not match (%d,%d,%d,%d) (net.cpp:750-785 would CHECK-fail)",
         op.layer.c_str(), cout, cin, K, K);
  const bool half = act_ == DType::F16;
  const float* W = cb[0].data.data();
  std::vector<float> ws(static_cast<size_t>(taps) * op.cin_p * op.cout_p, 0.f);
  for (int co = 0; co < cout; ++co)
    for (int ci = 0; ci < cin; ++ci)
      for (int t = 0; t < K * K; ++t) {
        float v = W[(static_cast<size_t>(co) * cin + ci) * K * K + t];
        int tap, cidx;
        slot(t, ci, tap, cidx);
        ws[(static_cast<size_t>(tap) * op.cin_p + cidx) * op.cout_p + co] = half ? through_half(v) : v;
      }
  op.h_w = ws;
  op.h_w_raw.assign(W, W + static_cast<size_t>(cout) * cin * K * K);
  op.w_simt.alloc(ws.size() * sizeof(float));
  SIVO_CUDA(cudaMemcpy(op.w_simt.p, ws.data(), ws.size() * sizeof(float), cudaMemcpyHostToDevice));
  if (half) {  // tensor-core layout: [tap][cout_p][cin_p] half, K(=cin)-major rows
    std::vector<__half> wt(static_cast<size_t>(taps) * op.cout_p * op.cin_p, __float2half_rn(0.f));
    for (int co = 0; co < cout; ++co)
      for (int ci = 0; ci < cin; ++ci)
        for (int t = 0; t < K * K; ++t) {
          int tap, cidx;
          slot(t, ci, tap, cidx);
          wt[(static_cast<size_t>(tap) * op.cout_p + co) * op.cin_p + cidx] =
              __float2half_rn(W[(static_cast<size_t>(co) * cin + ci) * K * K + t]);
        }
    op.w_tc.alloc(wt.size() * sizeof(__half));
    SIVO_CUDA(cudaMemcpy(op.w_tc.p, wt.data(), wt.size() * sizeof(__half), cudaMemcpyHostToDevice));
    if (!op.expand_k && (K == 7 || K == 3) && cin == 64 && cout == 64 && op.cin_p == 64 && op.cout_p == 64) {
      std::vector<__half> wp = conv_tc_pair_weights(W, K);
      op.w_tc_pair.alloc(wp.size() * sizeof(__half));
      SIVO_CUDA(cudaMemcpy(op.w_tc_pair.p, wp.data(), wp.size() * sizeof(__half), cudaMemcpyHostToDevice));
    }
  }
  if (op.split) {
    if (taps != K * K) fail(SIVO_EINVAL, "layer '%s': split-operand mode does not take folded / expanded first layers", op.layer.c_str());
    std::vector<__half> wt = conv_tc_split_weights(W, cout, cin, K, op.cout_p, op.cin_p, &op.acc_scale);
    op.w_tc.alloc(wt.size() * sizeof(__half));
    SIVO_CUDA(cudaMemcpy(op.w_tc.p, wt.data(), wt.size() * sizeof(__half), cudaMemcpyHostToDevice));
  }
  std::vector<float> b(op.cout_p, 0.f);
  if (cb.size() > 1) {
    if (static_cast<int>(cb[1].count()) != cout) fail(SIVO_EFORMAT, "layer '%s': bias blob size mismatch", op.layer.c_str());
    std::copy(cb[1].data.begin(), cb[1].data.end(), b.begin());
  }
  op.h_bias = b;
  op.bias.alloc(b.size() * sizeof(float));
  SIVO_CUDA(cudaMemcpy(op.bias.p, b.data(), b.size() * sizeof(float), cudaMemcpyHostToDevice));
  if (bn) {
    if (bn->size() < 2 || static_cast<int>((*bn)[0].count()) != cout || static_cast<int>((*bn)[1].count()) != cout)
      fail(SIVO_EFORMAT, "BN after '%s': expected scale and shift blobs of %d channels", op.layer.c_str(), cout);
    std::vector<float> sc(op.cout_p, 1.f), sh(op.cout_p, 0.f);
    std::copy((*bn)[0].data.begin(), (*bn)[0].data.end(), sc.begin());
    std::copy((*bn)[1].data.begin(), (*bn)[1].data.end(), sh.begin());
    op.h_bn_scale = sc;
    op.h_bn_shift = sh;
    op.bn_scale.alloc(sc.size() * sizeof(float));
    op.bn_shift.alloc(sh.size() * sizeof(float));
    SIVO_CUDA(cudaMemcpy(op.bn_scale.p, sc.data(), sc.size() * sizeof(float), cudaMemcpyHostToDevice));
    SIVO_CUDA(cudaMemcpy(op.bn_shift.p, sh.data(), sh.size() * sizeof(float), cudaMemcpyHostToDevice));
    op.has_bn = true;
  }
}

void SegNet::build(const NetSpec& net, const WeightMap& weights) {
  // consumers of each blob name, to spot the convolution feeding Softmax
  auto feeds_softmax = [&](size_t li, const std::string& top) {
    for (size_t j = li + 1; j < net.layers.size(); ++j)
      for (auto& b : net.layers[j].bottoms)
        if (b == top) return net.layers[j].type == LayerType::Softmax;
    return false;
  };
  int in_id = add_tensor(net.input_name, 1, 3, H_, W_, 4, act_);
  {
    Op op;
    op.kind = Op::Input;
    op.layer = "input";
    op.out = in_id;
    ops_.push_back(std::move(op));
  }
  auto blob_id = [&](const std::string& name) {
    auto it = by_name_.find(name);
    if (it == by_name_.end()) fail(SIVO_EFORMAT, "prototxt: blob '%s' is used before it is produced", name.c_str());
    // a fused kernel consumes this blob in registers and never writes it: a second consumer would read uninitialised memory
    if (tensors_[it->second]->elided)
      fail(SIVO_EFORMAT, "prototxt: blob '%s' has more than one consumer; the fused pool / unpool / dropout / classifier paths need a "
                         "single-consumer chain (create the net with keep_blobs to run it unfused)", name.c_str());
    return it->second;
  };
  int drop_idx = 0;
  bool saw_softmax = false;
  bool sampled = false;  // past the first sampling Dropout: tensors hold this handle's n_ samples
  for (size_t li = 0; li < net.layers.size(); ++li) {
    const LayerSpec& ly = net.layers[li];
    if (saw_softmax) fail(SIVO_EFORMAT, "prototxt: layers after Softmax are not on the path");
    int in = blob_id(ly.bottoms[0]);
    const TensorView iv = tensors_[in]->v;
    switch (ly.type) {
      case LayerType::LRN: {
        Op op;
        op.kind = Op::LRN;
        op.layer = ly.name;
        op.in = in;
        op.out = add_tensor(ly.tops[0], iv.n, iv.c, iv.h, iv.w, iv.cs, act_);
        op.lrn_size = ly.local_size; op.lrn_alpha = ly.alpha; op.lrn_beta = ly.beta; op.lrn_k = ly.k;
        ops_.push_back(std::move(op));
        break;
      }
      case LayerType::Convolution: {
        Op op;
        op.kind = Op::Conv;
        op.layer = ly.name;
        op.in = in;
        op.k = ly.kernel; op.pad = ly.pad; op.cin = iv.c; op.cout = ly.num_output;
        op.cin_p = iv.cs;
        if (sampled) op.plan_n = T_;  // a shard's per-sample layers run the unsharded handle's kernel variants
        const char* no_tc = std::getenv("SIVO_B200_NO_TC");
        if (iv.cs == 4 && iv.c == 3 && act_ == DType::F16 && opt_.engine != SIVO_ENGINE_SIMT && (ly.kernel == 7 || ly.kernel == 3) &&
            ly.num_output % 64 == 0 && !(no_tc && no_tc[0] == '1')) {
          // 3-channel first layer: expand the KxK taps into channels once, then it is a 1x1 tensor-core convolution
          const char* no_fold = std::getenv("SIVO_B200_NO_FOLD");
          Op ex;
          ex.kind = Op::Expand;
          ex.in = in;
          ex.k = ly.kernel;
          if (no_fold && no_fold[0] == '1') {
            // (A/B switch) materialise the taps as channels once, then it is a 1x1 tensor-core convolution
            const int blk = (ly.kernel * 4 + 15) / 16 * 16, cs_e = round_up(ly.kernel * blk, 64);
            ex.layer = ly.name + "/expand";
            ex.expand_blk = blk;
            ex.out = add_tensor("__expand_" + ly.name, iv.n, cs_e, iv.h, iv.w, cs_e, act_);
            ops_.push_back(std::move(ex));
            op.in = ops_.back().out;
            op.expand_k = ly.kernel; op.expand_blk = blk;
            op.k = 1; op.pad = 0; op.cin = cs_e; op.cin_p = cs_e;
          } else {
            // zero-pad to 8-channel pixels; the convolution's TMA reads overlapping 8-pixel windows of it (K x 1 layer)
            ex.layer = ly.name + "/pad8";
            ex.out = add_tensor("__pad8_" + ly.name, iv.n, 8, iv.h, iv.w + 8, 8, act_);
            const size_t no = ops_.size();
            if (!opt_.keep_blobs && no >= 2 && ops_[no - 1].kind == Op::LRN && ops_[no - 1].out == in && ops_[no - 2].kind == Op::Input &&
                ops_[no - 2].out == ops_[no - 1].in && iv.n == 1) {
              // input -> LRN -> pad8 collapse into one pass (the 'data' and 'norm' blobs are not materialised)
              ex.kind = Op::InputPad8;
              ex.lrn_size = ops_[no - 1].lrn_size; ex.lrn_alpha = ops_[no - 1].lrn_alpha;
              ex.lrn_beta = ops_[no - 1].lrn_beta; ex.lrn_k = ops_[no - 1].lrn_k;
              ex.layer = "input+" + ops_[no - 1].layer + "+" + ex.layer;
              tensors_[ops_[no - 1].out]->elided = tensors_[ops_[no - 2].out]->elided = true;
              ops_.pop_back();
              ops_.pop_back();
            }
            ops_.push_back(std::move(ex));
            op.in = ops_.back().out;
            op.fold_kw = ly.kernel;
            op.cin = 64; op.cin_p = 64;
          }
        }
        const TensorView civ = tensors_[op.in]->v;  // the tensor the convolution actually reads
        op.cout_p = round_up(op.cout, 64);
        const std::vector<Blob>* bn = nullptr;
        size_t lj = li + 1;
        for (; lj < net.layers.size(); ++lj) {  // absorb the in-place followers
          const LayerSpec& f = net.layers[lj];
          bool inplace = f.bottoms[0] == ly.tops[0] && f.tops[0] == ly.tops[0];
          if (!inplace) break;
          if (f.type == LayerType::BN && !bn && !op.relu) {
            auto it = weights.find(f.name);
            if (it == weights.end()) fail(SIVO_EFORMAT, "caffemodel has no blobs for BN layer '%s'", f.name.c_str());
            bn = &it->second;
          } else if (f.type == LayerType::ReLU && !op.relu) {
            op.relu = true;
            op.slope = f.negative_slope;
          } else {
            break;
          }
        }
        bool logits = feeds_softmax(lj - 1, ly.tops[0]);
        if (!logits && (op.cout % 8)) fail(SIVO_EFORMAT, "layer '%s': %d output channels (need a multiple of 8)", ly.name.c_str(), op.cout);
        int cs = logits ? round_up(op.cout, 16) : op.cout;
        op.out = add_tensor(ly.tops[0], iv.n, op.cout, iv.h, iv.w, cs, logits ? DType::F32 : act_);
        auto it = weights.find(ly.name);
        if (it == weights.end()) fail(SIVO_EFORMAT, "caffemodel has no blobs for layer '%s'", ly.name.c_str());
        // fp32 activations on the tensor-core engine: split-operand mode (three half MMAs per tap, fp32 accumulation)
        TensorView split_in = civ;
        if (act_ == DType::F32 && opt_.engine != SIVO_ENGINE_SIMT && !op.fold_kw && !op.expand_k && civ.cs % 64 == 0 && civ.c == civ.cs &&
            !(no_tc && no_tc[0] == '1')) {
          split_in.dt = DType::F16;
          split_in.cs = 2 * civ.cs;
          op.split = true;
          if (!conv_tc_supported(op, split_in, tensors_[op.out]->v)) op.split = false;
        }
        prepare_conv(op, it->second, bn);
        op.flops = 2.0 * iv.c * ly.kernel * ly.kernel * op.cout * iv.h * iv.w * iv.n;  // algorithmic, whatever the mapping
        op.flops_exec = op.split ? 3.0 * op.flops : op.flops;
        flops_dedup += op.flops;
        flops_naive += op.flops / iv.n * n_;
        if (logits && !opt_.keep_blobs && op.k == 1 && op.cin == 64 && op.cout <= 16 && !op.relu && !bn && !ops_.empty() &&
            ops_.back().kind == Op::Conv && ops_.back().use_tc && ops_.back().out == in && conv_tc_can_fuse_classifier(*ops_.back().tc)) {
          // 1x1 classifier straight after a tensor-core convolution: computed in that convolution's epilogue from the
          // half-rounded activations, so the 64-channel tensor is never written or re-read
          // No non-linearity sits between the two layers (Basic), so logits = (Wc W) * x + (Wc b + bc): ONE 64 -> 16 convolution
          // with weights composed in double and rounded to half once -- a quarter of the multiply-adds, and closer to the
          // reference's fp32 arithmetic than the two-step half path (the 64-channel activation is never rounded to half;
          // tests/test_gpu_parity.py, tools/compose_classifier_study.py).  Default; SIVO_B200_COMPOSE=0 keeps the two-step form.
          const char* compose = std::getenv("SIVO_B200_COMPOSE");
          Op& conv = ops_.back();
          if (!(compose && compose[0] == '0') && !conv.relu && !conv.has_bn && conv_tc_can_compose_classifier(*conv.tc)) {
            conv_tc_set_composed_classifier(*conv.tc, conv, op.h_w_raw.data(), op.h_bias.data(), op.cout,
                                            static_cast<float*>(tensors_[op.out]->v.p));
            conv.flops_exec = 2.0 * conv.cin * conv.k * conv.k * 16 * iv.h * iv.w * iv.n;  // the 16-wide composed layer
            conv.layer += "*" + ly.name;  // '*': composed, not merely fused
          } else {
            conv_tc_set_classifier(*conv.tc, op.h_w.data(), op.cout_p, op.h_bias.data(), std::min(16, op.cout_p),
                                   static_cast<float*>(tensors_[op.out]->v.p));
            conv.flops_exec += op.flops;
            conv.layer += "+" + ly.name;
          }
          conv.flops += op.flops;  // algorithmic: the reference runs both layers
          tensors_[in]->elided = true;
          fused_.push_back(std::move(op));
          li = lj - 1;
          break;
        }
        if (op.split) {
          op.a_split.alloc(split_in.elems() * sizeof(__half));
          split_in.p = op.a_split.p;
          op.tc = conv_tc_plan(op, split_in, tensors_[op.out]->v, op.w_tc.p);
          op.use_tc = true;
        } else if (opt_.engine != SIVO_ENGINE_SIMT && act_ == DType::F16 &&
            conv_tc_supported(op, civ, tensors_[op.out]->v)) {
          op.tc = conv_tc_plan(op, civ, tensors_[op.out]->v, op.w_tc.p);
          op.use_tc = true;
        } else if (op.fold_kw) {
          fail(SIVO_EINVAL, "layer '%s': window-folded first layer is not supported by the tensor-core kernel", ly.name.c_str());
        } else if (opt_.engine == SIVO_ENGINE_TCGEN05 && op.cin_p % 64 == 0 && (!logits || act_ == DType::F32)) {
          fail(SIVO_EINVAL, "layer '%s': tcgen05 engine requested but the shape is not supported", ly.name.c_str());
        }
        ops_.push_back(std::move(op));
        li = lj - 1;
        break;
      }
      case LayerType::ReLU:
      case LayerType::BN:
        fail(SIVO_EFORMAT, "layer '%s': %s must follow a convolution in place", ly.name.c_str(),
             ly.type == LayerType::BN ? "BN" : "ReLU");
      case LayerType::Pooling: {
        if ((iv.h | iv.w) & 1) fail(SIVO_EFORMAT, "layer '%s': odd input size %dx%d", ly.name.c_str(), iv.h, iv.w);
        if (iv.cs != iv.c) fail(SIVO_EFORMAT, "layer '%s': pooling a padded-channel tensor", ly.name.c_str());
        const int pooled = add_tensor(ly.tops[0], iv.n, iv.c, iv.h / 2, iv.w / 2, iv.cs, act_);
        const int pmask = add_tensor(ly.tops[1], iv.n, iv.c, iv.h / 2, iv.w / 2, iv.cs, act_, true);
        if (!opt_.keep_blobs && !ops_.empty() && ops_.back().kind == Op::Conv && ops_.back().use_tc && ops_.back().out == in &&
            iv.dt == DType::F16 && conv_tc_can_fuse_pool(*ops_.back().tc)) {
          // the producing tensor-core convolution pools in its epilogue: the full-resolution activations are never stored
          conv_tc_set_pool(*ops_.back().tc, tensors_[pooled]->v.p, tensors_[pmask]->buf.as<uint8_t>());
          tensors_[in]->elided = true;
          ops_.back().layer += "+" + ly.name;
          break;
        }
        Op op;
        op.kind = Op::Pool;
        op.layer = ly.name;
        op.in = in;
        op.out = pooled;
        op.out2 = pmask;
        ops_.push_back(std::move(op));
        break;
      }
      case LayerType::Upsample: {
        int m = blob_id(ly.bottoms[1]);
        const Tensor& mt = *tensors_[m];
        if (!mt.is_mask || mt.v.c != iv.c || mt.v.h != iv.h || mt.v.w != iv.w)
          fail(SIVO_EFORMAT, "layer '%s': mask blob '%s' does not match the input", ly.name.c_str(), ly.bottoms[1].c_str());
        const int up = add_tensor(ly.tops[0], iv.n, iv.c, iv.h * 2, iv.w * 2, iv.cs, act_);
        if (!opt_.keep_blobs && !ops_.empty() && ops_.back().kind == Op::Conv && ops_.back().use_tc && ops_.back().out == in &&
            iv.dt == DType::F16 && iv.cs == iv.c) {
          // the producing tensor-core convolution scatters straight into the unpooled tensor (its own output blob
          // is never materialised; keep_blobs keeps the two-kernel form so tests can read it)
          conv_tc_set_unpool(*ops_.back().tc, mt.buf.as<uint8_t>(), mt.v.n, tensors_[up]->v.p);
          tensors_[in]->elided = true;
          ops_.back().layer += "+" + ly.name;
          break;
        }
        if (!opt_.keep_blobs && !ops_.empty() && ops_.back().kind == Op::Dropout && ops_.back().out == in && iv.dt == DType::F16 &&
            iv.cs == iv.c && iv.cs % 8 == 0) {
          // sampling Dropout feeding the upsample: one pass writes the unpooled tensor (the dropped blob is not materialised)
          Op& d = ops_.back();
          tensors_[in]->elided = true;
          d.kind = Op::DropoutUnpool;
          d.in2 = m;
          d.out = up;
          d.layer += "+" + ly.name;
          break;
        }
        Op op;
        op.kind = Op::Unpool;
        op.layer = ly.name;
        op.in = in;
        op.in2 = m;
        op.out = up;
        ops_.push_back(std::move(op));
        break;
      }
      case LayerType::Dropout: {
        if (!ly.sample_weights_test) {  // plain test-time dropout is the identity (dropout_layer.cpp:43-45)
          by_name_[ly.tops[0]] = in;
          ++drop_idx;
          break;
        }
        if (ly.dropout_ratio != 0.5f)
          fail(SIVO_EFORMAT, "layer '%s': dropout_ratio %.3f (the keep-bit rule is specified for 0.5)", ly.name.c_str(), ly.dropout_ratio);
        if (sampled && !ops_.empty() && ops_.back().kind == Op::Conv && ops_.back().use_tc && ops_.back().out == in && iv.n == n_ &&
            iv.dt == DType::F16 && ly.tops[0] == ly.bottoms[0]) {
          // in-place sampling Dropout right after a tensor-core convolution: applied in its epilogue registers
          conv_tc_set_dropout(*ops_.back().tc, opt_.seed, d_frame_.as<uint64_t>(), drop_idx++, s0_, 1.f / (1.f - ly.dropout_ratio));
          ops_.back().layer += "+" + ly.name;
          break;
        }
        Op op;
        op.kind = Op::Dropout;
        op.layer = ly.name;
        op.in = in;
        op.drop_layer = drop_idx++;
        op.drop_scale = 1.f / (1.f - ly.dropout_ratio);
        op.out = add_tensor(ly.tops[0], n_, iv.c, iv.h, iv.w, iv.cs, act_);
        ops_.push_back(std::move(op));
        sampled = true;
        break;
      }
      case LayerType::Softmax: {
        if (iv.dt != DType::F32) fail(SIVO_EFORMAT, "Softmax must follow a convolution");
        n_classes_ = iv.c;
        Op op;
        op.kind = Op::Reduce;
        op.layer = ly.name;
        op.in = in;
        ops_.push_back(std::move(op));
        saw_softmax = true;
        break;
      }
    }
  }
  if (!saw_softmax) fail(SIVO_EFORMAT, "prototxt: no Softmax output layer ('prob')");
  if (!sampled && n_ != T_) fail(SIVO_EINVAL, "sample shard of a net without a sampling Dropout layer: every sample is the same");
}

SegNet::SegNet(const std::string& prototxt, const std::string& caffemodel, const sivo_segnet_options& opt, int first_sample,
               int n_samples)
    : opt_(opt) {
  // checkConfig (bayesian_segnet.cpp:80-89)
  if (prototxt.empty()) fail(SIVO_EINVAL, "model_file (.prototxt file) is empty!");
  if (caffemodel.empty()) fail(SIVO_EINVAL, "weights_file (.caffemodel file) is empty!");
  NetSpec net = parse_prototxt_file(prototxt);
  T_ = opt.T > 0 ? opt.T : net.dims[0];
  // bayesian_segnet.cpp:65-70
  if (net.dims[1] != 3) fail(SIVO_EINVAL, "Input layer must have 3 channels!");
  if (T_ <= 1) fail(SIVO_EINVAL, "Input layer must have a batch size greater than 1!");
  if (n_samples >= 0 && (first_sample < 0 || n_samples < 1 || first_sample > T_ - n_samples))
    fail(SIVO_EINVAL, "sample shard [%d, %d + %d) is not a non-empty range inside the T = %d Monte-Carlo samples", first_sample,
         first_sample, n_samples, T_);
  s0_ = n_samples >= 0 ? first_sample : 0;
  n_ = n_samples >= 0 ? n_samples : T_;
  H_ = net.dims[2];
  W_ = net.dims[3];
  if (H_ <= 0 || W_ <= 0) fail(SIVO_EFORMAT, "prototxt: bad input geometry %dx%d", W_, H_);
  act_ = opt.precision == SIVO_PRECISION_FP32 ? DType::F32 : DType::F16;
  WeightMap weights = read_caffemodel(caffemodel);
  device_ = opt.device;
  SIVO_CUDA(cudaSetDevice(device_));
  SIVO_CUDA(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  try {  // a malformed model throws out of build(): the destructor does not run for a half-built object
    d_frame_.alloc(sizeof(FrameArgs));
    build(net, weights);
    if (n_samples >= 0) {  // the partial / finalize kernels read 16-float logit pixels
      const TensorView& lv = tensors_[ops_.back().in]->v;
      if (lv.cs != 16 || lv.c > 16)
        fail(SIVO_EFORMAT, "sample shards need logits in the 16-channel layout (%d classes, channel stride %d)", lv.c, lv.cs);
    }
  } catch (...) {
    cudaStreamDestroy(stream_);
    stream_ = nullptr;
    throw;
  }
  const size_t hw = static_cast<size_t>(H_) * W_;
  d_bgr_.alloc(hw * 3);
  d_classes_.alloc(hw);
  d_conf_.alloc(hw * sizeof(double));
  d_ent_.alloc(hw * sizeof(double));
  h_in_.ensure(hw * 3);
  h_classes_.ensure(hw);
  h_conf_.ensure(hw * sizeof(double));
  h_ent_.ensure(hw * sizeof(double));
  SIVO_CUDA(cudaStreamSynchronize(stream_));
}

SegNet::~SegNet() {
  cudaSetDevice(device_);
  for (auto& g : graphs_) cudaGraphExecDestroy(g.exec);
  for (auto e : band_ev_) cudaEventDestroy(e);
  if (copy_stream_) cudaStreamDestroy(copy_stream_);
  for (auto e : events_) cudaEventDestroy(e);
  if (stream_) cudaStreamDestroy(stream_);
}

void SegNet::enqueue(const uint8_t* bgr_dev, uint8_t* classes_dev, double* conf_dev, double* ent_dev, cudaStream_t s, bool timed) {
  launches = 0;
  if (timed) SIVO_CUDA(cudaEventRecord(events_[0], s));
  for (size_t i = 0; i < ops_.size(); ++i) {
    Op& op = ops_[i];
    switch (op.kind) {
      case Op::Input:
        launch_input_u8(bgr_dev, tensors_[op.out]->v, s, d_frame_.as<FrameArgs>());
        break;
      case Op::Expand:
      case Op::InputPad8:
        if (op.kind == Op::InputPad8)
          launch_input_lrn_pad8(bgr_dev, tensors_[op.out]->v, op.lrn_size, op.lrn_alpha, op.lrn_beta, op.lrn_k, s, d_frame_.as<FrameArgs>());
        else if (op.expand_blk) launch_expand_taps(tensors_[op.in]->v, tensors_[op.out]->v, op.k, op.expand_blk, s);
        else launch_pad8(tensors_[op.in]->v, tensors_[op.out]->v, s);
        break;
      case Op::LRN:
        launch_lrn(tensors_[op.in]->v, tensors_[op.out]->v, op.lrn_size, op.lrn_alpha, op.lrn_beta, op.lrn_k, s);
        break;
      case Op::Conv: {
        if (op.use_tc) {
          if (op.split) {  // the float input as [hi | lo] half planes
            launch_split_hilo(tensors_[op.in]->v, op.a_split.p, s);
            ++launches;
          }
          conv_tc_launch(*op.tc, op, s);
        } else {
          ConvParams p;
          p.in = tensors_[op.in]->v;
          p.out = tensors_[op.out]->v;
          p.w_simt = op.w_simt.as<float>();
          p.bias = op.bias.as<float>();
          p.bn_scale = op.has_bn ? op.bn_scale.as<float>() : nullptr;
          p.bn_shift = op.has_bn ? op.bn_shift.as<float>() : nullptr;
          p.k = op.k; p.pad = op.pad; p.cin_p = op.cin_p; p.cout_p = op.cout_p;
          p.relu = op.relu; p.slope = op.slope;
          launch_conv_simt(p, s);
        }
        break;
      }
      case Op::Pool:
        launch_pool(tensors_[op.in]->v, tensors_[op.out]->v, tensors_[op.out2]->buf.as<uint8_t>(), s);
        break;
      case Op::Unpool:
        launch_unpool(tensors_[op.in]->v, tensors_[op.in2]->buf.as<uint8_t>(), tensors_[op.in2]->v.n, tensors_[op.out]->v, s);
        break;
      case Op::Dropout: {
        DropoutParams d;
        d.seed = opt_.seed;
        d.frame_dev = d_frame_.as<uint64_t>();
        d.layer = op.drop_layer;
        d.sample0 = s0_;
        launch_dropout(tensors_[op.in]->v, tensors_[op.out]->v, d, op.drop_scale, s);
        break;
      }
      case Op::DropoutUnpool: {
        DropoutParams d;
        d.seed = opt_.seed;
        d.frame_dev = d_frame_.as<uint64_t>();
        d.layer = op.drop_layer;
        d.sample0 = s0_;
        const Tensor& mt = *tensors_[op.in2];
        launch_dropout_unpool(tensors_[op.in]->v, n_, mt.buf.as<uint8_t>(), mt.v.n, tensors_[op.out]->v, d, op.drop_scale, s);
        break;
      }
      case Op::Reduce: {
        if (skip_reduce_) break;
        const TensorView& lv = tensors_[op.in]->v;
        if (partial_) {
          launch_mc_partial(static_cast<const float*>(lv.p), lv.n, lv.c, lv.cs, lv.h * lv.w, nullptr, 0, s, d_frame_.as<FrameArgs>());
          break;
        }
        launch_mc_reduce(static_cast<const float*>(lv.p), lv.n, lv.c, lv.cs, lv.h * lv.w, classes_dev, conf_dev, ent_dev, s, 0, -1,
                         d_frame_.as<FrameArgs>());
        break;
      }
    }
    ++launches;
    if (timed) SIVO_CUDA(cudaEventRecord(events_[i + 1], s));
  }
}

void SegNet::semantic_keys(const sivo_keypoint* kps, int n, int max_static_class, uint8_t* kp_class, double* kp_conf, double* kp_entropy,
                           int* keep_idx, int* n_keep) {
  if (n_keep) *n_keep = 0;
  if (n < 0 || (n > 0 && !kps)) fail(SIVO_EINVAL, "semantic_keys: bad keypoint array");
  if (!last_classes_ || !last_conf_ || !last_ent_) fail(SIVO_EINVAL, "semantic_keys: no segmentation result on the device yet (or a map pointer was NULL)");
  if (n == 0) return;
  SIVO_CUDA(cudaSetDevice(device_));
  cudaStream_t s = last_stream_;
  const size_t in_bytes = static_cast<size_t>(n) * sizeof(sivo_keypoint);
  const size_t out_bytes = static_cast<size_t>(n) * 17;  // n doubles, n doubles, n bytes
  if (d_kp_.bytes < in_bytes) d_kp_.alloc(in_bytes * 2);
  if (d_kp_out_.bytes < out_bytes) d_kp_out_.alloc(out_bytes * 2);
  h_kp_.ensure(in_bytes);
  h_kp_out_.ensure(out_bytes);
  memcpy(h_kp_.p, kps, in_bytes);
  SIVO_CUDA(cudaMemcpyAsync(d_kp_.p, h_kp_.p, in_bytes, cudaMemcpyHostToDevice, s));
  double* o_conf = d_kp_out_.as<double>();
  double* o_ent = o_conf + n;
  uint8_t* o_cls = reinterpret_cast<uint8_t*>(o_ent + n);
  launch_keypoint_lookup(d_kp_.as<sivo_keypoint>(), n, last_classes_, last_conf_, last_ent_, H_, W_, o_cls, o_conf, o_ent, s);
  SIVO_CUDA(cudaMemcpyAsync(h_kp_out_.p, d_kp_out_.p, out_bytes, cudaMemcpyDeviceToHost, s));
  SIVO_CUDA(cudaStreamSynchronize(s));
  const double* hc = h_kp_out_.as<double>();
  const double* he = hc + n;
  const uint8_t* hk = reinterpret_cast<const uint8_t*>(he + n);
  if (kp_conf) memcpy(kp_conf, hc, static_cast<size_t>(n) * sizeof(double));
  if (kp_entropy) memcpy(kp_entropy, he, static_cast<size_t>(n) * sizeof(double));
  if (kp_class) memcpy(kp_class, hk, n);
  int kept = 0;
  for (int i = 0; i < n; ++i)
    if (hk[i] != 255 && static_cast<int>(hk[i]) <= max_static_class) {  // `detection <= Classes::TERRAIN` (Frame.cc:190)
      if (keep_idx) keep_idx[kept] = i;
      ++kept;
    }
  if (n_keep) *n_keep = kept;
}

void SegNet::require_whole(const char* what) const {
  if (n_ != T_)
    fail(SIVO_EINVAL, "%s: this handle computes Monte-Carlo samples [%d, %d) of T = %d only; run it with run_device_partial and "
                      "finalize the summed probabilities", what, s0_, s0_ + n_, T_);
}

void SegNet::run_device(const uint8_t* bgr_dev, uint8_t* classes_dev, double* conf_dev, double* ent_dev, cudaStream_t s, float* conf32_dev,
                        float* ent32_dev) {
  require_whole("run_device");
  SIVO_CUDA(cudaSetDevice(device_));
  if (!s) s = stream_;
  last_classes_ = classes_dev; last_conf_ = conf_dev; last_ent_ = ent_dev; last_stream_ = s;
  FrameArgs fa{};
  fa.bgr = bgr_dev; fa.classes = classes_dev; fa.conf = conf_dev; fa.ent = ent_dev; fa.conf32 = conf32_dev; fa.ent32 = ent32_dev;
  run_frame(fa, s);
}

void SegNet::run_device_partial(const uint8_t* bgr_dev, double* prob_sum_dev, int accumulate, cudaStream_t s) {
  if (!prob_sum_dev) fail(SIVO_EINVAL, "run_device_partial: null probability-sum buffer");
  SIVO_CUDA(cudaSetDevice(device_));
  if (!s) s = stream_;
  FrameArgs fa{};
  fa.bgr = bgr_dev; fa.prob_sum = prob_sum_dev; fa.accumulate = accumulate ? 1 : 0;
  partial_ = true;
  try {
    run_frame(fa, s);
  } catch (...) {
    partial_ = false;
    throw;
  }
  partial_ = false;
}

void SegNet::finalize_device(const double* prob_sum_dev, uint8_t* classes_dev, double* conf_dev, double* ent_dev, float* conf32_dev,
                             float* ent32_dev, cudaStream_t s) {
  if (!prob_sum_dev) fail(SIVO_EINVAL, "finalize_device: null probability-sum buffer");
  SIVO_CUDA(cudaSetDevice(device_));
  if (!s) s = stream_;
  launch_mc_finalize(prob_sum_dev, T_, n_classes_, H_ * W_, classes_dev, conf_dev, ent_dev, conf32_dev, ent32_dev, s);
  last_classes_ = classes_dev; last_conf_ = conf_dev; last_ent_ = ent_dev; last_stream_ = s;
}

void SegNet::run_frame(const FrameArgs& frame_args, cudaStream_t s) {
  const uint8_t* bgr_dev = frame_args.bgr;
  uint8_t* classes_dev = frame_args.classes;
  double* conf_dev = frame_args.conf;
  double* ent_dev = frame_args.ent;
  // Everything that changes per frame -- the dropout frame counter and the caller's pointers -- goes to the device by value,
  // outside the captured graph (pipelined callers may issue the next frame before this one has started), so one graph per
  // stream serves every pointer set a caller cycles through
  FrameArgs fa = frame_args;
  fa.frame = frame_++;
  launch_set_frame_args(d_frame_.as<FrameArgs>(), fa, s);
  if (profiling_) {
    while (events_.size() < ops_.size() + 1) {
      cudaEvent_t e;
      SIVO_CUDA(cudaEventCreate(&e));
      events_.push_back(e);
    }
    enqueue(bgr_dev, classes_dev, conf_dev, ent_dev, s, true);
    SIVO_CUDA(cudaEventSynchronize(events_[ops_.size()]));
    conv_ms = other_ms = reduce_ms = 0;
    op_ms.assign(ops_.size(), 0.f);
    for (size_t i = 0; i < ops_.size(); ++i) {
      float ms = 0;
      SIVO_CUDA(cudaEventElapsedTime(&ms, events_[i], events_[i + 1]));
      op_ms[i] = ms;
      if (ops_[i].kind == Op::Conv) conv_ms += ms;
      else if (ops_[i].kind == Op::Reduce) reduce_ms += ms;
      else other_ms += ms;
    }
    SIVO_CUDA(cudaEventElapsedTime(&total_ms, events_[0], events_[ops_.size()]));
    return;
  }
  // Steady state: the whole op list is one CUDA graph launch.  Everything that changes per frame lives in device
  // memory (the frame counter read by the dropout code), so the captured kernels and their arguments never change.
  bool all_tc = true;
  for (const Op& op : ops_) if (op.kind == Op::Conv && !op.use_tc) all_tc = false;  // the SIMT launcher sets attributes per launch
  static const bool graphs_enabled = [] { const char* e = std::getenv("SIVO_B200_NO_GRAPH"); return !(e && e[0] == '1'); }();
  if (graphs_enabled && graph_ok_ && all_tc) {
    // the graph's kernels read the image / result pointers from FrameArgs: the key is the stream (and the op-list variant) only
    const void* key[5] = {nullptr, nullptr, nullptr, nullptr,
                          reinterpret_cast<const void*>(reinterpret_cast<uintptr_t>(s) ^ (skip_reduce_ ? 1u : 0u) ^ (partial_ ? 2u : 0u))};
    cudaGraphExec_t graph_exec_ = nullptr;
    for (size_t i = 0; i < graphs_.size(); ++i)
      if (memcmp(key, graphs_[i].key, sizeof key) == 0) {
        std::rotate(graphs_.begin(), graphs_.begin() + i, graphs_.begin() + i + 1);  // move to front
        graph_exec_ = graphs_.front().exec;
        break;
      }
    if (!graph_exec_) {
      cudaGraph_t g = nullptr;
      cudaError_t e = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal);
      if (e == cudaSuccess) {
        try {
          enqueue(bgr_dev, classes_dev, conf_dev, ent_dev, s, false);
        } catch (...) {
          cudaStreamEndCapture(s, &g);
          if (g) cudaGraphDestroy(g);
          graph_ok_ = false;
          throw;
        }
        e = cudaStreamEndCapture(s, &g);
        if (e == cudaSuccess) e = cudaGraphInstantiate(&graph_exec_, g, 0);
        if (g) cudaGraphDestroy(g);
      }
      if (e != cudaSuccess) {  // fall back to plain launches for this handle
        cudaGetLastError();
        graph_ok_ = false;
        graph_exec_ = nullptr;
      } else {
        if (graphs_.size() >= kMaxGraphs) {  // a caller cycling through more buffers than this re-captures the oldest
          cudaGraphExecDestroy(graphs_.back().exec);
          graphs_.pop_back();
        }
        GraphEntry ge;
        memcpy(ge.key, key, sizeof key);
        ge.exec = graph_exec_;
        graphs_.insert(graphs_.begin(), ge);
      }
    }
    if (graph_exec_) {
      SIVO_CUDA(cudaGraphLaunch(graph_exec_, s));
      return;
    }
  }
  enqueue(bgr_dev, classes_dev, conf_dev, ent_dev, s, false);
}

void SegNet::run_host(const uint8_t* bgr, int rows, int cols, size_t stride, uint8_t* classes, double* conf, double* ent) {
  require_whole("segmentImage");
  if (!bgr) fail(SIVO_EINVAL, "segmentImage: null image");
  // resizeImage (bayesian_segnet.cpp:142-162): exact size passes through, larger is centre-cropped;
  // smaller yields an empty Mat in the reference (and a crash downstream) -- here an error.
  if (rows < H_ || cols < W_) fail(SIVO_EINVAL, "segmentImage: image %dx%d is smaller than the network input %dx%d", cols, rows, W_, H_);
  if (stride < static_cast<size_t>(cols) * 3) fail(SIVO_EINVAL, "segmentImage: stride smaller than a row");
  int x_tl = 0, y_tl = 0;
  if (rows != H_ || cols != W_) {
    x_tl = cols / 2 - W_ / 2;
    y_tl = rows / 2 - H_ / 2;
  }
  SIVO_CUDA(cudaSetDevice(device_));
  const size_t hw = static_cast<size_t>(H_) * W_;
  const uint8_t* src = bgr + static_cast<size_t>(y_tl) * stride + static_cast<size_t>(x_tl) * 3;
  if (is_pinned_host(bgr)) {  // crop straight out of the caller's page-locked image
    SIVO_CUDA(cudaMemcpy2DAsync(d_bgr_.p, static_cast<size_t>(W_) * 3, src, stride, static_cast<size_t>(W_) * 3, H_,
                                cudaMemcpyHostToDevice, stream_));
  } else {
    uint8_t* stage = h_in_.as<uint8_t>();
    for (int y = 0; y < H_; ++y)
      memcpy(stage + static_cast<size_t>(y) * W_ * 3, src + static_cast<size_t>(y) * stride, static_cast<size_t>(W_) * 3);
    SIVO_CUDA(cudaMemcpyAsync(d_bgr_.p, stage, hw * 3, cudaMemcpyHostToDevice, stream_));
  }
  // outputs are caller-owned plain memory (Frame copies them into itself, Frame.cc:239-241): page-locked caller
  // buffers receive the device copy directly, pageable ones go through the pinned staging buffers
  const bool pc = is_pinned_host(classes), pf = is_pinned_host(conf), pe = is_pinned_host(ent);
  uint8_t* hc = pc ? classes : h_classes_.as<uint8_t>();
  double* hf = pf ? conf : h_conf_.as<double>();
  double* he = pe ? ent : h_ent_.as<double>();
  static const int n_bands = [] { const char* e = std::getenv("SIVO_B200_READBACK_BANDS"); return e ? std::max(1, std::min(16, atoi(e))) : 1; }();  // opt-in: measured no gain with the extractors' copies sharing the D2H engine
  const Op& last = ops_.back();
  const TensorView* lv = last.kind == Op::Reduce ? &tensors_[last.in]->v : nullptr;
  const bool to_record = rec_classes_ || rec_conf32_ || rec_ent32_;
  const bool banded = n_bands > 1 && !to_record && !profiling_ && lv && lv->cs == 16 && lv->c <= 16 && (classes || conf || ent) && H_ >= n_bands;
  if (!banded) {
    run_device(d_bgr_.as<uint8_t>(), d_classes_.as<uint8_t>(), d_conf_.as<double>(), d_ent_.as<double>(), stream_, rec_conf32_, rec_ent32_);
    if (classes) SIVO_CUDA(cudaMemcpyAsync(hc, d_classes_.p, hw, cudaMemcpyDeviceToHost, stream_));
    if (conf) SIVO_CUDA(cudaMemcpyAsync(hf, d_conf_.p, hw * sizeof(double), cudaMemcpyDeviceToHost, stream_));
    if (ent) SIVO_CUDA(cudaMemcpyAsync(he, d_ent_.p, hw * sizeof(double), cudaMemcpyDeviceToHost, stream_));
    if (rec_classes_) SIVO_CUDA(cudaMemcpyAsync(rec_classes_, d_classes_.p, hw, cudaMemcpyDeviceToDevice, stream_));
    SIVO_CUDA(cudaStreamSynchronize(stream_));
  } else {
    if (!copy_stream_) SIVO_CUDA(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking));
    while (static_cast<int>(band_ev_.size()) < n_bands) {
      cudaEvent_t e;
      SIVO_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      band_ev_.push_back(e);
    }
    skip_reduce_ = true;
    try {
      run_device(d_bgr_.as<uint8_t>(), d_classes_.as<uint8_t>(), d_conf_.as<double>(), d_ent_.as<double>(), stream_);
    } catch (...) {
      skip_reduce_ = false;
      throw;
    }
    skip_reduce_ = false;
    for (int b = 0; b < n_bands; ++b) {
      const int r0 = static_cast<int>(static_cast<long>(H_) * b / n_bands), r1 = static_cast<int>(static_cast<long>(H_) * (b + 1) / n_bands);
      const size_t p0 = static_cast<size_t>(r0) * W_, np = static_cast<size_t>(r1 - r0) * W_;
      launch_mc_reduce(static_cast<const float*>(lv->p), lv->n, lv->c, lv->cs, lv->h * lv->w, d_classes_.as<uint8_t>(), d_conf_.as<double>(),
                       d_ent_.as<double>(), stream_, static_cast<int>(p0), static_cast<int>(np));
      SIVO_CUDA(cudaEventRecord(band_ev_[b], stream_));
      SIVO_CUDA(cudaStreamWaitEvent(copy_stream_, band_ev_[b], 0));
      if (classes) SIVO_CUDA(cudaMemcpyAsync(hc + p0, d_classes_.as<uint8_t>() + p0, np, cudaMemcpyDeviceToHost, copy_stream_));
      if (conf) SIVO_CUDA(cudaMemcpyAsync(hf + p0, d_conf_.as<double>() + p0, np * sizeof(double), cudaMemcpyDeviceToHost, copy_stream_));
      if (ent) SIVO_CUDA(cudaMemcpyAsync(he + p0, d_ent_.as<double>() + p0, np * sizeof(double), cudaMemcpyDeviceToHost, copy_stream_));
    }
    launches = static_cast<int>(ops_.size()) - 1 + n_bands;  // the bands replace the single Reduce launch of the op list
    SIVO_CUDA(cudaStreamSynchronize(copy_stream_));
    SIVO_CUDA(cudaStreamSynchronize(stream_));
  }
  if (classes && !pc) memcpy(classes, h_classes_.p, hw);
  if (conf && !pf) memcpy(conf, h_conf_.p, hw * sizeof(double));
  if (ent && !pe) memcpy(ent, h_ent_.p, hw * sizeof(double));
}

void SegNet::blob(const std::string& name, float* out, size_t cap, int* n, int* c, int* h, int* w) {
  auto it = by_name_.find(name);
  if (it == by_name_.end()) fail(SIVO_EINVAL, "no blob named '%s'", name.c_str());
  const Tensor& t = *tensors_[it->second];
  if (t.elided && out)
    fail(SIVO_EINVAL, "blob '%s' is not materialised in this build (a fused kernel consumes it); create the net with keep_blobs", name.c_str());
  if (n) *n = t.v.n;
  if (c) *c = t.v.c;
  if (h) *h = t.v.h;
  if (w) *w = t.v.w;
  if (!out) return;
  size_t count = static_cast<size_t>(t.v.n) * t.v.c * t.v.h * t.v.w;
  if (cap < count) fail(SIVO_ERANGE, "blob '%s' has %zu values, buffer holds %zu", name.c_str(), count, cap);
  SIVO_CUDA(cudaSetDevice(device_));
  DevBuf tmp(count * sizeof(float));
  if (t.is_mask) {
    launch_mask_to_nchw(t.buf.as<uint8_t>(), t.v.n, t.v.c, t.v.h, t.v.w, tmp.as<int>(), stream_);
    std::vector<int> hi(count);
    SIVO_CUDA(cudaMemcpyAsync(hi.data(), tmp.p, count * sizeof(int), cudaMemcpyDeviceToHost, stream_));
    SIVO_CUDA(cudaStreamSynchronize(stream_));
    for (size_t i = 0; i < count; ++i) out[i] = static_cast<float>(hi[i]);  // Caffe stores the index as float
  } else {
    launch_act_to_nchw(t.v, tmp.as<float>(), stream_);
    SIVO_CUDA(cudaMemcpyAsync(out, tmp.p, count * sizeof(float), cudaMemcpyDeviceToHost, stream_));
    SIVO_CUDA(cudaStreamSynchronize(stream_));
  }
}

}  // namespace sivo
