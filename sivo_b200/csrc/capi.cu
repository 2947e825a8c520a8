// extern "C" boundary of libsivo_b200.so (include/sivo_b200.h).  No C++ type, exception or abort crosses it.
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>

#include "orb.h"
#include "segnet.h"

namespace sivo {
namespace {
thread_local std::string g_last_error;
}
void set_last_error(const std::string& m) { g_last_error = m; }
void stereo_hamming(int device, const sivo_keypoint* left, const uint8_t* dl, int nl, const sivo_keypoint* right,
                    const uint8_t* dr, int nr, const float* scale, int nlevels, int rows, float min_d, float max_d,
                    int* best_idx, int* best_dist);
void stereo_match(const Orb& left, const Orb& right, const sivo_keypoint* kl, const uint8_t* dl, int nl, const sivo_keypoint* kr,
                  const uint8_t* dr, int nr, float mb, float mbf, float* u_right, float* depth);
}  // namespace sivo

using namespace sivo;

struct sivo_segnet { SegNet* impl; };
struct sivo_orb { Orb* impl; };

extern "C" {

const char* sivo_last_error(void) { return g_last_error.c_str(); }
const char* sivo_version(void) { return "sivo_b200 0.1 (sm_100a)"; }

int sivo_segnet_create_ex(const char* prototxt, const char* caffemodel, const sivo_segnet_options* opt, sivo_segnet_t** out) {
  return guarded([&] {
    if (!out) fail(SIVO_EINVAL, "null output handle");
    *out = nullptr;
    sivo_segnet_options o{};
    if (opt) o = *opt;
    auto* impl = new SegNet(prototxt ? prototxt : "", caffemodel ? caffemodel : "", o);
    *out = new sivo_segnet{impl};
  });
}

int sivo_segnet_create_shard(const char* prototxt, const char* caffemodel, const sivo_segnet_options* opt, int first_sample,
                             int n_samples, sivo_segnet_t** out) {
  return guarded([&] {
    if (!out) fail(SIVO_EINVAL, "null output handle");
    *out = nullptr;
    if (n_samples < 1) fail(SIVO_EINVAL, "sample shard: n_samples = %d (need at least 1)", n_samples);
    sivo_segnet_options o{};
    if (opt) o = *opt;
    auto* impl = new SegNet(prototxt ? prototxt : "", caffemodel ? caffemodel : "", o, first_sample, n_samples);
    *out = new sivo_segnet{impl};
  });
}

int sivo_segnet_create(const char* prototxt, const char* caffemodel, int device, uint64_t seed, sivo_segnet_t** out) {
  sivo_segnet_options o{};
  o.device = device;
  o.seed = seed;
  // knobs with no slot in the reference's constructor come from the environment (the C++ shim calls this entry point):
  // SIVO_B200_PRECISION = fp16 (default: the fast mode) | fp32 (strict: split-operand tensor-core convolutions, fp32 activations);
  // SIVO_B200_ENGINE = auto | simt | tcgen05
  if (const char* e = std::getenv("SIVO_B200_PRECISION")) o.precision = (std::string(e) == "fp32") ? SIVO_PRECISION_FP32 : SIVO_PRECISION_FP16;
  if (const char* e = std::getenv("SIVO_B200_ENGINE"))
    o.engine = std::string(e) == "simt" ? SIVO_ENGINE_SIMT : std::string(e) == "tcgen05" ? SIVO_ENGINE_TCGEN05 : SIVO_ENGINE_AUTO;
  return sivo_segnet_create_ex(prototxt, caffemodel, &o, out);
}

int sivo_segnet_geometry(const sivo_segnet_t* h, int* width, int* height, int* T, int* n_classes) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    if (width) *width = h->impl->width();
    if (height) *height = h->impl->height();
    if (T) *T = h->impl->T();
    if (n_classes) *n_classes = h->impl->classes();
  });
}

int sivo_segnet_set_frame(sivo_segnet_t* h, uint64_t frame) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->set_frame(frame);
  });
}

int sivo_segnet_set_profiling(sivo_segnet_t* h, int on) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->set_profiling(on != 0);
  });
}

int sivo_segnet_run(sivo_segnet_t* h, const uint8_t* bgr, int rows, int cols, size_t stride, uint8_t* classes,
                    double* confidence, double* entropy) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->run_host(bgr, rows, cols, stride, classes, confidence, entropy);
  });
}

int sivo_segnet_run_device(sivo_segnet_t* h, const uint8_t* bgr_device, uint8_t* classes_device, double* confidence_device,
                           double* entropy_device, void* stream) {
  return guarded([&] {
    if (!h || !bgr_device) fail(SIVO_EINVAL, "null handle or image");
    h->impl->run_device(bgr_device, classes_device, confidence_device, entropy_device, static_cast<cudaStream_t>(stream));
  });
}

int sivo_segnet_set_record_outputs(sivo_segnet_t* h, uint8_t* classes_device, float* confidence_f32_device, float* entropy_f32_device) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->set_record_outputs(classes_device, confidence_f32_device, entropy_f32_device);
  });
}

int sivo_segnet_run_device_maps(sivo_segnet_t* h, const uint8_t* bgr_device, uint8_t* classes_device, double* confidence_device,
                                double* entropy_device, float* confidence_f32_device, float* entropy_f32_device, void* stream) {
  return guarded([&] {
    if (!h || !bgr_device) fail(SIVO_EINVAL, "null handle or image");
    h->impl->run_device(bgr_device, classes_device, confidence_device, entropy_device, static_cast<cudaStream_t>(stream),
                        confidence_f32_device, entropy_f32_device);
  });
}

int sivo_segnet_run_device_partial(sivo_segnet_t* h, const uint8_t* bgr_device, double* prob_sum_device, int accumulate, void* stream) {
  return guarded([&] {
    if (!h || !bgr_device) fail(SIVO_EINVAL, "null handle or image");
    h->impl->run_device_partial(bgr_device, prob_sum_device, accumulate, static_cast<cudaStream_t>(stream));
  });
}

int sivo_segnet_finalize_device(sivo_segnet_t* h, const double* prob_sum_device, uint8_t* classes_device, double* confidence_device,
                                double* entropy_device, float* confidence_f32_device, float* entropy_f32_device, void* stream) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->finalize_device(prob_sum_device, classes_device, confidence_device, entropy_device, confidence_f32_device, entropy_f32_device,
                             static_cast<cudaStream_t>(stream));
  });
}

int sivo_segnet_blob(sivo_segnet_t* h, const char* name, float* out, size_t cap, int* n, int* c, int* hh, int* ww) {
  return guarded([&] {
    if (!h || !name) fail(SIVO_EINVAL, "null handle or name");
    h->impl->blob(name, out, cap, n, c, hh, ww);
  });
}

int sivo_segnet_last_timing(const sivo_segnet_t* h, float* conv_ms, float* other_ms, float* reduce_ms, float* total_ms,
                            int* launches) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    if (conv_ms) *conv_ms = h->impl->conv_ms;
    if (other_ms) *other_ms = h->impl->other_ms;
    if (reduce_ms) *reduce_ms = h->impl->reduce_ms;
    if (total_ms) *total_ms = h->impl->total_ms;
    if (launches) *launches = h->impl->launches;
  });
}

int sivo_segnet_semantic_keys(sivo_segnet_t* h, const sivo_keypoint* kps, int n, int max_static_class, uint8_t* kp_class, double* kp_conf,
                              double* kp_entropy, int* keep_idx, int* n_keep) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->semantic_keys(kps, n, max_static_class, kp_class, kp_conf, kp_entropy, keep_idx, n_keep);
  });
}

int sivo_segnet_op_timing(const sivo_segnet_t* h, int index, char* name, size_t cap, float* ms, double* flops, int* n_ops) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    const int n = static_cast<int>(h->impl->n_ops());
    if (n_ops) *n_ops = n;
    if (index < 0) return;  // count query
    if (index >= n) fail(SIVO_ERANGE, "op index %d out of range (%d launches)", index, n);
    const Op& op = h->impl->op_at(index);
    if (name && cap) snprintf(name, cap, "%s", op.layer.c_str());
    if (ms) *ms = static_cast<size_t>(index) < h->impl->op_ms.size() ? h->impl->op_ms[index] : 0.f;
    if (flops) *flops = op.kind == Op::Conv ? op.flops : 0.0;
  });
}

int sivo_segnet_op_flops_executed(const sivo_segnet_t* h, int index, double* flops) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    const int n = static_cast<int>(h->impl->n_ops());
    if (index < 0 || index >= n) fail(SIVO_ERANGE, "op index %d out of range (%d launches)", index, n);
    const Op& op = h->impl->op_at(index);
    if (flops) *flops = op.kind == Op::Conv ? op.flops_exec : 0.0;
  });
}

int sivo_segnet_flops(const sivo_segnet_t* h, double* dedup, double* naive) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    if (dedup) *dedup = h->impl->flops_dedup;
    if (naive) *naive = h->impl->flops_naive;
  });
}

void sivo_segnet_destroy(sivo_segnet_t* h) {
  if (!h) return;
  delete h->impl;
  delete h;
}

// ---------------------------------------------------------------------------------------- ORB
int sivo_orb_create(int nfeatures, float scale_factor, int nlevels, int ini_th_fast, int min_th_fast, int device,
                    sivo_orb_t** out) {
  return guarded([&] {
    if (!out) fail(SIVO_EINVAL, "null output handle");
    *out = nullptr;
    auto* impl = new Orb(nfeatures, scale_factor, nlevels, ini_th_fast, min_th_fast, device);
    *out = new sivo_orb{impl};
  });
}

int sivo_orb_tables(const sivo_orb_t* h, float* scale, float* inv_scale, float* sigma2, float* inv_sigma2, int* per_level) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    const OrbTables& t = h->impl->tables();
    size_t n = t.scale.size();
    if (scale) memcpy(scale, t.scale.data(), n * sizeof(float));
    if (inv_scale) memcpy(inv_scale, t.inv_scale.data(), n * sizeof(float));
    if (sigma2) memcpy(sigma2, t.sigma2.data(), n * sizeof(float));
    if (inv_sigma2) memcpy(inv_sigma2, t.inv_sigma2.data(), n * sizeof(float));
    if (per_level) memcpy(per_level, t.per_level.data(), n * sizeof(int));
  });
}

int sivo_orb_run(sivo_orb_t* h, const uint8_t* gray, int rows, int cols, size_t stride, sivo_keypoint* kps, int cap, int* n,
                 uint8_t* desc32, uint8_t* const* pyramid_levels, const size_t* pyramid_strides) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->run(gray, rows, cols, stride, kps, cap, n, desc32, pyramid_levels, pyramid_strides);
  });
}

int sivo_orb_run_device_input(sivo_orb_t* h, const uint8_t* gray_device, int rows, int cols, size_t pitch, sivo_keypoint* kps,
                              int cap, int* n, uint8_t* desc32) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->run(gray_device, rows, cols, pitch, kps, cap, n, desc32, nullptr, nullptr, true);
  });
}

int sivo_orb_enqueue_device(sivo_orb_t* h, const uint8_t* gray_device, int rows, int cols, size_t pitch, sivo_keypoint* kps_device,
                            uint8_t* desc32_device, long long* count_device) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->enqueue_device(gray_device, rows, cols, pitch, kps_device, desc32_device, count_device);
  });
}

int sivo_orb_stream_wait(sivo_orb_t* h, void* consumer_cuda_stream) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->stream_wait(static_cast<cudaStream_t>(consumer_cuda_stream));
  });
}

int sivo_orb_wait_for_stream(sivo_orb_t* h, void* producer_cuda_stream) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->wait_for_stream(static_cast<cudaStream_t>(producer_cuda_stream));
  });
}

int sivo_orb_wait_event(sivo_orb_t* h, void* cuda_event) {
  return guarded([&] {
    if (!h || !cuda_event) fail(SIVO_EINVAL, "null argument");
    h->impl->wait_event(static_cast<cudaEvent_t>(cuda_event));
  });
}

int sivo_orb_device_status(sivo_orb_t* h, int* level_mask) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    const int m = h->impl->device_tree_status();
    if (level_mask) *level_mask = m;
  });
}

int sivo_orb_has_device_tree(const sivo_orb_t* h, int* yes) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    if (yes) *yes = h->impl->device_tree() ? 1 : 0;
  });
}

int sivo_orb_capacity(const sivo_orb_t* h, int* max_keypoints) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    if (max_keypoints) *max_keypoints = h->impl->capacity();
  });
}

int sivo_orb_level_size(const sivo_orb_t* h, int rows, int cols, int level, int* level_w, int* level_h) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->level_size(rows, cols, level, level_w, level_h);
  });
}

int sivo_orb_candidates(const sivo_orb_t* h, int level, int* xs, int* ys, int* resp, int cap, int* n) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    h->impl->candidates(level, xs, ys, resp, cap, n);
  });
}

int sivo_orb_last_timing(const sivo_orb_t* h, float* device_ms, float* host_tree_ms, int* launches) {
  return guarded([&] {
    if (!h) fail(SIVO_EINVAL, "null handle");
    if (device_ms) *device_ms = h->impl->device_ms;
    if (host_tree_ms) *host_tree_ms = h->impl->tree_ms;
    if (launches) *launches = h->impl->launches;
  });
}

void sivo_orb_destroy(sivo_orb_t* h) {
  if (!h) return;
  delete h->impl;
  delete h;
}

int sivo_orb_distribute(const float* xs, const float* ys, const float* resp, int n, int min_x, int max_x, int min_y, int max_y,
                        int n_target, int* keep, int cap) {
  int count = 0;
  int rc = guarded([&] {
    if (n > 0 && (!xs || !ys || !resp)) fail(SIVO_EINVAL, "null keypoint arrays");
    if (max_x <= min_x || max_y <= min_y) fail(SIVO_EINVAL, "empty distribution rectangle");
    std::vector<int> k = orb_distribute(xs, ys, resp, n, min_x, max_x, min_y, max_y, n_target);
    if (static_cast<int>(k.size()) > cap) fail(SIVO_ERANGE, "%zu kept keypoints, buffer holds %d", k.size(), cap);
    if (keep) memcpy(keep, k.data(), k.size() * sizeof(int));
    count = static_cast<int>(k.size());
  });
  return rc == SIVO_OK ? count : rc;
}

int sivo_dbg_orb_distribute_device(int device, const int* xs, const int* ys, const int* resp, int n, int min_x, int max_x, int min_y,
                                   int max_y, int n_target, int* out_x, int* out_y, int* out_resp, int cap) {
  int count = 0;
  int rc = guarded([&] {
    if (n > 0 && (!xs || !ys || !resp)) fail(SIVO_EINVAL, "null keypoint arrays");
    if (max_x <= min_x || max_y <= min_y) fail(SIVO_EINVAL, "empty distribution rectangle");
    SIVO_CUDA(cudaSetDevice(device));
    orb_tree_configure();
    OrbTreeParams prm{};
    int n_ini = static_cast<int>(std::round(static_cast<float>(max_x - min_x) / (max_y - min_y)));
    if (n_ini < 1) n_ini = 1;
    prm.n_target[0] = n_target; prm.n_ini[0] = n_ini; prm.height[0] = max_y - min_y;
    prm.hx[0] = static_cast<float>(max_x - min_x) / n_ini;
    prm.scale[0] = 1.f; prm.size[0] = 31.f; prm.min_b = 0;
    std::vector<uint32_t> packed(std::max(n, 1));
    for (int i = 0; i < n; ++i) {
      if (xs[i] < 0 || xs[i] > 4095 || ys[i] < 0 || ys[i] > 4095 || resp[i] < 0 || resp[i] > 255) fail(SIVO_EINVAL, "key %d out of range", i);
      packed[i] = static_cast<uint32_t>(xs[i]) | (static_cast<uint32_t>(ys[i]) << 12) | (static_cast<uint32_t>(resp[i]) << 24);
    }
    const int off[2] = {0, n};
    DevBuf d_cand(packed.size() * 4), d_off(sizeof off), d_sel(static_cast<size_t>(kTreeSelCap) * 4), d_cnt(2 * sizeof(int));
    SIVO_CUDA(cudaMemcpy(d_cand.p, packed.data(), packed.size() * 4, cudaMemcpyHostToDevice));
    SIVO_CUDA(cudaMemcpy(d_off.p, off, sizeof off, cudaMemcpyHostToDevice));
    SIVO_CUDA(cudaMemset(d_cnt.p, 0, 2 * sizeof(int)));
    orb_launch_distribute(d_cand.as<uint32_t>(), d_off.as<int>(), nullptr, nullptr, prm, 1, d_sel.as<uint32_t>(), d_cnt.as<int>(), d_cnt.as<int>() + 1, nullptr);
    int ce[2] = {0, 0};
    SIVO_CUDA(cudaMemcpy(ce, d_cnt.p, sizeof ce, cudaMemcpyDeviceToHost));
    if (ce[1]) fail(SIVO_ERANGE, "input exceeds the device quad tree's capacity");
    if (ce[0] > cap) fail(SIVO_ERANGE, "%d kept keypoints, buffer holds %d", ce[0], cap);
    std::vector<uint32_t> sel(std::max(ce[0], 1));
    SIVO_CUDA(cudaMemcpy(sel.data(), d_sel.p, static_cast<size_t>(ce[0]) * 4, cudaMemcpyDeviceToHost));
    for (int i = 0; i < ce[0]; ++i) {
      if (out_x) out_x[i] = static_cast<int>(sel[i] & 0xFFF);
      if (out_y) out_y[i] = static_cast<int>((sel[i] >> 12) & 0xFFF);
      if (out_resp) out_resp[i] = static_cast<int>(sel[i] >> 24);
    }
    count = ce[0];
  });
  return rc == SIVO_OK ? count : rc;
}

int sivo_stereo_hamming(int device, const sivo_keypoint* left, const uint8_t* desc_left, int n_left, const sivo_keypoint* right,
                        const uint8_t* desc_right, int n_right, const float* scale_factors, int nlevels, int rows, float min_d,
                        float max_d, int* best_idx, int* best_dist) {
  return guarded([&] {
    if (!scale_factors || !best_idx || !best_dist || (n_left && (!left || !desc_left)) || (n_right && (!right || !desc_right)))
      fail(SIVO_EINVAL, "null argument");
    stereo_hamming(device, left, desc_left, n_left, right, desc_right, n_right, scale_factors, nlevels, rows, min_d, max_d,
                   best_idx, best_dist);
  });
}

int sivo_hamming_best2(int device, const uint8_t* query_desc, int n_query, const uint8_t* train_desc, int n_train,
                       const int* cand_offsets, const int* cand_idx, const int* train_level, int* out5) {
  return guarded([&] {
    if (!out5 || !cand_offsets || (n_query && !query_desc) || (n_train && !train_desc) || (n_query > 0 && cand_offsets[n_query] && !cand_idx))
      fail(SIVO_EINVAL, "null argument");
    hamming_best2(device, query_desc, n_query, train_desc, n_train, cand_offsets, cand_idx, train_level, out5);
  });
}

int sivo_stereo_match(const sivo_orb_t* left, const sivo_orb_t* right, const sivo_keypoint* kp_left, const uint8_t* desc_left,
                      int n_left, const sivo_keypoint* kp_right, const uint8_t* desc_right, int n_right, float mb, float mbf,
                      float* u_right, float* depth) {
  return guarded([&] {
    if (!left || !right || !u_right || !depth || (n_left && (!kp_left || !desc_left)) || (n_right && (!kp_right || !desc_right)))
      fail(SIVO_EINVAL, "null argument");
    stereo_match(*left->impl, *right->impl, kp_left, desc_left, n_left, kp_right, desc_right, n_right, mb, mbf, u_right, depth);
  });
}

// ---------------------------------------------------------------------------------------- layer test hooks
namespace {
TensorView make_view(DevBuf& buf, int n, int c, int h, int w, int cs, DType dt) {
  TensorView v;
  v.n = n; v.c = c; v.h = h; v.w = w; v.cs = cs; v.dt = dt;
  buf.alloc(v.bytes());
  v.p = buf.p;
  return v;
}
void upload_nchw(const float* src, TensorView v) {
  size_t count = static_cast<size_t>(v.n) * v.c * v.h * v.w;
  DevBuf tmp(count * sizeof(float));
  SIVO_CUDA(cudaMemcpy(tmp.p, src, count * sizeof(float), cudaMemcpyHostToDevice));
  launch_nchw_to_act(tmp.as<float>(), v, nullptr);
  SIVO_CUDA(cudaDeviceSynchronize());
}
void download_nchw(TensorView v, float* dst) {
  size_t count = static_cast<size_t>(v.n) * v.c * v.h * v.w;
  DevBuf tmp(count * sizeof(float));
  launch_act_to_nchw(v, tmp.as<float>(), nullptr);
  SIVO_CUDA(cudaMemcpy(dst, tmp.p, count * sizeof(float), cudaMemcpyDeviceToHost));
}
}  // namespace

int sivo_dbg_pool(int device, const float* in, int n, int c, int h, int w, float* out, int* mask) {
  return guarded([&] {
    if (!in || n <= 0 || c <= 0 || (h & 1) || (w & 1)) fail(SIVO_EINVAL, "pool: bad arguments");
    SIVO_CUDA(cudaSetDevice(device));
    DevBuf bi, bo, bm(static_cast<size_t>(n) * c * (h / 2) * (w / 2)), bmi(static_cast<size_t>(n) * c * (h / 2) * (w / 2) * sizeof(int));
    TensorView vi = make_view(bi, n, c, h, w, c, DType::F32), vo = make_view(bo, n, c, h / 2, w / 2, c, DType::F32);
    upload_nchw(in, vi);
    launch_pool(vi, vo, bm.as<uint8_t>(), nullptr);
    if (out) download_nchw(vo, out);
    if (mask) {
      launch_mask_to_nchw(bm.as<uint8_t>(), n, c, h / 2, w / 2, bmi.as<int>(), nullptr);
      SIVO_CUDA(cudaMemcpy(mask, bmi.p, bmi.bytes, cudaMemcpyDeviceToHost));
    }
    SIVO_CUDA(cudaDeviceSynchronize());
  });
}

int sivo_dbg_unpool(int device, const float* in, const int* mask, int n, int c, int h, int w, float* out) {
  return guarded([&] {
    if (!in || !mask || !out) fail(SIVO_EINVAL, "unpool: null argument");
    SIVO_CUDA(cudaSetDevice(device));
    size_t cnt = static_cast<size_t>(n) * c * h * w;
    DevBuf bi, bo, bm(cnt), bmi(cnt * sizeof(int));
    TensorView vi = make_view(bi, n, c, h, w, c, DType::F32), vo = make_view(bo, n, c, h * 2, w * 2, c, DType::F32);
    upload_nchw(in, vi);
    SIVO_CUDA(cudaMemcpy(bmi.p, mask, cnt * sizeof(int), cudaMemcpyHostToDevice));
    launch_mask_from_nchw(bmi.as<int>(), n, c, h, w, bm.as<uint8_t>(), nullptr);
    launch_unpool(vi, bm.as<uint8_t>(), n, vo, nullptr);
    download_nchw(vo, out);
    SIVO_CUDA(cudaDeviceSynchronize());
  });
}

int sivo_dbg_lrn(int device, const float* in, int n, int c, int h, int w, int size, float alpha, float beta, float k, float* out) {
  return guarded([&] {
    if (!in || !out) fail(SIVO_EINVAL, "lrn: null argument");
    SIVO_CUDA(cudaSetDevice(device));
    DevBuf bi, bo;
    int cs = (c + 3) / 4 * 4;
    TensorView vi = make_view(bi, n, c, h, w, cs, DType::F32), vo = make_view(bo, n, c, h, w, cs, DType::F32);
    upload_nchw(in, vi);
    launch_lrn(vi, vo, size, alpha, beta, k, nullptr);
    download_nchw(vo, out);
    SIVO_CUDA(cudaDeviceSynchronize());
  });
}

int sivo_dbg_mc_reduce(int device, const float* logits, int T, int c, int h, int w, uint8_t* classes, double* confidence,
                       double* entropy) {
  return guarded([&] {
    if (!logits || T <= 0 || c <= 0) fail(SIVO_EINVAL, "mc_reduce: bad arguments");
    SIVO_CUDA(cudaSetDevice(device));
    DevBuf bl, bc(static_cast<size_t>(h) * w), bf(static_cast<size_t>(h) * w * 8), be(static_cast<size_t>(h) * w * 8);
    int cs = (c + 15) / 16 * 16;
    TensorView vl = make_view(bl, T, c, h, w, cs, DType::F32);
    upload_nchw(logits, vl);
    launch_mc_reduce(static_cast<const float*>(vl.p), T, c, cs, h * w, bc.as<uint8_t>(), bf.as<double>(), be.as<double>(), nullptr);
    SIVO_CUDA(cudaDeviceSynchronize());
    if (classes) SIVO_CUDA(cudaMemcpy(classes, bc.p, static_cast<size_t>(h) * w, cudaMemcpyDeviceToHost));
    if (confidence) SIVO_CUDA(cudaMemcpy(confidence, bf.p, static_cast<size_t>(h) * w * 8, cudaMemcpyDeviceToHost));
    if (entropy) SIVO_CUDA(cudaMemcpy(entropy, be.p, static_cast<size_t>(h) * w * 8, cudaMemcpyDeviceToHost));
  });
}

int sivo_dbg_mc_partial(int device, const float* logits, int T, int c, int h, int w, int accumulate, double* sums) {
  return guarded([&] {
    if (!logits || !sums || T <= 0 || c <= 0 || c > 16) fail(SIVO_EINVAL, "mc_partial: bad arguments");
    SIVO_CUDA(cudaSetDevice(device));
    const size_t bytes = static_cast<size_t>(c) * h * w * sizeof(double);
    DevBuf bl, bs(bytes);
    TensorView vl = make_view(bl, T, c, h, w, 16, DType::F32);
    upload_nchw(logits, vl);
    if (accumulate) SIVO_CUDA(cudaMemcpy(bs.p, sums, bytes, cudaMemcpyHostToDevice));
    launch_mc_partial(static_cast<const float*>(vl.p), T, c, 16, h * w, bs.as<double>(), accumulate, nullptr);
    SIVO_CUDA(cudaDeviceSynchronize());
    SIVO_CUDA(cudaMemcpy(sums, bs.p, bytes, cudaMemcpyDeviceToHost));
  });
}

int sivo_dbg_mc_finalize(int device, const double* sums, int T_total, int c, int h, int w, uint8_t* classes, double* confidence,
                         double* entropy) {
  return guarded([&] {
    if (!sums || T_total <= 0 || c <= 0 || c > 16) fail(SIVO_EINVAL, "mc_finalize: bad arguments");
    SIVO_CUDA(cudaSetDevice(device));
    const size_t hw = static_cast<size_t>(h) * w;
    DevBuf bs(static_cast<size_t>(c) * hw * sizeof(double)), bc(hw), bf(hw * 8), be(hw * 8);
    SIVO_CUDA(cudaMemcpy(bs.p, sums, bs.bytes, cudaMemcpyHostToDevice));
    launch_mc_finalize(bs.as<double>(), T_total, c, static_cast<int>(hw), bc.as<uint8_t>(), bf.as<double>(), be.as<double>(), nullptr,
                       nullptr, nullptr);
    SIVO_CUDA(cudaDeviceSynchronize());
    if (classes) SIVO_CUDA(cudaMemcpy(classes, bc.p, hw, cudaMemcpyDeviceToHost));
    if (confidence) SIVO_CUDA(cudaMemcpy(confidence, bf.p, hw * 8, cudaMemcpyDeviceToHost));
    if (entropy) SIVO_CUDA(cudaMemcpy(entropy, be.p, hw * 8, cudaMemcpyDeviceToHost));
  });
}

int sivo_dbg_dropout_mask(int device, uint64_t seed, uint64_t frame, int layer, int T, int c, int h, int w, uint8_t* keep) {
  return guarded([&] {
    if (!keep) fail(SIVO_EINVAL, "dropout_mask: null output");
    SIVO_CUDA(cudaSetDevice(device));
    size_t cnt = static_cast<size_t>(T) * c * h * w;
    DevBuf bk(cnt), bf(8);
    SIVO_CUDA(cudaMemcpy(bf.p, &frame, 8, cudaMemcpyHostToDevice));
    launch_dropout_bits(seed, bf.as<uint64_t>(), layer, T, c, h, w, bk.as<uint8_t>(), nullptr);
    SIVO_CUDA(cudaMemcpy(keep, bk.p, cnt, cudaMemcpyDeviceToHost));
  });
}

int sivo_dbg_conv(int device, int engine, int precision, const float* in, int n, int cin, int h, int w, const float* weight,
                  const float* bias, const float* bn_scale, const float* bn_shift, int cout, int k, int pad, int relu,
                  float* out) {
  return guarded([&] {
    if (!in || !weight || !out) fail(SIVO_EINVAL, "conv: null argument");
    if (pad != (k - 1) / 2) fail(SIVO_EINVAL, "conv: only 'same' padding");
    SIVO_CUDA(cudaSetDevice(device));
    DType dt = precision == SIVO_PRECISION_FP32 ? DType::F32 : DType::F16;
    int cs_in = cin < 8 ? 4 : cin;
    if (cin >= 8 && cin % 8) fail(SIVO_EINVAL, "conv: cin must be 3/4 or a multiple of 8");
    DevBuf bi, bo;
    TensorView vi = make_view(bi, n, cin, h, w, cs_in, dt);
    int cs_out = (cout % 8) ? (cout + 15) / 16 * 16 : cout;
    DType odt = (cout % 8) ? DType::F32 : dt;
    TensorView vo = make_view(bo, n, cout, h, w, cs_out, odt);
    upload_nchw(in, vi);
    Op op;
    op.kind = Op::Conv;
    op.layer = "dbg_conv";
    op.k = k; op.pad = pad; op.cin = cin; op.cout = cout; op.cin_p = cs_in; op.cout_p = (cout + 63) / 64 * 64;
    op.relu = relu != 0;
    // weights through the same preparation the executor uses
    auto th = [&](float x) { return dt == DType::F16 ? __half2float(__float2half_rn(x)) : x; };
    std::vector<float> ws(static_cast<size_t>(k) * k * op.cin_p * op.cout_p, 0.f);
    std::vector<__half> wt(static_cast<size_t>(k) * k * op.cout_p * op.cin_p, __float2half_rn(0.f));
    for (int co = 0; co < cout; ++co)
      for (int ci = 0; ci < cin; ++ci)
        for (int t = 0; t < k * k; ++t) {
          float v = weight[(static_cast<size_t>(co) * cin + ci) * k * k + t];
          ws[(static_cast<size_t>(t) * op.cin_p + ci) * op.cout_p + co] = th(v);
          wt[(static_cast<size_t>(t) * op.cout_p + co) * op.cin_p + ci] = __float2half_rn(v);
        }
    std::vector<float> b(op.cout_p, 0.f), sc(op.cout_p, 1.f), sh(op.cout_p, 0.f);
    if (bias) std::copy(bias, bias + cout, b.begin());
    if (bn_scale) std::copy(bn_scale, bn_scale + cout, sc.begin());
    if (bn_shift) std::copy(bn_shift, bn_shift + cout, sh.begin());
    op.h_bias = b; op.h_bn_scale = sc; op.h_bn_shift = sh;
    op.w_simt.alloc(ws.size() * 4);
    op.w_tc.alloc(wt.size() * 2);
    op.bias.alloc(b.size() * 4);
    op.bn_scale.alloc(sc.size() * 4);
    op.bn_shift.alloc(sh.size() * 4);
    SIVO_CUDA(cudaMemcpy(op.w_simt.p, ws.data(), ws.size() * 4, cudaMemcpyHostToDevice));
    SIVO_CUDA(cudaMemcpy(op.w_tc.p, wt.data(), wt.size() * 2, cudaMemcpyHostToDevice));
    if ((k == 7 || k == 3) && cin == 64 && cout == 64) {
      std::vector<__half> wp = conv_tc_pair_weights(weight, k);
      op.w_tc_pair.alloc(wp.size() * 2);
      SIVO_CUDA(cudaMemcpy(op.w_tc_pair.p, wp.data(), wp.size() * 2, cudaMemcpyHostToDevice));
    }
    SIVO_CUDA(cudaMemcpy(op.bias.p, b.data(), b.size() * 4, cudaMemcpyHostToDevice));
    SIVO_CUDA(cudaMemcpy(op.bn_scale.p, sc.data(), sc.size() * 4, cudaMemcpyHostToDevice));
    SIVO_CUDA(cudaMemcpy(op.bn_shift.p, sh.data(), sh.size() * 4, cudaMemcpyHostToDevice));
    op.has_bn = bn_scale != nullptr;
    // tensors for the tc plan live in a scratch vector; run on the default stream
    if (engine == SIVO_ENGINE_TCGEN05 && dt == DType::F32) {  // split-operand fp32 mode
      TensorView vs = vi;
      vs.dt = DType::F16;
      vs.cs = 2 * vi.cs;
      op.split = true;
      if (cin % 64 || !conv_tc_supported(op, vs, vo)) fail(SIVO_EINVAL, "conv: shape not supported by the split-operand tcgen05 mode");
      std::vector<__half> wsplit = conv_tc_split_weights(weight, cout, cin, k, op.cout_p, op.cin_p, &op.acc_scale);
      op.w_tc.alloc(wsplit.size() * 2);
      SIVO_CUDA(cudaMemcpy(op.w_tc.p, wsplit.data(), wsplit.size() * 2, cudaMemcpyHostToDevice));
      op.a_split.alloc(vs.elems() * 2);
      vs.p = op.a_split.p;
      op.tc = conv_tc_plan(op, vs, vo, op.w_tc.p);
      launch_split_hilo(vi, op.a_split.p, nullptr);
      conv_tc_launch(*op.tc, op, nullptr);
    } else if (engine == SIVO_ENGINE_TCGEN05) {
      if (dt != DType::F16 || !conv_tc_supported(op, vi, vo)) fail(SIVO_EINVAL, "conv: shape not supported by the tcgen05 engine");
      op.tc = conv_tc_plan(op, vi, vo, op.w_tc.p);
      conv_tc_launch(*op.tc, op, nullptr);
    } else {
      ConvParams p;
      p.in = vi; p.out = vo;
      p.w_simt = op.w_simt.as<float>();
      p.bias = op.bias.as<float>();
      p.bn_scale = op.has_bn ? op.bn_scale.as<float>() : nullptr;
      p.bn_shift = op.has_bn ? op.bn_shift.as<float>() : nullptr;
      p.k = k; p.pad = pad; p.cin_p = op.cin_p; p.cout_p = op.cout_p; p.relu = op.relu; p.slope = 0.f;
      launch_conv_simt(p, nullptr);
    }
    SIVO_CUDA(cudaDeviceSynchronize());
    download_nchw(vo, out);
    SIVO_CUDA(cudaDeviceSynchronize());
  });
}

}  // extern "C"
