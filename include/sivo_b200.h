/* sivo_b200 -- C ABI of the B200-native SIVO perception front-end (libsivo_b200.so).
 *
 * The reference has no FFI on this path: the "plugin API" is two C++ classes.  The shim classes in
 * integration/ keep their public signatures and forward to the entry points below, so src/sivo.cc,
 * src/orbslam/System.cc, Tracking.cc and Frame.cc compile unchanged (see INTEGRATION.md).
 *
 *   sivo_segnet_*   replaces  SIVO::BayesianSegNet            include/bayesian_segnet/bayesian_segnet.hpp:108-170
 *                             ctor                             src/bayesian_segnet/bayesian_segnet.cpp:46-78
 *                             segmentImage                     src/bayesian_segnet/bayesian_segnet.cpp:299-318
 *                             getInputGeometry                 include/bayesian_segnet/bayesian_segnet.hpp:139
 *   sivo_orb_*      replaces  SIVO::ORBextractor              include/orbslam/ORBextractor.h:46-125
 *                             ctor                             src/orbslam/ORBextractor.cc:412-475
 *                             operator()                       src/orbslam/ORBextractor.cc:1019-1083
 *                             mvImagePyramid (public member)   include/orbslam/ORBextractor.h:90
 *   sivo_stereo_*   replaces  the Hamming stage of Frame::ComputeStereoMatches   src/orbslam/Frame.cc:444-533
 *                             ORBmatcher::DescriptorDistance   src/orbslam/ORBmatcher.cc:1582-1596
 *
 * Conventions: every function returns 0 on success or a negative SIVO_E* code and never throws or aborts
 * across the boundary; sivo_last_error() returns a thread-local message for the last failure on the
 * calling thread.  Pointers are plain host pointers unless the name says `_device`.  Handles are
 * independent: two sivo_orb_t may be driven concurrently from two threads (Frame.cc:126-129); one handle
 * must not be used from two threads at once.
 */
#ifndef SIVO_B200_H_
#define SIVO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIVO_OK 0
#define SIVO_EINVAL (-22)   /* bad argument; the shim rethrows std::invalid_argument where the reference does */
#define SIVO_ENOENT (-2)    /* prototxt / caffemodel not readable */
#define SIVO_EFORMAT (-74)  /* prototxt / caffemodel malformed, unsupported layer, LFS stub, shape mismatch */
#define SIVO_ECUDA (-5)     /* CUDA runtime / driver error (message has the cudaError string) */
#define SIVO_ENOMEM (-12)
#define SIVO_ERANGE (-34)   /* output capacity too small */

typedef struct sivo_segnet sivo_segnet_t;
typedef struct sivo_orb sivo_orb_t;

/* bit-compatible with cv::KeyPoint (pt.x, pt.y, size, angle, response, octave, class_id) */
typedef struct sivo_keypoint {
  float x, y, size, angle, response;
  int32_t octave, class_id;
} sivo_keypoint;

/* precision of the convolution operands (accumulation is always fp32, the MC reduction fp64) */
enum { SIVO_PRECISION_FP16 = 0, SIVO_PRECISION_FP32 = 1 };
/* convolution engine */
enum { SIVO_ENGINE_AUTO = 0, SIVO_ENGINE_SIMT = 1, SIVO_ENGINE_TCGEN05 = 2 };

typedef struct sivo_segnet_options {
  int32_t device;      /* CUDA device ordinal */
  int32_t T;           /* MC samples; 0 = take the prototxt's first input dim */
  uint64_t seed;       /* dropout seed (oracle/philox.py spells out the mask rule) */
  int32_t precision;   /* SIVO_PRECISION_* */
  int32_t engine;      /* SIVO_ENGINE_* */
  int32_t keep_blobs;  /* 1 = keep every intermediate blob for sivo_segnet_blob (tests); disables fusion */
  int32_t reserved;
} sivo_segnet_options;

/* ---- Bayesian SegNet -------------------------------------------------------------------------- */
/* Fails with SIVO_EINVAL for NULL/empty paths, input C != 3, T <= 1 (bayesian_segnet.cpp:65-70,80-89). */
int sivo_segnet_create(const char* prototxt, const char* caffemodel, int device, uint64_t seed,
                       sivo_segnet_t** out);
int sivo_segnet_create_ex(const char* prototxt, const char* caffemodel, const sivo_segnet_options* opt,
                          sivo_segnet_t** out);
/* Sample shard (latency mode of SURVEY 8e): a handle that computes Monte-Carlo samples [first_sample, first_sample + n_samples)
 * of T (opt->T, or the prototxt's first dim).  T keeps the reference's rule T >= 2; a shard may hold a single sample.  Its op
 * list has batch n_samples after the first sampling Dropout, and its dropout keys use the global sample index, so the shards
 * of [0, T) compute exactly the samples of one unsharded handle.  SIVO_EINVAL if first_sample < 0, n_samples < 1 or
 * first_sample + n_samples > T; SIVO_EFORMAT if the logits are not the 16-channel layout the MC kernels need.  On a shard with
 * n_samples < T, sivo_segnet_run / _run_device / _run_device_maps return SIVO_EINVAL (their mean would be over the wrong
 * sample count); a shard [0, T) behaves exactly like a handle from sivo_segnet_create_ex. */
int sivo_segnet_create_shard(const char* prototxt, const char* caffemodel, const sivo_segnet_options* opt,
                             int first_sample, int n_samples, sivo_segnet_t** out);
/* T is the total sample count, also for a shard. */
int sivo_segnet_geometry(const sivo_segnet_t* h, int* width, int* height, int* T, int* n_classes);
/* Dropout masks are keyed by (seed, frame, layer, sample, element); frame auto-increments per run. */
int sivo_segnet_set_frame(sivo_segnet_t* h, uint64_t frame);
/* segmentImage: bgr is rows x cols x 3 u8 with `stride` bytes per row; larger images are centre-cropped
 * (resizeImage, bayesian_segnet.cpp:142-162), smaller ones are SIVO_EINVAL.  Outputs are row-major
 * height x width (MatXu / MatXd layout, bayesian_segnet.hpp:46-50); any of them may be NULL. */
int sivo_segnet_run(sivo_segnet_t* h, const uint8_t* bgr, int rows, int cols, size_t stride,
                    uint8_t* classes, double* confidence, double* entropy);
/* Same with device-resident buffers (already cropped height x width x 3, tightly packed) on `stream`
 * (a cudaStream_t; NULL = the handle's own stream).  No host synchronisation. */
int sivo_segnet_run_device(sivo_segnet_t* h, const uint8_t* bgr_device, uint8_t* classes_device,
                           double* confidence_device, double* entropy_device, void* stream);
/* Multi-GPU callers share a packed per-frame record (SURVEY 8e): after this call every sivo_segnet_run additionally leaves the
 * classes (u8) and single-precision copies of the confidence / entropy maps at these DEVICE addresses, complete when it returns,
 * so the record's maps never travel host -> device.  All NULL switches it off. */
int sivo_segnet_set_record_outputs(sivo_segnet_t* h, uint8_t* classes_device, float* confidence_f32_device, float* entropy_f32_device);
/* The same with additional single-precision copies of the two maps (any output may be NULL): what the packed per-frame record
 * of the multi-GPU path carries (SURVEY 8e: classes u8 + entropy f32 + confidence f32), written straight into it by the MC
 * reduction; the double maps stay the operator's outputs (bayesian_segnet.cpp:192-203, 262-276 compute in double). */
int sivo_segnet_run_device_maps(sivo_segnet_t* h, const uint8_t* bgr_device, uint8_t* classes_device, double* confidence_device,
                                double* entropy_device, float* confidence_f32_device, float* entropy_f32_device, void* stream);
/* The whole op list with the final reduction replaced by the per-pixel sum, in double, over this handle's samples of the
 * softmax probabilities: prob_sum_device[c * H*W + p], n_classes planes.  accumulate = 0 overwrites, 1 adds to what is
 * there (in sample order, so shards run one after another into one buffer give the unsharded sums bit for bit).  No host
 * synchronisation; advances the frame counter like sivo_segnet_run_device.  A NULL stream is the handle's own stream, so
 * shards that share one buffer are ordered by passing them one stream (or by events). */
int sivo_segnet_run_device_partial(sivo_segnet_t* h, const uint8_t* bgr_device, double* prob_sum_device, int accumulate,
                                   void* stream);
/* classes / confidence / entropy (+ optional f32 copies; any output may be NULL) from the summed probabilities of all T
 * samples, with the arithmetic of the single-handle reduction: equal sums give bit-identical maps.  The maps become the
 * handle's last result, the one sivo_segnet_semantic_keys reads.  Does not advance the frame counter. */
int sivo_segnet_finalize_device(sivo_segnet_t* h, const double* prob_sum_device, uint8_t* classes_device,
                                double* confidence_device, double* entropy_device, float* confidence_f32_device,
                                float* entropy_f32_device, void* stream);
/* Test hook: copies blob `name` (any top in the prototxt; needs keep_blobs) to `out` as float NCHW.
 * `*n`, `*c`, `*hh`, `*ww` receive its shape; `out` may be NULL to query the shape only. */
int sivo_segnet_blob(sivo_segnet_t* h, const char* name, float* out, size_t cap, int* n, int* c, int* hh,
                     int* ww);
/* Enables per-op CUDA-event timing (adds a host sync per run); off by default. */
/* Frame::SelectSemanticKeys (Frame.cc:177-203) plus the per-keypoint reads of the three maps that Tracking / LocalMapping
 * do later (Tracking.cc:487,538; LocalMapping.cc:483-485), evaluated on the device-resident maps of the last
 * sivo_segnet_run / _run_device -- so a caller that only needs per-keypoint values can pass NULL maps to sivo_segnet_run
 * and skip the 6.1 MB read-back.  For keypoint i: (row, col) = ((int) y, (int) x); kp_class/kp_conf/kp_entropy[i] = the map
 * values there (class 255, 0, 0 and never kept if outside the maps -- the reference would read out of bounds).
 * keep_idx[0..*n_keep) = indices with class <= max_static_class (Classes::TERRAIN = 8 in the reference), ascending, i.e. the
 * order mvKeysSemantic / mDescriptorsSemantic are built in.  Any output pointer may be NULL. */
int sivo_segnet_semantic_keys(sivo_segnet_t* h, const sivo_keypoint* kps, int n, int max_static_class, uint8_t* kp_class,
                              double* kp_conf, double* kp_entropy, int* keep_idx, int* n_keep);
int sivo_segnet_set_profiling(sivo_segnet_t* h, int on);
/* Per-stage device times (ms) of the last run: conv, other layers, MC reduction, total; counts kernels. */
int sivo_segnet_last_timing(const sivo_segnet_t* h, float* conv_ms, float* other_ms, float* reduce_ms,
                            float* total_ms, int* launches);
int sivo_segnet_flops(const sivo_segnet_t* h, double* conv_flops_dedup, double* conv_flops_naive);
/* One launch of the op list (index < 0: only `*n_ops`): layer name(s) it covers, its time in the last profiled run
 * (ms, CUDA events on the launching stream) and its algorithmic convolution flops (0 for non-convolution launches). */
int sivo_segnet_op_timing(const sivo_segnet_t* h, int index, char* name, size_t cap, float* ms, double* flops,
                          int* n_ops);
/* Multiply-add work a launch EXECUTES on the tensor / CUDA cores, as flops (2 x MACs).  Equals the algorithmic figure of
 * sivo_segnet_op_timing except where the library changes the operation count: the composed conv_decode1 x classifier layer
 * (one 64 -> 16 7x7 convolution instead of 64 -> 64 followed by 64 -> 15: 0.25x) and the split-operand fp32 mode (3x). */
int sivo_segnet_op_flops_executed(const sivo_segnet_t* h, int index, double* flops);
void sivo_segnet_destroy(sivo_segnet_t* h);

/* ---- ORB extractor ---------------------------------------------------------------------------- */
int sivo_orb_create(int nfeatures, float scale_factor, int nlevels, int ini_th_fast, int min_th_fast,
                    int device, sivo_orb_t** out);
/* Scale tables, each `nlevels` floats (GetScaleFactors & co, ORBextractor.h:66-88); any may be NULL. */
int sivo_orb_tables(const sivo_orb_t* h, float* scale, float* inv_scale, float* sigma2, float* inv_sigma2,
                    int* features_per_level);
/* operator(): gray is rows x cols u8.  Writes up to `cap` keypoints (level-major order) and cap x 32
 * descriptor bytes, *n = count (SIVO_ERANGE if cap is too small; nfeatures + 3*nlevels always suffices).
 * If pyramid_levels != NULL it must hold nlevels host pointers to buffers of
 * (level_h + 38) * pyramid_strides[l] bytes which receive the bordered level images, i.e. what
 * mvImagePyramid[l] is a (19,19)-offset ROI of (query sizes with sivo_orb_level_size). */
int sivo_orb_run(sivo_orb_t* h, const uint8_t* gray, int rows, int cols, size_t stride, sivo_keypoint* kps,
                 int cap, int* n, uint8_t* desc32, uint8_t* const* pyramid_levels,
                 const size_t* pyramid_strides);
/* Same operator with the gray image already resident in device memory (`pitch` bytes per row); the
 * candidate / selection round trip through the host quad tree stays inside the call. */
int sivo_orb_run_device_input(sivo_orb_t* h, const uint8_t* gray_device, int rows, int cols, size_t pitch,
                              sivo_keypoint* kps, int cap, int* n, uint8_t* desc32);
/* Fully asynchronous operator for device-resident pipelines (frame sharding across GPUs, CUDA-graph style callers): enqueues
 * pyramid -> FAST -> cells -> device quad tree -> blur -> rBRIEF on the handle's own stream and returns without synchronising.
 * kps_device needs room for sivo_orb_capacity(h) records, desc32_device for 32 bytes each; *count_device (int64) receives the
 * keypoint count.  sivo_orb_stream_wait makes another stream wait for the enqueued work; sivo_orb_device_status (synchronises)
 * returns a non-zero level mask if a level exceeded the device tree's capacity (use sivo_orb_run for such inputs). */
int sivo_orb_enqueue_device(sivo_orb_t* h, const uint8_t* gray_device, int rows, int cols, size_t pitch, sivo_keypoint* kps_device,
                            uint8_t* desc32_device, long long* count_device);
int sivo_orb_stream_wait(sivo_orb_t* h, void* consumer_cuda_stream);
/* The reverse edge: the handle's stream waits for everything enqueued on `producer_cuda_stream` so far (e.g. the collective
 * that still reads the buffers the next sivo_orb_enqueue_device will overwrite). */
int sivo_orb_wait_for_stream(sivo_orb_t* h, void* producer_cuda_stream);
/* The same edge for one recorded event (a cudaEvent_t): the handle's stream waits for exactly that point of another stream. */
int sivo_orb_wait_event(sivo_orb_t* h, void* cuda_event);
int sivo_orb_device_status(sivo_orb_t* h, int* level_mask);
int sivo_orb_capacity(const sivo_orb_t* h, int* max_keypoints);
int sivo_orb_has_device_tree(const sivo_orb_t* h, int* yes);
int sivo_orb_level_size(const sivo_orb_t* h, int rows, int cols, int level, int* level_w, int* level_h);
/* Test hook: FAST candidates of the last run before the quad tree, per level (x, y relative to the
 * (16,16) border origin as in ComputeKeyPointsOctTree, response). */
int sivo_orb_candidates(const sivo_orb_t* h, int level, int* xs, int* ys, int* resp, int cap, int* n);
int sivo_orb_last_timing(const sivo_orb_t* h, float* device_ms, float* host_tree_ms, int* launches);
void sivo_orb_destroy(sivo_orb_t* h);

/* Host-only DistributeOctTree (ORBextractor.cc:544-750), exported so that the shim, the library and the
 * tests share one implementation of the documented tie rule.  Returns the number of kept indices. */
int sivo_orb_distribute(const float* xs, const float* ys, const float* resp, int n, int min_x, int max_x,
                        int min_y, int max_y, int n_target, int* keep, int cap);

/* Test hook: the same distribution on the DEVICE quad tree (orb_tree.cu), integer key coordinates < 4096 and responses < 256
 * as the FAST stage produces them.  Writes the kept keys' (x, y, response) in list order; returns their count, or
 * SIVO_ERANGE if the input exceeds the device tree's capacity. */
int sivo_dbg_orb_distribute_device(int device, const int* xs, const int* ys, const int* resp, int n, int min_x, int max_x,
                                   int min_y, int max_y, int n_target, int* out_x, int* out_y, int* out_resp, int cap);

/* ---- stereo Hamming stage (next-row 1) -------------------------------------------------------- */
/* For each left keypoint: best right candidate in its row band (rows vL +- 2*scale[octave]), octave
 * within +-1, uR in [uL - max_d, uL - min_d], minimal DescriptorDistance; best_idx = -1 if none.
 * Mirrors Frame.cc:452-533 up to (not including) the SAD refinement. */
int sivo_stereo_hamming(int device, const sivo_keypoint* left, const uint8_t* desc_left, int n_left,
                        const sivo_keypoint* right, const uint8_t* desc_right, int n_right,
                        const float* scale_factors, int nlevels, int rows, float min_d, float max_d,
                        int* best_idx, int* best_dist);

/* The whole of Frame::ComputeStereoMatches (Frame.cc:444-629): Hamming search, 11x11 SAD slide (+-5 px) on the keypoint's
 * pyramid level, parabola sub-pixel fit, disparity gate [0, mbf/mb), median-based outlier cut.  Uses the device-resident
 * pyramids of the last sivo_orb_run of `left` / `right` (so mvImagePyramid need not travel to the host for it).
 * u_right / depth: n_left floats each = mvRight / mvDepth (-1 where unmatched). */
int sivo_stereo_match(const sivo_orb_t* left, const sivo_orb_t* right, const sivo_keypoint* kp_left, const uint8_t* desc_left,
                      int n_left, const sivo_keypoint* kp_right, const uint8_t* desc_right, int n_right, float mb, float mbf,
                      float* u_right, float* depth);

/* Best / second-best match over per-query candidate lists -- the inner loop of ORBmatcher::SearchByProjection
 * (ORBmatcher.cc:79-113), its last-frame / keyframe variants (:1278-, :1420-), SearchForTriangulation (:631-) and
 * SearchBySim3 (next row 4).  Query i's candidates are cand_idx[cand_offsets[i] .. cand_offsets[i+1]) (indices into the
 * train descriptors, in the order GetFeaturesInArea returned them; the caller has already dropped the ones its own
 * state excludes).  out5[5 i ..] = {bestIdx, bestDist, bestLevel, bestDist2, bestLevel2} exactly as the sequential loop
 * leaves them (strict '<', so the first minimum wins; 256 / -1 when there is no candidate).  train_level (octave per train
 * keypoint) may be NULL (levels reported as 0).  The TH_HIGH / mfNNratio / orientation-histogram decisions stay with the
 * caller, as does the in-loop `F.mvpMapPoints[bestIdx] = pMP` dependency between queries. */
int sivo_hamming_best2(int device, const uint8_t* query_desc, int n_query, const uint8_t* train_desc, int n_train,
                       const int* cand_offsets, const int* cand_idx, const int* train_level, int* out5);

/* ---- test hooks for single layers (float NCHW host arrays in/out; run the product kernels) ----- */
int sivo_dbg_pool(int device, const float* in, int n, int c, int h, int w, float* out, int* mask);
int sivo_dbg_unpool(int device, const float* in, const int* mask, int n, int c, int h, int w, float* out);
int sivo_dbg_conv(int device, int engine, int precision, const float* in, int n, int cin, int h, int w,
                  const float* weight, const float* bias, const float* bn_scale, const float* bn_shift,
                  int cout, int k, int pad, int relu, float* out);
int sivo_dbg_lrn(int device, const float* in, int n, int c, int h, int w, int size, float alpha, float beta,
                 float k, float* out);
int sivo_dbg_mc_reduce(int device, const float* logits, int T, int c, int h, int w, uint8_t* classes,
                       double* confidence, double* entropy);
/* The two halves of sivo_dbg_mc_reduce: sums[c][h][w] (+)= the softmax probabilities of T samples of logits (accumulate = 1
 * adds to the sums passed in), and the maps from sums of T_total samples. */
int sivo_dbg_mc_partial(int device, const float* logits, int T, int c, int h, int w, int accumulate, double* sums);
int sivo_dbg_mc_finalize(int device, const double* sums, int T_total, int c, int h, int w, uint8_t* classes,
                         double* confidence, double* entropy);
int sivo_dbg_dropout_mask(int device, uint64_t seed, uint64_t frame, int layer, int T, int c, int h, int w,
                          uint8_t* keep);

const char* sivo_last_error(void);
const char* sivo_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SIVO_B200_H_ */
