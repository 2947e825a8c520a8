// SegNet layer kernels, SIMT set: the strict-fp32 engine, the correctness anchor for the tcgen05
// convolution (conv_tc.cu), and every bandwidth-bound layer.  Semantics follow the Caffe layers the
// reference executes (SURVEY 2b); each kernel cites the layer it replaces.
#include <cuda_fp16.h>

#include "common.h"
#include "philox.cuh"
#include "segnet_kernels.h"

namespace sivo {
namespace {

template <typename T> __device__ __forceinline__ float ld_act(const T* p);
template <> __device__ __forceinline__ float ld_act<__half>(const __half* p) { return __half2float(*p); }
template <> __device__ __forceinline__ float ld_act<float>(const float* p) { return *p; }
template <typename T> __device__ __forceinline__ void st_act(T* p, float v);
template <> __device__ __forceinline__ void st_act<__half>(__half* p, float v) { *p = __float2half_rn(v); }
template <> __device__ __forceinline__ void st_act<float>(float* p, float v) { *p = v; }

// ---- input: wrapInputLayer + preprocessImage (bayesian_segnet.cpp:119-140,164-178): u8 BGR -> float, no
// mean / scale, planar split.  Here: one NHWC pixel of 4 channels (B, G, R, 0).
template <typename AT>
__global__ void k_input_u8(const uint8_t* __restrict__ bgr, AT* __restrict__ out, int npix, const FrameArgs* __restrict__ args) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  if (args) bgr = args->bgr;
  const uint8_t* s = bgr + 3 * static_cast<size_t>(i);
  AT* d = out + 4 * static_cast<size_t>(i);
  st_act(d + 0, static_cast<float>(s[0]));
  st_act(d + 1, static_cast<float>(s[1]));
  st_act(d + 2, static_cast<float>(s[2]));
  st_act(d + 3, 0.f);
}

// ---- LRN across channels (caffe lrn_layer.cpp:108-152): scale = k + alpha/size * sum_{window} x^2,
// y = x * scale^-beta.  Only ever applied to the 3-channel input, so one thread per pixel.
template <typename AT>
__global__ void k_lrn(const AT* __restrict__ in, AT* __restrict__ out, int npix, int c, int cs, int size,
                      float alpha_over_size, float beta, float k) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  const AT* s = in + static_cast<size_t>(i) * cs;
  AT* d = out + static_cast<size_t>(i) * cs;
  int pre = (size - 1) / 2;
  for (int ch = 0; ch < cs; ++ch) {
    if (ch >= c) { st_act(d + ch, 0.f); continue; }
    float acc = 0.f;
    for (int j = ch - pre; j <= ch - pre + size - 1; ++j)
      if (j >= 0 && j < c) { float x = ld_act(s + j); acc = __fadd_rn(acc, __fmul_rn(x, x)); }
    float scale = __fadd_rn(k, __fmul_rn(acc, alpha_over_size));
    st_act(d + ch, __fmul_rn(ld_act(s + ch), powf(scale, -beta)));
  }
}

// ---- direct convolution, fp32 FMA (conv_layer.cpp:25-40 / base_conv_layer.cpp:257-280; cuDNN fp32 in the
// reference's GPU mode).  Block = 8x16 pixels x 64 output channels; thread = 8 pixels of one row x 4 couts.
// Epilogue order matches the layer sequence: + bias, BN affine (mul then add, bn_layer.cpp:199-223), ReLU.
constexpr int kTH = 8, kTW = 16, kConvThreads = 256;

template <typename AT, typename OT, int K>
__global__ void __launch_bounds__(kConvThreads) k_conv_simt(ConvParams p, int CK, int tiles_w) {
  extern __shared__ float smem[];
  constexpr int IH = kTH + K - 1, IW = kTW + K - 1, IWP = IW | 1;
  float* s_w = smem;                          // [K*K][CK][64]
  float* s_in = smem + K * K * CK * 64;       // [CK][IH][IWP]
  const int tid = threadIdx.x;
  const int cg = tid & 15, pg = tid >> 4;
  const int row = pg >> 1, col0 = (pg & 1) * 8;
  const int tile_y = blockIdx.x / tiles_w, tile_x = blockIdx.x % tiles_w;
  const int y0 = tile_y * kTH, x0 = tile_x * kTW;
  const int co_base = blockIdx.y * 64;
  const int n = blockIdx.z;
  const int H = p.in.h, W = p.in.w, cs_in = p.in.cs;
  const AT* in = static_cast<const AT*>(p.in.p) + static_cast<size_t>(n) * H * W * cs_in;

  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int c0 = 0; c0 < p.cin_p; c0 += CK) {
    for (int e = tid; e < IH * IW * CK; e += kConvThreads) {
      int ci = e % CK, xy = e / CK;
      int x = xy % IW, y = xy / IW;
      int gy = y0 + y - p.pad, gx = x0 + x - p.pad;
      float v = 0.f;
      if (gy >= 0 && gy < H && gx >= 0 && gx < W && c0 + ci < cs_in)
        v = ld_act(in + (static_cast<size_t>(gy) * W + gx) * cs_in + c0 + ci);
      s_in[(ci * IH + y) * IWP + x] = v;
    }
    for (int e = tid; e < K * K * CK * 64; e += kConvThreads) {
      int co = e & 63, r = e >> 6;
      int ci = r % CK, tap = r / CK;
      s_w[e] = p.w_simt[(static_cast<size_t>(tap) * p.cin_p + c0 + ci) * p.cout_p + co_base + co];
    }
    __syncthreads();
    for (int ci = 0; ci < CK; ++ci) {
#pragma unroll
      for (int kh = 0; kh < K; ++kh) {
        float xr[8 + K - 1];
        const float* src = s_in + (ci * IH + row + kh) * IWP + col0;
#pragma unroll
        for (int i = 0; i < 8 + K - 1; ++i) xr[i] = src[i];
#pragma unroll
        for (int kw = 0; kw < K; ++kw) {
          const float4 w4 = *reinterpret_cast<const float4*>(s_w + ((kh * K + kw) * CK + ci) * 64 + cg * 4);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            acc[i][0] = fmaf(xr[i + kw], w4.x, acc[i][0]);
            acc[i][1] = fmaf(xr[i + kw], w4.y, acc[i][1]);
            acc[i][2] = fmaf(xr[i + kw], w4.z, acc[i][2]);
            acc[i][3] = fmaf(xr[i + kw], w4.w, acc[i][3]);
          }
        }
      }
    }
    __syncthreads();
  }

  const int gy = y0 + row;
  if (gy >= H) return;
  OT* out = static_cast<OT*>(p.out.p) + (static_cast<size_t>(n) * H + gy) * W * p.out.cs;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int gx = x0 + col0 + i;
    if (gx >= W) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int co = co_base + cg * 4 + j;
      if (co >= p.out.cs) continue;
      float v = __fadd_rn(acc[i][j], p.bias[co]);
      if (p.bn_scale) v = __fadd_rn(__fmul_rn(v, p.bn_scale[co]), p.bn_shift[co]);
      if (p.relu) v = v > 0.f ? v : __fmul_rn(p.slope, v);
      st_act(out + static_cast<size_t>(gx) * p.out.cs + co, v);
    }
  }
}

// ---- 2x2/2 max pool with argmax (pooling_layer.cpp:140-187): scan (0,0),(0,1),(1,0),(1,1) with strict '>'
// so the first maximum wins.  The mask is 2 bits (dh*2+dw) per element instead of Caffe's float plane index.
template <typename AT>
__global__ void k_pool(const AT* __restrict__ in, AT* __restrict__ out, uint8_t* __restrict__ mask, int N, int Ho,
                       int Wo, int cs) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t total = static_cast<size_t>(N) * Ho * Wo * cs;
  if (i >= total) return;
  int c = i % cs;
  size_t r = i / cs;
  int wo = r % Wo;
  r /= Wo;
  int ho = r % Ho;
  int n = r / Ho;
  int W = Wo * 2;
  const AT* s = in + ((static_cast<size_t>(n) * Ho * 2 + ho * 2) * W + wo * 2) * cs + c;
  float best = ld_act(s);
  int arg = 0;
  float v = ld_act(s + cs);
  if (v > best) { best = v; arg = 1; }
  v = ld_act(s + static_cast<size_t>(W) * cs);
  if (v > best) { best = v; arg = 2; }
  v = ld_act(s + static_cast<size_t>(W) * cs + cs);
  if (v > best) { best = v; arg = 3; }
  st_act(out + i, best);
  mask[i] = static_cast<uint8_t>(arg);
}

// ---- max-unpool (upsample_layer.cpp:74-103): zero fill + scatter, written densely per 2x2 block.
template <typename AT>
__global__ void k_unpool(const AT* __restrict__ in, const uint8_t* __restrict__ mask, int mask_n, AT* __restrict__ out,
                         int N, int Hi, int Wi, int cs) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t total = static_cast<size_t>(N) * Hi * Wi * cs;
  if (i >= total) return;
  int c = i % cs;
  size_t r = i / cs;
  int wi = r % Wi;
  r /= Wi;
  int hi = r % Hi;
  int n = r / Hi;
  size_t mi = ((static_cast<size_t>(n % mask_n) * Hi + hi) * Wi + wi) * cs + c;
  int arg = mask[mi];
  float v = ld_act(in + i);
  int W = Wi * 2;
  AT* d = out + ((static_cast<size_t>(n) * Hi * 2 + hi * 2) * W + wi * 2) * cs + c;
  st_act(d, arg == 0 ? v : 0.f);
  st_act(d + cs, arg == 1 ? v : 0.f);
  st_act(d + static_cast<size_t>(W) * cs, arg == 2 ? v : 0.f);
  st_act(d + static_cast<size_t>(W) * cs + cs, arg == 3 ? v : 0.f);
}

// ---- test-time dropout sampling (dropout_layer.cpp:31-46): y = x * keep * 1/(1-ratio).
template <typename AT>
__global__ void k_dropout(const AT* __restrict__ in, int in_n, AT* __restrict__ out, int N, int HW, int cs, int C,
                          uint64_t seed, const uint64_t* __restrict__ frame, int layer, int sample0, float scale) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;  // one thread per (n, pix, 32-ch word)
  int words = (cs + 31) / 32;
  size_t total = static_cast<size_t>(N) * HW * words;
  if (i >= total) return;
  int wd = i % words;
  size_t r = i / words;
  uint32_t pix = r % HW;
  int n = r / HW;
  uint32_t bits[4];
  dropout_bits128(seed, *frame, layer, sample0 + n, pix, wd >> 2, bits);
  uint32_t b = bits[wd & 3];
  const AT* s = in + (static_cast<size_t>(n % in_n) * HW + pix) * cs + wd * 32;
  AT* d = out + (static_cast<size_t>(n) * HW + pix) * cs + wd * 32;
  int lim = min(32, cs - wd * 32);
  for (int j = 0; j < lim; ++j) {
    float v = (wd * 32 + j < C && ((b >> j) & 1u)) ? __fmul_rn(ld_act(s + j), scale) : 0.f;
    st_act(d + j, v);
  }
}

// half activations, channel count a multiple of 8: one thread per (sample, pixel, 8-channel chunk), 16-byte accesses.
// y = x * 2 is exact in half, so this equals the generic kernel's float multiply + rounding.  With UNPOOL the result
// is scattered straight into the 2x2 block its pooling mask names (dropout -> upsample pair of the decoder entry).
template <bool UNPOOL>
__global__ void k_dropout_h8(const uint4* __restrict__ in, int in_n, uint4* __restrict__ out, int N, int Hi, int Wi, int cs,
                             uint64_t seed, const uint64_t* __restrict__ frame, int layer, int sample0, float scale,
                             const uint8_t* __restrict__ mask, int mask_n) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int chunks = cs >> 3;
  const int HW = Hi * Wi;
  if (i >= static_cast<size_t>(N) * HW * chunks) return;
  const int ch = static_cast<int>(i % chunks);
  const size_t r = i / chunks;
  const uint32_t pix = static_cast<uint32_t>(r % HW);
  const int n = static_cast<int>(r / HW);
  uint32_t bits[4];
  dropout_bits128(seed, *frame, layer, sample0 + n, pix, ch >> 4, bits);
  const uint32_t b = (bits[(ch >> 2) & 3] >> ((ch & 3) * 8)) & 0xFFu;
  const uint4 v = __ldg(in + (static_cast<size_t>(n % in_n) * HW + pix) * chunks + ch);
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  uint32_t o[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const __half2 s2 = __floats2half2_rn((b >> (2 * k)) & 1u ? scale : 0.f, (b >> (2 * k + 1)) & 1u ? scale : 0.f);
    const __half2 h = __hmul2(*reinterpret_cast<const __half2*>(&w[k]), s2);
    o[k] = *reinterpret_cast<const uint32_t*>(&h);
  }
  if (!UNPOOL) {
    out[i] = make_uint4(o[0], o[1], o[2], o[3]);
    return;
  }
  const uint2 m = __ldg(reinterpret_cast<const uint2*>(mask + ((static_cast<size_t>(n % mask_n) * HW + pix) * cs + ch * 8)));
  const uint32_t mw[2] = {m.x, m.y};
  const int hi = pix / Wi, wi = pix % Wi;
#pragma unroll
  for (int pos = 0; pos < 4; ++pos) {
    uint32_t sel[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t mb = mw[k >> 1] >> ((k & 1) * 16);
      const uint32_t lo = ((mb & 0xFFu) == static_cast<uint32_t>(pos)) ? 0x0000FFFFu : 0u;
      const uint32_t hi2 = (((mb >> 8) & 0xFFu) == static_cast<uint32_t>(pos)) ? 0xFFFF0000u : 0u;
      sel[k] = o[k] & (lo | hi2);
    }
    out[((static_cast<size_t>(n) * 2 * Hi + 2 * hi + (pos >> 1)) * (2 * Wi) + 2 * wi + (pos & 1)) * chunks + ch] =
        make_uint4(sel[0], sel[1], sel[2], sel[3]);
  }
}

__global__ void k_dropout_bits(uint64_t seed, const uint64_t* frame, int layer, int T, int C, int HW,
                               uint8_t* __restrict__ keep) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t total = static_cast<size_t>(T) * C * HW;
  if (i >= total) return;
  uint32_t pix = i % HW;
  int c = (i / HW) % C;
  int n = i / (static_cast<size_t>(HW) * C);
  uint32_t bits[4];
  dropout_bits128(seed, *frame, layer, n, pix, c >> 7, bits);
  keep[i] = (bits[(c >> 5) & 3] >> (c & 31)) & 1u;
}

// ---- Softmax over channels (softmax_layer.cpp:27-60, fp32) fused with the Monte-Carlo reduction the
// reference runs on the host in double (bayesian_segnet.cpp:278-318): mean over T, first-max argmax, max,
// -sum p log2 p with 0 log 0 := 0 (computeEntropy :38-44).  One thread per pixel; `prob` never exists.
template <int C>
__global__ void k_mc_reduce(const float* __restrict__ logits, int T, int cs, int hw, uint8_t* __restrict__ classes,
                            double* __restrict__ conf, double* __restrict__ entropy, const FrameArgs* __restrict__ args) {
  float *conf32 = nullptr, *ent32 = nullptr;
  if (args) { classes = args->classes; conf = args->conf; entropy = args->ent; conf32 = args->conf32; ent32 = args->ent32; }
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hw) return;
  double acc[C];
#pragma unroll
  for (int c = 0; c < C; ++c) acc[c] = 0.0;
  for (int t = 0; t < T; ++t) {
    const float* s = logits + (static_cast<size_t>(t) * hw + i) * cs;
    float x[16];
    if (cs == 16) {  // one 64-byte pixel: four 128-bit loads instead of 15 strided scalar ones
      const float4* s4 = reinterpret_cast<const float4*>(s);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 v = __ldg(s4 + q);
        x[4 * q] = v.x; x[4 * q + 1] = v.y; x[4 * q + 2] = v.z; x[4 * q + 3] = v.w;
      }
    } else {
#pragma unroll
      for (int c = 0; c < C; ++c) x[c] = s[c];
    }
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < C; ++c) m = fmaxf(m, x[c]);
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) { x[c] = expf(__fsub_rn(x[c], m)); sum = __fadd_rn(sum, x[c]); }
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] += static_cast<double>(__fdiv_rn(x[c], sum));
  }
  double best = -1.0, ent = 0.0;
  int arg = 0;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    double pm = acc[c] / static_cast<double>(T);
    if (pm > best) { best = pm; arg = c; }
    if (pm != 0.0) ent += -1.0 * pm * log2(pm);
  }
  if (classes) classes[i] = static_cast<uint8_t>(arg);
  if (conf) conf[i] = best;
  if (entropy) entropy[i] = ent;
  if (conf32) conf32[i] = static_cast<float>(best);
  if (ent32) ent32[i] = static_cast<float>(ent);
}

// Same reduction with four lanes per pixel (one float4 = 4 classes each): a warp reads 512 contiguous bytes per
// sample and there are 4x more threads in flight, which is what this HBM-bound pass needs.  The softmax max / sum and
// the final argmax / entropy are combined with xor-shuffles inside the 4-lane group (first maximum still wins).
// Instruction diet (ncu: the first version was issue-bound at 3400 instructions per warp, 0.8 TB/s): one IEEE
// reciprocal per sample instead of C divisions (p = e * (1/sum), <= 1 ulp from e/sum), mean = acc * (1/T) in double,
// and log2 evaluated in float on the double mean (relative error < 2^-22, i.e. < 1e-6 on the entropy, against the
// 1e-4 the contract allows); the products and the sums stay in double like computeEntropy (bayesian_segnet.cpp:38-44).
// The two halves -- per-sample softmax summed into acc, then mean / argmax / entropy -- are shared by the one-pass
// reduction and the partial / finalize pair of sample shards, so equal sums give bit-identical maps.

// lane q of pixel pp: acc[j] += softmax probability of class 4q + j, for samples 0..T-1 of `logits`, in sample order
__device__ __forceinline__ void mc_quad_accumulate(const float* __restrict__ logits, int T, int C, int hw, int pp, int q, double acc[4]) {
  constexpr int kBatch = 6;  // samples whose loads are issued together (memory-level parallelism: the pass is HBM-bound)
  for (int t0 = 0; t0 < T; t0 += kBatch) {
  float4 vb[kBatch];
#pragma unroll
  for (int b = 0; b < kBatch; ++b)
    if (t0 + b < T) vb[b] = __ldcs(reinterpret_cast<const float4*>(logits + (static_cast<size_t>(t0 + b) * hw + pp) * 16) + q);
#pragma unroll
  for (int b = 0; b < kBatch; ++b) {
    if (t0 + b >= T) break;
    const float4 v = vb[b];
    float x[4] = {v.x, v.y, v.z, v.w};
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j < 4; ++j) if (q * 4 + j < C) m = fmaxf(m, x[j]);
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 2));
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      x[j] = (q * 4 + j < C) ? __expf(__fsub_rn(x[j], m)) : 0.f;  // ex2.approx: <= 2 ulp on an argument in [-88, 0], 2e-7 on a probability
      sum = __fadd_rn(sum, x[j]);
    }
    sum = __fadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, 1));
    sum = __fadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, 2));
    const float inv = __frcp_rn(sum);
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[j] += static_cast<double>(__fmul_rn(x[j], inv));
  }
  }
}

// mean over T, first-max argmax and entropy from the 4-lane group's sums; every lane of the group ends with the pixel's result
__device__ __forceinline__ void mc_quad_finalize(const double acc[4], int T, int C, int q, double& best, int& arg, double& ent) {
  const double inv_t = 1.0 / static_cast<double>(T);
  best = -1.0;
  ent = 0.0;
  arg = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (q * 4 + j >= C) continue;
    const double pm = acc[j] * inv_t;
    if (pm > best) { best = pm; arg = q * 4 + j; }
    const float pf = static_cast<float>(pm);  // a mean below the float range contributes < 1e-43 bits: same as the 0 log 0 := 0 rule
    if (pf > 0.f) ent -= pm * static_cast<double>(log2f(pf));
  }
#pragma unroll
  for (int o = 1; o <= 2; o <<= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    ent += __shfl_xor_sync(0xffffffffu, ent, o);
    if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
  }
}

__global__ void k_mc_reduce_quad(const float* __restrict__ logits, int T, int C, int hw, uint8_t* __restrict__ classes,
                                 double* __restrict__ conf, double* __restrict__ entropy, int pix0, int pix_end,
                                 const FrameArgs* __restrict__ args) {
  float *conf32 = nullptr, *ent32 = nullptr;
  if (args) { classes = args->classes; conf = args->conf; entropy = args->ent; conf32 = args->conf32; ent32 = args->ent32; }
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int pix = pix0 + (gid >> 2), q = gid & 3;
  const bool live = pix < pix_end;
  const int pp = live ? pix : hw - 1;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  mc_quad_accumulate(logits, T, C, hw, pp, q, acc);
  double best, ent;
  int arg;
  mc_quad_finalize(acc, T, C, q, best, arg, ent);
  if (live && q == 0) {
    if (classes) classes[pix] = static_cast<uint8_t>(arg);
    if (conf) conf[pix] = best;
    if (entropy) entropy[pix] = ent;
    if (conf32) conf32[pix] = static_cast<float>(best);
    if (ent32) ent32[pix] = static_cast<float>(ent);
  }
}

// Sample shards, first half: the same 4-lane softmax, continued from the sums already in prob_sum ([C][hw] doubles) or from 0.
// Adding the shards of [0, T) one after another in sample order performs exactly k_mc_reduce_quad's sequence of double additions.
__global__ void k_mc_partial_quad(const float* __restrict__ logits, int n, int C, int hw, double* __restrict__ prob_sum, int accumulate,
                                  const FrameArgs* __restrict__ args) {
  if (args) { prob_sum = args->prob_sum; accumulate = args->accumulate; }
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int pix = gid >> 2, q = gid & 3;
  const bool live = pix < hw;
  const int pp = live ? pix : hw - 1;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  if (accumulate && live) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (q * 4 + j < C) acc[j] = prob_sum[static_cast<size_t>(q * 4 + j) * hw + pix];
  }
  mc_quad_accumulate(logits, n, C, hw, pp, q, acc);
  if (!live) return;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (q * 4 + j < C) prob_sum[static_cast<size_t>(q * 4 + j) * hw + pix] = acc[j];
}

// Second half: the maps from the summed probabilities of all T samples (the tail of k_mc_reduce_quad)
__global__ void k_mc_finalize(const double* __restrict__ prob_sum, int T, int C, int hw, uint8_t* __restrict__ classes,
                              double* __restrict__ conf, double* __restrict__ entropy, float* __restrict__ conf32,
                              float* __restrict__ ent32) {
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int pix = gid >> 2, q = gid & 3;
  const bool live = pix < hw;
  const int pp = live ? pix : hw - 1;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (q * 4 + j < C) acc[j] = prob_sum[static_cast<size_t>(q * 4 + j) * hw + pp];
  double best, ent;
  int arg;
  mc_quad_finalize(acc, T, C, q, best, arg, ent);
  if (live && q == 0) {
    if (classes) classes[pix] = static_cast<uint8_t>(arg);
    if (conf) conf[pix] = best;
    if (entropy) entropy[pix] = ent;
    if (conf32) conf32[pix] = static_cast<float>(best);
    if (ent32) ent32[pix] = static_cast<float>(ent);
  }
}

__global__ void k_mc_reduce_generic(const float* __restrict__ logits, int T, int C, int cs, int hw,
                                    uint8_t* __restrict__ classes, double* __restrict__ conf,
                                    double* __restrict__ entropy, const FrameArgs* __restrict__ args) {
  float *conf32 = nullptr, *ent32 = nullptr;
  if (args) { classes = args->classes; conf = args->conf; entropy = args->ent; conf32 = args->conf32; ent32 = args->ent32; }
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hw) return;
  double best = -1.0, ent = 0.0;
  int arg = 0;
  for (int c = 0; c < C; ++c) {
    double a = 0.0;
    for (int t = 0; t < T; ++t) {
      const float* s = logits + (static_cast<size_t>(t) * hw + i) * cs;
      float m = -INFINITY;
      for (int k = 0; k < C; ++k) m = fmaxf(m, s[k]);
      float sum = 0.f;
      for (int k = 0; k < C; ++k) sum = __fadd_rn(sum, expf(__fsub_rn(s[k], m)));
      a += static_cast<double>(__fdiv_rn(expf(__fsub_rn(s[c], m)), sum));
    }
    double pm = a / static_cast<double>(T);
    if (pm > best) { best = pm; arg = c; }
    if (pm != 0.0) ent += -1.0 * pm * log2(pm);
  }
  if (classes) classes[i] = static_cast<uint8_t>(arg);
  if (conf) conf[i] = best;
  if (entropy) entropy[i] = ent;
  if (conf32) conf32[i] = static_cast<float>(best);
  if (ent32) ent32[i] = static_cast<float>(ent);
}

// ---- tap expansion for the 3-channel first convolution: out[y][x][kh*blk + kw*4 + c] = in[y+kh-pad][x+kw-pad][c]
// (zero outside the image = the convolution's zero padding), so that conv1 becomes a 1x1 convolution over
// K*blk channels that the tensor-core kernel can run (K*K*3 = 147 of 256 K-slots useful for the 7x7 layer).
template <typename AT>
__global__ void k_expand_taps(const AT* __restrict__ in, AT* __restrict__ out, int N, int H, int W, int K, int blk, int cs_out) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;  // one thread per (n, y, x, kh-or-pad-block)
  const int groups = cs_out / blk;
  size_t total = static_cast<size_t>(N) * H * W * groups;
  if (i >= total) return;
  const int g = i % groups;
  size_t r = i / groups;
  const int x = r % W;
  r /= W;
  const int y = r % H;
  const int n = r / H;
  AT* d = out + ((static_cast<size_t>(n) * H + y) * W + x) * cs_out + g * blk;
  const int pad = (K - 1) / 2;
  const int yy = y + g - pad;
  const bool row_ok = g < K && yy >= 0 && yy < H;
  if (sizeof(AT) == 2) {  // half: one 4-channel pixel = 8 bytes; write the block as 16-byte vectors
    const uint2* src = reinterpret_cast<const uint2*>(in) + (static_cast<size_t>(n) * H + yy) * W;
    uint4* dst = reinterpret_cast<uint4*>(d);
    for (int q = 0; q < blk / 8; ++q) {
      uint2 a = make_uint2(0u, 0u), b = make_uint2(0u, 0u);
      const int xa = x + 2 * q - pad, xb = xa + 1;
      if (row_ok && 2 * q < K && xa >= 0 && xa < W) a = __ldg(src + xa);
      if (row_ok && 2 * q + 1 < K && xb >= 0 && xb < W) b = __ldg(src + xb);
      dst[q] = make_uint4(a.x, a.y, b.x, b.y);
    }
    return;
  }
  for (int j = 0; j < blk; ++j) {
    const int kw = j >> 2, c = j & 3;
    const int xx = x + kw - pad;
    float v = 0.f;
    if (row_ok && kw < K && xx >= 0 && xx < W) v = ld_act(in + ((static_cast<size_t>(n) * H + yy) * W + xx) * 4 + c);
    st_act(d + j, v);
  }
}

// Window-folded first layer (conv_tc.cu): the 4-channel half image, zero-padded to [H][W + 8] pixels of 8 channels.
__global__ void k_pad8(const uint2* __restrict__ in, uint4* __restrict__ out, int NH, int W) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int Wp = W + 8;
  if (i >= static_cast<size_t>(NH) * Wp) return;
  const int xp = static_cast<int>(i % Wp);
  const size_t row = i / Wp;
  const int x = xp - 3;
  uint2 v = make_uint2(0u, 0u);
  if (x >= 0 && x < W) v = __ldg(in + row * W + x);
  out[i] = make_uint4(v.x, v.y, 0u, 0u);
}

// k_input_u8 -> k_lrn<__half> -> k_pad8 in one pass over the padded image: identical operations on identical values
// (the u8 -> half conversion is exact, the LRN output is rounded to half once), hence bitwise the same operand.
__global__ void k_input_lrn_pad8(const uint8_t* __restrict__ bgr, uint4* __restrict__ out, int H, int W, int size,
                                 float alpha_over_size, float beta, float k, const FrameArgs* __restrict__ args) {
  if (args) bgr = args->bgr;
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int Wp = W + 8;
  if (i >= static_cast<size_t>(H) * Wp) return;
  const int x = static_cast<int>(i % Wp) - 3;
  const size_t row = i / Wp;
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  if (x >= 0 && x < W) {
    const uint8_t* s = bgr + 3 * (row * W + x);
    const float in[3] = {static_cast<float>(s[0]), static_cast<float>(s[1]), static_cast<float>(s[2])};
    const int pre = (size - 1) / 2;
    __half o[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      float acc = 0.f;
      for (int j = ch - pre; j <= ch - pre + size - 1; ++j)
        if (j >= 0 && j < 3) acc = __fadd_rn(acc, __fmul_rn(in[j], in[j]));
      const float scale = __fadd_rn(k, __fmul_rn(acc, alpha_over_size));
      o[ch] = __float2half_rn(__fmul_rn(in[ch], powf(scale, -beta)));
    }
    v.x = static_cast<uint32_t>(__half_as_ushort(o[0])) | (static_cast<uint32_t>(__half_as_ushort(o[1])) << 16);
    v.y = static_cast<uint32_t>(__half_as_ushort(o[2]));
  }
  out[i] = v;
}

// ---- layout converters for the test hooks
template <typename AT>
__global__ void k_nchw_to_act(const float* __restrict__ src, AT* __restrict__ dst, int N, int C, int HW, int cs) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t total = static_cast<size_t>(N) * HW * cs;
  if (i >= total) return;
  int c = i % cs;
  size_t r = i / cs;
  int pix = r % HW;
  int n = r / HW;
  st_act(dst + i, c < C ? src[(static_cast<size_t>(n) * C + c) * HW + pix] : 0.f);
}
template <typename AT>
__global__ void k_act_to_nchw(const AT* __restrict__ src, float* __restrict__ dst, int N, int C, int HW, int cs) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t total = static_cast<size_t>(N) * C * HW;
  if (i >= total) return;
  int pix = i % HW;
  int c = (i / HW) % C;
  int n = i / (static_cast<size_t>(HW) * C);
  dst[i] = ld_act(src + (static_cast<size_t>(n) * HW + pix) * cs + c);
}
// 2-bit mask <-> Caffe's plane-local index h*W+w of the *input* plane (pooling_layer.cpp:168)
__global__ void k_mask_to_nchw(const uint8_t* __restrict__ mask, int N, int C, int Ho, int Wo, int* __restrict__ dst) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t total = static_cast<size_t>(N) * C * Ho * Wo;
  if (i >= total) return;
  int wo = i % Wo;
  int ho = (i / Wo) % Ho;
  int c = (i / (static_cast<size_t>(Wo) * Ho)) % C;
  int n = i / (static_cast<size_t>(Wo) * Ho * C);
  int a = mask[((static_cast<size_t>(n) * Ho + ho) * Wo + wo) * C + c];
  dst[i] = (ho * 2 + (a >> 1)) * (Wo * 2) + wo * 2 + (a & 1);
}
__global__ void k_mask_from_nchw(const int* __restrict__ src, int N, int C, int Ho, int Wo, uint8_t* __restrict__ mask) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t total = static_cast<size_t>(N) * C * Ho * Wo;
  if (i >= total) return;
  int wo = i % Wo;
  int ho = (i / Wo) % Ho;
  int c = (i / (static_cast<size_t>(Wo) * Ho)) % C;
  int n = i / (static_cast<size_t>(Wo) * Ho * C);
  int idx = src[i];
  int y = idx / (Wo * 2), x = idx % (Wo * 2);
  mask[((static_cast<size_t>(n) * Ho + ho) * Wo + wo) * C + c] = static_cast<uint8_t>(((y - ho * 2) << 1) | (x - wo * 2));
}

inline unsigned blocks_for(size_t total, int threads) { return static_cast<unsigned>((total + threads - 1) / threads); }

template <typename AT, typename OT>
void conv_dispatch(const ConvParams& p, cudaStream_t s) {
  int tiles_w = ceil_div(p.in.w, kTW), tiles_h = ceil_div(p.in.h, kTH);
  dim3 grid(tiles_w * tiles_h, p.cout_p / 64, p.in.n);
  auto go = [&](auto kern, int K, int CK) {
    int IH = kTH + K - 1, IW = kTW + K - 1, IWP = IW | 1;
    size_t smem = (static_cast<size_t>(K) * K * CK * 64 + static_cast<size_t>(CK) * IH * IWP) * sizeof(float);
    SIVO_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    kern<<<grid, kConvThreads, smem, s>>>(p, CK, tiles_w);
    SIVO_CUDA(cudaGetLastError());
  };
  auto pick_ck = [&](int want) {
    int ck = want;
    while (p.cin_p % ck) ck >>= 1;
    return ck;
  };
  switch (p.k) {
    case 1: go(k_conv_simt<AT, OT, 1>, 1, pick_ck(16)); break;
    case 3: go(k_conv_simt<AT, OT, 3>, 3, pick_ck(16)); break;
    case 5: go(k_conv_simt<AT, OT, 5>, 5, pick_ck(8)); break;
    case 7: go(k_conv_simt<AT, OT, 7>, 7, pick_ck(4)); break;
    default: fail(SIVO_EFORMAT, "convolution kernel size %d is not supported (1, 3, 5, 7)", p.k);
  }
}

}  // namespace

#define DISPATCH_AT(dt, ...)                              \
  do {                                                    \
    if ((dt) == DType::F16) { using AT = __half; __VA_ARGS__; } \
    else { using AT = float; __VA_ARGS__; }               \
  } while (0)

void launch_input_u8(const uint8_t* bgr, TensorView out, cudaStream_t s, const FrameArgs* args) {
  int npix = out.h * out.w;
  DISPATCH_AT(out.dt, (k_input_u8<AT><<<blocks_for(npix, 256), 256, 0, s>>>(bgr, static_cast<AT*>(out.p), npix, args)));
  SIVO_CUDA(cudaGetLastError());
}

void launch_lrn(TensorView in, TensorView out, int size, float alpha, float beta, float k, cudaStream_t s) {
  int npix = in.n * in.h * in.w;
  float aos = alpha / static_cast<float>(size);
  DISPATCH_AT(in.dt, (k_lrn<AT><<<blocks_for(npix, 256), 256, 0, s>>>(static_cast<const AT*>(in.p), static_cast<AT*>(out.p),
                                                                      npix, in.c, in.cs, size, aos, beta, k)));
  SIVO_CUDA(cudaGetLastError());
}

void launch_conv_simt(const ConvParams& p, cudaStream_t s) {
  if (p.in.dt == DType::F16) {
    if (p.out.dt == DType::F16) conv_dispatch<__half, __half>(p, s);
    else conv_dispatch<__half, float>(p, s);
  } else {
    conv_dispatch<float, float>(p, s);
  }
}

void launch_expand_taps(TensorView in, TensorView out, int K, int blk, cudaStream_t s) {
  size_t total = static_cast<size_t>(out.n) * out.h * out.w * (out.cs / blk);
  DISPATCH_AT(in.dt, (k_expand_taps<AT><<<blocks_for(total, 256), 256, 0, s>>>(static_cast<const AT*>(in.p), static_cast<AT*>(out.p),
                                                                               out.n, out.h, out.w, K, blk, out.cs)));
  SIVO_CUDA(cudaGetLastError());
}

__global__ void k_keypoint_lookup(const sivo_keypoint* __restrict__ kps, int n, const uint8_t* __restrict__ classes,
                                  const double* __restrict__ conf, const double* __restrict__ ent, int H, int W,
                                  uint8_t* __restrict__ out_class, double* __restrict__ out_conf, double* __restrict__ out_ent) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int col = static_cast<int>(kps[i].x), row = static_cast<int>(kps[i].y);  // static_cast<int>(pt.x / pt.y): truncation
  const bool ok = col >= 0 && col < W && row >= 0 && row < H;
  const size_t o = ok ? static_cast<size_t>(row) * W + col : 0;
  out_class[i] = ok ? classes[o] : static_cast<uint8_t>(255);
  out_conf[i] = ok ? conf[o] : 0.0;
  out_ent[i] = ok ? ent[o] : 0.0;
}

void launch_keypoint_lookup(const sivo_keypoint* kps, int n, const uint8_t* classes, const double* conf, const double* ent, int H, int W,
                            uint8_t* out_class, double* out_conf, double* out_ent, cudaStream_t s) {
  if (n <= 0) return;
  k_keypoint_lookup<<<blocks_for(n, 128), 128, 0, s>>>(kps, n, classes, conf, ent, H, W, out_class, out_conf, out_ent);
  SIVO_CUDA(cudaGetLastError());
}

void launch_pad8(TensorView in, TensorView out, cudaStream_t s) {
  if (in.dt != DType::F16 || in.cs != 4 || out.cs != 8 || out.w != in.w + 8) fail(SIVO_EINVAL, "pad8: unexpected tensor layout");
  const size_t total = static_cast<size_t>(out.n) * out.h * out.w;
  k_pad8<<<blocks_for(total, 256), 256, 0, s>>>(static_cast<const uint2*>(in.p), static_cast<uint4*>(out.p), in.n * in.h, in.w);
  SIVO_CUDA(cudaGetLastError());
}

void launch_input_lrn_pad8(const uint8_t* bgr, TensorView out, int size, float alpha, float beta, float k, cudaStream_t s,
                           const FrameArgs* args) {
  if (out.dt != DType::F16 || out.cs != 8 || out.n != 1) fail(SIVO_EINVAL, "input_lrn_pad8: unexpected tensor layout");
  const size_t total = static_cast<size_t>(out.h) * out.w;
  k_input_lrn_pad8<<<blocks_for(total, 256), 256, 0, s>>>(bgr, static_cast<uint4*>(out.p), out.h, out.w - 8, size,
                                                          alpha / static_cast<float>(size), beta, k, args);
  SIVO_CUDA(cudaGetLastError());
}

// Split-operand fp32 mode: float NHWC [px][C] -> half [px][hi C | lo C] with hi = half(x), lo = half(x - hi) (both roundings
// to nearest; x - hi is exact in fp32), the A operand planes of the tcgen05 convolution (conv_tc.cu, TcParams::split).
__global__ void k_split_hilo(const float4* __restrict__ in, uint2* __restrict__ out, size_t npix, int c4) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= npix * c4) return;
  const size_t px = i / c4;
  const int q = static_cast<int>(i % c4);
  const float4 v = __ldg(in + i);
  const float f[4] = {v.x, v.y, v.z, v.w};
  __half hi[4], lo[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    hi[k] = __float2half_rn(f[k]);
    lo[k] = __float2half_rn(__fsub_rn(f[k], __half2float(hi[k])));
  }
  auto pack = [](const __half* h) {
    return make_uint2(static_cast<uint32_t>(__half_as_ushort(h[0])) | (static_cast<uint32_t>(__half_as_ushort(h[1])) << 16),
                      static_cast<uint32_t>(__half_as_ushort(h[2])) | (static_cast<uint32_t>(__half_as_ushort(h[3])) << 16));
  };
  out[px * 2 * c4 + q] = pack(hi);
  out[px * 2 * c4 + c4 + q] = pack(lo);
}

// The frame counter the dropout kernels read travels as a kernel argument (by value): an asynchronous copy from a single
// pinned slot could be overwritten by the next run_device() before it executes, giving two frames the same masks.
__global__ void k_set_frame_args(FrameArgs* dst, FrameArgs v) { *dst = v; }
void launch_set_frame_args(FrameArgs* dst, const FrameArgs& v, cudaStream_t s) {
  k_set_frame_args<<<1, 1, 0, s>>>(dst, v);
  SIVO_CUDA(cudaGetLastError());
}

void launch_split_hilo(TensorView in, void* out_half, cudaStream_t s) {
  if (in.dt != DType::F32 || in.cs % 4) fail(SIVO_EINVAL, "split_hilo: expects a float tensor with a channel stride that is a multiple of 4");
  const size_t npix = static_cast<size_t>(in.n) * in.h * in.w;
  const int c4 = in.cs / 4;
  k_split_hilo<<<blocks_for(npix * c4, 256), 256, 0, s>>>(static_cast<const float4*>(in.p), static_cast<uint2*>(out_half), npix, c4);
  SIVO_CUDA(cudaGetLastError());
}

void launch_pool(TensorView in, TensorView out, uint8_t* mask, cudaStream_t s) {
  size_t total = out.elems();
  DISPATCH_AT(in.dt, (k_pool<AT><<<blocks_for(total, 256), 256, 0, s>>>(static_cast<const AT*>(in.p), static_cast<AT*>(out.p),
                                                                        mask, out.n, out.h, out.w, out.cs)));
  SIVO_CUDA(cudaGetLastError());
}

void launch_unpool(TensorView in, const uint8_t* mask, int mask_n, TensorView out, cudaStream_t s) {
  size_t total = in.elems();
  DISPATCH_AT(in.dt, (k_unpool<AT><<<blocks_for(total, 256), 256, 0, s>>>(static_cast<const AT*>(in.p), mask, mask_n,
                                                                          static_cast<AT*>(out.p), in.n, in.h, in.w, in.cs)));
  SIVO_CUDA(cudaGetLastError());
}

void launch_dropout(TensorView in, TensorView out, const DropoutParams& d, float scale, cudaStream_t s) {
  if (in.dt == DType::F16 && out.dt == DType::F16 && out.cs % 8 == 0 && out.c == out.cs && in.cs == out.cs) {
    const size_t total = static_cast<size_t>(out.n) * out.h * out.w * (out.cs / 8);
    k_dropout_h8<false><<<blocks_for(total, 256), 256, 0, s>>>(static_cast<const uint4*>(in.p), in.n, static_cast<uint4*>(out.p), out.n,
                                                            out.h, out.w, out.cs, d.seed, d.frame_dev, d.layer, d.sample0, scale, nullptr, 1);
    SIVO_CUDA(cudaGetLastError());
    return;
  }
  int words = (out.cs + 31) / 32;
  size_t total = static_cast<size_t>(out.n) * out.h * out.w * words;
  DISPATCH_AT(in.dt, (k_dropout<AT><<<blocks_for(total, 256), 256, 0, s>>>(static_cast<const AT*>(in.p), in.n,
                                                                           static_cast<AT*>(out.p), out.n, out.h * out.w,
                                                                           out.cs, out.c, d.seed, d.frame_dev, d.layer, d.sample0, scale)));
  SIVO_CUDA(cudaGetLastError());
}

void launch_dropout_unpool(TensorView in, int T, const uint8_t* mask, int mask_n, TensorView out, const DropoutParams& d, float scale,
                           cudaStream_t s) {
  if (in.dt != DType::F16 || out.dt != DType::F16 || in.cs % 8 || in.c != in.cs || out.cs != in.cs || out.h != 2 * in.h || out.w != 2 * in.w ||
      out.n != T)
    fail(SIVO_EINVAL, "dropout+unpool: unexpected tensor layout");
  const size_t total = static_cast<size_t>(T) * in.h * in.w * (in.cs / 8);
  k_dropout_h8<true><<<blocks_for(total, 256), 256, 0, s>>>(static_cast<const uint4*>(in.p), in.n, static_cast<uint4*>(out.p), T, in.h, in.w,
                                                         in.cs, d.seed, d.frame_dev, d.layer, d.sample0, scale, mask, mask_n);
  SIVO_CUDA(cudaGetLastError());
}

void launch_mc_reduce(const float* logits, int T, int C, int cs, int hw, uint8_t* classes, double* conf, double* entropy,
                      cudaStream_t s, int pix0, int npix, const FrameArgs* args) {
  if (npix < 0) { pix0 = 0; npix = hw; }
  if (pix0 < 0 || pix0 + npix > hw) fail(SIVO_EINVAL, "mc_reduce: pixel range outside the map");
  if (npix == 0) return;
  if (cs == 16 && C <= 16) {
    k_mc_reduce_quad<<<blocks_for(static_cast<size_t>(npix) * 4, 256), 256, 0, s>>>(logits, T, C, hw, classes, conf, entropy, pix0, pix0 + npix, args);
    SIVO_CUDA(cudaGetLastError());
    return;
  }
  if (pix0 != 0 || npix != hw) fail(SIVO_EINVAL, "mc_reduce: pixel ranges need the 16-channel logits layout");
  if (C == 15) k_mc_reduce<15><<<blocks_for(hw, 128), 128, 0, s>>>(logits, T, cs, hw, classes, conf, entropy, args);
  else k_mc_reduce_generic<<<blocks_for(hw, 128), 128, 0, s>>>(logits, T, C, cs, hw, classes, conf, entropy, args);
  SIVO_CUDA(cudaGetLastError());
}

void launch_mc_partial(const float* logits, int n, int C, int cs, int hw, double* prob_sum, int accumulate, cudaStream_t s,
                       const FrameArgs* args) {
  if (cs != 16 || C > 16) fail(SIVO_EFORMAT, "mc_partial: needs the 16-channel logits layout (%d classes, stride %d)", C, cs);
  if (hw <= 0 || n <= 0) return;
  k_mc_partial_quad<<<blocks_for(static_cast<size_t>(hw) * 4, 256), 256, 0, s>>>(logits, n, C, hw, prob_sum, accumulate, args);
  SIVO_CUDA(cudaGetLastError());
}

void launch_mc_finalize(const double* prob_sum, int T, int C, int hw, uint8_t* classes, double* conf, double* entropy, float* conf32,
                        float* ent32, cudaStream_t s) {
  if (C > 16 || C <= 0 || T <= 0) fail(SIVO_EINVAL, "mc_finalize: %d classes, T = %d", C, T);
  if (hw <= 0) return;
  k_mc_finalize<<<blocks_for(static_cast<size_t>(hw) * 4, 256), 256, 0, s>>>(prob_sum, T, C, hw, classes, conf, entropy, conf32, ent32);
  SIVO_CUDA(cudaGetLastError());
}

void launch_dropout_bits(uint64_t seed, const uint64_t* frame_dev, int layer, int T, int C, int H, int W, uint8_t* keep,
                         cudaStream_t s) {
  size_t total = static_cast<size_t>(T) * C * H * W;
  k_dropout_bits<<<blocks_for(total, 256), 256, 0, s>>>(seed, frame_dev, layer, T, C, H * W, keep);
  SIVO_CUDA(cudaGetLastError());
}

void launch_nchw_to_act(const float* src, TensorView dst, cudaStream_t s) {
  size_t total = dst.elems();
  DISPATCH_AT(dst.dt, (k_nchw_to_act<AT><<<blocks_for(total, 256), 256, 0, s>>>(src, static_cast<AT*>(dst.p), dst.n, dst.c,
                                                                               dst.h * dst.w, dst.cs)));
  SIVO_CUDA(cudaGetLastError());
}

void launch_act_to_nchw(TensorView src, float* dst, cudaStream_t s) {
  size_t total = static_cast<size_t>(src.n) * src.c * src.h * src.w;
  DISPATCH_AT(src.dt, (k_act_to_nchw<AT><<<blocks_for(total, 256), 256, 0, s>>>(static_cast<const AT*>(src.p), dst, src.n,
                                                                               src.c, src.h * src.w, src.cs)));
  SIVO_CUDA(cudaGetLastError());
}

void launch_mask_to_nchw(const uint8_t* mask, int n, int c, int ho, int wo, int* dst, cudaStream_t s) {
  size_t total = static_cast<size_t>(n) * c * ho * wo;
  k_mask_to_nchw<<<blocks_for(total, 256), 256, 0, s>>>(mask, n, c, ho, wo, dst);
  SIVO_CUDA(cudaGetLastError());
}

void launch_mask_from_nchw(const int* src, int n, int c, int ho, int wo, uint8_t* mask, cudaStream_t s) {
  size_t total = static_cast<size_t>(n) * c * ho * wo;
  k_mask_from_nchw<<<blocks_for(total, 256), 256, 0, s>>>(src, n, c, ho, wo, mask);
  SIVO_CUDA(cudaGetLastError());
}

}  // namespace sivo
