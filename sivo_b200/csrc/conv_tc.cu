// tcgen05 implicit-GEMM convolution for sm_100a -- replaces cuDNN's fp32 `cudnnConvolutionForward`
// (caffe/src/caffe/layers/cudnn_conv_layer.cu:21-37) and the layers fused around it for every SegNet convolution
// (Basic: all eight 7x7 layers + the 1x1 classifier; Standard: all 26 3x3 layers).
//
// GEMM view per CTA:  D[128 pixels x N couts] += A[128 pixels x 64 cin] * B[64 cin x N couts]  per filter tap,
// M = 128 consecutive pixels of one output row, R = 4 (or 2) output rows -- a "row block" -- per accumulator stage.
//
//  * Activations are NHWC half, so one pixel's 64 input channels are one 128-byte row: exactly a
//    SWIZZLE_128B K-major UMMA operand row.  A TMA box {64 ch, 128+K-1 px, 1 row} of the input lands one
//    *halo row* in shared memory; out-of-image coordinates are zero-filled by TMA = the conv's zero padding.
//  * The A operand of tap (kh, kw) for output row r is the same halo row shifted by kw pixels: the UMMA
//    shared-memory descriptor simply starts kw*128 bytes later (the swizzle phase follows the absolute address), so
//    each input row is fetched from L2 once per K rows of output instead of K*K times.
//  * A CTA walks down a 128-px-wide column strip one row block at a time with a ring of halo rows: every input row is
//    loaded once per CTA (plus the K-1 overlap between vertically adjacent CTAs) and released as soon as its last tap
//    row has been issued.
//  * Weights stream through a TMA ring, one tile per tap (k_conv_tc: {64 cin x N cout}, [tap][cout][cin]) or per pair of
//    vertically adjacent taps (k_conv_tc_pair: two stacked tiles, N = 128, [kw][kh][cout][cin]).
//  * The 3-channel first layer reads a window-folded view of the zero-padded 8-channel image (KW = 1, see conv_tc_plan).
//  * Accumulators live in TMEM (2 stages x R x N fp32 columns) so the epilogue of block j overlaps the MMAs of block
//    j+1.  384 threads: warp 0 = halo-row TMA producer, warp 1 = weight TMA producer, warps 2-3 = MMA issuers (+ TMEM
//    alloc), warps 4-11 = epilogue (two per TMEM lane quarter; setmaxnreg 56 / 216): tcgen05.ld -> bias / BN affine / ReLU
//    -> half, then store | dropout | max-unpool scatter | 2x2 max-pool + argmax | 1x1 classifier -> float logits.
//  * Constants (bias, BN, classifier weights) are kernel parameters; stores are 4-lane transposed (quad_transpose): the
//    MMAs keep the shared-memory / L1 data path busy, so the epilogue must stay off it (DESIGN.md 4.1).
#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "philox.cuh"
#include "segnet.h"

namespace sivo {

namespace {

constexpr int kTcThreads = 12 * 32;  // warps: 0 halo TMA, 1 weight TMA, 2-3 MMA issuers, 4-11 epilogue (two per TMEM lane quarter)
constexpr int kEpiWarps = 8;
constexpr int kSlotBytes = 17 * 1024;  // one halo row: (128 + K - 1) px * 128 B, padded to a 1024-B multiple
constexpr int kMaxBStages = 6;

struct TcParams {
  int H, W, N_batch;       // spatial size and batch of input == output
  int cout_total;          // channel stride of the output tensor
  int n_tile;              // UMMA N (16 for the float logits layer, else 64 or 128)
  int chunks;              // Cin / 64
  int w_rep;               // weight tensor replicas in global memory (spreads the L2 hot spot all CTAs hammer)
  int dbg_noepi;           // timing experiment only: 1 = epilogue does nothing, 2 = TMEM loads only, 3 = no global stores
  int dbg_noshift;         // timing experiment only: ignore the kw shift of the A operand (wrong results)
  int dbg_noload;          // timing experiment only: halo rows are loaded once per ring slot and then reused (wrong results)
  int b_stages;            // weight ring depth (as many of kMaxBStages as fit in shared memory)
  int out_f32;             // 1: 16-channel float output (logits); 2: n_tile-wide float output (split-operand fp32 mode)
  int split;               // split-operand fp32 mode: A = [hi Cin | lo Cin] half planes of the float input, B K-axis = per real chunk
                           // [W_hi | W_lo | W_hi]; `chunks` then counts A chunks (2 * Cin / 64: hi and lo of each, interleaved)
  int cin_real;            // Cin (split mode: channel offset of the lo plane)
  float acc_scale;         // split mode: the weights were scaled by a power of two before the hi/lo split; 1 / that
  float rz_comp;           // split mode: expected truncation loss per accumulate step relative to the running sum (see seg_rows);
                           // each flushed segment of m steps is scaled by 1 + rz_comp * m before it is added (0 = off)
  int seg_rows;            // split mode: tap rows per accumulation segment.  The tensor core adds into its fp32 accumulator with
                           // truncation (measured: ~2^-25 relative per accumulate step, always towards zero, so it grows linearly
                           // with the chain length: 1.4e-5 for a 7x7x64 layer); the block's MMAs are therefore cut into segments
                           // of (A chunk, seg_rows tap rows) that each start a fresh accumulator, and the epilogue sums the
                           // segments in registers with round-to-nearest adds.
  int pairs_per_cta;       // row blocks (R output rows each) one CTA walks
  int strips;              // ceil(W / 128)
  int relu, has_bn, has_drop;
  float slope;
  void* out;
  // dropout fused into the epilogue (decoder convs of Basic: decdrop4 / decdrop3)
  uint64_t seed;
  const uint64_t* frame;
  int drop_layer;
  int drop_sample0;        // global index of batch image 0 (sample shards): the keep bits use drop_sample0 + img
  float drop_scale;
  // max-unpool fused into the epilogue (decoder convs): the output tensor is 2H x 2W and every pixel's channel
  // lands in the 2x2 position its pooling mask names, zeros elsewhere (upsample_layer.cpp:74-103)
  const uint8_t* unpool_mask;
  int mask_n;
  // 2x2/2 max pool with argmax fused into the epilogue (encoder convs): only the pooled tensor and its 2-bit mask are
  // written (pooling_layer.cpp:140-187: scan (0,0),(0,1),(1,0),(1,1), strict '>', so the first maximum wins)
  __half* pool_out;        // [N][H/2][W/2][cout_total]
  uint8_t* pool_mask;      // same shape
  // 1x1 classifier fused into the epilogue (the layer feeding Softmax): logits[j] = cls_b[j] + sum_c half(out[c]) * cls_w[c][j];
  // the 64-channel output itself is then never written
  int has_cls;
  float* cls_out;          // [N][H][W][16]
};

// Per-layer constants, passed by value as a kernel parameter so that the epilogue reads them from the constant bank
// (FFMA operands / LDC) instead of through L1 or shared memory, whose data path the MMA operand reads saturate.
constexpr int kMaxCout = 512;
struct TcConsts {
  float bias[kMaxCout], bn_scale[kMaxCout], bn_shift[kMaxCout];
  float cls_w[64 * 16];    // fused classifier: [cin][16] float (half-rounded values), j >= classes zero
  float cls_b[16];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a protocol bug must surface as a CUDA error, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  for (uint32_t spin = 0;; ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
    if (spin > (1u << 26)) asm volatile("trap;");  // inline: a __trap() call stub pins the whole kernel to the setmaxnreg minimum
  }
}

__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// K-major SWIZZLE_128B operand descriptor (cute::UMMA::SmemDescriptor): rows of 128 B, 8-row groups 1024 B apart.
// High word: stride byte offset 1024 >> 4 (bits 32-45), version 1 (bits 46-47), base_offset 0 (bits 49-51),
// layout SWIZZLE_128B = 2 (bits 61-63).  base_offset stays 0 even for operands that start kw*128 B into a
// 1024-B-aligned halo row: measured on B200 (profiles/r1_notes.md) the XOR phase follows the absolute
// shared-memory address bits [7:9]; writing (addr >> 7) & 7 there gives wrong products.
constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]),
        "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]),
        "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 4 x 4 transpose of 16-byte elements across each aligned group of four lanes: on entry lane c (of its group) holds
// e[0..3] = chunks 0..3 of its own pixel; on return e[j] = chunk c of the group's pixel j.  After it, one store
// instruction writes 64 contiguous bytes per pixel for 8 pixels instead of 16 bytes for 32: the epilogue's global
// stores share the L1 / shared-memory data path with the MMA operand reads, and a warp store that touches 32
// different lines holds that path four times longer (profiles/r1_notes.md).
template <typename V4>
__device__ __forceinline__ void quad_transpose(V4 (&e)[4], int lane) {
  static_assert(sizeof(V4) == 16, "16-byte elements");
  const bool odd = lane & 1, hi = lane & 2;
  auto xchg = [](V4 v, int m) {
    uint4 u = *reinterpret_cast<uint4*>(&v);
    u.x = __shfl_xor_sync(0xffffffffu, u.x, m);
    u.y = __shfl_xor_sync(0xffffffffu, u.y, m);
    u.z = __shfl_xor_sync(0xffffffffu, u.z, m);
    u.w = __shfl_xor_sync(0xffffffffu, u.w, m);
    return *reinterpret_cast<V4*>(&u);
  };
#pragma unroll
  for (int s = 0; s < 4; s += 2) {
    const V4 got = xchg(odd ? e[s] : e[s + 1], 1);
    if (odd) e[s] = got; else e[s + 1] = got;
  }
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const V4 got = xchg(hi ? e[s] : e[s + 2], 2);
    if (hi) e[s] = got; else e[s + 2] = got;
  }
}

// One output row of the epilogue for one thread (= one pixel x of row y): reads its accumulator columns from TMEM and
// applies the runtime-selected tail (see the file header).  `trow` = TMEM address of this row's first column for the
// thread's lane quarter, `n0` = first output channel of the CTA's tile.  Bias / BN / classifier constants come from the
// kernel parameters (constant bank): loads through L1 or shared memory would compete with the MMA operand reads.
// Must be called by all 32 lanes (warp shuffles); out-of-image pixels are masked at the stores.
__device__ __forceinline__ void epilogue_row(const TcParams& p, const TcConsts& cst, uint32_t trow, int img, int y, int x, int n0, int lane) {
    if (p.dbg_noepi == 1) return;
    if (p.dbg_noepi == 2) {
      for (int cc = 0; cc < p.n_tile; cc += 32) { uint32_t v[32]; tmem_ld32(trow + cc, v); if (v[0] == 0x12345678u && v[31] == 0x9abcdef0u) p.cls_out[0] = 1.f; }
      return;
    }
    if (p.dbg_noepi == 3) x += 1 << 20;  // every store is predicated off by the x < W test
    const int cl = lane & 3;          // this lane's 16-byte chunk after the transpose
    const int xg = x - cl;            // first pixel of the lane's group of four
    const bool row_ok = y < p.H && img < p.N_batch;  // img >= N: the odd image out of an image-pair tile (PK2)
    if (p.out_f32 == 1) {  // 16-channel float logits (the convolution feeding Softmax)
      uint32_t v[32];
      tmem_ld16(trow, v);
      float4 e[4];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float t = __fadd_rn(__uint_as_float(v[i]), cst.bias[i]);
        if (p.has_bn) t = __fadd_rn(__fmul_rn(t, cst.bn_scale[i]), cst.bn_shift[i]);
        if (p.relu) t = t > 0.f ? t : __fmul_rn(p.slope, t);
        reinterpret_cast<float*>(&e[i >> 2])[i & 3] = t;
      }
      quad_transpose(e, lane);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (row_ok && xg + j < p.W)
          *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + ((static_cast<size_t>(img) * p.H + y) * p.W + xg + j) * 16 + 4 * cl) = e[j];
      return;
    }
    if (p.has_cls) {  // conv (+bias) -> half rounding (as the unfused path stores it) -> 1x1 classifier -> float logits
      float l[16];
#pragma unroll
      for (int jj = 0; jj < 16; ++jj) l[jj] = cst.cls_b[jj];
#pragma unroll
      for (int cc = 0; cc < 64; cc += 32) {
        uint32_t v[32];
        tmem_ld32(trow + cc, v);
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float t = __fadd_rn(__uint_as_float(v[i]), cst.bias[cc + i]);
          if (p.has_bn) t = __fadd_rn(__fmul_rn(t, cst.bn_scale[cc + i]), cst.bn_shift[cc + i]);
          if (p.relu) t = t > 0.f ? t : __fmul_rn(p.slope, t);
          const float hv = __half2float(__float2half_rn(t));
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) l[jj] = fmaf(hv, cst.cls_w[(cc + i) * 16 + jj], l[jj]);
        }
      }
      float4 e[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) e[i] = make_float4(l[4 * i], l[4 * i + 1], l[4 * i + 2], l[4 * i + 3]);
      quad_transpose(e, lane);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (row_ok && xg + j < p.W)
          *reinterpret_cast<float4*>(p.cls_out + ((static_cast<size_t>(img) * p.H + y) * p.W + xg + j) * 16 + 4 * cl) = e[j];
      return;
    }
    uint32_t bits[4] = {0, 0, 0, 0};
    // max-unpool: fetch the 2-bit mask codes of the first 64 channels before touching TMEM, so the (DRAM / L2) latency
    // of the mask overlaps the accumulator loads.  Already in the transposed arrangement: lane (group, cl) reads the 8
    // codes of channels [8 cl, 8 cl + 8) of each of its group's four pixels.
    uint2 mrow[2][4] = {};
    const size_t mask_row = (static_cast<size_t>(img % p.mask_n) * p.H + y) * p.W;
    if (p.unpool_mask && row_ok) {
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (xg + j < p.W && h * 32 < p.n_tile)
            mrow[h][j] = __ldg(reinterpret_cast<const uint2*>(p.unpool_mask + (mask_row + xg + j) * p.cout_total + n0 + h * 32 + 8 * cl));
    }
    const bool inside = row_ok && x < p.W;
    for (int cc = 0; cc < p.n_tile; cc += 32) {
      uint32_t v[32];
      tmem_ld32(trow + cc, v);
      const int c0 = n0 + cc;
      if (p.has_drop && inside && ((c0 & 127) == 0 || cc == 0))
        dropout_bits128(p.seed, *p.frame, p.drop_layer, p.drop_sample0 + img, static_cast<uint32_t>(y * p.W + x), c0 >> 7, bits);
      const int wsel = (c0 >> 5) & 3;  // selects, not a dynamically indexed (= local-memory) array
      const uint32_t keep = !p.has_drop ? 0xFFFFFFFFu : wsel == 0 ? bits[0] : wsel == 1 ? bits[1] : wsel == 2 ? bits[2] : bits[3];
      uint4 e[4];
#pragma unroll
      for (int i = 0; i < 32; i += 2) {
        float f[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const int c = c0 + i + k;
          float t = __fadd_rn(__uint_as_float(v[i + k]), cst.bias[c]);
          if (p.has_bn) t = __fadd_rn(__fmul_rn(t, cst.bn_scale[c]), cst.bn_shift[c]);
          if (p.relu) t = t > 0.f ? t : __fmul_rn(p.slope, t);
          f[k] = t;
        }
        __half2 h = __floats2half2_rn(f[0], f[1]);
        if (p.has_drop) {  // y = x * keep * 2 on the stored half value (exact)
          __half2 sc = __floats2half2_rn((keep >> i) & 1u ? p.drop_scale : 0.f, (keep >> (i + 1)) & 1u ? p.drop_scale : 0.f);
          h = __hmul2(h, sc);
        }
        reinterpret_cast<uint32_t*>(&e[i >> 3])[(i >> 1) & 3] = *reinterpret_cast<uint32_t*>(&h);
      }
      quad_transpose(e, lane);  // e[j] = channels [c0 + 8 cl, c0 + 8 cl + 8) of pixel xg + j
      if (p.unpool_mask) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint2 m;
          if (cc == 0) m = mrow[0][j];
          else if (cc == 32) m = mrow[1][j];
          else {
            m = make_uint2(0u, 0u);
            if (row_ok && xg + j < p.W)
              m = __ldg(reinterpret_cast<const uint2*>(p.unpool_mask + (mask_row + xg + j) * p.cout_total + c0 + 8 * cl));
          }
          if (!(row_ok && xg + j < p.W)) continue;
          const uint32_t ew[4] = {e[j].x, e[j].y, e[j].z, e[j].w};         // half2 i = channels 2i, 2i+1 -> mask bytes 2i, 2i+1
          // the last block's epilogue is exposed at the end of every CTA, so its instruction count matters: one address per
          // output pixel (the four positions are constant offsets from it) and the eight mask bytes compared four at a time
          __half* const ob = static_cast<__half*>(p.out) +
              ((static_cast<size_t>(img) * 2 * p.H + 2 * y) * (2 * p.W) + 2 * (xg + j)) * p.cout_total + c0 + 8 * cl;
          const size_t row_step = static_cast<size_t>(2 * p.W) * p.cout_total;
#pragma unroll
          for (int pos = 0; pos < 4; ++pos) {
            const uint32_t eq0 = __vcmpeq4(m.x, 0x01010101u * pos), eq1 = __vcmpeq4(m.y, 0x01010101u * pos);  // 0xFF per matching byte
            // bytes (2i, 2i+1) of the mask widen to the two halves of word i
            const uint32_t s0 = ew[0] & __byte_perm(eq0, 0u, 0x1100), s1 = ew[1] & __byte_perm(eq0, 0u, 0x3322);
            const uint32_t s2 = ew[2] & __byte_perm(eq1, 0u, 0x1100), s3 = ew[3] & __byte_perm(eq1, 0u, 0x3322);
            *reinterpret_cast<uint4*>(ob + (pos >> 1) * row_step + (pos & 1) * p.cout_total) = make_uint4(s0, s1, s2, s3);
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (row_ok && xg + j < p.W)
            *reinterpret_cast<uint4*>(static_cast<__half*>(p.out) + ((static_cast<size_t>(img) * p.H + y) * p.W + xg + j) * p.cout_total + c0 + 8 * cl) = e[j];
      }
    }
}

// Two vertically adjacent output rows (y even) with the pooling epilogue: bias / BN / ReLU -> half (the value the
// unfused path would store) -> 2x2 max with first-maximum argmax; the horizontal neighbour lives in the adjacent lane.
__device__ __forceinline__ void epilogue_pool_rows(const TcParams& p, const TcConsts& cst, uint32_t trow0, uint32_t trow1, int img, int y, int x, int n0, int lane) {
  if (p.dbg_noepi) return;
  const bool writer = (lane & 1) == 0 && y + 1 < p.H && x + 1 < p.W && img < p.N_batch;
  for (int cc = 0; cc < p.n_tile; cc += 32) {
    uint32_t v0[32], v1[32];
    tmem_ld32(trow0 + cc, v0);
    tmem_ld32(trow1 + cc, v1);
    const int c0 = n0 + cc;
    uint32_t outv[16], outm[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) outm[i] = 0;
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
      __half2 h[2];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        float f[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int c = c0 + i + e;
          float t = __fadd_rn(__uint_as_float(r ? v1[i + e] : v0[i + e]), cst.bias[c]);
          if (p.has_bn) t = __fadd_rn(__fmul_rn(t, cst.bn_scale[c]), cst.bn_shift[c]);
          if (p.relu) t = t > 0.f ? t : __fmul_rn(p.slope, t);
          f[e] = t;
        }
        h[r] = __floats2half2_rn(f[0], f[1]);
      }
      const uint32_t a = *reinterpret_cast<uint32_t*>(&h[0]), c = *reinterpret_cast<uint32_t*>(&h[1]);
      const uint32_t b = __shfl_xor_sync(0xffffffffu, a, 1), d = __shfl_xor_sync(0xffffffffu, c, 1);
      // window in scan order: a = (y, x), b = (y, x+1), c = (y+1, x), d = (y+1, x+1); two channels per register
      uint32_t best = a, arg = 0;
      const uint32_t cand[3] = {b, c, d};
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        // strict '>' per half (false on NaN, like __hgt): 0xFFFF where the candidate wins
        const uint32_t sel = __hgt2_mask(*reinterpret_cast<const __half2*>(&cand[k]), *reinterpret_cast<const __half2*>(&best));
        best = (best & ~sel) | (cand[k] & sel);
        const uint32_t selb = __byte_perm(sel, 0u, 0x4420);  // the two half masks as two byte masks (bytes 0 and 1)
        arg = (arg & ~selb) | ((0x0101u * static_cast<uint32_t>(k + 1)) & selb);
      }
      outv[i >> 1] = best;
      outm[i >> 2] |= arg << (((i >> 1) & 1) * 16);  // two mask bytes per half2, four per 32-bit word
    }
    if (writer) {
      const size_t o = ((static_cast<size_t>(img) * (p.H >> 1) + (y >> 1)) * (p.W >> 1) + (x >> 1)) * p.cout_total + c0;
      uint4* dv = reinterpret_cast<uint4*>(p.pool_out + o);
#pragma unroll
      for (int i = 0; i < 4; ++i) dv[i] = make_uint4(outv[4 * i], outv[4 * i + 1], outv[4 * i + 2], outv[4 * i + 3]);
      uint4* dm = reinterpret_cast<uint4*>(p.pool_mask + o);
      dm[0] = make_uint4(outm[0], outm[1], outm[2], outm[3]);
      dm[1] = make_uint4(outm[4], outm[5], outm[6], outm[7]);
    }
  }
}

// ROLL = true : one 64-channel chunk (Cin == 64); halo rows persist in the ring while the CTA walks down its
//               strip, so each input row is fetched once per CTA.
// ROLL = false: Cin = 64 * NC; per (row pair, chunk) the kRows+K-1 halo rows of that chunk are fetched, used by
//               the K*K taps and released; the ring double-buffers chunks.
// KW < K : the kernel is K x KW over a *window-folded* input (KW = 1: every pixel's 64 "channels" are the 8-pixel x
//               8-channel window starting at it, so a 3-channel K x K layer is a K x 1 layer; see conv_tc_plan).
// PK2 (only with !ROLL): layers at most 64 pixels wide (Standard's conv5_x at 22x64) would fill half of every 128-pixel M tile.
//               Two images share a tile instead (rows 0-63: image 2z, rows 64-127: image 2z+1), and because the kw shift of a
//               shared-memory row would run from one image into the other, the shift is done by TMA: per (chunk, kw) the halo rows
//               are fetched as two 64-pixel boxes starting at pixel kw - 1 (out-of-range pixels and images zero-filled), so the
//               A operand of tap (kh, kw) is an unshifted, fully populated tile.  3x the halo traffic, which these small layers
//               have to spare; weights arrive in (kw, kh) order.
template <int K, bool ROLL, int kRows, int KW = K, bool PK2 = false>
__global__ void __launch_bounds__(kTcThreads, 1)
k_conv_tc(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const __grid_constant__ TcParams p,
          const __grid_constant__ TcConsts cst) {
  asm volatile("griddepcontrol.launch_dependents;");  // the next kernel's CTAs may be scheduled as soon as all of ours have started
  constexpr int RK = kRows + K - 1;                  // halo rows one row pair reads (per chunk)
  // rows are released as soon as their last tap row is issued; !ROLL double-buffers chunks where that fits (K = 7: RK + 2)
  constexpr int kSlots = ROLL ? RK : (K == 7 ? RK + 2 : 2 * RK);
  constexpr int kPad = (K - 1) / 2, kPadW = (KW - 1) / 2;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* a_slots = smem;
  uint8_t* b_stages = smem + kSlots * kSlotBytes;
  const int b_bytes = p.n_tile * 128;
  const int b_stride = (b_bytes + 1023) & ~1023;
  const int kBStages = p.b_stages;
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_stages + kBStages * b_stride);
  uint64_t* a_full = bars;                       // [kSlots]
  uint64_t* a_empty = a_full + kSlots;           // [kSlots]
  uint64_t* b_full = a_empty + kSlots;           // [kBStages]
  uint64_t* b_empty = b_full + kBStages;         // [kBStages]
  uint64_t* t_full = b_empty + kBStages;         // [2]
  uint64_t* t_empty = t_full + 2;                // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int strip = blockIdx.x % p.strips, rowblk = blockIdx.x / p.strips;
  static_assert(!PK2 || (!ROLL && KW == K), "image-pair tiles use the chunked kernel");
  constexpr int UPC = PK2 ? KW * RK : RK;          // halo units per (row block, chunk)
  const int n0 = blockIdx.y * p.n_tile;
  const int img = PK2 ? 2 * blockIdx.z : blockIdx.z;
  const int x0 = strip * 128;
  const int NC = ROLL ? 1 : p.chunks;
  const int total_pairs = (p.H + kRows - 1) / kRows;
  const int pair0 = rowblk * p.pairs_per_cta;
  const int npairs = min(p.pairs_per_cta, total_pairs - pair0);
  const int y_base = pair0 * kRows;              // first output row of this CTA
  const int n_units = ROLL ? npairs * kRows + K - 1 : npairs * NC * UPC;
  uint32_t tmem_cols = 32;
  while (tmem_cols < static_cast<uint32_t>(2 * kRows * p.n_tile)) tmem_cols <<= 1;

  if (threadIdx.x == 0) {
    // two MMA issuer warps (each owns half of the output rows): every consumer-side release needs both commits
    for (int i = 0; i < kSlots; ++i) { mbar_init(a_full + i, 1); mbar_init(a_empty + i, 2); }
    for (int i = 0; i < kBStages; ++i) { mbar_init(b_full + i, 1); mbar_init(b_empty + i, 2); }
    for (int i = 0; i < 2; ++i) { mbar_init(t_full + i, 2); mbar_init(t_empty + i, kEpiWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  // everything above touched only this CTA's shared / tensor memory; the producing kernel's results are needed from here on
  asm volatile("griddepcontrol.wait;" ::: "memory");

  // 384 threads start with 168 registers each; the TMA / MMA-issue warpgroup needs few, the two epilogue warpgroups
  // (32 accumulator words + packed outputs + masks per thread) need many: 128 x 56 + 256 x 216 = 62 464 <= 65 536
  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 56;" ::: "memory");
  if (warp == 0) {
    // ===== halo-row producer =====
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
      for (int u = 0; u < n_units; ++u) {
        const int slot = u % kSlots;
        const uint32_t round = static_cast<uint32_t>(u / kSlots);
        int ch = 0, yy, kw_p = 0;
        if (ROLL) {
          yy = y_base - kPad + u;
        } else {
          const int j = u / (NC * UPC), rem = u % (NC * UPC);
          ch = rem / UPC;
          kw_p = (rem % UPC) / RK;
          yy = y_base + j * kRows - kPad + rem % RK;
        }
        mbar_wait(a_empty + slot, (round & 1) ^ 1);
        const int a_ch = p.split ? (ch & 1) * p.cin_real + (ch >> 1) * 64 : ch * 64;  // split: chunk = (real chunk, hi | lo plane)
        if (PK2) {
          mbar_expect_tx(a_full + slot, static_cast<uint32_t>(2 * 64 * 128));
          tma_load_4d(a_slots + slot * kSlotBytes, &map_a, a_full + slot, a_ch, kw_p - kPadW, yy, img);
          tma_load_4d(a_slots + slot * kSlotBytes + 64 * 128, &map_a, a_full + slot, a_ch, kw_p - kPadW, yy, img + 1);
          continue;
        }
        mbar_expect_tx(a_full + slot, static_cast<uint32_t>((128 + KW - 1) * 128));
        tma_load_4d(a_slots + slot * kSlotBytes, &map_a, a_full + slot, a_ch, x0 - kPadW, yy, img);
      }
    }
  } else if (warp == 1) {
    // ===== weight producer =====
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_b)) : "memory");
      const int w_replica = static_cast<int>((blockIdx.x + blockIdx.z) % static_cast<unsigned>(p.w_rep));
      uint32_t it = 0;
      for (int j = 0; j < npairs; ++j)
        for (int ch = 0; ch < NC; ++ch) {
          // split: a hi chunk meets W_hi and W_lo (two tiles per tap), a lo chunk W_hi only; K-axis = [W_hi | W_lo | W_hi] per real chunk
          const int nrep = p.split && !(ch & 1) ? 2 : 1;
          for (int tap = 0; tap < K * KW; ++tap)
            for (int rep = 0; rep < nrep; ++rep, ++it) {
              const int st = it % kBStages;
              mbar_wait(b_empty + st, ((it / kBStages) & 1) ^ 1);
              mbar_expect_tx(b_full + st, static_cast<uint32_t>(b_bytes));
              const int kc = p.split ? (3 * (ch >> 1) + ((ch & 1) ? 2 : rep)) * 64 : ch * 64;
              const int tap_w = PK2 ? (tap % K) * K + tap / K : tap;  // PK2 consumes taps kw-major: (kw, kh) -> kh * K + kw
              tma_load_3d(b_stages + st * b_stride, &map_b, b_full + st, kc, n0, tap_w + w_replica * K * KW);
            }
        }
    }
  } else if (warp == 2 || warp == 3) {
    // ===== MMA issuers: warp 2 owns output rows [0, kRows/2), warp 3 the rest.  The loops are warp-uniform (all 32
    // lanes wait on the barriers) and one elected lane issues, so addresses stay in uniform registers: with N = 64 an
    // MMA retires every 32 tensor cycles and a single issuing thread running ~14 instructions per MMA was the limiter
    // (profiles/r1_notes.md).
    constexpr int kMine = kRows / 2;
    const int r_first = (warp - 2) * kMine;
    const uint32_t idesc = (1u << 4) | (static_cast<uint32_t>(p.n_tile >> 3) << 17) | (8u << 24);  // f16 x f16 -> f32, M = 128
    const uint32_t a_base = smem_u32(a_slots), b_base = smem_u32(b_stages);
    int st = 0;
    uint32_t b_phase = 0;
    int waited = 0;  // halo units whose TMA has been observed
    int seg = 0;  // accumulation segments issued so far (== row blocks unless split mode cuts a block into several)
    const int S = p.split ? p.seg_rows : K;
    for (int j = 0; j < npairs; ++j) {
      int acc = seg & 1;
      for (int ch = 0; ch < NC; ++ch)
      for (int kwo = 0; kwo < (PK2 ? KW : 1); ++kwo) {  // PK2: the kw shift is done by TMA, one set of halo rows per tap column
        const int base_u = ROLL ? j * kRows : PK2 ? ((j * NC + ch) * KW + kwo) * RK : (j * NC + ch) * RK;
        for (int kh = 0; kh < K; ++kh) {
          const bool seg_start = p.split ? (kh % S == 0) : (ch == 0 && kwo == 0 && kh == 0);
          const bool seg_end = p.split ? (kh % S == S - 1 || kh == K - 1) : (ch == NC - 1 && kwo == (PK2 ? KW - 1 : 0) && kh == K - 1);
          if (seg_start) {
            acc = seg & 1;
            mbar_wait(t_empty + acc, ((seg >> 1) & 1) ^ 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          }
          while (waited <= base_u + kh + kRows - 1 && waited < n_units) {
            mbar_wait(a_full + waited % kSlots, (waited / kSlots) & 1);
            ++waited;
          }
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          uint32_t a_row_lo[kMine], d_row[kMine];
#pragma unroll
          for (int m = 0; m < kMine; ++m) {
            const int unit = base_u + r_first + m + kh;
            a_row_lo[m] = (((a_base + (unit % kSlots) * kSlotBytes) & 0x3FFFFu) >> 4) | (1u << 16);
            d_row[m] = tmem_base + static_cast<uint32_t>((acc * kRows + r_first + m) * p.n_tile);
          }
          const uint32_t first_row = p.split ? (kh % S ? 1u : 0u) : ((ch | kwo | kh) ? 1u : 0u);  // 0: the segment's first MMAs clear
          const uint32_t kw_step = (p.dbg_noshift || PK2) ? 0u : 8u;
          const int nrep = p.split && !(ch & 1) ? 2 : 1;
#pragma unroll
          for (int kw = 0; kw < (PK2 ? 1 : KW); ++kw)
          for (int rep = 0; rep < nrep; ++rep) {
            mbar_wait(b_full + st, b_phase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            // descriptors: the high word is constant; the low word is (address >> 4) | LBO; a K step of 16 halfs
            // advances it by 32 B >> 4 = 2, a tap column by 128 B >> 4 = 8
            const uint32_t b_lo = (((b_base + st * b_stride) & 0x3FFFFu) >> 4) | (1u << 16);
            if (elect_one()) {
              // K step outer, row inner: consecutive MMAs go to different accumulators (an MMA chain on one
              // accumulator is serialised by the accumulate dependency; see profiles/r1_notes.md)
#pragma unroll
              for (int k = 0; k < 4; ++k) {
#pragma unroll
                for (int m = 0; m < kMine; ++m)
                  umma_f16(d_row[m], (static_cast<uint64_t>(kDescHi) << 32) | (a_row_lo[m] + kw_step * kw + 2 * k),
                           (static_cast<uint64_t>(kDescHi) << 32) | (b_lo + 2 * k), idesc, first_row | static_cast<uint32_t>(kw | k | rep));
              }
              umma_commit(b_empty + st);  // weight stage is free once both issuers' MMAs retire
            }
            __syncwarp();
            if (++st == kBStages) { st = 0; b_phase ^= 1; }
          }
          // halo row base_u + kh is only read by tap rows <= kh of this block.  ROLL: rows >= kRows are also the next block's, so
          // only kh < kRows goes back to the producer now (the next block's rows stream in behind the MMAs); !ROLL: every
          // chunk fetches its own rows, so row kh is dead after tap row kh
          if ((!ROLL || kh < kRows) && elect_one()) umma_commit(a_empty + (base_u + kh) % kSlots);
          __syncwarp();
          if (seg_end) {
            if (elect_one()) umma_commit(t_full + acc);
            __syncwarp();
            ++seg;
          }
        }
        if (elect_one()) {
          if (ROLL && K < kRows)  // fewer tap rows than output rows: release the rest of this block's own rows
            for (int i = K; i < kRows; ++i) umma_commit(a_empty + (base_u + i) % kSlots);
          if (!ROLL)  // the chunk's remaining halo rows (last read by tap row K - 1) are dead
            for (int i = K; i < RK; ++i) umma_commit(a_empty + (base_u + i) % kSlots);
        }
        __syncwarp();
      }
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;" ::: "memory");
    // ===== epilogue: TMEM -> registers -> bias / BN / ReLU / dropout -> half (or float logits) -> global =====
    // Measured (profiles/r1_notes.md): with four epilogue warps the stores + arithmetic of block j outlast the MMAs of
    // block j+1 (30 % of the frame's conv time).  Eight warps -- warps w and w+4 share a TMEM lane quarter and split the
    // rows of a block between them -- halve the epilogue's duration so it fits under the MMAs again.
    const int q = warp & 3;           // TMEM lane quarter this warp may access
    const int eset = (warp - 4) >> 2;  // 0: first half of the block's rows, 1: second half
    const int x = PK2 ? ((q * 32 + lane) & 63) : x0 + q * 32 + lane;  // PK2: tile rows 64-127 are the second image
    const int img_e = PK2 ? img + ((q * 32 + lane) >> 6) : img;
    if (!ROLL && kRows == 2 && p.split) {
      // split-operand fp32 mode: a block arrives as NC * ceil(K / seg_rows) accumulation segments; each epilogue warp owns one
      // of the block's two rows, sums the segments in registers (round-to-nearest) and finishes the row after the last one
      const int segs = NC * ((K + p.seg_rows - 1) / p.seg_rows);
      const int y_row = eset;  // kRows == 2: set 0 takes row 0, set 1 row 1
      int seg = 0;
      for (int j = 0; j < npairs; ++j) {
        float accr[128];
#pragma unroll
        for (int i = 0; i < 128; ++i) accr[i] = 0.f;
        const int segs_per_chunk = (K + p.seg_rows - 1) / p.seg_rows;
        for (int sg = 0; sg < segs; ++sg, ++seg) {
          const int acc = seg & 1;
          // accumulate steps of this segment: (tap rows) x KW x 4 K steps x (2 weight tiles for a hi chunk, 1 for a lo chunk).
          // The tensor core truncates each add towards zero: mean loss 0.36 x 2^-23 of the running sum per step (half an ulp,
          // ulp / |x| averaging 0.72 x 2^-23 over a binade), and a sum growing from 0 averages ~0.6 of its final value, so the
          // segment comes back short by ~0.216 x 2^-23 x m of itself: scaled back up here (leaves the zero-mean part).
          const int ch_s = sg / segs_per_chunk, kh0 = (sg % segs_per_chunk) * p.seg_rows;
          const int m_steps = min(p.seg_rows, K - kh0) * KW * 4 * ((ch_s & 1) ? 1 : 2);
          const float comp = 1.f + p.rz_comp * static_cast<float>(m_steps);
          mbar_wait(t_full + acc, (seg >> 1) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t trow = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>((acc * kRows + y_row) * p.n_tile);
          if (p.n_tile == 16) {
            uint32_t v[32];
            tmem_ld16(trow, v);
#pragma unroll
            for (int i = 0; i < 16; ++i) accr[i] = __fmaf_rn(__uint_as_float(v[i]), comp, accr[i]);
          } else {
#pragma unroll
            for (int cc = 0; cc < 128; cc += 32)
              if (cc < p.n_tile) {
                uint32_t v[32];
                tmem_ld32(trow + cc, v);
#pragma unroll
                for (int i = 0; i < 32; ++i) accr[cc + i] = __fmaf_rn(__uint_as_float(v[i]), comp, accr[cc + i]);
              }
          }
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive(t_empty + acc);
        }
        // finish the row: x 2^-s, bias, BN affine, ReLU in fp32 (as the reference), float NHWC store (4-lane transposed)
        const int y = y_base + j * kRows + y_row;
        const bool row_ok = y < p.H;
        const int cl = lane & 3, xg = x - cl;
        if (p.n_tile == 16) {
          float4 e[4];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float t = __fadd_rn(__fmul_rn(accr[i], p.acc_scale), cst.bias[i]);
            if (p.has_bn) t = __fadd_rn(__fmul_rn(t, cst.bn_scale[i]), cst.bn_shift[i]);
            if (p.relu) t = t > 0.f ? t : __fmul_rn(p.slope, t);
            reinterpret_cast<float*>(&e[i >> 2])[i & 3] = t;
          }
          quad_transpose(e, lane);
#pragma unroll
          for (int jj = 0; jj < 4; ++jj)
            if (row_ok && xg + jj < p.W)
              *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + ((static_cast<size_t>(img) * p.H + y) * p.W + xg + jj) * 16 + 4 * cl) = e[jj];
        } else {
#pragma unroll
          for (int cc = 0; cc < 128; cc += 32)
            if (cc < p.n_tile) {
              const int c0 = n0 + cc;
              float4 ea[4], eb[4];
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                float t = __fadd_rn(__fmul_rn(accr[cc + i], p.acc_scale), cst.bias[c0 + i]);
                if (p.has_bn) t = __fadd_rn(__fmul_rn(t, cst.bn_scale[c0 + i]), cst.bn_shift[c0 + i]);
                if (p.relu) t = t > 0.f ? t : __fmul_rn(p.slope, t);
                if (i < 16) reinterpret_cast<float*>(&ea[i >> 2])[i & 3] = t;
                else reinterpret_cast<float*>(&eb[(i - 16) >> 2])[i & 3] = t;
              }
              quad_transpose(ea, lane);  // ea[jj] = channels [c0 + 4 cl, +4) of pixel xg + jj; eb the same 16 channels further
              quad_transpose(eb, lane);
#pragma unroll
              for (int jj = 0; jj < 4; ++jj)
                if (row_ok && xg + jj < p.W) {
                  float* o = reinterpret_cast<float*>(p.out) + ((static_cast<size_t>(img) * p.H + y) * p.W + xg + jj) * p.cout_total + c0 + 4 * cl;
                  *reinterpret_cast<float4*>(o) = ea[jj];
                  *reinterpret_cast<float4*>(o + 16) = eb[jj];
                }
            }
        }
      }
    } else
    for (int j = 0; j < npairs; ++j) {
      const int acc = j & 1;
      mbar_wait(t_full + acc, (j >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      constexpr int kPer = kRows / 2;  // rows per epilogue set
      if (p.pool_out) {
        if (kRows == 4 || eset == 0) {  // a row pair per set (kRows == 2: one pair, taken by set 0)
          const int r = kRows == 4 ? 2 * eset : 0;
          const uint32_t trow = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>((acc * kRows + r) * p.n_tile);
          epilogue_pool_rows(p, cst, trow, trow + p.n_tile, img_e, y_base + j * kRows + r, x, n0, lane);
        }
      } else {
#pragma unroll
        for (int rr = 0; rr < kPer; ++rr) {
          const int r = eset * kPer + rr;
          const int y = y_base + j * kRows + r;
          const uint32_t trow = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>((acc * kRows + r) * p.n_tile);
          epilogue_row(p, cst, trow, img_e, y, x, n0, lane);
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(t_empty + acc);
    }
  }
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Paired-tap variant (64 -> 64 channels, 4-row blocks).  With N = 64 every MMA re-reads its 16 KB A tile from shared
// memory for 8 KB of weights: 192 B/clk of operand traffic against the SM's 128 B/clk, i.e. <= 67 % of the tensor
// rate.  But output row r at tap row kh and output row r-1 at tap row kh+1 read the SAME input row, so with the four
// accumulators laid out in decreasing row order one N = 128 MMA whose B tile stacks W(kh, kw) over W(kh+1, kw)
// updates acc(r) | acc(r-1) from a single A read.  Per (tap-row pair, kw) that is 5 MMA groups (N = 64, 128, 128,
// 128, 64) instead of 8: A traffic 80 KB instead of 128 KB per 1024 tensor cycles (141 B/clk), and 20 instead of 32
// instructions.  Weights come as [kw][kh][cout][cin] so one TMA box of 128 rows lands both taps of a pair.
// TRIPLE (K = 7): the last three tap rows (4, 5, 6) are stacked as well -- input row i of that group feeds acc(r) for every
// r with 0 <= i - r <= 2, one MMA of N = 64 / 128 / 192 / 192 / 128 / 64 per (input row, kw): 1664 tensor cycles instead of
// 1152 + 768 for a pair plus a single.  The weight stages grow to 24 KB (three 64-row boxes); the halo ring shrinks from
// K + 3 to 9 slots to pay for it (a block keeps at most 6 rows live, the rest is prefetch depth).
// NW = accumulator width = output channels per tap tile: 64 for the 64 -> 64 layers; 16 for conv_decode1 composed with the 1x1
// classifier (float logits straight from the accumulators; needs TRIPLE: its weight boxes are one tap each).
template <int K, bool TRIPLE = false, int NW = 64>
__global__ void __launch_bounds__(kTcThreads, 1)
k_conv_tc_pair(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const __grid_constant__ TcParams p,
               const __grid_constant__ TcConsts cst) {
  asm volatile("griddepcontrol.launch_dependents;");
  static_assert(!TRIPLE || K == 7, "the triple group is taps 4..6 of a 7-row filter");
  static_assert(NW == 64 || (NW == 16 && TRIPLE), "accumulator width");
  constexpr int kTapBytes = NW * 128;            // one tap's weight tile: NW rows of 64 half
  constexpr uint32_t kTapLo = kTapBytes >> 4;    // the same in descriptor units
  constexpr int kRows = 4, RK = kRows + K - 1, kSlots = TRIPLE ? 9 : RK, kPad = (K - 1) / 2, NP = TRIPLE ? 3 : (K + 1) / 2;
  constexpr int kBBytes = (TRIPLE ? 3 : 2) * kTapBytes;  // stacked weight tiles: stage stride
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* a_slots = smem;
  uint8_t* b_stages = smem + kSlots * kSlotBytes;
  const int kBStages = p.b_stages;
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_stages + kBStages * kBBytes);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + kSlots;
  uint64_t* b_full = a_empty + kSlots;
  uint64_t* b_empty = b_full + kBStages;
  uint64_t* t_full = b_empty + kBStages;
  uint64_t* t_empty = t_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int strip = blockIdx.x % p.strips, rowblk = blockIdx.x / p.strips;
  const int img = blockIdx.z;
  const int x0 = strip * 128;
  const int total_pairs = (p.H + kRows - 1) / kRows;
  const int pair0 = rowblk * p.pairs_per_cta;
  const int npairs = min(p.pairs_per_cta, total_pairs - pair0);
  const int y_base = pair0 * kRows;
  const int n_units = npairs * kRows + K - 1;
  constexpr uint32_t tmem_cols = 2 * kRows * NW;  // 2 stages x 4 rows x NW columns (512 or 128)

  if (threadIdx.x == 0) {
    for (int i = 0; i < kSlots; ++i) { mbar_init(a_full + i, 1); mbar_init(a_empty + i, 1); }
    for (int i = 0; i < kBStages; ++i) { mbar_init(b_full + i, 1); mbar_init(b_empty + i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(t_full + i, 1); mbar_init(t_empty + i, kEpiWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  // everything above touched only this CTA's shared / tensor memory; the producing kernel's results are needed from here on
  asm volatile("griddepcontrol.wait;" ::: "memory");

  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 56;" ::: "memory");
  if (warp == 0) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
      for (int u = 0; u < n_units; ++u) {
        const int slot = u % kSlots;
        mbar_wait(a_empty + slot, ((static_cast<uint32_t>(u / kSlots)) & 1) ^ 1);
        mbar_expect_tx(a_full + slot, static_cast<uint32_t>((128 + K - 1) * 128));
        tma_load_4d(a_slots + slot * kSlotBytes, &map_a, a_full + slot, 0, x0 - kPad, y_base - kPad + u, img);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_b)) : "memory");
      const int w_replica = static_cast<int>((blockIdx.x + blockIdx.z) % static_cast<unsigned>(p.w_rep));
      int st = 0;
      uint32_t ph = 0;
      for (int j = 0; j < npairs; ++j)
        for (int pp = 0; pp < NP; ++pp)
          for (int kw = 0; kw < K; ++kw) {
            mbar_wait(b_empty + st, ph ^ 1);
            if (TRIPLE) {  // 64-row boxes: two for a pair, three for the triple group
              const int nt = pp == 2 ? 3 : 2;
              mbar_expect_tx(b_full + st, static_cast<uint32_t>(nt * kTapBytes));
              for (int t = 0; t < nt; ++t)
                tma_load_3d(b_stages + st * kBBytes + t * kTapBytes, &map_b, b_full + st, 0, (kw * K + 2 * pp + t) * NW, w_replica);
            } else {
              mbar_expect_tx(b_full + st, static_cast<uint32_t>(kBBytes));
              // rows (kw*K + 2pp)*64 .. +127 of the [kw][kh][cout] x cin matrix; the odd last tap row drags in 64 rows it
              // never uses (the next kw's first tap, or zero fill past the end)
              tma_load_3d(b_stages + st * kBBytes, &map_b, b_full + st, 0, (kw * K + 2 * pp) * 64, w_replica);
            }
            if (++st == kBStages) { st = 0; ph ^= 1; }
          }
    }
  } else if (warp == 2) {
    // ===== MMA issuer (one warp: with N = 128 an MMA lasts 64 tensor cycles and costs 1-2 issue instructions) =====
    // one, two or three tap tiles wide (the names keep the NW = 64 widths)
    const uint32_t idesc64 = (1u << 4) | (static_cast<uint32_t>(NW >> 3) << 17) | (8u << 24);
    const uint32_t idesc128 = (1u << 4) | (static_cast<uint32_t>(2 * NW >> 3) << 17) | (8u << 24);
    const uint32_t idesc192 = (1u << 4) | (static_cast<uint32_t>(3 * NW >> 3) << 17) | (8u << 24);
    const uint32_t a_base = smem_u32(a_slots), b_base = smem_u32(b_stages);
    int st = 0;
    uint32_t b_phase = 0;
    int waited = 0;
    for (int j = 0; j < npairs; ++j) {
      const int acc = j & 1;
      mbar_wait(t_empty + acc, ((j >> 1) & 1) ^ 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int base_u = j * kRows;
      const uint32_t d0 = tmem_base + static_cast<uint32_t>(acc * kRows * NW);  // column of acc(row 3); acc(r) sits at d0 + (3 - r) * NW
      for (int pp = 0; pp < NP; ++pp) {
        const int kh0 = 2 * pp;
        const bool triple = TRIPLE && pp == 2;
        const bool paired = kh0 + 1 < K;
        const int last_unit = base_u + kh0 + (triple ? 2 : paired ? 1 : 0) + kRows - 1;
        while (waited <= last_unit && waited < n_units) {
          mbar_wait(a_full + waited % kSlots, (waited / kSlots) & 1);
          ++waited;
        }
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        uint32_t a_lo[kRows + 2];
#pragma unroll
        for (int i = 0; i <= kRows + 1; ++i)
          a_lo[i] = (((a_base + ((base_u + kh0 + i) % kSlots) * kSlotBytes) & 0x3FFFFu) >> 4) | (1u << 16);
#pragma unroll
        for (int kw = 0; kw < K; ++kw) {
          mbar_wait(b_full + st, b_phase);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t b_lo = (((b_base + st * kBBytes) & 0x3FFFFu) >> 4) | (1u << 16);
          if (elect_one()) {
            const uint64_t hi = static_cast<uint64_t>(kDescHi) << 32;
            if (pp == 0 && kw == 0) {
              // first tap pair of the block: plain N = 64 MMAs so that each accumulator's first MMA can clear it
#pragma unroll
              for (int t = 0; t < 2; ++t)
#pragma unroll
                for (int r = 0; r < kRows; ++r)
#pragma unroll
                  for (int k = 0; k < 4; ++k)
                    umma_f16(d0 + (3 - r) * NW, hi | (a_lo[r + t] + 2 * k), hi | (b_lo + kTapLo * t + 2 * k), idesc64,
                             static_cast<uint32_t>(t | k));
            } else if (triple) {
              // input row i of the group (block row 4 + i) x taps 4..6: acc(r) for r = i, i-1, i-2 where they exist.
              // Accumulators sit in decreasing row order, weights in increasing tap order, so each MMA is one contiguous
              // D range and one contiguous B range: (first acc column, first B row / 64, N)
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t ak = 8 * kw + 2 * k;
                umma_f16(d0 + 3 * NW, hi | (a_lo[0] + ak), hi | (b_lo + 2 * k), idesc64, 1u);          // row 4: acc0 <- W4
                umma_f16(d0 + 2 * NW, hi | (a_lo[1] + ak), hi | (b_lo + 2 * k), idesc128, 1u);         // row 5: acc1|acc0 <- W4|W5
                umma_f16(d0 + 1 * NW, hi | (a_lo[2] + ak), hi | (b_lo + 2 * k), idesc192, 1u);         // row 6: acc2|acc1|acc0 <- W4|W5|W6
                umma_f16(d0, hi | (a_lo[3] + ak), hi | (b_lo + 2 * k), idesc192, 1u);                  // row 7: acc3|acc2|acc1 <- W4|W5|W6
                umma_f16(d0, hi | (a_lo[4] + ak), hi | (b_lo + kTapLo + 2 * k), idesc128, 1u);         // row 8: acc3|acc2 <- W5|W6
                umma_f16(d0, hi | (a_lo[5] + ak), hi | (b_lo + 2 * kTapLo + 2 * k), idesc64, 1u);      // row 9: acc3 <- W6
              }
            } else if (paired) {
#pragma unroll
              for (int k = 0; k < 4; ++k) umma_f16(d0 + 3 * NW, hi | (a_lo[0] + 8 * kw + 2 * k), hi | (b_lo + 2 * k), idesc64, 1u);
#pragma unroll
              for (int i = 1; i < kRows; ++i)
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  umma_f16(d0 + (3 - i) * NW, hi | (a_lo[i] + 8 * kw + 2 * k), hi | (b_lo + 2 * k), idesc128, 1u);
#pragma unroll
              for (int k = 0; k < 4; ++k) umma_f16(d0, hi | (a_lo[kRows] + 8 * kw + 2 * k), hi | (b_lo + kTapLo + 2 * k), idesc64, 1u);
            } else {
#pragma unroll
              for (int r = 0; r < kRows; ++r)
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  umma_f16(d0 + (3 - r) * NW, hi | (a_lo[r] + 8 * kw + 2 * k), hi | (b_lo + 2 * k), idesc64, 1u);
            }
            umma_commit(b_empty + st);
          }
          __syncwarp();
          if (++st == kBStages) { st = 0; b_phase ^= 1; }
        }
        // halo rows base_u + kh0 (and + kh0 + 1) are read by no later tap row of this block and by no later block
        if (elect_one()) {
          if (kh0 < kRows) umma_commit(a_empty + (base_u + kh0) % kSlots);
          if (paired && kh0 + 1 < kRows) umma_commit(a_empty + (base_u + kh0 + 1) % kSlots);
        }
        __syncwarp();
      }
      if (elect_one()) {
        for (int i = K; i < kRows; ++i) umma_commit(a_empty + (base_u + i) % kSlots);  // K < 4: rows no tap row released
        umma_commit(t_full + acc);
      }
      __syncwarp();
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;" ::: "memory");
    const int q = warp & 3;
    const int eset = (warp - 4) >> 2;  // two warps per TMEM lane quarter: rows {0,1} and {2,3}
    const int x = x0 + q * 32 + lane;
    for (int j = 0; j < npairs; ++j) {
      const int acc = j & 1;
      mbar_wait(t_full + acc, (j >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (p.pool_out) {  // accumulators sit in decreasing row order: row r+1 is 64 columns below row r
        const int r = 2 * eset;
        const uint32_t trow = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>((acc * kRows + (3 - r)) * NW);
        epilogue_pool_rows(p, cst, trow, trow - NW, img, y_base + j * kRows + r, x, 0, lane);
      } else {
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          const int r = 2 * eset + rr;
          const int y = y_base + j * kRows + r;
          const uint32_t trow = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>((acc * kRows + (3 - r)) * NW);
          epilogue_row(p, cst, trow, img, y, x, 0, lane);
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(t_empty + acc);
    }
  }
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Full-stack variant for the composed 64 -> 16 layer (Basic: conv_decode1 x the 1x1 classifier as ONE 7x7 convolution with
// 16 output columns, see conv_tc_set_composed_classifier).  With N = 16 per tap an MMA is bound by its 4 KB A read, so ALL
// seven tap rows are stacked along N: input row i of a block feeds acc(r) for every output row r with 0 <= i - r <= 6, one
// MMA of N = 16 x (number of such rows) <= 112 per (input row, kw, K step).  Accumulators sit in decreasing row order and
// the weights in increasing tap order, so each MMA covers one contiguous TMEM column range and one contiguous weight range.
//  * R = 16 output rows per block, 2 accumulator stages x 16 rows x 16 columns = all 512 TMEM columns.
//  * The composed weights (49 taps x 16 x 64 half = 98 KB) stay resident in shared memory: no weight ring.
//  * Every input row is consumed by 28 consecutive MMAs and then dead: the halo ring is pure prefetch depth (7 slots).
//  * Model: per (kw, K step) a block issues MMAs of N = 16, 32, .., 96, 112 x 10, 96, .., 16 for its 22 input rows =
//    1152 cycles (N = 112: 56 tensor cycles against 60 of shared-memory operand reads) -> 32 K cycles per 16 x 128 px.
// K = 3: the same for a 3x3 layer with <= 16 float outputs (Standard's conv1_1_D): N = 16, 32, 48 x 14, 32, 16 per (kw, K step).
constexpr int kStackRows = 16, kStackSlots = 7;
template <int K>
__global__ void __launch_bounds__(kTcThreads, 1)
k_conv_tc_stack16(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const __grid_constant__ TcParams p,
                  const __grid_constant__ TcConsts cst) {
  asm volatile("griddepcontrol.launch_dependents;");
  constexpr int R = kStackRows, kSlots = kStackSlots, kPad = (K - 1) / 2, NW = 16;
  constexpr int kTapBytes = NW * 128, kKwBytes = K * kTapBytes, kWBytes = K * kKwBytes;  // 2 KB, 14 KB, 98 KB
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* w_smem = smem;                         // [kw][kh][16][64] half, K-major SWIZZLE_128B rows
  uint8_t* a_slots = smem + ((kWBytes + 1023) & ~1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(a_slots + kSlots * kSlotBytes);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + kSlots;
  uint64_t* w_full = a_empty + kSlots;
  uint64_t* t_full = w_full + 1;
  uint64_t* t_empty = t_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int strip = blockIdx.x % p.strips, rowblk = blockIdx.x / p.strips;
  const int img = blockIdx.z;
  const int x0 = strip * 128;
  const int total_blocks = (p.H + R - 1) / R;
  const int blk0 = rowblk * p.pairs_per_cta;
  const int nblk = min(p.pairs_per_cta, total_blocks - blk0);
  constexpr uint32_t tmem_cols = 2 * R * NW;  // 512

  if (threadIdx.x == 0) {
    for (int i = 0; i < kSlots; ++i) { mbar_init(a_full + i, 1); mbar_init(a_empty + i, 1); }
    mbar_init(w_full, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(t_full + i, 1); mbar_init(t_empty + i, kEpiWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  asm volatile("griddepcontrol.wait;" ::: "memory");

  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 56;" ::: "memory");
  if (warp == 0) {
    // ===== halo-row producer: R + 6 input rows per block, in order, through the ring =====
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
      uint32_t u = 0;
      for (int j = 0; j < nblk; ++j) {
        const int y0 = (blk0 + j) * R;
        for (int i = 0; i < R + K - 1; ++i, ++u) {
          const int slot = u % kSlots;
          mbar_wait(a_empty + slot, ((u / kSlots) & 1) ^ 1);
          if (p.dbg_noload && u >= static_cast<uint32_t>(kSlots)) { mbar_arrive(a_full + slot); continue; }
          mbar_expect_tx(a_full + slot, static_cast<uint32_t>((128 + K - 1) * 128));
          tma_load_4d(a_slots + slot * kSlotBytes, &map_a, a_full + slot, 0, x0 - kPad, y0 - kPad + i, img);
        }
      }
    }
  } else if (warp == 1) {
    // ===== weights: loaded once, resident =====
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_b)) : "memory");
      mbar_expect_tx(w_full, static_cast<uint32_t>(kWBytes));
      for (int kw = 0; kw < K; ++kw)  // one box {64 cin, 7 taps x 16 rows} per tap column
        tma_load_3d(w_smem + kw * kKwBytes, &map_b, w_full, 0, kw * K * NW, 0);
    }
  } else if (warp == 2) {
    // ===== MMA issuer =====
    const uint32_t a_base = smem_u32(a_slots), w_base = smem_u32(w_smem);
    const uint64_t hi = static_cast<uint64_t>(kDescHi) << 32;
    mbar_wait(w_full, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    uint32_t u = 0;
    for (int j = 0; j < nblk; ++j) {
      const int acc = j & 1;
      mbar_wait(t_empty + acc, ((j >> 1) & 1) ^ 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t d0 = tmem_base + static_cast<uint32_t>(acc * R * NW);  // acc(r) sits at d0 + (R - 1 - r) * NW
      for (int i = 0; i < R + K - 1; ++i, ++u) {
        const int slot = u % kSlots;
        mbar_wait(a_full + slot, (u / kSlots) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int r_hi = min(R - 1, i), r_lo = max(0, i - (K - 1));
        const int cnt = r_hi - r_lo + 1;             // output rows this input row feeds
        const int kh_lo = i - r_hi;                  // tap row meeting acc(r_hi); acc(r_hi - t) meets tap kh_lo + t
        const uint32_t d = d0 + static_cast<uint32_t>((R - 1 - r_hi) * NW);
        const uint32_t a_lo = (((a_base + slot * kSlotBytes) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t b_lo = (((w_base + kh_lo * kTapBytes) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t idesc = (1u << 4) | (static_cast<uint32_t>((cnt * NW) >> 3) << 17) | (8u << 24);
        if (elect_one()) {
          if (i < R) {
            // acc(i) meets its first tap here (kh = 0, kw = 0, K step 0): that MMA must clear it, the rest of the stack accumulates
            const uint32_t idesc1 = (1u << 4) | (static_cast<uint32_t>(NW >> 3) << 17) | (8u << 24);
            umma_f16(d, hi | a_lo, hi | b_lo, idesc1, 0u);
            if (cnt > 1) {
              const uint32_t idesc_r = (1u << 4) | (static_cast<uint32_t>(((cnt - 1) * NW) >> 3) << 17) | (8u << 24);
              umma_f16(d + NW, hi | a_lo, hi | (b_lo + (kTapBytes >> 4)), idesc_r, 1u);
            }
#pragma unroll
            for (int k = 1; k < 4; ++k) umma_f16(d, hi | (a_lo + 2 * k), hi | (b_lo + 2 * k), idesc, 1u);
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16(d, hi | (a_lo + 2 * k), hi | (b_lo + 2 * k), idesc, 1u);
          }
#pragma unroll
          for (int kw = 1; kw < K; ++kw)
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16(d, hi | (a_lo + 8 * kw + 2 * k), hi | (b_lo + kw * (kKwBytes >> 4) + 2 * k), idesc, 1u);
          umma_commit(a_empty + slot);   // the row is dead once these MMAs retire
          if (i == R + K - 2) umma_commit(t_full + acc);
        }
        __syncwarp();
      }
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;" ::: "memory");
    // ===== epilogue: 16 float logits per pixel straight from the accumulators (+ composed bias), 4-lane transposed stores =====
    const int q = warp & 3;
    const int eset = (warp - 4) >> 2;  // two warps per TMEM lane quarter: rows [0, 8) and [8, 16) of the block
    const int x = x0 + q * 32 + lane;
    for (int j = 0; j < nblk; ++j) {
      const int acc = j & 1;
      mbar_wait(t_full + acc, (j >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 2
      for (int rr = 0; rr < R / 2; ++rr) {
        const int r = eset * (R / 2) + rr;
        const int y = (blk0 + j) * R + r;
        const uint32_t trow = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * R * NW + (R - 1 - r) * NW);
        epilogue_row(p, cst, trow, img, y, x, 0, lane);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(t_empty + acc);
    }
  }
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

// ---- host: tensor maps through the driver entry point (no -lcuda at link time)
using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                              const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn encode_fn() {
  static EncodeFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  });
  if (!fn) fail(SIVO_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
  return fn;
}

void encode(CUtensorMap* m, void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes, const cuuint32_t* box) {
  cuuint32_t elem[5] = {1, 1, 1, 1, 1};
  CUresult r = encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, rank, base, dims, strides_bytes, box, elem, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) fail(SIVO_ECUDA, "cuTensorMapEncodeTiled failed with %d", static_cast<int>(r));
}

}  // namespace

struct ConvTcPlan {
  CUtensorMap map_a, map_b;
  TcParams p;
  TcConsts cst;
  dim3 grid;
  size_t smem;
  int k, rows;
  int kw;             // filter width the kernel walks (== k, or 1 for a window-folded layer)
  bool roll;
  bool pair = false;  // paired-tap kernel (64 -> 64 channels, 4-row blocks)
  bool triple = false;  // ... with taps 4..6 stacked three-high (K = 7)
  bool nw16 = false;    // ... with 16-wide accumulators: conv composed with the 1x1 classifier
  bool pk2 = false;     // two images per 128-pixel M tile (layers at most 64 pixels wide, chunked 3x3 kernel)
  bool stack16 = false; // composed 64 -> 16 layer on the full-stack kernel (all seven tap rows stacked along N, resident weights)
  DevBuf w_replicas;  // private replicated copy of the weights (w_rep > 1)
};

namespace {
// one place that names every instantiation: configure == true sets the dynamic shared-memory limit, else launches
void conv_tc_dispatch(const ConvTcPlan& plan, cudaStream_t s, bool configure) {
  auto go = [&](auto kern) {
    // the limit is per kernel function, not per launch: always raise it to the full 227 KB so that plans of different
    // sizes that share an instantiation (e.g. the 16-wide logits tile and a 64-wide layer) cannot lower it for each other
    if (configure) SIVO_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    else {
      // Programmatic dependent launch: the CTAs of this launch may start while the previous kernel of the stream is still
      // draining (on SMs it has already left, or never used) and run their prologue -- barrier init, TMEM allocation,
      // descriptor prefetch -- up to griddepcontrol.wait, which returns once that kernel has completed and flushed.
      // Opt-in (SIVO_B200_PDL=1): measured on B200 it shaves ~20 us off a lone SegNet frame (1.22 -> 1.20 ms) but the early
      // CTAs sit on SMs the concurrent extractor kernels could have used, so the three-call frame gets no faster.
      static const bool pdl = [] { const char* e = std::getenv("SIVO_B200_PDL"); return e && e[0] == '1'; }();
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = plan.grid;
      cfg.blockDim = dim3(kTcThreads);
      cfg.dynamicSmemBytes = plan.smem;
      cfg.stream = s;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = attr;
      cfg.numAttrs = pdl ? 1 : 0;
      SIVO_CUDA(cudaLaunchKernelEx(&cfg, kern, plan.map_a, plan.map_b, plan.p, plan.cst));
    }
  };
  const int K = plan.k;
  if (plan.stack16) { if (plan.k == 7) go(k_conv_tc_stack16<7>); else go(k_conv_tc_stack16<3>); }
  else if (plan.pair && plan.nw16) go(k_conv_tc_pair<7, true, 16>);
  else if (plan.pair) { if (K == 7 && plan.triple) go(k_conv_tc_pair<7, true>); else if (K == 7) go(k_conv_tc_pair<7>); else go(k_conv_tc_pair<3>); }
  else if (plan.kw == 1 && K > 1) {  // window-folded first layer (K x 1)
    if (!plan.roll) fail(SIVO_EINVAL, "window-folded convolution needs the rolling kernel");
    if (plan.rows == 4) { if (K == 7) go(k_conv_tc<7, true, 4, 1>); else go(k_conv_tc<3, true, 4, 1>); }
    else { if (K == 7) go(k_conv_tc<7, true, 2, 1>); else go(k_conv_tc<3, true, 2, 1>); }
  }
  else if (plan.roll && plan.rows == 4) { if (K == 7) go(k_conv_tc<7, true, 4>); else if (K == 3) go(k_conv_tc<3, true, 4>); else go(k_conv_tc<1, true, 4>); }
  else if (plan.roll) { if (K == 7) go(k_conv_tc<7, true, 2>); else if (K == 3) go(k_conv_tc<3, true, 2>); else go(k_conv_tc<1, true, 2>); }
  else if (plan.pk2) go(k_conv_tc<3, false, 2, 3, true>);
  else { if (K == 7) go(k_conv_tc<7, false, 2>); else if (K == 3) go(k_conv_tc<3, false, 2>); else go(k_conv_tc<1, false, 2>); }
}
}  // namespace

namespace {
void conv_tc_use_stack16(ConvTcPlan& plan, int K);  // below
// Upper bound on the row blocks one CTA walks.  Long-lived CTAs (one wave of 144 CTAs x 8 blocks = 0.19 ms) amortise the
// prologue best, but while they run no SM frees up, so the extractors' short dependent kernels -- highest stream priority
// notwithstanding -- each wait for a whole CTA lifetime; SIVO_B200_TC_MAX_PPC trades the two (unit: row blocks of this kernel;
// the 16-row full-stack blocks count `scale` x as much).
int tc_max_ppc(int scale = 1) {
  static const int v = [] { const char* e = std::getenv("SIVO_B200_TC_MAX_PPC"); return e ? std::max(1, atoi(e)) : 24; }();
  return std::max(1, v / scale);
}
// Output rows per accumulator stage.  4 rows share each weight tile (TMEM: 2 stages x rows x n_tile <= 512 columns), but
// a layer too small to give every SM a 4-row block runs 2-row blocks instead: twice the CTAs, half the work each.
int tc_rows(int K, bool roll, int n_tile, int columns = 1 << 30, int H = 1 << 20) {
  if (!(roll && n_tile <= 64)) return 2;
  return static_cast<long>(columns) * ceil_div(H, 4) < 148 ? 2 : 4;
}
size_t tc_smem_bytes(int K, bool roll, int n_tile, int stages) {
  const int rows = tc_rows(K, roll, n_tile);  // the 4-row variant is the larger footprint
  const int rk = rows + K - 1;
  const int slots = roll ? rk : (K == 7 ? rk + 2 : 2 * rk);  // k_conv_tc's kSlots
  const int b_stride = (n_tile * 128 + 1023) & ~1023;
  return 1024 + static_cast<size_t>(slots) * kSlotBytes + static_cast<size_t>(stages) * b_stride + (2 * slots + 2 * stages + 4) * 8 + 16 + 64 * 16 * 4;  // barriers, TMEM slot, fused-classifier weights
}
int tc_stages(int K, bool roll, int n_tile) {  // deepest weight ring that fits (0 = configuration does not fit)
  for (int st = kMaxBStages; st >= 3; --st)
    if (tc_smem_bytes(K, roll, n_tile, st) <= 227 * 1024) return st;
  return 0;
}
int tc_pick_n(const Op& op, const TensorView& out, bool roll) {
  if (out.dt == DType::F32 && out.cs <= 16) return 16;  // the float logits layer
  int n = (op.cout_p % 128 == 0) ? 128 : 64;
  if (!tc_stages(op.k, roll, n)) n = 64;
  return n;
}
}  // namespace

bool conv_tc_supported(const Op& op, const TensorView& in, const TensorView& out) {
  if (const char* e = std::getenv("SIVO_B200_NO_TC")) if (e[0] == '1') return false;
  if (in.dt != DType::F16) return false;
  if (op.k != 1 && op.k != 3 && op.k != 7) return false;
  if (op.cout_p > kMaxCout) return false;
  if (op.fold_kw) {
    if (in.cs != 8 || op.cin_p != 64 || (op.k != 3 && op.k != 7) || out.dt != DType::F16 || op.cout % 64 || out.cs != op.cout) return false;
    return tc_stages(op.k, true, tc_pick_n(op, out, true)) > 0;
  }
  if (op.split) {  // `in` = the [hi Cin | lo Cin] half planes of the float input
    if (op.cin % 64 || in.cs != 2 * op.cin || out.dt != DType::F32) return false;
    if (!((out.cs == op.cout && op.cout % 64 == 0) || (out.cs == 16 && op.cout <= 16))) return false;
    return tc_stages(op.k, false, tc_pick_n(op, out, false)) > 0;
  }
  if (in.cs % 64 || op.cin != in.cs) return false;
  if (out.dt == DType::F16) {
    if (op.cout % 64 || out.cs != op.cout) return false;
  } else {
    if (out.cs != 16 || op.cout > 16) return false;  // float logits, 16-channel pixels
  }
  const bool roll = in.cs == 64;
  return tc_stages(op.k, roll, tc_pick_n(op, out, roll)) > 0;
}

std::shared_ptr<ConvTcPlan> conv_tc_plan(const Op& op, const TensorView& in, const TensorView& out, const void* w_tc) {
  auto plan = std::make_shared<ConvTcPlan>();
  const int K = op.k;
  const int KW = op.fold_kw ? 1 : K;
  const bool roll = (in.cs == 64 || op.fold_kw) && !op.split;
  // the kernel variant (image pairs, rows per block and with them the paired-tap kernel) follows the planning batch; only the
  // grid follows the real one
  const int plan_n = op.plan_n > 0 ? op.plan_n : in.n;
  if (op.fold_kw) {
    // window-folded input: `in` is the zero-padded 8-channel image [N][H][W + 8][8] half (3 zero pixels left, 5 right);
    // "pixel" x of the operand is the 128-byte window of 8 pixels x 8 channels starting at padded pixel x, i.e. image
    // pixels x-3 .. x+4: a tensor whose W stride (16 B) is smaller than its row (128 B).  TMA only needs 16-byte
    // multiples, so one box {64, 128, 1, 1} lands the K = kw*8 + c operand rows of 128 output pixels, and the K x K
    // layer over 3 channels becomes a K x 1 layer over these 64 -- no expanded tensor in HBM.  `in.w` counts the padded row.
    const int w_valid = in.w - 8;
    cuuint64_t dims[4] = {64, static_cast<cuuint64_t>(w_valid), static_cast<cuuint64_t>(in.h), static_cast<cuuint64_t>(in.n)};
    cuuint64_t strides[3] = {16, static_cast<cuuint64_t>(in.w) * 16, static_cast<cuuint64_t>(in.h) * in.w * 16};
    cuuint32_t box[4] = {64, 128, 1, 1};
    encode(&plan->map_a, in.p, 4, dims, strides, box);
  } else {  // input: NHWC half, dims (C, W, H, N)
    cuuint64_t dims[4] = {static_cast<cuuint64_t>(in.cs), static_cast<cuuint64_t>(in.w), static_cast<cuuint64_t>(in.h),
                          static_cast<cuuint64_t>(in.n)};
    cuuint64_t strides[3] = {static_cast<cuuint64_t>(in.cs) * 2, static_cast<cuuint64_t>(in.w) * in.cs * 2,
                             static_cast<cuuint64_t>(in.h) * in.w * in.cs * 2};
    const char* pk2_env = std::getenv("SIVO_B200_TC_PK2");
    plan->pk2 = !roll && !op.split && K == 3 && in.w <= 64 && plan_n >= 2 && !(pk2_env && pk2_env[0] == '0');
    cuuint32_t box[4] = {64, static_cast<cuuint32_t>(plan->pk2 ? 64 : 128 + K - 1), 1, 1};
    encode(&plan->map_a, in.p, 4, dims, strides, box);
  }
  const int n_tile = tc_pick_n(op, out, roll);
  int w_rep = 1;
  if (const char* e = std::getenv("SIVO_B200_TC_WREP")) w_rep = std::max(1, std::min(16, atoi(e)));
  {  // weights: [replica][tap][cout_p][cin_p] half, dims (cin, cout, replica * tap)
    const size_t one = static_cast<size_t>(K) * KW * op.cout_p * op.cin_p * 2 * (op.split ? 3 : 1);
    void* wbase = const_cast<void*>(w_tc);
    if (w_rep > 1) {
      plan->w_replicas.alloc(one * w_rep);
      for (int r = 0; r < w_rep; ++r)
        SIVO_CUDA(cudaMemcpy(plan->w_replicas.as<uint8_t>() + r * one, w_tc, one, cudaMemcpyDeviceToDevice));
      wbase = plan->w_replicas.p;
    }
    const int kext = op.split ? 3 * op.cin_p : op.cin_p;  // split: [W_hi | W_lo | W_hi] per 64-channel chunk along K
    cuuint64_t dims[3] = {static_cast<cuuint64_t>(kext), static_cast<cuuint64_t>(op.cout_p), static_cast<cuuint64_t>(K * KW * w_rep)};
    cuuint64_t strides[2] = {static_cast<cuuint64_t>(kext) * 2, static_cast<cuuint64_t>(op.cout_p) * kext * 2};
    cuuint32_t box[3] = {64, static_cast<cuuint32_t>(n_tile), 1};
    encode(&plan->map_b, wbase, 3, dims, strides, box);
  }
  TcParams& p = plan->p;
  p.H = in.h; p.W = op.fold_kw ? in.w - 8 : in.w; p.N_batch = in.n;
  p.cout_total = out.cs;
  p.n_tile = n_tile;
  p.chunks = op.fold_kw ? 1 : in.cs / 64;
  p.w_rep = w_rep;
  p.out_f32 = out.dt == DType::F32 ? (n_tile == 16 ? 1 : 2) : 0;
  p.split = op.split ? 1 : 0;
  p.cin_real = op.cin;
  p.acc_scale = op.split ? op.acc_scale : 1.f;
  p.seg_rows = 1;  // a segment per (chunk, tap row): 7x7 56 / 28 accumulate steps, 3x3 24 / 12, 1x1 8 / 4 (measured: profiles/r2_parity.md)
  if (const char* e = std::getenv("SIVO_B200_SPLIT_SEG")) p.seg_rows = std::max(1, std::min(K, atoi(e)));
  p.rz_comp = 0.216f * 1.1920929e-7f;  // x 2^-23
  if (const char* e = std::getenv("SIVO_B200_SPLIT_RZ")) p.rz_comp = static_cast<float>(atof(e)) * 1.1920929e-7f;
  p.strips = ceil_div(p.W, 128);
  const int cout_tiles = p.out_f32 == 1 ? 1 : op.cout_p / n_tile;
  const int n_z = plan->pk2 ? ceil_div(in.n, 2) : in.n;  // PK2: an image pair per tile
  const int columns = p.strips * n_z * cout_tiles;
  const int rows = tc_rows(K, roll, n_tile, p.strips * (plan->pk2 ? ceil_div(plan_n, 2) : plan_n) * cout_tiles, in.h);
  const int total_pairs = ceil_div(in.h, rows);
  // row blocks per CTA: minimise (waves of 148 SMs) x (blocks per CTA + ~1 block of prologue / halo overhead)
  int ppc = 1;
  double best_cost = 1e30;
  for (int c = 1; c <= std::min(total_pairs, tc_max_ppc()); ++c) {
    const long ctas = static_cast<long>(columns) * ceil_div(total_pairs, c);
    const double cost = static_cast<double>((ctas + 147) / 148) * (c + (roll ? (K - 1.0) / rows * 0.5 + 0.5 : 0.3));
    if (cost < best_cost - 1e-9) { best_cost = cost; ppc = c; }
  }
  p.pairs_per_cta = ppc;
  p.relu = op.relu; p.has_bn = op.has_bn; p.slope = op.slope;
  std::memset(&plan->cst, 0, sizeof(TcConsts));
  if (static_cast<int>(op.h_bias.size()) != op.cout_p || (op.has_bn && (static_cast<int>(op.h_bn_scale.size()) != op.cout_p ||
                                                                         static_cast<int>(op.h_bn_shift.size()) != op.cout_p)))
    fail(SIVO_EINVAL, "conv_tc_plan: host copies of the bias / BN constants are missing");
  std::copy(op.h_bias.begin(), op.h_bias.end(), plan->cst.bias);
  if (op.has_bn) {
    std::copy(op.h_bn_scale.begin(), op.h_bn_scale.end(), plan->cst.bn_scale);
    std::copy(op.h_bn_shift.begin(), op.h_bn_shift.end(), plan->cst.bn_shift);
  }
  p.out = out.p;
  p.has_drop = 0; p.seed = 0; p.frame = nullptr; p.drop_layer = 0; p.drop_sample0 = 0; p.drop_scale = 2.f;
  p.unpool_mask = nullptr; p.mask_n = 1;
  p.dbg_noshift = 0;
  p.dbg_noepi = 0;
  if (const char* e = std::getenv("SIVO_B200_TC_NOEPI")) p.dbg_noepi = atoi(e);
  if (const char* e = std::getenv("SIVO_B200_TC_NOSHIFT")) p.dbg_noshift = e[0] == '1';
  p.dbg_noload = 0;
  if (const char* e = std::getenv("SIVO_B200_TC_NOLOAD")) p.dbg_noload = e[0] == '1';
  p.pool_out = nullptr; p.pool_mask = nullptr;
  p.has_cls = 0; p.cls_out = nullptr;
  plan->grid = dim3(p.strips * ceil_div(total_pairs, ppc), cout_tiles, n_z);
  p.b_stages = tc_stages(K, roll, n_tile);
  if (const char* e = std::getenv("SIVO_B200_TC_BSTAGES")) p.b_stages = std::max(2, std::min(p.b_stages, atoi(e)));  // experiment knob
  plan->smem = tc_smem_bytes(K, roll, n_tile, p.b_stages);
  const char* pair_env = std::getenv("SIVO_B200_TC_PAIR");
  if (roll && !op.fold_kw && rows == 4 && n_tile == 64 && op.cout_p == 64 && !p.out_f32 && (K == 7 || K == 3) && op.w_tc_pair.p &&
      !(pair_env && pair_env[0] == '0')) {  // default on: ~2 % faster than the N = 64 kernel (profiles/r1_notes.md)
    // paired-tap kernel: weights as one [K*K*64 rows][64 cin] matrix in (kw, kh, cout) row order, 128-row boxes
    const size_t one = static_cast<size_t>(K) * K * 64 * 128;
    void* wbase = op.w_tc_pair.p;
    if (w_rep > 1) {
      plan->w_replicas.alloc(one * w_rep);
      for (int r = 0; r < w_rep; ++r)
        SIVO_CUDA(cudaMemcpy(plan->w_replicas.as<uint8_t>() + r * one, op.w_tc_pair.p, one, cudaMemcpyDeviceToDevice));
      wbase = plan->w_replicas.p;
    }
    const char* triple_env = std::getenv("SIVO_B200_TC_TRIPLE");
    plan->triple = K == 7 && !(triple_env && triple_env[0] == '0');
    cuuint64_t dims[3] = {64, static_cast<cuuint64_t>(K) * K * 64, static_cast<cuuint64_t>(w_rep)};
    cuuint64_t strides[2] = {128, one};
    cuuint32_t box[3] = {64, static_cast<cuuint32_t>(plan->triple ? 64 : 128), 1};
    encode(&plan->map_b, wbase, 3, dims, strides, box);
    plan->pair = true;
    const int slots = plan->triple ? 9 : rows + K - 1;
    const size_t stage = plan->triple ? 24576 : 16384;
    int st = plan->triple ? 3 : 6;
    auto bytes = [&](int n) { return 1024 + static_cast<size_t>(slots) * kSlotBytes + static_cast<size_t>(n) * stage + (2 * slots + 2 * n + 4) * 8 + 16; };
    while (st > 2 && bytes(st) > 227 * 1024) --st;
    if (bytes(st) > 227 * 1024) fail(SIVO_EINVAL, "paired-tap kernel does not fit in shared memory");
    p.b_stages = st;
    plan->smem = bytes(st);
  }
  plan->k = K;
  plan->kw = KW;
  plan->roll = roll;
  plan->rows = rows;
  const char* stack_env = std::getenv("SIVO_B200_STACK16");
  if (roll && !op.fold_kw && !op.split && p.out_f32 == 1 && (K == 3 || K == 7) && op.cin == 64 && op.cout <= 16 &&
      op.h_w_raw.size() == static_cast<size_t>(op.cout) * 64 * K * K && !(stack_env && stack_env[0] == '0')) {
    // the float logits layer (Standard: conv1_1_D, 64 -> 15, 3x3): all K tap rows stacked along N on the full-stack kernel
    std::vector<__half> w(static_cast<size_t>(K) * K * 16 * 64, __float2half_rn(0.f));
    for (int o = 0; o < op.cout; ++o)
      for (int i = 0; i < 64; ++i)
        for (int kh = 0; kh < K; ++kh)
          for (int kw = 0; kw < K; ++kw)
            w[((static_cast<size_t>(kw) * K + kh) * 16 + o) * 64 + i] =
                __float2half_rn(op.h_w_raw[((static_cast<size_t>(o) * 64 + i) * K + kh) * K + kw]);
    plan->w_replicas.alloc(w.size() * sizeof(__half));
    SIVO_CUDA(cudaMemcpy(plan->w_replicas.p, w.data(), w.size() * sizeof(__half), cudaMemcpyHostToDevice));
    conv_tc_use_stack16(*plan, K);
  }
  conv_tc_dispatch(*plan, nullptr, true);
  return plan;
}

void conv_tc_set_dropout(ConvTcPlan& plan, uint64_t seed, const uint64_t* frame_dev, int layer, int sample0, float scale) {
  plan.p.has_drop = 1;
  plan.p.seed = seed;
  plan.p.frame = frame_dev;
  plan.p.drop_layer = layer;
  plan.p.drop_sample0 = sample0;
  plan.p.drop_scale = scale;
}

void conv_tc_set_unpool(ConvTcPlan& plan, const uint8_t* mask, int mask_n, void* out_2h_2w) {
  plan.p.unpool_mask = mask;
  plan.p.mask_n = mask_n;
  plan.p.out = out_2h_2w;
}

std::vector<__half> conv_tc_pair_weights(const float* w_cout_cin_k_k, int K) {
  // [kw][kh][cout = 64][cin = 64] half from Caffe's (cout, cin, kh, kw) float blob
  std::vector<__half> out(static_cast<size_t>(K) * K * 64 * 64);
  for (int kw = 0; kw < K; ++kw)
    for (int kh = 0; kh < K; ++kh)
      for (int co = 0; co < 64; ++co)
        for (int ci = 0; ci < 64; ++ci)
          out[((static_cast<size_t>(kw) * K + kh) * 64 + co) * 64 + ci] =
              __float2half_rn(w_cout_cin_k_k[((static_cast<size_t>(co) * 64 + ci) * K + kh) * K + kw]);
  return out;
}

std::vector<__half> conv_tc_split_weights(const float* W, int cout, int cin, int K, int cout_p, int cin_p, float* acc_scale) {
  // [tap][cout_p][3 cin_p] half: per 64-channel chunk c of the K axis [W_hi(c) | W_lo(c) | W_hi(c)], where W * 2^s = W_hi + W_lo.
  // The power-of-two scale lifts the low parts out of half's subnormal range (|w| ~ 1e-2 has ulp(hi) ~ 2^-17 < 2^-14); the
  // epilogue multiplies the accumulator by 2^-s, which is exact.
  float wmax = 0.f;
  for (size_t i = 0; i < static_cast<size_t>(cout) * cin * K * K; ++i) wmax = std::max(wmax, std::fabs(W[i]));
  int e = 0;
  if (wmax > 0.f && std::isfinite(wmax)) { std::frexp(wmax, &e); e = 8 - e; }  // wmax * 2^e in [128, 256)
  e = std::max(-24, std::min(24, e));
  const float up = std::ldexp(1.f, e);
  *acc_scale = std::ldexp(1.f, -e);
  const int kext = 3 * cin_p;
  std::vector<__half> wt(static_cast<size_t>(K) * K * cout_p * kext, __float2half_rn(0.f));
  for (int co = 0; co < cout; ++co)
    for (int ci = 0; ci < cin; ++ci)
      for (int t = 0; t < K * K; ++t) {
        const float v = W[(static_cast<size_t>(co) * cin + ci) * K * K + t] * up;
        const __half hi = __float2half_rn(v), lo = __float2half_rn(v - __half2float(hi));
        __half* row = wt.data() + (static_cast<size_t>(t) * cout_p + co) * kext + (ci / 64) * 192 + ci % 64;
        row[0] = hi; row[64] = lo; row[128] = hi;
      }
  return wt;
}

bool conv_tc_can_fuse_pool(const ConvTcPlan& plan) {
  return !plan.p.out_f32 && !plan.p.unpool_mask && !plan.p.has_drop && !plan.p.has_cls && (plan.p.H % 2) == 0 && (plan.p.W % 2) == 0;
}

void conv_tc_set_pool(ConvTcPlan& plan, void* pooled, uint8_t* mask) {
  plan.p.pool_out = static_cast<__half*>(pooled);
  plan.p.pool_mask = mask;
}

bool conv_tc_can_fuse_classifier(const ConvTcPlan& plan) {
  return plan.roll && plan.p.n_tile == 64 && plan.p.cout_total == 64 && !plan.p.out_f32 && !plan.p.unpool_mask && !plan.p.has_drop && !plan.p.pool_out;
}

void conv_tc_set_classifier(ConvTcPlan& plan, const float* w_cin_by_cout, int stride, const float* bias, int n_bias, float* logits) {
  for (int c = 0; c < 64; ++c)
    for (int j = 0; j < 16; ++j) plan.cst.cls_w[c * 16 + j] = j < stride ? w_cin_by_cout[static_cast<size_t>(c) * stride + j] : 0.f;
  for (int j = 0; j < 16; ++j) plan.cst.cls_b[j] = j < n_bias ? bias[j] : 0.f;
  plan.p.has_cls = 1;
  plan.p.cls_out = logits;
}

namespace {
// Points a plan whose weights sit in plan.w_replicas as [kw][kh][16][64] half at the full-stack kernel (k_conv_tc_stack16<K>).
void conv_tc_use_stack16(ConvTcPlan& plan, int K) {
  TcParams& p = plan.p;
  cuuint64_t dims[3] = {64, static_cast<cuuint64_t>(K) * K * 16, 1};
  cuuint64_t strides[2] = {128, static_cast<cuuint64_t>(K) * K * 16 * 128};
  cuuint32_t box_s[3] = {64, static_cast<cuuint32_t>(K * 16), 1};  // one box per tap column: K taps x 16 rows
  encode(&plan.map_b, plan.w_replicas.p, 3, dims, strides, box_s);
  plan.stack16 = true;
  plan.pair = plan.triple = plan.nw16 = false;
  const int total_blocks = ceil_div(p.H, kStackRows);
  const int columns = p.strips * p.N_batch;
  int ppc = 1;
  double best_cost = 1e30;
  for (int c = 1; c <= std::min(total_blocks, tc_max_ppc(2)); ++c) {  // (waves of 148 SMs) x (blocks per CTA + weight load / prologue)
    const long ctas = static_cast<long>(columns) * ceil_div(total_blocks, c);
    const double cost = static_cast<double>((ctas + 147) / 148) * (c + 0.35);
    if (cost < best_cost - 1e-9) { best_cost = cost; ppc = c; }
  }
  p.pairs_per_cta = ppc;
  plan.grid = dim3(p.strips * ceil_div(total_blocks, ppc), 1, p.N_batch);
  const size_t wbytes = (static_cast<size_t>(K) * K * 16 * 128 + 1023) & ~static_cast<size_t>(1023);
  plan.smem = 1024 + wbytes + static_cast<size_t>(kStackSlots) * kSlotBytes + (2 * kStackSlots + 1 + 4) * 8 + 16;
}
}  // namespace

bool conv_tc_can_compose_classifier(const ConvTcPlan& plan) {
  return plan.pair && plan.triple && plan.k == 7 && !plan.p.out_f32 && !plan.p.unpool_mask && !plan.p.has_drop && !plan.p.pool_out &&
         !plan.p.has_cls && !plan.p.relu && !plan.p.has_bn && plan.p.cout_total == 64;
}

void conv_tc_set_composed_classifier(ConvTcPlan& plan, const Op& conv, const float* wc, const float* bc, int n_cls, float* logits) {
  const int K = 7;
  if (n_cls > 16 || conv.h_w_raw.size() != static_cast<size_t>(64) * 64 * K * K || conv.h_bias.size() < 64)
    fail(SIVO_EINVAL, "composed classifier: unexpected layer shapes");
  // W'[o][i][kh][kw] = sum_c wc[o][c] W[c][i][kh][kw] in double, rounded once to half; rows o >= n_cls stay zero.
  // Device layout [kw][kh][16][64]: one 16-row TMA box per tap, K-major rows like every other B tile.
  std::vector<__half> w(static_cast<size_t>(K) * K * 16 * 64, __float2half_rn(0.f));
  const float* W = conv.h_w_raw.data();
  for (int o = 0; o < n_cls; ++o)
    for (int i = 0; i < 64; ++i)
      for (int kh = 0; kh < K; ++kh)
        for (int kw = 0; kw < K; ++kw) {
          double acc = 0.0;
          for (int c = 0; c < 64; ++c) acc += static_cast<double>(wc[o * 64 + c]) * W[((static_cast<size_t>(c) * 64 + i) * K + kh) * K + kw];
          w[((static_cast<size_t>(kw) * K + kh) * 16 + o) * 64 + i] = __float2half_rn(static_cast<float>(acc));
        }
  plan.w_replicas.alloc(w.size() * sizeof(__half));
  SIVO_CUDA(cudaMemcpy(plan.w_replicas.p, w.data(), w.size() * sizeof(__half), cudaMemcpyHostToDevice));
  cuuint64_t dims[3] = {64, static_cast<cuuint64_t>(K) * K * 16, 1};
  cuuint64_t strides[2] = {128, static_cast<cuuint64_t>(K) * K * 16 * 128};
  cuuint32_t box[3] = {64, 16, 1};
  encode(&plan.map_b, plan.w_replicas.p, 3, dims, strides, box);
  std::memset(&plan.cst, 0, sizeof(TcConsts));
  for (int o = 0; o < n_cls; ++o) {
    double acc = bc[o];
    for (int c = 0; c < 64; ++c) acc += static_cast<double>(wc[o * 64 + c]) * conv.h_bias[c];
    plan.cst.bias[o] = static_cast<float>(acc);
  }
  TcParams& p = plan.p;
  p.out_f32 = 1;
  p.n_tile = 16;
  p.cout_total = 16;
  p.out = logits;
  p.w_rep = 1;
  const char* stack_env = std::getenv("SIVO_B200_STACK16");
  if (!(stack_env && stack_env[0] == '0')) {
    conv_tc_use_stack16(plan, K);
  } else {
    p.b_stages = 6;
    plan.nw16 = true;
    plan.smem = 1024 + static_cast<size_t>(9) * kSlotBytes + static_cast<size_t>(p.b_stages) * 3 * 16 * 128 + (2 * 9 + 2 * p.b_stages + 4) * 8 + 16;
  }
  conv_tc_dispatch(plan, nullptr, true);
}

void conv_tc_launch(const ConvTcPlan& plan, const Op& op, cudaStream_t s) {
  (void)op;
  conv_tc_dispatch(plan, s, false);
  SIVO_CUDA(cudaGetLastError());
}

}  // namespace sivo
