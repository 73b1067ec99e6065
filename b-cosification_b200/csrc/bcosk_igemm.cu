// bcosk_igemm.cu -- implicit-GEMM B-cos convolution / linear, forward and explain-dgrad, for sm_100a.
//
//   D[m, n] = sum_k A[m, k] * B[n, k],  fp32 accumulation in TMEM
//     A: NHWC 16-bit activations gathered by TMA *im2col* loads (one [128 pixel x kch channel] box per
//        filter tap / channel chunk, zero fill for padding and tails) into 128B- (or 64B-) swizzled smem
//     B: packed K-major weights, TMA tiled loads
//     MMA: tcgen05.mma.cta_group::1.kind::f16, M=128, N=BN, K=16, issued by one elected thread
//   warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..5 = epilogue (tcgen05.ld).
//   Non-persistent; two CTAs are co-resident per SM (BN <= 128) so one CTA's epilogue overlaps the other's
//   main loop.  Epilogues are documented in include/bcosk.h (struct bcosk_igemm_params).
//   Epilogue I/O (throughput mode): the big per-element tensors move as 128x64 tiles through shared memory with
//   TMA bulk copies - one input tile (residual / producer gain) is prefetched during the main loop, the two output
//   tiles (y + gain, or y + out2) are staged in the drained pipeline slots and written with TMA stores - so the
//   HBM-bound layers keep >100 KB per SM in flight without spending registers or warps on it.
#include <cuda.h>
#include <cstring>

#include "../../include/bcosk.h"
#include "bcosk_common.cuh"
#include "bcosk_host.h"
#include "bcosk_igemm_epi.cuh"

namespace bcosk {

int launch_hp(const bcosk_igemm_params& p, cudaStream_t st);   // bcosk_igemm_hp.cu

constexpr int BM = 128;       // CTA tile M (= UMMA M, one TMEM lane per output pixel)
constexpr int STAGE_K = 64;   // K elements per pipeline stage (128 bytes of 16-bit data per row)
constexpr int A_STAGE_BYTES = BM * STAGE_K * 2;
constexpr int NUM_THREADS = 192;
#ifndef BCOSK_BN128_STAGES
// Ring slots / CTAs per SM of the 128-wide per-tile kernel.  Three CTAs with two 32 KB stages each beat two CTAs with
// three (measured: -0.63 ms of 14.3 per step, every 128-wide launch 4-20 % faster): a tile's load -> MMA -> epilogue ->
// store chain is latency bound, so independent tiles in flight matter more than the depth of one tile's ring.
#define BCOSK_BN128_STAGES 2
#define BCOSK_BN128_BLOCKS 3
#endif
#ifndef BCOSK_LIGHT2_BLOCKS
#define BCOSK_LIGHT2_BLOCKS 4   // CTAs per SM of the single-stage forward variant (5 spills ~200 B per thread)
#endif

// LIGHT: 3 small slots and 3 CTAs per SM - for the bandwidth-bound launches with a short K loop, where what matters is
// how many tiles (i.e. how many bytes) are in flight per SM, not the depth of the MMA pipeline.
// LIGHT = 2: two slots and 4 CTAs per SM for forward launches whose K loop is ONE stage (K = 64).  Slot 0 is the stage and
// afterwards the y tile; slot 1 holds the residual tile and the gain tile is staged over it - every thread reads its own
// residual words before it writes the same words of the gain tile, so the alias is safe.
template <int BN, int LIGHT = 0> struct TileCfg {
  static constexpr int kStages = LIGHT == 2 ? 2 : (LIGHT ? 3 : (BN == 128 ? BCOSK_BN128_STAGES : 4));   // pipeline slots; the last may hold the input tile
  static constexpr int kMinBlocks = LIGHT == 2 ? BCOSK_LIGHT2_BLOCKS : (LIGHT ? 3 : (BN == 128 ? BCOSK_BN128_BLOCKS : 2));
  static constexpr int kBStageBytes = BN * STAGE_K * 2;
  static constexpr int kSlotBytes = A_STAGE_BYTES + kBStageBytes;   // A stage followed by its B stage
  static constexpr int kTileBytes = BM * BN * 2;                    // one 16-bit epilogue tile (BN/64 boxes of 16 KB)
  static constexpr bool kTmaEpilogue = BN == 64 || BN == 128;
  static constexpr int kTmemCols = BN;                              // one fp32 accumulator column per tile column
  static constexpr int kBarOffset = kStages * (A_STAGE_BYTES + kBStageBytes);
  // stages + 1 KB alignment slack + barriers/params
  static constexpr int kSmemBytes = kBarOffset + 1024 + 256 + 2 * BN * 4;
};

// One 32-column slice of one output row: everything after the accumulator is in registers.
// Generic (scalar) form: any scale mode, precision planes, fp32 side tensors.  An out-of-line call, because in the
// kernels it serves only as the fallback of the fast form and would otherwise cost them their register budget; the
// arrays passed by reference live in local memory there.
template <int MODE, typename T>
__device__ __noinline__ void epilogue_chunk_generic(const bcosk_igemm_params& p, const RowInfo& ri, int64_t yrow, float inv_norm,
                                               int64_t add_row, const float* s_alpha, const float* s_beta, int j, int c0,
                                               int ncols, float (&v)[32], float& sq_acc, const EpiTiles& tl, int row) {
  T* y16 = reinterpret_cast<T*>(p.y);
  float* y32 = reinterpret_cast<float*>(p.y);
  if (MODE == BCOSK_MODE_FWD) {
    if (p.lin_bias != nullptr) {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (i < ncols) v[i] += __ldg(p.lin_bias + c0 + i);
    }
    if (p.max_out > 1) {      // MaxOut: n / max_out columns leave this row (per-row stores; see maxout_fwd_tail)
      sq_acc += maxout_fwd_tail<T, 32>(p, v, inv_norm, ri.m, yrow, c0, ncols);
      return;
    }
    float t[32];
    if (p.scale_mode == BCOSK_SCALE_B2) {
#pragma unroll
      for (int i = 0; i < 32; ++i) t[i] = fabsf(v[i]) * inv_norm * s_alpha[j * 32 + i];
    } else if (p.scale_mode == BCOSK_SCALE_POW) {
      const float e = p.b_exp - 1.f;
#pragma unroll
      for (int i = 0; i < 32; ++i) t[i] = __powf(fabsf(v[i]) * inv_norm + 1e-6f, e) * s_alpha[j * 32 + i];
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) t[i] = s_alpha[j * 32 + i];
    }
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = fmaf(v[i], t[i], s_beta[j * 32 + i]);
    if (p.res != nullptr) {
      float r[32];
      if (tl.in != 0) tile_load32<T>(tl.in, row, j, r);
      else load32_planes<T>(reinterpret_cast<const T*>(p.res) + (size_t)ri.m * p.res_ld + c0, p.res_planes,
                            p.res_plane_stride, ncols, r);
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] += r[i];
    }
    uint32_t mbits = 0xffffffffu;
    if (p.relu) {
      mbits = 0;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const bool pos = v[i] > 0.f;
        mbits |= (pos ? 1u : 0u) << i;
        v[i] = pos ? v[i] : 0.f;
        t[i] = pos ? t[i] : 0.f;
      }
    }
    if (p.maskbits != nullptr) p.maskbits[(size_t)ri.m * p.mask_ld + (c0 >> 5)] = mbits;
    if (p.gain != nullptr) {
      if (tl.out2 != 0) {
        tile_store32<T>(tl.out2, row, j, t);
      } else if (p.gain_f32) {
        store32_f32(reinterpret_cast<float*>(p.gain) + (size_t)ri.m * p.gain_ld + c0, ncols, t);
      } else {
        store32_planes<T>(reinterpret_cast<T*>(p.gain) + (size_t)ri.m * p.gain_ld + c0, 1, 0, ncols, t);
      }
    }
    if (tl.out1 != 0) {
      tile_store32<T>(tl.out1, row, j, v);
    } else if (p.y_f32) {
      store32_f32(y32 + (size_t)yrow * p.y_ld + c0, ncols, v);
    } else {
      store32_planes<T>(y16 + (size_t)yrow * p.y_ld + c0, p.y_planes, p.y_plane_stride, ncols, v);
    }
    if (p.sq_out != nullptr) {
#pragma unroll
      for (int i = 0; i < 32; ++i) sq_acc = fmaf(v[i], v[i], sq_acc);  // columns >= n are exact zeros
    }
  } else {
    // ---------------- explain-dgrad epilogue ----------------
    if (add_row >= 0) {
      float a[32];
      load32_planes<T>(reinterpret_cast<const T*>(p.add) + (size_t)add_row * p.add_ld + c0, p.add_planes,
                       p.add_plane_stride, ncols, a);
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] += a[i];
    }
    if (p.out2 != nullptr) {
      float o[32];
      if (p.mul2 != nullptr) {
        if (p.mul2_f32) load32_f32(reinterpret_cast<const float*>(p.mul2) + (size_t)ri.m * p.mul2_ld + c0, ncols, o);
        else load32_planes<T>(reinterpret_cast<const T*>(p.mul2) + (size_t)ri.m * p.mul2_ld + c0, 1, 0, ncols, o);
#pragma unroll
        for (int i = 0; i < 32; ++i) o[i] *= v[i];
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) o[i] = v[i];
      }
      if (p.mask2 != nullptr) {
        const uint32_t mb = __ldg(p.mask2 + (size_t)ri.m * p.mask2_ld + (c0 >> 5));
#pragma unroll
        for (int i = 0; i < 32; ++i) o[i] = ((mb >> i) & 1u) ? o[i] : 0.f;
      }
      if (tl.out2 != 0) tile_store32<T>(tl.out2, row, j, o);
      else store32_planes<T>(reinterpret_cast<T*>(p.out2) + (size_t)ri.m * p.out2_ld + c0, p.out2_planes,
                             p.out2_plane_stride, ncols, o);
    }
    if (p.mul1 != nullptr) {
      float g[32];
      if (tl.in != 0) tile_load32<T>(tl.in, row, j, g);
      else if (p.mul1_f32) load32_f32(reinterpret_cast<const float*>(p.mul1) + (size_t)ri.m * p.mul1_ld + c0, ncols, g);
      else load32_planes<T>(reinterpret_cast<const T*>(p.mul1) + (size_t)ri.m * p.mul1_ld + c0, 1, 0, ncols, g);
      if (p.mul1_sqrt_scale != nullptr) {
#pragma unroll
        for (int i = 0; i < 32; ++i) g[i] = fast_sqrt(g[i] * ri.gscale);
      }
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] *= g[i];
    }
    if (tl.out1 != 0) {
      tile_store32<T>(tl.out1, row, j, v);
    } else if (p.y_f32) {
      store32_f32(y32 + (size_t)yrow * p.y_ld + c0, ncols, v);
    } else {
      store32_planes<T>(y16 + (size_t)yrow * p.y_ld + c0, p.y_planes, p.y_plane_stride, ncols, v);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Fast form for the throughput mode (single 16-bit plane, B=2 or no scale): the math runs on float2 pairs with the
// sm_100 packed-fp32 instructions (FMUL2 / FFMA2 / FADD2), ReLU and the gain mask are applied on the packed 16-bit
// words, per-channel vectors are read with 128-bit shared loads.  ~3x fewer instructions than the generic form -
// the epilogue, not HBM, was the limiter of the bandwidth-bound layers (profiles/r01_*).
// ---------------------------------------------------------------------------------------------
template <typename T> struct Pk;
template <> struct Pk<__nv_bfloat16> {
  static __device__ __forceinline__ uint32_t gt0_mask(uint32_t w) {
    return __hgt2_mask(*reinterpret_cast<__nv_bfloat162*>(&w), __floats2bfloat162_rn(0.f, 0.f));
  }
};
template <> struct Pk<__half> {
  static __device__ __forceinline__ uint32_t gt0_mask(uint32_t w) {
    return __hgt2_mask(*reinterpret_cast<__half2*>(&w), __floats2half2_rn(0.f, 0.f));
  }
};

__device__ __forceinline__ void tile_load_words(uint32_t tile, int r, int j, uint32_t (&w)[16]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const uint4 u = lds128(tile_ptr(tile, r, j, g));
    w[g * 4 + 0] = u.x; w[g * 4 + 1] = u.y; w[g * 4 + 2] = u.z; w[g * 4 + 3] = u.w;
  }
}
__device__ __forceinline__ void tile_store_words(uint32_t tile, int r, int j, const uint32_t (&w)[16]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) sts128(tile_ptr(tile, r, j, g), make_uint4(w[g * 4], w[g * 4 + 1], w[g * 4 + 2], w[g * 4 + 3]));
}
__device__ __forceinline__ void global_load_words(const void* ptr, int ncols, uint32_t (&w)[16]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    uint4 u = make_uint4(0, 0, 0, 0);
    if (g * 8 < ncols) u = __ldg(reinterpret_cast<const uint4*>(ptr) + g);
    w[g * 4 + 0] = u.x; w[g * 4 + 1] = u.y; w[g * 4 + 2] = u.z; w[g * 4 + 3] = u.w;
  }
}
__device__ __forceinline__ void global_store_words(void* ptr, int ncols, const uint32_t (&w)[16]) {
#pragma unroll
  for (int g = 0; g < 4; ++g)
    if (g * 8 < ncols) reinterpret_cast<uint4*>(ptr)[g] = make_uint4(w[g * 4], w[g * 4 + 1], w[g * 4 + 2], w[g * 4 + 3]);
}

// Forward, B=2 scale: branch-free over the 16 column pairs so the compiler can interleave them (all launch-uniform
// options are folded into data: a zero residual word, an all-ones ReLU mask, ...).
template <typename T, bool MASK, bool AFFINE, int ACT = 0>
__device__ __forceinline__ void epilogue_fwd_fast(const bcosk_igemm_params& p, const RowInfo& ri, int64_t yrow,
                                                  float inv_norm, const float* s_alpha, const float* s_beta, int j, int c0,
                                                  int ncols, const float (&v)[32], float& sq_acc, const EpiTiles& tl, int row) {
  uint32_t yw[16], tw[16], rw[16];
  if (p.res != nullptr) {
    if (tl.in != 0) tile_load_words(tl.in, row, j, rw);
    else global_load_words(reinterpret_cast<const T*>(p.res) + (size_t)ri.m * p.res_ld + c0, ncols, rw);
  } else {
#pragma unroll
    for (int k = 0; k < 16; ++k) rw[k] = 0u;
  }
  const uint32_t a4 = smem_u32(s_alpha + j * 32), b4 = smem_u32(s_beta + j * 32);
  const float2 inv2 = make_float2(inv_norm, inv_norm);
  const uint32_t relu_off = p.relu ? 0u : 0xffffffffu;
  const bool plain = p.scale_mode == BCOSK_SCALE_NONE;       // plain linear map (the ViT's to_qkv): the multiplier is alpha alone
  float2 sq2 = make_float2(0.f, 0.f);
  uint32_t mbits = 0;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    float4 al = make_float4(1.f, 1.f, 1.f, 1.f), be = make_float4(0.f, 0.f, 0.f, 0.f);
    if (AFFINE) {
      al = lds_f4(a4 + q * 16);
      be = lds_f4(b4 + q * 16);
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int k = q * 2 + h;  // pair index: columns 2k, 2k+1
      const float2 vv = make_float2(v[2 * k], v[2 * k + 1]);
      float2 t, y;
      if (AFFINE) {
        const float2 kk = __fmul2_rn(h ? make_float2(al.z, al.w) : make_float2(al.x, al.y), inv2);
        t = make_float2(fabsf(vv.x) * kk.x, fabsf(vv.y) * kk.y);                   // |lin| / ||patch|| * alpha
        if (plain) t = h ? make_float2(al.z, al.w) : make_float2(al.x, al.y);
        y = __ffma2_rn(vv, t, h ? make_float2(be.z, be.w) : make_float2(be.x, be.y));
        y = __fadd2_rn(y, Cvt<T>::unpack2(rw[k]));
      } else {
        // the plan folded sqrt(BN multiplier) into the weights: nothing per channel is left
        t = plain ? make_float2(1.f, 1.f) : make_float2(fabsf(vv.x) * inv_norm, fabsf(vv.y) * inv_norm);
        y = __ffma2_rn(vv, t, Cvt<T>::unpack2(rw[k]));
      }
      if (ACT == 1) {      // MyGELU behind the transform: gate = Phi(y), detached in the explanation pass (folded into the gain)
        const float2 gate = make_float2(0.5f * (1.0f + erff(y.x * 0.70710678118654752440f)),
                                        0.5f * (1.0f + erff(y.y * 0.70710678118654752440f)));
        y = __fmul2_rn(y, gate);
        t = __fmul2_rn(t, gate);
      } else if (ACT == 2) {   // QuickGELU y sigmoid(1.702 y), NOT detached (CLIP/clip/model.py:166-168): the gain takes its derivative
        const float2 sg = make_float2(1.0f / (1.0f + expf(-1.702f * y.x)), 1.0f / (1.0f + expf(-1.702f * y.y)));
        t = __fmul2_rn(t, make_float2(sg.x + 1.702f * y.x * sg.x * (1.0f - sg.x), sg.y + 1.702f * y.y * sg.y * (1.0f - sg.y)));
        y = __fmul2_rn(y, sg);
      }
      const uint32_t ywk = Cvt<T>::pack2(y.x, y.y);
      const uint32_t m = Pk<T>::gt0_mask(ywk) | relu_off;                          // 0xFFFF per kept half
      yw[k] = ywk & m;
      tw[k] = Cvt<T>::pack2(t.x, t.y) & m;
#ifndef BCOSK_EXP_SKIP
      if (MASK) mbits |= ((m & 1u) | ((m >> 15) & 2u)) << (2 * k);
      const float2 ym = Cvt<T>::unpack2(yw[k]);                                    // what the consumer will read
      sq2 = __ffma2_rn(ym, ym, sq2);
#endif
    }
  }
  if (MASK) p.maskbits[(size_t)ri.m * p.mask_ld + (c0 >> 5)] = mbits;
  if (p.gain != nullptr) {
    if (tl.out2 != 0) tile_store_words(tl.out2, row, j, tw);
    else global_store_words(reinterpret_cast<T*>(p.gain) + (size_t)ri.m * p.gain_ld + c0, ncols, tw);
  }
  if (tl.out1 != 0) tile_store_words(tl.out1, row, j, yw);
  else global_store_words(reinterpret_cast<T*>(p.y) + (size_t)yrow * p.y_ld + c0, ncols, yw);
  sq_acc += sq2.x + sq2.y;
}

template <typename T>
__device__ __forceinline__ void epilogue_explain_fast(const bcosk_igemm_params& p, const RowInfo& ri, int64_t yrow,
                                                      int64_t add_row, int j, int c0, int ncols, float (&v)[32],
                                                      const EpiTiles& tl, int row, uint32_t mb) {
  uint32_t w[16];
  if (add_row >= 0) {
    if (tl.in2 != 0) tile_load_words(tl.in2, row, j, w);
    else global_load_words(reinterpret_cast<const T*>(p.add) + (size_t)add_row * p.add_ld + c0, ncols, w);
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float2 a = __fadd2_rn(make_float2(v[2 * k], v[2 * k + 1]), Cvt<T>::unpack2(w[k]));
      v[2 * k] = a.x;
      v[2 * k + 1] = a.y;
    }
  }
  if (p.out2 != nullptr) {
    uint32_t ow[16];
    if (p.mul2 != nullptr) {
      global_load_words(reinterpret_cast<const T*>(p.mul2) + (size_t)ri.m * p.mul2_ld + c0, ncols, w);
    } else {
      const uint32_t one2 = Cvt<T>::pack2(1.f, 1.f);
#pragma unroll
      for (int k = 0; k < 16; ++k) w[k] = one2;
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float2 o = __fmul2_rn(make_float2(v[2 * k], v[2 * k + 1]), Cvt<T>::unpack2(w[k]));
      // bit 2k -> low half, bit 2k+1 -> high half of an AND mask for the packed word
      const uint32_t sel = ((mb >> (2 * k)) & 1u) * 0xffffu + ((mb >> (2 * k + 1)) & 1u) * 0xffff0000u;
      ow[k] = Cvt<T>::pack2(o.x, o.y) & sel;
    }
    if (tl.out2 != 0) tile_store_words(tl.out2, row, j, ow);
    else global_store_words(reinterpret_cast<T*>(p.out2) + (size_t)ri.m * p.out2_ld + c0, ncols, ow);
  }
  if (p.mul1 != nullptr) {
    if (tl.in != 0) tile_load_words(tl.in, row, j, w);
    else global_load_words(reinterpret_cast<const T*>(p.mul1) + (size_t)ri.m * p.mul1_ld + c0, ncols, w);
    if (p.mul1_sqrt_scale != nullptr) {
      // mul1 holds the producer's ReLU output: gain = sqrt(y / ||patch||)
      const float2 s2 = make_float2(ri.gscale, ri.gscale);
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const float2 ys = __fmul2_rn(Cvt<T>::unpack2(w[k]), s2);
        v[2 * k] *= fast_sqrt(ys.x);
        v[2 * k + 1] *= fast_sqrt(ys.y);
      }
    } else {
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const float2 g = __fmul2_rn(make_float2(v[2 * k], v[2 * k + 1]), Cvt<T>::unpack2(w[k]));
        v[2 * k] = g.x;
        v[2 * k + 1] = g.y;
      }
    }
  }
  if (p.y_f32) {
    store32_f32(reinterpret_cast<float*>(p.y) + (size_t)yrow * p.y_ld + c0, ncols, v);
  } else {
    uint32_t yw[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) yw[k] = Cvt<T>::pack2(v[2 * k], v[2 * k + 1]);
    if (tl.out1 != 0) tile_store_words(tl.out1, row, j, yw);
    else global_store_words(reinterpret_cast<T*>(p.y) + (size_t)yrow * p.y_ld + c0, ncols, yw);
  }
}

template <int MODE, typename T>
__device__ __forceinline__ void epilogue_chunk_fast(const bcosk_igemm_params& p, const RowInfo& ri, int64_t yrow,
                                                    float inv_norm, int64_t add_row, const float* s_alpha,
                                                    const float* s_beta, int j, int c0, int ncols, float (&v)[32],
                                                    float& sq_acc, const EpiTiles& tl, int row, uint32_t mb) {
  if (MODE == BCOSK_MODE_FWD) {
    const bool affine = p.alpha != nullptr || p.beta != nullptr;
    if (p.act == 1) {          // (validated: no mask bits, no ReLU)
      if (affine) epilogue_fwd_fast<T, false, true, 1>(p, ri, yrow, inv_norm, s_alpha, s_beta, j, c0, ncols, v, sq_acc, tl, row);
      else epilogue_fwd_fast<T, false, false, 1>(p, ri, yrow, inv_norm, s_alpha, s_beta, j, c0, ncols, v, sq_acc, tl, row);
    } else if (p.act == 2) {
      if (affine) epilogue_fwd_fast<T, false, true, 2>(p, ri, yrow, inv_norm, s_alpha, s_beta, j, c0, ncols, v, sq_acc, tl, row);
      else epilogue_fwd_fast<T, false, false, 2>(p, ri, yrow, inv_norm, s_alpha, s_beta, j, c0, ncols, v, sq_acc, tl, row);
    } else if (p.maskbits != nullptr) {
      if (affine) epilogue_fwd_fast<T, true, true>(p, ri, yrow, inv_norm, s_alpha, s_beta, j, c0, ncols, v, sq_acc, tl, row);
      else epilogue_fwd_fast<T, true, false>(p, ri, yrow, inv_norm, s_alpha, s_beta, j, c0, ncols, v, sq_acc, tl, row);
    } else {
      if (affine) epilogue_fwd_fast<T, false, true>(p, ri, yrow, inv_norm, s_alpha, s_beta, j, c0, ncols, v, sq_acc, tl, row);
      else epilogue_fwd_fast<T, false, false>(p, ri, yrow, inv_norm, s_alpha, s_beta, j, c0, ncols, v, sq_acc, tl, row);
    }
  } else {
    epilogue_explain_fast<T>(p, ri, yrow, add_row, j, c0, ncols, v, tl, row, mb);
  }
}

// register-resident select of a[j] for a small compile-time sized array (avoids a local-memory array)
template <int N>
__device__ __forceinline__ uint32_t pick_word(const uint32_t (&a)[N], int j) {
  uint32_t r = a[0];
#pragma unroll
  for (int i = 1; i < N; ++i) r = (j == i) ? a[i] : r;
  return r;
}

// eligibility of the fast form (uniform over the launch)
template <int MODE>
__device__ __forceinline__ bool epilogue_fast_ok(const bcosk_igemm_params& p) {
  if (MODE == BCOSK_MODE_FWD)
    return !p.y_f32 && p.y_planes == 1 && (p.gain == nullptr || !p.gain_f32) && (p.res == nullptr || p.res_planes == 1) &&
           (p.scale_mode == BCOSK_SCALE_B2 || p.scale_mode == BCOSK_SCALE_NONE) && p.lin_bias == nullptr && p.max_out <= 1;
  return (p.y_f32 || p.y_planes == 1) && (p.add == nullptr || p.add_planes == 1) && (p.mul1 == nullptr || !p.mul1_f32) &&
         (p.out2 == nullptr || p.out2_planes == 1) && (p.mul2 == nullptr || !p.mul2_f32);
}

template <int MODE, typename T>
__device__ __forceinline__ void epilogue_chunk(const bcosk_igemm_params& p, const RowInfo& ri, int64_t yrow, float inv_norm,
                                               int64_t add_row, const float* s_alpha, const float* s_beta, int j, int c0,
                                               int ncols, float (&v)[32], float& sq_acc, const EpiTiles& tl, int row,
                                               bool fast, uint32_t mb) {
  if (fast) {
    epilogue_chunk_fast<MODE, T>(p, ri, yrow, inv_norm, add_row, s_alpha, s_beta, j, c0, ncols, v, sq_acc, tl, row, mb);
  } else {
    // the generic form is an out-of-line call: give it its own copies so that `v` stays in registers on the fast path
    float vv[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) vv[i] = v[i];
    float sq_local = sq_acc;
    const RowInfo ri_copy = ri;
    const EpiTiles tl_copy = tl;
    epilogue_chunk_generic<MODE, T>(p, ri_copy, yrow, inv_norm, add_row, s_alpha, s_beta, j, c0, ncols, vv, sq_local, tl_copy,
                                    row);
    sq_acc = sq_local;
  }
}

template <int BN, int MODE, typename T, int LIGHT = 0>
__global__ void __launch_bounds__(NUM_THREADS, TileCfg<BN, LIGHT>::kMinBlocks)
bcosk_igemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                   const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_in2,
                   const __grid_constant__ CUtensorMap tmap_out1, const __grid_constant__ CUtensorMap tmap_out2,
                   const __grid_constant__ bcosk_igemm_params p, const IgemmAux aux) {
  using Cfg = TileCfg<BN, LIGHT>;
  constexpr int kSlots = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment required by the 128B swizzle atoms
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // slot s = [A stage 16 KB | B stage BN*128 B]; after the main loop slots 0/1 hold the output tiles, and when an
  // epilogue input tile is prefetched it owns the last slot (the ring then has kSlots-1 stages)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::kBarOffset);
  uint64_t* empty_bar = full_bar + kSlots;
  uint64_t* tmem_full_bar = empty_bar + kSlots;    // accumulator complete
  uint64_t* in_bar = tmem_full_bar + 1;            // epilogue input tile landed
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(in_bar + 1);
  float* s_alpha = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);
  float* s_beta = s_alpha + BN;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_tiles = (p.n + BN - 1) / BN;
  const int tile = blockIdx.x;
  const int tile_n = tile % n_tiles;
  const int tile_m = tile / n_tiles;
  const int M = p.a_nb * p.op * p.oq;
  const int m0 = tile_m * BM;
  const int n0 = tile_n * BN;

  const int chunks_per_stage = STAGE_K / p.kch;  // 1 (kch = 64) or 2 (kch = 32)
  const int total_chunks = p.num_segs * p.num_taps * p.chunks_per_tap;
  const int num_iters = total_chunks / chunks_per_stage;  // host guarantees divisibility
  const bool use_in_tile = Cfg::kTmaEpilogue && aux.tma_in != 0;
  const bool use_in2_tile = use_in_tile && aux.tma_in2 != 0;   // host guarantees >= 2 ring stages remain
  const bool late_in = use_in_tile && !use_in2_tile && aux.late_in != 0;
  const int num_stages = kSlots - ((use_in_tile && !late_in) ? 1 : 0) - (use_in2_tile ? 1 : 0);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < kSlots; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    mbar_init(in_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      if (use_in_tile && !late_in) {
        // residual (forward) / producer gain (explain): whole 128 x BN tile, lands while the main loop runs
        uint8_t* dst = smem + (kSlots - 1) * Cfg::kSlotBytes;
        mbar_arrive_expect_tx(in_bar, Cfg::kTileBytes * (use_in2_tile ? 2 : 1));
        for (int b = 0; b < BN / 64; ++b) tma_load_2d(dst + b * 16384, &tmap_in, in_bar, n0 + b * 64, m0);
        if (use_in2_tile) {
          uint8_t* dst2 = smem + (kSlots - 2) * Cfg::kSlotBytes;
          for (int b = 0; b < BN / 64; ++b) tma_load_2d(dst2 + b * 16384, &tmap_in2, in_bar, n0 + b * 64, m0);
        }
      }
      // first output pixel of this tile -> im2col base coordinates
      const int opq = p.op * p.oq;
      const int img = m0 / opq;
      const int rem = m0 - img * opq;
      const int pp = rem / p.oq;
      const int qq = rem - pp * p.oq;
      const int base_w = p.lo_w + qq * p.stride_w;
      const int base_h = p.lo_h + pp * p.stride_h;
      const uint32_t a_chunk_bytes = BM * p.kch * 2;
      const uint32_t b_chunk_bytes = BN * p.kch * 2;
      int stage = 0;
      uint32_t phase = 0;
      int seg = 0, tap = 0, kc = 0;
      for (int it = 0; it < num_iters; ++it) {
        uint8_t* slot = smem + stage * Cfg::kSlotBytes;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        mbar_arrive_expect_tx(&full_bar[stage], Cfg::kSlotBytes);
        for (int j = 0; j < chunks_per_stage; ++j) {
          const int ci = it * chunks_per_stage + j;
          tma_load_im2col_4d(slot + j * a_chunk_bytes, &tmap_a, &full_bar[stage], p.seg_a_choff[seg] + kc * p.kch, base_w,
                             base_h, img, p.tap_off_w[tap], p.tap_off_h[tap]);
          tma_load_2d(slot + A_STAGE_BYTES + j * b_chunk_bytes, &tmap_b, &full_bar[stage], ci * p.kch, n0);
          if (++kc == p.chunks_per_tap) {
            kc = 0;
            if (++tap == p.num_taps) { tap = 0; ++seg; }
          }
        }
        if (++stage == num_stages) { stage = 0; phase ^= 1; }
      }
      if (late_in) {
        // the last slot's final stage has been consumed -> it now takes the epilogue input tile
        while (stage != kSlots - 1) {
          if (++stage == num_stages) { stage = 0; phase ^= 1; }
        }
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* dst = smem + (kSlots - 1) * Cfg::kSlotBytes;
        mbar_arrive_expect_tx(in_bar, Cfg::kTileBytes);
        for (int b = 0; b < BN / 64; ++b) tma_load_2d(dst + b * 16384, &tmap_in, in_bar, n0 + b * 64, m0);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_f16((uint32_t)p.dtype, BM, BN);
      const uint32_t row_bytes = p.kch * 2;
      const uint32_t a_chunk_bytes = BM * p.kch * 2;
      const uint32_t b_chunk_bytes = BN * p.kch * 2;
      const int mma_per_chunk = p.kch / 16;
      const uint64_t da_stage0 = umma_smem_desc_kmajor(smem_u32(smem), 128);
      const uint64_t slot16 = Cfg::kSlotBytes >> 4;
      int stage = 0;
      uint32_t phase = 0;
      uint32_t accumulate = 0;
      for (int it = 0; it < num_iters; ++it) {
        uint8_t* slot = smem + stage * Cfg::kSlotBytes;
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (chunks_per_stage == 1) {
          // 64-channel chunks: four K steps per stage, descriptors differ by constants only (the issuing thread must
          // stay below the 64 cycles a 128 x 128 x 16 MMA takes; the generic loop below costs ~170 per MMA)
          const uint64_t da = da_stage0 + (uint64_t)stage * slot16;
          const uint64_t db = da + (A_STAGE_BYTES >> 4);
          umma_f16(tmem_base, da, db, idesc, accumulate);
          umma_f16(tmem_base, da + 2, db + 2, idesc, 1);
          umma_f16(tmem_base, da + 4, db + 4, idesc, 1);
          umma_f16(tmem_base, da + 6, db + 6, idesc, 1);
          accumulate = 1;
        } else {
          for (int j = 0; j < chunks_per_stage; ++j) {
            const uint64_t da = umma_smem_desc_kmajor(smem_u32(slot + j * a_chunk_bytes), row_bytes);
            const uint64_t db = umma_smem_desc_kmajor(smem_u32(slot + A_STAGE_BYTES + j * b_chunk_bytes), row_bytes);
            for (int k = 0; k < mma_per_chunk; ++k) {
              // advance 16 K-elements = 32 bytes inside the swizzle atom: +2 in the (addr >> 4) field
              umma_f16(tmem_base, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, accumulate);
              accumulate = 1;
            }
          }
        }
        umma_commit(&empty_bar[stage]);   // frees the smem slot once these MMAs have read it
        if (++stage == num_stages) { stage = 0; phase ^= 1; }
      }
      umma_commit(tmem_full_bar);  // accumulator complete
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    const int quad = warp & 3;  // TMEM lane quadrant this warp may read
    const int row = quad * 32 + lane;
    const int et = (warp - 2) * 32 + lane;  // 0..127
    // stage per-channel vectors while the main loop runs
    if (MODE == BCOSK_MODE_FWD) {
      for (int i = et; i < BN; i += 128) {
        const int c = n0 + i;
        s_alpha[i] = (p.alpha != nullptr && c < p.n) ? __ldg(p.alpha + c) : 1.f;
        s_beta[i] = (p.beta != nullptr && c < p.n) ? __ldg(p.beta + c) : 0.f;
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
    }
    RowInfo ri;
    ri.m = m0 + row;
    ri.valid = ri.m < M;
    {
      const int opq = p.op * p.oq;
      const int mm = ri.valid ? ri.m : 0;
      ri.img = mm / opq;
      const int rem = mm - ri.img * opq;
      ri.p = rem / p.oq;
      ri.q = rem - ri.p * p.oq;
    }
    const int64_t yrow = p.os_0 + (int64_t)ri.img * p.os_n + (int64_t)ri.p * p.os_p + (int64_t)ri.q * p.os_q;
    if (MODE == BCOSK_MODE_EXPLAIN && p.side_mapped) ri.m = (int)yrow;   // side tensors follow the mapped output row
    ri.gscale = (MODE == BCOSK_MODE_EXPLAIN && p.mul1_sqrt_scale != nullptr && ri.valid) ? __ldg(p.mul1_sqrt_scale + ri.m) : 1.f;
    float inv_norm = 1.f;
    int64_t add_row = -1;
    if (MODE == BCOSK_MODE_FWD) {
      if (p.scale_mode != BCOSK_SCALE_NONE && ri.valid) {
        if (p.inv_norm != nullptr) {
          inv_norm = __ldg(p.inv_norm + ri.m);
        } else {
          // patch norm from the producer's per-pixel sums of squares (reference calc_patch_norms, bcosconv2d.py:196-231)
          const size_t part_stride = (size_t)p.a_nb * p.sq_h * p.sq_w;
          float acc = 0.f;
          for (int dy = 0; dy < p.sq_k; ++dy) {
            const int yy = ri.p * p.sq_stride - p.sq_pad + dy;
            if (yy < 0 || yy >= p.sq_h) continue;
            for (int dx = 0; dx < p.sq_k; ++dx) {
              const int xx = ri.q * p.sq_stride - p.sq_pad + dx;
              if (xx < 0 || xx >= p.sq_w) continue;
              const size_t o = ((size_t)ri.img * p.sq_h + yy) * p.sq_w + xx;
              for (int t = 0; t < p.sq_parts; ++t) acc += __ldg(p.sq_in + t * part_stride + o);
            }
          }
          inv_norm = 1.0f / (sqrtf(acc + p.sq_eps_in) + p.sq_eps_out);
        }
      }
    } else {
      if (p.add != nullptr && ri.valid) {
        const int s = p.add_stride;
        if (ri.p % s == 0 && ri.q % s == 0 && ri.p / s < p.add_p && ri.q / s < p.add_q)
          add_row = ((int64_t)ri.img * p.add_p + ri.p / s) * p.add_q + ri.q / s;
      }
    }
    float sq_acc = 0.f;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    EpiTiles tl;
    tl.in = use_in_tile ? smem_u32(smem + (kSlots - 1) * Cfg::kSlotBytes) : 0u;
    tl.in2 = use_in2_tile ? smem_u32(smem + (kSlots - 2) * Cfg::kSlotBytes) : 0u;
    // two-slot rings: the input tile shares slot 1 with an output tile.  Forward reads the residual before it writes the
    // gain (out2 in slot 1); explain writes out2 BEFORE it reads the producer gain, so there y (out1) takes slot 1 - it is
    // written after the gain words of the same thread were read - and out2 goes to slot 0.
    constexpr bool kSwapOut = MODE == BCOSK_MODE_EXPLAIN && kSlots == 2;
    tl.out1 = (Cfg::kTmaEpilogue && aux.tma_out1) ? smem_u32(smem + (kSwapOut ? Cfg::kSlotBytes : 0)) : 0u;
    tl.out2 = (Cfg::kTmaEpilogue && aux.tma_out2) ? smem_u32(smem + (kSwapOut ? 0 : Cfg::kSlotBytes)) : 0u;

    const bool fast = epilogue_fast_ok<MODE>(p);
    // explain: the previous block's ReLU mask words of this row (one per 32 columns), fetched before any waiting
    uint32_t mb_pre[BN / 32];
#pragma unroll
    for (int j = 0; j < BN / 32; ++j) {
      mb_pre[j] = 0xffffffffu;
      if (MODE == BCOSK_MODE_EXPLAIN && p.mask2 != nullptr && ri.valid && n0 + j * 32 < p.n)
        mb_pre[j] = __ldg(p.mask2 + (size_t)ri.m * p.mask2_ld + ((n0 + j * 32) >> 5));
    }
    if (use_in_tile) mbar_wait(in_bar, 0);
    mbar_wait(tmem_full_bar, 0);  // all MMAs done: accumulator complete AND every pipeline slot is drained
    tc_fence_after();
#pragma unroll 1
    for (int j = 0; j < BN / 32; ++j) {
      const int c0 = n0 + j * 32;
      if (c0 >= p.n) break;  // warp-uniform
      uint32_t raw[32];
      tmem_ld_32x32(tmem_base + lane_base + (uint32_t)(j * 32), raw);
      tmem_ld_wait();
      if (!ri.valid) continue;
      float v[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(raw[i]);
      epilogue_chunk<MODE, T>(p, ri, yrow, inv_norm, add_row, s_alpha, s_beta, j, c0, min(32, p.n - c0), v, sq_acc, tl,
                              row, fast, pick_word<BN / 32>(mb_pre, j));
    }
    if (tl.out1 != 0 || tl.out2 != 0) {
      // generic-proxy smem writes -> visible to the async proxy, then one thread issues the bulk tensor stores
      fence_proxy_async_smem();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (et == 0) {
        for (int b = 0; b < BN / 64; ++b) {
          const int c = n0 + b * 64;
          if (c >= p.n) break;
          if (tl.out1 != 0) tma_store_2d_addr(&tmap_out1, tl.out1 + b * 16384, c, m0);
          if (tl.out2 != 0) tma_store_2d_addr(&tmap_out2, tl.out2 + b * 16384, c, m0);
        }
        tma_store_commit_and_wait_read();
      }
    }
    if (MODE == BCOSK_MODE_FWD) {
      if (p.sq_out != nullptr && ri.valid) p.sq_out[(size_t)tile_n * M + ri.m] = sq_acc;
      if (p.inv_norm_out != nullptr && tile_n == 0 && ri.valid && warp >= 2) p.inv_norm_out[ri.m] = inv_norm;
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// =================================================================================================
// Persistent variant for the bandwidth-bound launches (64-wide tiles, short K loop): one CTA per SM walks tiles
// t = blockIdx.x, +gridDim.x, ...  Everything a tile needs is prefetched by dedicated warps while the previous tile is
// still in its epilogue, so the SM always has loads, math and stores of different tiles in flight:
//   warp 0  A/B TMA producer (3-slot ring, runs ahead across tiles)
//   warp 1  TMEM allocator + MMA issuer, two accumulator buffers (tile i -> buffer i&1)
//   warp 2  epilogue-input producer: residual / producer-gain tile and the extra-gradient tile, double buffered
//   warp 3  row-side producer: 1/||patch|| per row (forward) or the ReLU-mask words (explain) + per-channel vectors
//   warps 4..11  epilogue: warp w reads TMEM lane quadrant w%4, columns 32*((w-4)/4) .., and stages the two output
//                tiles in shared memory (double buffered); one thread issues the TMA stores of tile i, whose
//                shared-memory reads overlap the math of tile i+1.  One named barrier per tile.
// =================================================================================================
// i-th tile of this CTA, or -1 past the end.  order 1 keeps the n tiles of a row block on one CTA back to back, so the
// 128-byte segments of each output row reach L2 together and the A tile is fetched once.
__device__ __forceinline__ int persist_tile(int i, int n_tiles, int m_tiles, int order) {
  if (order == 0) {
    const int t = blockIdx.x + i * gridDim.x;
    return t < m_tiles * n_tiles ? t : -1;
  }
  const int g = blockIdx.x + (i / n_tiles) * gridDim.x;
  return g < m_tiles ? g * n_tiles + i % n_tiles : -1;
}

constexpr int P_THREADS = 384;
constexpr int P_EPI_THREADS = 256;
constexpr int P_BN = 64;

struct PersistCfg {
  static constexpr int kSlots = 3;
  static constexpr int kBStageBytes = P_BN * STAGE_K * 2;
  static constexpr int kSlotBytes = A_STAGE_BYTES + kBStageBytes;        // 24 KB
  static constexpr int kTileBytes = BM * P_BN * 2;                       // 16 KB: one 128 x 64 16-bit tile (one TMA box)
  static constexpr int kTmemCols = 2 * P_BN;
  static constexpr int kRingBytes = kSlots * kSlotBytes;                 // 72 KB
  // ring | in[2] | in2[2] | out1[2] | out2[2] | barriers (256 B) | row-side [2][BM] words x2 | alpha/beta [2][2][BN] | sq [2][2][BM]
  static constexpr int kSideWords = 2 * BM * 2 + 2 * 2 * P_BN + 2 * 2 * BM;
  static constexpr int kSmemBytes = kRingBytes + 8 * kTileBytes + 256 + kSideWords * 4;
};

template <int MODE, typename T>
__global__ void __launch_bounds__(P_THREADS, 1)
bcosk_igemm_persistent_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                              const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_in2,
                              const __grid_constant__ CUtensorMap tmap_out1, const __grid_constant__ CUtensorMap tmap_out2,
                              const __grid_constant__ bcosk_igemm_params p, const IgemmAux aux) {
  using Cfg = PersistCfg;
  constexpr int BN = P_BN;
  constexpr int kSlots = Cfg::kSlots;
  extern __shared__ __align__(1024) uint8_t smem_dyn[];
  uint8_t* smem = smem_dyn;   // no static shared memory in this kernel: the dynamic window starts 1024-byte aligned
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint8_t* in_tile = smem + Cfg::kRingBytes;                 // [2][kTileBytes]
  uint8_t* in2_tile = in_tile + 2 * Cfg::kTileBytes;         // [2]
  uint8_t* out1_tile = in2_tile + 2 * Cfg::kTileBytes;       // [2]
  uint8_t* out2_tile = out1_tile + 2 * Cfg::kTileBytes;      // [2]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(out2_tile + 2 * Cfg::kTileBytes);
  uint64_t* empty_bar = full_bar + kSlots;
  uint64_t* acc_full_bar = empty_bar + kSlots;               // [2]
  uint64_t* acc_empty_bar = acc_full_bar + 2;                // [2]
  uint64_t* in_full_bar = acc_empty_bar + 2;                 // [2]
  uint64_t* in_empty_bar = in_full_bar + 2;                  // [2]
  uint64_t* side_full_bar = in_empty_bar + 2;                // [2]
  uint64_t* side_empty_bar = side_full_bar + 2;              // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(side_empty_bar + 2);
  uint32_t* s_side = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(full_bar) + 256);   // [2][BM][2]: inv_norm | mask words
  float* s_ab = reinterpret_cast<float*>(s_side + 2 * BM * 2);                                   // [2][alpha BN | beta BN]
  float* s_sq = s_ab + 2 * 2 * BN;                                                               // [2][2][BM]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_tiles = (p.n + BN - 1) / BN;
  const int M = p.a_nb * p.op * p.oq;
  const int m_tiles = (M + BM - 1) / BM;
  const int chunks_per_stage = STAGE_K / p.kch;
  const int num_iters = (p.num_segs * p.num_taps * p.chunks_per_tap) / chunks_per_stage;
  const bool use_in_tile = aux.tma_in != 0;
  const bool use_in2_tile = use_in_tile && aux.tma_in2 != 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < kSlots; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&acc_full_bar[s], 1);
      mbar_init(&acc_empty_bar[s], 8);   // one arrival per epilogue warp
      mbar_init(&in_full_bar[s], 1);
      mbar_init(&in_empty_bar[s], 8);
      mbar_init(&side_full_bar[s], 1);
      mbar_init(&side_empty_bar[s], 8);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== A/B producer =====================
    if (lane == 0) {
      const int opq = p.op * p.oq;
      const uint32_t a_chunk_bytes = BM * p.kch * 2;
      const uint32_t b_chunk_bytes = BN * p.kch * 2;
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0, t; (t = persist_tile(it, n_tiles, m_tiles, aux.order)) >= 0; ++it) {
        const int m0 = (t / n_tiles) * BM, n0 = (t % n_tiles) * BN;
        const int img = m0 / opq;
        const int rem = m0 - img * opq;
        const int pp = rem / p.oq;
        const int qq = rem - pp * p.oq;
        const int base_w = p.lo_w + qq * p.stride_w;
        const int base_h = p.lo_h + pp * p.stride_h;
        int seg = 0, tap = 0, kc = 0;
        for (int it = 0; it < num_iters; ++it) {
          uint8_t* slot = smem + stage * Cfg::kSlotBytes;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], Cfg::kSlotBytes);
          for (int j = 0; j < chunks_per_stage; ++j) {
            const int ci = it * chunks_per_stage + j;
            tma_load_im2col_4d(slot + j * a_chunk_bytes, &tmap_a, &full_bar[stage], p.seg_a_choff[seg] + kc * p.kch, base_w,
                               base_h, img, p.tap_off_w[tap], p.tap_off_h[tap]);
            tma_load_2d(slot + A_STAGE_BYTES + j * b_chunk_bytes, &tmap_b, &full_bar[stage], ci * p.kch, n0);
            if (++kc == p.chunks_per_tap) {
              kc = 0;
              if (++tap == p.num_taps) { tap = 0; ++seg; }
            }
          }
          if (++stage == kSlots) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_f16((uint32_t)p.dtype, BM, BN);
      const uint32_t row_bytes = p.kch * 2;
      const uint32_t a_chunk_bytes = BM * p.kch * 2;
      const uint32_t b_chunk_bytes = BN * p.kch * 2;
      const int mma_per_chunk = p.kch / 16;
      int stage = 0;
      uint32_t phase = 0;
      uint32_t i = 0;
      for (int t; (t = persist_tile((int)i, n_tiles, m_tiles, aux.order)) >= 0; ++i) {
        const uint32_t buf = i & 1u;
        mbar_wait(&acc_empty_bar[buf], ((i >> 1) & 1u) ^ 1u);   // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + buf * BN;
        uint32_t accumulate = 0;
        for (int it = 0; it < num_iters; ++it) {
          uint8_t* slot = smem + stage * Cfg::kSlotBytes;
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          for (int j = 0; j < chunks_per_stage; ++j) {
            const uint64_t da = umma_smem_desc_kmajor(smem_u32(slot + j * a_chunk_bytes), row_bytes);
            const uint64_t db = umma_smem_desc_kmajor(smem_u32(slot + A_STAGE_BYTES + j * b_chunk_bytes), row_bytes);
            for (int k = 0; k < mma_per_chunk; ++k) {
              umma_f16(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, accumulate);
              accumulate = 1;
            }
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == kSlots) { stage = 0; phase ^= 1; }
        }
        umma_commit(&acc_full_bar[buf]);
      }
    }
  } else if (warp == 2) {
    // ===================== epilogue-input producer =====================
    if (lane == 0 && use_in_tile) {
      uint32_t i = 0;
      for (int t; (t = persist_tile((int)i, n_tiles, m_tiles, aux.order)) >= 0; ++i) {
        const uint32_t buf = i & 1u;
        const int m0 = (t / n_tiles) * BM, n0 = (t % n_tiles) * BN;
        mbar_wait(&in_empty_bar[buf], ((i >> 1) & 1u) ^ 1u);
        mbar_arrive_expect_tx(&in_full_bar[buf], Cfg::kTileBytes * (use_in2_tile ? 2 : 1));
        tma_load_2d(in_tile + buf * Cfg::kTileBytes, &tmap_in, &in_full_bar[buf], n0, m0);
        if (use_in2_tile) tma_load_2d(in2_tile + buf * Cfg::kTileBytes, &tmap_in2, &in_full_bar[buf], n0, m0);
      }
    }
  } else if (warp == 3) {
    // ===================== row-side producer =====================
    uint32_t i = 0;
    const int opq = p.op * p.oq;
    for (int t; (t = persist_tile((int)i, n_tiles, m_tiles, aux.order)) >= 0; ++i) {
      const uint32_t buf = i & 1u;
      const int m0 = (t / n_tiles) * BM, n0 = (t % n_tiles) * BN;
      mbar_wait(&side_empty_bar[buf], ((i >> 1) & 1u) ^ 1u);
      uint32_t* side = s_side + buf * (BM * 2);
      if (MODE == BCOSK_MODE_FWD) {
        // 1/||patch|| for rows lane, lane+32, lane+64, lane+96: the (tap, part) loops are outermost and the four rows
        // innermost, so every step issues four independent loads (one dependent-load round trip per step, not per row)
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        int img_r[4], pp_r[4], qq_r[4];
        bool ok_r[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int m = m0 + lane + 32 * r;
          ok_r[r] = m < M;
          const int mm = ok_r[r] ? m : 0;
          img_r[r] = mm / opq;
          const int rem = mm - img_r[r] * opq;
          pp_r[r] = rem / p.oq;
          qq_r[r] = rem - pp_r[r] * p.oq;
        }
        if (p.scale_mode == BCOSK_SCALE_NONE) {
#pragma unroll
          for (int r = 0; r < 4; ++r) acc[r] = 1.f;
        } else if (p.inv_norm != nullptr) {
#pragma unroll
          for (int r = 0; r < 4; ++r) acc[r] = ok_r[r] ? __ldg(p.inv_norm + m0 + lane + 32 * r) : 1.f;
        } else {
          const size_t part_stride = (size_t)p.a_nb * p.sq_h * p.sq_w;
          for (int dy = 0; dy < p.sq_k; ++dy) {
            for (int dx = 0; dx < p.sq_k; ++dx) {
              size_t off[4];
              bool in_r[4];
#pragma unroll
              for (int r = 0; r < 4; ++r) {
                const int yy = pp_r[r] * p.sq_stride - p.sq_pad + dy;
                const int xx = qq_r[r] * p.sq_stride - p.sq_pad + dx;
                in_r[r] = ok_r[r] && yy >= 0 && yy < p.sq_h && xx >= 0 && xx < p.sq_w;
                off[r] = in_r[r] ? ((size_t)img_r[r] * p.sq_h + yy) * p.sq_w + xx : 0;
              }
              for (int tt = 0; tt < p.sq_parts; ++tt) {
                float x[4];
#pragma unroll
                for (int r = 0; r < 4; ++r) x[r] = in_r[r] ? __ldg(p.sq_in + tt * part_stride + off[r]) : 0.f;
#pragma unroll
                for (int r = 0; r < 4; ++r) acc[r] += x[r];
              }
            }
          }
#pragma unroll
          for (int r = 0; r < 4; ++r) acc[r] = 1.0f / (sqrtf(acc[r] + p.sq_eps_in) + p.sq_eps_out);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          side[(lane + 32 * r) * 2] = __float_as_uint(acc[r]);
          side[(lane + 32 * r) * 2 + 1] = 0xffffffffu;
        }
      } else {
        // ReLU mask words of the previous block for this row's 64 columns
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int m = m0 + lane + 32 * r;
          uint32_t w0 = 0xffffffffu, w1 = 0xffffffffu;
          if (m < M && p.mask2 != nullptr) {
            w0 = __ldg(p.mask2 + (size_t)m * p.mask2_ld + (n0 >> 5));
            w1 = (n0 + 32 < p.n) ? __ldg(p.mask2 + (size_t)m * p.mask2_ld + (n0 >> 5) + 1) : 0u;
          }
          side[(lane + 32 * r) * 2] = w0;
          side[(lane + 32 * r) * 2 + 1] = w1;
        }
      }
      if (MODE == BCOSK_MODE_FWD) {
        float* ab = s_ab + buf * (2 * BN);
        for (int c = lane; c < BN; c += 32) {
          const int cc = n0 + c;
          ab[c] = (p.alpha != nullptr && cc < p.n) ? __ldg(p.alpha + cc) : 1.f;
          ab[BN + c] = (p.beta != nullptr && cc < p.n) ? __ldg(p.beta + cc) : 0.f;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&side_full_bar[buf]);
    }
  } else {
    // ===================== epilogue (warps 4..11) =====================
    const int quad = warp & 3;
    const int half = (warp - 4) >> 2;                  // 32-column half of the tile handled by this warp
    const int row = quad * 32 + lane;
    const int et = threadIdx.x - 128;                  // 0..255
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const bool any_out_tile = aux.tma_out1 || aux.tma_out2;
    const bool fast = epilogue_fast_ok<MODE>(p);
    const bool want_sq = MODE == BCOSK_MODE_FWD && p.sq_out != nullptr;
    const int opq = p.op * p.oq;
    uint32_t i = 0;
    for (int t; (t = persist_tile((int)i, n_tiles, m_tiles, aux.order)) >= 0; ++i) {
      const uint32_t buf = i & 1u;
      const uint32_t par = (i >> 1) & 1u;
      const int tile_n = t % n_tiles;
      const int m0 = (t / n_tiles) * BM, n0 = tile_n * BN;
      RowInfo ri;
      ri.m = m0 + row;
      ri.valid = ri.m < M;
      {
        const int mm = ri.valid ? ri.m : 0;
        ri.img = mm / opq;
        const int rem = mm - ri.img * opq;
        ri.p = rem / p.oq;
        ri.q = rem - ri.p * p.oq;
      }
      const int64_t yrow = p.os_0 + (int64_t)ri.img * p.os_n + (int64_t)ri.p * p.os_p + (int64_t)ri.q * p.os_q;
    if (MODE == BCOSK_MODE_EXPLAIN && p.side_mapped) ri.m = (int)yrow;   // side tensors follow the mapped output row
    ri.gscale = (MODE == BCOSK_MODE_EXPLAIN && p.mul1_sqrt_scale != nullptr && ri.valid) ? __ldg(p.mul1_sqrt_scale + ri.m) : 1.f;
      int64_t add_row = -1;
      if (MODE == BCOSK_MODE_EXPLAIN && p.add != nullptr && ri.valid) {
        const int s = p.add_stride;
        if (ri.p % s == 0 && ri.q % s == 0 && ri.p / s < p.add_p && ri.q / s < p.add_q)
          add_row = ((int64_t)ri.img * p.add_p + ri.p / s) * p.add_q + ri.q / s;
      }
      EpiTiles tl;
      tl.in = use_in_tile ? smem_u32(in_tile + buf * Cfg::kTileBytes) : 0u;
      tl.in2 = use_in2_tile ? smem_u32(in2_tile + buf * Cfg::kTileBytes) : 0u;
      tl.out1 = aux.tma_out1 ? smem_u32(out1_tile + buf * Cfg::kTileBytes) : 0u;
      tl.out2 = aux.tma_out2 ? smem_u32(out2_tile + buf * Cfg::kTileBytes) : 0u;

      mbar_wait(&side_full_bar[buf], par);
      const uint32_t side0 = s_side[buf * (BM * 2) + row * 2];
      const uint32_t side1 = s_side[buf * (BM * 2) + row * 2 + 1];
      const float inv_norm = (MODE == BCOSK_MODE_FWD) ? __uint_as_float(side0) : 1.f;
      const uint32_t mb = (MODE == BCOSK_MODE_EXPLAIN) ? (half ? side1 : side0) : 0xffffffffu;
      if (use_in_tile) mbar_wait(&in_full_bar[buf], par);
      mbar_wait(&acc_full_bar[buf], par);
      tc_fence_after();

      float sq_acc = 0.f;
      const int j = half;                       // chunk index inside the 64-wide tile
      const int c0 = n0 + j * 32;
      if (c0 < p.n) {                           // warp-uniform
        uint32_t raw[32];
        tmem_ld_32x32(tmem_base + lane_base + (uint32_t)(buf * BN + j * 32), raw);
        tmem_ld_wait();
        if (ri.valid) {
          float v[32];
#pragma unroll
          for (int k = 0; k < 32; ++k) v[k] = __uint_as_float(raw[k]);
          epilogue_chunk<MODE, T>(p, ri, yrow, inv_norm, add_row, s_ab + buf * (2 * BN), s_ab + buf * (2 * BN) + BN, j, c0,
                                  min(32, p.n - c0), v, sq_acc, tl, row, fast, mb);
        }
      }
      // accumulator, input tiles and row-side values are consumed: hand the buffers back
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&acc_empty_bar[buf]);
        if (use_in_tile) mbar_arrive(&in_empty_bar[buf]);
        mbar_arrive(&side_empty_bar[buf]);
      }
      if (want_sq) s_sq[(buf * 2 + half) * BM + row] = sq_acc;
      if (any_out_tile) {
        fence_proxy_async_smem();
        // the stores of tile i-1 (other staging buffer) must have read their tiles before tile i+1 overwrites them
        if (et == 0) tma_store_wait_read();
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (any_out_tile && et == 0 && n0 < p.n) {
        if (tl.out1 != 0) tma_store_2d_addr(&tmap_out1, tl.out1, n0, m0);
        if (tl.out2 != 0) tma_store_2d_addr(&tmap_out2, tl.out2, n0, m0);
        tma_store_commit();
      }
      if (want_sq && half == 0 && ri.valid)
        p.sq_out[(size_t)tile_n * M + ri.m] = s_sq[(buf * 2) * BM + row] + s_sq[(buf * 2 + 1) * BM + row];
      if (MODE == BCOSK_MODE_FWD && p.inv_norm_out != nullptr && tile_n == 0 && half == 0 && ri.valid)
        p.inv_norm_out[ri.m] = inv_norm;
    }
    if (any_out_tile && et == 0) tma_store_wait_read();
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// =================================================================================================
// Flat-window variant (bcosk_igemm_params.a_flat): stride-1 k x k gathers over a zero-bordered buffer.
// Persistent, one CTA per SM.  The packed weights stay resident in shared memory, every tile fetches ONE window of
// 128 + max tap offset pixel rows with <= 2 tiled TMA boxes (double buffered) and each tap's MMA reads it through a
// descriptor shifted by (off_h * a_wp + off_w) rows.  Per tile that is ~4x fewer bytes from L2 than one im2col box
// per tap for the 4 x 4 stem (16 boxes), which is what bounded it.
//   warp 0  producer (weights once, then windows)   warp 1  TMEM allocator + MMA issuer (two accumulators)
//   warps 2..  epilogue: one TMEM lane quadrant x 32-column slice each; 16-bit outputs are staged in swizzled tiles
//              and copied out as full 128-byte lines (the tile's rows belong to up to three image rows; positions
//              x >= oq are skipped)
// =================================================================================================
struct FlatGeom {
  int box_rows;    // rows per window box (multiple of 8, <= 256)
  int nbox;        // 1 or 2
  int tiles_img;   // 128-position tiles per image
  int pitch;       // pixels per (padded) row of the flattened positions
  int dense;       // 1: `a` is a plain dense tensor; the zero borders exist only in shared memory (one 4-D TMA box of
                   // `nrows` x `pitch` pixels per tile whose out-of-range pixels are zero filled)
  int nrows;
  int tma_store;   // 1: a tile is a whole number of image rows (128 % pitch == 0): staged outputs leave through clipped
                   // 3-D TMA stores with non-negative start coordinates (one per image row) instead of the copy-out loop
};

template <int BN>
struct FlatCfg {
  static constexpr int kEpiWarps = (BN / 32) * 4;
  static constexpr int kThreads = 64 + kEpiWarps * 32;
  static constexpr int kTileBytes = BM * 128;          // one staged output tile (64 x 16-bit columns)
  static constexpr int kTmemCols = 2 * BN < 32 ? 32 : 2 * BN;
};

template <int BN, int MODE, typename T>
__global__ void __launch_bounds__(FlatCfg<BN>::kThreads, 1)
bcosk_igemm_flat_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                        const __grid_constant__ CUtensorMap tmap_out1, const __grid_constant__ CUtensorMap tmap_out2,
                        const __grid_constant__ bcosk_igemm_params p, const IgemmAux aux, const FlatGeom geo) {
  using Cfg = FlatCfg<BN>;
  extern __shared__ __align__(1024) uint8_t smem_dyn[];
  uint8_t* smem = smem_dyn;
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  const uint32_t row_bytes = (uint32_t)p.kch * 2;
  const uint32_t b_chunk_bytes = BN * row_bytes;
  const uint32_t b_bytes = (uint32_t)p.num_taps * b_chunk_bytes;
  const uint32_t win_bytes = geo.dense ? (uint32_t)geo.nrows * geo.pitch * row_bytes : (uint32_t)geo.nbox * geo.box_rows * row_bytes;
  const bool any_out_tile = aux.tma_out1 || aux.tma_out2;
  uint8_t* s_b = smem;
  uint8_t* s_win = s_b + ((b_bytes + 1023u) & ~1023u);                         // [2][win_bytes], 1024-aligned
  const uint32_t win_stride = (win_bytes + 1023u) & ~1023u;
  uint8_t* s_out = s_win + 2 * win_stride;                                     // [2 bufs][out1 | out2] (if staged)
  uint8_t* s_tail = s_out + (any_out_tile ? 4 * Cfg::kTileBytes : 0);
  uint64_t* b_full_bar = reinterpret_cast<uint64_t*>(s_tail);
  uint64_t* win_full_bar = b_full_bar + 1;      // [2]
  uint64_t* win_empty_bar = win_full_bar + 2;   // [2]
  uint64_t* acc_full_bar = win_empty_bar + 2;   // [2]
  uint64_t* acc_empty_bar = acc_full_bar + 2;   // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(acc_empty_bar + 2);
  float* s_ab = reinterpret_cast<float*>(s_tail + 128);                        // [alpha BN | beta BN]
  float* s_sq = s_ab + 2 * BN;                                                 // [2][BN/32][BM]
  uint32_t* s_aoff = reinterpret_cast<uint32_t*>(s_sq + 2 * (BN / 32) * BM);   // [BCOSK_MAX_TAPS] tap offsets >> 4

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.a_nb * geo.tiles_img;
  const int img_rows = p.a_hp * p.a_wp;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    mbar_init(b_full_bar, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&win_full_bar[s], 1);
      mbar_init(&win_empty_bar[s], 1);
      mbar_init(&acc_full_bar[s], 1);
      mbar_init(&acc_empty_bar[s], Cfg::kEpiWarps);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, Cfg::kTmemCols);
    tmem_relinquish();
    for (int t = lane; t < p.num_taps; t += 32)
      s_aoff[t] = ((uint32_t)(p.tap_off_h[t] * geo.pitch + p.tap_off_w[t]) * row_bytes) >> 4;
  }
  if (MODE == BCOSK_MODE_FWD && warp >= 2) {
    for (int c = threadIdx.x - 64; c < BN; c += Cfg::kEpiWarps * 32) {
      s_ab[c] = (p.alpha != nullptr && c < p.n) ? __ldg(p.alpha + c) : 1.f;
      s_ab[BN + c] = (p.beta != nullptr && c < p.n) ? __ldg(p.beta + c) : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== producer =====================
    if (lane == 0) {
      mbar_arrive_expect_tx(b_full_bar, b_bytes);
      for (int c = 0; c < p.num_taps; ++c) tma_load_2d(s_b + c * b_chunk_bytes, &tmap_b, b_full_bar, c * p.kch, 0);
      uint32_t i = 0;
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++i) {
        const uint32_t buf = i & 1u, par = (i >> 1) & 1u;
        const int img = t / geo.tiles_img;
        const int m0 = (t - img * geo.tiles_img) * BM;
        mbar_wait(&win_empty_bar[buf], par ^ 1u);
        mbar_arrive_expect_tx(&win_full_bar[buf], win_bytes);
        if (geo.dense) {
          // input rows p0 + lo_h .. of this image, pixels lo_w .. lo_w + pitch - 1: borders arrive as zeros
          tma_load_4d(s_win + buf * win_stride, &tmap_a, &win_full_bar[buf], 0, p.lo_w, m0 / geo.pitch + p.lo_h, img);
        } else {
          for (int bx = 0; bx < geo.nbox; ++bx)
            tma_load_2d(s_win + buf * win_stride + bx * geo.box_rows * row_bytes, &tmap_a, &win_full_bar[buf], 0,
                        img * img_rows + m0 + bx * geo.box_rows);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_f16(p.dtype == BCOSK_DTYPE_BF16 ? 1u : 0u, BM, BN);
      const int ksteps = p.kch / 16;
      const uint64_t db0 = umma_smem_desc_kmajor(smem_u32(s_b), row_bytes);
      const uint64_t b_chunk16 = b_chunk_bytes >> 4;
      mbar_wait(b_full_bar, 0);
      uint32_t i = 0;
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++i) {
        const uint32_t buf = i & 1u, par = (i >> 1) & 1u;
        mbar_wait(&acc_empty_bar[buf], par ^ 1u);
        mbar_wait(&win_full_bar[buf], par);
        tc_fence_after();
        // one LDS + two 64-bit adds per tap, then the K steps unrolled: the issuing thread must stay well under the
        // ~48 cycles a 128 x 64 x 16 MMA takes (measured: scripts/exp/mma_rate.cu), a naive loop costs ~240 per MMA
        uint64_t da0 = umma_smem_desc_kmajor(smem_u32(s_win + buf * win_stride), row_bytes);
        if (geo.dense) {
          const int m0 = (t % geo.tiles_img) * BM;
          da0 += ((uint32_t)(m0 % geo.pitch) * row_bytes) >> 4;      // the window starts at the tile's first image row
        }
        uint64_t db = db0;
        const uint32_t tmem_d = tmem_base + buf * BN;
        {
          const uint64_t da = da0 + s_aoff[0];
          umma_f16(tmem_d, da, db, idesc, 0);
          umma_f16(tmem_d, da + 2, db + 2, idesc, 1);
          if (ksteps == 4) {
            umma_f16(tmem_d, da + 4, db + 4, idesc, 1);
            umma_f16(tmem_d, da + 6, db + 6, idesc, 1);
          }
        }
#pragma unroll 1
        for (int tap = 1; tap < p.num_taps; ++tap) {
          const uint64_t da = da0 + s_aoff[tap];
          db += b_chunk16;
          umma_f16(tmem_d, da, db, idesc, 1);
          umma_f16(tmem_d, da + 2, db + 2, idesc, 1);
          if (ksteps == 4) {
            umma_f16(tmem_d, da + 4, db + 4, idesc, 1);
            umma_f16(tmem_d, da + 6, db + 6, idesc, 1);
          }
        }
        umma_commit(&win_empty_bar[buf]);
        umma_commit(&acc_full_bar[buf]);
      }
    }
  } else {
    // ===================== epilogue =====================
    const int quad = warp & 3;
    const int j = (warp - 2) >> 2;                     // 32-column slice of the tile handled by this warp
    const int row = quad * 32 + lane;
    const int et = threadIdx.x - 64;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const bool fast = epilogue_fast_ok<MODE>(p);
    const bool want_sq = MODE == BCOSK_MODE_FWD && p.sq_out != nullptr;
    const int c0 = j * 32;
    uint32_t i = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++i) {
      const uint32_t buf = i & 1u, par = (i >> 1) & 1u;
      const int img = t / geo.tiles_img;
      const int m0 = (t - img * geo.tiles_img) * BM;
      const int mf = m0 + row;                         // flattened position p * a_wp + x
      RowInfo ri;
      ri.img = img;
      ri.p = mf / geo.pitch;
      ri.q = mf - ri.p * geo.pitch;
      ri.valid = ri.p < p.op && ri.q < p.oq;
      ri.m = ri.valid ? (img * p.op + ri.p) * p.oq + ri.q : 0;
      const int64_t yrow = p.os_0 + (int64_t)ri.img * p.os_n + (int64_t)ri.p * p.os_p + (int64_t)ri.q * p.os_q;
    if (MODE == BCOSK_MODE_EXPLAIN && p.side_mapped) ri.m = (int)yrow;   // side tensors follow the mapped output row
    ri.gscale = (MODE == BCOSK_MODE_EXPLAIN && p.mul1_sqrt_scale != nullptr && ri.valid) ? __ldg(p.mul1_sqrt_scale + ri.m) : 1.f;
      float inv_norm = 1.f;
      uint32_t mb = 0xffffffffu;
      int64_t add_row = -1;
      if (ri.valid) {
        if (MODE == BCOSK_MODE_FWD && p.scale_mode != BCOSK_SCALE_NONE) inv_norm = __ldg(p.inv_norm + ri.m);
        if (MODE == BCOSK_MODE_EXPLAIN && p.mask2 != nullptr && c0 < p.n)
          mb = __ldg(p.mask2 + (size_t)ri.m * p.mask2_ld + (c0 >> 5));
        if (MODE == BCOSK_MODE_EXPLAIN && p.add != nullptr) {
          const int s = p.add_stride;
          if (ri.p % s == 0 && ri.q % s == 0 && ri.p / s < p.add_p && ri.q / s < p.add_q)
            add_row = ((int64_t)ri.img * p.add_p + ri.p / s) * p.add_q + ri.q / s;
        }
      }
      EpiTiles tl;
      tl.in = 0u;
      tl.in2 = 0u;
      tl.out1 = aux.tma_out1 ? smem_u32(s_out + (buf * 2) * Cfg::kTileBytes) : 0u;
      tl.out2 = aux.tma_out2 ? smem_u32(s_out + (buf * 2 + 1) * Cfg::kTileBytes) : 0u;

      mbar_wait(&acc_full_bar[buf], par);
      tc_fence_after();
      float sq_acc = 0.f;
      if (c0 < p.n) {
        uint32_t raw[32];
        tmem_ld_32x32(tmem_base + lane_base + (uint32_t)(buf * BN + c0), raw);
        tmem_ld_wait();
        if (ri.valid) {
          float v[32];
#pragma unroll
          for (int k = 0; k < 32; ++k) v[k] = __uint_as_float(raw[k]);
          epilogue_chunk<MODE, T>(p, ri, yrow, inv_norm, add_row, s_ab, s_ab + BN, j, c0, min(32, p.n - c0), v, sq_acc, tl,
                                  row, fast, mb);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty_bar[buf]);
      float* sq_buf = s_sq + buf * (BN / 32) * BM;
      if (want_sq) sq_buf[j * BM + row] = sq_acc;
      if (any_out_tile && geo.tma_store) {
        fence_proxy_async_smem();
        if (et == 0) tma_store_wait_read();           // tile i-1's stores have read the other staging buffer
      }
      asm volatile("bar.sync 1, %0;" ::"n"(Cfg::kEpiWarps * 32) : "memory");
      if (any_out_tile && geo.tma_store) {
        if (et == 0) {
          const int p0 = m0 / geo.pitch;              // the tile starts at x = 0 of image row p0
          for (int k = 0; k < BM / geo.pitch && p0 + k < p.op; ++k) {
            const uint32_t off = (uint32_t)(k * geo.pitch) << 7;
            if (tl.out1 != 0) tma_store_3d_addr(&tmap_out1, tl.out1 + off, 0, 0, img * p.op + p0 + k);
            if (tl.out2 != 0) tma_store_3d_addr(&tmap_out2, tl.out2 + off, 0, 0, img * p.op + p0 + k);
          }
          tma_store_commit();
        }
      } else if (any_out_tile) {
        // copy the staged tiles out: 8 lanes per row write one 128-byte line each, rows at x >= oq are skipped.
        // (TMA stores cannot do this: a tile's rows belong to up to three image rows and a negative start coordinate
        // is an illegal instruction for cp.async.bulk.tensor stores - scripts/exp/tma_store3d.cu.)
        T* y16 = reinterpret_cast<T*>(p.y);
        T* g16 = reinterpret_cast<T*>(MODE == BCOSK_MODE_FWD ? p.gain : p.out2);
        const int g_ld = MODE == BCOSK_MODE_FWD ? p.gain_ld : p.out2_ld;
        for (int it = et; it < BM * 8; it += Cfg::kEpiWarps * 32) {
          const int r = it >> 3, u = it & 7;
          const int mfr = m0 + r;
          const int pr = mfr / geo.pitch;
          const int xr = mfr - pr * geo.pitch;
          if (pr < p.op && xr < p.oq && u * 8 < p.n) {
            const size_t d = (size_t)(img * p.op + pr) * p.oq + xr;
            const uint32_t off = (uint32_t)(r << 7) + (uint32_t)((u ^ (r & 7)) << 4);
            if (tl.out1 != 0) *reinterpret_cast<uint4*>(y16 + d * p.y_ld + u * 8) = lds128(tl.out1 + off);
            if (tl.out2 != 0) *reinterpret_cast<uint4*>(g16 + d * g_ld + u * 8) = lds128(tl.out2 + off);
          }
        }
      }
      if (want_sq && j == 0 && ri.valid) {
        float s = sq_buf[row];
#pragma unroll
        for (int h = 1; h < BN / 32; ++h) s += sq_buf[h * BM + row];
        p.sq_out[ri.m] = s;
      }
      if (MODE == BCOSK_MODE_FWD && p.inv_norm_out != nullptr && j == 0 && ri.valid) p.inv_norm_out[ri.m] = inv_norm;
    }
    if (any_out_tile && geo.tma_store && et == 0) tma_store_wait_read();
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------
// debug: land one A chunk in smem via the im2col tensor map and copy it out de-swizzled
// ---------------------------------------------------------------------------------------------
__global__ void bcosk_debug_a_tile_kernel(const __grid_constant__ CUtensorMap tmap_a,
                                          const __grid_constant__ bcosk_igemm_params p, int tile_m, int chunk,
                                          uint16_t* out) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t bar;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int m0 = tile_m * BM;
    const int opq = p.op * p.oq;
    const int img = m0 / opq, rem = m0 % opq;
    const int pp = rem / p.oq, qq = rem % p.oq;
    const int kc = chunk % p.chunks_per_tap;
    const int t = chunk / p.chunks_per_tap;
    const int tap = t % p.num_taps, seg = t / p.num_taps;
    mbar_arrive_expect_tx(&bar, BM * p.kch * 2);
    tma_load_im2col_4d(smem, &tmap_a, &bar, p.seg_a_choff[seg] + kc * p.kch, p.lo_w + qq * p.stride_w,
                       p.lo_h + pp * p.stride_h, img, p.tap_off_w[tap], p.tap_off_h[tap]);
  }
  mbar_wait(&bar, 0);
  const int row_bytes = p.kch * 2;
  for (int i = threadIdx.x; i < BM * p.kch; i += blockDim.x) {
    const int r = i / p.kch, c = i % p.kch;
    const int u = (c * 2) / 16;  // logical 16-byte unit inside the row
    // Swizzle<3,4,3> (128B rows): unit ^= row % 8;  Swizzle<2,4,3> (64B rows): unit ^= (row / 2) % 4
    const int pu = (row_bytes == 128) ? (u ^ (r & 7)) : (u ^ ((r >> 1) & 3));
    const int byte = r * row_bytes + pu * 16 + (c * 2) % 16;
    out[i] = *reinterpret_cast<uint16_t*>(smem + byte);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct LaunchMaps {
  CUtensorMap a, b, in, in2, out1, out2;
};

template <int BN, int MODE, int LIGHT = 0>
static int launch_igemm(const LaunchMaps& mp, const bcosk_igemm_params& p, const IgemmAux& aux, cudaStream_t st) {
  using Cfg = TileCfg<BN, LIGHT>;
  auto kern = bcosk_igemm_kernel<BN, MODE, __nv_bfloat16, LIGHT>;
  auto kern_h = bcosk_igemm_kernel<BN, MODE, __half, LIGHT>;
  const void* fn = (p.dtype == BCOSK_DTYPE_BF16) ? (const void*)kern : (const void*)kern_h;
  // per launch: the attribute belongs to (function, device); a process may drive several GPUs and threads
  BCOSK_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
  const long long M = (long long)p.a_nb * p.op * p.oq;
  const long long m_tiles = (M + BM - 1) / BM;
  const long long n_tiles = (p.n + BN - 1) / BN;
  if (m_tiles * n_tiles > 0x7fffffffLL) return set_error(BCOSK_EUNSUPPORTED, "igemm: grid too large");
  dim3 grid((unsigned)(m_tiles * n_tiles));
  if (p.dtype == BCOSK_DTYPE_BF16)
    kern<<<grid, NUM_THREADS, Cfg::kSmemBytes, st>>>(mp.a, mp.b, mp.in, mp.in2, mp.out1, mp.out2, p, aux);
  else
    kern_h<<<grid, NUM_THREADS, Cfg::kSmemBytes, st>>>(mp.a, mp.b, mp.in, mp.in2, mp.out1, mp.out2, p, aux);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

static int g_num_sms = 0;             // refreshed per launch from the current device (a process may drive several GPUs)
static int g_late_in_iters = 2;        // K stages from which the epilogue input tile is fetched after the main loop (0 = never)
static bool g_light_enabled = true;
static bool g_light4_enabled = true;
static int g_light4_max_iters = 4;

template <int MODE>
static int launch_persistent(const LaunchMaps& mp, const bcosk_igemm_params& p, const IgemmAux& aux, cudaStream_t st) {
  using Cfg = PersistCfg;
  auto kern = bcosk_igemm_persistent_kernel<MODE, __nv_bfloat16>;
  auto kern_h = bcosk_igemm_persistent_kernel<MODE, __half>;
  const void* fn = (p.dtype == BCOSK_DTYPE_BF16) ? (const void*)kern : (const void*)kern_h;
  // per launch: the attribute belongs to (function, device); a process may drive several GPUs and threads
  BCOSK_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
  {
    int dev = 0;
    BCOSK_CUDA_CHECK(cudaGetDevice(&dev));
    BCOSK_CUDA_CHECK(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const long long M = (long long)p.a_nb * p.op * p.oq;
  const long long tiles = ((M + BM - 1) / BM) * ((p.n + P_BN - 1) / P_BN);
  if (tiles > 0x7fffffffLL) return set_error(BCOSK_EUNSUPPORTED, "igemm: too many tiles");
  dim3 grid((unsigned)(tiles < g_num_sms ? tiles : g_num_sms));
  if (p.dtype == BCOSK_DTYPE_BF16)
    kern<<<grid, P_THREADS, Cfg::kSmemBytes, st>>>(mp.a, mp.b, mp.in, mp.in2, mp.out1, mp.out2, p, aux);
  else
    kern_h<<<grid, P_THREADS, Cfg::kSmemBytes, st>>>(mp.a, mp.b, mp.in, mp.in2, mp.out1, mp.out2, p, aux);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

template <int BN, int MODE>
static int launch_flat_bn(const bcosk_igemm_params& p, cudaStream_t st) {
  using Cfg = FlatCfg<BN>;
  const bool dense = p.a_flat == 2;
  int kw = 1, kh = 1;
  for (int t = 0; t < p.num_taps; ++t) {
    if (p.tap_off_h[t] < 0 || p.tap_off_w[t] < 0) return set_error(BCOSK_EINVAL, "igemm(flat): negative tap offset");
    kw = max(kw, p.tap_off_w[t] + 1);
    kh = max(kh, p.tap_off_h[t] + 1);
  }
  FlatGeom geo;
  memset(&geo, 0, sizeof(geo));
  geo.dense = dense ? 1 : 0;
  // dense input: the pitch only exists in shared memory; rows must start on a swizzle-pattern boundary (8 pixels)
  geo.pitch = dense ? ((p.a_w + kw - 1 + 7) & ~7) : p.a_wp;
  const int wp = geo.pitch, hp = dense ? p.a_h : p.a_hp;
  const int max_off = (kh - 1) * wp + (kw - 1);
  const int need = BM + max_off;
  geo.nbox = need <= 256 ? 1 : 2;
  geo.box_rows = (((need + geo.nbox - 1) / geo.nbox) + 7) & ~7;
  if (!dense && geo.box_rows > 256)
    return set_error(BCOSK_EUNSUPPORTED, "igemm(flat): window of %d rows does not fit two TMA boxes", need);
  geo.tiles_img = ((p.op - 1) * wp + p.oq + BM - 1) / BM;
  // dense: image rows touched by a tile that may start at any position of a row, plus the taps' rows
  geo.nrows = ((BM % wp == 0 ? 0 : wp - 1) + BM - 1) / wp + kh;
  if (dense && (geo.nrows > 256 || wp > 256)) return set_error(BCOSK_EUNSUPPORTED, "igemm(flat): window too large for one TMA box");
  const int row_bytes = p.kch * 2;
  const long long b_bytes = (long long)p.num_taps * BN * row_bytes;
  const long long win_stride = dense ? (((long long)geo.nrows * wp * row_bytes + 1023) & ~1023ll)
                                     : (((long long)geo.nbox * geo.box_rows * row_bytes + 1023) & ~1023ll);

  LaunchMaps mp;
  memset(&mp, 0, sizeof(mp));
  IgemmAux aux{};
  {
    int rc;
    if (dense) {
      const long long dims[4] = {p.a_c, p.a_w, p.a_h, p.a_nb};
      const long long strides[3] = {(long long)p.a_c * 2, (long long)p.a_w * p.a_c * 2, (long long)p.a_h * p.a_w * p.a_c * 2};
      const int box[4] = {p.kch, wp, geo.nrows, 1};
      rc = make_tiled_map_nd(&mp.a, p.a, 2, 4, dims, strides, box, row_bytes);
    } else {
      const uint8_t* origin = reinterpret_cast<const uint8_t*>(p.a) + ((long long)p.lo_h * wp + p.lo_w) * p.a_c * 2;
      const long long dims[2] = {p.a_c, p.a_flat_rows};
      const long long strides[1] = {(long long)p.a_c * 2};
      const int box[2] = {p.kch, geo.box_rows};
      rc = make_tiled_map_nd(&mp.a, origin, 2, 2, dims, strides, box, row_bytes);
    }
    if (rc) return rc;
    rc = make_tiled_map_2d(&mp.b, p.b, (long long)p.num_taps * p.kch, p.n, p.kch, BN, row_bytes);
    if (rc) return rc;
  }
  const bool dense_out = p.os_0 == 0 && p.os_q == 1 && p.os_p == p.oq && p.os_n == (long long)p.op * p.oq;
  auto stageable = [&](const void* base, int ld) -> bool {
    return (reinterpret_cast<uintptr_t>(base) & 15) == 0 && ld % 8 == 0;
  };
  if (BN == 64 && dense_out) {   // 16-bit outputs staged in shared memory, written as full lines
    if (!p.y_f32 && p.y_planes == 1) aux.tma_out1 = stageable(p.y, p.y_ld) ? 1 : 0;
    if (MODE == BCOSK_MODE_FWD && p.gain && !p.gain_f32) aux.tma_out2 = stageable(p.gain, p.gain_ld) ? 1 : 0;
    if (MODE == BCOSK_MODE_EXPLAIN && p.out2 && p.out2_planes == 1) aux.tma_out2 = stageable(p.out2, p.out2_ld) ? 1 : 0;
  }
  if ((aux.tma_out1 || aux.tma_out2) && BM % wp == 0) {
    // a tile is BM / pitch whole image rows: one clipped 3-D store per row and tensor (x >= oq falls outside the map)
    auto map_out = [&](CUtensorMap* m, const void* base, int ld) -> bool {
      const long long dims[3] = {p.n, p.oq, (long long)p.a_nb * p.op};
      const long long strides[2] = {(long long)ld * 2, (long long)p.oq * ld * 2};
      const int box[3] = {64, wp, 1};
      return make_tiled_map_nd(m, base, 2, 3, dims, strides, box, 128) == BCOSK_OK;
    };
    const void* o2 = MODE == BCOSK_MODE_FWD ? p.gain : p.out2;
    const int o2_ld = MODE == BCOSK_MODE_FWD ? p.gain_ld : p.out2_ld;
    geo.tma_store = (!aux.tma_out1 || map_out(&mp.out1, p.y, p.y_ld)) && (!aux.tma_out2 || map_out(&mp.out2, o2, o2_ld)) ? 1 : 0;
  }
  const long long smem = ((b_bytes + 1023) & ~1023ll) + 2 * win_stride +
                         ((aux.tma_out1 || aux.tma_out2) ? 4 * Cfg::kTileBytes : 0) + 128 + 2 * BN * 4 +
                         2 * (BN / 32) * BM * 4 + BCOSK_MAX_TAPS * 4;
  if (smem > 227 * 1024) return set_error(BCOSK_EUNSUPPORTED, "igemm(flat): %lld bytes of shared memory needed", smem);
  auto kern = bcosk_igemm_flat_kernel<BN, MODE, __nv_bfloat16>;
  auto kern_h = bcosk_igemm_flat_kernel<BN, MODE, __half>;
  const void* fn = (p.dtype == BCOSK_DTYPE_BF16) ? (const void*)kern : (const void*)kern_h;
  BCOSK_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  {
    int dev = 0;
    BCOSK_CUDA_CHECK(cudaGetDevice(&dev));
    BCOSK_CUDA_CHECK(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const long long tiles = (long long)p.a_nb * geo.tiles_img;
  if (tiles > 0x7fffffffLL || (long long)p.a_nb * hp * wp > 0x7fffffffLL) return set_error(BCOSK_EUNSUPPORTED, "igemm(flat): too large");
  dim3 grid((unsigned)(tiles < g_num_sms ? tiles : g_num_sms));
  if (p.dtype == BCOSK_DTYPE_BF16)
    kern<<<grid, Cfg::kThreads, (size_t)smem, st>>>(mp.a, mp.b, mp.out1, mp.out2, p, aux, geo);
  else
    kern_h<<<grid, Cfg::kThreads, (size_t)smem, st>>>(mp.a, mp.b, mp.out1, mp.out2, p, aux, geo);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

static int launch_flat(const bcosk_igemm_params& p, cudaStream_t st) {
  if (p.hp_accum || p.num_segs != 1 || p.chunks_per_tap != 1 || p.stride_w != 1 || p.stride_h != 1 || p.n > 64)
    return set_error(BCOSK_EUNSUPPORTED, "igemm(flat): needs stride 1, one segment, one chunk per tap, n <= 64, no hp_accum");
  if (p.a_c < p.kch || p.seg_a_choff[0] != 0) return set_error(BCOSK_EINVAL, "igemm(flat): bad channel geometry");
  if (p.a_flat == 1) {
    if (p.a_wp < p.a_w || p.a_hp < p.a_h || p.a_flat_rows < 1) return set_error(BCOSK_EINVAL, "igemm(flat): bad buffer geometry");
    if (p.oq > p.a_wp) return set_error(BCOSK_EINVAL, "igemm(flat): oq exceeds the buffer pitch");
  } else if (p.a_flat != 2) {
    return set_error(BCOSK_EINVAL, "igemm(flat): a_flat must be 1 or 2");
  }
  if (p.mode == BCOSK_MODE_FWD && p.scale_mode != BCOSK_SCALE_NONE && !p.inv_norm)
    return set_error(BCOSK_EUNSUPPORTED, "igemm(flat): inv_norm must be precomputed");
  if (p.res_planes > 1 || p.y_planes > 1 && !p.y_f32) return set_error(BCOSK_EUNSUPPORTED, "igemm(flat): single plane only");
  if (p.mode == BCOSK_MODE_FWD)
    return p.n <= 32 ? launch_flat_bn<32, BCOSK_MODE_FWD>(p, st) : launch_flat_bn<64, BCOSK_MODE_FWD>(p, st);
  return p.n <= 32 ? launch_flat_bn<32, BCOSK_MODE_EXPLAIN>(p, st) : launch_flat_bn<64, BCOSK_MODE_EXPLAIN>(p, st);
}

static int validate(const bcosk_igemm_params& p) {
  if (!p.a || !p.b || !p.y) return set_error(BCOSK_EINVAL, "igemm: null a/b/y");
  if (p.kch != 64 && p.kch != 32) return set_error(BCOSK_EINVAL, "igemm: kch must be 32 or 64");
  if (p.num_taps < 1 || p.num_taps > BCOSK_MAX_TAPS) return set_error(BCOSK_EINVAL, "igemm: num_taps out of range");
  if (p.num_segs < 1 || p.num_segs > BCOSK_MAX_SEGS) return set_error(BCOSK_EINVAL, "igemm: num_segs out of range");
  if (p.chunks_per_tap < 1) return set_error(BCOSK_EINVAL, "igemm: chunks_per_tap < 1");
  const int total = p.num_segs * p.num_taps * p.chunks_per_tap;
  if (total % (STAGE_K / p.kch) != 0) return set_error(BCOSK_EINVAL, "igemm: chunk count not a multiple of the stage");
  if (p.a_c % 8 != 0) return set_error(BCOSK_EINVAL, "igemm: a_c must be a multiple of 8 (16-byte pixels)");
  if (p.n < 8 || p.n % 8 != 0) return set_error(BCOSK_EINVAL, "igemm: n must be a positive multiple of 8");
  if (p.dtype != BCOSK_DTYPE_BF16 && p.dtype != BCOSK_DTYPE_F16) return set_error(BCOSK_EINVAL, "igemm: dtype");
  if (p.mode == BCOSK_MODE_FWD && p.scale_mode != BCOSK_SCALE_NONE && !p.inv_norm && !p.sq_in)
    return set_error(BCOSK_EINVAL, "igemm: inv_norm or sq_in required for a B-cos scale");
  if (!p.inv_norm && p.sq_in && (p.sq_parts < 1 || p.sq_k < 1 || p.sq_stride < 1 || p.sq_h < 1 || p.sq_w < 1))
    return set_error(BCOSK_EINVAL, "igemm: bad sq_in geometry");
  if (p.a_nb < 1 || p.op < 1 || p.oq < 1) return set_error(BCOSK_EINVAL, "igemm: empty problem");
  if (p.mul1_sqrt_scale && (p.mode != BCOSK_MODE_EXPLAIN || !p.mul1 || p.mul1_f32))
    return set_error(BCOSK_EINVAL, "igemm: mul1_sqrt_scale needs explain mode and a 16-bit mul1");
  if (p.inv_norm_out && p.mode != BCOSK_MODE_FWD) return set_error(BCOSK_EINVAL, "igemm: inv_norm_out is a forward output");
  if (p.side_mapped && (p.mode != BCOSK_MODE_EXPLAIN || p.add != nullptr))
    return set_error(BCOSK_EINVAL, "igemm: side_mapped needs explain mode without an extra gradient");
  if (p.act != 0) {
    if (p.act != 1 && p.act != 2) return set_error(BCOSK_EINVAL, "igemm: act must be 0 (none), 1 (GELU, detached gate) or 2 (QuickGELU)");
    if (p.mode != BCOSK_MODE_FWD || p.hp_accum || p.y_f32 || p.y_planes != 1 || (p.gain && p.gain_f32) || (p.res && p.res_planes != 1) ||
        (p.scale_mode != BCOSK_SCALE_B2 && p.scale_mode != BCOSK_SCALE_NONE) || p.lin_bias || p.max_out > 1 || p.relu || p.maskbits)
      return set_error(BCOSK_EUNSUPPORTED, "igemm: act belongs to a one-plane 16-bit forward launch without ReLU / mask bits / MaxOut / bias");
  }
  if (p.max_out > 1) {
    if (p.mode != BCOSK_MODE_FWD || (p.max_out != 2 && p.max_out != 4 && p.max_out != 8) || p.n % p.max_out != 0)
      return set_error(BCOSK_EINVAL, "igemm: max_out must be 2, 4 or 8, divide n, and belongs to a forward launch");
    if (p.alpha || p.beta || p.res || p.relu || p.maskbits || p.a_flat || p.inv_norm_out)
      return set_error(BCOSK_EINVAL, "igemm: max_out is not combined with alpha / beta / res / relu / maskbits / a_flat / inv_norm_out");
    if (p.amax && p.amax_ld < p.n / p.max_out) return set_error(BCOSK_EINVAL, "igemm: amax_ld < n / max_out");
    if (p.y_ld < p.n / p.max_out || (p.gain && p.gain_ld < p.n / p.max_out))
      return set_error(BCOSK_EINVAL, "igemm: y_ld / gain_ld < n / max_out");
  } else if (p.y_ld % (p.y_f32 ? 4 : 8) != 0) {
    return set_error(BCOSK_EINVAL, "igemm: y_ld alignment");
  }
  return BCOSK_OK;
}

static int make_maps(const bcosk_igemm_params& p, int bn, LaunchMaps* mp, IgemmAux* aux) {
  memset(mp, 0, sizeof(*mp));
  memset(aux, 0, sizeof(*aux));
  int rc = make_im2col_map_nhwc(&mp->a, p.a, p.a_nb, p.a_h, p.a_w, p.a_c, p.lo_w, p.lo_h, p.up_w, p.up_h, p.stride_w,
                                p.stride_h, p.kch, BM, p.kch == 64 ? 128 : 64);
  if (rc) return rc;
  const long long ktot = (long long)p.num_segs * p.num_taps * p.chunks_per_tap * p.kch;
  rc = make_tiled_map_2d(&mp->b, p.b, ktot, p.n, p.kch, bn, p.kch == 64 ? 128 : 64);
  if (rc) return rc;
  // ---- TMA epilogue (throughput mode): 16-bit single-plane tensors addressed densely by output row
  const long long M = (long long)p.a_nb * p.op * p.oq;
  const bool tile_ok = (bn == 64 || bn == 128) && p.max_out <= 1;   // MaxOut rows leave with per-row stores
  const bool dense_out = p.os_0 == 0 && p.os_q == 1 && p.os_p == p.oq && p.os_n == (long long)p.op * p.oq;
  auto map16 = [&](CUtensorMap* m, const void* base, int ld) -> bool {
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || ld % 8 != 0) return false;
    return make_tiled_map_2d(m, base, ld, M, 64, BM, 128) == BCOSK_OK;
  };
  if (tile_ok) {
    if (p.y && !p.y_f32 && p.y_planes == 1 && dense_out) aux->tma_out1 = map16(&mp->out1, p.y, p.y_ld) ? 1 : 0;
    if (p.mode == BCOSK_MODE_FWD) {
      if (p.gain && !p.gain_f32) aux->tma_out2 = map16(&mp->out2, p.gain, p.gain_ld) ? 1 : 0;
      if (p.res && p.res_planes == 1) aux->tma_in = map16(&mp->in, p.res, p.res_ld) ? 1 : 0;
    } else {
      if (p.out2 && p.out2_planes == 1 && !p.side_mapped) aux->tma_out2 = map16(&mp->out2, p.out2, p.out2_ld) ? 1 : 0;
      if (p.mul1 && !p.mul1_f32 && !p.side_mapped) aux->tma_in = map16(&mp->in, p.mul1, p.mul1_ld) ? 2 : 0;
      // second input tile: the extra gradient, when it is dense over the same rows (identity shortcuts) and the tile
      // shape leaves two ring stages (64-wide tiles have 4 slots)
      if (aux->tma_in && bn == 64 && p.add && p.add_planes == 1 && p.add_stride == 1 && p.add_p == p.op && p.add_q == p.oq)
        aux->tma_in2 = map16(&mp->in2, p.add, p.add_ld) ? 1 : 0;
    }
  }
  return BCOSK_OK;
}

}  // namespace bcosk

using namespace bcosk;

extern "C" int bcosk_igemm(const bcosk_igemm_params* pp, void* stream) {
  if (!pp) return set_error(BCOSK_EINVAL, "igemm: null params");
  bcosk_igemm_params p = *pp;
  int rc = validate(p);
  if (rc) return rc;
  int bn = p.block_n;
  if (bn == 0) bn = p.n <= 32 ? 32 : ((p.n <= 64 || p.hp_accum) ? 64 : 128);
  if (bn != 32 && bn != 64 && bn != 128) return set_error(BCOSK_EINVAL, "igemm: block_n");
  p.block_n = bn;
  if (p.max_out > 1) p.sched = 1;        // MaxOut: the per-tile kernel (generic epilogue, per-row stores)
  if (p.a_flat) return launch_flat(p, reinterpret_cast<cudaStream_t>(stream));
  if (p.hp_accum) return launch_hp(p, reinterpret_cast<cudaStream_t>(stream));   // parity mode: bcosk_igemm_hp.cu
  LaunchMaps mp;
  IgemmAux aux{};
  rc = make_maps(p, bn, &mp, &aux);
  if (rc) return rc;
  {
    const int iters = p.num_segs * p.num_taps * p.chunks_per_tap / (STAGE_K / p.kch);
    aux.late_in = (g_late_in_iters > 0 && bn == 128 && iters >= g_late_in_iters) ? 1 : 0;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
#define BCOSK_DISPATCH(BN_)                                                                         \
  case BN_:                                                                                         \
    return p.mode == BCOSK_MODE_FWD ? launch_igemm<BN_, BCOSK_MODE_FWD>(mp, p, aux, st)             \
                                    : launch_igemm<BN_, BCOSK_MODE_EXPLAIN>(mp, p, aux, st);
  if (p.sched < 0 || p.sched > 3) return set_error(BCOSK_EINVAL, "igemm: sched must be 0..3");
  if (p.sched >= 2 && bn == 64) {   // 0 / 1 one CTA per tile, 2 persistent strided, 3 persistent in row-block order
    aux.order = p.sched == 3 ? 1 : 0;
    return p.mode == BCOSK_MODE_FWD ? launch_persistent<BCOSK_MODE_FWD>(mp, p, aux, st)
                                    : launch_persistent<BCOSK_MODE_EXPLAIN>(mp, p, aux, st);
  }
  {
    // explain launches with ONE K stage and both input tiles (producer gain + extra gradient): the 3-slot variant fits
    // them too - stage | extra-gradient tile | gain tile - with out2 staged over the extra-gradient tile, whose words
    // every thread has consumed before it writes the same words of out2 (epilogue_explain_fast order)
    const int iters = p.num_segs * p.num_taps * p.chunks_per_tap / (STAGE_K / p.kch);
    if (bn == 64 && g_light_enabled && aux.tma_in2 && iters == 1 && p.mode == BCOSK_MODE_EXPLAIN && aux.tma_in &&
        aux.tma_out1 && (aux.tma_out2 || !p.out2) && !p.y_f32 && p.y_planes == 1 && !p.mul2_f32)
      return launch_igemm<64, BCOSK_MODE_EXPLAIN, 1>(mp, p, aux, st);
  }
  if (bn == 64 && g_light_enabled && !aux.tma_in2) {
    // short K loop (<= 4 stages): the 3-CTA/SM variant
    const int iters = p.num_segs * p.num_taps * p.chunks_per_tap / (STAGE_K / p.kch);
    // two-slot variant, 4 CTAs per SM: one K stage with the input tile prefetched, or up to four stages with the input
    // tile fetched after the loop (aux.late_in); the second output tile is staged over the consumed input tile
    const bool out_tiles = aux.tma_out1 && (aux.tma_out2 || !(p.mode == BCOSK_MODE_FWD ? p.gain : p.out2));
    if (iters <= g_light4_max_iters && g_light4_enabled && out_tiles) {
      aux.late_in = (aux.tma_in && iters >= 2) ? 1 : 0;
      return p.mode == BCOSK_MODE_FWD ? launch_igemm<64, BCOSK_MODE_FWD, 2>(mp, p, aux, st)
                                      : launch_igemm<64, BCOSK_MODE_EXPLAIN, 2>(mp, p, aux, st);
    }
    if (iters <= 4)
      return p.mode == BCOSK_MODE_FWD ? launch_igemm<64, BCOSK_MODE_FWD, 1>(mp, p, aux, st)
                                      : launch_igemm<64, BCOSK_MODE_EXPLAIN, 1>(mp, p, aux, st);
  }
  switch (bn) {
    BCOSK_DISPATCH(32)
    BCOSK_DISPATCH(64)
    BCOSK_DISPATCH(128)
  }
#undef BCOSK_DISPATCH
  return set_error(BCOSK_EINVAL, "igemm: unreachable");
}

extern "C" int bcosk_set_late_input(int32_t min_k_stages) {
  const int prev = g_late_in_iters;
  g_late_in_iters = min_k_stages;
  return prev;
}

extern "C" int bcosk_set_light(int32_t enabled) {
  const int prev = (g_light_enabled ? 1 : 0) | (g_light4_enabled ? 2 : 0);
  g_light_enabled = (enabled & 1) != 0;
  g_light4_enabled = (enabled & 2) != 0;
  g_light4_max_iters = (enabled & 4) ? 1 : ((enabled & 8) ? 1 << 20 : 4);   // bit 2: single-stage launches only; bit 3: any K (A/B)
  return prev;
}

extern "C" int bcosk_debug_a_tile(const bcosk_igemm_params* pp, int32_t tile_m, int32_t chunk, void* out, void* stream) {
  if (!pp || !out) return set_error(BCOSK_EINVAL, "debug_a_tile: null");
  bcosk_igemm_params p = *pp;
  CUtensorMap ta;
  int rc = make_im2col_map_nhwc(&ta, p.a, p.a_nb, p.a_h, p.a_w, p.a_c, p.lo_w, p.lo_h, p.up_w, p.up_h, p.stride_w,
                                p.stride_h, p.kch, BM, p.kch == 64 ? 128 : 64);
  if (rc) return rc;
  bcosk_debug_a_tile_kernel<<<1, 128, BM * 128 + 1024, reinterpret_cast<cudaStream_t>(stream)>>>(
      ta, p, tile_m, chunk, reinterpret_cast<uint16_t*>(out));
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}
