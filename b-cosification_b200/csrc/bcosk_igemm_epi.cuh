// bcosk_igemm_epi.cuh -- epilogue building blocks shared by the implicit-GEMM kernels (bcosk_igemm.cu, bcosk_igemm_hp.cu):
// per-row bookkeeping, precision-plane loads / stores, and the 128B-swizzled shared-memory tiles that TMA bulk copies move.
#pragma once
#include "../../include/bcosk.h"
#include "bcosk_common.cuh"

namespace bcosk {
struct RowInfo {
  int m, img, p, q;
  bool valid;
  float gscale;   // explain: mul1_sqrt_scale[row] (the multiplier is sqrt(mul1 * gscale)) or unused
};

// 16-bit row segment (32 columns starting at `ptr`) -> 32 floats, adding over precision planes
template <typename T>
__device__ __forceinline__ void load32_planes(const T* ptr, int planes, int plane_stride, int ncols, float (&v)[32]) {
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = 0.f;
  for (int pl = 0; pl < planes; ++pl) {
    const uint4* src = reinterpret_cast<const uint4*>(ptr + (size_t)pl * plane_stride);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      if (g * 8 < ncols) {
        uint4 u = __ldg(src + g);
        float2 f;
        f = Cvt<T>::unpack2(u.x); v[g * 8 + 0] += f.x; v[g * 8 + 1] += f.y;
        f = Cvt<T>::unpack2(u.y); v[g * 8 + 2] += f.x; v[g * 8 + 3] += f.y;
        f = Cvt<T>::unpack2(u.z); v[g * 8 + 4] += f.x; v[g * 8 + 5] += f.y;
        f = Cvt<T>::unpack2(u.w); v[g * 8 + 6] += f.x; v[g * 8 + 7] += f.y;
      }
    }
  }
}

// fp32 row segment (32 columns) -> v
__device__ __forceinline__ void load32_f32(const float* ptr, int ncols, float (&v)[32]) {
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    if (g * 4 < ncols) {
      float4 f = __ldg(reinterpret_cast<const float4*>(ptr) + g);
      v[g * 4 + 0] = f.x; v[g * 4 + 1] = f.y; v[g * 4 + 2] = f.z; v[g * 4 + 3] = f.w;
    } else {
      v[g * 4 + 0] = v[g * 4 + 1] = v[g * 4 + 2] = v[g * 4 + 3] = 0.f;
    }
  }
}

// store 32 floats as 16-bit precision planes: plane 0 = rn(v), plane 1 = rn(v - plane0), ...
// returns in `v` the value actually representable by the stored planes (sum of planes).
template <typename T>
__device__ __forceinline__ void store32_planes(T* ptr, int planes, int plane_stride, int ncols, float (&v)[32]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float r[8], acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { r[i] = v[g * 8 + i]; acc[i] = 0.f; }
    for (int pl = 0; pl < planes; ++pl) {
      uint32_t w[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        w[j] = Cvt<T>::pack2(r[2 * j], r[2 * j + 1]);
        const float2 f = Cvt<T>::unpack2(w[j]);
        r[2 * j] -= f.x; r[2 * j + 1] -= f.y;
        acc[2 * j] += f.x; acc[2 * j + 1] += f.y;
      }
      if (g * 8 < ncols)
        reinterpret_cast<uint4*>(ptr + (size_t)pl * plane_stride)[g] = make_uint4(w[0], w[1], w[2], w[3]);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) v[g * 8 + i] = acc[i];
  }
}

__device__ __forceinline__ void store32_f32(float* ptr, int ncols, const float (&v)[32]) {
#pragma unroll
  for (int g = 0; g < 8; ++g)
    if (g * 4 < ncols)
      reinterpret_cast<float4*>(ptr)[g] = make_float4(v[g * 4], v[g * 4 + 1], v[g * 4 + 2], v[g * 4 + 3]);
}

// ---------------------------------------------------------------------------------------------
// MaxOut forward tail (include/bcosk.h `max_out`): NV consecutive accumulator columns of one output row (bias already
// added), first GEMM column c0 (a multiple of NV), NV % G == 0.  Keeps the largest unit of every group of G adjacent
// columns (first one on ties), applies the B-cos scale of the kept unit and writes the NV/G results of this row at
// column c0/G: y (fp32 or precision planes), gain, amax.  Returns the sum of the squared outputs as stored.
// Per-row scalar stores: the MaxOut layers belong to the module-level path, not to the benchmarked plans.
// ---------------------------------------------------------------------------------------------
template <typename T, int NV, int G>
__device__ __forceinline__ float maxout_fwd_tail_g(const bcosk_igemm_params& p, const float (&v)[NV], float inv_norm, int64_t m_row,
                                                   int64_t yrow, int c0, int ncols) {
  constexpr int NO = NV / G;
  const int o0 = c0 / G;
  float sq = 0.f;
#pragma unroll
  for (int o = 0; o < NO; ++o) {
    if (o * G < ncols) {
      float best = v[o * G];
      int bi = 0;
#pragma unroll
      for (int k = 1; k < G; ++k) {
        const bool gt = v[o * G + k] > best;
        best = gt ? v[o * G + k] : best;
        bi = gt ? k : bi;
      }
      float t = 1.f;
      if (p.scale_mode == BCOSK_SCALE_B2) t = fabsf(best) * inv_norm;
      else if (p.scale_mode == BCOSK_SCALE_POW) t = __powf(fabsf(best) * inv_norm + 1e-6f, p.b_exp - 1.f);
      float y = best * t;
      if (p.y_f32) {
        reinterpret_cast<float*>(p.y)[(size_t)yrow * p.y_ld + o0 + o] = y;
      } else {
        T* yp = reinterpret_cast<T*>(p.y) + (size_t)yrow * p.y_ld + o0 + o;
        float r = y, acc = 0.f;
        for (int pl = 0; pl < p.y_planes; ++pl) {
          const float h = Cvt<T>::round1(r);
          yp[(size_t)pl * p.y_plane_stride] = T(h);
          r -= h;
          acc += h;
        }
        y = acc;
      }
      if (p.gain != nullptr) {
        if (p.gain_f32) reinterpret_cast<float*>(p.gain)[(size_t)m_row * p.gain_ld + o0 + o] = t;
        else reinterpret_cast<T*>(p.gain)[(size_t)m_row * p.gain_ld + o0 + o] = T(t);
      }
      if (p.amax != nullptr) p.amax[(size_t)m_row * p.amax_ld + o0 + o] = (uint8_t)bi;
      sq = fmaf(y, y, sq);
    }
  }
  return sq;
}

template <typename T, int NV>
__device__ __forceinline__ float maxout_fwd_tail(const bcosk_igemm_params& p, const float (&v)[NV], float inv_norm, int64_t m_row,
                                                 int64_t yrow, int c0, int ncols) {
  if (p.max_out == 2) return maxout_fwd_tail_g<T, NV, 2>(p, v, inv_norm, m_row, yrow, c0, ncols);
  if (p.max_out == 4) return maxout_fwd_tail_g<T, NV, 4>(p, v, inv_norm, m_row, yrow, c0, ncols);
  return maxout_fwd_tail_g<T, NV, 8>(p, v, inv_norm, m_row, yrow, c0, ncols);
}

// Library-internal launch state (decided by the host launcher, see launch_igemm)
struct IgemmAux {
  int tma_in;    // 0 none, 1 = forward residual, 2 = explain mul1: prefetched as a tile into the last pipeline slot
  int tma_in2;   // explain: the extra gradient `add` (dense, same rows as y) prefetched into the slot before it
  int tma_out1;  // primary output y staged in slot 0 and written with TMA
  int tma_out2;  // forward: gain, explain: out2 - staged in slot 1 and written with TMA
  int order;     // persistent kernel: 0 = tiles strided over the grid, 1 = a CTA walks all n tiles of one row block
  int late_in;   // long K loops: fetch the epilogue input tile AFTER the main loop (into the last slot, once its final
                 // stage is consumed) so that the ring keeps all its stages while the MMAs run
};

// Shared-memory tiles of the TMA epilogue: [BN/64 boxes][128 rows][128 bytes], 16-byte units XOR-swizzled by row
// (CU_TENSOR_MAP_SWIZZLE_128B).  Thread = row r, chunk j = 32 columns = 4 units.
// Tiles are addressed in the shared window (32-bit addresses, 0 = absent) with explicit ld.shared / st.shared so that
// the compiler never falls back to generic-space accesses.
struct EpiTiles {
  uint32_t in;
  uint32_t in2;
  uint32_t out1;
  uint32_t out2;
};
__device__ __forceinline__ uint32_t tile_ptr(uint32_t tile, int r, int j, int g) {
  const int u = ((j & 1) << 2) + g;
  return tile + ((j >> 1) << 14) + (r << 7) + ((u ^ (r & 7)) << 4);
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 u;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(addr));
  return u;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& u) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(u.x), "r"(u.y), "r"(u.z), "r"(u.w) : "memory");
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 f;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(f.x), "=f"(f.y), "=f"(f.z), "=f"(f.w) : "r"(addr));
  return f;
}
template <typename T>
__device__ __forceinline__ void tile_load32(uint32_t tile, int r, int j, float (&v)[32]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const uint4 u = lds128(tile_ptr(tile, r, j, g));
    float2 f;
    f = Cvt<T>::unpack2(u.x); v[g * 8 + 0] = f.x; v[g * 8 + 1] = f.y;
    f = Cvt<T>::unpack2(u.y); v[g * 8 + 2] = f.x; v[g * 8 + 3] = f.y;
    f = Cvt<T>::unpack2(u.z); v[g * 8 + 4] = f.x; v[g * 8 + 5] = f.y;
    f = Cvt<T>::unpack2(u.w); v[g * 8 + 6] = f.x; v[g * 8 + 7] = f.y;
  }
}
// rounds v to 16 bit (v returns the stored value) and writes the 32 columns of this row into the tile
template <typename T>
__device__ __forceinline__ void tile_store32(uint32_t tile, int r, int j, float (&v)[32]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      w[k] = Cvt<T>::pack2(v[g * 8 + 2 * k], v[g * 8 + 2 * k + 1]);
      const float2 f = Cvt<T>::unpack2(w[k]);
      v[g * 8 + 2 * k] = f.x; v[g * 8 + 2 * k + 1] = f.y;
    }
    sts128(tile_ptr(tile, r, j, g), make_uint4(w[0], w[1], w[2], w[3]));
  }
}

}  // namespace bcosk
