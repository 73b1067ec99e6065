// bcosk_elementwise.cu -- bandwidth kernels around the implicit GEMM (sm_100a).
//
// All tensors are NHWC; 16-bit tensors are moved with 16-byte vector accesses (8 channels per thread),
// reductions use warp shuffles, and every kernel is sized so that consecutive lanes touch consecutive
// addresses.  Each entry point is documented in include/bcosk.h with the reference code it replaces.
#include "../../include/bcosk.h"
#include "bcosk_common.cuh"
#include "bcosk_host.h"

namespace bcosk {

static inline unsigned blocks_for(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

template <typename T>
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  float2 a;
  a = Cvt<T>::unpack2(u.x); f[0] = a.x; f[1] = a.y;
  a = Cvt<T>::unpack2(u.y); f[2] = a.x; f[3] = a.y;
  a = Cvt<T>::unpack2(u.z); f[4] = a.x; f[5] = a.y;
  a = Cvt<T>::unpack2(u.w); f[6] = a.x; f[7] = a.y;
}
template <typename T>
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(Cvt<T>::pack2(f[0], f[1]), Cvt<T>::pack2(f[2], f[3]), Cvt<T>::pack2(f[4], f[5]),
                    Cvt<T>::pack2(f[6], f[7]));
}
// 8 channels summed over precision planes
template <typename T>
__device__ __forceinline__ void load8_planes(const T* ptr, int planes, int plane_stride, float (&f)[8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i) f[i] = 0.f;
  for (int pl = 0; pl < planes; ++pl) {
    float g[8];
    unpack8<T>(__ldg(reinterpret_cast<const uint4*>(ptr + (size_t)pl * plane_stride)), g);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] += g[i];
  }
}
// compile-time single-plane variant: a bare 16-byte load, so unrolled callers can overlap many of them
template <typename T, bool ONE>
__device__ __forceinline__ void load8_pl(const T* ptr, int planes, int plane_stride, float (&f)[8]) {
  if (ONE) unpack8<T>(__ldg(reinterpret_cast<const uint4*>(ptr)), f);
  else load8_planes<T>(ptr, planes, plane_stride, f);
}

// split-store 8 channels into planes; f returns the stored (representable) value
template <typename T>
__device__ __forceinline__ void store8_planes(T* ptr, int planes, int plane_stride, float (&f)[8]) {
  float r[8], acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { r[i] = f[i]; acc[i] = 0.f; }
  for (int pl = 0; pl < planes; ++pl) {
    uint4 u = pack8<T>(r);
    float g[8];
    unpack8<T>(u, g);
#pragma unroll
    for (int i = 0; i < 8; ++i) { r[i] -= g[i]; acc[i] += g[i]; }
    *reinterpret_cast<uint4*>(ptr + (size_t)pl * plane_stride) = u;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) f[i] = acc[i];
}

// ------------------------------------------------------------------------------------------------
// input normalise + NCHW fp32 -> NHWC 16-bit + 2x2 space-to-depth (+ per-pixel sum of squares)
// ------------------------------------------------------------------------------------------------
struct Norm6 { float mean[6]; float inv_std[6]; };

// 2x2 patch of the 6-channel [x, 1-x] input at (img, 2r.., 2s..): either fp32 NCHW with 6 channels, or uint8 NCHW RGB
// (x = u8/255, the inverse channels are formed on the fly: AddInverse, reference bcos/data/transforms.py:42-55)
template <typename SRC>
__device__ __forceinline__ void load_patch6(const SRC* __restrict__ x, int img, int r, int s, int h, int w, float (&raw)[24]);
template <>
__device__ __forceinline__ void load_patch6<float>(const float* __restrict__ x, int img, int r, int s, int h, int w,
                                                   float (&raw)[24]) {
  const size_t plane = (size_t)h * w;
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const float* src = x + ((size_t)img * 6 + c) * plane + (size_t)(2 * r) * w + 2 * s;
    const float2 top = __ldg(reinterpret_cast<const float2*>(src));
    const float2 bot = __ldg(reinterpret_cast<const float2*>(src + w));
    raw[0 * 6 + c] = top.x; raw[1 * 6 + c] = top.y; raw[2 * 6 + c] = bot.x; raw[3 * 6 + c] = bot.y;
  }
}
template <>
__device__ __forceinline__ void load_patch6<uint8_t>(const uint8_t* __restrict__ x, int img, int r, int s, int h, int w,
                                                     float (&raw)[24]) {
  const size_t plane = (size_t)h * w;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const uint8_t* src = x + ((size_t)img * 3 + c) * plane + (size_t)(2 * r) * w + 2 * s;
    const uchar2 top = __ldg(reinterpret_cast<const uchar2*>(src));
    const uchar2 bot = __ldg(reinterpret_cast<const uchar2*>(src + w));
    const float v0 = (float)top.x / 255.0f, v1 = (float)top.y / 255.0f, v2 = (float)bot.x / 255.0f, v3 = (float)bot.y / 255.0f;
    raw[0 * 6 + c] = v0; raw[1 * 6 + c] = v1; raw[2 * 6 + c] = v2; raw[3 * 6 + c] = v3;
    raw[0 * 6 + c + 3] = 1.0f - v0; raw[1 * 6 + c + 3] = 1.0f - v1; raw[2 * 6 + c + 3] = 1.0f - v2; raw[3 * 6 + c + 3] = 1.0f - v3;
  }
}

template <typename T, typename SRC>
__global__ void input_prep_s2d_kernel(const SRC* __restrict__ x, int nb, int h, int w, Norm6 nm, T* __restrict__ out,
                                      int cp, int planes, float* __restrict__ sq, int row_pitch, int img_pitch) {
  const int h2 = h >> 1, w2 = w >> 1;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;        // 32-bit index math, the image on blockIdx.y
  if (idx >= h2 * w2) return;
  const int r = idx / w2;
  const int s = idx - r * w2;
  const int img = blockIdx.y;
  float v[24];  // channel (dy*2+dx)*6 + c
  load_patch6<SRC>(x, img, r, s, h, w, v);
  const size_t plane = (size_t)h * w;
#pragma unroll
  for (int d = 0; d < 4; ++d)
#pragma unroll
    for (int c = 0; c < 6; ++c) v[d * 6 + c] = (v[d * 6 + c] - nm.mean[c]) * nm.inv_std[c];
  T* dst = out + ((size_t)img * img_pitch + (size_t)r * row_pitch + s) * ((size_t)planes * cp);
  float st[24];
#pragma unroll
  for (int g = 0; g < 3; ++g) {
    float f[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = v[g * 8 + i];
    store8_planes<T>(dst + g * 8, planes, cp, f);
#pragma unroll
    for (int i = 0; i < 8; ++i) st[g * 8 + i] = f[i];
  }
  const uint4 z = make_uint4(0, 0, 0, 0);
  for (int pl = 0; pl < planes; ++pl)
    for (int g = 3; g < cp / 8; ++g) *reinterpret_cast<uint4*>(dst + (size_t)pl * cp + g * 8) = z;
  if (sq != nullptr) {
    float q[4];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      float a = 0.f;
#pragma unroll
      for (int c = 0; c < 6; ++c) a = fmaf(st[d * 6 + c], st[d * 6 + c], a);
      q[d] = a;
    }
    float* sp = sq + (size_t)img * plane + (size_t)(2 * r) * w + 2 * s;
    *reinterpret_cast<float2*>(sp) = make_float2(q[0], q[1]);
    *reinterpret_cast<float2*>(sp + w) = make_float2(q[2], q[3]);
  }
}

// ------------------------------------------------------------------------------------------------
// patch norm from per-pixel sums of squares
// ------------------------------------------------------------------------------------------------
// Block = 16 x 16 outputs of one image.  The (15*stride + k)^2 window of summed partial maps is staged in shared memory
// (zero outside the image), then every thread adds its k x k taps from shared memory: no per-tap bounds checks or
// 64-bit index arithmetic (the first version was instruction bound: 860 instructions per output for the 7x7 stem).
constexpr int PN_TILE = 16;
__global__ void patch_inv_norm_kernel(const float* __restrict__ sq, int parts, int nb, int h, int w, int kh, int kw,
                                      int stride, int pad, float eps_in, float eps_out, float* __restrict__ inv_norm,
                                      int op, int oq) {
  extern __shared__ float tile[];
  const int img = blockIdx.z;
  const int p0 = blockIdx.y * PN_TILE, q0 = blockIdx.x * PN_TILE;
  const int th = (PN_TILE - 1) * stride + kh, tw = (PN_TILE - 1) * stride + kw;
  const int y0 = p0 * stride - pad, x0 = q0 * stride - pad;
  const size_t part_stride = (size_t)nb * h * w;
  const float* base = sq + (size_t)img * h * w;
  for (int i = threadIdx.x; i < th * tw; i += blockDim.x) {
    const int ty = i / tw, tx = i - ty * tw;
    const int yy = y0 + ty, xx = x0 + tx;
    float v = 0.f;
    if (yy >= 0 && yy < h && xx >= 0 && xx < w) {
      const int o = yy * w + xx;
      for (int t = 0; t < parts; ++t) v += __ldg(base + t * part_stride + o);
    }
    tile[i] = v;
  }
  __syncthreads();
  const int lp = threadIdx.x / PN_TILE, lq = threadIdx.x % PN_TILE;
  const int p = p0 + lp, q = q0 + lq;
  if (p >= op || q >= oq) return;
  float acc = 0.f;
  const float* t0 = tile + (lp * stride) * tw + lq * stride;
  for (int dy = 0; dy < kh; ++dy)
    for (int dx = 0; dx < kw; ++dx) acc += t0[dy * tw + dx];
  inv_norm[((size_t)img * op + p) * oq + q] = 1.0f / (sqrtf(acc + eps_in) + eps_out);
}

// ------------------------------------------------------------------------------------------------
// sum_c x^2 per pixel (one warp per row)
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void pixel_sqsum_kernel(const T* __restrict__ x, long long rows, int c, int planes, int plane_stride, int ld,
                                   float* __restrict__ sq) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const T* src = x + (size_t)row * ld;
  float acc = 0.f;
  for (int g = lane; g < c / 8; g += 32) {
    float f[8];
    load8_planes<T>(src + g * 8, planes, plane_stride, f);
#pragma unroll
    for (int i = 0; i < 8; ++i) acc = fmaf(f[i], f[i], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) sq[row] = acc;
}

// ------------------------------------------------------------------------------------------------
// average pooling (count_include_pad=True) forward / explain-backward
// ------------------------------------------------------------------------------------------------
// lanes_per_pix = min(32, c/8) (a power of two); a warp covers 32/lanes_per_pix output pixels.
template <typename T, int KT, bool ONE>
__global__ void avgpool_fwd_kernel(const T* __restrict__ x, int nb, int h, int w, int c, int planes, int k_rt, int stride,
                                   int pad, T* __restrict__ y, int op, int oq, float* __restrict__ sq, int lpp) {
  const int k = KT > 0 ? KT : k_rt;   // compile-time window => the tap loops unroll and their loads overlap
  const int lane = threadIdx.x & 31;
  const int img = blockIdx.y;
  const unsigned warp_id = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int ppw = 32 / lpp;  // pixels per warp
  const unsigned ipix = warp_id * ppw + lane / lpp;          // pixel inside the image (32-bit math: no 64-bit divisions)
  const bool valid = ipix < (unsigned)(op * oq);
  const size_t pix = (size_t)img * op * oq + ipix;
  const int sub = lane % lpp;
  float sqacc = 0.f;
  if (valid) {
    const int p = (int)(ipix / (unsigned)oq);
    const int q = (int)(ipix - (unsigned)p * oq);
    const float inv = 1.0f / (float)(k * k);
    const int ld = planes * c;
    for (int g = sub; g < c / 8; g += lpp) {
      float acc[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll
      for (int dy = 0; dy < (KT > 0 ? KT : 1); ++dy) {
#pragma unroll
        for (int dx = 0; dx < (KT > 0 ? KT : 1); ++dx) {
          if (KT > 0) {
            const int yy = p * stride - pad + dy, xx = q * stride - pad + dx;
            if (yy >= 0 && yy < h && xx >= 0 && xx < w) {
              float f[8];
              load8_pl<T, ONE>(x + (((size_t)img * h + yy) * w + xx) * ld + g * 8, planes, c, f);
#pragma unroll
              for (int i = 0; i < 8; ++i) acc[i] += f[i];
            }
          }
        }
      }
      if (KT == 0) {
        for (int dy = 0; dy < k; ++dy) {
          const int yy = p * stride - pad + dy;
          if (yy < 0 || yy >= h) continue;
          for (int dx = 0; dx < k; ++dx) {
            const int xx = q * stride - pad + dx;
            if (xx < 0 || xx >= w) continue;
            float f[8];
            load8_planes<T>(x + (((size_t)img * h + yy) * w + xx) * ld + g * 8, planes, c, f);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] += f[i];
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] *= inv;
      store8_planes<T>(y + (size_t)pix * ld + g * 8, planes, c, acc);
#pragma unroll
      for (int i = 0; i < 8; ++i) sqacc = fmaf(acc[i], acc[i], sqacc);
    }
  }
  if (sq != nullptr) {
    for (int o = lpp >> 1; o > 0; o >>= 1) sqacc += __shfl_xor_sync(0xffffffffu, sqacc, o);
    if (valid && sub == 0) sq[pix] = sqacc;
  }
}

template <typename T, bool ONE>
__global__ void avgpool_bwd_mul_kernel(const T* __restrict__ gy, int nb, int h, int w, int c, int planes, int k,
                                       int stride, int pad, int op, int oq, const void* __restrict__ gain, int gain_f32,
                                       T* __restrict__ gx, int row_pitch, int img_pitch) {
  const int cg = c / 8;
  const int img = blockIdx.y;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;     // (pixel, channel group) inside the image, 32-bit math
  if (idx >= (unsigned)(h * w * cg)) return;
  const unsigned ipix = idx / (unsigned)cg;
  const int g = (int)(idx - ipix * cg);
  const int yy = (int)(ipix / (unsigned)w);
  const int xx = (int)(ipix - (unsigned)yy * w);
  const size_t pix = (size_t)img * h * w + ipix;
  const int ld = planes * c;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  // output rows p with p*stride - pad <= yy <= p*stride - pad + k - 1
  const int p_lo = max(0, (yy + pad - k + 1 + stride - 1) / stride);
  const int p_hi = min(op - 1, (yy + pad) / stride);
  const int q_lo = max(0, (xx + pad - k + 1 + stride - 1) / stride);
  const int q_hi = min(oq - 1, (xx + pad) / stride);
  if (p_hi - p_lo <= 1 && q_hi - q_lo <= 1) {
    // at most 2 x 2 windows cover an input pixel (k <= 2 * stride): unrolled, the loads overlap
#pragma unroll
    for (int dp = 0; dp < 2; ++dp)
#pragma unroll
      for (int dq = 0; dq < 2; ++dq) {
        const int p = p_lo + dp, q = q_lo + dq;
        if (p <= p_hi && q <= q_hi) {
          float f[8];
          load8_pl<T, ONE>(gy + (((size_t)img * op + p) * oq + q) * ld + g * 8, planes, c, f);
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[i] += f[i];
        }
      }
  } else {
    for (int p = p_lo; p <= p_hi; ++p)
      for (int q = q_lo; q <= q_hi; ++q) {
        float f[8];
        load8_planes<T>(gy + (((size_t)img * op + p) * oq + q) * ld + g * 8, planes, c, f);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] += f[i];
      }
  }
  const float inv = 1.0f / (float)(k * k);
  float gn[8];
  if (gain == nullptr) {
#pragma unroll
    for (int i = 0; i < 8; ++i) gn[i] = 1.f;
  } else if (gain_f32) {
    const float4* gp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(gain) + (size_t)pix * c + g * 8);
    const float4 a = __ldg(gp), b = __ldg(gp + 1);
    gn[0] = a.x; gn[1] = a.y; gn[2] = a.z; gn[3] = a.w; gn[4] = b.x; gn[5] = b.y; gn[6] = b.z; gn[7] = b.w;
  } else {
    unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(gain) + (size_t)pix * c + g * 8)), gn);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] *= inv * gn[i];
  store8_planes<T>(gx + ((size_t)img * img_pitch + (size_t)yy * row_pitch + xx) * ld + g * 8, planes, c, acc);
}

// ------------------------------------------------------------------------------------------------
// Row-staged variants (single plane, 16-bit, c/8 a power of two <= 32).  One block per (image, output row) resp.
// (image, input row): whole rows are fetched into shared memory with 1-D bulk copies, so a block has tens of KB in
// flight from a single instruction instead of one 16-byte load per thread and tap (the direct kernels above were
// latency bound at 1.3 / 2.4 TB/s; profiles/r01_pool_kernels.md).  Same arithmetic order as the direct kernels.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
avgpool_fwd_rows_kernel(const T* __restrict__ x, int h, int w, int c, int planes, int k, int stride, int pad, T* __restrict__ y,
                        int op, int oq, float* __restrict__ sq, int split) {
  extern __shared__ __align__(128) uint8_t pool_smem[];
  __shared__ __align__(8) uint64_t bar;
  // `split` CTAs share an output row (each stages only the input pixels its outputs read: more CTAs per SM, more loads in flight)
  const int img = blockIdx.y, p = blockIdx.x / split, part = blockIdx.x - p * split;
  const int ld = planes * c;                               // precision planes side by side in every pixel
  const int q_lo = (int)((long long)oq * part / split), q_hi = (int)((long long)oq * (part + 1) / split);
  const int x_lo = max(0, q_lo * stride - pad), x_hi = min(w, (q_hi - 1) * stride - pad + k);
  const uint32_t row_bytes = (uint32_t)(x_hi - x_lo) * ld * sizeof(T);
  const int y0 = p * stride - pad;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
    uint32_t total = 0;
    for (int dy = 0; dy < k; ++dy)
      if (y0 + dy >= 0 && y0 + dy < h) total += row_bytes;
    mbar_arrive_expect_tx(&bar, total);
    for (int dy = 0; dy < k; ++dy) {
      const int yy = y0 + dy;
      if (yy >= 0 && yy < h) bulk_load_1d(pool_smem + dy * row_bytes, x + (((size_t)img * h + yy) * w + x_lo) * ld, row_bytes, &bar);
    }
  }
  __syncthreads();
  mbar_wait(&bar, 0);
  const int cg = c / 8;
  const float inv = 1.0f / (float)(k * k);
  const int items = (q_hi - q_lo) * cg;
  const int items_pad = (items + 31) & ~31;
  for (int it = threadIdx.x; it < items_pad; it += blockDim.x) {
    const bool valid = it < items;
    const int q = q_lo + it / cg, g = it % cg;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    float sqacc = 0.f;
    if (valid) {
      for (int dy = 0; dy < k; ++dy) {
        if (y0 + dy < 0 || y0 + dy >= h) continue;
        for (int dx = 0; dx < k; ++dx) {
          const int xx = q * stride - pad + dx;
          if (xx < 0 || xx >= w) continue;
          // the tap's fp32 value first (sum of its planes: exact), then the running sum - the order F.avg_pool2d adds in
          float f[8];
          unpack8<T>(*reinterpret_cast<const uint4*>(pool_smem + dy * row_bytes + ((size_t)(xx - x_lo) * ld + g * 8) * sizeof(T)), f);
          for (int pl = 1; pl < planes; ++pl) {
            float f2[8];
            unpack8<T>(*reinterpret_cast<const uint4*>(pool_smem + dy * row_bytes + ((size_t)(xx - x_lo) * ld + pl * c + g * 8) * sizeof(T)), f2);
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] += f2[i];
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[i] += f[i];
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] *= inv;
      store8_planes<T>(y + (((size_t)img * op + p) * oq + q) * ld + g * 8, planes, c, acc);
#pragma unroll
      for (int i = 0; i < 8; ++i) sqacc = fmaf(acc[i], acc[i], sqacc);
    }
    if (sq != nullptr) {
      for (int o = cg >> 1; o > 0; o >>= 1) sqacc += __shfl_xor_sync(0xffffffffu, sqacc, o);
      if (valid && g == 0) sq[((size_t)img * op + p) * oq + q] = sqacc;
    }
  }
}

// gx[yy, :, :] = gain[yy, :, :] * (sum of the <= 2 x 2 output gradients whose windows cover the pixel) / k^2, staged and
// written back as one row.
template <typename T>
__global__ void __launch_bounds__(256)
avgpool_bwd_mul_rows_kernel(const T* __restrict__ gy, int h, int w, int c, int k, int stride, int pad, int op, int oq,
                            const T* __restrict__ gain, T* __restrict__ gx, int row_pitch, int img_pitch,
                            const float* __restrict__ gain_sqrt_scale) {
  extern __shared__ __align__(128) uint8_t pool_smem[];
  __shared__ __align__(8) uint64_t bar;
  const int img = blockIdx.y, yy = blockIdx.x;
  const uint32_t row_bytes = (uint32_t)w * c * sizeof(T);
  const uint32_t grow_bytes = (uint32_t)oq * c * sizeof(T);
  const int p_lo = max(0, (yy + pad - k + 1 + stride - 1) / stride);
  const int p_hi = min(op - 1, (yy + pad) / stride);
  uint8_t* s_gain = pool_smem;                 // [w][c], overwritten with the result
  uint8_t* s_gy = pool_smem + row_bytes;       // [2][oq][c]
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
    mbar_arrive_expect_tx(&bar, row_bytes + (uint32_t)(p_hi - p_lo + 1) * grow_bytes);
    bulk_load_1d(s_gain, gain + ((size_t)img * h + yy) * w * c, row_bytes, &bar);
    for (int p = p_lo; p <= p_hi; ++p)
      bulk_load_1d(s_gy + (p - p_lo) * grow_bytes, gy + ((size_t)img * op + p) * oq * c, grow_bytes, &bar);
  }
  __syncthreads();
  mbar_wait(&bar, 0);
  const int cg = c / 8;
  const float inv = 1.0f / (float)(k * k);
  for (int it = threadIdx.x; it < w * cg; it += blockDim.x) {
    const int xx = it / cg, g = it - xx * cg;
    const int q_lo = max(0, (xx + pad - k + 1 + stride - 1) / stride);
    const int q_hi = min(oq - 1, (xx + pad) / stride);
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    for (int p = p_lo; p <= p_hi; ++p)
      for (int q = q_lo; q <= q_hi; ++q) {
        float f[8];
        unpack8<T>(*reinterpret_cast<const uint4*>(s_gy + (p - p_lo) * grow_bytes + ((size_t)q * c + g * 8) * sizeof(T)), f);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] += f[i];
      }
    uint4* slot = reinterpret_cast<uint4*>(s_gain + ((size_t)xx * c + g * 8) * sizeof(T));
    float gn[8];
    unpack8<T>(*slot, gn);
    if (gain_sqrt_scale != nullptr) {
      // `gain` holds the producer's ReLU output: the multiplier is sqrt(y / ||patch||)
      const float sc = __ldg(gain_sqrt_scale + ((size_t)img * h + yy) * w + xx);
#pragma unroll
      for (int i = 0; i < 8; ++i) gn[i] = fast_sqrt(gn[i] * sc);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] *= inv * gn[i];
    uint4 o;
    o.x = Cvt<T>::pack2(acc[0], acc[1]);
    o.y = Cvt<T>::pack2(acc[2], acc[3]);
    o.z = Cvt<T>::pack2(acc[4], acc[5]);
    o.w = Cvt<T>::pack2(acc[6], acc[7]);
    *slot = o;
  }
  fence_proxy_async_smem();
  __syncthreads();
  if (threadIdx.x == 0) {
    bulk_store_1d(gx + ((size_t)img * img_pitch + (size_t)yy * row_pitch) * c, s_gain, row_bytes);
    tma_store_commit_and_wait_read();
  }
}

// ------------------------------------------------------------------------------------------------
// classifier tail: GAP + logit layer + argmax (one block per image)
// ------------------------------------------------------------------------------------------------
// torch.argmax order: NaN above every number, then the larger value, then the smaller index.  The starting candidate
// (-inf, INT_MAX) loses to every class, so a row of -inf gives 0 and `pred` is always a class index.
__device__ __forceinline__ bool argmax_before(float v, int i, float bv, int bi) {
  const bool vn = v != v, bn = bv != bv;
  if (vn != bn) return vn;
  if (vn || v == bv) return i < bi;
  return v > bv;
}

__global__ void gap_logits_kernel(const float* __restrict__ fc, int npix, int ncls, float inv_temp, float bias,
                                  float* __restrict__ logits, int* __restrict__ pred) {
  const int img = blockIdx.x;
  const float* src = fc + (size_t)img * npix * ncls;
  float best = -INFINITY;
  int best_i = 0x7fffffff;
  const float invn = 1.0f / (float)npix;
  for (int cls = threadIdx.x; cls < ncls; cls += blockDim.x) {
    float acc = 0.f;
    for (int px = 0; px < npix; ++px) acc += __ldg(src + (size_t)px * ncls + cls);
    const float l = acc * invn * inv_temp + bias;
    logits[(size_t)img * ncls + cls] = l;
    if (argmax_before(l, cls, best, best_i)) { best = l; best_i = cls; }
  }
  // block arg-max
  __shared__ float s_v[32];
  __shared__ int s_i[32];
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
    if (argmax_before(ov, oi, best, best_i)) { best = ov; best_i = oi; }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { s_v[warp] = best; s_i[warp] = best_i; }
  __syncthreads();
  if (warp == 0) {
    const int nw = blockDim.x >> 5;
    best = lane < nw ? s_v[lane] : -INFINITY;
    best_i = lane < nw ? s_i[lane] : 0x7fffffff;
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
      if (argmax_before(ov, oi, best, best_i)) { best = ov; best_i = oi; }
    }
    if (lane == 0 && pred != nullptr) pred[img] = best_i;
  }
}

// ------------------------------------------------------------------------------------------------
// explain seed through GAP + classifier for a one-hot logit gradient
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void fc_seed_dgrad_kernel(const int* __restrict__ target, const void* __restrict__ gain_fc, int gain_f32,
                                     const float* __restrict__ w_fc, int nb, int npix, int ncls, int c, float coef,
                                     const void* __restrict__ mul1, int mul1_f32, T* __restrict__ out1,
                                     const uint32_t* __restrict__ mask2, T* __restrict__ out2, int planes) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int cg = c / 8;
  const long long total = (long long)nb * npix * cg;
  if (idx >= total) return;
  const int g = (int)(idx % cg);
  const long long row = idx / cg;  // img * npix + pix
  const int img = (int)(row / npix);
  const int cls = __ldg(target + img);
  float gf;
  if (gain_f32) gf = __ldg(reinterpret_cast<const float*>(gain_fc) + (size_t)row * ncls + cls);
  else gf = Cvt<T>::unpack2((uint32_t)__ldg(reinterpret_cast<const uint16_t*>(gain_fc) + (size_t)row * ncls + cls)).x;
  const float s = coef * gf;
  const float4* wp = reinterpret_cast<const float4*>(w_fc + (size_t)cls * c + g * 8);
  const float4 wa = __ldg(wp), wb = __ldg(wp + 1);
  float v[8] = {s * wa.x, s * wa.y, s * wa.z, s * wa.w, s * wb.x, s * wb.y, s * wb.z, s * wb.w};
  const int ld = planes * c;
  if (out2 != nullptr) {
    float o[8];
    const uint32_t mb = mask2 ? __ldg(mask2 + (size_t)row * ((c + 31) / 32) + (g >> 2)) : 0xffffffffu;
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = ((mb >> ((g & 3) * 8 + i)) & 1u) ? v[i] : 0.f;
    store8_planes<T>(out2 + (size_t)row * ld + g * 8, planes, c, o);
  }
  if (mul1 != nullptr) {
    float gn[8];
    if (mul1_f32) {
      const float4* gp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(mul1) + (size_t)row * c + g * 8);
      const float4 a = __ldg(gp), b = __ldg(gp + 1);
      gn[0] = a.x; gn[1] = a.y; gn[2] = a.z; gn[3] = a.w; gn[4] = b.x; gn[5] = b.y; gn[6] = b.z; gn[7] = b.w;
    } else {
      unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(mul1) + (size_t)row * c + g * 8)), gn);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] *= gn[i];
  }
  store8_planes<T>(out1 + (size_t)row * ld + g * 8, planes, c, v);
}

// ------------------------------------------------------------------------------------------------
// contribution map from the stem dgrad (space-to-depth layout)
// ------------------------------------------------------------------------------------------------
struct InvStd6 { float v[6]; };

template <typename SRC>
__global__ void contrib_map_s2d_kernel(const float* __restrict__ g, const SRC* __restrict__ x, int nb, int h, int w,
                                       int cp, InvStd6 is, float out_scale, float* __restrict__ cmap,
                                       float* __restrict__ grad6) {
  const int h2 = h >> 1, w2 = w >> 1;
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;        // 32-bit index math, the image on blockIdx.y
  if (pix >= h2 * w2) return;
  const int r = pix / w2;
  const int s = pix - r * w2;
  const int img = blockIdx.y;
  const float4* gp = reinterpret_cast<const float4*>(g + ((size_t)img * h2 * w2 + pix) * cp);
  float gv[24];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const float4 a = __ldg(gp + i);
    gv[4 * i] = a.x; gv[4 * i + 1] = a.y; gv[4 * i + 2] = a.z; gv[4 * i + 3] = a.w;
  }
  float xv[24];
  load_patch6<SRC>(x, img, r, s, h, w, xv);
  const size_t plane = (size_t)h * w;
  float cm[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const size_t off = ((size_t)img * 6 + c) * plane + (size_t)(2 * r) * w + 2 * s;
    const float k = is.v[c] * out_scale;
    const float g0 = gv[0 * 6 + c] * k, g1 = gv[1 * 6 + c] * k, g2 = gv[2 * 6 + c] * k, g3 = gv[3 * 6 + c] * k;
    cm[0] = fmaf(xv[0 * 6 + c], g0, cm[0]);
    cm[1] = fmaf(xv[1 * 6 + c], g1, cm[1]);
    cm[2] = fmaf(xv[2 * 6 + c], g2, cm[2]);
    cm[3] = fmaf(xv[3 * 6 + c], g3, cm[3]);
    if (grad6 != nullptr) {
      *reinterpret_cast<float2*>(grad6 + off) = make_float2(g0, g1);
      *reinterpret_cast<float2*>(grad6 + off + w) = make_float2(g2, g3);
    }
  }
  float* cp_out = cmap + (size_t)img * plane + (size_t)(2 * r) * w + 2 * s;
  *reinterpret_cast<float2*>(cp_out) = make_float2(cm[0], cm[1]);
  *reinterpret_cast<float2*>(cp_out + w) = make_float2(cm[2], cm[3]);
}

// ------------------------------------------------------------------------------------------------
// generic element-wise helpers
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void channel_affine_kernel(const T* __restrict__ x, long long rows, int c, const float* __restrict__ alpha,
                                      const float* __restrict__ beta, int relu, T* __restrict__ y) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int cg = c / 8;
  if (idx >= rows * cg) return;
  const int g = (int)(idx % cg);
  float f[8];
  unpack8<T>(__ldg(reinterpret_cast<const uint4*>(x) + idx), f);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float a = alpha ? __ldg(alpha + g * 8 + i) : 1.f;
    const float b = beta ? __ldg(beta + g * 8 + i) : 0.f;
    float v = fmaf(f[i], a, b);
    f[i] = (relu && v < 0.f) ? 0.f : v;
  }
  reinterpret_cast<uint4*>(y)[idx] = pack8<T>(f);
}

template <typename T>
__global__ void mul_kernel(const T* __restrict__ a, const T* __restrict__ b, long long n8, T* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n8) return;
  float fa[8], fb[8];
  unpack8<T>(__ldg(reinterpret_cast<const uint4*>(a) + idx), fa);
  unpack8<T>(__ldg(reinterpret_cast<const uint4*>(b) + idx), fb);
#pragma unroll
  for (int i = 0; i < 8; ++i) fa[i] *= fb[i];
  reinterpret_cast<uint4*>(out)[idx] = pack8<T>(fa);
}

}  // namespace bcosk

using namespace bcosk;

#define BCOSK_DTYPE_SWITCH(dtype, ...)                                              \
  if ((dtype) == BCOSK_DTYPE_BF16) { using T = __nv_bfloat16; __VA_ARGS__ }         \
  else if ((dtype) == BCOSK_DTYPE_F16) { using T = __half; __VA_ARGS__ }            \
  else return set_error(BCOSK_EINVAL, "bad dtype %d", (int)(dtype));

static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

template <typename SRC>
static int input_prep_impl(const SRC* x, int32_t nb, int32_t h, int32_t w, const float* mean6, const float* inv_std6,
                           void* out, int32_t cp, int32_t planes, int32_t dtype, float* sq, int32_t row_pitch,
                           int32_t img_pitch, void* stream) {
  if (!x || !out || !mean6 || !inv_std6) return set_error(BCOSK_EINVAL, "input_prep: null pointer");
  if (row_pitch == 0) row_pitch = w / 2;
  if (img_pitch == 0) img_pitch = (h / 2) * row_pitch;
  if (row_pitch < w / 2 || img_pitch < (h / 2) * row_pitch) return set_error(BCOSK_EINVAL, "input_prep: bad output pitch");
  if (h % 2 || w % 2 || cp < 24 || cp % 8) return set_error(BCOSK_EINVAL, "input_prep: need even h,w and cp>=24, cp%%8==0");
  Norm6 nm;
  for (int i = 0; i < 6; ++i) { nm.mean[i] = mean6[i]; nm.inv_std[i] = inv_std6[i]; }  // host pointers
  if (nb < 1 || nb > 65535) return set_error(BCOSK_EINVAL, "input_prep: batch must be in [1, 65535]");
  const dim3 grid((unsigned)(((h / 2) * (w / 2) + 255) / 256), (unsigned)nb);
  BCOSK_DTYPE_SWITCH(dtype, input_prep_s2d_kernel<T, SRC><<<grid, 256, 0, S(stream)>>>(
      x, nb, h, w, nm, reinterpret_cast<T*>(out), cp, planes, sq, row_pitch, img_pitch);)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_input_prep_s2d(const float* x, int32_t nb, int32_t h, int32_t w, const float* mean6,
                                    const float* inv_std6, void* out, int32_t cp, int32_t planes, int32_t dtype, float* sq,
                                    int32_t out_row_pitch, int32_t out_img_pitch, void* stream) {
  return input_prep_impl<float>(x, nb, h, w, mean6, inv_std6, out, cp, planes, dtype, sq, out_row_pitch, out_img_pitch, stream);
}

extern "C" int bcosk_input_prep_s2d_u8(const uint8_t* x, int32_t nb, int32_t h, int32_t w, const float* mean6,
                                       const float* inv_std6, void* out, int32_t cp, int32_t planes, int32_t dtype,
                                       float* sq, int32_t out_row_pitch, int32_t out_img_pitch, void* stream) {
  return input_prep_impl<uint8_t>(x, nb, h, w, mean6, inv_std6, out, cp, planes, dtype, sq, out_row_pitch, out_img_pitch,
                                  stream);
}

extern "C" int bcosk_patch_inv_norm(const float* sq, int32_t parts, int32_t nb, int32_t h, int32_t w, int32_t kh,
                                    int32_t kw, int32_t stride, int32_t pad, float eps_in, float eps_out, float* inv_norm,
                                    int32_t op, int32_t oq, void* stream) {
  if (!sq || !inv_norm || parts < 1) return set_error(BCOSK_EINVAL, "patch_inv_norm: bad argument");
  if (nb > 65535) return set_error(BCOSK_EUNSUPPORTED, "patch_inv_norm: batch too large for the grid");
  const int th = (PN_TILE - 1) * stride + kh, tw = (PN_TILE - 1) * stride + kw;
  const size_t smem = (size_t)th * tw * sizeof(float);
  if (smem > 48 * 1024) return set_error(BCOSK_EUNSUPPORTED, "patch_inv_norm: window too large");
  dim3 grid((oq + PN_TILE - 1) / PN_TILE, (op + PN_TILE - 1) / PN_TILE, nb);
  patch_inv_norm_kernel<<<grid, PN_TILE * PN_TILE, smem, S(stream)>>>(sq, parts, nb, h, w, kh, kw, stride, pad, eps_in,
                                                                        eps_out, inv_norm, op, oq);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_pixel_sqsum(const void* x, int64_t rows, int32_t c, int32_t planes, int32_t plane_stride, int32_t ld,
                                 int32_t dtype, float* sq, void* stream) {
  if (!x || !sq || c % 8) return set_error(BCOSK_EINVAL, "pixel_sqsum: bad argument");
  BCOSK_DTYPE_SWITCH(dtype, pixel_sqsum_kernel<T><<<blocks_for(rows, 8), 256, 0, S(stream)>>>(
      reinterpret_cast<const T*>(x), rows, c, planes, plane_stride, ld, sq);)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

// lanes that share one pixel in the direct pooling kernels: the largest power of two <= min(32, c / 8); every lane walks the 8-channel
// groups g = lane, lane + lanes, ... < c / 8 (any channel count that is a multiple of 8: DenseNet-169 / -201 transitions have 320 / 448)
static int lanes_per_pixel(int c) {
  const int g = c / 8;
  if (c % 8 || g < 1) return 0;
  int l = 1;
  while (l * 2 <= g && l * 2 <= 32) l *= 2;
  return l;
}

extern "C" int bcosk_avgpool_fwd(const void* x, int32_t nb, int32_t h, int32_t w, int32_t c, int32_t planes, int32_t k,
                                 int32_t stride, int32_t pad, void* y, int32_t op, int32_t oq, int32_t dtype, float* sq,
                                 void* stream) {
  const int lpp = lanes_per_pixel(c);
  if (!x || !y || lpp == 0) return set_error(BCOSK_EUNSUPPORTED, "avgpool_fwd: c must be a positive multiple of 8");
  if (nb > 65535) return set_error(BCOSK_EUNSUPPORTED, "avgpool_fwd: batch too large for the grid");
  if (op < 1 || oq < 1) return set_error(BCOSK_EINVAL, "avgpool_fwd: empty output");
  {
    // row-staged kernel: <= 32 lanes per pixel, k full input rows (all planes) fit shared memory
    const size_t smem_row = (size_t)k * w * planes * c * 2;
    if (c / 8 <= 32 && (c / 8 & (c / 8 - 1)) == 0 && c % 8 == 0 && smem_row <= 100 * 1024 && op <= 32767) {
      // long rows: two or three CTAs per output row (<= ~44 KB each: five CTAs per SM instead of two); never more parts than
      // output columns, or a part would own no column and stage a negative input range (a global 7 x 7 pool has oq = 1)
      int split = smem_row > 88 * 1024 ? 3 : (smem_row > 44 * 1024 ? 2 : 1);
      if (split > oq) split = oq;
      const int span = ((oq + split - 1) / split - 1) * stride + k + stride;          // input pixels one part reads (upper bound)
      size_t smem = (size_t)k * (span < w ? span : w) * planes * c * 2;
      if (smem > 48 * 1024) {
        BCOSK_DTYPE_SWITCH(dtype, BCOSK_CUDA_CHECK(cudaFuncSetAttribute(avgpool_fwd_rows_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                                         100 * 1024));)
      }
      BCOSK_DTYPE_SWITCH(dtype, avgpool_fwd_rows_kernel<T><<<dim3(op * split, nb), 256, smem, S(stream)>>>(
          reinterpret_cast<const T*>(x), h, w, c, planes, k, stride, pad, reinterpret_cast<T*>(y), op, oq, sq, split);)
      BCOSK_CUDA_CHECK(cudaGetLastError());
      return BCOSK_OK;
    }
  }
  const long long pix = (long long)op * oq;                       // per image; grid.y walks the images
  const long long warps = (pix + (32 / lpp) - 1) / (32 / lpp);
  const dim3 pgrid(blocks_for(warps, 8), nb);
#define BCOSK_POOL_FWD(KT_, ONE_)                                                                                      \
  BCOSK_DTYPE_SWITCH(dtype, avgpool_fwd_kernel<T, KT_, ONE_><<<pgrid, 256, 0, S(stream)>>>(                                \
      reinterpret_cast<const T*>(x), nb, h, w, c, planes, k, stride, pad, reinterpret_cast<T*>(y), op, oq, sq, lpp);)
  if (k == 3 && planes == 1) { BCOSK_POOL_FWD(3, true) }
  else if (k == 3) { BCOSK_POOL_FWD(3, false) }
  else if (k == 2 && planes == 1) { BCOSK_POOL_FWD(2, true) }
  else if (k == 2) { BCOSK_POOL_FWD(2, false) }
  else { BCOSK_POOL_FWD(0, false) }
#undef BCOSK_POOL_FWD
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_avgpool_bwd_mul(const void* gy, int32_t nb, int32_t h, int32_t w, int32_t c, int32_t planes, int32_t k,
                                     int32_t stride, int32_t pad, int32_t op, int32_t oq, const void* gain, int32_t gain_f32,
                                     void* gx, int32_t dtype, int32_t row_pitch, int32_t img_pitch,
                                     const float* gain_sqrt_scale, void* stream) {
  if (!gy || !gx || c % 8) return set_error(BCOSK_EINVAL, "avgpool_bwd_mul: bad argument");
  if (row_pitch == 0) row_pitch = w;
  if (img_pitch == 0) img_pitch = h * row_pitch;
  if (row_pitch < w || img_pitch < h * row_pitch) return set_error(BCOSK_EINVAL, "avgpool_bwd_mul: bad output pitch");
  if (nb > 65535) return set_error(BCOSK_EUNSUPPORTED, "avgpool_bwd_mul: batch too large for the grid");
  {
    // row-staged kernel: single plane, 16-bit gain, at most two output rows cover an input row (k <= 2 * stride)
    const size_t smem = ((size_t)w + 2 * (size_t)oq) * c * 2;
    if (planes == 1 && gain != nullptr && !gain_f32 && k <= 2 * stride && smem <= 48 * 1024 && h <= 65535) {
      BCOSK_DTYPE_SWITCH(dtype, avgpool_bwd_mul_rows_kernel<T><<<dim3(h, nb), 256, smem, S(stream)>>>(
          reinterpret_cast<const T*>(gy), h, w, c, k, stride, pad, op, oq, reinterpret_cast<const T*>(gain),
          reinterpret_cast<T*>(gx), row_pitch, img_pitch, gain_sqrt_scale);)
      BCOSK_CUDA_CHECK(cudaGetLastError());
      return BCOSK_OK;
    }
  }
  if (gain_sqrt_scale != nullptr)
    return set_error(BCOSK_EUNSUPPORTED, "avgpool_bwd_mul: gain_sqrt_scale needs the row-staged path (one 16-bit plane, k <= 2*stride)");
  const long long n = (long long)h * w * (c / 8);
  const dim3 bgrid(blocks_for(n, 256), nb);
  if (planes == 1) {
    BCOSK_DTYPE_SWITCH(dtype, avgpool_bwd_mul_kernel<T, true><<<bgrid, 256, 0, S(stream)>>>(
        reinterpret_cast<const T*>(gy), nb, h, w, c, planes, k, stride, pad, op, oq, gain, gain_f32, reinterpret_cast<T*>(gx),
        row_pitch, img_pitch);)
  } else {
    BCOSK_DTYPE_SWITCH(dtype, avgpool_bwd_mul_kernel<T, false><<<bgrid, 256, 0, S(stream)>>>(
        reinterpret_cast<const T*>(gy), nb, h, w, c, planes, k, stride, pad, op, oq, gain, gain_f32, reinterpret_cast<T*>(gx),
        row_pitch, img_pitch);)
  }
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_gap_logits(const float* fc, int32_t nb, int32_t npix, int32_t ncls, float inv_temp, float bias,
                                float* logits, int32_t* pred, void* stream) {
  if (!fc || !logits) return set_error(BCOSK_EINVAL, "gap_logits: null pointer");
  if (nb < 1 || npix < 1 || ncls < 1) return set_error(BCOSK_EINVAL, "gap_logits: bad shape");
  gap_logits_kernel<<<nb, 256, 0, S(stream)>>>(fc, npix, ncls, inv_temp, bias, logits, pred);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_fc_seed_dgrad(const int32_t* target, const void* gain_fc, int32_t gain_f32, const float* w_fc,
                                   int32_t nb, int32_t npix, int32_t ncls, int32_t c, float inv_temp, float seed_scale,
                                   const void* mul1, int32_t mul1_f32, void* out1, const uint32_t* mask2, void* out2,
                                   int32_t planes, int32_t dtype, void* stream) {
  if (!target || !gain_fc || !w_fc || !out1 || c % 8) return set_error(BCOSK_EINVAL, "fc_seed_dgrad: bad argument");
  const long long n = (long long)nb * npix * (c / 8);
  const float coef = inv_temp * seed_scale / (float)npix;
  BCOSK_DTYPE_SWITCH(dtype, fc_seed_dgrad_kernel<T><<<blocks_for(n, 256), 256, 0, S(stream)>>>(
      target, gain_fc, gain_f32, w_fc, nb, npix, ncls, c, coef, mul1, mul1_f32, reinterpret_cast<T*>(out1), mask2,
      reinterpret_cast<T*>(out2), planes);)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

template <typename SRC>
static int contrib_map_impl(const float* g, const SRC* x, int32_t nb, int32_t h, int32_t w, int32_t cp,
                            const float* inv_std6, float out_scale, float* cmap, float* grad6, void* stream) {
  if (!g || !x || !cmap || !inv_std6 || cp < 24 || cp % 4) return set_error(BCOSK_EINVAL, "contrib_map: bad argument");
  // one thread per 2x2 block, written with float2 stores: an odd size would leave the last row / column unwritten
  if (h < 2 || w < 2 || h % 2 || w % 2) return set_error(BCOSK_EINVAL, "contrib_map: need even h, w (as input_prep)");
  InvStd6 is;
  for (int i = 0; i < 6; ++i) is.v[i] = inv_std6[i];
  if (nb < 1 || nb > 65535) return set_error(BCOSK_EINVAL, "contrib_map: batch must be in [1, 65535]");
  const dim3 grid((unsigned)(((h / 2) * (w / 2) + 255) / 256), (unsigned)nb);
  contrib_map_s2d_kernel<SRC><<<grid, 256, 0, S(stream)>>>(g, x, nb, h, w, cp, is, out_scale, cmap, grad6);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_contrib_map_s2d(const float* g, const float* x, int32_t nb, int32_t h, int32_t w, int32_t cp,
                                     const float* inv_std6, float out_scale, float* cmap, float* grad6, void* stream) {
  return contrib_map_impl<float>(g, x, nb, h, w, cp, inv_std6, out_scale, cmap, grad6, stream);
}

extern "C" int bcosk_contrib_map_s2d_u8(const float* g, const uint8_t* x, int32_t nb, int32_t h, int32_t w, int32_t cp,
                                        const float* inv_std6, float out_scale, float* cmap, float* grad6, void* stream) {
  return contrib_map_impl<uint8_t>(g, x, nb, h, w, cp, inv_std6, out_scale, cmap, grad6, stream);
}

extern "C" int bcosk_channel_affine(const void* x, int64_t rows, int32_t c, const float* alpha, const float* beta,
                                    int32_t relu, void* y, int32_t dtype, void* stream) {
  if (!x || !y || c % 8) return set_error(BCOSK_EINVAL, "channel_affine: bad argument");
  const long long n = rows * (c / 8);
  BCOSK_DTYPE_SWITCH(dtype, channel_affine_kernel<T><<<blocks_for(n, 256), 256, 0, S(stream)>>>(
      reinterpret_cast<const T*>(x), rows, c, alpha, beta, relu, reinterpret_cast<T*>(y));)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_mul(const void* a, const void* b, int64_t n, void* out, int32_t dtype, void* stream) {
  if (!a || !b || !out || n % 8) return set_error(BCOSK_EINVAL, "mul: bad argument");
  BCOSK_DTYPE_SWITCH(dtype, mul_kernel<T><<<blocks_for(n / 8, 256), 256, 0, S(stream)>>>(
      reinterpret_cast<const T*>(a), reinterpret_cast<const T*>(b), n / 8, reinterpret_cast<T*>(out));)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}
