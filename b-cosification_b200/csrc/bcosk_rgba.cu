// RGBA explanation images from dynamic linear weights, on the device, for whole batches.
// Replaces gradient_to_image (bcos/common.py:387-436): per pixel colour from the normalised, clamped weight vector,
// alpha = ||w||_2 where the contribution is non-negative, smooth x smooth box filter (zero padded, divided by smooth^2
// like F.avg_pool2d with count_include_pad), division by the per-image alpha percentile (torch.quantile, linear
// interpolation between the two neighbouring order statistics) and clipping to [0, 1].
#include <cstdint>

#include "../../include/bcosk.h"
#include "bcosk_host.h"

namespace bcosk {

static inline cudaStream_t S2(void* s) { return reinterpret_cast<cudaStream_t>(s); }

__device__ __forceinline__ float x6_value(const float* x, size_t img, int c, size_t plane, size_t pix) {
  return __ldg(x + (img * 6 + c) * plane + pix);
}
__device__ __forceinline__ float x6_value(const uint8_t* x, size_t img, int c, size_t plane, size_t pix) {
  const float v = (float)__ldg(x + (img * 3 + (c % 3)) * plane + pix) / 255.0f;
  return c < 3 ? v : 1.0f - v;                       // AddInverse (bcos/data/transforms.py:42-55)
}

// colour + raw alpha per pixel (common.py:412-428)
template <typename SRC>
__global__ void rgba_pixel_kernel(const float* __restrict__ g, const SRC* __restrict__ x, int h, int w,
                                  float* __restrict__ out, float* __restrict__ alpha0) {
  const size_t plane = (size_t)h * w;
  const size_t img = blockIdx.y;
  const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= plane) return;
  float gv[6];
  float contrib = 0.f, maxabs = 0.f, sq = 0.f;
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    gv[c] = __ldg(g + (img * 6 + c) * plane + pix);
    contrib += x6_value(x, img, c, plane, pix) * gv[c];
    maxabs = fmaxf(maxabs, fabsf(gv[c]));
    sq += gv[c] * gv[c];
  }
  float r[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) r[c] = fmaxf(gv[c] / (maxabs + 1e-12f), 0.f);
  float* o = out + (img * plane + pix) * 4;
#pragma unroll
  for (int c = 0; c < 3; ++c) o[c] = r[c] / (r[c] + r[c + 3] + 1e-12f);
  alpha0[img * plane + pix] = contrib < 0.f ? 1e-12f : sqrtf(sq);
}

// one direction of the box filter (zero padded); the second pass also divides by smooth^2
__global__ void box_filter_kernel(const float* __restrict__ src, int h, int w, int radius, int vertical, float scale,
                                  float* __restrict__ dst) {
  const size_t plane = (size_t)h * w;
  const size_t img = blockIdx.y;
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= (int)plane) return;
  const int y = pix / w, xx = pix - y * w;
  const float* s = src + img * plane;
  float acc = 0.f;
  for (int d = -radius; d <= radius; ++d) {
    const int yy = vertical ? y + d : y, xq = vertical ? xx : xx + d;
    if (yy >= 0 && yy < h && xq >= 0 && xq < w) acc += __ldg(s + (size_t)yy * w + xq);
  }
  dst[img * plane + pix] = acc * scale;
}

// torch.quantile(alpha, q) per image: radix select of the order statistics k = floor(q (n-1)) and k + 1 over the
// (non-negative) float bit patterns, 8 bits per pass, one block per image; then linear interpolation.
__global__ void __launch_bounds__(1024) alpha_quantile_kernel(const float* __restrict__ alpha, int n, float q,
                                                               float* __restrict__ qv) {
  __shared__ unsigned int hist[256];
  __shared__ unsigned int s_prefix, s_rank;
  const uint32_t* a = reinterpret_cast<const uint32_t*>(alpha) + (size_t)blockIdx.x * n;
  const float pos = q * (float)(n - 1);
  const int k = (int)floorf(pos);
  const float frac = pos - (float)k;
  float vals[2];
  for (int which = 0; which < 2; ++which) {
    const int rank0 = min(k + which, n - 1);
    if (threadIdx.x == 0) { s_prefix = 0u; s_rank = (unsigned)rank0; }
    for (int shift = 24; shift >= 0; shift -= 8) {
      for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0u;
      __syncthreads();
      const unsigned prefix = s_prefix;
      const unsigned mask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const unsigned v = a[i];
        if ((v & mask) == prefix) atomicAdd(&hist[(v >> shift) & 0xffu], 1u);
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        unsigned rank = s_rank, cum = 0;
        int b = 0;
        for (; b < 256; ++b) {
          if (cum + hist[b] > rank) break;
          cum += hist[b];
        }
        s_prefix = prefix | ((unsigned)b << shift);
        s_rank = rank - cum;
      }
      __syncthreads();
    }
    vals[which] = __uint_as_float(s_prefix);
    __syncthreads();
  }
  if (threadIdx.x == 0) qv[blockIdx.x] = vals[0] + (vals[1] - vals[0]) * frac;   // torch lerp(lower, upper, weight)
}

__global__ void rgba_finalize_kernel(const float* __restrict__ alpha, const float* __restrict__ qv, int plane,
                                     float* __restrict__ out) {
  const size_t img = blockIdx.y;
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= plane) return;
  const float a = alpha[img * plane + pix] / qv[img];
  // torch.clamp keeps NaN: a zero quantile over zero alpha (an all-zero gradient image) is 0/0 in the reference too
  out[(img * plane + pix) * 4 + 3] = a != a ? a : fminf(fmaxf(a, 0.f), 1.f);
}

template <typename SRC>
static int rgba_impl(const float* grad6, const SRC* x, int nb, int h, int w, int smooth, float percentile, float* tmp,
                     float* out, void* stream) {
  if (!grad6 || !x || !tmp || !out) return set_error(BCOSK_EINVAL, "explanation_rgba: null pointer");
  if (nb < 1 || nb > 65535 || h < 1 || w < 1) return set_error(BCOSK_EINVAL, "explanation_rgba: bad shape");
  if (smooth < 0 || (smooth > 0 && smooth % 2 == 0))
    return set_error(BCOSK_EUNSUPPORTED, "explanation_rgba: the smoothing window must be odd (0 = none)");
  if (!(percentile >= 0.f && percentile <= 100.f)) return set_error(BCOSK_EINVAL, "explanation_rgba: percentile");
  const int plane = h * w;
  float* a0 = tmp;
  float* a1 = tmp + (size_t)nb * plane;
  float* qv = tmp + 2 * (size_t)nb * plane;
  const dim3 grid((plane + 255) / 256, nb);
  rgba_pixel_kernel<SRC><<<grid, 256, 0, S2(stream)>>>(grad6, x, h, w, out, a0);
  const float* smoothed = a0;
  if (smooth > 1) {
    box_filter_kernel<<<grid, 256, 0, S2(stream)>>>(a0, h, w, smooth / 2, 0, 1.0f, a1);
    box_filter_kernel<<<grid, 256, 0, S2(stream)>>>(a1, h, w, smooth / 2, 1, 1.0f / (float)(smooth * smooth), a0);
    smoothed = a0;
  }
  alpha_quantile_kernel<<<nb, 1024, 0, S2(stream)>>>(smoothed, plane, percentile / 100.0f, qv);
  rgba_finalize_kernel<<<grid, 256, 0, S2(stream)>>>(smoothed, qv, plane, out);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}


// ------------------------------------------------------------------------------------------------
// Localisation ("grid pointing game") scores: interpretability/analyses/localisation.py:306-388.
// attributions [T, C, H, W] (x * grad per target of a grid image) -> channel sum -> smooth x smooth box average (zero
// padded, stride 1) -> optional sign flip -> clamp(min = 0) -> mean over each cell x cell region -> fraction of the
// total per target, 0 where total * contrib <= 0.  Region r of the output is column-major (col * rows + row), the order
// `.permute(0, 1, 3, 2).reshape(T, -1)` produces.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void channel_sum_kernel(const float* __restrict__ a, int c, int plane, float* __restrict__ out) {
  const size_t img = blockIdx.y;
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= plane) return;
  const float* s = a + img * (size_t)c * plane + pix;
  float acc = 0.f;
  for (int ch = 0; ch < c; ++ch) acc += __ldg(s + (size_t)ch * plane);
  out[img * plane + pix] = acc;
}

// one block per (region, target): mean over the region of max(sign * v, 0)
__global__ void __launch_bounds__(256) region_mean_kernel(const float* __restrict__ a, int h, int w, int cell, int rows, int cols,
                                                          float sign, float* __restrict__ raw) {
  __shared__ float red[8];
  const int r = blockIdx.x, t = blockIdx.y;
  const int col = r / rows, row = r - col * rows;            // column-major region index
  const float* s = a + (size_t)t * h * w + (size_t)row * cell * w + (size_t)col * cell;
  float acc = 0.f;
  for (int i = threadIdx.x; i < cell * cell; i += 256) {
    const int y = i / cell, x = i - y * cell;
    acc += fmaxf(sign * __ldg(s + (size_t)y * w + x), 0.f);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) raw[(size_t)t * rows * cols + r] = v / (float)(cell * cell);
  }
}

// one warp per target: contribs / total where total * contrib > 0, else 0
__global__ void region_fraction_kernel(const float* __restrict__ raw, int nt, int regions, float* __restrict__ out) {
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= nt) return;
  const int lane = threadIdx.x & 31;
  float s = 0.f;
  for (int r = lane; r < regions; r += 32) s += __ldg(raw + (size_t)t * regions + r);
  const float total = warp_sum(s);
  for (int r = lane; r < regions; r += 32) {
    const float v = __ldg(raw + (size_t)t * regions + r);
    out[(size_t)t * regions + r] = total * v > 0.f ? v / total : 0.f;
  }
}

}  // namespace bcosk

using namespace bcosk;

extern "C" int bcosk_explanation_rgba(const float* grad6, const float* x, int32_t nb, int32_t h, int32_t w, int32_t smooth,
                                      float percentile, float* tmp, float* out, void* stream) {
  return rgba_impl<float>(grad6, x, nb, h, w, smooth, percentile, tmp, out, stream);
}

extern "C" int bcosk_explanation_rgba_u8(const float* grad6, const uint8_t* x, int32_t nb, int32_t h, int32_t w,
                                         int32_t smooth, float percentile, float* tmp, float* out, void* stream) {
  return rgba_impl<uint8_t>(grad6, x, nb, h, w, smooth, percentile, tmp, out, stream);
}

extern "C" int bcosk_localisation_scores(const float* attr, int32_t nt, int32_t c, int32_t h, int32_t w, int32_t smooth,
                                         int32_t cell, int32_t negate, float* tmp, float* out, void* stream) {
  if (!attr || !tmp || !out) return set_error(BCOSK_EINVAL, "localisation_scores: null pointer");
  if (nt < 1 || nt > 65535 || c < 1 || h < 1 || w < 1 || cell < 1 || cell > h || cell > w)
    return set_error(BCOSK_EINVAL, "localisation_scores: bad shape");
  if (smooth < 0 || (smooth > 0 && smooth % 2 == 0))
    return set_error(BCOSK_EUNSUPPORTED, "localisation_scores: the smoothing window must be odd (0 = none)");
  const int plane = h * w, rows = h / cell, cols = w / cell, regions = rows * cols;
  float* a0 = tmp;
  float* a1 = tmp + (size_t)nt * plane;
  float* raw = tmp + 2 * (size_t)nt * plane;
  const dim3 grid((plane + 255) / 256, nt);
  channel_sum_kernel<<<grid, 256, 0, S2(stream)>>>(attr, c, plane, a0);
  if (smooth > 1) {
    box_filter_kernel<<<grid, 256, 0, S2(stream)>>>(a0, h, w, smooth / 2, 0, 1.0f, a1);
    box_filter_kernel<<<grid, 256, 0, S2(stream)>>>(a1, h, w, smooth / 2, 1, 1.0f / (float)(smooth * smooth), a0);
  }
  region_mean_kernel<<<dim3(regions, nt), 256, 0, S2(stream)>>>(a0, h, w, cell, rows, cols, negate ? -1.f : 1.f, raw);
  region_fraction_kernel<<<(nt + 7) / 8, 256, 0, S2(stream)>>>(raw, nt, regions, out);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}
