// bcosk_dense_train.cu -- bandwidth kernels of the DenseNet fine-tuning step (engine/train.py DenseNetTrainPlan), sm_100a.
//
// A dense block keeps ONE feature tensor F [rows][C_total] (16-bit); layer l's 3x3 conv writes its slice, and every consumer
// (dense-layer norm1, transition norm, norm5) normalises a prefix F[:, :C_l] with the BATCH statistics of those channels
// (batchnorm_uncentered.py:36-43: centred biased variance, uncentred output x * w * rstd).  The statistics of a channel do not
// depend on the consumer, so they are computed once, when the slice is written:
//
//   forward   dense_slice_stats          mean, var, rstd of F[:, col0 : col0 + c]           (after the block-input copy and every 3x3)
//             dense_consumer_finalize    alpha_l = w_l * rstd, running_var_l EMA            (then bcosk_dense_bn_relu_fwd applies it)
//   backward  dense_consumer_bwd         g_y = (g_t + t * gnT) * [t > 0];  G[:, :C_l] += g_y * alpha_l;  partials of S_l = sum g_y * F
//             dense_consumer_bwd_finalize  g_w = S_l * rstd;  K += k_l = -rstd^3 w_l S_l / M
//             dense_slice_bwd            g_out = G[:, slice] + (F[:, slice] - mean) * K -> g_lin = 2 s g_out and gnT (a 3x3 slice),
//                                        or g_out itself (the block's input channels)
// The batch-statistics term of consumer l is linear in (F - mean), so the consumers only add their k_l into K and the producer of
// the slice applies the sum once: one fused pass per consumer.  Per-block partials in a fixed order, no atomics.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "../../include/bcosk.h"
#include "bcosk_common.cuh"
#include "bcosk_host.h"

namespace bcosk {
namespace {

template <typename T>
__device__ __forceinline__ void dt_unpack8(const uint4& u, float (&f)[8]) {
  float2 a;
  a = Cvt<T>::unpack2(u.x); f[0] = a.x; f[1] = a.y;
  a = Cvt<T>::unpack2(u.y); f[2] = a.x; f[3] = a.y;
  a = Cvt<T>::unpack2(u.z); f[4] = a.x; f[5] = a.y;
  a = Cvt<T>::unpack2(u.w); f[6] = a.x; f[7] = a.y;
}
template <typename T>
__device__ __forceinline__ uint4 dt_pack8(const float (&f)[8]) {
  return make_uint4(Cvt<T>::pack2(f[0], f[1]), Cvt<T>::pack2(f[2], f[3]), Cvt<T>::pack2(f[4], f[5]), Cvt<T>::pack2(f[6], f[7]));
}
template <typename T>
__device__ __forceinline__ void dt_load8(const T* p, float (&f)[8]) {
  dt_unpack8<T>(__ldg(reinterpret_cast<const uint4*>(p)), f);
}
__device__ __forceinline__ void dt_load8f(const float* p, float (&f)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}

// Reductions over rows: thread = (row lane rl, 8-channel group g); G = c / 8 groups (<= 256), RP = 256 / G rows per pass.
// Block b owns row b of the partials; the caller's finalize sums them in block order (fp64).
template <typename T>
__global__ void __launch_bounds__(256) dense_slice_stats_kernel(const T* __restrict__ F, long long rows, int ld, int col0, int c,
                                                                float* __restrict__ partials) {
  extern __shared__ float sm[];          // [RP][2][c]
  const int G = c >> 3, RP = 256 / G;
  const int g = threadIdx.x % G, rl = threadIdx.x / G;
  if (rl < RP) {
    float s1[8], s2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s1[i] = s2[i] = 0.f;
    for (long long r = (long long)blockIdx.x * RP + rl; r < rows; r += (long long)gridDim.x * RP) {
      float f[8];
      dt_load8<T>(F + (size_t)r * ld + col0 + g * 8, f);
#pragma unroll
      for (int i = 0; i < 8; ++i) { s1[i] += f[i]; s2[i] = fmaf(f[i], f[i], s2[i]); }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      sm[(rl * 2) * c + g * 8 + i] = s1[i];
      sm[(rl * 2 + 1) * c + g * 8 + i] = s2[i];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * c; i += 256) {
    float a = 0.f;
    for (int r = 0; r < RP; ++r) a += sm[r * 2 * c + i];
    partials[(size_t)blockIdx.x * 2 * c + i] = a;
  }
}

// same arithmetic as bnu_finalize (csrc/bcosk_train.cu): fp64 sums, var = E[x^2] - E[x]^2 clamped at 0
__global__ void dense_slice_stats_finalize_kernel(const float* __restrict__ partials, int nblk, double inv_m, int c, float eps,
                                                  float* __restrict__ mean, float* __restrict__ var, float* __restrict__ rstd) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  double s1 = 0.0, s2 = 0.0;
  for (int b = 0; b < nblk; ++b) {
    s1 += (double)partials[(size_t)b * 2 * c + ch];
    s2 += (double)partials[(size_t)b * 2 * c + c + ch];
  }
  const double m = s1 * inv_m;
  double v = s2 * inv_m - m * m;
  if (v < 0.0) v = 0.0;
  mean[ch] = (float)m;
  var[ch] = (float)v;
  rstd[ch] = (float)(1.0 / sqrt(v + (double)eps));
}

__global__ void dense_consumer_finalize_kernel(const float* __restrict__ var, const float* __restrict__ rstd, const float* __restrict__ w,
                                               int c, float momentum, float* __restrict__ running_var, float* __restrict__ alpha) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  alpha[ch] = (w != nullptr ? w[ch] : 1.f) * rstd[ch];
  if (running_var != nullptr) running_var[ch] = (1.f - momentum) * running_var[ch] + momentum * var[ch];
}

template <typename T>
__global__ void __launch_bounds__(256) dense_consumer_bwd_kernel(const void* __restrict__ g_t, int gt_f32, const T* __restrict__ t,
                                                                 const float* __restrict__ gnt, const float* __restrict__ alpha,
                                                                 const T* __restrict__ F, int ld, long long rows, int c,
                                                                 float* __restrict__ Gm, int accumulate, float* __restrict__ partials) {
  extern __shared__ float sm[];          // [RP][c]
  const int G = c >> 3, RP = 256 / G;
  const int g = threadIdx.x % G, rl = threadIdx.x / G;
  if (rl < RP) {
    float s[8], a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] = 0.f;
    dt_load8f(alpha + g * 8, a);
    for (long long r = (long long)blockIdx.x * RP + rl; r < rows; r += (long long)gridDim.x * RP) {
      float gz[8], tv[8], f[8];
      if (gt_f32) dt_load8f(reinterpret_cast<const float*>(g_t) + (size_t)r * c + g * 8, gz);
      else dt_load8<T>(reinterpret_cast<const T*>(g_t) + (size_t)r * c + g * 8, gz);
      dt_load8<T>(t + (size_t)r * c + g * 8, tv);
      dt_load8<T>(F + (size_t)r * ld + g * 8, f);
      const float tn = __ldg(gnt + r);
      float* gp = Gm + (size_t)r * ld + g * 8;
      float o[8];
      if (accumulate) {
        const float4 p0 = *reinterpret_cast<const float4*>(gp), p1 = *reinterpret_cast<const float4*>(gp + 4);
        o[0] = p0.x; o[1] = p0.y; o[2] = p0.z; o[3] = p0.w; o[4] = p1.x; o[5] = p1.y; o[6] = p1.z; o[7] = p1.w;
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = 0.f;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float gy = tv[i] > 0.f ? fmaf(tv[i], tn, gz[i]) : 0.f;     // t = relu(F alpha): t > 0 is the ReLU mask
        s[i] = fmaf(gy, f[i], s[i]);
        o[i] = fmaf(gy, a[i], o[i]);
      }
      reinterpret_cast<float4*>(gp)[0] = make_float4(o[0], o[1], o[2], o[3]);
      reinterpret_cast<float4*>(gp)[1] = make_float4(o[4], o[5], o[6], o[7]);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) sm[rl * c + g * 8 + i] = s[i];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < c; i += 256) {
    float acc = 0.f;
    for (int r = 0; r < RP; ++r) acc += sm[r * c + i];
    partials[(size_t)blockIdx.x * c + i] = acc;
  }
}

__global__ void dense_consumer_bwd_finalize_kernel(const float* __restrict__ partials, int nblk, const float* __restrict__ rstd,
                                                   const float* __restrict__ w, double inv_m, int c, int accumulate, float* __restrict__ K,
                                                   float* __restrict__ g_w) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  double S = 0.0;
  for (int b = 0; b < nblk; ++b) S += (double)partials[(size_t)b * c + ch];
  const float r = rstd[ch], ww = w != nullptr ? w[ch] : 1.f;
  const float k = (float)(-(double)r * r * r * ww * S * inv_m);
  K[ch] = accumulate ? K[ch] + k : k;
  if (g_w != nullptr) g_w[ch] = (float)(S * r);
}

// one warp covers 32 / lpr rows, lpr = lanes per row (a power of two >= min(G, 32)); gnT is a shuffle reduction over those lanes
template <typename T>
__global__ void __launch_bounds__(256) dense_slice_bwd_kernel(const float* __restrict__ Gm, const T* __restrict__ F, int ld, int col0,
                                                              long long rows, int c, int lpr, const float* __restrict__ mean,
                                                              const float* __restrict__ K, const T* __restrict__ scale,
                                                              const float* __restrict__ inv_n, T* __restrict__ out,
                                                              float* __restrict__ gnt) {
  const int G = c >> 3;
  const int lane = threadIdx.x & 31;
  const long long warp = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long row = warp * (32 / lpr) + lane / lpr;
  const int sub = lane % lpr;
  float acc = 0.f;
  if (row < rows) {
    for (int g = sub; g < G; g += lpr) {
      float go[8], f[8], mu[8], k[8];
      dt_load8f(Gm + (size_t)row * ld + col0 + g * 8, go);
      dt_load8<T>(F + (size_t)row * ld + col0 + g * 8, f);
      dt_load8f(mean + col0 + g * 8, mu);
      dt_load8f(K + col0 + g * 8, k);
#pragma unroll
      for (int i = 0; i < 8; ++i) go[i] = fmaf(f[i] - mu[i], k[i], go[i]);
      if (scale != nullptr) {
        float sc[8];
        dt_load8<T>(scale + (size_t)row * c + g * 8, sc);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          acc = fmaf(go[i], f[i], acc);
          go[i] = 2.f * go[i] * sc[i];
        }
      }
      *reinterpret_cast<uint4*>(out + (size_t)row * c + g * 8) = dt_pack8<T>(go);
    }
  }
  if (gnt != nullptr) {
    for (int o = lpr >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (row < rows && sub == 0) {
      const float in = __ldg(inv_n + row);
      gnt[row] = -acc * in * in;
    }
  }
}

inline cudaStream_t S_(void* s) { return reinterpret_cast<cudaStream_t>(s); }

int check_prefix(int c, int col0, int ld, const char* who) {
  if (c < 8 || c % 8 != 0 || c > 2048 || col0 < 0 || col0 % 8 != 0 || ld % 8 != 0 || col0 + c > ld)
    return set_error(BCOSK_EINVAL, "%s: need c %% 8 == 0, 8 <= c <= 2048, col0 %% 8 == 0, ld %% 8 == 0, col0 + c <= ld (c %d col0 %d ld %d)",
                     who, c, col0, ld);
  return BCOSK_OK;
}

}  // namespace
}  // namespace bcosk

using namespace bcosk;

#define BCOSK_DT_SWITCH(dtype, who, ...)                                            \
  if ((dtype) == BCOSK_DTYPE_BF16) { using T = __nv_bfloat16; __VA_ARGS__ }         \
  else if ((dtype) == BCOSK_DTYPE_F16) { using T = __half; __VA_ARGS__ }            \
  else return set_error(BCOSK_EINVAL, "%s: bad dtype %d", who, (int)(dtype));

extern "C" int bcosk_dense_slice_stats(const void* F, int64_t rows, int32_t ld, int32_t col0, int32_t c, float eps, float* partials, int32_t nblk,
                                       float* mean, float* var, float* rstd, int32_t dtype, void* stream) {
  if (!F || !partials || !mean || !var || !rstd || rows < 1 || nblk < 1) return set_error(BCOSK_EINVAL, "dense_slice_stats: bad argument");
  int rc = check_prefix(c, col0, ld, "dense_slice_stats");
  if (rc) return rc;
  const size_t smem = (size_t)(256 / (c / 8)) * 2 * c * sizeof(float);
  BCOSK_DT_SWITCH(dtype, "dense_slice_stats", dense_slice_stats_kernel<T><<<(unsigned)nblk, 256, smem, S_(stream)>>>(
      reinterpret_cast<const T*>(F), rows, ld, col0, c, partials);)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  dense_slice_stats_finalize_kernel<<<(c + 127) / 128, 128, 0, S_(stream)>>>(partials, nblk, 1.0 / (double)rows, c, eps, mean + col0,
                                                                            var + col0, rstd + col0);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_dense_consumer_finalize(const float* var, const float* rstd, const float* weight, int32_t c, float momentum,
                                             float* running_var, float* alpha, void* stream) {
  if (!var || !rstd || !alpha || c < 1) return set_error(BCOSK_EINVAL, "dense_consumer_finalize: bad argument");
  dense_consumer_finalize_kernel<<<(c + 127) / 128, 128, 0, S_(stream)>>>(var, rstd, weight, c, momentum, running_var, alpha);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_dense_consumer_bwd(const void* g_t, int32_t g_t_f32, const void* t, const float* gnt, const float* alpha, const void* F,
                                        int32_t ld, int64_t rows, int32_t c, float* G, int32_t accumulate, float* partials, int32_t nblk,
                                        int32_t dtype, void* stream) {
  if (!g_t || !t || !gnt || !alpha || !F || !G || !partials || rows < 1 || nblk < 1)
    return set_error(BCOSK_EINVAL, "dense_consumer_bwd: bad argument");
  int rc = check_prefix(c, 0, ld, "dense_consumer_bwd");
  if (rc) return rc;
  const size_t smem = (size_t)(256 / (c / 8)) * c * sizeof(float);
  BCOSK_DT_SWITCH(dtype, "dense_consumer_bwd", dense_consumer_bwd_kernel<T><<<(unsigned)nblk, 256, smem, S_(stream)>>>(
      g_t, g_t_f32, reinterpret_cast<const T*>(t), gnt, alpha, reinterpret_cast<const T*>(F), ld, rows, c, G, accumulate, partials);)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_dense_consumer_bwd_finalize(const float* partials, int32_t nblk, const float* rstd, const float* weight, int64_t rows,
                                                 int32_t c, int32_t accumulate, float* K, float* g_weight, void* stream) {
  if (!partials || nblk < 1 || !rstd || !K || rows < 1 || c < 1) return set_error(BCOSK_EINVAL, "dense_consumer_bwd_finalize: bad argument");
  dense_consumer_bwd_finalize_kernel<<<(c + 127) / 128, 128, 0, S_(stream)>>>(partials, nblk, rstd, weight, 1.0 / (double)rows, c, accumulate,
                                                                             K, g_weight);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_dense_slice_bwd(const float* G, const void* F, int32_t ld, int32_t col0, int64_t rows, int32_t c, const float* mean,
                                     const float* K, const void* scale, const float* inv_norm, void* out, float* gnt, int32_t dtype,
                                     void* stream) {
  if (!G || !F || !mean || !K || !out || rows < 1) return set_error(BCOSK_EINVAL, "dense_slice_bwd: bad argument");
  if ((gnt != nullptr) != (scale != nullptr) || (gnt && !inv_norm))
    return set_error(BCOSK_EINVAL, "dense_slice_bwd: scale, gnt and inv_norm go together");
  int rc = check_prefix(c, col0, ld, "dense_slice_bwd");
  if (rc) return rc;
  const int groups = c / 8;
  int lpr = 1;
  while (lpr < groups && lpr < 32) lpr <<= 1;
  const long long warps = (rows + (32 / lpr) - 1) / (32 / lpr);
  const unsigned grid = (unsigned)((warps + 7) / 8);
  BCOSK_DT_SWITCH(dtype, "dense_slice_bwd", dense_slice_bwd_kernel<T><<<grid, 256, 0, S_(stream)>>>(
      G, reinterpret_cast<const T*>(F), ld, col0, rows, c, lpr, mean, K, reinterpret_cast<const T*>(scale), inv_norm,
      reinterpret_cast<T*>(out), gnt);)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}
