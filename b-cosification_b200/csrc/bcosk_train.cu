// bcosk_train.cu -- bandwidth kernels of the B-cosification fine-tuning step (SURVEY 8f row 2, BASELINE config 5), sm_100a.
//
// The fine-tuning step runs the network in train mode (reference: bcos/training/trainer.py:666-784): uncentred batch norm with
// BATCH statistics (batchnorm_uncentered.py:36-43), B-cos scales that are NOT detached (bcosconv2d.py:172-194), the
// UniformOffLabelsBCEWithLogitsLoss (bcos/modules/losses.py:99-139), adaptive gradient clipping (bcos/training/agc.py:28-42)
// and AdamW.  The contractions (forward, data gradient, weight gradient) are tcgen05 kernels (bcosk_igemm*.cu, bcosk_wgrad.cu);
// this file holds everything between them, on NHWC 16-bit activations / gradients with fp32 per-channel and per-pixel vectors:
//
//   forward   conv -> [bnu_stats -> bnu_finalize -> bnu_apply (+ residual, ReLU, per-pixel sum of squares for the next patch norm)]
//   backward  g_z = gA + gB + x_post * T   (data gradients of the consumers + their patch-norm path, see below)
//             g_y = g_z * [x_post > 0]
//             S[c] = sum_m g_y * out                                   train_bwd_reduce
//             g_out = g_y * alpha[c] + (out - mean[c]) * kcoef[c]      kcoef = -rstd^3 w S / M   (batch-statistics path)
//             g_lin = g_out * 2 s            (d(lin |lin| / n)/d lin = 2 |lin| / n, the scale is part of the graph)
//             gnT[m] = -sum_c g_out * out / n[m]^2                     train_bwd_apply
//             T = transposed sum-pool of gnT                           (d n / d x = x / n over the patch)  sumpool_transpose
//   optimizer unit-wise AGC + AdamW on fp32 master weights             agc_adamw
// 16-byte vector accesses, consecutive lanes on consecutive addresses, warp-shuffle / shared-memory reductions.
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
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  float2 a;
  a = Cvt<T>::unpack2(u.x); f[0] = a.x; f[1] = a.y;
  a = Cvt<T>::unpack2(u.y); f[2] = a.x; f[3] = a.y;
  a = Cvt<T>::unpack2(u.z); f[4] = a.x; f[5] = a.y;
  a = Cvt<T>::unpack2(u.w); f[6] = a.x; f[7] = a.y;
}
template <typename T>
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(Cvt<T>::pack2(f[0], f[1]), Cvt<T>::pack2(f[2], f[3]), Cvt<T>::pack2(f[4], f[5]), Cvt<T>::pack2(f[6], f[7]));
}
__device__ __forceinline__ void load8f(const float* p, float (&f)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
// 8 channels of row `row`: 16-bit tensor, or fp32 when f32
template <typename T>
__device__ __forceinline__ void load_row8(const void* base, bool f32, size_t row, int ld, int c8, float (&f)[8]) {
  if (f32) load8f(reinterpret_cast<const float*>(base) + row * ld + c8, f);
  else unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(base) + row * ld + c8)), f);
}

// thread -> (row lane, channel group): G = C/8 channel groups (<= 256), RP = 256 / G rows per pass
struct SlabMap {
  int G, RP;
  __device__ SlabMap(int C) {
    G = C >> 3;
    RP = 256 / G;
    if (RP < 1) RP = 1;
  }
};

// ---------------------------------------------------------------- per-channel sums (sum x, sum x^2) over the rows
template <typename T>
__global__ void __launch_bounds__(256) bnu_stats_kernel(const T* __restrict__ x, long long M, int C, float* __restrict__ partials) {
  extern __shared__ float sm[];          // [RP][2][C]
  const SlabMap mp(C);
  const int g = threadIdx.x % mp.G, rl = threadIdx.x / mp.G;
  float s1[8], s2[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s1[i] = s2[i] = 0.f;
  if (rl < mp.RP) {
    for (long long r = (long long)blockIdx.x * mp.RP + rl; r < M; r += (long long)gridDim.x * mp.RP) {
      float f[8];
      unpack8<T>(__ldg(reinterpret_cast<const uint4*>(x + (size_t)r * C + g * 8)), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) { s1[i] += f[i]; s2[i] = fmaf(f[i], f[i], s2[i]); }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      sm[(rl * 2) * C + g * 8 + i] = s1[i];
      sm[(rl * 2 + 1) * C + g * 8 + i] = s2[i];
    }
  }
  __syncthreads();
  // every block owns one row of `partials` (fixed summation order: the statistics are bit-reproducible run to run - a
  // random-init deep B-cos net amplifies even fp32 reordering noise of the statistics into O(10 %) gradient differences)
  for (int i = threadIdx.x; i < 2 * C; i += 256) {
    float a = 0.f;
    for (int r = 0; r < mp.RP; ++r) a += sm[r * 2 * C + i];
    partials[(size_t)blockIdx.x * 2 * C + i] = a;
  }
}

// mean, biased centred variance -> rstd, alpha = w * rstd; running_var <- (1 - momentum) running_var + momentum var
__global__ void bnu_finalize_kernel(const float* __restrict__ partials, int nblk, double inv_m, int C, const float* __restrict__ w,
                                    float eps, float momentum, float* __restrict__ running_var, float* __restrict__ alpha,
                                    float* __restrict__ mean, float* __restrict__ rstd) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s1 = 0.0, s2 = 0.0;
  for (int b = 0; b < nblk; ++b) {
    s1 += (double)partials[(size_t)b * 2 * C + c];
    s2 += (double)partials[(size_t)b * 2 * C + C + c];
  }
  const double m = s1 * inv_m;
  double var = s2 * inv_m - m * m;
  if (var < 0.0) var = 0.0;
  const float r = (float)(1.0 / sqrt(var + (double)eps));
  mean[c] = (float)m;
  rstd[c] = r;
  alpha[c] = (w != nullptr ? w[c] : 1.f) * r;
  if (running_var != nullptr) running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)var;
}

// y = relu?(x * alpha[c] + res), sq[m] = sum_c y^2
template <typename T>
__global__ void __launch_bounds__(256) bnu_apply_kernel(const T* __restrict__ x, long long M, int C, const float* __restrict__ alpha,
                                                        const T* __restrict__ res, int relu, T* __restrict__ y, float* __restrict__ sq) {
  const int G = C >> 3;
  const int lpr = G < 32 ? G : 32;                       // lanes per row (G < 32: a power of two)
  const int rpw = 32 / lpr;
  const int lane = threadIdx.x & 31;
  const long long warp = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long row = warp * rpw + lane / lpr;
  const int sub = lane % lpr;
  float acc = 0.f;
  if (row < M) {
    for (int g = sub; g < G; g += lpr) {
      float f[8], a[8];
      unpack8<T>(__ldg(reinterpret_cast<const uint4*>(x + (size_t)row * C + g * 8)), f);
      load8f(alpha + g * 8, a);
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] *= a[i];
      if (res != nullptr) {
        float r[8];
        unpack8<T>(__ldg(reinterpret_cast<const uint4*>(res + (size_t)row * C + g * 8)), r);
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] += r[i];
      }
      if (relu) {
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = fmaxf(f[i], 0.f);
      }
      const uint4 u = pack8<T>(f);
      *reinterpret_cast<uint4*>(y + (size_t)row * C + g * 8) = u;
      float q[8];
      unpack8<T>(u, q);                                  // what the consumer reads
#pragma unroll
      for (int i = 0; i < 8; ++i) acc = fmaf(q[i], q[i], acc);
    }
  }
  if (sq != nullptr) {
    for (int o = lpr >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (row < M && sub == 0) sq[row] = acc;
  }
}

// g_y of one row x 8 channels: (gA + gB + x_post * T[row]) * [x_post > 0]
template <typename T>
__device__ __forceinline__ void grad_in8(const void* gA, bool ga_f32, const T* gB, const T* xpost, const float* Tn, int relu, size_t row,
                                         int C, int c8, float (&g)[8]) {
  load_row8<T>(gA, ga_f32, row, C, c8, g);
  if (gB != nullptr) {
    float b[8];
    unpack8<T>(__ldg(reinterpret_cast<const uint4*>(gB + row * C + c8)), b);
#pragma unroll
    for (int i = 0; i < 8; ++i) g[i] += b[i];
  }
  if (xpost != nullptr && (Tn != nullptr || relu)) {
    float xp[8];
    unpack8<T>(__ldg(reinterpret_cast<const uint4*>(xpost + row * C + c8)), xp);
    if (Tn != nullptr) {
      const float t = __ldg(Tn + row);
#pragma unroll
      for (int i = 0; i < 8; ++i) g[i] = fmaf(xp[i], t, g[i]);
    }
    if (relu) {
#pragma unroll
      for (int i = 0; i < 8; ++i) g[i] = xp[i] > 0.f ? g[i] : 0.f;
    }
  }
}

// S[c] += sum_rows g_y * out
template <typename T>
__global__ void __launch_bounds__(256) train_bwd_reduce_kernel(const void* __restrict__ gA, int ga_f32, const T* __restrict__ gB,
                                                               const T* __restrict__ xpost, const float* __restrict__ Tn, int relu,
                                                               const void* __restrict__ out, int out_f32, long long M, int C,
                                                               float* __restrict__ partials) {
  extern __shared__ float sm[];          // [RP][C]
  const SlabMap mp(C);
  const int g = threadIdx.x % mp.G, rl = threadIdx.x / mp.G;
  float s[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = 0.f;
  if (rl < mp.RP) {
    for (long long r = (long long)blockIdx.x * mp.RP + rl; r < M; r += (long long)gridDim.x * mp.RP) {
      float gy[8], o[8];
      grad_in8<T>(gA, ga_f32 != 0, gB, xpost, Tn, relu, (size_t)r, C, g * 8, gy);
      load_row8<T>(out, out_f32 != 0, (size_t)r, C, g * 8, o);
#pragma unroll
      for (int i = 0; i < 8; ++i) s[i] = fmaf(gy[i], o[i], s[i]);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) sm[rl * C + g * 8 + i] = s[i];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += 256) {
    float a = 0.f;
    for (int r = 0; r < mp.RP; ++r) a += sm[r * C + i];
    partials[(size_t)blockIdx.x * C + i] = a;            // one row per block: fixed summation order
  }
}

// kcoef[c] = -rstd^3 w S / M;  g_w[c] += S rstd  (d z / d w = out * rstd)
__global__ void bnu_bwd_finalize_kernel(const float* __restrict__ partials, int nblk, const float* __restrict__ rstd,
                                        const float* __restrict__ w, double inv_m, int C, float* __restrict__ kcoef,
                                        float* __restrict__ g_w, float* __restrict__ s_out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double S = 0.0;
  for (int b = 0; b < nblk; ++b) S += (double)partials[(size_t)b * C + c];
  const float r = rstd[c], ww = w != nullptr ? w[c] : 1.f;
  kcoef[c] = (float)(-(double)r * r * r * ww * S * inv_m);
  if (g_w != nullptr) g_w[c] = (float)(S * r);
  if (s_out != nullptr) s_out[c] = (float)S;
}

// g_lin, gnT (and optionally g_y) of one layer
template <typename T>
__global__ void __launch_bounds__(256) train_bwd_apply_kernel(const void* __restrict__ gA, int ga_f32, const T* __restrict__ gB,
                                                              const T* __restrict__ xpost, const float* __restrict__ Tn, int relu,
                                                              const void* __restrict__ out, int out_f32, const T* __restrict__ s,
                                                              const float* __restrict__ alpha, const float* __restrict__ kcoef,
                                                              const float* __restrict__ mean, const float* __restrict__ inv_n,
                                                              long long M, int C, T* __restrict__ g_lin, float* __restrict__ gnT,
                                                              T* __restrict__ g_y) {
  const int G = C >> 3;
  const int lpr = G < 32 ? G : 32;
  const int rpw = 32 / lpr;
  const int lane = threadIdx.x & 31;
  const long long warp = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long row = warp * rpw + lane / lpr;
  const int sub = lane % lpr;
  float acc = 0.f;
  if (row < M) {
    for (int g = sub; g < G; g += lpr) {
      float gy[8], o[8], sc[8];
      grad_in8<T>(gA, ga_f32 != 0, gB, xpost, Tn, relu, (size_t)row, C, g * 8, gy);
      if (g_y != nullptr) *reinterpret_cast<uint4*>(g_y + (size_t)row * C + g * 8) = pack8<T>(gy);
      load_row8<T>(out, out_f32 != 0, (size_t)row, C, g * 8, o);
      unpack8<T>(__ldg(reinterpret_cast<const uint4*>(s + (size_t)row * C + g * 8)), sc);
      float go[8];
      if (alpha != nullptr) {
        float a[8], k[8], mu[8];
        load8f(alpha + g * 8, a);
        load8f(kcoef + g * 8, k);
        load8f(mean + g * 8, mu);
#pragma unroll
        for (int i = 0; i < 8; ++i) go[i] = fmaf(gy[i], a[i], (o[i] - mu[i]) * k[i]);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) go[i] = gy[i];
      }
      float gl[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        gl[i] = 2.f * go[i] * sc[i];
        acc = fmaf(go[i], o[i], acc);
      }
      *reinterpret_cast<uint4*>(g_lin + (size_t)row * C + g * 8) = pack8<T>(gl);
    }
  }
  if (gnT != nullptr) {
    for (int o = lpr >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (row < M && sub == 0) {
      const float in = __ldg(inv_n + row);
      gnT[row] = -acc * in * in;
    }
  }
}

// out = gA + gB + x * T[row]   (gradient of a tensor that feeds convolutions but is not a norm layer's output: the pooled stem)
template <typename T>
__global__ void grad_combine_kernel(const T* __restrict__ gA, const T* __restrict__ gB, const T* __restrict__ x, const float* __restrict__ Tn,
                                    long long M, int C, T* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int G = C >> 3;
  if (idx >= M * G) return;
  const size_t row = (size_t)(idx / G);
  const int g = (int)(idx % G);
  float f[8];
  grad_in8<T>(gA, false, gB, x, Tn, 0, row, C, g * 8, f);
  *reinterpret_cast<uint4*>(out + row * C + g * 8) = pack8<T>(f);
}

// Backward of AvgPool2d(k) (stride k, no padding: the anti-aliasing pools of the CLIP ResNets) fused with the consumers' terms
// at the pooled resolution: gx[img, y, x, :] (+)= (gA + gB + xp * T)[img, y / k, x / k, :] / k^2.  One thread per input pixel and
// 8 channels; pixels past the last full window get zero.  Every output element is written by one thread (no atomics).
template <typename T>
__global__ void pool_bwd_norm_kernel(const void* __restrict__ gA, int ga_f32, const T* __restrict__ gB, const T* __restrict__ xp,
                                     const float* __restrict__ Tn, int nb, int h, int w, int C, int k, int accumulate, T* __restrict__ gx) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int G = C >> 3;
  if (idx >= (long long)nb * h * w * G) return;
  const long long pix = idx / G;
  const int g = (int)(idx - pix * G);
  const int x = (int)(pix % w), y = (int)((pix / w) % h), img = (int)(pix / ((long long)w * h));
  const int op = h / k, oq = w / k;
  float f[8];
  if (y / k < op && x / k < oq) {
    const size_t row = ((size_t)img * op + y / k) * oq + x / k;
    grad_in8<T>(gA, ga_f32 != 0, gB, xp, Tn, 0, row, C, g * 8, f);
    const float inv = 1.0f / (float)(k * k);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] *= inv;
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = 0.f;
  }
  uint4* dst = reinterpret_cast<uint4*>(gx + (size_t)pix * C + g * 8);
  if (accumulate) {
    float o[8];
    unpack8<T>(*dst, o);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] += o[i];
  }
  *dst = pack8<T>(f);
}

// T[img, y, x] (+)= sum over the output pixels (p, q) whose k x k window (stride, pad) covers (y, x) of gnT[img, p, q]
__global__ void sumpool_transpose_kernel(const float* __restrict__ gnT, int nb, int h, int w, int k, int stride, int pad, int op, int oq,
                                         int accumulate, float* __restrict__ Tn) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)nb * h * w) return;
  const int x = (int)(idx % w);
  const int y = (int)((idx / w) % h);
  const int img = (int)(idx / ((long long)w * h));
  float a = 0.f;
  for (int dy = 0; dy < k; ++dy) {
    const int py = y + pad - dy;
    if (py < 0 || py % stride != 0 || py / stride >= op) continue;
    for (int dx = 0; dx < k; ++dx) {
      const int px = x + pad - dx;
      if (px < 0 || px % stride != 0 || px / stride >= oq) continue;
      a += __ldg(gnT + ((size_t)img * op + py / stride) * oq + px / stride);
    }
  }
  Tn[idx] = accumulate ? Tn[idx] + a : a;
}

// UniformOffLabelsBCEWithLogitsLoss (losses.py:99-139, reduction "mean"): target = clamp(one_hot, min = off);
// loss += sum BCE / (N C);  g_fc[n, pix, c] = (sigmoid(x) - t) / (N C) * inv_temp / npix  (through LogitLayer and the global average pool)
template <typename T>
__global__ void bce_uniform_off_kernel(const float* __restrict__ logits, const int32_t* __restrict__ labels, int N, int C, float off,
                                       float inv_temp, int npix, float grad_scale, float* __restrict__ loss, T* __restrict__ g_fc,
                                       float* __restrict__ g_logits) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  float l = 0.f;
  if (idx < (long long)N * C) {
    const int n = (int)(idx / C), c = (int)(idx % C);
    const float x = logits[idx];
    const float t = (labels[n] == c) ? 1.f : off;
    // stable BCE with logits: max(x, 0) - x t + log(1 + exp(-|x|))
    l = fmaxf(x, 0.f) - x * t + log1pf(expf(-fabsf(x)));
    const float sg = 1.f / (1.f + expf(-x));
    const float g = (sg - t) / (float)((long long)N * C);
    if (g_logits != nullptr) g_logits[idx] = g;
    const float gp = g * inv_temp / (float)npix * grad_scale;
    if (g_fc != nullptr) {
      const uint32_t pk = Cvt<T>::pack2(gp, gp);
      unsigned short h = (unsigned short)(pk & 0xffffu);
      unsigned short* dst = reinterpret_cast<unsigned short*>(g_fc);
      for (int p = 0; p < npix; ++p) dst[((size_t)n * npix + p) * C + c] = h;
    }
  }
  l = warp_sum(l);
  if ((threadIdx.x & 31) == 0 && l != 0.f) atomicAdd(loss, l / (float)((long long)N * C));
}

// out[i] = idx[i] >= 0 ? src[idx[i]] : 0   (fp32 master weights -> packed 16-bit operand layouts)
template <typename T>
__global__ void gather_cast_kernel(const float* __restrict__ src, const int32_t* __restrict__ idx, long long n, T* __restrict__ out) {
  const long long i2 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 2;
  if (i2 >= n) return;
  const int32_t a = idx[i2], b = (i2 + 1 < n) ? idx[i2 + 1] : -1;
  const float fa = a >= 0 ? __ldg(src + a) : 0.f, fb = b >= 0 ? __ldg(src + b) : 0.f;
  if (i2 + 1 < n) *reinterpret_cast<uint32_t*>(out + i2) = Cvt<T>::pack2(fa, fb);
  else out[i2] = (T)fa;
}

// Unit-wise adaptive gradient clipping (agc.py:28-42) + AdamW (decoupled weight decay) on one parameter tensor.
// One block per unit (output channel row of `cols` elements; 1-D parameters are ONE unit).  g is gathered through gidx
// (the weight-gradient kernel writes the packed operand layout), scaled by gscale (1 / world size after the all-reduce sum).
__global__ void __launch_bounds__(256) agc_adamw_kernel(float* __restrict__ w, const float* __restrict__ g, const int32_t* __restrict__ gidx,
                                                        float* __restrict__ m, float* __restrict__ v, int cols, float gscale, float lr,
                                                        float beta1, float beta2, float eps, float wd, float clip, float agc_eps,
                                                        float bc1, float bc2) {
  __shared__ float red[2][8];
  const size_t base = (size_t)blockIdx.x * cols;
  float sw = 0.f, sg = 0.f;
  for (int i = threadIdx.x; i < cols; i += 256) {
    const float ww = w[base + i];
    const float gg = g[gidx != nullptr ? (size_t)gidx[base + i] : base + i] * gscale;
    sw = fmaf(ww, ww, sw);
    sg = fmaf(gg, gg, sg);
  }
  sw = warp_sum(sw);
  sg = warp_sum(sg);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = sw; red[1][threadIdx.x >> 5] = sg; }
  __syncthreads();
  float nw = 0.f, ng = 0.f;
  for (int i = 0; i < 8; ++i) { nw += red[0][i]; ng += red[1][i]; }
  nw = sqrtf(nw);
  ng = sqrtf(ng);
  float factor = 1.f;
  if (clip > 0.f) {
    const float max_norm = fmaxf(nw, agc_eps) * clip;
    if (!(ng < max_norm)) factor = max_norm / fmaxf(ng, 1e-6f);
  }
  for (int i = threadIdx.x; i < cols; i += 256) {
    const float gg = g[gidx != nullptr ? (size_t)gidx[base + i] : base + i] * gscale * factor;
    float ww = w[base + i];
    const float mm = beta1 * m[base + i] + (1.f - beta1) * gg;
    const float vv = beta2 * v[base + i] + (1.f - beta2) * gg * gg;
    m[base + i] = mm;
    v[base + i] = vv;
    ww -= lr * wd * ww;
    ww -= lr * (mm / bc1) / (sqrtf(vv / bc2) + eps);
    w[base + i] = ww;
  }
}

// ---- whole-model variants (one launch each; CUDA-graph friendly: the step counter lives in device memory) ----------------------
// adam state [3] = {step, 1 - beta1^step, 1 - beta2^step}: advanced on the device so that a captured graph can be replayed
__global__ void adam_state_step_kernel(float* __restrict__ st, float beta1, float beta2) {
  const float step = st[0] + 1.f;
  st[0] = step;
  st[1] = 1.f - powf(beta1, step);
  st[2] = 1.f - powf(beta2, step);
}

// unit u of the whole model: cols[u] consecutive master weights starting at off[u] (one block per unit)
__global__ void __launch_bounds__(256) agc_adamw_multi_kernel(float* __restrict__ w, const float* __restrict__ g, const int32_t* __restrict__ gidx,
                                                              float* __restrict__ m, float* __restrict__ v, const long long* __restrict__ off,
                                                              const int32_t* __restrict__ ncols, float gscale, float lr, float beta1,
                                                              float beta2, float eps, float wd, float clip, float agc_eps,
                                                              const float* __restrict__ st) {
  __shared__ float red[2][8];
  const size_t base = (size_t)off[blockIdx.x];
  const int cols = ncols[blockIdx.x];
  const float bc1 = st[1], bc2 = st[2];
  float sw = 0.f, sg = 0.f;
  for (int i = threadIdx.x; i < cols; i += 256) {
    const float ww = w[base + i];
    const float gg = g[(size_t)gidx[base + i]] * gscale;
    sw = fmaf(ww, ww, sw);
    sg = fmaf(gg, gg, sg);
  }
  sw = warp_sum(sw);
  sg = warp_sum(sg);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = sw; red[1][threadIdx.x >> 5] = sg; }
  __syncthreads();
  float nw = 0.f, ng = 0.f;
  for (int i = 0; i < 8; ++i) { nw += red[0][i]; ng += red[1][i]; }
  nw = sqrtf(nw);
  ng = sqrtf(ng);
  float factor = 1.f;
  if (clip > 0.f) {
    const float max_norm = fmaxf(nw, agc_eps) * clip;
    if (!(ng < max_norm)) factor = max_norm / fmaxf(ng, 1e-6f);
  }
  for (int i = threadIdx.x; i < cols; i += 256) {
    const float gg = g[(size_t)gidx[base + i]] * gscale * factor;
    float ww = w[base + i];
    const float mm = beta1 * m[base + i] + (1.f - beta1) * gg;
    const float vv = beta2 * v[base + i] + (1.f - beta2) * gg * gg;
    m[base + i] = mm;
    v[base + i] = vv;
    ww -= lr * wd * ww;
    ww -= lr * (mm / bc1) / (sqrtf(vv / bc2) + eps);
    w[base + i] = ww;
  }
}

// table[p] = {index pointer, output pointer, n}: every packed operand of the model refreshed in one launch (blockIdx.y = pack)
template <typename T>
__global__ void gather_cast_multi_kernel(const float* __restrict__ src, const long long* __restrict__ table) {
  const long long* e = table + 3 * (long long)blockIdx.y;
  const int32_t* idx = reinterpret_cast<const int32_t*>(e[0]);
  T* out = reinterpret_cast<T*>(e[1]);
  const long long n = e[2];
  for (long long i2 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 2; i2 < n; i2 += (long long)gridDim.x * blockDim.x * 2) {
    const int32_t a = idx[i2], b = (i2 + 1 < n) ? idx[i2 + 1] : -1;
    const float fa = a >= 0 ? __ldg(src + a) : 0.f, fb = b >= 0 ? __ldg(src + b) : 0.f;
    if (i2 + 1 < n) *reinterpret_cast<uint32_t*>(out + i2) = Cvt<T>::pack2(fa, fb);
    else out[i2] = (T)fa;
  }
}

inline cudaStream_t S_(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline unsigned grid_for(long long items, int per_block, unsigned cap = 0x7fffffffu) {
  long long b = (items + per_block - 1) / per_block;
  if (b < 1) b = 1;
  return (unsigned)(b > (long long)cap ? cap : b);
}

}  // namespace
}  // namespace bcosk

using namespace bcosk;

#define BCOSK_T_SWITCH(dtype, ...)                                                  \
  if ((dtype) == BCOSK_DTYPE_BF16) { using T = __nv_bfloat16; __VA_ARGS__ }         \
  else if ((dtype) == BCOSK_DTYPE_F16) { using T = __half; __VA_ARGS__ }            \
  else return set_error(BCOSK_EINVAL, "bad dtype %d", (int)(dtype));

static int check_channels(int c, const char* who) {
  const int g = c / 8;
  if (c % 8 != 0 || g < 1 || g > 256 || (g < 32 && (g & (g - 1)) != 0))
    return set_error(BCOSK_EUNSUPPORTED, "%s: channels must be a multiple of 8, <= 2048, and 8 x a power of two below 256 (got %d)", who, c);
  return BCOSK_OK;
}

extern "C" int bcosk_bnu_stats_nhwc(const void* x, int64_t rows, int32_t c, int32_t dtype, float* partials, int32_t nblk, void* stream) {
  if (!x || !partials || nblk < 1) return set_error(BCOSK_EINVAL, "bnu_stats: bad argument");
  int rc = check_channels(c, "bnu_stats");
  if (rc) return rc;
  const int G = c / 8, RP = 256 / G < 1 ? 1 : 256 / G;
  const size_t smem = (size_t)RP * 2 * c * sizeof(float);
  BCOSK_T_SWITCH(dtype, bnu_stats_kernel<T><<<(unsigned)nblk, 256, smem, S_(stream)>>>(reinterpret_cast<const T*>(x), rows, c, partials);)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_bnu_finalize(const float* partials, int32_t nblk, int64_t rows, int32_t c, const float* weight, float eps,
                                  float momentum, float* running_var, float* alpha, float* mean, float* rstd, void* stream) {
  if (!partials || nblk < 1 || !alpha || !mean || !rstd || rows < 1) return set_error(BCOSK_EINVAL, "bnu_finalize: bad argument");
  bnu_finalize_kernel<<<(c + 127) / 128, 128, 0, S_(stream)>>>(partials, nblk, 1.0 / (double)rows, c, weight, eps, momentum, running_var,
                                                             alpha, mean, rstd);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_bnu_apply_nhwc(const void* x, int64_t rows, int32_t c, const float* alpha, const void* res, int32_t relu, void* y,
                                    float* sq, int32_t dtype, void* stream) {
  if (!x || !alpha || !y) return set_error(BCOSK_EINVAL, "bnu_apply: null pointer");
  int rc = check_channels(c, "bnu_apply");
  if (rc) return rc;
  const int G = c / 8, lpr = G < 32 ? G : 32;
  const long long warps = (rows + (32 / lpr) - 1) / (32 / lpr);
  BCOSK_T_SWITCH(dtype, bnu_apply_kernel<T><<<grid_for(warps, 8), 256, 0, S_(stream)>>>(
      reinterpret_cast<const T*>(x), rows, c, alpha, reinterpret_cast<const T*>(res), relu, reinterpret_cast<T*>(y), sq);)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_train_bwd_reduce(const void* ga, int32_t ga_f32, const void* gb, const void* xpost, const float* tn, int32_t relu,
                                      const void* out, int32_t out_f32, int64_t rows, int32_t c, float* partials, int32_t nblk,
                                      int32_t dtype, void* stream) {
  if (!ga || !out || !partials || nblk < 1) return set_error(BCOSK_EINVAL, "train_bwd_reduce: bad argument");
  if ((relu || tn) && !xpost) return set_error(BCOSK_EINVAL, "train_bwd_reduce: ReLU mask / norm path need the layer's output tensor");
  int rc = check_channels(c, "train_bwd_reduce");
  if (rc) return rc;
  const int G = c / 8, RP = 256 / G < 1 ? 1 : 256 / G;
  const size_t smem = (size_t)RP * c * sizeof(float);
  BCOSK_T_SWITCH(dtype, train_bwd_reduce_kernel<T><<<(unsigned)nblk, 256, smem, S_(stream)>>>(
      ga, ga_f32, reinterpret_cast<const T*>(gb), reinterpret_cast<const T*>(xpost), tn, relu, out, out_f32, rows, c, partials);)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_bnu_bwd_finalize(const float* partials, int32_t nblk, const float* rstd, const float* weight, int64_t rows, int32_t c,
                                      float* kcoef, float* g_weight, float* s_out, void* stream) {
  if (!partials || nblk < 1 || !rstd || !kcoef || rows < 1) return set_error(BCOSK_EINVAL, "bnu_bwd_finalize: bad argument");
  bnu_bwd_finalize_kernel<<<(c + 127) / 128, 128, 0, S_(stream)>>>(partials, nblk, rstd, weight, 1.0 / (double)rows, c, kcoef, g_weight,
                                                                 s_out);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_train_bwd_apply(const void* ga, int32_t ga_f32, const void* gb, const void* xpost, const float* tn, int32_t relu,
                                     const void* out, int32_t out_f32, const void* scale, const float* alpha, const float* kcoef,
                                     const float* mean, const float* inv_norm, int64_t rows, int32_t c, void* g_lin, float* gnt, void* g_y,
                                     int32_t dtype, void* stream) {
  if (!ga || !out || !scale || !g_lin) return set_error(BCOSK_EINVAL, "train_bwd_apply: null pointer");
  if ((relu || tn) && !xpost) return set_error(BCOSK_EINVAL, "train_bwd_apply: ReLU mask / norm path need the layer's output tensor");
  if (alpha && (!kcoef || !mean)) return set_error(BCOSK_EINVAL, "train_bwd_apply: alpha needs kcoef and mean");
  if (gnt && !inv_norm) return set_error(BCOSK_EINVAL, "train_bwd_apply: gnT needs inv_norm");
  int rc = check_channels(c, "train_bwd_apply");
  if (rc) return rc;
  const int G = c / 8, lpr = G < 32 ? G : 32;
  const long long warps = (rows + (32 / lpr) - 1) / (32 / lpr);
  BCOSK_T_SWITCH(dtype, train_bwd_apply_kernel<T><<<grid_for(warps, 8), 256, 0, S_(stream)>>>(
      ga, ga_f32, reinterpret_cast<const T*>(gb), reinterpret_cast<const T*>(xpost), tn, relu, out, out_f32,
      reinterpret_cast<const T*>(scale), alpha, kcoef, mean, inv_norm, rows, c, reinterpret_cast<T*>(g_lin), gnt,
      reinterpret_cast<T*>(g_y));)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_grad_combine(const void* ga, const void* gb, const void* x, const float* tn, int64_t rows, int32_t c, void* out,
                                  int32_t dtype, void* stream) {
  if (!ga || !out || c % 8 != 0 || (tn && !x)) return set_error(BCOSK_EINVAL, "grad_combine: bad argument");
  BCOSK_T_SWITCH(dtype, grad_combine_kernel<T><<<grid_for(rows * (c / 8), 256), 256, 0, S_(stream)>>>(
      reinterpret_cast<const T*>(ga), reinterpret_cast<const T*>(gb), reinterpret_cast<const T*>(x), tn, rows, c,
      reinterpret_cast<T*>(out));)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_pool_bwd_norm(const void* ga, int32_t ga_f32, const void* gb, const void* x, const float* tn, int32_t nb, int32_t h,
                                   int32_t w, int32_t c, int32_t k, int32_t accumulate, void* gx, int32_t dtype, void* stream) {
  if (!ga || !gx || nb < 1 || h < k || w < k || k < 1 || c < 8 || c % 8 != 0 || (tn && !x))
    return set_error(BCOSK_EINVAL, "pool_bwd_norm: bad argument");
  const long long n = (long long)nb * h * w * (c / 8);
  BCOSK_T_SWITCH(dtype, pool_bwd_norm_kernel<T><<<grid_for(n, 256), 256, 0, S_(stream)>>>(
      ga, ga_f32, reinterpret_cast<const T*>(gb), reinterpret_cast<const T*>(x), tn, nb, h, w, c, k, accumulate, reinterpret_cast<T*>(gx));)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_sumpool_transpose(const float* gnt, int32_t nb, int32_t h, int32_t w, int32_t k, int32_t stride, int32_t pad,
                                       int32_t op, int32_t oq, int32_t accumulate, float* tn, void* stream) {
  if (!gnt || !tn || k < 1 || stride < 1) return set_error(BCOSK_EINVAL, "sumpool_transpose: bad argument");
  const long long n = (long long)nb * h * w;
  sumpool_transpose_kernel<<<grid_for(n, 256), 256, 0, S_(stream)>>>(gnt, nb, h, w, k, stride, pad, op, oq, accumulate, tn);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_bce_uniform_off(const float* logits, const int32_t* labels, int32_t n, int32_t c, float off_label, float inv_temp,
                                     int32_t npix, float grad_scale, float* loss, void* g_fc, float* g_logits, int32_t dtype,
                                     void* stream) {
  if (!logits || !labels || !loss) return set_error(BCOSK_EINVAL, "bce_uniform_off: null pointer");
  const long long items = (long long)n * c;
  BCOSK_T_SWITCH(dtype, bce_uniform_off_kernel<T><<<grid_for(items, 256), 256, 0, S_(stream)>>>(
      logits, labels, n, c, off_label, inv_temp, npix, grad_scale, loss, reinterpret_cast<T*>(g_fc), g_logits);)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_gather_cast(const float* src, const int32_t* idx, int64_t n, void* out, int32_t dtype, void* stream) {
  if (!src || !idx || !out) return set_error(BCOSK_EINVAL, "gather_cast: null pointer");
  BCOSK_T_SWITCH(dtype, gather_cast_kernel<T><<<grid_for((n + 1) / 2, 256), 256, 0, S_(stream)>>>(src, idx, n, reinterpret_cast<T*>(out));)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_agc_adamw(float* w, const float* g, const int32_t* gidx, float* m, float* v, int32_t units, int32_t cols,
                               float grad_scale, float lr, float beta1, float beta2, float eps, float weight_decay, float clip_factor,
                               float agc_eps, int32_t step, void* stream) {
  if (!w || !g || !m || !v || units < 1 || cols < 1 || step < 1) return set_error(BCOSK_EINVAL, "agc_adamw: bad argument");
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  agc_adamw_kernel<<<units, 256, 0, S_(stream)>>>(w, g, gidx, m, v, cols, grad_scale, lr, beta1, beta2, eps, weight_decay, clip_factor,
                                                 agc_eps, bc1, bc2);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_adam_state_step(float* state, float beta1, float beta2, void* stream) {
  if (!state) return set_error(BCOSK_EINVAL, "adam_state_step: null pointer");
  adam_state_step_kernel<<<1, 1, 0, S_(stream)>>>(state, beta1, beta2);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_agc_adamw_multi(float* w, const float* g, const int32_t* gidx, float* m, float* v, const int64_t* unit_off,
                                     const int32_t* unit_cols, int32_t units, float grad_scale, float lr, float beta1, float beta2, float eps,
                                     float weight_decay, float clip_factor, float agc_eps, const float* adam_state, void* stream) {
  if (!w || !g || !gidx || !m || !v || !unit_off || !unit_cols || !adam_state || units < 1)
    return set_error(BCOSK_EINVAL, "agc_adamw_multi: bad argument");
  agc_adamw_multi_kernel<<<units, 256, 0, S_(stream)>>>(w, g, gidx, m, v, reinterpret_cast<const long long*>(unit_off), unit_cols, grad_scale, lr,
                                                       beta1, beta2, eps, weight_decay, clip_factor, agc_eps, adam_state);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_gather_cast_multi(const float* src, const int64_t* table, int32_t npacks, int64_t max_n, int32_t dtype, void* stream) {
  if (!src || !table || npacks < 1 || npacks > 65535 || max_n < 1) return set_error(BCOSK_EINVAL, "gather_cast_multi: bad argument");
  dim3 grid(grid_for((max_n + 1) / 2, 256, 1024), npacks);
  BCOSK_T_SWITCH(dtype, gather_cast_multi_kernel<T><<<grid, 256, 0, S_(stream)>>>(src, reinterpret_cast<const long long*>(table));)
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}
