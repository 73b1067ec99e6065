// bcosk_vit.cu -- bandwidth kernels of the fused SimpleViT plan (engine/vit.py) for sm_100a.
//
// The plan keeps every token tensor as [rows = images * tokens][planes * d] 16-bit precision planes (value = sum of planes),
// so the B-cos / plain linear layers run as 1x1 launches of the tcgen05 implicit GEMM with nothing in between but these
// kernels.  Reference: bcos/models/vit.py:143-158 (Attention), :160-185 (FeedForward), :290-339 (SimpleViT.forward),
// bcosify_vit.py:27-32 (MyGELU), bcos/modules/norms/centered_norms.py:187-224 (DetachableLayerNorm).
//
//   vit_patchify[_u8]    image -> patch rows "b c (h p1) (w p2) -> b h w (p1 p2 c)", normalised, + sum of squares per patch
//   vit_ln_fwd           LayerNorm over d of plane rows -> plane rows, 1/std per row (kept for the explanation pass)
//   vit_gelu_fwd         a = u * Phi(u) on plane rows + sum of squares per row; the saved gain of the producing B-cos linear
//                        is multiplied by the (detached) gate Phi(u), so the consumer's explain epilogue applies both at once
//   vit_ln_bwd           explanation backward of the LayerNorm (variance detached, mean in the graph) + residual-stream add:
//                        G_out = G_in + rstd * (g w - mean_d(g w)),  ghat = G_out * gain of the previous B-cos linear
//   vit_contrib_map[_u8] (x * grad).sum(channels) from the patch-embedding data gradient
//
// One warp per row, 16-byte vector accesses, warp-shuffle reductions, fp32 arithmetic.
#include "../../include/bcosk.h"
#include "bcosk_common.cuh"
#include "bcosk_host.h"

namespace bcosk {

struct F6 { float v[6]; };
static inline cudaStream_t SV(void* s) { return reinterpret_cast<cudaStream_t>(s); }

template <typename T>
__device__ __forceinline__ void unpack8v(const uint4& u, float (&f)[8]) {
  float2 q;
  q = Cvt<T>::unpack2(u.x); f[0] = q.x; f[1] = q.y;
  q = Cvt<T>::unpack2(u.y); f[2] = q.x; f[3] = q.y;
  q = Cvt<T>::unpack2(u.z); f[4] = q.x; f[5] = q.y;
  q = Cvt<T>::unpack2(u.w); f[6] = q.x; f[7] = q.y;
}

// 8 columns of a plane row -> fp32 (sum of planes)
template <typename T>
__device__ __forceinline__ void load8_row(const T* row, int planes, int plane_stride, int col, float (&f)[8]) {
  // all plane loads are issued before the first use (at most three planes; a runtime loop would serialise them)
  uint4 u[3];
  u[0] = __ldg(reinterpret_cast<const uint4*>(row + col));
#pragma unroll
  for (int pl = 1; pl < 3; ++pl)
    u[pl] = pl < planes ? __ldg(reinterpret_cast<const uint4*>(row + (size_t)pl * plane_stride + col)) : make_uint4(0u, 0u, 0u, 0u);
  unpack8v<T>(u[0], f);
#pragma unroll
  for (int pl = 1; pl < 3; ++pl) {
    float g[8];
    unpack8v<T>(u[pl], g);        // zero words unpack to +0.0 for both 16-bit formats
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] += g[i];
  }
}

// 8 values -> planes (plane 0 = rn(v), plane 1 = rn(v - plane 0), ...); v returns the stored value
template <typename T>
__device__ __forceinline__ void store8_row(T* row, int planes, int plane_stride, int col, float (&v)[8]) {
  float r[8], acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { r[i] = v[i]; acc[i] = 0.f; }
  for (int pl = 0; pl < planes; ++pl) {
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      w[k] = Cvt<T>::pack2(r[2 * k], r[2 * k + 1]);
      const float2 q = Cvt<T>::unpack2(w[k]);
      r[2 * k] -= q.x; r[2 * k + 1] -= q.y;
      acc[2 * k] += q.x; acc[2 * k + 1] += q.y;
    }
    *reinterpret_cast<uint4*>(row + (size_t)pl * plane_stride + col) = make_uint4(w[0], w[1], w[2], w[3]);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = acc[i];
}

__device__ __forceinline__ void load8_f32(const float* p, float (&f)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
__device__ __forceinline__ void store8_f32(float* p, const float (&f)[8]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(f[0], f[1], f[2], f[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(f[4], f[5], f[6], f[7]);
}

// ------------------------------------------------------------------------------------------------ patchify
// One CTA per patch, one thread per pixel of the patch (p*p threads).  out row = patch, column (p1*p + p2)*6 + c.
template <typename T, typename X>
__global__ void vit_patchify_kernel(const X* __restrict__ x, int H, int W, int p, F6 mean, F6 istd, T* __restrict__ out, int planes,
                                    float* __restrict__ sq) {
  __shared__ float red[32];
  const int gw = W / p, gh = H / p;
  const int patch = blockIdx.x;
  const int img = patch / (gh * gw), pr = patch - img * gh * gw;
  const int ph = pr / gw, pw = pr - ph * gw;
  const int t = threadIdx.x, p1 = t / p, p2 = t - p1 * p;
  const int yy = ph * p + p1, xx = pw * p + p2;
  float v[6];
  if (sizeof(X) == 1) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float r = (float)x[(((size_t)img * 3 + c) * H + yy) * W + xx] / 255.0f;
      v[c] = r;
      v[c + 3] = 1.0f - r;
    }
  } else {
#pragma unroll
    for (int c = 0; c < 6; ++c) v[c] = (float)x[(((size_t)img * 6 + c) * H + yy) * W + xx];
  }
#pragma unroll
  for (int c = 0; c < 6; ++c) v[c] = (v[c] - mean.v[c]) * istd.v[c];
  const int D = p * p * 6;
  T* row = out + (size_t)patch * planes * D + t * 6;
  float r[6], acc[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) { r[c] = v[c]; acc[c] = 0.f; }
  for (int pl = 0; pl < planes; ++pl) {
    uint32_t w[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      w[k] = Cvt<T>::pack2(r[2 * k], r[2 * k + 1]);
      const float2 q = Cvt<T>::unpack2(w[k]);
      r[2 * k] -= q.x; r[2 * k + 1] -= q.y;
      acc[2 * k] += q.x; acc[2 * k + 1] += q.y;
    }
    uint32_t* dst = reinterpret_cast<uint32_t*>(row + (size_t)pl * D);
    dst[0] = w[0]; dst[1] = w[1]; dst[2] = w[2];
  }
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < 6; ++c) s = fmaf(acc[c], acc[c], s);
  s = warp_sum(s);
  if ((t & 31) == 0) red[t >> 5] = s;
  __syncthreads();
  if (t < 32) {
    float a = t < (int)(blockDim.x >> 5) ? red[t] : 0.f;
    a = warp_sum(a);
    if (t == 0 && sq != nullptr) sq[patch] = a;
  }
}

// cmap[img, y, x] = sum_c x6[c] * g[patch, (p1 p + p2) 6 + c] * istd[c] * out_scale     (+ grad6 [img, 6, H, W])
template <typename X>
__global__ void vit_contrib_map_kernel(const float* __restrict__ g, const X* __restrict__ x, int H, int W, int p, F6 istd,
                                       float out_scale, float* __restrict__ cmap, float* __restrict__ grad6) {
  const int gw = W / p, gh = H / p;
  const int patch = blockIdx.x;
  const int img = patch / (gh * gw), pr = patch - img * gh * gw;
  const int ph = pr / gw, pw = pr - ph * gw;
  const int t = threadIdx.x, p1 = t / p, p2 = t - p1 * p;
  const int yy = ph * p + p1, xx = pw * p + p2;
  const float* gr = g + (size_t)patch * (p * p * 6) + t * 6;
  float acc = 0.f;
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    float xv;
    if (sizeof(X) == 1) {
      const float r = (float)x[(((size_t)img * 3 + (c % 3)) * H + yy) * W + xx] / 255.0f;
      xv = c < 3 ? r : 1.0f - r;
    } else {
      xv = (float)x[(((size_t)img * 6 + c) * H + yy) * W + xx];
    }
    const float g6 = __ldg(gr + c) * istd.v[c] * out_scale;
    acc = fmaf(xv, g6, acc);
    if (grad6 != nullptr) grad6[(((size_t)img * 6 + c) * H + yy) * W + xx] = g6;
  }
  cmap[((size_t)img * H + yy) * W + xx] = acc;
}

// ------------------------------------------------------------------------------------------------ LayerNorm forward
constexpr int LN_MAXV = 4;   // 8-column vectors per lane: d <= 1024
template <typename T>
__global__ void vit_ln_fwd_kernel(const T* __restrict__ x, long long rows, int d, int planes, int out_planes, const float* __restrict__ w,
                                  float eps, T* __restrict__ y, float* __restrict__ rstd_out, float* __restrict__ sq) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31, nvec = d >> 3;
  const T* xr = x + row * (long long)planes * d;
  float f[LN_MAXV][8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nvec) {
      load8_row<T>(xr, planes, d, v * 8, f[i]);
#pragma unroll
      for (int k = 0; k < 8; ++k) s += f[i][k];
    }
  }
  const float mean = warp_sum(s) / (float)d;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nvec) {
#pragma unroll
      for (int k = 0; k < 8; ++k) { f[i][k] -= mean; q = fmaf(f[i][k], f[i][k], q); }
    }
  }
  const float var = warp_sum(q) / (float)d;            // biased, like F.layer_norm
  const float rstd = 1.0f / sqrtf(var + eps);
  T* yr = y + row * (long long)out_planes * d;
  float sacc = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nvec) {
      float wv[8];
      load8_f32(w + v * 8, wv);
      float o[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = f[i][k] * rstd * wv[k];
      store8_row<T>(yr, out_planes, d, v * 8, o);
#pragma unroll
      for (int k = 0; k < 8; ++k) sacc = fmaf(o[k], o[k], sacc);
    }
  }
  sacc = warp_sum(sacc);
  if (lane == 0) {
    rstd_out[row] = rstd;
    if (sq != nullptr) sq[row] = sacc;
  }
}

// ------------------------------------------------------------------------------------------------ LayerNorm explanation backward
// g: gradient wrt the LayerNorm output ([rows][d], fp32 or one 16-bit plane); G_in / G_out: residual-stream gradient (fp32);
// ghat = G_out * gain ([rows][d] one 16-bit plane; gain 16-bit or fp32), the A operand of the previous linear's data gradient.
template <typename T>
__global__ void vit_ln_bwd_kernel(const void* __restrict__ g, int g_f32, const float* __restrict__ G_in, long long rows, int d,
                                  const float* __restrict__ w, const float* __restrict__ rstd, float* __restrict__ G_out,
                                  const void* __restrict__ gain, int gain_f32, T* __restrict__ ghat) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31, nvec = d >> 3;
  float f[LN_MAXV][8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nvec) {
      if (g_f32) load8_f32(reinterpret_cast<const float*>(g) + row * d + v * 8, f[i]);
      else unpack8v<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(g) + row * d + v * 8)), f[i]);
      float wv[8];
      load8_f32(w + v * 8, wv);
#pragma unroll
      for (int k = 0; k < 8; ++k) { f[i][k] *= wv[k]; s += f[i][k]; }
    }
  }
  const float mean = warp_sum(s) / (float)d;
  const float r = __ldg(rstd + row);
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nvec) {
      float o[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = r * (f[i][k] - mean);
      if (G_in != nullptr) {
        float a[8];
        load8_f32(G_in + row * d + v * 8, a);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] += a[k];
      }
      if (G_out != nullptr) store8_f32(G_out + row * d + v * 8, o);
      if (ghat != nullptr) {
        if (gain != nullptr) {
          float gn[8];
          if (gain_f32) load8_f32(reinterpret_cast<const float*>(gain) + row * d + v * 8, gn);
          else unpack8v<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(gain) + row * d + v * 8)), gn);
#pragma unroll
          for (int k = 0; k < 8; ++k) o[k] *= gn[k];
        }
        store8_row<T>(ghat + row * d, 1, 0, v * 8, o);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ GELU forward
template <typename T>
__global__ void vit_gelu_fwd_kernel(const T* __restrict__ u, long long rows, int d, int planes, T* __restrict__ a, float* __restrict__ sq,
                                    void* __restrict__ gain, int gain_f32) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31, nvec = d >> 3;
  const T* ur = u + row * (long long)planes * d;
  T* ar = a + row * (long long)planes * d;
  float sacc = 0.f;
  for (int v = lane; v < nvec; v += 32) {
    float f[8], gate[8];
    load8_row<T>(ur, planes, d, v * 8, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      gate[k] = 0.5f * (1.0f + erff(f[k] * 0.70710678118654752440f));
      f[k] *= gate[k];
    }
    store8_row<T>(ar, planes, d, v * 8, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) sacc = fmaf(f[k], f[k], sacc);
    if (gain != nullptr) {
      float gn[8];
      if (gain_f32) {
        float* gp = reinterpret_cast<float*>(gain) + row * d + v * 8;
        load8_f32(gp, gn);
#pragma unroll
        for (int k = 0; k < 8; ++k) gn[k] *= gate[k];
        store8_f32(gp, gn);
      } else {
        T* gp = reinterpret_cast<T*>(gain) + row * d + v * 8;
        unpack8v<T>(*reinterpret_cast<const uint4*>(gp), gn);
#pragma unroll
        for (int k = 0; k < 8; ++k) gn[k] *= gate[k];
        store8_row<T>(gp, 1, 0, 0, gn);
      }
    }
  }
  sacc = warp_sum(sacc);
  if (lane == 0 && sq != nullptr) sq[row] = sacc;
}

// ------------------------------------------------------------------------------------------------ attention on plane rows
// One CTA per (image, head).  qkv rows: [n tokens][planes * 3*H*D] (q | k | v blocks of every plane, head h at h*D), D = 64.
//   forward : out[n][planes * H*D] = softmax(q k^T * scale) v                     (written as planes)
//   backward: gv [n][H*D] one 16-bit plane = P^T g,  g: [n][H*D] fp32            (q, k frozen: bcos/models/vit.py:148-150)
// P (n x n fp32) lives in shared memory, recomputed from q, k in the backward.
constexpr int VAT_D = 64;
template <typename T, bool BWD>
__global__ void __launch_bounds__(256, 1)
vit_attention_kernel(const T* __restrict__ qkv, int planes, const float* __restrict__ g, int n, int heads, float scale, T* __restrict__ out) {
  extern __shared__ float sm[];
  float* P = sm;                       // [n][n]
  float* buf = sm + (size_t)n * n;     // [n][VAT_D + 1]
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int hd = heads * VAT_D, pst = 3 * hd, ld = planes * pst;
  const T* base = qkv + (size_t)b * n * ld + h * VAT_D;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  constexpr int LDB = VAT_D + 1;
  auto stage = [&](int block_off) {      // q / k / v block of this head -> buf (fp32, planes summed); 8 columns per thread step
    for (int i = threadIdx.x; i < n * (VAT_D / 8); i += blockDim.x) {
      const int r = i / (VAT_D / 8), c8 = (i % (VAT_D / 8)) * 8;
      float f[8];
      load8_row<T>(base + (size_t)r * ld + block_off, planes, pst, c8, f);
#pragma unroll
      for (int k = 0; k < 8; ++k) buf[r * LDB + c8 + k] = f[k];
    }
  };
  stage(hd);                             // K
  __syncthreads();
  for (int i = warp; i < n; i += nw) {
    // lane l holds columns l and l + 32 of query row i (planes summed)
    float qi0 = 0.f, qi1 = 0.f;
    for (int pl = 0; pl < planes; ++pl) {
      qi0 += (float)base[(size_t)i * ld + (size_t)pl * pst + lane];
      qi1 += (float)base[(size_t)i * ld + (size_t)pl * pst + lane + 32];
    }
    float mx = -INFINITY;
    for (int j0 = 0; j0 < n; j0 += 32) {
      const int j = j0 + lane;
      float s = 0.f;
#pragma unroll
      for (int dd = 0; dd < 32; ++dd) {
        const float q0 = __shfl_sync(0xffffffffu, qi0, dd), q1 = __shfl_sync(0xffffffffu, qi1, dd);
        if (j < n) s = fmaf(q0, buf[j * LDB + dd], fmaf(q1, buf[j * LDB + dd + 32], s));
      }
      s *= scale;
      if (j < n) { P[(size_t)i * n + j] = s; mx = fmaxf(mx, s); }
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int j = lane; j < n; j += 32) {
      const float e = expf(P[(size_t)i * n + j] - mx);
      P[(size_t)i * n + j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    for (int j = lane; j < n; j += 32) P[(size_t)i * n + j] *= inv;
  }
  __syncthreads();
  if (!BWD) {
    stage(2 * hd);                       // V
  } else {
    const float* gh = g + (size_t)b * n * hd + h * VAT_D;
    for (int i = threadIdx.x; i < n * VAT_D; i += blockDim.x)
      buf[(i / VAT_D) * LDB + (i % VAT_D)] = __ldg(gh + (size_t)(i / VAT_D) * hd + (i % VAT_D));
  }
  __syncthreads();
  for (int r = warp; r < n; r += nw) {
    float a0 = 0.f, a1 = 0.f;
    for (int t = 0; t < n; ++t) {
      const float pw = BWD ? P[(size_t)t * n + r] : P[(size_t)r * n + t];
      a0 = fmaf(pw, buf[t * LDB + lane], a0);
      a1 = fmaf(pw, buf[t * LDB + lane + 32], a1);
    }
    const int op = BWD ? 1 : planes;
    T* o = out + ((size_t)b * n + r) * (op * hd) + h * VAT_D;
    float r0 = a0, r1 = a1;
    for (int pl = 0; pl < op; ++pl) {
      const float h0 = Cvt<T>::round1(r0), h1 = Cvt<T>::round1(r1);
      o[(size_t)pl * hd + lane] = T(h0);
      o[(size_t)pl * hd + lane + 32] = T(h1);
      r0 -= h0; r1 -= h1;
    }
  }
}

// ------------------------------------------------------------------------------------------------ CLIP ViT encoder (engine/clip_vit.py)
// The reference leaves CLIP's LayerNorm, QuickGELU and nn.MultiheadAttention untouched (bcosify.py:74-113 converts only conv1 and the
// MLP linears), so its explanation pass differentiates them exactly: these are the TRUE backward forms.

// LayerNorm backward (nothing detached): with xh = (x - mean) rstd and gw = g w,
//   G_out = G_in + rstd * (gw - mean_d(gw) - xh * mean_d(gw xh));  ghat = G_out (* gain) as one 16-bit plane.
template <typename T>
__global__ void vit_ln_bwd_full_kernel(const void* __restrict__ g, int g_f32, const T* __restrict__ x, int planes, const float* __restrict__ G_in,
                                       long long rows, int d, const float* __restrict__ w, const float* __restrict__ rstd,
                                       float* __restrict__ G_out, const void* __restrict__ gain, int gain_f32, T* __restrict__ ghat) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31, nvec = d >> 3;
  const T* xr = x + row * (long long)planes * d;
  float f[LN_MAXV][8], xh[LN_MAXV][8];
  float s = 0.f, sx = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nvec) {
      if (g_f32) load8_f32(reinterpret_cast<const float*>(g) + row * d + v * 8, f[i]);
      else unpack8v<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(g) + row * d + v * 8)), f[i]);
      float wv[8];
      load8_f32(w + v * 8, wv);
      load8_row<T>(xr, planes, d, v * 8, xh[i]);
#pragma unroll
      for (int k = 0; k < 8; ++k) { f[i][k] *= wv[k]; s += f[i][k]; sx += xh[i][k]; }
    }
  }
  const float mean_g = warp_sum(s) / (float)d;
  const float mean_x = warp_sum(sx) / (float)d;
  const float r = __ldg(rstd + row);
  float sgx = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nvec) {
#pragma unroll
      for (int k = 0; k < 8; ++k) { xh[i][k] = (xh[i][k] - mean_x) * r; sgx = fmaf(f[i][k], xh[i][k], sgx); }
    }
  }
  const float mean_gx = warp_sum(sgx) / (float)d;
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nvec) {
      float o[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = r * (f[i][k] - mean_g - xh[i][k] * mean_gx);
      if (G_in != nullptr) {
        float a[8];
        load8_f32(G_in + row * d + v * 8, a);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] += a[k];
      }
      if (G_out != nullptr) store8_f32(G_out + row * d + v * 8, o);
      if (ghat != nullptr) {
        if (gain != nullptr) {
          float gn[8];
          if (gain_f32) load8_f32(reinterpret_cast<const float*>(gain) + row * d + v * 8, gn);
          else unpack8v<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(gain) + row * d + v * 8)), gn);
#pragma unroll
          for (int k = 0; k < 8; ++k) o[k] *= gn[k];
        }
        store8_row<T>(ghat + row * d, 1, 0, v * 8, o);
      }
    }
  }
}

// QuickGELU (CLIP/clip/model.py:166-168): a = u * sigmoid(1.702 u); the saved gain of the producing B-cos linear is multiplied by the
// TRUE derivative sigmoid + 1.702 u sigmoid (1 - sigmoid) (the reference does not detach this activation).
template <typename T>
__global__ void vit_quickgelu_fwd_kernel(const T* __restrict__ u, long long rows, int d, int planes, T* __restrict__ a, float* __restrict__ sq,
                                         void* __restrict__ gain, int gain_f32) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31, nvec = d >> 3;
  const T* ur = u + row * (long long)planes * d;
  T* ar = a + row * (long long)planes * d;
  float sacc = 0.f;
  for (int v = lane; v < nvec; v += 32) {
    float f[8], dv[8];
    load8_row<T>(ur, planes, d, v * 8, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float sg = 1.0f / (1.0f + expf(-1.702f * f[k]));
      dv[k] = sg + 1.702f * f[k] * sg * (1.0f - sg);
      f[k] *= sg;
    }
    store8_row<T>(ar, planes, d, v * 8, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) sacc = fmaf(f[k], f[k], sacc);
    if (gain != nullptr) {
      float gn[8];
      if (gain_f32) {
        float* gp = reinterpret_cast<float*>(gain) + row * d + v * 8;
        load8_f32(gp, gn);
#pragma unroll
        for (int k = 0; k < 8; ++k) gn[k] *= dv[k];
        store8_f32(gp, gn);
      } else {
        T* gp = reinterpret_cast<T*>(gain) + row * d + v * 8;
        unpack8v<T>(*reinterpret_cast<const uint4*>(gp), gn);
#pragma unroll
        for (int k = 0; k < 8; ++k) gn[k] *= dv[k];
        store8_row<T>(gp, 1, 0, 0, gn);
      }
    }
  }
  sacc = warp_sum(sacc);
  if (lane == 0 && sq != nullptr) sq[row] = sacc;
}

// Full attention backward (nothing frozen), one CTA per (image, head), n <= 112 tokens (shared memory), D = 64.  With z = scale q k^T, P = softmax(z):
//   dV = P^T g;  dP = g V^T;  dz = P o (dP - rowsum(P o dP));  dQ = scale dz K;  dK = scale dz^T Q.
// out [n][3*H*D] one 16-bit plane (q | k | v blocks): the A operand of the in_proj data gradient.
template <typename T>
__global__ void __launch_bounds__(256, 1)
vit_attention_bwd_full_kernel(const T* __restrict__ qkv, int planes, const float* __restrict__ g, int n, int heads, float scale, T* __restrict__ out) {
  extern __shared__ float sm[];
  constexpr int LDB = VAT_D + 1;
  float* P = sm;                                   // [n][n]  probabilities
  float* DZ = P + (size_t)n * n;                    // [n][n]  dP, then dz * scale
  float* sq_ = DZ + (size_t)n * n;                  // [n][LDB] q
  float* sk = sq_ + (size_t)n * LDB;                // k
  float* sv = sk + (size_t)n * LDB;                 // v
  float* sg = sv + (size_t)n * LDB;                 // g
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int hd = heads * VAT_D, pst = 3 * hd, ld = planes * pst;
  const T* base = qkv + (size_t)b * n * ld + h * VAT_D;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int i = threadIdx.x; i < n * (VAT_D / 8); i += blockDim.x) {
    const int r = i / (VAT_D / 8), c8 = (i % (VAT_D / 8)) * 8;
    float f[8];
    load8_row<T>(base + (size_t)r * ld, planes, pst, c8, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) sq_[r * LDB + c8 + k] = f[k];
    load8_row<T>(base + (size_t)r * ld + hd, planes, pst, c8, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) sk[r * LDB + c8 + k] = f[k];
    load8_row<T>(base + (size_t)r * ld + 2 * hd, planes, pst, c8, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) sv[r * LDB + c8 + k] = f[k];
  }
  const float* gh = g + (size_t)b * n * hd + h * VAT_D;
  for (int i = threadIdx.x; i < n * VAT_D; i += blockDim.x) sg[(i / VAT_D) * LDB + (i % VAT_D)] = __ldg(gh + (size_t)(i / VAT_D) * hd + (i % VAT_D));
  __syncthreads();
  // rows of P and dz (one warp per query row; lane = key j, j + 32, ...)
  for (int i = warp; i < n; i += nw) {
    float mx = -INFINITY;
    for (int j = lane; j < n; j += 32) {
      float s = 0.f;
#pragma unroll 16
      for (int dd = 0; dd < VAT_D; ++dd) s = fmaf(sq_[i * LDB + dd], sk[j * LDB + dd], s);
      s *= scale;
      P[(size_t)i * n + j] = s;
      mx = fmaxf(mx, s);
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int j = lane; j < n; j += 32) {
      const float e = expf(P[(size_t)i * n + j] - mx);
      P[(size_t)i * n + j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    for (int j = lane; j < n; j += 32) P[(size_t)i * n + j] *= inv;
  }
  __syncthreads();
  // dV[j] = sum_i P[i][j] g[i]
  T* obase = out + (size_t)b * n * pst + h * VAT_D;
  for (int j = warp; j < n; j += nw) {
    float a0 = 0.f, a1 = 0.f;
    for (int i = 0; i < n; ++i) {
      const float pw = P[(size_t)i * n + j];
      a0 = fmaf(pw, sg[i * LDB + lane], a0);
      a1 = fmaf(pw, sg[i * LDB + lane + 32], a1);
    }
    obase[(size_t)j * pst + 2 * hd + lane] = T(a0);
    obase[(size_t)j * pst + 2 * hd + lane + 32] = T(a1);
  }
  __syncthreads();
  // dz[i][j] = P (dP - sum_j P dP) * scale, dP[i][j] = g[i] . v[j]   (one warp per query row; dz goes to its own n x n buffer)
  for (int i = warp; i < n; i += nw) {
    float acc = 0.f;
    for (int jj = lane; jj < n; jj += 32) {
      float dp = 0.f;
#pragma unroll 16
      for (int dd = 0; dd < VAT_D; ++dd) dp = fmaf(sg[i * LDB + dd], sv[jj * LDB + dd], dp);
      DZ[(size_t)i * n + jj] = dp;
      acc = fmaf(P[(size_t)i * n + jj], dp, acc);
    }
    acc = warp_sum(acc);
    for (int jj = lane; jj < n; jj += 32) DZ[(size_t)i * n + jj] = P[(size_t)i * n + jj] * (DZ[(size_t)i * n + jj] - acc) * scale;
  }
  __syncthreads();
  // dQ[i] = sum_j dz[i][j] k[j];  dK[j] = sum_i dz[i][j] q[i]
  for (int r = warp; r < n; r += nw) {
    float q0 = 0.f, q1 = 0.f, k0 = 0.f, k1 = 0.f;
    for (int t = 0; t < n; ++t) {
      const float a = DZ[(size_t)r * n + t], bb = DZ[(size_t)t * n + r];
      q0 = fmaf(a, sk[t * LDB + lane], q0);
      q1 = fmaf(a, sk[t * LDB + lane + 32], q1);
      k0 = fmaf(bb, sq_[t * LDB + lane], k0);
      k1 = fmaf(bb, sq_[t * LDB + lane + 32], k1);
    }
    obase[(size_t)r * pst + lane] = T(q0);
    obase[(size_t)r * pst + lane + 32] = T(q1);
    obase[(size_t)r * pst + hd + lane] = T(k0);
    obase[(size_t)r * pst + hd + lane + 32] = T(k1);
  }
}

// The same gradients for longer sequences (113..208 tokens: CLIP ViT-B/16 has 197), where two n x n fp32 blocks no longer fit shared memory:
// nothing n x n is kept.  Pass 1 (a warp per query row) leaves the softmax statistics m_i, l_i and D_i = sum_j P_ij dP_ij; pass 2 (per
// query row) and pass 3 (per key column) recompute s_ij, P_ij, dP_ij and dz_ij = P_ij (dP_ij - D_i) scale from q, k, v, g in shared
// memory and reduce them through one per-warp row buffer.  3x the dot products of the block form, same formulas.
template <typename T>
__global__ void __launch_bounds__(256, 1)
vit_attention_bwd_full_long_kernel(const T* __restrict__ qkv, int planes, const float* __restrict__ g, int n, int heads, float scale, T* __restrict__ out) {
  extern __shared__ float sm[];
  constexpr int LDB = VAT_D + 1;
  float* sq_ = sm;                                  // [n][LDB] q
  float* sk = sq_ + (size_t)n * LDB;                // k
  float* sv = sk + (size_t)n * LDB;                 // v
  float* sg = sv + (size_t)n * LDB;                 // g
  float* sm_ = sg + (size_t)n * LDB;                // [n] row maximum of z
  float* sl = sm_ + n;                              // [n] 1 / sum exp
  float* sD = sl + n;                               // [n] sum_j P dP
  const int nw = blockDim.x >> 5;
  float* rowA = sD + n;                             // [nw][n] per-warp row buffers
  float* rowB = rowA + (size_t)nw * n;
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int hd = heads * VAT_D, pst = 3 * hd, ld = planes * pst;
  const T* base = qkv + (size_t)b * n * ld + h * VAT_D;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < n * (VAT_D / 8); i += blockDim.x) {
    const int r = i / (VAT_D / 8), c8 = (i % (VAT_D / 8)) * 8;
    float f[8];
    load8_row<T>(base + (size_t)r * ld, planes, pst, c8, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) sq_[r * LDB + c8 + k] = f[k];
    load8_row<T>(base + (size_t)r * ld + hd, planes, pst, c8, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) sk[r * LDB + c8 + k] = f[k];
    load8_row<T>(base + (size_t)r * ld + 2 * hd, planes, pst, c8, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) sv[r * LDB + c8 + k] = f[k];
  }
  const float* gh = g + (size_t)b * n * hd + h * VAT_D;
  for (int i = threadIdx.x; i < n * VAT_D; i += blockDim.x) sg[(i / VAT_D) * LDB + (i % VAT_D)] = __ldg(gh + (size_t)(i / VAT_D) * hd + (i % VAT_D));
  __syncthreads();
  auto dot = [&](const float* a, const float* c) {
    float s = 0.f;
#pragma unroll 16
    for (int dd = 0; dd < VAT_D; ++dd) s = fmaf(a[dd], c[dd], s);
    return s;
  };
  float* ra = rowA + (size_t)warp * n;
  float* rb = rowB + (size_t)warp * n;
  T* obase = out + (size_t)b * n * pst + h * VAT_D;
  // ---- pass 1 + 2: a warp per query row i: statistics, then dz_i[.] -> dQ_i
  for (int i = warp; i < n; i += nw) {
    float mx = -INFINITY;
    for (int j = lane; j < n; j += 32) {
      const float s = dot(sq_ + i * LDB, sk + j * LDB) * scale;
      ra[j] = s;
      mx = fmaxf(mx, s);
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int j = lane; j < n; j += 32) {
      const float e = expf(ra[j] - mx);
      ra[j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    float acc = 0.f;
    for (int j = lane; j < n; j += 32) {
      const float pj = ra[j] * inv;
      const float dp = dot(sg + i * LDB, sv + j * LDB);
      ra[j] = pj;
      rb[j] = dp;
      acc = fmaf(pj, dp, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) { sm_[i] = mx; sl[i] = inv; sD[i] = acc; }
    for (int j = lane; j < n; j += 32) rb[j] = ra[j] * (rb[j] - acc) * scale;      // dz_i[j]
    __syncwarp();
    float q0 = 0.f, q1 = 0.f;
    for (int t = 0; t < n; ++t) {
      const float a = rb[t];
      q0 = fmaf(a, sk[t * LDB + lane], q0);
      q1 = fmaf(a, sk[t * LDB + lane + 32], q1);
    }
    obase[(size_t)i * pst + lane] = T(q0);
    obase[(size_t)i * pst + lane + 32] = T(q1);
    __syncwarp();
  }
  __syncthreads();
  // ---- pass 3: a warp per key column j: P_.j and dz_.j recomputed -> dV_j, dK_j
  for (int j = warp; j < n; j += nw) {
    for (int i = lane; i < n; i += 32) {
      const float s = dot(sq_ + i * LDB, sk + j * LDB) * scale;
      const float pj = expf(s - sm_[i]) * sl[i];
      const float dp = dot(sg + i * LDB, sv + j * LDB);
      ra[i] = pj;
      rb[i] = pj * (dp - sD[i]) * scale;
    }
    __syncwarp();
    float v0 = 0.f, v1 = 0.f, k0 = 0.f, k1 = 0.f;
    for (int t = 0; t < n; ++t) {
      const float pw = ra[t], dz = rb[t];
      v0 = fmaf(pw, sg[t * LDB + lane], v0);
      v1 = fmaf(pw, sg[t * LDB + lane + 32], v1);
      k0 = fmaf(dz, sq_[t * LDB + lane], k0);
      k1 = fmaf(dz, sq_[t * LDB + lane + 32], k1);
    }
    obase[(size_t)j * pst + 2 * hd + lane] = T(v0);
    obase[(size_t)j * pst + 2 * hd + lane + 32] = T(v1);
    obase[(size_t)j * pst + hd + lane] = T(k0);
    obase[(size_t)j * pst + hd + lane + 32] = T(k1);
    __syncwarp();
  }
}

}  // namespace bcosk

using namespace bcosk;

#define VIT_DISPATCH(dtype, CALL_BF16, CALL_F16)                         \
  if ((dtype) == BCOSK_DTYPE_BF16) { CALL_BF16; }                        \
  else if ((dtype) == BCOSK_DTYPE_F16) { CALL_F16; }                     \
  else return set_error(BCOSK_EINVAL, "vit kernel: dtype");

static F6 make_f6(const float* p) {
  F6 f;
  for (int i = 0; i < 6; ++i) f.v[i] = p[i];
  return f;
}

template <typename X>
static int vit_patchify_impl(const X* x, int32_t nb, int32_t h, int32_t w, int32_t p, const float* mean6, const float* inv_std6,
                             void* out, int32_t planes, int32_t dtype, float* sq, void* stream) {
  if (!x || !out || !mean6 || !inv_std6 || nb < 1 || p < 2 || h % p || w % p || (p * p) % 32 || p * p > 1024 || planes < 1 || planes > 3)
    return set_error(BCOSK_EINVAL, "vit_patchify: bad argument");
  const unsigned grid = (unsigned)((long long)nb * (h / p) * (w / p));
  const F6 m = make_f6(mean6), s = make_f6(inv_std6);
  VIT_DISPATCH(dtype,
               (vit_patchify_kernel<__nv_bfloat16, X><<<grid, p * p, 0, SV(stream)>>>(x, h, w, p, m, s, reinterpret_cast<__nv_bfloat16*>(out), planes, sq)),
               (vit_patchify_kernel<__half, X><<<grid, p * p, 0, SV(stream)>>>(x, h, w, p, m, s, reinterpret_cast<__half*>(out), planes, sq)))
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_vit_patchify(const float* x, int32_t nb, int32_t h, int32_t w, int32_t p, const float* mean6, const float* inv_std6,
                                  void* out, int32_t planes, int32_t dtype, float* sq, void* stream) {
  return vit_patchify_impl<float>(x, nb, h, w, p, mean6, inv_std6, out, planes, dtype, sq, stream);
}
extern "C" int bcosk_vit_patchify_u8(const uint8_t* x, int32_t nb, int32_t h, int32_t w, int32_t p, const float* mean6,
                                     const float* inv_std6, void* out, int32_t planes, int32_t dtype, float* sq, void* stream) {
  return vit_patchify_impl<uint8_t>(x, nb, h, w, p, mean6, inv_std6, out, planes, dtype, sq, stream);
}

template <typename X>
static int vit_contrib_impl(const float* g, const X* x, int32_t nb, int32_t h, int32_t w, int32_t p, const float* inv_std6, float out_scale,
                            float* cmap, float* grad6, void* stream) {
  if (!g || !x || !cmap || !inv_std6 || nb < 1 || p < 2 || h % p || w % p || p * p > 1024)
    return set_error(BCOSK_EINVAL, "vit_contrib_map: bad argument");
  const unsigned grid = (unsigned)((long long)nb * (h / p) * (w / p));
  vit_contrib_map_kernel<X><<<grid, p * p, 0, SV(stream)>>>(g, x, h, w, p, make_f6(inv_std6), out_scale, cmap, grad6);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}
extern "C" int bcosk_vit_contrib_map(const float* g, const float* x, int32_t nb, int32_t h, int32_t w, int32_t p, const float* inv_std6,
                                     float out_scale, float* cmap, float* grad6, void* stream) {
  return vit_contrib_impl<float>(g, x, nb, h, w, p, inv_std6, out_scale, cmap, grad6, stream);
}
extern "C" int bcosk_vit_contrib_map_u8(const float* g, const uint8_t* x, int32_t nb, int32_t h, int32_t w, int32_t p,
                                        const float* inv_std6, float out_scale, float* cmap, float* grad6, void* stream) {
  return vit_contrib_impl<uint8_t>(g, x, nb, h, w, p, inv_std6, out_scale, cmap, grad6, stream);
}

extern "C" int bcosk_vit_ln_fwd(const void* x, int64_t rows, int32_t d, int32_t planes, int32_t out_planes, const float* w, float eps, void* y,
                                float* rstd, float* sq, int32_t dtype, void* stream) {
  if (out_planes == 0) out_planes = planes;
  if (!x || !y || !w || !rstd || rows < 1 || d % 8 || d > 256 * LN_MAXV || planes < 1 || planes > 3 || out_planes < 1 || out_planes > 3)
    return set_error(BCOSK_EINVAL, "vit_ln_fwd: bad argument (d must be a multiple of 8, <= 1024)");
  const unsigned grid = (unsigned)((rows + 7) / 8);
  VIT_DISPATCH(dtype,
               (vit_ln_fwd_kernel<__nv_bfloat16><<<grid, 256, 0, SV(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(x), rows, d, planes, out_planes, w, eps,
                                                                             reinterpret_cast<__nv_bfloat16*>(y), rstd, sq)),
               (vit_ln_fwd_kernel<__half><<<grid, 256, 0, SV(stream)>>>(reinterpret_cast<const __half*>(x), rows, d, planes, out_planes, w, eps,
                                                                      reinterpret_cast<__half*>(y), rstd, sq)))
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_vit_ln_bwd(const void* g, int32_t g_f32, const float* G_in, int64_t rows, int32_t d, const float* w, const float* rstd,
                                float* G_out, const void* gain, int32_t gain_f32, void* ghat, int32_t dtype, void* stream) {
  if (!g || !w || !rstd || (!G_out && !ghat) || rows < 1 || d % 8 || d > 256 * LN_MAXV)
    return set_error(BCOSK_EINVAL, "vit_ln_bwd: bad argument");
  const unsigned grid = (unsigned)((rows + 7) / 8);
  VIT_DISPATCH(dtype,
               (vit_ln_bwd_kernel<__nv_bfloat16><<<grid, 256, 0, SV(stream)>>>(g, g_f32, G_in, rows, d, w, rstd, G_out, gain, gain_f32,
                                                                             reinterpret_cast<__nv_bfloat16*>(ghat))),
               (vit_ln_bwd_kernel<__half><<<grid, 256, 0, SV(stream)>>>(g, g_f32, G_in, rows, d, w, rstd, G_out, gain, gain_f32,
                                                                      reinterpret_cast<__half*>(ghat))))
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_vit_gelu_fwd(const void* u, int64_t rows, int32_t d, int32_t planes, void* a, float* sq, void* gain, int32_t gain_f32,
                                  int32_t dtype, void* stream) {
  if (!u || !a || rows < 1 || d % 8 || planes < 1 || planes > 3) return set_error(BCOSK_EINVAL, "vit_gelu_fwd: bad argument");
  const unsigned grid = (unsigned)((rows + 7) / 8);
  VIT_DISPATCH(dtype,
               (vit_gelu_fwd_kernel<__nv_bfloat16><<<grid, 256, 0, SV(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(u), rows, d, planes,
                                                                               reinterpret_cast<__nv_bfloat16*>(a), sq, gain, gain_f32)),
               (vit_gelu_fwd_kernel<__half><<<grid, 256, 0, SV(stream)>>>(reinterpret_cast<const __half*>(u), rows, d, planes,
                                                                        reinterpret_cast<__half*>(a), sq, gain, gain_f32)))
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_vit_attention(const void* qkv, int32_t planes, const float* g, int32_t batch, int32_t n, int32_t heads, int32_t dim_head,
                                   float scale, int32_t backward, void* out, int32_t dtype, void* stream) {
  if (!qkv || !out || (backward && !g) || planes < 1 || planes > 3) return set_error(BCOSK_EINVAL, "vit_attention: bad argument");
  if (dim_head != VAT_D) return set_error(BCOSK_EUNSUPPORTED, "vit_attention: dim_head must be 64");
  const size_t smem = ((size_t)n * n + (size_t)n * (VAT_D + 1)) * sizeof(float);
  if (smem > 227 * 1024) return set_error(BCOSK_EUNSUPPORTED, "vit_attention: sequence too long for the shared-memory kernel (n <= 208)");
#define VAT_LAUNCH(T_, BWD_)                                                                                                      \
  do {                                                                                                                            \
    BCOSK_CUDA_CHECK(cudaFuncSetAttribute(vit_attention_kernel<T_, BWD_>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); \
    vit_attention_kernel<T_, BWD_><<<batch * heads, 256, smem, SV(stream)>>>(reinterpret_cast<const T_*>(qkv), planes, g, n, heads,   \
                                                                            scale, reinterpret_cast<T_*>(out));                     \
  } while (0)
  if (dtype == BCOSK_DTYPE_BF16) {
    if (backward) VAT_LAUNCH(__nv_bfloat16, true); else VAT_LAUNCH(__nv_bfloat16, false);
  } else if (dtype == BCOSK_DTYPE_F16) {
    if (backward) VAT_LAUNCH(__half, true); else VAT_LAUNCH(__half, false);
  } else {
    return set_error(BCOSK_EINVAL, "vit_attention: dtype");
  }
#undef VAT_LAUNCH
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_vit_ln_bwd_full(const void* g, int32_t g_f32, const void* x, int32_t planes, const float* G_in, int64_t rows, int32_t d,
                                     const float* w, const float* rstd, float* G_out, const void* gain, int32_t gain_f32, void* ghat,
                                     int32_t dtype, void* stream) {
  if (!g || !x || !w || !rstd || (!G_out && !ghat) || rows < 1 || d % 8 || d > 256 * LN_MAXV || planes < 1 || planes > 3)
    return set_error(BCOSK_EINVAL, "vit_ln_bwd_full: bad argument");
  const unsigned grid = (unsigned)((rows + 7) / 8);
  VIT_DISPATCH(dtype,
               (vit_ln_bwd_full_kernel<__nv_bfloat16><<<grid, 256, 0, SV(stream)>>>(g, g_f32, reinterpret_cast<const __nv_bfloat16*>(x), planes, G_in, rows, d, w,
                                                                                  rstd, G_out, gain, gain_f32, reinterpret_cast<__nv_bfloat16*>(ghat))),
               (vit_ln_bwd_full_kernel<__half><<<grid, 256, 0, SV(stream)>>>(g, g_f32, reinterpret_cast<const __half*>(x), planes, G_in, rows, d, w, rstd,
                                                                           G_out, gain, gain_f32, reinterpret_cast<__half*>(ghat))))
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_vit_quickgelu_fwd(const void* u, int64_t rows, int32_t d, int32_t planes, void* a, float* sq, void* gain, int32_t gain_f32,
                                       int32_t dtype, void* stream) {
  if (!u || !a || rows < 1 || d % 8 || planes < 1 || planes > 3) return set_error(BCOSK_EINVAL, "vit_quickgelu_fwd: bad argument");
  const unsigned grid = (unsigned)((rows + 7) / 8);
  VIT_DISPATCH(dtype,
               (vit_quickgelu_fwd_kernel<__nv_bfloat16><<<grid, 256, 0, SV(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(u), rows, d, planes,
                                                                                    reinterpret_cast<__nv_bfloat16*>(a), sq, gain, gain_f32)),
               (vit_quickgelu_fwd_kernel<__half><<<grid, 256, 0, SV(stream)>>>(reinterpret_cast<const __half*>(u), rows, d, planes,
                                                                             reinterpret_cast<__half*>(a), sq, gain, gain_f32)))
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_vit_attention_bwd_full(const void* qkv, int32_t planes, const float* g, int32_t batch, int32_t n, int32_t heads, int32_t dim_head,
                                            float scale, void* out, int32_t dtype, void* stream) {
  if (!qkv || !g || !out || planes < 1 || planes > 3 || batch < 1) return set_error(BCOSK_EINVAL, "vit_attention_bwd_full: bad argument");
  if (dim_head != VAT_D) return set_error(BCOSK_EUNSUPPORTED, "vit_attention_bwd_full: dim_head must be 64");
  size_t smem = (2 * (size_t)n * n + 4 * (size_t)n * (VAT_D + 1)) * sizeof(float);
  if (smem > 227 * 1024) {
    // longer sequences (CLIP ViT-B/16: 197 tokens): the recomputing form, nothing n x n in shared memory
    smem = (4 * (size_t)n * (VAT_D + 1) + 3 * (size_t)n + 2 * 8 * (size_t)n) * sizeof(float);
    if (smem > 227 * 1024) return set_error(BCOSK_EUNSUPPORTED, "vit_attention_bwd_full: sequence too long for the shared-memory kernels (n <= 208)");
    if (dtype == BCOSK_DTYPE_BF16) {
      BCOSK_CUDA_CHECK(cudaFuncSetAttribute(vit_attention_bwd_full_long_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      vit_attention_bwd_full_long_kernel<__nv_bfloat16><<<batch * heads, 256, smem, SV(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(qkv), planes, g, n, heads,
                                                                                                 scale, reinterpret_cast<__nv_bfloat16*>(out));
    } else if (dtype == BCOSK_DTYPE_F16) {
      BCOSK_CUDA_CHECK(cudaFuncSetAttribute(vit_attention_bwd_full_long_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      vit_attention_bwd_full_long_kernel<__half><<<batch * heads, 256, smem, SV(stream)>>>(reinterpret_cast<const __half*>(qkv), planes, g, n, heads, scale,
                                                                                          reinterpret_cast<__half*>(out));
    } else {
      return set_error(BCOSK_EINVAL, "vit_attention_bwd_full: dtype");
    }
    BCOSK_CUDA_CHECK(cudaGetLastError());
    return BCOSK_OK;
  }
  if (dtype == BCOSK_DTYPE_BF16) {
    BCOSK_CUDA_CHECK(cudaFuncSetAttribute(vit_attention_bwd_full_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    vit_attention_bwd_full_kernel<__nv_bfloat16><<<batch * heads, 256, smem, SV(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(qkv), planes, g, n, heads, scale,
                                                                                          reinterpret_cast<__nv_bfloat16*>(out));
  } else if (dtype == BCOSK_DTYPE_F16) {
    BCOSK_CUDA_CHECK(cudaFuncSetAttribute(vit_attention_bwd_full_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    vit_attention_bwd_full_kernel<__half><<<batch * heads, 256, smem, SV(stream)>>>(reinterpret_cast<const __half*>(qkv), planes, g, n, heads, scale,
                                                                                   reinterpret_cast<__half*>(out));
  } else {
    return set_error(BCOSK_EINVAL, "vit_attention_bwd_full: dtype");
  }
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}
