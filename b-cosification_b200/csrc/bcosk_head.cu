// bcosk_head.cu -- the attention-pool head of the CLIP ResNet encoders inside the fused plan (engine/clip_rn.py), sm_100a.
//
// Reference: BcosAttentionPool2d.forward bcos/modules/bcosattnpool.py:34-59 (pooled mode: the query is the mean token, q and k are
// detached in explanation mode, bias-free projections, c_proj used as a plain linear map).  Only the mean token's output is kept, so
// the projections commute with the pooling: per head h
//     s_j = q_h . (W_k,h x_j) = (W_k,h^T q_h) . x_j            p = softmax_j(s)
//     o_h = sum_j p_j (W_v,h x_j) = W_v,h (sum_j p_j x_j)
// i.e. three token-equivalents of 2048 x 2048 projections per image instead of 150 (q, k, v of 50 tokens), plus small batched
// products.  Everything here is fp32 on the CUDA cores (32 GFLOP per 512 images): a strided-batched SGEMM, the token gather with the
// mean token, and a row softmax.  The explanation backward (p constant) is three more SGEMM calls.
#include "../../include/bcosk.h"
#include "bcosk_common.cuh"
#include "bcosk_host.h"

namespace bcosk {

static inline cudaStream_t SH(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// C[b] (M x N, row pitch ldc) = alpha * op(A[b]) (M x K) * op(B[b]) (K x N); row-major storage, op = transpose when the flag is set
// (A stored K x M / B stored N x K).  64 x 64 x 16 tiles, 256 threads, 4 x 4 outputs per thread.
template <bool TA, bool TB, int TM>
__global__ void __launch_bounds__(256)
sgemm_batched_kernel(int M, int N, int K, const float* __restrict__ A, long long lda, long long sA, const float* __restrict__ B, long long ldb,
                     long long sB, float* __restrict__ C, long long ldc, long long sC, float alpha, int accumulate) {
  constexpr int R = TM / 16;                       // outputs per thread and dimension (4 for 64 x 64 tiles, 2 for 32 x 32)
  __shared__ float As[16][TM + 4];
  __shared__ float Bs[16][TM + 4];
  const int bz = blockIdx.z;
  A += (size_t)bz * sA;
  B += (size_t)bz * sB;
  C += (size_t)bz * sC;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TM;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[R][R];
#pragma unroll
  for (int i = 0; i < R; ++i)
#pragma unroll
    for (int j = 0; j < R; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += 16) {
    // 16 * TM elements per tile; the fast index of the load follows the contiguous axis of the operand
    for (int e = threadIdx.x; e < 16 * TM; e += 256) {
      int kk, mm;
      if (TA) { mm = e % TM; kk = e / TM; } else { kk = e & 15; mm = e >> 4; }
      const int m = m0 + mm, k = k0 + kk;
      As[kk][mm] = (m < M && k < K) ? __ldg(TA ? A + (size_t)k * lda + m : A + (size_t)m * lda + k) : 0.f;
      int nn;
      if (TB) { kk = e & 15; nn = e >> 4; } else { nn = e % TM; kk = e / TM; }
      const int n = n0 + nn;
      const int k2 = k0 + kk;
      Bs[kk][nn] = (n < N && k2 < K) ? __ldg(TB ? B + (size_t)n * ldb + k2 : B + (size_t)k2 * ldb + n) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[R], b[R];
#pragma unroll
      for (int i = 0; i < R; ++i) a[i] = As[kk][ty * R + i];
#pragma unroll
      for (int j = 0; j < R; ++j) b[j] = Bs[kk][tx * R + j];
#pragma unroll
      for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < R; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < R; ++i) {
    const int m = m0 + ty * R + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < R; ++j) {
      const int n = n0 + tx * R + j;
      if (n < N) C[(size_t)m * ldc + n] = accumulate ? C[(size_t)m * ldc + n] + alpha * acc[i][j] : alpha * acc[i][j];
    }
  }
}

// tokens [nb][npix + 1][c] fp32 from the trunk output planes [nb][npix][planes * c]: token 0 = mean over the pixels, token j+1 = pixel j
template <typename T>
__global__ void head_tokens_kernel(const T* __restrict__ x, int npix, int c, int planes, float* __restrict__ tok) {
  const int img = blockIdx.y;
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  const T* src = x + (size_t)img * npix * planes * c + ch;
  float* dst = tok + (size_t)img * (npix + 1) * c + ch;
  float sum = 0.f;
  for (int j = 0; j < npix; ++j) {
    float v = 0.f;
    for (int pl = 0; pl < planes; ++pl) v += (float)src[(size_t)j * planes * c + (size_t)pl * c];
    dst[(size_t)(j + 1) * c] = v;
    sum += v;
  }
  dst[0] = sum / (float)npix;
}

// in-place softmax over rows of `n` (one warp per row)
__global__ void row_softmax_kernel(float* __restrict__ s, long long rows, int n) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  float* r = s + row * n;
  float mx = -INFINITY;
  for (int j = lane; j < n; j += 32) mx = fmaxf(mx, r[j]);
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
  for (int j = lane; j < n; j += 32) {
    const float e = expf(r[j] - mx);
    r[j] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  const float inv = 1.0f / sum;
  for (int j = lane; j < n; j += 32) r[j] *= inv;
}

// softmax backward per row of n: ds = p * (dp - sum_j p_j dp_j) (one warp per row, fixed reduction order; ds may alias dp)
__global__ void softmax_bwd_kernel(const float* __restrict__ p, const float* dp, long long rows, int n, float* ds) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* pr = p + row * n;
  const float* dr = dp + row * n;
  float dot = 0.f;
  for (int j = lane; j < n; j += 32) dot = fmaf(__ldg(pr + j), dr[j], dot);
  dot = warp_sum(dot);
  float* out = ds + row * n;
  for (int j = lane; j < n; j += 32) out[j] = __ldg(pr + j) * (dr[j] - dot);
}

// gradient wrt the trunk output pixels from the gradient wrt the tokens: g[img][pix][ch] = gt[img][pix + 1][ch] + gt[img][0][ch] / npix,
// then as the last block's gradient tensors: out1 = planes(g * scale * mul1), out2 = planes(g * scale [* mul2]) masked by mask2
template <typename T>
__global__ void seed_from_tokens_kernel(const float* __restrict__ gt, int nb, int npix, int c, float scale, const void* __restrict__ mul1,
                                        int mul1_f32, T* __restrict__ out1, const uint32_t* __restrict__ mask2, const void* __restrict__ mul2,
                                        int mul2_f32, T* __restrict__ out2, int planes) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;     // (pixel row, 8-channel group)
  const int nvec = c >> 3;
  if (idx >= (long long)nb * npix * nvec) return;
  const long long row = idx / nvec;
  const int v = (int)(idx - row * nvec);
  const int img = (int)(row / npix), pix = (int)(row - (long long)img * npix);
  const float* g1 = gt + ((size_t)img * (npix + 1) + pix + 1) * c + v * 8;
  const float* g0 = gt + (size_t)img * (npix + 1) * c + v * 8;
  float g[8];
  const float invn = 1.0f / (float)npix;
#pragma unroll
  for (int i = 0; i < 8; ++i) g[i] = (__ldg(g1 + i) + __ldg(g0 + i) * invn) * scale;
  auto side = [&](const void* base, int f32, float (&m)[8]) {
    if (f32) {
#pragma unroll
      for (int i = 0; i < 8; ++i) m[i] = __ldg(reinterpret_cast<const float*>(base) + row * c + v * 8 + i);
    } else {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(base) + row * c + v * 8));
      float2 f;
      f = Cvt<T>::unpack2(u.x); m[0] = f.x; m[1] = f.y;
      f = Cvt<T>::unpack2(u.y); m[2] = f.x; m[3] = f.y;
      f = Cvt<T>::unpack2(u.z); m[4] = f.x; m[5] = f.y;
      f = Cvt<T>::unpack2(u.w); m[6] = f.x; m[7] = f.y;
    }
  };
  auto store = [&](T* dst, const float (&val)[8]) {
    float r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = val[i];
    for (int pl = 0; pl < planes; ++pl) {
      uint32_t w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        w[k] = Cvt<T>::pack2(r[2 * k], r[2 * k + 1]);
        const float2 q = Cvt<T>::unpack2(w[k]);
        r[2 * k] -= q.x; r[2 * k + 1] -= q.y;
      }
      *reinterpret_cast<uint4*>(dst + row * ((long long)planes * c) + (size_t)pl * c + v * 8) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  };
  if (out1 != nullptr) {
    float o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = g[i];
    if (mul1 != nullptr) {
      float m[8];
      side(mul1, mul1_f32, m);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] *= m[i];
    }
    store(out1, o);
  }
  if (out2 != nullptr) {
    float o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = g[i];
    if (mul2 != nullptr) {
      float m[8];
      side(mul2, mul2_f32, m);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] *= m[i];
    }
    if (mask2 != nullptr) {
      const uint32_t mb = __ldg(mask2 + row * ((c + 31) / 32) + (v >> 2)) >> ((v & 3) * 8);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = ((mb >> i) & 1u) ? o[i] : 0.f;
    }
    store(out2, o);
  }
}

}  // namespace bcosk

using namespace bcosk;

static int sgemm_batched(int32_t trans_a, int32_t trans_b, int32_t m, int32_t n, int32_t k, const float* a, int64_t lda, int64_t stride_a,
                         const float* b, int64_t ldb, int64_t stride_b, float* c, int64_t ldc, int64_t stride_c, int32_t batch, float alpha,
                         int accumulate, void* stream) {
  if (!a || !b || !c || m < 1 || n < 1 || k < 1 || batch < 1 || batch > 65535) return set_error(BCOSK_EINVAL, "sgemm_batched: bad argument");
  // few 64 x 64 tiles (the projections of 512 mean tokens: 128-256 CTAs looping over K = 2048) leave SMs idle: 32 x 32 tiles then
  const long long tiles64 = (long long)((n + 63) / 64) * ((m + 63) / 64) * batch;
  const int tm = tiles64 < 2 * 148 ? 32 : 64;
  dim3 grid((n + tm - 1) / tm, (m + tm - 1) / tm, batch);
  if (grid.y > 65535) return set_error(BCOSK_EUNSUPPORTED, "sgemm_batched: m too large for the grid");
#define SG(TA_, TB_)                                                                                                                   \
  do {                                                                                                                                 \
    if (tm == 32) sgemm_batched_kernel<TA_, TB_, 32><<<grid, 256, 0, SH(stream)>>>(m, n, k, a, lda, stride_a, b, ldb, stride_b, c, ldc, stride_c, alpha, accumulate); \
    else sgemm_batched_kernel<TA_, TB_, 64><<<grid, 256, 0, SH(stream)>>>(m, n, k, a, lda, stride_a, b, ldb, stride_b, c, ldc, stride_c, alpha, accumulate);          \
  } while (0)
  if (trans_a) { if (trans_b) SG(true, true); else SG(true, false); }
  else { if (trans_b) SG(false, true); else SG(false, false); }
#undef SG
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_sgemm_batched(int32_t trans_a, int32_t trans_b, int32_t m, int32_t n, int32_t k, const float* a, int64_t lda,
                                   int64_t stride_a, const float* b, int64_t ldb, int64_t stride_b, float* c, int64_t ldc, int64_t stride_c,
                                   int32_t batch, float alpha, void* stream) {
  return sgemm_batched(trans_a, trans_b, m, n, k, a, lda, stride_a, b, ldb, stride_b, c, ldc, stride_c, batch, alpha, 0, stream);
}

extern "C" int bcosk_sgemm_batched_acc(int32_t trans_a, int32_t trans_b, int32_t m, int32_t n, int32_t k, const float* a, int64_t lda,
                                       int64_t stride_a, const float* b, int64_t ldb, int64_t stride_b, float* c, int64_t ldc, int64_t stride_c,
                                       int32_t batch, float alpha, void* stream) {
  return sgemm_batched(trans_a, trans_b, m, n, k, a, lda, stride_a, b, ldb, stride_b, c, ldc, stride_c, batch, alpha, 1, stream);
}

extern "C" int bcosk_head_tokens(const void* x, int32_t nb, int32_t npix, int32_t c, int32_t planes, int32_t dtype, float* tokens, void* stream) {
  if (!x || !tokens || nb < 1 || nb > 65535 || npix < 1 || c < 1 || planes < 1) return set_error(BCOSK_EINVAL, "head_tokens: bad argument");
  dim3 grid((c + 127) / 128, nb);
  if (dtype == BCOSK_DTYPE_BF16) head_tokens_kernel<__nv_bfloat16><<<grid, 128, 0, SH(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(x), npix, c, planes, tokens);
  else if (dtype == BCOSK_DTYPE_F16) head_tokens_kernel<__half><<<grid, 128, 0, SH(stream)>>>(reinterpret_cast<const __half*>(x), npix, c, planes, tokens);
  else return set_error(BCOSK_EINVAL, "head_tokens: dtype");
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_row_softmax(float* s, int64_t rows, int32_t n, void* stream) {
  if (!s || rows < 1 || n < 1) return set_error(BCOSK_EINVAL, "row_softmax: bad argument");
  row_softmax_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, SH(stream)>>>(s, rows, n);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_softmax_bwd(const float* p, const float* dp, int64_t rows, int32_t n, float* ds, void* stream) {
  if (!p || !dp || !ds || rows < 1 || n < 1) return set_error(BCOSK_EINVAL, "softmax_bwd: bad argument");
  softmax_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, SH(stream)>>>(p, dp, rows, n, ds);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

extern "C" int bcosk_seed_from_tokens(const float* g_tokens, int32_t nb, int32_t npix, int32_t c, float scale, const void* mul1, int32_t mul1_f32,
                                      void* out1, const uint32_t* mask2, const void* mul2, int32_t mul2_f32, void* out2, int32_t planes,
                                      int32_t dtype, void* stream) {
  if (!g_tokens || (!out1 && !out2) || nb < 1 || npix < 1 || c < 8 || c % 8 || planes < 1 || planes > 3)
    return set_error(BCOSK_EINVAL, "seed_from_tokens: bad argument");
  const long long n = (long long)nb * npix * (c / 8);
  const unsigned grid = (unsigned)((n + 255) / 256);
  if (dtype == BCOSK_DTYPE_BF16)
    seed_from_tokens_kernel<__nv_bfloat16><<<grid, 256, 0, SH(stream)>>>(g_tokens, nb, npix, c, scale, mul1, mul1_f32, reinterpret_cast<__nv_bfloat16*>(out1),
                                                                       mask2, mul2, mul2_f32, reinterpret_cast<__nv_bfloat16*>(out2), planes);
  else if (dtype == BCOSK_DTYPE_F16)
    seed_from_tokens_kernel<__half><<<grid, 256, 0, SH(stream)>>>(g_tokens, nb, npix, c, scale, mul1, mul1_f32, reinterpret_cast<__half*>(out1), mask2, mul2,
                                                                mul2_f32, reinterpret_cast<__half*>(out2), planes);
  else
    return set_error(BCOSK_EINVAL, "seed_from_tokens: dtype");
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}
