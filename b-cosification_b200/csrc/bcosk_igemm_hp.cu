// bcosk_igemm_hp.cu -- the parity-mode implicit GEMM (bcosk_igemm_params.hp_accum = 1) for sm_100a.
//
// Same contraction as bcosk_igemm.cu (D[m, n] = sum_k A[m, k] B[n, k], A gathered by TMA im2col, B packed K-major,
// tcgen05.mma kind::f16 into TMEM), for operands that carry precision planes (value = sum of 16-bit planes) and results
// that must match the reference's fp32 arithmetic (BcosifyConv2d.forward_impl bcosifyconv2d.py:50-102 and the autograd
// data gradient reached from BcosUtilMixin.explain bcos/common.py:163-181) to ~1e-6:
//
//   * K order: segment 0 is (a-plane 0 x b-plane 0), the remaining segments are the cross terms (a0 b1, a1 b0, ...), each
//     2^-11 (fp16) / 2^-8 (bf16) of the leading one.  The tensor core truncates when it aligns an addend to a large
//     running sum (measured: relative error ~ K 2^-26, biased), so the LEADING segment is accumulated `chunk` K stages at a
//     time into one of two TMEM accumulators and the epilogue warps sum those partials in registers with round-to-nearest
//     fp32 adds; with fp16 planes all cross-term segments run back to back in ONE further accumulation (its truncation error
//     is below 2^-34 of the result), with bf16 planes they are chunked like the leading segment.
//   * Epilogue I/O goes through shared memory and TMA like the throughput kernels: every plane of a 16-bit tensor is a
//     [128 rows][64 columns] SWIZZLE_128B box at a column offset of the same 2-D tensor, fp32 side tensors (saved gain /
//     producer gain) are [128][32]-float boxes.  Output boxes are staged in the drained pipeline ring (or over the input
//     box they replace: every thread reads its own words of an input box before it writes the same words of the output
//     box) and leave with bulk tensor stores.  Input boxes (residual planes; producer gain + extra-gradient planes) are
//     fetched at kernel start into memory next to the ring when the K loop is short (bandwidth-bound launches), or after
//     the last MMA into ring space when it is long (their lines are pulled into L2 by TMA prefetches meanwhile).
//   * 320 threads: TMA producer warp, MMA warp, 8 epilogue warps (TMEM lane quadrant x 32-column half each, 32
//     accumulator registers per thread), two CTAs per SM (256 TMEM columns and <= 113 KB of shared memory each).  64-wide
//     forward launches may instead run 192 threads, three CTAs per SM (hp::Cfg<64, 3>, bcosk_igemm_params.sched = 3).
//   * The common case (two planes, B = 2, everything boxed) runs a packed-fp32 epilogue (FMUL2 / FFMA2 / FADD2);
//     anything else falls back, per tensor, to a generic form with per-row 16-byte accesses.
#include <cuda.h>
#include <cfloat>
#include <cstring>

#include "../../include/bcosk.h"
#include "bcosk_common.cuh"
#include "bcosk_host.h"
#include "bcosk_igemm_epi.cuh"

namespace bcosk {

namespace hp {
constexpr int BM = 128;
constexpr int STAGE_K = 64;
constexpr int A_BYTES = BM * STAGE_K * 2;      // 16 KB
constexpr int BOX_BYTES = BM * 128;            // one [128 rows][128 bytes] swizzled box
constexpr int MAX_STAGES = 8;
// Tile width.  64: two CTAs per SM (<= 113 KB of shared memory, 256 TMEM columns each).  128 (forward launches with the packed
// epilogue only): one CTA per SM, 64 KB paired stages - 98 instead of 65 FLOP per byte of L2 -> shared-memory fill, which is what
// bounds the K >= 1024 launches (DESIGN.md 3.6); every epilogue warp then owns two 32-column groups.
// CTAS_ = 3 (64-wide forward launches with the packed epilogue only, `sched` 3): three CTAs per SM - more independent tiles in
// flight for the latency-bound short-K launches.  128 TMEM columns (ONE partial accumulator + the cross-term accumulator: the MMA
// warp waits for the epilogue to drain the partial before the next chunk), 6 warps (4 epilogue warps, each walks both 32-column
// groups of its lane quadrant), one paired stage as the ring, <= 75 KB of shared memory.  CTAS_ = 4 (`sched` 4): the same kernel
// for launches whose leading segment is one accumulation (no stash), <= 56 KB of shared memory and <= 80 registers.
template <int BN_, int CTAS_ = (BN_ == 64 ? 2 : 1)>
struct Cfg {
  static constexpr int BN = BN_;
  static constexpr bool SLIM = CTAS_ >= 3;                  // one partial accumulator, four epilogue warps
  static constexpr bool ONE_DRAIN = CTAS_ >= 4;             // launches whose leading segment is one accumulation (no stash)
  static constexpr int EPI_WARPS = SLIM ? 4 : 8;
  static constexpr int THREADS = 64 + 32 * EPI_WARPS;       // TMA producer, MMA issuer, epilogue warps
  static constexpr int GS = EPI_WARPS / 4;                  // epilogue warps per lane quadrant: warp j owns groups jj = j + GS h
  static constexpr int NB = BN_ / 64;                       // 64-column boxes per plane of a 16-bit tensor
  static constexpr int NG = BN_ / (32 * GS);                // 32-column groups per epilogue warp
  static constexpr int NACC = SLIM ? 1 : 2;                 // partial accumulators of the leading segment
  static constexpr int B_BYTES = BN_ * STAGE_K * 2;         // 8 / 16 KB
  static constexpr int SLOT_BYTES = A_BYTES + B_BYTES;      // 24 / 32 KB
  static constexpr int PAIR_BYTES = 2 * A_BYTES + 2 * B_BYTES;   // paired stage: [A plane 0 | A plane 1 | B plane 0 | B plane 1] = 48 / 64 KB
  static constexpr int PLANE_BYTES = NB * BOX_BYTES;        // boxes of one plane lie back to back
  static constexpr int TMEM_COLS = SLIM ? 2 * BN_ : 4 * BN_;    // partial accumulator(s) + the cross-term accumulator (power of two)
  static constexpr int TAIL_BYTES = 256 + 2 * BN_ * 4 + BM * 4;   // barriers | alpha, beta | sum-of-squares exchange
  // (228 KB - CTAS x 1 KB reserved) / CTAS; one CTA: 225 KB
  static constexpr int MAX_SMEM = CTAS_ == 1 ? 230400 : (233472 - CTAS_ * 1024) / CTAS_ / 128 * 128;
  static constexpr int MIN_SMEM = BN_ == 64 ? 0 : 118784;   // wide tiles allocate all of TMEM: keep a second CTA off the SM
  static constexpr int MIN_BLOCKS = CTAS_;
  static constexpr int MAX_RING_PAIRED = SLIM ? 1 : (BN_ == 64 ? 2 : 3);
  static constexpr int MAX_RING = SLIM ? 2 : (BN_ == 64 ? 4 : 6);
};
}  // namespace hp

struct HpAux {
  int stages;        // ring slots (2..8)
  int chunk;         // K stages of segment 0 summed by the tensor core before the epilogue warps take over
  int xchunk;        // the same for the cross-term segments (all of them back to back)
  int paired;        // two-plane operands: one stage carries both planes of A and B for one (tap, channel chunk) and feeds three
                     // MMA groups (a0 b0 -> partial accumulator, a0 b1 + a1 b0 -> cross-term accumulator): 48 KB per 3 groups
                     // instead of 72 KB (a0 is fetched once, not twice)
  int in16_planes;   // forward: residual planes / explain: extra-gradient planes fetched as boxes (0 = per-row loads)
  int in32;          // explain: fp32 producer gain fetched as boxes
  int early_in;      // input boxes live outside the ring and are fetched at kernel start (else after the last MMA)
  int out1_planes;   // y planes staged and written with TMA (0 = per-row stores)
  int out2_kind;     // 0 = per-row / none, 1 = forward fp32 gain boxes, 2 = explain out2 planes, 3 = forward 16-bit gain box
  int out2_planes;
  int fast;          // the packed two-plane epilogue applies
  uint32_t off_in16, off_in32;     // byte offsets of the box regions from the start of shared memory
  uint32_t off_out1, off_out2;
  uint32_t off_stash;              // three-CTA kernel with more than one drain: running sums of the groups after the first (fp32 boxes)
  uint32_t tail;                   // barriers etc. (after the ring and the extra input area)
};

__device__ __forceinline__ void tma_prefetch_2d(const void* desc, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(desc)), "r"(c0),
               "r"(c1)
               : "memory");
}

// address of 16-byte unit `u` (0..7) of row r in a swizzled box
__device__ __forceinline__ uint32_t box_unit(uint32_t box, int r, int u) { return box + (r << 7) + ((u ^ (r & 7)) << 4); }

// 8 values -> `planes` 16-bit planes (plane 0 = rn(v), plane 1 = rn(v - plane 0), ...); w[pl] receives the packed words,
// v returns the value the planes represent
template <typename T>
__device__ __forceinline__ void split8(float (&v)[8], int planes, uint4 (&w)[3]) {
  float r[8], a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { r[i] = v[i]; a[i] = 0.f; }
#pragma unroll
  for (int pl = 0; pl < 3; ++pl) {
    if (pl < planes) {
      uint32_t x[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        x[k] = Cvt<T>::pack2(r[2 * k], r[2 * k + 1]);
        const float2 f = Cvt<T>::unpack2(x[k]);
        r[2 * k] -= f.x; r[2 * k + 1] -= f.y;
        a[2 * k] += f.x; a[2 * k + 1] += f.y;
      }
      w[pl] = make_uint4(x[0], x[1], x[2], x[3]);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = a[i];
}

template <typename T>
__device__ __forceinline__ void add8(const uint4& u, float (&v)[8]) {
  float2 f;
  f = Cvt<T>::unpack2(u.x); v[0] += f.x; v[1] += f.y;
  f = Cvt<T>::unpack2(u.y); v[2] += f.x; v[3] += f.y;
  f = Cvt<T>::unpack2(u.z); v[4] += f.x; v[5] += f.y;
  f = Cvt<T>::unpack2(u.w); v[6] += f.x; v[7] += f.y;
}

__device__ __forceinline__ uint32_t pick4(const uint4& u, int k) { return k == 0 ? u.x : (k == 1 ? u.y : (k == 2 ? u.z : u.w)); }
__device__ __forceinline__ float2 pair4(const float4& lo, const float4& hi, int k) {
  return k == 0 ? make_float2(lo.x, lo.y) : (k == 1 ? make_float2(lo.z, lo.w) : (k == 2 ? make_float2(hi.x, hi.y) : make_float2(hi.z, hi.w)));
}
// y -> two 16-bit planes (packed pair)
template <typename T>
__device__ __forceinline__ void split_pair(const float2 y, uint32_t& w0, uint32_t& w1) {
  w0 = Cvt<T>::pack2(y.x, y.y);
  const float2 f = Cvt<T>::unpack2(w0);
  w1 = Cvt<T>::pack2(y.x - f.x, y.y - f.y);
}

// Packed forward epilogue of one row x 32 columns (two planes, B = 2 scale, everything boxed).
//   t = |lin| * inv_norm * alpha;  y = lin * t + beta + res;  ReLU;  y -> two planes, gain = t (0 where clamped), sum y^2
template <typename T>
__device__ __forceinline__ void hp_fwd_fast(const float* acc /* [32] */, float inv_norm, uint32_t ab /* smem: alpha[32] of this group, beta at + 4 BN bytes */,
                                            uint32_t res0 /* plane-0 box or 0 */, uint32_t y0, uint32_t gbox /* fp32 gain box or 0 */,
                                            uint32_t g16 /* 16-bit gain box or 0 */, int row, int j, bool relu, float& sq_acc,
                                            uint32_t& mbits, bool plain /* scale mode NONE: multiplier = alpha */,
                                            uint32_t pstep /* bytes from plane 0 to plane 1 of a boxed tensor */, uint32_t beta_off) {
  using namespace hp;
  const float floor_v = relu ? 0.f : -FLT_MAX;
  const float2 inv2 = make_float2(inv_norm, inv_norm);
  float2 sq2 = make_float2(0.f, 0.f);
  uint32_t mb = 0;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const float4 a_lo = lds_f4(ab + g * 32), a_hi = lds_f4(ab + g * 32 + 16);
    const float4 b_lo = lds_f4(ab + beta_off + g * 32), b_hi = lds_f4(ab + beta_off + g * 32 + 16);
    uint4 r0 = make_uint4(0, 0, 0, 0), r1 = make_uint4(0, 0, 0, 0);
    if (res0 != 0) {
      r0 = lds128(tile_ptr(res0, row, j, g));
      r1 = lds128(tile_ptr(res0 + pstep, row, j, g));
    }
    uint32_t w0[4], w1[4];
    float tt[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 vv = make_float2(acc[g * 8 + 2 * k], acc[g * 8 + 2 * k + 1]);
      const float2 kk = __fmul2_rn(pair4(a_lo, a_hi, k), inv2);
      float2 t = make_float2(fabsf(vv.x) * kk.x, fabsf(vv.y) * kk.y);
      if (plain) t = pair4(a_lo, a_hi, k);
      float2 y = __ffma2_rn(vv, t, pair4(b_lo, b_hi, k));
      y = __fadd2_rn(y, Cvt<T>::unpack2(pick4(r0, k)));
      y = __fadd2_rn(y, Cvt<T>::unpack2(pick4(r1, k)));
      const bool px = y.x > floor_v, py = y.y > floor_v;
      y.x = px ? y.x : 0.f;
      y.y = py ? y.y : 0.f;
      t.x = px ? t.x : 0.f;
      t.y = py ? t.y : 0.f;
      mb |= ((px ? 1u : 0u) | (py ? 2u : 0u)) << (g * 8 + 2 * k);
      split_pair<T>(y, w0[k], w1[k]);
      sq2 = __ffma2_rn(y, y, sq2);
      tt[2 * k] = t.x;
      tt[2 * k + 1] = t.y;
    }
    if (gbox != 0) {
      sts128(box_unit(gbox, row, 2 * g), make_uint4(__float_as_uint(tt[0]), __float_as_uint(tt[1]), __float_as_uint(tt[2]), __float_as_uint(tt[3])));
      sts128(box_unit(gbox, row, 2 * g + 1), make_uint4(__float_as_uint(tt[4]), __float_as_uint(tt[5]), __float_as_uint(tt[6]), __float_as_uint(tt[7])));
    } else if (g16 != 0) {
      sts128(tile_ptr(g16, row, j, g), make_uint4(Cvt<T>::pack2(tt[0], tt[1]), Cvt<T>::pack2(tt[2], tt[3]), Cvt<T>::pack2(tt[4], tt[5]),
                                                  Cvt<T>::pack2(tt[6], tt[7])));
    }
    sts128(tile_ptr(y0, row, j, g), make_uint4(w0[0], w0[1], w0[2], w0[3]));
    sts128(tile_ptr(y0 + pstep, row, j, g), make_uint4(w1[0], w1[1], w1[2], w1[3]));
  }
  sq_acc += sq2.x + sq2.y;
  mbits = mb;
}

// Packed explain epilogue of one row x 32 columns (two planes, everything boxed except the optional fp32 mul2).
//   tot = D + add;  out2 = tot * mul2 * mask2 bit;  y = tot * mul1
template <typename T>
__device__ __forceinline__ void hp_explain_fast(const float* acc /* [32] */, uint32_t add0 /* plane-0 box or 0 */, uint32_t gbox /* fp32 mul1 box or 0 */,
                                                uint32_t y0, uint32_t o20 /* out2 plane-0 box or 0 */, const float* mul2_row /* global or null */,
                                                uint32_t mb2, int row, int j, uint32_t pstep) {
  using namespace hp;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    uint4 a0 = make_uint4(0, 0, 0, 0), a1 = make_uint4(0, 0, 0, 0);
    if (add0 != 0) {
      a0 = lds128(tile_ptr(add0, row, j, g));
      a1 = lds128(tile_ptr(add0 + pstep, row, j, g));
    }
    float4 g_lo = make_float4(1.f, 1.f, 1.f, 1.f), g_hi = g_lo;
    if (gbox != 0) {
      g_lo = lds_f4(box_unit(gbox, row, 2 * g));
      g_hi = lds_f4(box_unit(gbox, row, 2 * g + 1));
    }
    float4 m_lo = make_float4(1.f, 1.f, 1.f, 1.f), m_hi = m_lo;
    if (o20 != 0 && mul2_row != nullptr) {
      m_lo = __ldg(reinterpret_cast<const float4*>(mul2_row + g * 8));
      m_hi = __ldg(reinterpret_cast<const float4*>(mul2_row + g * 8 + 4));
    }
    uint32_t yw0[4], yw1[4], ow0[4], ow1[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float2 tot = make_float2(acc[g * 8 + 2 * k], acc[g * 8 + 2 * k + 1]);
      tot = __fadd2_rn(tot, Cvt<T>::unpack2(pick4(a0, k)));
      tot = __fadd2_rn(tot, Cvt<T>::unpack2(pick4(a1, k)));
      if (o20 != 0) {
        float2 o = __fmul2_rn(tot, pair4(m_lo, m_hi, k));
        const uint32_t bits = mb2 >> (g * 8 + 2 * k);
        o.x = (bits & 1u) ? o.x : 0.f;
        o.y = (bits & 2u) ? o.y : 0.f;
        split_pair<T>(o, ow0[k], ow1[k]);
      }
      split_pair<T>(__fmul2_rn(tot, pair4(g_lo, g_hi, k)), yw0[k], yw1[k]);
    }
    if (o20 != 0) {
      sts128(tile_ptr(o20, row, j, g), make_uint4(ow0[0], ow0[1], ow0[2], ow0[3]));
      sts128(tile_ptr(o20 + pstep, row, j, g), make_uint4(ow1[0], ow1[1], ow1[2], ow1[3]));
    }
    sts128(tile_ptr(y0, row, j, g), make_uint4(yw0[0], yw0[1], yw0[2], yw0[3]));
    sts128(tile_ptr(y0 + pstep, row, j, g), make_uint4(yw1[0], yw1[1], yw1[2], yw1[3]));
  }
}

template <int MODE, typename T, int BN_, int CTAS_>
__global__ void __launch_bounds__(hp::Cfg<BN_, CTAS_>::THREADS, hp::Cfg<BN_, CTAS_>::MIN_BLOCKS)
bcosk_igemm_hp_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                      const __grid_constant__ CUtensorMap tmap_in16, const __grid_constant__ CUtensorMap tmap_in32,
                      const __grid_constant__ CUtensorMap tmap_out1, const __grid_constant__ CUtensorMap tmap_out2,
                      const __grid_constant__ bcosk_igemm_params p, const HpAux aux) {
  using namespace hp;
  using C = Cfg<BN_, CTAS_>;
  constexpr int BN = C::BN, NB = C::NB, NG = C::NG, GS = C::GS, NACC = C::NACC, EPI_THREADS = 32 * C::EPI_WARPS;
  static_assert(!C::SLIM || MODE == BCOSK_MODE_FWD, "the three- and four-CTA kernels run forward launches only");
  constexpr int B_BYTES = C::B_BYTES, SLOT_BYTES = C::SLOT_BYTES, PAIR_BYTES = C::PAIR_BYTES, PLANE_BYTES = C::PLANE_BYTES;
  constexpr int TMEM_COLS = C::TMEM_COLS;
  extern __shared__ __align__(1024) uint8_t smem[];   // no static shared memory: the dynamic window starts 1024-byte aligned
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  const int stages = aux.stages;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + aux.tail);
  uint64_t* empty_bar = full_bar + MAX_STAGES;
  uint64_t* acc_full_bar = empty_bar + MAX_STAGES;   // [3] partial accumulator complete; [2] = cross-term accumulator (paired mode)
  uint64_t* acc_empty_bar = acc_full_bar + 3;        // [2] partial accumulator drained
  uint64_t* mma_done_bar = acc_empty_bar + 2;        // every MMA has read its operands: the ring is free
  uint64_t* in_bar = mma_done_bar + 1;               // epilogue input boxes landed
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(in_bar + 1);
  float* s_alpha = reinterpret_cast<float*>(smem + aux.tail + 256);
  float* s_beta = s_alpha + BN;
  float* s_sq = s_beta + BN;                         // [BM] sums of squares of the upper column half

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_tiles = (p.n + BN - 1) / BN;
  const int tile_n = blockIdx.x % n_tiles;
  const int tile_m = blockIdx.x / n_tiles;
  const int M = p.a_nb * p.op * p.oq;
  const int m0 = tile_m * BM;
  const int n0 = tile_n * BN;

  const int chunks_per_stage = STAGE_K / p.kch;                                  // 1 (kch = 64) or 2 (kch = 32)
  const int seg_iters = (p.num_taps * p.chunks_per_tap) / chunks_per_stage;      // K stages per segment (host: divisible)
  const int num_iters = aux.paired ? seg_iters : p.num_segs * seg_iters;    // paired: one stage per (tap, chunk), both planes
  const int main_drains = (seg_iters + aux.chunk - 1) / aux.chunk;
  const int num_drains = aux.paired ? main_drains : main_drains + (num_iters - seg_iters + aux.xchunk - 1) / aux.xchunk;
  const int boxes32 = min(BN / 32, (p.n - n0 + 31) >> 5);                        // fp32 boxes of this tile inside the tensor
  const int boxes16 = min(NB, (p.n - n0 + 63) >> 6);                             // 64-column boxes per plane inside the tensor
  const bool any_in = aux.in16_planes != 0 || aux.in32 != 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < NACC; ++s) {
      mbar_init(&acc_full_bar[s], 1);
      mbar_init(&acc_empty_bar[s], C::EPI_WARPS);   // one arrival per epilogue warp
    }
    mbar_init(&acc_full_bar[2], 1);
    mbar_init(mma_done_bar, 1);
    mbar_init(in_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      const int ps16 = MODE == BCOSK_MODE_FWD ? p.res_plane_stride : p.add_plane_stride;
      auto load_inputs = [&]() {
        mbar_arrive_expect_tx(in_bar, (uint32_t)(aux.in16_planes * boxes16 * BOX_BYTES + (aux.in32 ? boxes32 * BOX_BYTES : 0)));
        for (int pl = 0; pl < aux.in16_planes; ++pl)
          for (int b = 0; b < boxes16; ++b)
            tma_load_2d(smem + aux.off_in16 + pl * PLANE_BYTES + b * BOX_BYTES, &tmap_in16, in_bar, pl * ps16 + n0 + b * 64, m0);
        if (aux.in32)
          for (int b = 0; b < boxes32; ++b) tma_load_2d(smem + aux.off_in32 + b * BOX_BYTES, &tmap_in32, in_bar, n0 + b * 32, m0);
      };
      if (any_in) {
        if (aux.early_in) {
          load_inputs();                 // their boxes are not part of the ring
        } else {
          // pull the lines into L2 while the K loop runs; the boxes are fetched into the ring after it
          for (int pl = 0; pl < aux.in16_planes; ++pl)
            for (int b = 0; b < boxes16; ++b) tma_prefetch_2d(&tmap_in16, pl * ps16 + n0 + b * 64, m0);
          if (aux.in32)
            for (int b = 0; b < boxes32; ++b) tma_prefetch_2d(&tmap_in32, n0 + b * 32, m0);
        }
      }
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
      if (aux.paired) {
        // segments are {a0 b0, a0 b1, a1 b0} (engine/pack.py SEGMENTS[2]): stage = [a0 | a1 | b0 | b1] of one (tap, chunk)
        const int seg_cols = p.num_taps * p.chunks_per_tap * p.kch;      // B columns per segment
        for (int it = 0; it < num_iters; ++it) {
          uint8_t* slot = smem + stage * PAIR_BYTES;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], aux.paired == 2 ? PAIR_BYTES - A_BYTES : PAIR_BYTES);
          tma_load_im2col_4d(slot, &tmap_a, &full_bar[stage], p.seg_a_choff[0] + kc * p.kch, base_w, base_h, img, p.tap_off_w[tap],
                             p.tap_off_h[tap]);
          if (aux.paired != 2)
            tma_load_im2col_4d(slot + A_BYTES, &tmap_a, &full_bar[stage], p.seg_a_choff[2] + kc * p.kch, base_w, base_h, img,
                               p.tap_off_w[tap], p.tap_off_h[tap]);
          tma_load_2d(slot + 2 * A_BYTES, &tmap_b, &full_bar[stage], it * p.kch, n0);
          tma_load_2d(slot + 2 * A_BYTES + B_BYTES, &tmap_b, &full_bar[stage], seg_cols + it * p.kch, n0);
          if (++kc == p.chunks_per_tap) { kc = 0; ++tap; }
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      } else
      for (int it = 0; it < num_iters; ++it) {
        uint8_t* slot = smem + stage * SLOT_BYTES;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        mbar_arrive_expect_tx(&full_bar[stage], SLOT_BYTES);
        for (int j = 0; j < chunks_per_stage; ++j) {
          const int ci = it * chunks_per_stage + j;
          tma_load_im2col_4d(slot + j * a_chunk_bytes, &tmap_a, &full_bar[stage], p.seg_a_choff[seg] + kc * p.kch, base_w, base_h,
                             img, p.tap_off_w[tap], p.tap_off_h[tap]);
          tma_load_2d(slot + A_BYTES + j * b_chunk_bytes, &tmap_b, &full_bar[stage], ci * p.kch, n0);
          if (++kc == p.chunks_per_tap) {
            kc = 0;
            if (++tap == p.num_taps) { tap = 0; ++seg; }
          }
        }
        if (++stage == stages) { stage = 0; phase ^= 1; }
      }
      if (any_in && !aux.early_in) {
        mbar_wait(mma_done_bar, 0);      // the ring is free: it now receives the epilogue's input boxes
        load_inputs();
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
      const uint64_t slot16 = SLOT_BYTES >> 4;
      int stage = 0;
      uint32_t phase = 0;
      uint32_t accumulate = 0;
      int d = 0;                        // accumulation (drain) index
      if (aux.paired) {
        const uint64_t pair16 = PAIR_BYTES >> 4;
        const uint32_t tmem_x = tmem_base + NACC * BN;   // cross-term accumulator
        for (int it = 0; it < num_iters; ++it) {
          const bool first = it % aux.chunk == 0;
          const bool last = it % aux.chunk == aux.chunk - 1 || it == num_iters - 1;
          const uint32_t buf = (uint32_t)d % NACC;
          if (first) {
            mbar_wait(&acc_empty_bar[buf], (((uint32_t)d / NACC) & 1u) ^ 1u);
            tc_fence_after();
          }
          const uint32_t tmem_d = tmem_base + buf * BN;
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t da0 = da_stage0 + (uint64_t)stage * pair16;
          const uint64_t da1 = da0 + (A_BYTES >> 4);
          const uint64_t db0 = da0 + (2 * A_BYTES >> 4);
          const uint64_t db1 = db0 + (B_BYTES >> 4);
          // a0 b0 -> partial accumulator of the leading term
          umma_f16(tmem_d, da0, db0, idesc, first ? 0u : 1u);
          umma_f16(tmem_d, da0 + 2, db0 + 2, idesc, 1);
          umma_f16(tmem_d, da0 + 4, db0 + 4, idesc, 1);
          umma_f16(tmem_d, da0 + 6, db0 + 6, idesc, 1);
          if (last) {
            umma_commit(&acc_full_bar[buf]);
            ++d;
          }
          // a0 b1 + a1 b0 -> cross-term accumulator (one accumulation over all of K)
          umma_f16(tmem_x, da0, db1, idesc, it == 0 ? 0u : 1u);
          umma_f16(tmem_x, da0 + 2, db1 + 2, idesc, 1);
          umma_f16(tmem_x, da0 + 4, db1 + 4, idesc, 1);
          umma_f16(tmem_x, da0 + 6, db1 + 6, idesc, 1);
          if (aux.paired != 2) {
            umma_f16(tmem_x, da1, db0, idesc, 1);
            umma_f16(tmem_x, da1 + 2, db0 + 2, idesc, 1);
            umma_f16(tmem_x, da1 + 4, db0 + 4, idesc, 1);
            umma_f16(tmem_x, da1 + 6, db0 + 6, idesc, 1);
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&acc_full_bar[2]);
        umma_commit(mma_done_bar);
      } else {
      for (int it = 0; it < num_iters; ++it) {
        const int xi = it - seg_iters;   // position among the cross-term stages
        const bool first = it < seg_iters ? (it % aux.chunk == 0) : (xi % aux.xchunk == 0);
        const bool last = it < seg_iters ? (it % aux.chunk == aux.chunk - 1 || it == seg_iters - 1)
                                         : (xi % aux.xchunk == aux.xchunk - 1 || it == num_iters - 1);
        const uint32_t buf = (uint32_t)d % NACC;
        if (first) {
          mbar_wait(&acc_empty_bar[buf], (((uint32_t)d / NACC) & 1u) ^ 1u);
          tc_fence_after();
          accumulate = 0;
        }
        const uint32_t tmem_d = tmem_base + buf * BN;
        uint8_t* slot = smem + stage * SLOT_BYTES;
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (chunks_per_stage == 1) {
          const uint64_t da = da_stage0 + (uint64_t)stage * slot16;
          const uint64_t db = da + (A_BYTES >> 4);
          umma_f16(tmem_d, da, db, idesc, accumulate);
          umma_f16(tmem_d, da + 2, db + 2, idesc, 1);
          umma_f16(tmem_d, da + 4, db + 4, idesc, 1);
          umma_f16(tmem_d, da + 6, db + 6, idesc, 1);
          accumulate = 1;
        } else {
          for (int j = 0; j < chunks_per_stage; ++j) {
            const uint64_t da = umma_smem_desc_kmajor(smem_u32(slot + j * a_chunk_bytes), row_bytes);
            const uint64_t db = umma_smem_desc_kmajor(smem_u32(slot + A_BYTES + j * b_chunk_bytes), row_bytes);
            for (int k = 0; k < mma_per_chunk; ++k) {
              umma_f16(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, accumulate);
              accumulate = 1;
            }
          }
        }
        umma_commit(&empty_bar[stage]);
        if (last) {
          umma_commit(&acc_full_bar[buf]);
          ++d;
        }
        if (++stage == stages) { stage = 0; phase ^= 1; }
      }
      umma_commit(mma_done_bar);
      }
    }
  } else {
    // ===================== epilogue (warps 2 .. 2 + EPI_WARPS - 1) =====================
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may read
    const int j = (warp - 2) >> 2;             // this warp owns the 32-column groups jj = j + GS h, h < NG (warp-uniform)
    const int row = quad * 32 + lane;
    const int et = threadIdx.x - 64;           // 0 .. EPI_THREADS - 1
    if (MODE == BCOSK_MODE_FWD) {
      if (et < BN) {
        const int c = n0 + et;
        s_alpha[et] = (p.alpha != nullptr && c < p.n) ? __ldg(p.alpha + c) : 1.f;
        s_beta[et] = (p.beta != nullptr && c < p.n) ? __ldg(p.beta + c) : 0.f;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
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
    if (MODE == BCOSK_MODE_EXPLAIN && p.side_mapped) ri.m = (int)yrow;
    float inv_norm = 1.f;
    int64_t add_row = -1;
    if (MODE == BCOSK_MODE_FWD) {
      if (p.scale_mode != BCOSK_SCALE_NONE && ri.valid) {
        if (p.inv_norm != nullptr) {
          inv_norm = __ldg(p.inv_norm + ri.m);
        } else {
          // patch norm from the producer's per-pixel sums of squares (calc_patch_norms, bcosconv2d.py:196-231)
          const size_t part_stride = (size_t)p.a_nb * p.sq_h * p.sq_w;
          float s = 0.f;
          for (int dy = 0; dy < p.sq_k; ++dy) {
            const int yy = ri.p * p.sq_stride - p.sq_pad + dy;
            if (yy < 0 || yy >= p.sq_h) continue;
            for (int dx = 0; dx < p.sq_k; ++dx) {
              const int xx = ri.q * p.sq_stride - p.sq_pad + dx;
              if (xx < 0 || xx >= p.sq_w) continue;
              const size_t o = ((size_t)ri.img * p.sq_h + yy) * p.sq_w + xx;
              for (int t = 0; t < p.sq_parts; ++t) s += __ldg(p.sq_in + t * part_stride + o);
            }
          }
          inv_norm = 1.0f / (sqrtf(s + p.sq_eps_in) + p.sq_eps_out);
        }
      }
    } else if (p.add != nullptr && ri.valid) {
      const int s = p.add_stride;
      if (ri.p % s == 0 && ri.q % s == 0 && ri.p / s < p.add_p && ri.q / s < p.add_q)
        add_row = ((int64_t)ri.img * p.add_p + ri.p / s) * p.add_q + ri.q / s;
    }
    uint32_t mb2s[NG];
#pragma unroll
    for (int h = 0; h < NG; ++h) {
      const int c0 = n0 + (j + GS * h) * 32;
      mb2s[h] = 0xffffffffu;
      if (MODE == BCOSK_MODE_EXPLAIN && p.mask2 != nullptr && ri.valid && c0 < p.n) mb2s[h] = __ldg(p.mask2 + (size_t)ri.m * p.mask2_ld + (c0 >> 5));
    }
    // side tensors read with per-row loads after the last drain: pull their lines into L2 now
#pragma unroll
    for (int h = 0; h < NG; ++h) {
      const int c0 = n0 + (j + GS * h) * 32;
      if (!(ri.valid && c0 < p.n)) continue;
      const int ncols_pf = min(32, p.n - c0);
      auto prefetch_row = [&](const void* base, size_t elem_off, int elem_bytes) {
        const char* b = reinterpret_cast<const char*>(base) + elem_off * (size_t)elem_bytes;
        const char* e = b + (size_t)ncols_pf * elem_bytes;
        for (const char* q = reinterpret_cast<const char*>(reinterpret_cast<uintptr_t>(b) & ~(uintptr_t)127); q < e; q += 128)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(q));
      };
      if (MODE == BCOSK_MODE_FWD) {
        if (p.res != nullptr && aux.in16_planes == 0)
          for (int pl = 0; pl < p.res_planes; ++pl) prefetch_row(p.res, (size_t)ri.m * p.res_ld + c0 + (size_t)pl * p.res_plane_stride, 2);
      } else {
        if (add_row >= 0 && aux.in16_planes == 0)
          for (int pl = 0; pl < p.add_planes; ++pl)
            prefetch_row(p.add, (size_t)add_row * p.add_ld + c0 + (size_t)pl * p.add_plane_stride, 2);
        if (p.mul1 != nullptr && !aux.in32) prefetch_row(p.mul1, (size_t)ri.m * p.mul1_ld + c0, p.mul1_f32 ? 4 : 2);
        if (p.out2 != nullptr && p.mul2 != nullptr) prefetch_row(p.mul2, (size_t)ri.m * p.mul2_ld + c0, p.mul2_f32 ? 4 : 2);
      }
    }

    // ---- sum the partial accumulators of this thread's 32-column groups (round-to-nearest fp32 adds, in drain order, then
    //      the cross-term accumulator)
    const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(j * 32);     // group h: + 32 GS h columns
    constexpr int NGR = C::SLIM ? 1 : NG;      // groups whose sums live in registers across the drains
    float acc[NGR][32];
#pragma unroll
    for (int h = 0; h < NGR; ++h)
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[h][i] = 0.f;
    if constexpr (!C::SLIM) {
      for (int d = 0; d < num_drains; ++d) {
        const uint32_t buf = (uint32_t)d % NACC;
        mbar_wait(&acc_full_bar[buf], ((uint32_t)d / NACC) & 1u);
        tc_fence_after();
        uint32_t raw[NG][32];
#pragma unroll
        for (int h = 0; h < NG; ++h) tmem_ld_32x32(taddr + buf * BN + h * 32 * GS, raw[h]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty_bar[buf]);
#pragma unroll
        for (int h = 0; h < NG; ++h)
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[h][i] += __uint_as_float(raw[h][i]);
      }
      if (aux.paired) {
        mbar_wait(&acc_full_bar[2], 0);
        tc_fence_after();
        uint32_t raw[NG][32];
#pragma unroll
        for (int h = 0; h < NG; ++h) tmem_ld_32x32(taddr + NACC * BN + h * 32 * GS, raw[h]);
        tmem_ld_wait();
        tc_fence_before();
#pragma unroll
        for (int h = 0; h < NG; ++h)
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[h][i] += __uint_as_float(raw[h][i]);
      }
    } else {
      // One partial accumulator: every drain but the last is added here - group 0 into registers, the other groups into
      // their stash boxes - and handed back to the MMA warp.  The last drain and the cross terms are added per group
      // below, right before that group's epilogue, so at most 32 accumulator columns are live at a time.
      const uint32_t stash = smem_u32(smem) + aux.off_stash;
      for (int d = 0; !C::ONE_DRAIN && d + 1 < num_drains; ++d) {
        mbar_wait(&acc_full_bar[0], (uint32_t)d & 1u);
        tc_fence_after();
        uint32_t raw[32];
        tmem_ld_32x32(taddr, raw);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[0][i] += __uint_as_float(raw[i]);
#pragma unroll 1
        for (int h = 1; h < NG; ++h) {
          tmem_ld_32x32(taddr + h * 32, raw);
          tmem_ld_wait();
          const uint32_t sb = stash + (uint32_t)((h - 1) * BOX_BYTES);
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            float4 s = d == 0 ? make_float4(0.f, 0.f, 0.f, 0.f) : lds_f4(box_unit(sb, row, u));
            s.x += __uint_as_float(raw[4 * u]);
            s.y += __uint_as_float(raw[4 * u + 1]);
            s.z += __uint_as_float(raw[4 * u + 2]);
            s.w += __uint_as_float(raw[4 * u + 3]);
            sts128(box_unit(sb, row, u), make_uint4(__float_as_uint(s.x), __float_as_uint(s.y), __float_as_uint(s.z), __float_as_uint(s.w)));
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty_bar[0]);
      }
      mbar_wait(&acc_full_bar[0], (uint32_t)(num_drains - 1) & 1u);
      if (aux.paired) mbar_wait(&acc_full_bar[2], 0);
      tc_fence_after();
    }
    if (any_in) mbar_wait(in_bar, 0);

    const uint32_t sbase = smem_u32(smem);
    const uint32_t r_in16 = sbase + aux.off_in16, r_in32 = sbase + aux.off_in32;
    const uint32_t r_out1 = sbase + aux.off_out1, r_out2 = sbase + aux.off_out2;
    T* y16 = reinterpret_cast<T*>(p.y);
    float* y32 = reinterpret_cast<float*>(p.y);
    float sq_acc = 0.f;

#pragma unroll
    for (int h = 0; h < NG; ++h) {
      const int jj = j + GS * h;               // 32-column group of the tile
      const int c0 = n0 + jj * 32;
      float accs[C::SLIM ? 32 : 1];
      if constexpr (C::SLIM) {
        // (running sum or 0) + last drain + cross terms; tcgen05.ld is warp-wide, so before any lane leaves the loop
        if (C::ONE_DRAIN || h == 0 || num_drains == 1) {
#pragma unroll
          for (int i = 0; i < 32; ++i) accs[i] = h == 0 ? acc[0][i] : 0.f;
        } else {
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float4 s = lds_f4(box_unit(smem_u32(smem) + aux.off_stash + (uint32_t)((h - 1) * BOX_BYTES), row, u));
            accs[4 * u] = s.x; accs[4 * u + 1] = s.y; accs[4 * u + 2] = s.z; accs[4 * u + 3] = s.w;
          }
        }
        uint32_t raw[32];
        tmem_ld_32x32(taddr + h * 32, raw);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) accs[i] += __uint_as_float(raw[i]);
        if (aux.paired) {
          tmem_ld_32x32(taddr + BN + h * 32, raw);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) accs[i] += __uint_as_float(raw[i]);
        }
      }
      if (!(ri.valid && c0 < p.n)) continue;
      const int ncols = min(32, p.n - c0);
      const float* accv = C::SLIM ? accs : acc[C::SLIM ? 0 : h];
      const uint32_t mb2 = mb2s[h];
      if (C::SLIM || aux.fast) {
        if (MODE == BCOSK_MODE_FWD) {
          uint32_t mbits;
          hp_fwd_fast<T>(accv, inv_norm, smem_u32(s_alpha + jj * 32), aux.in16_planes ? r_in16 : 0u, r_out1,
                         aux.out2_kind == 1 ? r_out2 + jj * BOX_BYTES : 0u, aux.out2_kind == 3 ? r_out2 : 0u, row, jj, p.relu != 0, sq_acc,
                         mbits, p.scale_mode == BCOSK_SCALE_NONE, (uint32_t)PLANE_BYTES, (uint32_t)(BN * 4));
          if (p.maskbits != nullptr) p.maskbits[(size_t)ri.m * p.mask_ld + (c0 >> 5)] = mbits;
        } else {
          hp_explain_fast<T>(accv, aux.in16_planes ? r_in16 : 0u, aux.in32 ? r_in32 + jj * BOX_BYTES : 0u, r_out1,
                             aux.out2_kind == 2 ? r_out2 : 0u,
                             p.mul2 != nullptr ? reinterpret_cast<const float*>(p.mul2) + (size_t)ri.m * p.mul2_ld + c0 : nullptr, mb2, row, jj, (uint32_t)PLANE_BYTES);
        }
      } else {
        uint32_t mbits = 0;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          if (g * 8 < ncols) {     // n is a multiple of 8
            const int cg = c0 + g * 8;
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = accv[g * 8 + i];
            uint4 w[3];
            if (MODE == BCOSK_MODE_FWD) {
              // ---------------- forward: scale, BN multiplier, residual, ReLU; writes y planes, gain, mask, sum y^2
              if (p.lin_bias != nullptr) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] += __ldg(p.lin_bias + cg + i);
              }
              if (p.max_out > 1) {     // MaxOut: 8 / max_out columns of this row leave through per-row stores
                sq_acc += maxout_fwd_tail<T, 8>(p, v, inv_norm, ri.m, yrow, cg, 8);
                continue;
              }
              // (the operation order of hp_fwd_fast wherever both forms apply: |lin| * (alpha * inv_norm), then the residual planes
              //  added one at a time, so that the packed and the generic epilogue write the same bits)
              float t[8];
              const float4 a0 = *reinterpret_cast<const float4*>(s_alpha + jj * 32 + g * 8);
              const float4 a1 = *reinterpret_cast<const float4*>(s_alpha + jj * 32 + g * 8 + 4);
              const float al[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
              if (p.scale_mode == BCOSK_SCALE_B2) {
#pragma unroll
                for (int i = 0; i < 8; ++i) t[i] = fabsf(v[i]) * (al[i] * inv_norm);
              } else if (p.scale_mode == BCOSK_SCALE_POW) {
                const float e = p.b_exp - 1.f;
#pragma unroll
                for (int i = 0; i < 8; ++i) t[i] = __powf(fabsf(v[i]) * inv_norm + 1e-6f, e) * al[i];
              } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) t[i] = al[i];
              }
              const float4 b0 = *reinterpret_cast<const float4*>(s_beta + jj * 32 + g * 8);
              const float4 b1 = *reinterpret_cast<const float4*>(s_beta + jj * 32 + g * 8 + 4);
              const float be[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] = fmaf(v[i], t[i], be[i]);
              if (p.res != nullptr) {
                if (aux.in16_planes) {
                  for (int pl = 0; pl < aux.in16_planes; ++pl) add8<T>(lds128(tile_ptr(r_in16 + pl * PLANE_BYTES, row, jj, g)), v);
                } else {
                  const T* rp = reinterpret_cast<const T*>(p.res) + (size_t)ri.m * p.res_ld + cg;
                  for (int pl = 0; pl < p.res_planes; ++pl)
                    add8<T>(__ldg(reinterpret_cast<const uint4*>(rp + (size_t)pl * p.res_plane_stride)), v);
                }
              }
              if (p.relu) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const bool pos = v[i] > 0.f;
                  mbits |= (pos ? 1u : 0u) << (g * 8 + i);
                  v[i] = pos ? v[i] : 0.f;
                  t[i] = pos ? t[i] : 0.f;
                }
              } else {
                mbits |= 0xffu << (g * 8);
              }
              if (p.gain != nullptr) {
                if (aux.out2_kind == 1) {
                  sts128(box_unit(r_out2 + jj * BOX_BYTES, row, 2 * g), make_uint4(__float_as_uint(t[0]), __float_as_uint(t[1]),
                                                                                 __float_as_uint(t[2]), __float_as_uint(t[3])));
                  sts128(box_unit(r_out2 + jj * BOX_BYTES, row, 2 * g + 1), make_uint4(__float_as_uint(t[4]), __float_as_uint(t[5]),
                                                                                     __float_as_uint(t[6]), __float_as_uint(t[7])));
                } else if (aux.out2_kind == 3) {
                  split8<T>(t, 1, w);
                  sts128(tile_ptr(r_out2, row, jj, g), w[0]);
                } else if (p.gain_f32) {
                  float4* gp = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.gain) + (size_t)ri.m * p.gain_ld + cg);
                  gp[0] = make_float4(t[0], t[1], t[2], t[3]);
                  gp[1] = make_float4(t[4], t[5], t[6], t[7]);
                } else {
                  split8<T>(t, 1, w);
                  *reinterpret_cast<uint4*>(reinterpret_cast<T*>(p.gain) + (size_t)ri.m * p.gain_ld + cg) = w[0];
                }
              }
              if (p.y_f32) {
                float4* yp = reinterpret_cast<float4*>(y32 + (size_t)yrow * p.y_ld + cg);
                yp[0] = make_float4(v[0], v[1], v[2], v[3]);
                yp[1] = make_float4(v[4], v[5], v[6], v[7]);
              } else {
                split8<T>(v, p.y_planes, w);
                if (aux.out1_planes) {
#pragma unroll
                  for (int pl = 0; pl < 3; ++pl)
                    if (pl < aux.out1_planes) sts128(tile_ptr(r_out1 + pl * PLANE_BYTES, row, jj, g), w[pl]);
                } else {
                  T* yp = y16 + (size_t)yrow * p.y_ld + cg;
#pragma unroll
                  for (int pl = 0; pl < 3; ++pl)
                    if (pl < p.y_planes) *reinterpret_cast<uint4*>(yp + (size_t)pl * p.y_plane_stride) = w[pl];
                }
              }
              if (p.sq_out != nullptr) {
#pragma unroll
                for (int i = 0; i < 8; ++i) sq_acc = fmaf(v[i], v[i], sq_acc);
              }
            } else {
              // ---------------- explain: tot = D + add;  out2 = tot * mul2 * mask2;  y = tot * mul1
              if (add_row >= 0) {
                if (aux.in16_planes) {
                  for (int pl = 0; pl < aux.in16_planes; ++pl) add8<T>(lds128(tile_ptr(r_in16 + pl * PLANE_BYTES, row, jj, g)), v);
                } else {
                  const T* ap = reinterpret_cast<const T*>(p.add) + (size_t)add_row * p.add_ld + cg;
                  for (int pl = 0; pl < p.add_planes; ++pl)
                    add8<T>(__ldg(reinterpret_cast<const uint4*>(ap + (size_t)pl * p.add_plane_stride)), v);
                }
              }
              if (p.out2 != nullptr) {
                float o[8];
                if (p.mul2 != nullptr) {
                  if (p.mul2_f32) {
                    const float4* mp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.mul2) + (size_t)ri.m * p.mul2_ld + cg);
                    const float4 m0v = __ldg(mp), m1v = __ldg(mp + 1);
                    o[0] = m0v.x; o[1] = m0v.y; o[2] = m0v.z; o[3] = m0v.w; o[4] = m1v.x; o[5] = m1v.y; o[6] = m1v.z; o[7] = m1v.w;
                  } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) o[i] = 0.f;
                    add8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.mul2) + (size_t)ri.m * p.mul2_ld + cg)), o);
                  }
#pragma unroll
                  for (int i = 0; i < 8; ++i) o[i] *= v[i];
                } else {
#pragma unroll
                  for (int i = 0; i < 8; ++i) o[i] = v[i];
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] = ((mb2 >> (g * 8 + i)) & 1u) ? o[i] : 0.f;
                split8<T>(o, p.out2_planes, w);
                if (aux.out2_kind == 2) {
#pragma unroll
                  for (int pl = 0; pl < 3; ++pl)
                    if (pl < aux.out2_planes) sts128(tile_ptr(r_out2 + pl * PLANE_BYTES, row, jj, g), w[pl]);
                } else {
                  T* op = reinterpret_cast<T*>(p.out2) + (size_t)ri.m * p.out2_ld + cg;
#pragma unroll
                  for (int pl = 0; pl < 3; ++pl)
                    if (pl < p.out2_planes) *reinterpret_cast<uint4*>(op + (size_t)pl * p.out2_plane_stride) = w[pl];
                }
              }
              if (p.mul1 != nullptr) {
                float gq[8];
                if (aux.in32) {
                  const float4 g0 = lds_f4(box_unit(r_in32 + jj * BOX_BYTES, row, 2 * g));
                  const float4 g1 = lds_f4(box_unit(r_in32 + jj * BOX_BYTES, row, 2 * g + 1));
                  gq[0] = g0.x; gq[1] = g0.y; gq[2] = g0.z; gq[3] = g0.w; gq[4] = g1.x; gq[5] = g1.y; gq[6] = g1.z; gq[7] = g1.w;
                } else if (p.mul1_f32) {
                  const float4* mp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.mul1) + (size_t)ri.m * p.mul1_ld + cg);
                  const float4 g0 = __ldg(mp), g1 = __ldg(mp + 1);
                  gq[0] = g0.x; gq[1] = g0.y; gq[2] = g0.z; gq[3] = g0.w; gq[4] = g1.x; gq[5] = g1.y; gq[6] = g1.z; gq[7] = g1.w;
                } else {
#pragma unroll
                  for (int i = 0; i < 8; ++i) gq[i] = 0.f;
                  add8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.mul1) + (size_t)ri.m * p.mul1_ld + cg)), gq);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] *= gq[i];
              }
              if (p.y_f32) {
                float4* yp = reinterpret_cast<float4*>(y32 + (size_t)yrow * p.y_ld + cg);
                yp[0] = make_float4(v[0], v[1], v[2], v[3]);
                yp[1] = make_float4(v[4], v[5], v[6], v[7]);
              } else {
                split8<T>(v, p.y_planes, w);
                if (aux.out1_planes) {
#pragma unroll
                  for (int pl = 0; pl < 3; ++pl)
                    if (pl < aux.out1_planes) sts128(tile_ptr(r_out1 + pl * PLANE_BYTES, row, jj, g), w[pl]);
                } else {
                  T* yp = y16 + (size_t)yrow * p.y_ld + cg;
#pragma unroll
                  for (int pl = 0; pl < 3; ++pl)
                    if (pl < p.y_planes) *reinterpret_cast<uint4*>(yp + (size_t)pl * p.y_plane_stride) = w[pl];
                }
              }
            }
          }
        }
        if (MODE == BCOSK_MODE_FWD && p.maskbits != nullptr) p.maskbits[(size_t)ri.m * p.mask_ld + (c0 >> 5)] = mbits;
      }
    }
    const bool want_sq = MODE == BCOSK_MODE_FWD && p.sq_out != nullptr;
    if (want_sq && j == 1) s_sq[row] = sq_acc;  // (GS = 2: the upper column half's sum goes to the warp of the lower one)
    // generic-proxy writes of the staged boxes -> visible to the async proxy, then one thread issues the bulk stores
    if (aux.out1_planes != 0 || aux.out2_kind != 0) fence_proxy_async_smem();
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
    if ((aux.out1_planes != 0 || aux.out2_kind != 0) && et == 0) {
      for (int pl = 0; pl < aux.out1_planes; ++pl)
        for (int b = 0; b < boxes16; ++b)
          tma_store_2d_addr(&tmap_out1, r_out1 + pl * PLANE_BYTES + b * BOX_BYTES, pl * p.y_plane_stride + n0 + b * 64, m0);
      if (aux.out2_kind == 1) {
        for (int b = 0; b < boxes32; ++b) tma_store_2d_addr(&tmap_out2, r_out2 + b * BOX_BYTES, n0 + b * 32, m0);
      } else if (aux.out2_kind == 2) {
        for (int pl = 0; pl < aux.out2_planes; ++pl)
          for (int b = 0; b < boxes16; ++b)
            tma_store_2d_addr(&tmap_out2, r_out2 + pl * PLANE_BYTES + b * BOX_BYTES, pl * p.out2_plane_stride + n0 + b * 64, m0);
      } else if (aux.out2_kind == 3) {
        for (int b = 0; b < boxes16; ++b) tma_store_2d_addr(&tmap_out2, r_out2 + b * BOX_BYTES, n0 + b * 64, m0);
      }
      tma_store_commit_and_wait_read();
    }
    if (MODE == BCOSK_MODE_FWD && j == 0 && ri.valid) {
      if (want_sq) p.sq_out[(size_t)tile_n * M + ri.m] = GS == 1 ? sq_acc : sq_acc + (n0 + 32 < p.n ? s_sq[row] : 0.f);
      if (p.inv_norm_out != nullptr && tile_n == 0) p.inv_norm_out[ri.m] = inv_norm;
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int g_hp_chunk = 2;       // default K stages of the leading segment per TMEM accumulation (bcosk_set_hp_chunk)
static int g_hp_xchunk = 0;      // experiment override of the cross-term accumulation length (0 = by operand format)
static int g_hp_stage_boxes = 1; // 0 = per-row epilogue I/O everywhere (A/B measurements)
static int g_hp_early_iters = 4; // K loops of at most this many stages fetch their input boxes at kernel start

// The three- and four-CTA kernels (CTAS_ = 3, 4) set *declined and launches nothing where it does not apply (no packed epilogue, or its
// boxes do not fit one paired stage): the caller then runs the two-CTA kernel, which gives the same bits.
template <int MODE, int BN_, int CTAS_ = (BN_ == 64 ? 2 : 1)>
static int launch_hp_mode(const bcosk_igemm_params& p, cudaStream_t st, bool* declined = nullptr, int32_t* info = nullptr) {
  using namespace hp;
  using C = Cfg<BN_, CTAS_>;
  constexpr int BN = C::BN;
  constexpr int SLOT_BYTES = C::SLOT_BYTES, PAIR_BYTES = C::PAIR_BYTES, PLANE_BYTES = C::PLANE_BYTES, TAIL_BYTES = C::TAIL_BYTES;
  constexpr int MAX_SMEM = C::MAX_SMEM;
  CUtensorMap ma, mb, min16, min32, mout1, mout2;
  memset(&min16, 0, sizeof(min16));
  memset(&min32, 0, sizeof(min32));
  memset(&mout1, 0, sizeof(mout1));
  memset(&mout2, 0, sizeof(mout2));
  int rc = make_im2col_map_nhwc(&ma, p.a, p.a_nb, p.a_h, p.a_w, p.a_c, p.lo_w, p.lo_h, p.up_w, p.up_h, p.stride_w, p.stride_h,
                                p.kch, BM, p.kch == 64 ? 128 : 64);
  if (rc) return rc;
  const long long ktot = (long long)p.num_segs * p.num_taps * p.chunks_per_tap * p.kch;
  rc = make_tiled_map_2d(&mb, p.b, ktot, p.n, p.kch, BN, p.kch == 64 ? 128 : 64);
  if (rc) return rc;
  const long long M = (long long)p.a_nb * p.op * p.oq;
  const bool dense_out = p.os_0 == 0 && p.os_q == 1 && p.os_p == p.oq && p.os_n == (long long)p.op * p.oq;
  auto planes_ok = [&](int planes) { return planes == 1 || p.n % BN == 0; };   // a ragged tile would spill into the next plane
  auto map16 = [&](CUtensorMap* m, const void* base, int ld, long long rows) -> bool {
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || ld % 8 != 0) return false;
    return make_tiled_map_2d(m, base, ld, rows, 64, BM, 128) == BCOSK_OK;
  };
  auto map32 = [&](CUtensorMap* m, const void* base, int ld, long long rows) -> bool {
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || ld % 4 != 0) return false;
    const long long dims[2] = {ld, rows};
    const long long strides[1] = {(long long)ld * 4};
    const int box[2] = {32, BM};
    return make_tiled_map_nd(m, base, 4, 2, dims, strides, box, 128) == BCOSK_OK;
  };
  HpAux aux;
  memset(&aux, 0, sizeof(aux));
  aux.chunk = p.hp_chunk > 0 ? p.hp_chunk : g_hp_chunk;
  // cross terms are 2^-11 of the leading segment with fp16 planes: one accumulation over all of them adds a truncation
  // error below 2^-34 of the result.  bf16 planes (2^-8, and second-order terms at 2^-16 on top of first-order ones) keep
  // the chunk length of the leading segment.
  aux.xchunk = p.dtype == BCOSK_DTYPE_F16 ? (1 << 20) : aux.chunk;
  if (g_hp_xchunk > 0) aux.xchunk = g_hp_xchunk;
  if ((g_hp_stage_boxes & 1) && p.max_out <= 1) {      // MaxOut rows (n / max_out columns) leave with per-row stores
    if (!p.y_f32 && dense_out && planes_ok(p.y_planes) && p.y_planes <= 3 && map16(&mout1, p.y, p.y_ld, M)) aux.out1_planes = p.y_planes;
    if (MODE == BCOSK_MODE_FWD) {
      if (p.gain && p.gain_f32 && map32(&mout2, p.gain, p.gain_ld, M)) aux.out2_kind = 1;
      if (p.gain && !p.gain_f32 && map16(&mout2, p.gain, p.gain_ld, M)) aux.out2_kind = 3;   // 16-bit gain: one box
      if (p.res && planes_ok(p.res_planes) && p.res_planes <= 3 && map16(&min16, p.res, p.res_ld, M)) aux.in16_planes = p.res_planes;
    } else {
      if (p.mul1 && p.mul1_f32 && !p.side_mapped && map32(&min32, p.mul1, p.mul1_ld, M)) aux.in32 = 1;
      if (p.add && p.add_stride == 1 && p.add_p == p.op && p.add_q == p.oq && planes_ok(p.add_planes) && p.add_planes <= 3 &&
          map16(&min16, p.add, p.add_ld, M))
        aux.in16_planes = p.add_planes;
      if (p.out2 && !p.side_mapped && planes_ok(p.out2_planes) && p.out2_planes <= 3 && map16(&mout2, p.out2, p.out2_ld, M)) {
        aux.out2_kind = 2;
        aux.out2_planes = p.out2_planes;
      }
    }
  }
  // ---- placement of the boxes.  Outputs are staged in the (drained) ring; y goes over the 16-bit input planes it
  //      replaces.  Inputs: next to the ring and fetched at kernel start when the K loop is short, else into the ring
  //      after the last MMA.  When the boxes do not fit two CTAs per SM, tensors drop back to per-row accesses one by one.
  const int tail_bytes = MODE == BCOSK_MODE_FWD ? TAIL_BYTES : 256;
  // two-plane operands in the canonical segment order {a0 b0, a0 b1, a1 b0}: paired stages (a0 fetched once)
  aux.paired = (g_hp_stage_boxes & 4) == 0 && p.kch == 64 && p.num_segs == 3 && p.seg_b_plane[0] == 0 && p.seg_b_plane[1] == 1 &&
               p.seg_b_plane[2] == 0 && p.seg_a_choff[0] == p.seg_a_choff[1] && p.seg_a_choff[2] != p.seg_a_choff[0];
  // one-plane input against two-plane weights {a0 b0, a0 b1} (exact byte patch matrix of the stem, one-plane branch operands added into a
  // two-plane residual stream): the same paired stage without the a1 box and without the a1 b0 product
  if (!aux.paired && (g_hp_stage_boxes & 4) == 0 && p.kch == 64 && p.num_segs == 2 && p.seg_b_plane[0] == 0 && p.seg_b_plane[1] == 1 &&
      p.seg_a_choff[0] == p.seg_a_choff[1])
    aux.paired = 2;
  const int slot_b = aux.paired ? PAIR_BYTES : SLOT_BYTES;
  const int max_ring = aux.paired ? C::MAX_RING_PAIRED : C::MAX_RING;        // ring slots that fit the CTAs of one SM
  const int iters = aux.paired ? p.num_taps * p.chunks_per_tap : p.num_segs * p.num_taps * p.chunks_per_tap / (STAGE_K / p.kch);
  // (three CTAs: input boxes always after the last MMA - the other CTAs of the SM hide the fetch)
  const int early_iters = C::SLIM ? 0 : (aux.paired ? (g_hp_early_iters + 2) / 3 : g_hp_early_iters);
  // three CTAs with more than one drain of the single partial accumulator: the running sums of the column groups after the
  // first wait in a stash between the ring and the tail
  int stash_b = 0;
  if (C::SLIM) {
    const int seg_iters = p.num_taps * p.chunks_per_tap / (STAGE_K / p.kch);
    const int main_drains = (seg_iters + aux.chunk - 1) / aux.chunk;
    const int num_drains = aux.paired ? main_drains : main_drains + (iters - seg_iters + aux.xchunk - 1) / aux.xchunk;
    if (num_drains > 1) stash_b = (C::NG - 1) * BOX_BYTES;
  }
  int stages = 0, extra = 0;
  auto place = [&]() -> bool {
    const int in16_b = aux.in16_planes * PLANE_BYTES, in32_b = aux.in32 ? (BN / 32) * BOX_BYTES : 0;
    const int out1_b = aux.out1_planes * PLANE_BYTES;
    const int out2_b = aux.out2_kind == 1 ? (BN / 32) * BOX_BYTES
                                          : (aux.out2_kind == 2 ? aux.out2_planes * PLANE_BYTES : (aux.out2_kind == 3 ? PLANE_BYTES : 0));
    aux.early_in = 0;
    extra = 0;
    if ((in16_b || in32_b) && iters <= early_iters) {
      // early inputs: [ring | in16 | in32]; y over in16 when present (same plane count), else in the ring; out2 in the ring
      const bool y_over_in = in16_b != 0 && aux.out1_planes == aux.in16_planes;
      const int ring_need = (y_over_in ? 0 : out1_b) + out2_b;
      int s = (ring_need + slot_b - 1) / slot_b;
      if (s < (aux.paired ? 1 : 2)) s = aux.paired ? 1 : 2;
      if (s <= max_ring && s * slot_b + in16_b + in32_b + tail_bytes <= MAX_SMEM) {
        // the deepest useful ring that still fits
        while (s < max_ring && s < iters && (s + 1) * slot_b + in16_b + in32_b + tail_bytes <= MAX_SMEM) ++s;
        stages = s;
        extra = in16_b + in32_b;
        aux.early_in = 1;
        aux.off_in16 = (uint32_t)(stages * slot_b);
        aux.off_in32 = aux.off_in16 + (uint32_t)in16_b;
        aux.off_out1 = y_over_in ? aux.off_in16 : 0u;
        aux.off_out2 = y_over_in ? 0u : (uint32_t)out1_b;
        return true;
      }
    }
    // everything inside the ring: [in16 / y | in32 or forward gain | explain out2]
    const int a_b = in16_b > out1_b ? in16_b : out1_b;
    const int b_b = MODE == BCOSK_MODE_FWD ? out2_b : in32_b;
    const int c_b = MODE == BCOSK_MODE_FWD ? 0 : out2_b;
    const int need = a_b + b_b + c_b;
    stages = (need + slot_b - 1) / slot_b;
    if (stages < max_ring) stages = max_ring;
    // three CTAs: one paired stage, plus the stash box behind it.  fp32 gains (two boxes) may overrun the stage by exactly
    // one box, the gain box of the second column group, which then shares the stash's place: each thread reads its row of
    // the stash before it writes its row of that gain box.
    int over = 0;
    if (C::SLIM && stages > max_ring) {
      over = need - max_ring * slot_b;
      if (!(MODE == BCOSK_MODE_FWD && aux.out2_kind == 1 && over == BOX_BYTES)) return false;
      stages = max_ring;
    }
    if (C::ONE_DRAIN && (stash_b != 0 || over != 0)) return false;   // four CTAs: the ring and the tail only
    extra = stash_b > over ? stash_b : over;
    if (stages > MAX_STAGES || stages * slot_b + extra + tail_bytes > MAX_SMEM) return false;
    aux.off_stash = (uint32_t)(stages * slot_b);
    aux.off_in16 = 0;
    aux.off_out1 = 0;
    aux.off_in32 = (uint32_t)a_b;
    aux.off_out2 = MODE == BCOSK_MODE_FWD ? (uint32_t)a_b : (uint32_t)(a_b + b_b);
    return true;
  };
  if (C::SLIM && !place()) {
    *declined = true;
    return BCOSK_OK;
  }
  while (!place()) {
    if (MODE == BCOSK_MODE_EXPLAIN && aux.out2_kind == 2) aux.out2_kind = 0, aux.out2_planes = 0;
    else if (aux.in16_planes) aux.in16_planes = 0;
    else if (aux.out2_kind) aux.out2_kind = 0;
    else if (aux.in32) aux.in32 = 0;
    else if (aux.out1_planes) aux.out1_planes = 0;
    else return set_error(BCOSK_EUNSUPPORTED, "igemm(hp): no shared-memory placement");
  }
  // ---- the packed two-plane epilogue
  if (MODE == BCOSK_MODE_FWD)
    aux.fast = (p.scale_mode == BCOSK_SCALE_B2 || p.scale_mode == BCOSK_SCALE_NONE) && !p.lin_bias && !p.y_f32 && p.y_planes == 2 && aux.out1_planes == 2 &&
               (!p.res || aux.in16_planes == 2) && (!p.gain || aux.out2_kind == 1 || aux.out2_kind == 3);
  else
    aux.fast = !p.y_f32 && p.y_planes == 2 && aux.out1_planes == 2 && (!p.add || aux.in16_planes == 2) && (!p.mul1 || aux.in32) &&
               (!p.out2 || (aux.out2_kind == 2 && aux.out2_planes == 2)) && (!p.mul2 || p.mul2_f32);
  if (g_hp_stage_boxes & 2) aux.fast = 0;      // A/B: generic epilogue arithmetic over the same boxes
  if (C::SLIM && !aux.fast) {
    *declined = true;
    return BCOSK_OK;
  }
  aux.stages = stages;
  aux.tail = (uint32_t)(stages * slot_b + extra);
  if (BN_ > 64 && !aux.fast)
    return set_error(BCOSK_EUNSUPPORTED, "igemm(hp): 128-wide tiles need the packed two-plane epilogue (two boxed planes, B = 2 or plain scale)");
  int smem = (int)aux.tail + tail_bytes;
  if (smem < C::MIN_SMEM) smem = C::MIN_SMEM;
  auto kern = bcosk_igemm_hp_kernel<MODE, __nv_bfloat16, BN_, CTAS_>;
  auto kern_h = bcosk_igemm_hp_kernel<MODE, __half, BN_, CTAS_>;
  const void* fn = (p.dtype == BCOSK_DTYPE_BF16) ? (const void*)kern : (const void*)kern_h;
  BCOSK_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_SMEM));
  BCOSK_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  if (info != nullptr) {        // bcosk_igemm_hp_config: report the configuration instead of launching
    int blocks = 0;
    BCOSK_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, fn, C::THREADS, (size_t)smem));
    cudaFuncAttributes fa;
    BCOSK_CUDA_CHECK(cudaFuncGetAttributes(&fa, fn));
    info[0] = CTAS_;
    info[1] = C::THREADS;
    info[2] = smem;
    info[3] = blocks;
    info[4] = fa.numRegs;
    info[5] = (int32_t)fa.localSizeBytes;
    return BCOSK_OK;
  }
  const long long m_tiles = (M + BM - 1) / BM;
  const long long n_tiles = (p.n + BN - 1) / BN;
  if (m_tiles * n_tiles > 0x7fffffffLL) return set_error(BCOSK_EUNSUPPORTED, "igemm(hp): grid too large");
  dim3 grid((unsigned)(m_tiles * n_tiles));
  if (p.dtype == BCOSK_DTYPE_BF16)
    kern<<<grid, C::THREADS, smem, st>>>(ma, mb, min16, min32, mout1, mout2, p, aux);
  else
    kern_h<<<grid, C::THREADS, smem, st>>>(ma, mb, min16, min32, mout1, mout2, p, aux);
  BCOSK_CUDA_CHECK(cudaGetLastError());
  return BCOSK_OK;
}

static int dispatch_hp(const bcosk_igemm_params& p, cudaStream_t st, int32_t* info) {
  const int cps = hp::STAGE_K / p.kch;
  if ((p.num_taps * p.chunks_per_tap) % cps != 0)
    return set_error(BCOSK_EINVAL, "igemm(hp): a segment must be a whole number of K stages");
  if (p.hp_chunk < 0) return set_error(BCOSK_EINVAL, "igemm(hp): hp_chunk < 0");
  if (p.mul1_sqrt_scale) return set_error(BCOSK_EUNSUPPORTED, "igemm(hp): recomputed gains (mul1_sqrt_scale) are a throughput-mode option");
  if (p.block_n == 128) {
    if (p.mode != BCOSK_MODE_FWD) return set_error(BCOSK_EUNSUPPORTED, "igemm(hp): 128-wide tiles are a forward-launch option");
    return launch_hp_mode<BCOSK_MODE_FWD, 128>(p, st, nullptr, info);
  }
  if (p.sched == 4 && p.mode == BCOSK_MODE_FWD) {
    bool declined = false;
    const int rc = launch_hp_mode<BCOSK_MODE_FWD, 64, 4>(p, st, &declined, info);
    if (!declined) return rc;
  }
  if ((p.sched == 3 || p.sched == 4) && p.mode == BCOSK_MODE_FWD) {
    bool declined = false;
    const int rc = launch_hp_mode<BCOSK_MODE_FWD, 64, 3>(p, st, &declined, info);
    if (!declined) return rc;
  }
  return p.mode == BCOSK_MODE_FWD ? launch_hp_mode<BCOSK_MODE_FWD, 64>(p, st, nullptr, info)
                                  : launch_hp_mode<BCOSK_MODE_EXPLAIN, 64>(p, st, nullptr, info);
}

int launch_hp(const bcosk_igemm_params& p, cudaStream_t st) { return dispatch_hp(p, st, nullptr); }

}  // namespace bcosk

extern "C" int bcosk_igemm_hp_config(const bcosk_igemm_params* p, int32_t* info) {
  if (!p || !info || !p->hp_accum) return bcosk::set_error(BCOSK_EINVAL, "igemm_hp_config: needs hp_accum params and info[6]");
  bcosk_igemm_params q = *p;
  if (q.block_n == 0) q.block_n = 64;
  return bcosk::dispatch_hp(q, 0, info);
}

extern "C" int bcosk_set_hp_chunk(int32_t stages) {
  const int prev = bcosk::g_hp_chunk | (bcosk::g_hp_xchunk << 16);
  if ((stages & 0xffff) >= 1) bcosk::g_hp_chunk = stages & 0xffff;
  bcosk::g_hp_xchunk = stages >> 16;            // bits 16..: experiment override of the cross-term accumulation length
  return prev;
}

extern "C" int bcosk_set_hp_boxes(int32_t enabled) {
  // the previous setting in the encoding the argument uses (bits 8.. = 1 + threshold), so that passing it back restores it
  const int prev = bcosk::g_hp_stage_boxes | ((bcosk::g_hp_early_iters + 1) << 8);
  bcosk::g_hp_stage_boxes = enabled & 7;        // bit 0: boxes, bit 1: generic arithmetic, bit 2: no paired stages
  if (enabled >> 8) bcosk::g_hp_early_iters = (enabled >> 8) - 1;   // bits 8..: 1 + K stages up to which input boxes are fetched early
  return prev;
}
