// bcosk_common.cuh -- sm_100a PTX wrappers shared by the bcosk kernels.
//
// mbarrier, TMA (cp.async.bulk.tensor: tiled + im2col), tcgen05 (alloc / mma / commit / ld),
// UMMA shared-memory + instruction descriptors.  Hand-written inline PTX; encodings follow the
// PTX ISA 8.7 tables (cross-checked against the descriptor bit-fields documented in CUTLASS'
// cute/arch/mma_sm100_desc.hpp).  Compile only with -gencode arch=compute_100a,code=sm_100a.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#ifndef BCOSK_SPIN_LIMIT
// A wedged pipeline traps (-> cudaErrorLaunchFailure) instead of hanging the GPU forever.
#define BCOSK_SPIN_LIMIT (1u << 24)
#endif

namespace bcosk {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > BCOSK_SPIN_LIMIT) __trap();
  }
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(desc)) : "memory");
}
// 2-D tiled load: coordinates (c0 = innermost, c1)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* desc, uint64_t* bar, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// 4-D tiled load (c0 innermost); out-of-range coordinates (also negative ones) are zero filled
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const void* desc, uint64_t* bar, int32_t c0, int32_t c1, int32_t c2,
                                            int32_t c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// 4-D im2col load over an NHWC tensor described as (C, W, H, N); (off_w, off_h) = filter tap offset
__device__ __forceinline__ void tma_load_im2col_4d(void* smem_dst, const void* desc, uint64_t* bar, int32_t c,
                                                   int32_t w, int32_t h, int32_t n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h),
      "r"(n), "h"(off_w), "h"(off_h)
      : "memory");
}

// 2-D tiled store smem -> global (bulk async group); out-of-bounds parts of the box are clipped
__device__ __forceinline__ void tma_store_2d(const void* desc, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_2d_addr(const void* desc, uint32_t smem_addr, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_addr), "r"(c0), "r"(c1)
               : "memory");
}
// close the bulk group and wait until the TMA unit has finished READING shared memory (stores may still be in flight)
__device__ __forceinline__ void tma_store_3d_addr(const void* desc, uint32_t smem_addr, int32_t c0, int32_t c1, int32_t c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(desc), "r"(smem_addr),
               "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit_and_wait_read() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// 1-D bulk copies (contiguous bytes, 16-byte aligned, size % 16 == 0): global -> shared with mbarrier completion, shared -> global
// as a bulk group.
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_store_1d(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// ------------------------------------------------------------------ tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], bf16/fp16 inputs, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// All previously issued MMAs of this thread arrive on `bar` when complete (implies fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (thread i <- lane base+i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------ UMMA descriptors
// K-major operand tile whose rows are `row_bytes` (= swizzle span) wide: 128 -> SWIZZLE_128B, 64 -> SWIZZLE_64B.
// 8-row groups are contiguous, so the stride-byte-offset is 8*row_bytes. LBO is unused for swizzled K-major (set 1).
// Bits: [0,14) addr>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 (Blackwell) | [61,64) layout type.
__device__ __forceinline__ uint64_t umma_smem_desc_kmajor(uint32_t smem_addr, uint32_t row_bytes) {
  const uint64_t layout = (row_bytes == 128) ? 2ull : (row_bytes == 64 ? 4ull : 6ull);
  uint64_t d = (uint64_t)((smem_addr >> 4) & 0x3FFFu);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(((8u * row_bytes) >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= layout << 61;
  return d;
}
// A tile may start at any ROW of a larger swizzled buffer (start address = base + r * row_bytes, base 1024-aligned):
// the tensor core, like the TMA unit, derives the swizzle phase from the absolute shared-memory address, so the same
// descriptor form is correct and bits [49,52) ("base offset") stay 0 (measured: scripts/exp, tests flat_*; setting
// them to (addr >> 7) & 7 reads the wrong rows).
// kind::f16 instruction descriptor: fp32 accumulate, A/B both K-major, `fmt` 0 = fp16, 1 = bf16.
// Bits: [4,6) c_format=1 | [7,10) a_format | [10,13) b_format | 15 a_major=0 | 16 b_major=0 | [17,23) N>>3 | [24,29) M>>4.
__host__ __device__ __forceinline__ uint32_t umma_idesc_f16(uint32_t fmt, uint32_t M, uint32_t N) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// ------------------------------------------------------------------ small helpers
template <typename T> struct Cvt;
template <> struct Cvt<__nv_bfloat16> {
  static __device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  static __device__ __forceinline__ float2 unpack2(uint32_t u) {
    return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u));
  }
  static __device__ __forceinline__ float round1(float a) { return __bfloat162float(__float2bfloat16_rn(a)); }
};
template <> struct Cvt<__half> {
  static __device__ __forceinline__ uint32_t pack2(float a, float b) {
    __half2 v = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  static __device__ __forceinline__ float2 unpack2(uint32_t u) { return __half22float2(*reinterpret_cast<__half2*>(&u)); }
  static __device__ __forceinline__ float round1(float a) { return __half2float(__float2half_rn(a)); }
};

// one MUFU instruction (sqrt(0) = 0); the IEEE sqrtf costs ~20 instructions per element in an epilogue
__device__ __forceinline__ float fast_sqrt(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace bcosk
