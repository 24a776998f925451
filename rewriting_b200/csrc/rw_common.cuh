// rw_common.cuh — sm_100a device primitives shared by the rewriting_b200 kernels.
//
// Thin inline-PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor), tcgen05
// (alloc / mma / commit / ld) and the bf16 hi/lo split used by every
// tensor-core kernel in this library.  Nothing here is derived from the
// reference (davidbau/rewriting has no tensor-core code at all); the layouts
// follow the PTX ISA "tcgen05 matrix descriptor" / "instruction descriptor"
// tables.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>

namespace rw {

// ---------------------------------------------------------------------------
// error plumbing (C-ABI never throws; see include/rewriting_b200.h)
// ---------------------------------------------------------------------------
enum : int {
  RW_OK = 0,
  RW_ERR_BAD_ARG = -1,
  RW_ERR_CUDA = -2,
  RW_ERR_NO_DRIVER_SYMBOL = -3,
  RW_ERR_UNSUPPORTED = -4,
};
void set_last_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

// spin bound for every mbarrier wait: a protocol bug traps (-> CUDA error)
// instead of hanging the GPU box.
#ifndef RW_SPIN_LIMIT
#define RW_SPIN_LIMIT (1u << 26)
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > RW_SPIN_LIMIT) __trap();
  }
}

// ---------------------------------------------------------------------------
// TMA (tiled mode, 2-D), completes on an mbarrier
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c_inner, int32_t c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];\n" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c_inner), "r"(c_outer)
      : "memory");
}

// ---------------------------------------------------------------------------
// tcgen05: TMEM allocation, MMA, commit, load
// ---------------------------------------------------------------------------
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {
  static_assert(kCols == 32 || kCols == 64 || kCols == 128 || kCols == 256 || kCols == 512, "");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(
                   smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(kCols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, single CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when complete
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(
          smem_u32(bar))
      : "memory");
}
// ---- cta_group::2 (CTA pair) variants: one MMA spans the two SMs of a cluster; the leader
// CTA (cluster rank 0) issues it, each CTA stages its own A rows and half of B. --------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // clears the CTA-rank bit of a shared address

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// TMA load whose completion bytes are credited to the LEADER CTA's mbarrier
__device__ __forceinline__ void tma_load_2d_cg2(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                                int32_t c_inner, int32_t c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];\n" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c_inner),
      "r"(c_outer)
      : "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* smem_result) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(
                   smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(kCols)
               : "memory");
}
__device__ __forceinline__ void umma_bf16_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the barrier at this offset in BOTH CTAs of the pair when the MMAs complete
__device__ __forceinline__ void umma_commit_cg2_mc(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64"
      " [%0], %1;\n" ::"r"(smem_u32(bar)),
      "h"(mask)
      : "memory");
}
// arrive on the LEADER CTA's copy of a barrier (from either CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];\n" ::"r"(smem_u32(bar) & kPeerBitMask)
               : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
        "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
        "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// 16-column form for the narrow (BN = 32) tiles
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}

// ---------------------------------------------------------------------------
// descriptors
// ---------------------------------------------------------------------------
// Shared-memory matrix descriptor (PTX ISA "tcgen05 matrix descriptor"):
//  [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 |
//  [49,52) base offset | [52] lbo mode | [61,64) swizzle (2 = 128B, 4 = 64B)
__host__ __device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes,
                                                            uint32_t sbo_bytes,
                                                            uint32_t layout_type) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFFu);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout_type & 7u) << 61;
  return d;
}
constexpr uint32_t kSwizzle128B = 2;
constexpr uint32_t kSwizzle64B = 4;

// Instruction descriptor for kind::f16, bf16 x bf16 -> fp32.
//  [4,6) D fmt (1=f32) | [7,10) A fmt (1=bf16) | [10,13) B fmt | [15] A major
//  (0=K,1=MN) | [16] B major | [17,23) N>>3 | [24,29) M>>4
__host__ __device__ constexpr uint32_t make_idesc_bf16(uint32_t M, uint32_t N, uint32_t a_mn_major,
                                                       uint32_t b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (a_mn_major << 15) | (b_mn_major << 16) |
         ((N >> 3) << 17) | ((M >> 4) << 24);
}

// ---------------------------------------------------------------------------
// bf16 hi/lo split:  x ~= hi + lo with |x-(hi+lo)| <= 2^-17 |x|
// ---------------------------------------------------------------------------
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

// ---------------------------------------------------------------------------
// host: TMA descriptor encode through the driver entry point (no -lcuda)
// ---------------------------------------------------------------------------
// swizzle_bytes: 128 (box rows of 128 B) or 64 (box rows of 64 B)
int make_tmap_2d_bf16(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer,
                      uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer,
                      uint32_t swizzle_bytes = 128);

int device_sm_count();

}  // namespace rw
