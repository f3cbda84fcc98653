// Shared device helpers of the tcgen05 kernels (policy_tc.cu: rollout forward; bptt_tc.cu: backward): PTX wrappers
// for mbarriers, bulk / tensor copies, tcgen05.mma / commit / ld, UMMA shared-memory descriptors, and the fp16 hi/lo
// operand split.
#pragma once
#include <cuda_fp16.h>

#include "ic3_common.cuh"

constexpr uint32_t WATCHDOG_SPINS = 1u << 26;   // bounded mbarrier wait: a broken pipeline raises a flag instead of hanging
constexpr float SCALE_A = 16.f, SCALE_B = 256.f, INV_SCALE = 1.f / 4096.f;

__device__ __forceinline__ void split_f16(float v, float scale, __half& hi, __half& lo) {
  const float s = v * scale;            // power of two: exact
  hi = __float2half_rn(s);
  lo = __float2half_rn(s - __half2float(hi));
}

__device__ __forceinline__ void store_split4(__half* img, size_t off_hi, size_t off_lo, const float4& v, float scale) {
  __half h[4], l[4];
  split_f16(v.x, scale, h[0], l[0]);
  split_f16(v.y, scale, h[1], l[1]);
  split_f16(v.z, scale, h[2], l[2]);
  split_f16(v.w, scale, h[3], l[3]);
  uint2 ph, pl;
  ph.x = (uint32_t)__half_as_ushort(h[0]) | ((uint32_t)__half_as_ushort(h[1]) << 16);
  ph.y = (uint32_t)__half_as_ushort(h[2]) | ((uint32_t)__half_as_ushort(h[3]) << 16);
  pl.x = (uint32_t)__half_as_ushort(l[0]) | ((uint32_t)__half_as_ushort(l[1]) << 16);
  pl.y = (uint32_t)__half_as_ushort(l[2]) | ((uint32_t)__half_as_ushort(l[3]) << 16);
  *reinterpret_cast<uint2*>(img + off_hi) = ph;
  *reinterpret_cast<uint2*>(img + off_lo) = pl;
}

// ---- PTX wrappers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded wait: a mis-programmed pipeline must never hang the GPU; it raises the flag instead.
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, int32_t* err) {
  if (mbar_try(bar, parity)) return true;       // common case in the steady state: already complete
#pragma unroll 1
  for (uint32_t spin = 0; spin < WATCHDOG_SPINS; ++spin)
    if (mbar_try(bar, parity)) return true;
  if (err) atomicOr(err, IC3_ERR_PIPELINE);
  return false;
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, kind::f16 (fp16 inputs, fp32 accumulate), one CTA
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// K-major, no swizzle: core matrices of 8 rows x 16 B; LBO = byte distance between the two
// K-adjacent core matrices of one MMA, SBO = distance between 8-row groups (both >> 4).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;                 // descriptor version 1 (sm_100)
  return d;                               // base_offset = 0, lbo_mode = 0, layout_type = SWIZZLE_NONE (0)
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

