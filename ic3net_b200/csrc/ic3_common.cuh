// Shared device/host helpers for the ic3net_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ic3net_b200.h"

#define IC3_FULL_MASK 0xffffffffu
#define IC3_ENV_WARPS 8      // envs per CTA of an env step launched without an observation block (warp = env)

// predator-prey: agent rows per environment (the prey is row N with --enemy_comm, predator_prey_env.py:203-207)
__host__ __device__ __forceinline__ int ic3_pp_agents(const ic3_pp_cfg& c) { return c.N + (c.enemy_comm != 0 ? 1 : 0); }

extern unsigned long long g_ic3_launches;  // c_api.cu

#define IC3_LAUNCH_CHECK()                         \
  do {                                             \
    ++g_ic3_launches;                              \
    cudaError_t _e = cudaGetLastError();           \
    if (_e != cudaSuccess) return (int)_e;         \
  } while (0)

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  Same stream layout as oracle/philox.py:
//   key = (seed_lo, seed_hi), counter = (env_id, tick, stream, index)
// Every draw is reduced to 24 bits so u = u24 * 2^-24 is exact in fp32.
// ---------------------------------------------------------------------------
enum { IC3_STREAM_PP_RESET = 1, IC3_STREAM_TJ_SPAWN = 2, IC3_STREAM_ACTION = 3 };

__host__ __device__ __forceinline__ void ic3_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#ifdef __CUDA_ARCH__
  hi = __umulhi(a, b);
  lo = a * b;
#else
  unsigned long long p = (unsigned long long)a * b;
  hi = (uint32_t)(p >> 32);
  lo = (uint32_t)p;
#endif
}

__host__ __device__ __forceinline__ uint4 ic3_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                    uint64_t seed) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    ic3_mulhilo(0xD2511F53u, c0, hi0, lo0);
    ic3_mulhilo(0xCD9E8D57u, c2, hi1, lo1);
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

// four 24-bit draws for (env, tick, stream, index)
__host__ __device__ __forceinline__ uint4 ic3_draw24(uint64_t seed, uint32_t env, uint32_t tick,
                                                    uint32_t stream, uint32_t index) {
  uint4 w = ic3_philox(env, tick, stream, index, seed);
  return make_uint4(w.x >> 8, w.y >> 8, w.z >> 8, w.w >> 8);
}

// floor(u * k) for u = u24 * 2^-24, as an integer operation
__host__ __device__ __forceinline__ uint32_t ic3_pick(uint32_t u24, uint32_t k) {
  return (uint32_t)(((unsigned long long)u24 * k) >> 24);
}

__device__ __forceinline__ uint32_t ic3_word(const uint4& w, int i) {
  return i == 0 ? w.x : (i == 1 ? w.y : (i == 2 ? w.z : w.w));
}

// ---------------------------------------------------------------------------
// streaming (evict-first) vector stores / loads for write-once / read-once data
// ---------------------------------------------------------------------------
__device__ __forceinline__ void ic3_st_stream(float4* p, const float4& v) { __stcs(p, v); }
__device__ __forceinline__ void ic3_st_stream(float* p, float v) { __stcs(p, v); }
// keep = true: plain write-back store (the consumer kernel follows while the lines are still in L2)
__device__ __forceinline__ void ic3_st_obs(float4* p, const float4& v, bool keep) {
  if (keep) *p = v;
  else __stcs(p, v);
}
__device__ __forceinline__ void ic3_st_obs(float* p, float v, bool keep) {
  if (keep) *p = v;
  else __stcs(p, v);
}
// Observation batches up to this size are written with plain stores so that the encoder launched right after
// them reads L2 instead of HBM (126 MB L2 on B200); larger ones stream with evict-first stores.
constexpr size_t IC3_OBS_L2_KEEP_BYTES = (size_t)96 << 20;
__device__ __forceinline__ float4 ic3_ld_stream(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ float ic3_ld_stream(const float* p) { return __ldcs(p); }
