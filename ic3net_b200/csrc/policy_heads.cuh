// Value / action heads, log-softmax and inverse-CDF sampling for one agent row, executed by
// one warp (reference: comm.py:228-239, action_utils.py:32-36), for the fp32 SIMT policy
// kernel (policy.cu).
#pragma once
#include "ic3_common.cuh"

// log-softmax + inverse-CDF sampling of one head; logits live one per lane
// (lane off+a holds logit a).  Every lane of the warp executes this.
__device__ __forceinline__ void head_logp_sample(float mylogit, int off, int na, float u, bool do_sample,
                                                 float& mylogp, int& action) {
  float m = -INFINITY;
  for (int a = 0; a < na; ++a) m = fmaxf(m, __shfl_sync(IC3_FULL_MASK, mylogit, off + a));
  float s = 0.f;
  for (int a = 0; a < na; ++a) s += expf(__shfl_sync(IC3_FULL_MASK, mylogit, off + a) - m);
  const float lse = m + logf(s);
  mylogp = mylogit - lse;
  action = na - 1;
  if (do_sample) {
    float cdf = 0.f;
    bool found = false;
    for (int a = 0; a < na; ++a) {
      cdf += expf(__shfl_sync(IC3_FULL_MASK, mylogp, off + a));
      if (!found && cdf > u) {
        action = a;
        found = true;
      }
    }
  }
}

// hv[m] = h'[row][lane + 32*m].  grow = global agent row, e = env, i = agent in env.
template <int H>
__device__ __forceinline__ void heads_for_row(const ic3_policy_cfg& cfg, const float* __restrict__ head_w,
                                              const float* __restrict__ head_b, const float (&hv)[H / 32],
                                              size_t grow, int e, int i, int lane, const uint32_t* tick,
                                              const uint32_t* draws, float* __restrict__ value,
                                              float* __restrict__ logp, int32_t* __restrict__ action) {
  int atot = 0;
  for (int k = 0; k < cfg.nheads; ++k) atot += cfg.head_dim[k];
  const int nout = 1 + atot;
  float mylogit = 0.f;
  for (int o = 0; o < nout; ++o) {
    float part = 0.f;
#pragma unroll
    for (int m = 0; m < H / 32; ++m) part = fmaf(hv[m], __ldg(head_w + (size_t)o * H + lane + 32 * m), part);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) part += __shfl_xor_sync(IC3_FULL_MASK, part, s);
    if (lane == o) mylogit = part + __ldg(head_b + o);
  }
  if (lane == 0) value[grow] = mylogit;
  uint4 w = make_uint4(0, 0, 0, 0);
  const bool do_sample = action != nullptr;
  if (do_sample && !draws)
    w = ic3_draw24(cfg.seed, cfg.env_id0 + (uint32_t)e, tick ? tick[e] : 0u, IC3_STREAM_ACTION, (uint32_t)i);
  int off = 1;
  for (int k = 0; k < cfg.nheads; ++k) {
    const int na = cfg.head_dim[k];
    uint32_t u24 = 0;
    if (do_sample) u24 = draws ? draws[grow * cfg.nheads + k] : ic3_word(w, k);
    float mylogp;
    int act;
    head_logp_sample(mylogit, off, na, (float)u24 * 5.9604644775390625e-08f, do_sample, mylogp, act);
    if (lane >= off && lane < off + na) logp[grow * atot + (off - 1) + (lane - off)] = mylogp;
    if (do_sample && lane == 0) action[grow * cfg.nheads + k] = act;
    off += na;
  }
}
