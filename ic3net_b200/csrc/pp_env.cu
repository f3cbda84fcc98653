// Predator-prey environment kernels (reference: ic3net_envs/predator_prey_env.py).
//
// Layout in HBM: loc [B, N+1, 2] int32 (predators, then the prey), reached [B,N] u8,
// done [B] u8.  With cfg.enemy_comm the prey is agent row N of act / reward / obs (NA = N + 1 rows per env).  One CTA per environment; warp 0 owns the integer state (lane = agent,
// reductions are ballots), all warps stream the observation block of the env:
// [N * W*W cells][V] floats, contiguous, written once with 16-byte evict-first stores.
#include <algorithm>
#include <cstring>

#include "ic3_common.cuh"
#include "rollout_tail.cuh"

namespace {

struct PPArgs {
  ic3_pp_cfg cfg;
  ic3_pp_state st;
};

// reset(): predator_prey_env.py:146-168, _get_cordinates :173-175.
// N+1 distinct cells by rejection from the spawn stream; executed by one warp.
__device__ __forceinline__ void pp_reset_env(const PPArgs& a, int e, int lane) {
  const int N = a.cfg.N, D = a.cfg.dim, need = N + 1;
  const uint32_t ncell = (uint32_t)(D * D);
  const uint32_t epi = a.st.episode[e];
  int mycell = -1, cnt = 0;
  for (uint32_t blk = 0; cnt < need && blk < 4096u; ++blk) {
    const uint4 w = ic3_draw24(a.cfg.seed, a.cfg.env_id0 + (uint32_t)e, epi, IC3_STREAM_PP_RESET, blk);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (cnt < need) {
        const int cand = (int)ic3_pick(ic3_word(w, i), ncell);
        const bool dup = __any_sync(IC3_FULL_MASK, lane < cnt && mycell == cand);
        if (!dup) {
          if (lane == cnt) mycell = cand;
          ++cnt;
        }
      }
    }
  }
  if (lane < need) {
    int* l = a.st.loc + ((size_t)e * need + lane) * 2;
    l[0] = mycell / D;
    l[1] = mycell % D;
  }
  if (lane < N) a.st.reached[(size_t)e * N + lane] = 0;
  if (lane == 0) {
    a.st.episode[e] = epi + 1;
    a.st.done[e] = 0;
    a.st.success[e] = -1;
  }
}

__global__ void pp_reset_kernel(PPArgs a, const uint8_t* __restrict__ mask) {
  const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= a.cfg.B) return;
  if (mask && !mask[e]) return;
  pp_reset_env(a, e, threadIdx.x & 31);
}

// _get_obs (:188-210) + _flatten_obs (env_wrappers.py:98): the env's block of
// N*W*W cells, V floats each.  s_cell packs (cls | npred << 16 | nprey << 24).
template <bool VEC4>
__device__ __forceinline__ void pp_write_obs(const ic3_pp_cfg& cfg, const int* s_r, const int* s_c,
                                            uint32_t* s_cell, float* __restrict__ obs_env, bool keep) {
  const int N = cfg.N, D = cfg.dim, v = cfg.vision, W = 2 * v + 1, WW = W * W;
  const int V = D * D + 4, OUTSIDE = D * D + 1;
  const int ncell = ic3_pp_agents(cfg) * WW;      // row N (enemy_comm): the window around the prey (:203-207)
  for (int c = threadIdx.x; c < ncell; c += blockDim.x) {
    const int i = c / WW, w = c - i * WW, dy = w / W, dx = w - dy * W;
    const int rr = s_r[i] - v + dy, cc = s_c[i] - v + dx;
    uint32_t info = (uint32_t)OUTSIDE;
    if (rr >= 0 && rr < D && cc >= 0 && cc < D) {
      int npred = 0;
      for (int j = 0; j < N; ++j) npred += (s_r[j] == rr && s_c[j] == cc);
      const int nprey = (s_r[N] == rr && s_c[N] == cc);
      info = (uint32_t)(rr * D + cc) | ((uint32_t)npred << 16) | ((uint32_t)nprey << 24);
    }
    s_cell[c] = info;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  for (int c = warp; c < ncell; c += nwarp) {
    const uint32_t info = s_cell[c];
    const int cls = (int)(info & 0xffffu);
    const float npred = (float)((info >> 16) & 0xffu), nprey = (float)(info >> 24);
    float* dst = obs_env + (size_t)c * V;
    if (VEC4) {
      const int V4 = V >> 2, qc = cls >> 2, qp = (V - 1) >> 2, qy = (V - 2) >> 2;
      for (int q = lane; q < V4; q += 32) {
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q == qc) {
          const int k = cls & 3;
          o.x = k == 0 ? 1.f : 0.f; o.y = k == 1 ? 1.f : 0.f; o.z = k == 2 ? 1.f : 0.f; o.w = k == 3 ? 1.f : 0.f;
        }
        if (q == qy) {  // PREY class = V-2 (V % 4 == 0 -> component 2)
          o.z = nprey;
        }
        if (q == qp) {  // PREDATOR class = V-1 -> component 3
          o.w = npred;
        }
        ic3_st_obs(reinterpret_cast<float4*>(dst) + q, o, keep);
      }
    } else {
      for (int q = lane; q < V; q += 32) {
        float o = (q == cls) ? 1.f : 0.f;
        if (q == V - 2) o = nprey;
        if (q == V - 1) o = npred;
        ic3_st_obs(dst + q, o, keep);
      }
    }
  }
}

// step(): predator_prey_env.py:112-144.  One CTA per env.
template <bool VEC4>
__global__ void pp_step_kernel(PPArgs a, const int32_t* __restrict__ act, int act_stride,
                               float* __restrict__ reward, float* __restrict__ obs, int32_t* err,
                               RolloutOpt r, int do_step, int keep_l2) {
  extern __shared__ uint32_t s_cell[];
  __shared__ int s_r[IC3_MAX_AGENTS + 1], s_c[IC3_MAX_AGENTS + 1];
  const int N = a.cfg.N, D = a.cfg.dim;
  const int NA = ic3_pp_agents(a.cfg);      // agent rows (N predators [+ the prey with enemy_comm])
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // with an observation block to write: one CTA per env, warp 0 owns the state.  Without (index-form encoder /
  // observation handles): the state update is all there is, one WARP per env, several envs per CTA
  const int e = obs ? (int)blockIdx.x : (int)(blockIdx.x * (blockDim.x >> 5)) + warp;
  if (obs ? warp == 0 : e < a.cfg.B) {
    int rr = 0, cc = 0, rch = 0;
    if (lane <= N) {
      const int* l = a.st.loc + ((size_t)e * (N + 1) + lane) * 2;
      rr = l[0];
      cc = l[1];
    }
    if (lane < N) rch = a.st.reached[(size_t)e * N + lane];
    if (do_step && r.has && ic3_rollout_halted(r.io, e, a.cfg.B, NA, lane)) {
      // this slot has completed its batch (trainer.py:231): nothing moves, null records
    } else if (do_step) {
      if (a.st.done[e]) {  // :129-130 RuntimeError("Episode is done")
        if (lane == 0) atomicOr(err, IC3_ERR_EPISODE_DONE);
      } else {
        int av = 4;
        if (lane < NA) av = act[((size_t)e * NA + lane) * act_stride];
        if (lane >= NA) av = 4;
        if (lane < NA && (av < 0 || av > a.cfg.naction)) atomicOr(err, IC3_ERR_BAD_ACTION);  // :137 (sic, <=)
        if (lane < N && !rch) {  // _take_action :212-252: every move is a clamped move
          if (av == 0) rr = max(0, rr - 1);
          else if (av == 1) cc = min(D - 1, cc + 1);
          else if (av == 2) rr = min(D - 1, rr + 1);
          else if (av == 3) cc = max(0, cc - 1);
        }
        // _get_reward :254-290
        const int pr = __shfl_sync(IC3_FULL_MASK, rr, N), pc = __shfl_sync(IC3_FULL_MASK, cc, N);
        const bool on = lane < N && rr == pr && cc == pc;
        const int n_on = __popc(__ballot_sync(IC3_FULL_MASK, on));
        double rew = -0.05;  // TIMESTEP_PENALTY :40
        if (on) {
          if (a.cfg.mode == IC3_PP_COOPERATIVE) rew = 0.05 * (double)n_on;       // :262-263
          else if (a.cfg.mode == IC3_PP_COMPETITIVE) rew = 0.05 / (double)n_on;  // :264-266
          else rew = 0.0;                                                         // :267-268 PREY_REWARD
        }
        if (lane == N) rew = n_on == 0 ? 0.05 : 0.0;   // prey reward (enemy_comm row), :276-281
        rch |= on ? 1 : 0;  // :271
        const bool allr = __ballot_sync(IC3_FULL_MASK, lane >= N || rch) == IC3_FULL_MASK;
        const bool done = (a.cfg.mode == IC3_PP_MIXED) && allr;  // :273-274
        int success = a.st.success[e];
        if (a.cfg.mode != IC3_PP_COMPETITIVE) success = (n_on == N) ? 1 : 0;  // :284-288
        if (lane < N) {
          int* l = a.st.loc + ((size_t)e * (N + 1) + lane) * 2;
          l[0] = rr;
          l[1] = cc;
          a.st.reached[(size_t)e * N + lane] = (uint8_t)rch;
        }
        if (lane < NA) reward[(size_t)e * NA + lane] = (float)rew;
        if (lane == 0) {
          a.st.done[e] = done ? 1 : 0;
          a.st.success[e] = success;
          a.st.tick[e] += 1;
        }
        if (r.has) {
          const bool done_t = ic3_rollout_tail(r.io, e, a.cfg.B, NA, lane, (float)rew, done, 1, 0, success);
          if (done_t) {
            __syncwarp();
            pp_reset_env(a, e, lane);
            __syncwarp();
            if (lane <= N) {
              const int* l = a.st.loc + ((size_t)e * (N + 1) + lane) * 2;
              rr = l[0];
              cc = l[1];
            }
          }
        }
      }
    }
    if (do_step && r.has && r.io.snap_T > 0) {          // inputs of the next policy step, for compute_grad
      __syncwarp();
      ic3_rollout_snapshot(r.io, e, a.cfg.B, NA, lane);
      if (r.io.snap_pp_loc && r.io.t + 1 < r.io.snap_T && lane <= N) {
        int* d = r.io.snap_pp_loc + (((size_t)(r.io.t + 1) * a.cfg.B + e) * (N + 1) + lane) * 2;
        d[0] = rr;
        d[1] = cc;
      }
    }
    if (obs && lane <= N) {
      s_r[lane] = rr;
      s_c[lane] = cc;
    }
  }
  if (obs == nullptr) return;
  __syncthreads();
  const int W = 2 * a.cfg.vision + 1;
  pp_write_obs<VEC4>(a.cfg, s_r, s_c, s_cell, obs + (size_t)e * NA * W * W * (D * D + 4), keep_l2 != 0);
}

int pp_check(const ic3_pp_cfg* cfg, const ic3_pp_state* st) {
  if (!cfg || !st) return IC3_E_NULL;
  if (!st->loc || !st->reached || !st->done || !st->success || !st->episode || !st->tick) return IC3_E_NULL;
  if (cfg->B <= 0 || cfg->N <= 0 || cfg->N >= IC3_MAX_AGENTS) return IC3_E_RANGE;  // lane N holds the prey
  if (cfg->dim <= 0 || cfg->dim > 181 || cfg->vision < 0 || cfg->vision > 7) return IC3_E_RANGE;
  if (cfg->N + 1 > cfg->dim * cfg->dim) return IC3_E_RANGE;
  if (cfg->mode < 0 || cfg->mode > 2) return IC3_E_RANGE;  // :269 "Incorrect mode"
  if (cfg->naction != 4 && cfg->naction != 5) return IC3_E_RANGE;
  return IC3_OK;
}

// Residency bound of the observation-writing launch (one 256-thread CTA per env): at most 4 CTAs per SM.  The kernel's
// 46-48 registers would let 5 CTAs share an SM, and the observation write is then slower: on B200 (predator-prey hard,
// 8192 envs, 1000 W) 0.190 ms at 5 CTAs/SM against 0.184 ms at 4.  Requesting more than a fifth of the SM's shared
// memory per CTA (dynamic shared memory, unused beyond the kernel's own cell buffer) keeps the fifth CTA out.
constexpr int PP_OBS_CTAS_PER_SM = 4;
size_t pp_obs_smem_floor() {
  static size_t floor = 0;
  if (floor == 0) {
    int dev = 0, per_sm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    floor = (size_t)per_sm / (PP_OBS_CTAS_PER_SM + 1) + 1;
    if (floor > 48 * 1024) floor = 48 * 1024;      // the default dynamic shared-memory limit of a launch
  }
  return floor;
}

int pp_launch(const ic3_pp_cfg* cfg, const ic3_pp_state* st, const int32_t* act, int act_stride,
              float* reward, float* obs, int32_t* err, const ic3_rollout_io* r, int do_step,
              cudaStream_t s) {
  PPArgs a{*cfg, *st};
  const int W = 2 * cfg->vision + 1;
  const int V = cfg->dim * cfg->dim + 4;
  const int NA = ic3_pp_agents(*cfg);
  const size_t smem = obs ? std::max((size_t)NA * W * W * sizeof(uint32_t), pp_obs_smem_floor()) : 0;
  const int threads = obs ? 256 : 32 * IC3_ENV_WARPS;
  const int grid = obs ? cfg->B : (cfg->B + IC3_ENV_WARPS - 1) / IC3_ENV_WARPS;
  const bool vec4 = (V % 4 == 0) && ((reinterpret_cast<uintptr_t>(obs) & 15) == 0);
  RolloutOpt ro = make_rollout_opt(r);
  // small observation batches stay in L2 for the encoder that follows (see IC3_OBS_L2_KEEP_BYTES)
  const int keep = obs && (size_t)cfg->B * NA * W * W * V * sizeof(float) <= IC3_OBS_L2_KEEP_BYTES;
  if (vec4) pp_step_kernel<true><<<grid, threads, smem, s>>>(a, act, act_stride, reward, obs, err, ro, do_step, keep);
  else pp_step_kernel<false><<<grid, threads, smem, s>>>(a, act, act_stride, reward, obs, err, ro, do_step, keep);
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}

}  // namespace

extern "C" int ic3_pp_reset(const ic3_pp_cfg* cfg, const ic3_pp_state* st, const uint8_t* mask,
                            float* obs, void* stream) {
  int rc = pp_check(cfg, st);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  PPArgs a{*cfg, *st};
  const int wpb = 4;
  pp_reset_kernel<<<(cfg->B + wpb - 1) / wpb, wpb * 32, 0, s>>>(a, mask);
  IC3_LAUNCH_CHECK();
  if (obs) return pp_launch(cfg, st, nullptr, 0, nullptr, obs, nullptr, nullptr, 0, s);
  return IC3_OK;
}

extern "C" int ic3_pp_step(const ic3_pp_cfg* cfg, const ic3_pp_state* st, const int32_t* act,
                           int32_t act_stride, float* reward, float* obs, int32_t* err,
                           const ic3_rollout_io* r, void* stream) {
  int rc = pp_check(cfg, st);
  if (rc) return rc;
  if (!act || !reward || !err || act_stride < 1) return IC3_E_NULL;
  if (r && (!r->t_ep || !r->fresh || !r->alive_next || (r->hard_attn && (!r->comm_next || !r->action))))
    return IC3_E_NULL;
  return pp_launch(cfg, st, act, act_stride, reward, obs, err, r, 1, (cudaStream_t)stream);
}

extern "C" int ic3_pp_obs(const ic3_pp_cfg* cfg, const ic3_pp_state* st, float* obs, void* stream) {
  int rc = pp_check(cfg, st);
  if (rc) return rc;
  if (!obs) return IC3_E_NULL;
  return pp_launch(cfg, st, nullptr, 0, nullptr, obs, nullptr, nullptr, 0, (cudaStream_t)stream);
}
