// Traffic-junction environment kernels (reference: ic3net_envs/traffic_junction_env.py).
//
// One CTA per environment; warp 0 owns the car state (lane = car slot).  The only
// sequential part of the reference step -- _add_cars looping over arrival groups with
// an early exit and a dead-slot choice (:369-393, :614-618) -- stays a warp-uniform
// loop: dead slots are a ballot, "the j-th dead slot" is __fns on that ballot.
// Static tables (road-id grid, routes) are read-only device arrays built once on host.
#include <cstring>

#include "ic3_common.cuh"
#include "rollout_tail.cuh"

namespace {

struct TJArgs {
  ic3_tj_cfg cfg;
  ic3_tj_state st;
};

// reset(): traffic_junction_env.py:160-204 (state part)
__device__ __forceinline__ void tj_reset_env(const TJArgs& a, int e, int lane) {
  const int N = a.cfg.N;
  if (lane < N) {
    const size_t i = (size_t)e * N + lane;
    a.st.loc[i * 2] = 0;
    a.st.loc[i * 2 + 1] = 0;
    a.st.alive[i] = 0;
    a.st.wait[i] = 0;
    a.st.route_id[i] = -1;
    a.st.route_pos[i] = -1;
    a.st.last_act[i] = 0;
    a.st.completed[i] = 0;
  }
  if (lane == 0) {
    a.st.cars_in_sys[e] = 0;
    a.st.has_failed[e] = 0;
  }
}

__global__ void tj_reset_kernel(TJArgs a, const uint8_t* __restrict__ mask) {
  const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= a.cfg.B) return;
  if (mask && !mask[e]) return;
  tj_reset_env(a, e, threadIdx.x & 31);
}

// _get_obs (:321-366) + _flatten_obs (env_wrappers.py:88-98): row i =
// [last_act, route_id/(npath-1), W*W cells x V classes]; all zero for dead cars.
// s_cell packs (cls | count << 16).
__device__ __forceinline__ void tj_write_obs(const ic3_tj_cfg& cfg, const int* s_r, const int* s_c,
                                            const int* s_alive, const int* s_rid, const int* s_lact,
                                            uint32_t* s_cell, float* __restrict__ obs_env, bool keep) {
  const int N = cfg.N, v = cfg.vision, W = 2 * v + 1, WW = W * W, V = cfg.vocab;
  const int O = 2 + WW * V;
  const int ncell = N * WW;
  for (int c = threadIdx.x; c < ncell; c += blockDim.x) {
    const int i = c / WW, w = c - i * WW, dy = w / W, dx = w - dy * W;
    const int rr = s_r[i] - v + dy, cc = s_c[i] - v + dx;
    uint32_t info = (uint32_t)cfg.outside_cls;  // padding is OUTSIDE (:316)
    if (rr >= 0 && rr < cfg.h && cc >= 0 && cc < cfg.w) {
      int cnt = 0;  // every slot counts, dead ones are parked at (0,0) (:326-327)
      for (int j = 0; j < N; ++j) cnt += (s_r[j] == rr && s_c[j] == cc);
      info = (uint32_t)cfg.grid[rr * cfg.w + cc] | ((uint32_t)cnt << 16);
    }
    s_cell[c] = info;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  for (int c = warp; c < ncell; c += nwarp) {
    const int i = c / WW, w = c - i * WW;
    const uint32_t info = s_cell[c];
    const int cls = (int)(info & 0xffffu);
    const float cnt = (float)(info >> 16);
    const bool live = s_alive[i] != 0;
    float* dst = obs_env + (size_t)i * O + 2 + (size_t)w * V;
    for (int q = lane; q < V; q += 32) {
      float o = (q == cls) ? 1.f : 0.f;
      if (q == cfg.car_cls) o += cnt;
      ic3_st_obs(dst + q, live ? o : 0.f, keep);
    }
  }
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const bool live = s_alive[i] != 0;
    float* dst = obs_env + (size_t)i * O;
    dst[0] = live ? (float)s_lact[i] : 0.f;                                    // / (naction-1) == 1
    dst[1] = live ? (float)s_rid[i] / (float)(cfg.npath - 1) : 0.f;            // :341
  }
}

__global__ void tj_step_kernel(TJArgs a, const int32_t* __restrict__ act, int act_stride,
                               const uint32_t* __restrict__ draws, float* __restrict__ reward,
                               float* __restrict__ obs, int32_t* err, RolloutOpt r, int do_step, int keep_l2) {
  extern __shared__ uint32_t s_cell[];
  __shared__ int s_r[IC3_MAX_AGENTS], s_c[IC3_MAX_AGENTS], s_alive[IC3_MAX_AGENTS], s_rid[IC3_MAX_AGENTS],
      s_lact[IC3_MAX_AGENTS];
  const ic3_tj_cfg& cfg = a.cfg;
  const int N = cfg.N;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // with an observation block to write: one CTA per env, warp 0 owns the state; without: one WARP per env (pp_env.cu)
  const int e = obs ? (int)blockIdx.x : (int)(blockIdx.x * (blockDim.x >> 5)) + warp;
  if (obs ? warp == 0 : e < cfg.B) {
    const size_t i = (size_t)e * N + lane;
    int rr = 0, cc = 0, alive = 0, wait = 0, rid = -1, rpos = -1, lact = 0;
    if (lane < N) {
      rr = a.st.loc[i * 2];
      cc = a.st.loc[i * 2 + 1];
      alive = a.st.alive[i];
      wait = a.st.wait[i];
      rid = a.st.route_id[i];
      rpos = a.st.route_pos[i];
      lact = a.st.last_act[i];
    }
    if (do_step && r.has && ic3_rollout_halted(r.io, e, cfg.B, N, lane)) {
      // this slot has completed its batch (trainer.py:231): nothing moves, null records
    } else if (do_step) {
      // ---- _take_action :540-581 ----
      int completed = 0;
      int av = 1;
      if (lane < N) av = act[i * act_stride];
      if (lane >= N) av = 1;
      if (lane < N && (av < 0 || av > 2)) atomicOr(err, IC3_ERR_BAD_ACTION);  // :228 (sic, <=)
      if (lane < N && alive) {
        wait += 1;                       // :546
        if (av == 1) {
          lact = 1;                      // BRAKE :549-551
        } else if (av == 0) {            // GAS :554
          rpos += 1;
          const int len = cfg.route_len[rid];
          if (rpos == len) {             // :560-568
            alive = 0;
            wait = 0;
            rr = 0;
            cc = 0;
            completed = 1;
          } else if (rpos > len) {
            atomicOr(err, IC3_ERR_ROUTE_OVERRUN);  // :570-572
          } else {
            const int cell = cfg.route_cells[(size_t)rid * cfg.Lmax + rpos];
            rr = cell >> 16;
            cc = cell & 0xffff;
            lact = 0;                    // :581
          }
        }
      }
      int cars = a.st.cars_in_sys[e] - __popc(__ballot_sync(IC3_FULL_MASK, completed));
      // ---- _add_cars :369-393 ----
      const uint32_t tick = a.st.tick[e];
      for (int g = 0; g < cfg.G; ++g) {
        if (cars >= N) break;            // :371-372
        uint32_t w0, w1, w2;
        if (draws) {
          const uint32_t* d = draws + ((size_t)e * cfg.G + g) * 3;
          w0 = d[0]; w1 = d[1]; w2 = d[2];
        } else {
          const uint4 w = ic3_draw24(cfg.seed, cfg.env_id0 + (uint32_t)e, tick, IC3_STREAM_TJ_SPAWN, (uint32_t)g);
          w0 = w.x; w1 = w.y; w2 = w.z;
        }
        if (w0 <= cfg.spawn_thr) {       // np.random.uniform() <= add_rate :375
          const unsigned dead = __ballot_sync(IC3_FULL_MASK, lane < N && !alive);
          const int k = __popc(dead);    // > 0 because cars < N
          const int j = (int)ic3_pick(w1, (uint32_t)k);
          const int slot = (int)__fns(dead, 0, j + 1);      // _choose_dead :614-618
          const int p = (int)ic3_pick(w2, (uint32_t)cfg.P); // :383
          if (lane == slot) {
            alive = 1;
            rid = p + g * cfg.P;         // :385
            rpos = 0;
            const int cell = cfg.route_cells[(size_t)rid * cfg.Lmax];
            rr = cell >> 16;
            cc = cell & 0xffff;
          }
          cars += 1;
        }
      }
      // ---- _get_reward :585-595 ----
      int crash = 0;
      for (int j = 0; j < N; ++j) {
        const int rj = __shfl_sync(IC3_FULL_MASK, rr, j), cj = __shfl_sync(IC3_FULL_MASK, cc, j);
        crash |= (j != lane && rj == rr && cj == cc && (rr | cc) != 0);
      }
      crash = (lane < N) ? crash : 0;
      const bool any_crash = __any_sync(IC3_FULL_MASK, crash);
      double rew = -0.01 * (double)wait;         // TIMESTEP_PENALTY * wait :586
      if (crash) rew += -10.0;                   // CRASH_PENALTY :591
      rew = alive ? rew : 0.0;                   // :594
      int failed = a.st.has_failed[e];
      failed |= any_crash ? 1 : 0;
      if (lane < N) {
        a.st.loc[i * 2] = rr;
        a.st.loc[i * 2 + 1] = cc;
        a.st.alive[i] = (uint8_t)alive;
        a.st.wait[i] = wait;
        a.st.route_id[i] = rid;
        a.st.route_pos[i] = rpos;
        a.st.last_act[i] = (uint8_t)lact;
        a.st.completed[i] = (uint8_t)completed;
        reward[i] = (float)rew;
      }
      if (lane == 0) {
        a.st.cars_in_sys[e] = cars;
        a.st.has_failed[e] = (uint8_t)failed;
        a.st.tick[e] = tick + 1;
      }
      if (r.has) {
        // episode_over is never set by the reference env (:219,252): episodes end on max_steps
        const bool done_t = ic3_rollout_tail(r.io, e, cfg.B, N, lane, (float)rew, false, (uint8_t)alive,
                                             (uint8_t)completed, 1 - failed);
        if (done_t) {
          __syncwarp();
          tj_reset_env(a, e, lane);
          rr = cc = alive = wait = lact = 0;
          rid = rpos = -1;
        }
      }
    }
    if (do_step && r.has && r.io.snap_T > 0) {          // inputs of the next policy step, for compute_grad
      __syncwarp();
      ic3_rollout_snapshot(r.io, e, cfg.B, N, lane);
      if (r.io.t + 1 < r.io.snap_T && lane < N) {
        const size_t k = ((size_t)(r.io.t + 1) * cfg.B + e) * N + lane;
        if (r.io.snap_tj_loc) {
          r.io.snap_tj_loc[2 * k] = rr;
          r.io.snap_tj_loc[2 * k + 1] = cc;
        }
        if (r.io.snap_tj_alive) r.io.snap_tj_alive[k] = (uint8_t)alive;
        if (r.io.snap_tj_last_act) r.io.snap_tj_last_act[k] = (uint8_t)lact;
        if (r.io.snap_tj_route_id) r.io.snap_tj_route_id[k] = rid;
      }
    }
    if (obs && lane < N) {
      s_r[lane] = rr;
      s_c[lane] = cc;
      s_alive[lane] = alive;
      s_rid[lane] = rid;
      s_lact[lane] = lact;
    }
  }
  if (obs == nullptr) return;
  __syncthreads();
  const int W = 2 * cfg.vision + 1;
  tj_write_obs(cfg, s_r, s_c, s_alive, s_rid, s_lact, s_cell, obs + (size_t)e * N * (2 + W * W * cfg.vocab), keep_l2 != 0);
}

int tj_check(const ic3_tj_cfg* cfg, const ic3_tj_state* st) {
  if (!cfg || !st) return IC3_E_NULL;
  if (!st->loc || !st->alive || !st->wait || !st->route_id || !st->route_pos || !st->last_act ||
      !st->completed || !st->cars_in_sys || !st->has_failed || !st->tick)
    return IC3_E_NULL;
  if (!cfg->grid || !cfg->route_len || !cfg->route_cells) return IC3_E_NULL;
  if (cfg->B <= 0 || cfg->N <= 0 || cfg->N > IC3_MAX_AGENTS) return IC3_E_RANGE;
  if (cfg->h <= 0 || cfg->w <= 0 || cfg->h > 32767 || cfg->w > 32767) return IC3_E_RANGE;
  if (cfg->vision < 0 || cfg->vision > 7) return IC3_E_RANGE;
  if (cfg->G <= 0 || cfg->P <= 0 || cfg->Lmax <= 0 || cfg->npath < 2 || cfg->vocab <= 0 || cfg->vocab > 65535)
    return IC3_E_RANGE;
  return IC3_OK;
}

int tj_launch(const ic3_tj_cfg* cfg, const ic3_tj_state* st, const int32_t* act, int act_stride,
              const uint32_t* draws, float* reward, float* obs, int32_t* err, const ic3_rollout_io* r,
              int do_step, cudaStream_t s) {
  TJArgs a{*cfg, *st};
  const int W = 2 * cfg->vision + 1;
  const size_t smem = obs ? (size_t)cfg->N * W * W * sizeof(uint32_t) : 0;
  const int threads = obs ? 128 : 32 * IC3_ENV_WARPS;
  const int grid = obs ? cfg->B : (cfg->B + IC3_ENV_WARPS - 1) / IC3_ENV_WARPS;
  RolloutOpt ro = make_rollout_opt(r);
  const int keep = obs && (size_t)cfg->B * cfg->N * (2 + W * W * cfg->vocab) * sizeof(float) <= IC3_OBS_L2_KEEP_BYTES;
  tj_step_kernel<<<grid, threads, smem, s>>>(a, act, act_stride, draws, reward, obs, err, ro, do_step, keep);
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}

}  // namespace

extern "C" int ic3_tj_reset(const ic3_tj_cfg* cfg, const ic3_tj_state* st, const uint8_t* mask,
                            float* obs, void* stream) {
  int rc = tj_check(cfg, st);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  TJArgs a{*cfg, *st};
  const int wpb = 4;
  tj_reset_kernel<<<(cfg->B + wpb - 1) / wpb, wpb * 32, 0, s>>>(a, mask);
  IC3_LAUNCH_CHECK();
  if (obs) return tj_launch(cfg, st, nullptr, 0, nullptr, nullptr, obs, nullptr, nullptr, 0, s);
  return IC3_OK;
}

extern "C" int ic3_tj_step(const ic3_tj_cfg* cfg, const ic3_tj_state* st, const int32_t* act,
                           int32_t act_stride, const uint32_t* draws, float* reward, float* obs,
                           int32_t* err, const ic3_rollout_io* r, void* stream) {
  int rc = tj_check(cfg, st);
  if (rc) return rc;
  if (!act || !reward || !err || act_stride < 1) return IC3_E_NULL;
  if (r && (!r->t_ep || !r->fresh || !r->alive_next || (r->hard_attn && (!r->comm_next || !r->action))))
    return IC3_E_NULL;
  return tj_launch(cfg, st, act, act_stride, draws, reward, obs, err, r, 1, (cudaStream_t)stream);
}

extern "C" int ic3_tj_obs(const ic3_tj_cfg* cfg, const ic3_tj_state* st, float* obs, void* stream) {
  int rc = tj_check(cfg, st);
  if (rc) return rc;
  if (!obs) return IC3_E_NULL;
  return tj_launch(cfg, st, nullptr, 0, nullptr, nullptr, obs, nullptr, nullptr, 0, (cudaStream_t)stream);
}
