// Per-step tail of Trainer.get_episode (reference trainer.py:69-125), executed by
// the warp that owns one environment (lane = agent) right after the env step.
#pragma once
#include "ic3_common.cuh"

struct RolloutOpt {
  int has;            // 0: plain gym semantics (ic3_rollout_io* was NULL)
  ic3_rollout_io io;
};

static inline RolloutOpt make_rollout_opt(const ic3_rollout_io* r) {
  RolloutOpt o;
  o.has = r != nullptr;
  if (r) o.io = *r;
  else memset(&o.io, 0, sizeof(o.io));
  return o;
}

// Reference batch boundary (trainer.py:231-237): a worker plays whole episodes until it holds >= batch_size steps,
// so its last episode overshoots.  With r.batch_size > 0 a slot HALTS at the first episode end at which its step
// count has reached batch_size; from then on the lock-step iterations skip it: no env step, no statistics, null
// records (rec_valid = 0, alive = 0, reward = 0, episode_mask = 0).  Returns true for a halted slot.
__device__ __forceinline__ bool ic3_rollout_halted(const ic3_rollout_io& r, int e, int B, int N, int lane) {
  if (r.batch_size <= 0 || !r.halted || !r.halted[e]) return false;
  if (lane < N) {
    const size_t idx = ((size_t)r.t * B + e) * N + lane;
    if (r.rec_reward) r.rec_reward[idx] = 0.f;
    if (r.rec_mini_mask) r.rec_mini_mask[idx] = 1;
    if (r.rec_alive) r.rec_alive[idx] = 0;
  }
  if (lane == 0) {
    if (r.rec_episode_mask) r.rec_episode_mask[(size_t)r.t * B + e] = 0;
    if (r.rec_valid) r.rec_valid[(size_t)r.t * B + e] = 0;
  }
  return true;
}

// Returns true when the episode of env `e` ends at this step
// (env done, or t == max_steps-1: trainer.py:90, or the batch is cut here).
__device__ __forceinline__ bool ic3_rollout_tail(const ic3_rollout_io& r, int e, int B, int N, int lane,
                                                 float reward, bool env_done, uint8_t alive_post,
                                                 uint8_t completed, int success) {
  const int tep = r.t_ep[e];
  __syncwarp();
  const bool done_t = env_done || (tep == r.max_steps - 1) || (r.last != 0);
  if (lane < N) {
    const size_t idx = ((size_t)r.t * B + e) * N + lane;
    const int a = e * N + lane;
    if (r.rec_reward) r.rec_reward[idx] = reward;                                  // trainer.py:104
    if (r.rec_mini_mask) r.rec_mini_mask[idx] = done_t ? 1 : (uint8_t)(1 - completed);  // :97-99
    if (r.rec_alive) r.rec_alive[idx] = alive_post;                                // :78-81
    if (r.hard_attn) {                                                             // :70-73
      const uint8_t comm =
          r.comm_action_one ? 1 : (uint8_t)(r.action[(size_t)a * r.nheads + (r.nheads - 1)] != 0);
      r.comm_next[a] = comm;
      if (r.stat_comm) r.stat_comm[a] += (float)comm;
    }
    r.alive_next[a] = alive_post;
    if (r.stat_reward) r.stat_reward[a] += reward;                                 // :86
  }
  if (lane == 0) {
    if (r.rec_episode_mask) r.rec_episode_mask[(size_t)r.t * B + e] = done_t ? 0 : 1;  // :92-96
    if (r.rec_valid) r.rec_valid[(size_t)r.t * B + e] = 1;
    r.fresh[e] = done_t ? 1 : 0;
    r.t_ep[e] = done_t ? 0 : tep + 1;
    int nsteps = 0;
    if (r.stat_steps) nsteps = (r.stat_steps[e] += 1);                             // :109
    if (done_t) {
      if (r.batch_size > 0 && r.halted && nsteps >= r.batch_size) r.halted[e] = 1; // trainer.py:231 loop condition
      if (r.stat_episodes) r.stat_episodes[e] += 1;                                // :235
      if (r.stat_success && success > 0) r.stat_success[e] += success;             // :124-125
    }
  }
  return done_t;
}

// Snapshot of what the NEXT policy step will see (ic3_rollout_io.snap_*): called by the env step kernels after the
// tail / auto-reset, with the slot's current fresh / comm / alive / step index already final.
__device__ __forceinline__ void ic3_rollout_snapshot(const ic3_rollout_io& r, int e, int B, int N, int lane) {
  const int t1 = r.t + 1;
  if (r.snap_T <= 0 || t1 >= r.snap_T) return;
  if (lane < N) {
    const size_t idx = ((size_t)t1 * B + e) * N + lane;
    const int a = e * N + lane;
    if (r.snap_comm && r.hard_attn) r.snap_comm[idx] = r.comm_next[a];
    if (r.snap_alive) r.snap_alive[idx] = r.alive_next[a];
  }
  if (lane == 0) {
    if (r.snap_fresh) r.snap_fresh[(size_t)t1 * B + e] = r.fresh[e];
    if (r.snap_tep) r.snap_tep[(size_t)t1 * B + e] = r.t_ep[e];
  }
}
