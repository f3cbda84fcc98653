/*
 * ic3net_b200 -- C ABI of the B200-native IC3Net rollout hot path.
 *
 * The reference (IC3Net/IC3Net) is pure Python and has no FFI layer; its boundary
 * for this path is the duck-typed Python surface listed below.  Every entry
 * point here names the reference interface (file:line under /root/reference) it
 * replaces; the Python classes in ic3net_b200/ keep that surface and call these
 * functions through ctypes (see INTEGRATION.md for the binding a maintainer adds).
 *
 * Conventions
 *   - plain C types only; every pointer inside the *_state / *_io / *_weights
 *     structs is a DEVICE pointer owned by the caller (PyTorch is only the
 *     container); the structs themselves live in host memory;
 *   - every call enqueues work on the caller's `stream` (a cudaStream_t passed
 *     as void*) and returns immediately: 0 = ok, <0 = IC3_E_* argument error,
 *     >0 = cudaError_t of the launch;
 *   - misuse that the reference reports with a Python exception *during* a step
 *     ("Episode is done", predator_prey_env.py:129-130, traffic_junction_env.py:
 *     222-223; route overrun :570-572) is recorded in a caller-supplied device
 *     flag word `err` (bit IC3_ERR_*), which the Python layer turns into the same
 *     exception at its next host read;
 *   - one host thread per GPU, no re-entrancy (the reference is single-threaded,
 *     multi_processing.py:7).
 *
 * Randomness: counter-based Philox4x32-10, key = seed, counter =
 * (env_id0 + env, tick, stream, index); see ic3net_b200/csrc/ic3_common.cuh.  Every
 * stochastic entry point also accepts explicit 24-bit draws ("tape") instead.
 */
#ifndef IC3NET_B200_H
#define IC3NET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IC3_MAX_AGENTS 32   /* one warp lane per agent */
#define IC3_MAX_HEADS 4
#define IC3_MAX_HEAD_DIM 16

enum {
  IC3_OK = 0,
  IC3_E_NULL = -1,        /* required pointer missing */
  IC3_E_RANGE = -2,       /* size / enum out of the supported range */
  IC3_E_UNSUPPORTED = -3  /* configuration the kernels do not implement */
};

enum {
  IC3_ERR_EPISODE_DONE = 1, /* step() on a finished episode */
  IC3_ERR_ROUTE_OVERRUN = 2,
  IC3_ERR_BAD_ACTION = 4,   /* action > naction (reference asserts, :137 / :228) */
  IC3_ERR_PIPELINE = 0x100, /* tcgen05 path: an mbarrier wait ran into its watchdog (mis-programmed pipeline) */
  IC3_ERR_FP16_RANGE = 0x200 /* tcgen05 path: an activation (|a| >= 4094) or folded weight (|w| >= 255) left the range of
                               the fp16 hi/lo operand split; results of that step are not trustworthy -> use the
                               fp32 SIMT kernels (policy_impl = 'simt') for such a model */
};

enum { IC3_PP_MIXED = 0, IC3_PP_COOPERATIVE = 1, IC3_PP_COMPETITIVE = 2 };

const char* ic3_version(void);
const char* ic3_strerror(int code);
/* number of kernels launched by this library since load (bench.py "gpu_launches") */
uint64_t ic3_launch_count(void);

/* ------------------------------------------------------------------------
 * Predator-prey  (ic3net_envs/predator_prey_env.py)
 * ---------------------------------------------------------------------- */
typedef struct {
  int32_t B;        /* environments in the batch */
  int32_t N;        /* predators (args.nfriendly, :79) ; one fixed prey (:78).  Rows of act / reward / obs per env:
                       N + (enemy_comm != 0) */
  int32_t dim;      /* board is dim x dim (:80) */
  int32_t vision;   /* window is (2v+1)^2 (:107) */
  int32_t mode;     /* IC3_PP_* (:262-269) */
  int32_t naction;  /* 5, or 4 with --no_stay (:88-92) */
  uint32_t env_id0; /* global id of env 0 (rank * B): RNG stream selector */
  int32_t enemy_comm; /* --enemy_comm (:69, :203-207, :255, :276-281; main.py:124-131): the prey is one more agent of
                         the policy -- row N of obs / reward / act (its action is ignored, :214-217; its reward is
                         +0.05 while no predator stands on it, else 0) */
  uint64_t seed;
} ic3_pp_cfg;

typedef struct {
  int32_t* loc;      /* [B, N+1, 2] (row, col); predators then prey (:158-159) */
  uint8_t* reached;  /* [B, N] reached_prey (:155,271) */
  uint8_t* done;     /* [B] episode_over (:154,273-274) */
  int32_t* success;  /* [B] stat['success'] (:284-288), -1 when unset */
  uint32_t* episode; /* [B] resets so far (tick of the spawn stream) */
  uint32_t* tick;    /* [B] env steps so far (tick of the action stream) */
} ic3_pp_state;

/* Trainer-side bookkeeping fused into the env step kernels when `r` is non-NULL:
 * the per-step tail of Trainer.get_episode (trainer.py:69-108) plus auto-reset,
 * so a batch of B independent env slots can run T lock-step iterations with no
 * host round trip.  All pointers are device pointers; rec_* may be NULL. */
typedef struct {
  int32_t t;               /* lock-step index into the rec_* arrays */
  int32_t max_steps;       /* args.max_steps (trainer.py:43,90) */
  int32_t nheads;          /* columns of `action` */
  int32_t hard_attn;       /* args.hard_attn && args.commnet (trainer.py:70) */
  int32_t comm_action_one; /* args.comm_action_one (trainer.py:71) */
  int32_t last;            /* 1 on the final lock-step of the batch: open episodes are cut (treated like max_steps) */
  const int32_t* action;   /* [B, N, nheads] sampled this step; env consumes head 0 (env_wrappers.py:76-77) */
  int32_t* t_ep;           /* [B] step index inside the current episode */
  uint8_t* fresh;          /* [B] out: next policy step starts an episode (h=c=0, nobody talks, all alive; trainer.py:45-51) */
  uint8_t* comm_next;      /* [B, N] out: info['comm_action'] for the next policy step (trainer.py:70-71) */
  uint8_t* alive_next;     /* [B, N] out: info['alive_mask'] for the next policy step (comm.py:102-104) */
  float* rec_reward;       /* [T, B, N] */
  uint8_t* rec_episode_mask; /* [T, B]  0 on the last step of an episode (trainer.py:92-96) */
  uint8_t* rec_mini_mask;  /* [T, B, N] 1 - is_completed on non-final steps (trainer.py:97-99) */
  uint8_t* rec_alive;      /* [T, B, N] misc['alive_mask'] (trainer.py:78-81) */
  float* stat_reward;      /* [B, N] += reward          (trainer.py:86) */
  float* stat_comm;        /* [B, N] += comm_next       (trainer.py:73) */
  int32_t* stat_success;   /* [B] += env.stat['success'] at episode end (trainer.py:124-125) */
  int32_t* stat_episodes;  /* [B] += 1 at episode end   (trainer.py:235) */
  int32_t* stat_steps;     /* [B] += 1 every step       (trainer.py:109) */
  /* Reference batch boundary (trainer.py:227-237: whole episodes until the worker holds >= batch_size steps, the
   * last episode overshoots).  batch_size > 0 with halted != NULL: a slot halts at the first episode end at which
   * stat_steps[slot] >= batch_size and is skipped by every later lock-step (null records).  With
   * T >= batch_size + max_steps - 1 lock-steps every slot halts by itself and `last` stays 0.  0 / NULL: off. */
  int32_t batch_size;
  int32_t reserved0;
  uint8_t* halted;         /* [B] in/out: slot has completed its batch */
  uint8_t* rec_valid;      /* [T, B] 1 = a real step of this slot, 0 = slot already halted (may be NULL) */
  /* Inputs of the NEXT policy step, recorded for Trainer.compute_grad (all optional; written at index t + 1 when
   * t + 1 < snap_T; index 0 is the caller's): what the policy will see as fresh / comm_action / alive_mask / step
   * index, and the environment state its observation is taken from. */
  int32_t snap_T;
  int32_t reserved1;
  uint8_t* snap_fresh;     /* [T, B] */
  uint8_t* snap_comm;      /* [T, B, N] */
  uint8_t* snap_alive;     /* [T, B, N] */
  int32_t* snap_tep;       /* [T, B] */
  int32_t* snap_pp_loc;    /* [T, B, N+1, 2]   predator_prey */
  int32_t* snap_tj_loc;    /* [T, B, N, 2]     traffic_junction ... */
  uint8_t* snap_tj_alive;  /* [T, B, N] */
  uint8_t* snap_tj_last_act; /* [T, B, N] */
  int32_t* snap_tj_route_id; /* [T, B, N] */
} ic3_rollout_io;

/* reset(): predator_prey_env.py:146-168.  Draws N+1 distinct cells per env from
 * the spawn stream (law of np.random.choice(dim*dim, N+1, replace=False), :174).
 * mask: [B] uint8 or NULL (= all).  obs: [B,N,O] float or NULL. */
int ic3_pp_reset(const ic3_pp_cfg* cfg, const ic3_pp_state* st, const uint8_t* mask,
                 float* obs, void* stream);
/* step(action): predator_prey_env.py:112-144 (+ _take_action :212-252, _get_reward
 * :254-290, _get_obs :188-210 when obs != NULL).  act: [B,N] int32 (stride
 * act_stride ints per agent, so a [B,N,heads] action tensor can be passed directly).
 * reward: [B,N] float.  err: device flag word. */
int ic3_pp_step(const ic3_pp_cfg* cfg, const ic3_pp_state* st, const int32_t* act, int32_t act_stride,
                float* reward, float* obs, int32_t* err, const ic3_rollout_io* r, void* stream);
/* _get_obs + env_wrappers._flatten_obs: predator_prey_env.py:188-210, env_wrappers.py:88-100.
 * obs: [B, N, W*W*V] float32, window-major then class. */
int ic3_pp_obs(const ic3_pp_cfg* cfg, const ic3_pp_state* st, float* obs, void* stream);

/* ------------------------------------------------------------------------
 * Traffic junction  (ic3net_envs/traffic_junction_env.py, traffic_helper.py)
 * ---------------------------------------------------------------------- */
typedef struct {
  int32_t B, N, vision;
  int32_t h, w;            /* dims (already +1 for easy, :112-115) */
  int32_t G, P, Lmax;      /* arrival groups, paths per group, longest path */
  int32_t outside_cls;     /* OUTSIDE_CLASS = BASE (:129) */
  int32_t car_cls;         /* CAR_CLASS = BASE + 2 (:130) */
  int32_t vocab;           /* vocab_size = BASE + 3 (:132) */
  int32_t npath;           /* nPr(nroad, 2) (:126) */
  uint32_t spawn_thr;      /* floor(add_rate * 2^24): u <= add_rate (:375) on 24-bit draws */
  uint32_t env_id0;
  uint64_t seed;
  const int32_t* grid;        /* [h, w] road ids / OUTSIDE (:300-316) */
  const int32_t* route_len;   /* [G, P] */
  const int32_t* route_cells; /* [G, P, Lmax] (row << 16 | col) (traffic_helper.py:156-209) */
} ic3_tj_cfg;

typedef struct {
  int32_t* loc;        /* [B, N, 2] car_loc; dead cars sit at (0,0) (:185,565) */
  uint8_t* alive;      /* [B, N] alive_mask */
  int32_t* wait;       /* [B, N] */
  int32_t* route_id;   /* [B, N] p + g*P, -1 before the first spawn (:177,385) */
  int32_t* route_pos;  /* [B, N] car_route_loc (:188) */
  uint8_t* last_act;   /* [B, N] car_last_act (:186), survives respawn */
  uint8_t* completed;  /* [B, N] is_completed of the last step (:233) */
  int32_t* cars_in_sys;/* [B] */
  uint8_t* has_failed; /* [B] sticky per episode (:171,592) */
  uint32_t* tick;      /* [B] env steps so far */
} ic3_tj_state;

/* reset(epoch): traffic_junction_env.py:160-204 (the curriculum, :196-200,620-626,
 * is host arithmetic that only changes cfg->spawn_thr). */
int ic3_tj_reset(const ic3_tj_cfg* cfg, const ic3_tj_state* st, const uint8_t* mask,
                 float* obs, void* stream);
/* step(action): traffic_junction_env.py:206-252 (_take_action :540-581, _add_cars
 * :369-393, _choose_dead :614-618, _get_reward :585-595).  draws: [B,G,3] 24-bit
 * ints (spawn test, dead slot, path) or NULL for the Philox spawn stream. */
int ic3_tj_step(const ic3_tj_cfg* cfg, const ic3_tj_state* st, const int32_t* act, int32_t act_stride,
                const uint32_t* draws, float* reward, float* obs, int32_t* err,
                const ic3_rollout_io* r, void* stream);
/* _get_obs + _flatten_obs: traffic_junction_env.py:321-366, env_wrappers.py:88-100.
 * obs: [B, N, 2 + W*W*V] float32. */
int ic3_tj_obs(const ic3_tj_cfg* cfg, const ic3_tj_state* st, float* obs, void* stream);

/* ------------------------------------------------------------------------
 * CommNet / IC3Net policy step  (comm.py:134-244, action_utils.py:27-36)
 * ---------------------------------------------------------------------- */
typedef struct {
  int32_t B, N, H, O;      /* envs, agents, hid_size (32|64|128), obs dim */
  int32_t nheads;          /* len(args.naction_heads) */
  int32_t head_dim[IC3_MAX_HEADS];
  int32_t hard_attn;       /* args.hard_attn (comm.py:171) */
  int32_t comm_avg;        /* args.comm_mode == 'avg' (comm.py:194) */
  int32_t comm_mask_zero;  /* args.comm_mask_zero (comm.py:39-43) */
  uint32_t env_id0;
  uint64_t seed;
  /* Observation layout hint for the encoder sum x = b + sum_f obs[f] * W_e[:, f] (comm.py:119).  With
   * obs_vocab = V > 0 the features f >= obs_off form cells of V entries whose first V - obs_ncount entries
   * are a one-hot position class and whose last obs_ncount entries are counts: every encoder (dense, index,
   * fused) then accumulates the class terms and the remaining terms separately,
   *   x = (b + sum_class ...) + (0 + sum_other ...),  each sum in increasing feature order,
   * so that the class part can come from a per-position table (ic3_*_encoder_table) and all forms stay
   * bit-identical.  predator_prey: (0, D*D+4, 2); traffic_junction: (2, vocab, 1).  obs_vocab = 0: one sum. */
  int32_t obs_off, obs_vocab, obs_ncount;
  /* Policy variants of comm.py / models.py (all zero = the recurrent LSTM CommNet / IC3Net with one comm pass):
   *   cell      IC3_CELL_LSTM: (h, c) = LSTMCell(x + C_i(S), (h, c))                       (comm.py:213-218)
   *             IC3_CELL_TANH: h = tanh(x + f_i(h) + C_i(S))                               (comm.py:220-224; models.py:25,
   *                            84 with comm_mask_zero: the MLP / RNN baselines)
   *   passes    comm passes per forward, 1..IC3_MAX_PASSES (comm.py:179), weights C_i / f_i per pass (share_weights:
   *             the same pointers)
   *   x_tanh    x = tanh(encoder(obs)) (non-recurrent branch, comm.py:127-128; models.py:24)
   *   h_from_x  the hidden state entering the first pass is x itself instead of io->h (comm.py:129)
   * Variants run on the fp32 SIMT kernel (the tcgen05 path implements the all-zero configuration). */
  int32_t cell, passes, x_tanh, h_from_x;
  int32_t reserved0;
} ic3_policy_cfg;

enum { IC3_CELL_LSTM = 0, IC3_CELL_TANH = 1 };
#define IC3_MAX_PASSES 4

/* Parameters in the reference state_dict layout (device, fp32). */
typedef struct {
  const float* encoder_w;  /* [H, O] */
  const float* encoder_b;  /* [H] */
  const float* c_w;        /* C_modules.0.weight [H, H] */
  const float* c_b;        /* [H] */
  const float* w_ih;       /* f_module.weight_ih [4H, H] gate order i,f,g,o */
  const float* w_hh;       /* f_module.weight_hh [4H, H] */
  const float* b_ih;       /* [4H] */
  const float* b_hh;       /* [4H] */
  const float* value_w;    /* value_head.weight [1, H] */
  const float* value_b;    /* [1] */
  const float* head_w[IC3_MAX_HEADS]; /* heads.k.weight [na_k, H] */
  const float* head_b[IC3_MAX_HEADS]; /* [na_k] */
  /* variants (ic3_policy_cfg.cell / passes); all NULL for the default configuration */
  const float* c_w_pass[IC3_MAX_PASSES]; /* C_modules.i.weight [H, H] for pass i >= 1 (index 0 unused: c_w) */
  const float* c_b_pass[IC3_MAX_PASSES];
  const float* f_w_pass[IC3_MAX_PASSES]; /* IC3_CELL_TANH: f_modules.i.weight [H, H], every pass */
  const float* f_b_pass[IC3_MAX_PASSES];
} ic3_policy_params;

/* Kernel-side layout, produced once per weight update by ic3_policy_pack. */
typedef struct {
  float* enc_wT;   /* [O, H]       encoder.weight^T: one contiguous H-row per obs feature */
  float* enc_b;    /* [H] */
  float* c_wT;     /* [H, H]       c_wT[k][n] = C.weight[n][k] */
  float* c_b;      /* [H] */
  float* lstm_wT;  /* [2H, 4H]     rows 0..H-1 <- w_ih^T, rows H..2H-1 <- w_hh^T; column 4*u+gate */
  float* lstm_b;   /* [4H]         b_ih + b_hh, column 4*u+gate */
  float* head_w;   /* [1+sum(na), H]  row 0 = value head, then heads in order */
  float* head_b;   /* [1+sum(na)] */
  /* tcgen05 path (H == 128 only; both NULL selects the fp32 SIMT kernel):
   * lstm_img: fp16 hi/lo split of 256 * [W_ih ; W_ih.C ; W_hh] (K = 384) as ready-made
   *   shared-memory images, [2 column halves][12 K-chunks][hi,lo][core-matrix layout] = 786432 bytes;
   * bias_cat: [4H] b_ih + b_hh + W_ih.c_b, column 4*u+gate.
   * comm_passes > 1 (LSTM cell only): `passes` such images / bias vectors one after the other, pass i folded
   *   with C_modules[i] (comm.py:63-70). */
  void* lstm_img;
  float* bias_cat;
  /* variants: c_wT / c_b hold `passes` consecutive [H, H] / [H] blocks; IC3_CELL_TANH: f_wT [passes][H, H]
   * (f_wT[i][k][n] = f_i.weight[n][k]) and f_b [passes][H]; NULL otherwise */
  float* f_wT;
  float* f_b;
  int32_t* flags;  /* device word written by ic3_policy_pack (IC3_ERR_FP16_RANGE when a folded weight does not fit the
                      operand split), OR-ed into ic3_policy_io.err by every policy step; may be NULL */
} ic3_policy_packed;

#define IC3_LSTM_IMG_BYTES 786432

int ic3_policy_pack(const ic3_policy_cfg* cfg, const ic3_policy_params* p,
                    const ic3_policy_packed* out, void* stream);

/* x = encoder(obs): comm.py:119.  Exact for any dense obs; cost scales with the
 * number of non-zeros per row (one-hot observations: ~1% dense). */
int ic3_encoder_dense(const ic3_policy_cfg* cfg, const ic3_policy_packed* w, const float* obs,
                      float* x, void* stream);
/* Same x computed straight from the env state (no [B,N,O] tensor is materialised). */
int ic3_pp_encoder_index(const ic3_pp_cfg* env, const ic3_pp_state* st, const ic3_policy_cfg* cfg,
                         const ic3_policy_packed* w, float* x, void* stream);
int ic3_tj_encoder_index(const ic3_tj_cfg* env, const ic3_tj_state* st, const ic3_policy_cfg* cfg,
                         const ic3_policy_packed* w, float* x, void* stream);
/* Class part of the encoder sum per agent position: table[(r*D + c)*H + n] = b[n] + sum over the window cells
 * (row-major) of W_e[n, cell*V + class(cell)] -- the one-hot grid of predator_prey_env.py:176-186 /
 * traffic_junction_env.py:300-319 depends on the position alone.  Rebuild after every weight update.
 * table: [dim*dim, H] (predator_prey) / [h*w, H] (traffic_junction) float32. */
int ic3_pp_encoder_table(const ic3_pp_cfg* env, const ic3_policy_cfg* cfg, const ic3_policy_packed* w,
                         float* table, void* stream);
int ic3_tj_encoder_table(const ic3_tj_cfg* env, const ic3_policy_cfg* cfg, const ic3_policy_packed* w,
                         float* table, void* stream);

typedef struct {
  const float* x;             /* [B*N, H] encoder output */
  const float* h;             /* [B*N, H] prev hidden  (comm.py:122) */
  const float* c;             /* [B*N, H] prev cell */
  const uint8_t* comm_action; /* [B, N] info['comm_action'] (required when hard_attn) */
  const uint8_t* alive;       /* [B, N] info['alive_mask'] or NULL = all alive (comm.py:102-107) */
  const uint8_t* fresh;       /* [B] or NULL; 1 = episode start: h=c=0, comm_action=0, alive=1 (trainer.py:45-51) */
  const uint32_t* tick;       /* [B] action-stream tick per env, or NULL = 0 */
  const uint32_t* draws;      /* [B, N, nheads] 24-bit draws, or NULL = Philox action stream */
  float* h_out;               /* [B*N, H] */
  float* c_out;               /* [B*N, H] */
  float* value;               /* [B*N]    value_head (comm.py:228) */
  float* logp;                /* [B, N, sum(na)] log_softmax per head, heads concatenated (comm.py:239) */
  int32_t* action;            /* [B, N, nheads] sampled actions or NULL (action_utils.py:32-36) */
  void* workspace;            /* tcgen05 path: ic3_policy_workspace_bytes(cfg) bytes of scratch (operand images), else NULL */
  int32_t* err;               /* tcgen05 path: device flag word (pipeline watchdog), may be NULL */
  /* tcgen05 path only: when x == NULL the encoder output is computed from the environment state inside the
   * policy step (fused index encoder, vision <= 2); exactly one pair must then be set (HOST pointers). */
  const ic3_pp_cfg* pp_env;
  const ic3_pp_state* pp_state;
  const ic3_tj_cfg* tj_env;
  const ic3_tj_state* tj_state;
  /* optional, fused index encoder only: [positions, H] table of ic3_pp_encoder_table / ic3_tj_encoder_table
   * for the CURRENT weights (device pointer); needs cfg->obs_vocab > 0. */
  const float* x_table;
  int32_t pass_index;         /* callers pass 0.  comm_passes > 1 on the tcgen05 path: the library runs the step once per
                                 pass on a private copy of this struct and numbers the copies here (a fresh episode's
                                 zero state applies to pass 0 only; its masks to every pass, comm.py:179-218) */
} ic3_policy_io;

/* Scratch the tcgen05 policy path needs for a batch of cfg->B environments (0 when unsupported). */
uint64_t ic3_policy_workspace_bytes(const ic3_policy_cfg* cfg);

/* One CommNetMLP.forward (recurrent branch, comm_passes = 1) + select_action. */
int ic3_policy_step(const ic3_policy_cfg* cfg, const ic3_policy_packed* w, const ic3_policy_io* io,
                    void* stream);
/* Measurement aid (bench.py "roofline_tensor"): ic3_policy_step on the tcgen05 path with CUDA events between its
 * kernels; synchronises the stream and returns ms[3] = device time of {operand preparation (+ fused encoder),
 * LSTM/comm tensor-core kernel, heads + sampling}.  Not for the production loop. */
int ic3_policy_step_profile(const ic3_policy_cfg* cfg, const ic3_policy_packed* w, const ic3_policy_io* io,
                            void* stream, float* ms);
/* select_action alone (action_utils.py:32-36) on given log-probabilities. */
int ic3_sample_actions(const ic3_policy_cfg* cfg, const float* logp, const uint32_t* tick,
                       const uint32_t* draws, int32_t* action, void* stream);

/* ------------------------------------------------------------------------
 * REINFORCE returns  (trainer.py:160-173), the first step of Trainer.compute_grad
 * ---------------------------------------------------------------------- */
/* reward, mini_mask: [T,B,N]; episode_mask: [T,B]; returns out: [T,B,N] float32 (float64 accumulation). */
int ic3_returns_scan(int32_t T, int32_t B, int32_t N, float gamma, float mean_ratio, const float* reward,
                     const uint8_t* episode_mask, const uint8_t* mini_mask, float* returns, void* stream);

/* Batch statistics of Trainer.run_batch (trainer.py:73-75,86-88,109-110,124-125,235; merged over workers by
 * multi_processing.py:86-88): the per-slot accumulators of ic3_rollout_io summed over the B env slots of this GPU
 * into one float64 device vector  out[4 + 2N] = [num_episodes, num_steps, success, err flag word, reward[N],
 * comm_action[N]]  (stat_comm may be NULL: zeros).  One device->host copy per update instead of one per key; the
 * data-parallel trainer all-reduces the vector before reading it. */
int ic3_stat_reduce(int32_t B, int32_t N, const int32_t* stat_episodes, const int32_t* stat_steps,
                    const int32_t* stat_success, const int32_t* err, const float* stat_reward,
                    const float* stat_comm, double* out, void* stream);

/* ------------------------------------------------------------------------
 * Back-propagation through time of the rollout loss (Trainer.compute_grad, trainer.py:128-225;
 * utils.multinomials_log_density utils.py:42-46) over the records of a lock-step rollout, hid_size 128,
 * at most 7 action logits.  The host walks the lock-step iterations t = T-1 .. 0:
 *     ic3_bptt_begin(plan, max |c| of the record, stream)
 *     for t in reversed(range(T)): ic3_bptt_step(plan, &io_t, stream)
 *     ic3_bptt_finish(plan, params, grads, losses, stream)
 * Per step: d loss / d (value, logits) from the recorded log-probs / actions / advantages / masks, LSTM cell and
 * comm backward, and the three GEMMs (gate re-computation, d gates . W, (d gates)^T . features) on the tensor cores
 * with the forward's fp16 hi/lo operand split.  Parameter gradients are ADDED to the `grads` buffers (the caller
 * zeroes them, trainer.py:248) and are not divided by num_steps (trainer.py:251-253 does that).
 * ---------------------------------------------------------------------- */
typedef struct {
  const ic3_policy_cfg* cfg;    /* HOST pointers: same structs the rollout used */
  const ic3_policy_packed* w;
  const ic3_pp_cfg* pp_env;     /* exactly one of pp_env / tj_env */
  const ic3_tj_cfg* tj_env;
  const float* x_table;         /* device: ic3_*_encoder_table of the CURRENT weights (required) */
  float value_coeff;            /* args.value_coeff (trainer.py:209) */
  float entr;                   /* args.entr (trainer.py:211-220) */
  void* workspace;              /* device scratch of ic3_bptt_workspace_bytes(plan) bytes */
} ic3_bptt_plan;

typedef struct {
  int32_t t;                    /* lock-step index (its parity selects the operand-image set of the step) */
  int32_t reserved0;
  /* state entering / leaving policy step t */
  const float* h_prev;          /* [B*N, H] h_{t-1} as fed to the step (ignored for fresh slots) */
  const float* c_prev;          /* [B*N, H] */
  const float* h_new;           /* [B*N, H] h'_t */
  /* inputs of policy step t as recorded */
  const uint8_t* fresh;         /* [B] */
  const uint8_t* comm;          /* [B, N] info['comm_action'] (required with hard_attn) */
  const uint8_t* alive;         /* [B, N] info['alive_mask'] or NULL */
  const uint8_t* cut;           /* [B] or NULL: (h', c') of step t were detached, (t_ep + 1) % detach_gap == 0 (trainer.py:56-60) */
  /* environment state the observation of step t was taken from */
  const int32_t* pp_loc;        /* [B, N+1, 2] */
  const int32_t* tj_loc;        /* [B, N, 2] */
  const uint8_t* tj_alive;      /* [B, N] */
  const uint8_t* tj_last_act;   /* [B, N] */
  const int32_t* tj_route_id;   /* [B, N] */
  /* outputs of step t and their learning signals */
  const float* logp;            /* [B*N, sum(na)] */
  const int32_t* action;        /* [B*N, nheads] */
  const float* value;           /* [B*N] */
  const float* ret;             /* [B*N] returns (ic3_returns_scan) */
  const float* adv;             /* [B*N] advantages (returns - value, optionally normalised, trainer.py:176-180) */
  const uint8_t* alive_post;    /* [B*N] misc['alive_mask'] of the step (trainer.py:186-190) */
  const uint8_t* valid;         /* [B] or NULL: 0 = slot had already completed its batch (ic3_rollout_io.rec_valid) */
  /* recursion: in = d loss / d (h'_t, c'_t) from later steps, out = d loss / d (h_{t-1}, c_{t-1}) */
  float* dh;                    /* [B*N, H] */
  float* dc;                    /* [B*N, H] */
  int32_t* err;                 /* device flag word (IC3_ERR_PIPELINE / IC3_ERR_FP16_RANGE), may be NULL */
} ic3_bptt_step_io;

uint64_t ic3_bptt_workspace_bytes(const ic3_bptt_plan* plan);   /* 0 = configuration not supported by the kernels */
int ic3_bptt_begin(const ic3_bptt_plan* plan, float c_abs_max, void* stream);
int ic3_bptt_step(const ic3_bptt_plan* plan, const ic3_bptt_step_io* io, void* stream);
/* Optional look-ahead: launches the recursion-independent kernels of step io->t (heads gradient, operand images) on the
 * library's side stream so that they overlap the tensor-core kernels of step t + 1; call it for step t - 1 right before
 * ic3_bptt_step(t) (and once for t = T - 1 after ic3_bptt_begin).  The step's records must not change until
 * ic3_bptt_step(io->t) has been issued. */
int ic3_bptt_prepare(const ic3_bptt_plan* plan, const ic3_bptt_step_io* io, void* stream);
/* params: the CURRENT parameters; grads: same struct holding the gradient buffers (reference layouts);
 * losses: device double[3] = action_loss, value_loss, entropy sums (trainer.py:198-216). */
int ic3_bptt_finish(const ic3_bptt_plan* plan, const ic3_policy_params* params, const ic3_policy_params* grads,
                    double* losses, void* stream);

/* ------------------------------------------------------------------------
 * Optimizer step  (trainer.py:21-22 RMSprop(lr, alpha=0.97, eps=1e-6); trainer.py:251-256 and
 * multi_processing.py:95-97: summed gradient / global num_steps, then one step)
 * ---------------------------------------------------------------------- */
/* All live parameters, their gradients and the RMSprop second-moment state as three flat,
 * 16-byte aligned float32 buffers of n elements:  g = grad / grad_div (stored back into grad);
 * square_avg = alpha*square_avg + (1-alpha)*g*g;  param -= lr * g / (sqrt(square_avg) + eps). */
int ic3_rmsprop_step(int64_t n, float lr, float alpha, float eps, float grad_div, float* grad,
                     float* param, float* square_avg, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IC3NET_B200_H */
