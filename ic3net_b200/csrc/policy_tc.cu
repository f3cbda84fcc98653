// CommNet / IC3Net policy step on the 5th-generation tensor cores ("policy v2", H = 128).
//
// Math.  With S the gated hidden-state mean (comm.py:181-205), the LSTM pre-activations of
// comm.py:206-218 are ONE contraction over K = 384:
//   gates = W_ih (x + C S + c_b) + W_hh h + b_ih + b_hh
//         = [x | S | h] . [W_ih ; W_ih C ; W_hh]^T + (b_ih + b_hh + W_ih c_b)
// (W_ih C is formed once per weight update in float64.)  fp32 accuracy on fp16 tensor cores:
// a * 16 = a_hi + a_lo and w * 256 = w_hi + w_lo with fp16 halves (11 significant bits each,
// power-of-two pre-scaling keeps both halves in the fp16 normal range for |a| < 4094, |w| < 255);
//   D = a_hi w_hi + a_lo w_hi + a_hi w_lo   (3 tcgen05.mma kind::f16, fp32 accumulate in TMEM)
// drops only a_lo w_lo (2^-22 relative) and gates = D * 2^-12 + bias.
//
// Data movement.  Both operands are stored in global memory as ready-made shared-memory
// images in the no-swizzle K-major core-matrix layout (8 rows x 16 bytes per core matrix),
// so a stage of the pipeline is two plain cp.async.bulk copies (A: 16 KB, B: 32 KB) that
// complete on an mbarrier, and the MMA descriptors are fixed offsets into the stage:
//   prep kernel   x, h (fp32), gate masks  ->  A image [tile][12 chunks][hi,lo][4 kcore][16 rcore][8][8]
//   pack kernel   weights                  ->  B image [2 halves][12 chunks][hi,lo][4 kcore][32 ncore][8][8]
//   lstm kernel   persistent, one CTA per SM looping over work items (128-row tile, 256-column half):
//                 warp 16 = bulk-copy producer (4-stage ring) + TMEM allocator, warp 17 = MMA issuer
//                 (one thread) into two 256-column TMEM accumulators, warps 0-15 = epilogue
//                 (tcgen05.ld -> LSTM cell -> c', h' + partial head logits) of item i while the
//                 MMAs of item i+1 run.
//   heads kernel  value / action heads + sampling: heads_finish_kernel sums the epilogue's partial
//                 logits (thread per row, <= 7 action logits); heads_kernel<P> otherwise.
#include "policy_tc_kernels.cuh"


// Persistent grid: as many CTAs as can be co-resident (one per SM: 148 on B200), each looping over work items.
static int launch_lstm(const ic3_policy_cfg* cfg, const ic3_policy_io* io, const ic3_policy_packed* w, const __half* a_img,
                       int ntiles, size_t smem, int nout, float* partial, cudaStream_t s) {
  static int max_ctas = 0;
  if (max_ctas == 0) {
    cudaError_t e = cudaFuncSetAttribute(lstm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    int dev = 0, nsm = 0, per_sm = 0;
    e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lstm_tc_kernel, TC_P_THREADS, smem);
    if (e != cudaSuccess) return (int)e;
    if (per_sm <= 0) return IC3_E_RANGE;
    max_ctas = nsm * per_sm;
  }
  const int nitems = 2 * ntiles;                                   // (row tile, column half)
  const int grid = nitems < max_ctas ? nitems : max_ctas;
  const __half* b_img = reinterpret_cast<const __half*>(w->lstm_img) + (size_t)io->pass_index * B_IMG_HALFS;
  lstm_tc_kernel<<<grid, TC_P_THREADS, smem, s>>>(*cfg, *io, a_img, b_img, w->bias_cat + (size_t)io->pass_index * 4 * TC_H,
                                                  nitems, w->head_w, nout, partial);
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}

uint64_t ic3_tc_workspace_bytes(const ic3_policy_cfg* cfg) {
  if (!cfg || cfg->H != TC_H) return 0;
  const long R = (long)cfg->B * cfg->N;
  const long ntiles = (R + TC_M - 1) / TC_M;
  // operand image + per-slot partial logits [R][NSLOT][HEAD_PAD] (+ comm_passes > 1: two (h, c) pairs that carry the
  // state from one pass to the next)
  const uint64_t carry = cfg->passes > 1 ? (uint64_t)4 * R * TC_H * sizeof(float) : 0;
  return (uint64_t)ntiles * TC_NCHUNK * A_CHUNK_BYTES + (uint64_t)R * NSLOT * HEAD_PAD * sizeof(float) + carry;
}

int ic3_tc_pack(const ic3_policy_cfg* cfg, const ic3_policy_params* p, const ic3_policy_packed* out, cudaStream_t s) {
  if (cfg->H != TC_H) return IC3_E_UNSUPPORTED;
  const int total = 4 * TC_H * TC_K;
  if (out->flags) {
    cudaError_t e = cudaMemsetAsync(out->flags, 0, sizeof(int32_t), s);
    if (e != cudaSuccess) return (int)e;
  }
  const int P = cfg->passes > 1 ? cfg->passes : 1;
  for (int ps = 0; ps < P; ++ps) {           // pass i folds C_modules[i] (comm.py:63-70; share_weights: the same module)
    ic3_policy_params q = *p;
    if (ps > 0 && p->c_w_pass[ps]) q.c_w = p->c_w_pass[ps];
    if (ps > 0 && p->c_b_pass[ps]) q.c_b = p->c_b_pass[ps];
    pack_tc_kernel<<<(total + 255) / 256, 256, 0, s>>>(q, reinterpret_cast<__half*>(out->lstm_img) + (size_t)ps * B_IMG_HALFS,
                                                       out->bias_cat + (size_t)ps * 4 * TC_H, out->flags);
    IC3_LAUNCH_CHECK();
  }
  return IC3_OK;
}

// Per-kernel timing hook (ic3_policy_step_profile): when set, events are recorded on the stream before the first
// kernel of the step and after each of its kernels.  Host-side only; nullptr in normal operation.
static cudaEvent_t* g_prof_ev = nullptr;
static inline void prof_mark(int i, cudaStream_t s) {
  if (g_prof_ev) cudaEventRecord(g_prof_ev[i], s);
}

extern "C" int ic3_policy_step_profile(const ic3_policy_cfg* cfg, const ic3_policy_packed* w, const ic3_policy_io* io,
                                       void* stream, float* ms) {
  static cudaEvent_t ev[4];
  static bool made = false;
  if (!ms) return IC3_E_NULL;
  if (!made) {
    for (int i = 0; i < 4; ++i) {
      cudaError_t e = cudaEventCreate(&ev[i]);
      if (e != cudaSuccess) return (int)e;
    }
    made = true;
  }
  g_prof_ev = ev;
  const int rc = ic3_policy_step(cfg, w, io, stream);
  g_prof_ev = nullptr;
  if (rc) return rc;
  cudaError_t e = cudaEventSynchronize(ev[3]);
  if (e != cudaSuccess) return (int)e;
  for (int i = 0; i < 3; ++i) {
    e = cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]);
    if (e != cudaSuccess) return (int)e;
  }
  return IC3_OK;
}

static int tc_pass(const ic3_policy_cfg* cfg, const ic3_policy_packed* w, const ic3_policy_io* io, cudaStream_t s, bool last);

// comm.py:179-218: `passes` rounds of (communicate, LSTM cell) on the same encoded observation.  Pass i reads the
// state pass i-1 wrote (two carry buffers behind the workspace, alternating) and uses weight image i; only the last
// pass writes the caller's h_out / c_out and finishes the heads.
int ic3_tc_policy_step(const ic3_policy_cfg* cfg, const ic3_policy_packed* w, const ic3_policy_io* io, cudaStream_t s) {
  if (cfg->H != TC_H) return IC3_E_UNSUPPORTED;
  if (!io->workspace || !w->lstm_img || !w->bias_cat) return IC3_E_NULL;
  const int P = cfg->passes > 1 ? cfg->passes : 1;
  if (P == 1) return tc_pass(cfg, w, io, s, true);
  const long R = (long)cfg->B * cfg->N;
  ic3_policy_cfg c1 = *cfg;
  c1.passes = 1;
  float* carry = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(io->workspace) + ic3_tc_workspace_bytes(&c1));
  const size_t RH = (size_t)R * TC_H;
  for (int ps = 0; ps < P; ++ps) {
    ic3_policy_io q = *io;
    q.pass_index = ps;
    if (ps > 0) {
      q.h = carry + (size_t)((ps - 1) & 1) * 2 * RH;
      q.c = q.h + RH;
    }
    if (ps < P - 1) {
      q.h_out = carry + (size_t)(ps & 1) * 2 * RH;
      q.c_out = q.h_out + RH;
    }
    const int rc = tc_pass(cfg, w, &q, s, ps == P - 1);
    if (rc) return rc;
  }
  return IC3_OK;
}

static int tc_pass(const ic3_policy_cfg* cfg, const ic3_policy_packed* w, const ic3_policy_io* io, cudaStream_t s, bool last) {
  const long R = (long)cfg->B * cfg->N;
  const int ntiles = (int)((R + TC_M - 1) / TC_M);
  __half* img = reinterpret_cast<__half*>(io->workspace);
  PrepSrc src;
  memset(&src, 0, sizeof(src));
  src.wT = w->enc_wT;
  src.bias = w->enc_b;
  src.split = cfg->obs_vocab > 0;
  src.table = io->x_table;
  src.wflags = w->flags;
  if (src.table && !src.split) return IC3_E_RANGE;      // the table IS the first of the two sums
  prof_mark(0, s);
  if (io->x) {
    prep_kernel<XSRC_TENSOR, false><<<2 * ntiles, PREP_THREADS, prep_T_bytes(cfg->N), s>>>(*cfg, *io, img, src, PrepBwd{});
  } else if (io->pp_env && io->pp_state) {       // fused index encoder, predator-prey
    const int W = 2 * io->pp_env->vision + 1;
    if (W * W > PREP_MAX_WW || io->pp_env->B != cfg->B || ic3_pp_agents(*io->pp_env) != cfg->N) return IC3_E_RANGE;
    if (cfg->O != W * W * (io->pp_env->dim * io->pp_env->dim + 4)) return IC3_E_RANGE;
    src.pp = *io->pp_env;
    src.pps = *io->pp_state;
    if (int lrc = ic3_pp_layout_check(io->pp_env, cfg)) return lrc;
    if (src.table) {
      prep_kernel<XSRC_PP, true><<<2 * ntiles, PREP_THREADS, prep_T_bytes(cfg->N), s>>>(*cfg, *io, img, src, PrepBwd{});
    } else {
      static bool cfgd = false;
      if (!cfgd) {
        cudaError_t e = cudaFuncSetAttribute(prep_kernel<XSRC_PP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PREP_X_BYTES + (PREP_ROWS + 2) * TC_H * 4);
        if (e != cudaSuccess) return (int)e;
        cfgd = true;
      }
      prep_kernel<XSRC_PP, false><<<2 * ntiles, 256, PREP_X_BYTES + prep_T_bytes(cfg->N), s>>>(*cfg, *io, img, src, PrepBwd{});
    }
  } else if (io->tj_env && io->tj_state) {       // fused index encoder, traffic junction
    const int W = 2 * io->tj_env->vision + 1;
    if (W * W > PREP_MAX_WW || io->tj_env->B != cfg->B || io->tj_env->N != cfg->N) return IC3_E_RANGE;
    if (cfg->O != 2 + W * W * io->tj_env->vocab) return IC3_E_RANGE;
    src.tj = *io->tj_env;
    src.tjs = *io->tj_state;
    if (int lrc = ic3_tj_layout_check(io->tj_env, cfg)) return lrc;
    if (src.table) {
      prep_kernel<XSRC_TJ, true><<<2 * ntiles, PREP_THREADS, prep_T_bytes(cfg->N), s>>>(*cfg, *io, img, src, PrepBwd{});
    } else {
      static bool cfgd = false;
      if (!cfgd) {
        cudaError_t e = cudaFuncSetAttribute(prep_kernel<XSRC_TJ, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PREP_X_BYTES + (PREP_ROWS + 2) * TC_H * 4);
        if (e != cudaSuccess) return (int)e;
        cfgd = true;
      }
      prep_kernel<XSRC_TJ, false><<<2 * ntiles, 256, PREP_X_BYTES + prep_T_bytes(cfg->N), s>>>(*cfg, *io, img, src, PrepBwd{});
    }
  } else {
    return IC3_E_NULL;
  }
  IC3_LAUNCH_CHECK();
  prof_mark(1, s);
  const size_t smem = NSTAGE_P * STAGE_BYTES + 256 + TC_H * HEAD_PAD * sizeof(float) + 4 * TC_H * sizeof(float);
  int nout = 1;
  for (int k = 0; k < cfg->nheads; ++k) nout += cfg->head_dim[k];
  const bool fused_heads = nout <= HEAD_PAD;
  float* partial = fused_heads ? reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(io->workspace) +
                                                           (size_t)ntiles * TC_NCHUNK * A_CHUNK_BYTES)
                               : nullptr;
  const int rc = launch_lstm(cfg, io, w, img, ntiles, smem, nout, partial, s);
  if (rc) return rc;
  prof_mark(2, s);
  if (!last) return IC3_OK;                  // heads after the last comm pass only
  if (fused_heads) {
    heads_finish_kernel<<<(unsigned)((R + 127) / 128), 128, 0, s>>>(*cfg, *w, *io, partial);
    IC3_LAUNCH_CHECK();
    prof_mark(3, s);
    return IC3_OK;
  }
  const int P = nout <= 8 ? 8 : (nout <= 16 ? 16 : 32);
  const long rows_per_block = 8L * (32 / P);
  const int hgrid = (int)((R + rows_per_block - 1) / rows_per_block);
  if (P == 8) heads_kernel<8><<<hgrid, 256, 0, s>>>(*cfg, *w, *io);
  else if (P == 16) heads_kernel<16><<<hgrid, 256, 0, s>>>(*cfg, *w, *io);
  else heads_kernel<32><<<hgrid, 256, 0, s>>>(*cfg, *w, *io);
  IC3_LAUNCH_CHECK();
  prof_mark(3, s);
  return IC3_OK;
}
