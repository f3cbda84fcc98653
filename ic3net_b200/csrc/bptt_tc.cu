// Back-propagation through time of the rollout loss (Trainer.compute_grad, reference trainer.py:128-225) as
// hand-written sm_100a kernels (H = 128).  One call of ic3_bptt_step differentiates ONE lock-step iteration t of
// the recorded rollout for all env slots; the host walks t = T-1 .. 0.  Per step:
//
//   heads      d(loss)/d(value, logits) from the records (advantages, log-probs, actions, masks), the value /
//              action-head weight gradients, the three loss sums                               [bptt_heads_kernel]
//   scale      power-of-two scale of this step's gate gradients for the fp16 hi/lo operand split [bptt_scale_kernel]
//   prep       [x | S | h_{t-1}] operand image (the forward's own kernel, fed from the records) + the sparse
//              observation pattern P + the comm gate factors                                    [prep_kernel<.., BWD>]
//   gates      tcgen05: gate pre-activations re-computed exactly like the forward (K = 384), LSTM cell backward in
//              the epilogue -> d gates (fp16 hi/lo image), d c_{t-1}                            [bptt_gates_kernel]
//   dgrad      tcgen05: [dS | dh] = d gates . [W_ih C | W_hh]   (K = 512, N = 256)              [bptt_dgrad_kernel]
//   comm       backward of the gated hidden-state mean + episode-start / detach cuts -> d h_{t-1} [bptt_comm_kernel]
//   wgrad      tcgen05: G += (d gates)^T . [x | S | h | P]  -- both operands MN-major views of the images the other
//              kernels already wrote, contraction over the agent rows; per-CTA accumulators     [bptt_wgrad_kernel]
//
// After the last step ic3_bptt_finish folds G into the parameter gradients (float64):
//   dW_hh = G_h,  dW_ih = G_x + G_S C^T + g1 c_b^T,  db_ih = db_hh = g1,  dC = W_ih^T G_S,  dc_b = W_ih^T g1,
//   d encoder = W_ih^T (d gates)^T P scattered back through the observation layout (one-hot class per window cell
//   of the agent position, count / scalar features), with g1 = column of ones of P.
//
// Arithmetic of the three GEMMs: the forward's fp16 hi/lo split (3 MMAs, fp32 accumulate).  d gates of a step are
// scaled by a power of two s_t chosen from an upper bound of their magnitude (so hi stays below 2^14 and lo keeps
// 2^-35 of the step's largest element); products are unscaled when they leave the tensor memory.
#include <cuda.h>

#include "policy_tc_kernels.cuh"

namespace {

constexpr int BP_HEADS = HEAD_PAD;                 // value + action logits handled by the fused heads backward (<= 8)
constexpr int DG_TILE_HALFS = 2 * 64 * 16 * 64;    // d gates image per tile: [hi, lo][cg 64][rg 16][8][8]
constexpr int DG_PART_HALFS = 64 * 16 * 64;
constexpr int WG_MAX_NP = 512;                     // columns of P the weight-gradient kernel can hold in tensor memory

struct BpttScalars {      // device-resident scalars of the recursion
  unsigned dhmax;         // bits of max |dh| entering the next step to be processed (atomicMax on non-negative floats)
  unsigned dcmax;
  unsigned hbound[2];     // bound of the heads' contribution to |dh| of step t, slot t & 1 (heads of step t - 1 run early)
  float cmax;             // max |c| over the whole record (set by the host once per compute_grad)
  float scale[2];         // s_t, indexed by t & 1: the weight-gradient kernel of step t runs on a side stream while
  float inv_scale[2];     // 1 / s_t          the main stream already prepares step t - 1
};

// ------------------------------------------------------------------------------------------------------------------
// heads: d loss / d outputs of step t  (trainer.py:176-220, utils.py:42-46)
// ------------------------------------------------------------------------------------------------------------------
struct HeadsArgs {
  int R, N, nheads, atot;
  int head_dim[IC3_MAX_HEADS];
  float value_coeff, entr;
  const float* logp;          // [R, atot]
  const int32_t* action;      // [R, nheads]
  const float* value;         // [R]
  const float* ret;           // [R]
  const float* adv;           // [R]
  const uint8_t* alive_post;  // [R]
  const uint8_t* valid;       // [B] or NULL
  const float* h_new;         // [R, H] h'_t
  const float* head_w;        // packed [1 + atot, H]
  float* dout;                // [R, 8]
  float* gw_part;             // [nblocks][8][H]  per-block partial sums of d head weights (block-private, += every step)
  double* gs_part;            // [nblocks][8 + 3] per-block: d head biases (8), action_loss, value_loss, entropy
  BpttScalars* sc;
  int q;                      // t & 1
};

constexpr int HB_ROWS = 256;   // rows per block of the heads kernel

// <= 36 registers: one CTA of this kernel fits beside a resident bptt_gates_kernel CTA (576 threads x 96 registers), so it
// overlaps the tensor-core kernels of the previous step when launched ahead on the side stream (ic3_bptt_prepare)
__global__ void __launch_bounds__(256, 7) bptt_heads_kernel(HeadsArgs a) {
  __shared__ __align__(16) float s_dout[HB_ROWS][BP_HEADS];
  __shared__ float s_wmax[BP_HEADS];
  __shared__ double s_red[8][BP_HEADS + 3];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int row = blockIdx.x * HB_ROWS + tid;
  const int nout = 1 + a.atot;
  if (tid < BP_HEADS) {
    float m = 0.f;
    if (tid < nout)
      for (int k = 0; k < TC_H; ++k) m = fmaxf(m, fabsf(__ldg(a.head_w + (size_t)tid * TC_H + k)));
    s_wmax[tid] = m;
  }
  float d[BP_HEADS];
#pragma unroll
  for (int o = 0; o < BP_HEADS; ++o) d[o] = 0.f;
  double al = 0.0, vl = 0.0, en = 0.0;
  if (row < a.R) {
    const float alive = a.alive_post[row] ? 1.f : 0.f;
    const float vmask = (a.valid == nullptr || a.valid[row / a.N]) ? 1.f : 0.f;
    const float value = a.value[row], ret = a.ret[row], adv = a.adv[row];
    d[0] = 2.f * a.value_coeff * alive * (value - ret);                       // trainer.py:205-208
    vl = (double)((value - ret) * (value - ret) * alive);
    float lp_taken = 0.f;
    int off = 0;
    for (int m = 0; m < a.nheads; ++m) {
      const int na = a.head_dim[m];
      const int act = a.action[(size_t)row * a.nheads + m];
      float Hm = 0.f;
      for (int j = 0; j < na; ++j) {
        const float lp = a.logp[(size_t)row * a.atot + off + j];
        Hm -= lp * __expf(lp);
      }
      en += (double)(Hm * vmask);                                             // trainer.py:211-216 (not alive-masked)
      for (int j = 0; j < na; ++j) {
        const float lp = a.logp[(size_t)row * a.atot + off + j];
        const float pj = __expf(lp);
        float g = (-adv * alive) * ((j == act ? 1.f : 0.f) - pj);             // d(-A logp[act]) / d logit_j
        if (a.entr > 0.f) g += a.entr * pj * (lp + Hm) * vmask;               // d(-entr * H) / d logit_j
        if (1 + off + j < BP_HEADS) d[1 + off + j] = g;
        if (j == act) lp_taken += lp;
      }
      off += na;
    }
    al = (double)(-adv * lp_taken * alive);                                   // trainer.py:198-201
    *reinterpret_cast<float4*>(a.dout + (size_t)row * BP_HEADS) = make_float4(d[0], d[1], d[2], d[3]);
    *reinterpret_cast<float4*>(a.dout + (size_t)row * BP_HEADS + 4) = make_float4(d[4], d[5], d[6], d[7]);
  }
#pragma unroll
  for (int o = 0; o < BP_HEADS; ++o) s_dout[tid][o] = d[o];
  __syncthreads();
  // bound of the heads' contribution to |dh| of a row: sum_o |dout_o| max_u |W[o][u]|
  float hb = 0.f;
#pragma unroll
  for (int o = 0; o < BP_HEADS; ++o) hb += fabsf(d[o]) * s_wmax[o];
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) hb = fmaxf(hb, __shfl_xor_sync(IC3_FULL_MASK, hb, s));
  if (lane == 0 && hb > 0.f) atomicMax(&a.sc->hbound[a.q], __float_as_uint(hb));
  // block sums: bias gradients + losses (double)
  double v[BP_HEADS + 3];
#pragma unroll
  for (int o = 0; o < BP_HEADS; ++o) v[o] = (double)d[o];
  v[BP_HEADS] = al; v[BP_HEADS + 1] = vl; v[BP_HEADS + 2] = en;
#pragma unroll
  for (int o = 0; o < BP_HEADS + 3; ++o) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) v[o] += __shfl_xor_sync(IC3_FULL_MASK, v[o], s);
    if (lane == 0) s_red[warp][o] = v[o];
  }
  __syncthreads();
  if (tid < BP_HEADS + 3) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += s_red[w][tid];
    a.gs_part[(size_t)blockIdx.x * (BP_HEADS + 3) + tid] += t;
  }
  // head weight gradients: thread = (hidden unit u, half of the block's rows); fixed summation order
  const int u = tid & (TC_H - 1), half = tid >> 7;
  float acc[BP_HEADS];
#pragma unroll
  for (int o = 0; o < BP_HEADS; ++o) acc[o] = 0.f;
  const int r0 = blockIdx.x * HB_ROWS + half * (HB_ROWS / 2);
  const int nr = min(HB_ROWS / 2, a.R - r0);                 // rows of this half that exist (<= 0: none)
  const float* hp = a.h_new + (size_t)r0 * TC_H + u;
  int r = 0;
  for (; r + 8 <= nr; r += 8) {                               // 8 independent loads in flight per thread
    float hv[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) hv[q] = __ldg(hp + (size_t)(r + q) * TC_H);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 d0 = *reinterpret_cast<const float4*>(&s_dout[half * (HB_ROWS / 2) + r + q][0]);
      const float4 d1 = *reinterpret_cast<const float4*>(&s_dout[half * (HB_ROWS / 2) + r + q][4]);
      acc[0] = fmaf(d0.x, hv[q], acc[0]); acc[1] = fmaf(d0.y, hv[q], acc[1]);
      acc[2] = fmaf(d0.z, hv[q], acc[2]); acc[3] = fmaf(d0.w, hv[q], acc[3]);
      acc[4] = fmaf(d1.x, hv[q], acc[4]); acc[5] = fmaf(d1.y, hv[q], acc[5]);
      acc[6] = fmaf(d1.z, hv[q], acc[6]); acc[7] = fmaf(d1.w, hv[q], acc[7]);
    }
  }
  for (; r < nr; ++r) {
    const float hv = __ldg(hp + (size_t)r * TC_H);
    const float* dr = s_dout[half * (HB_ROWS / 2) + r];
#pragma unroll
    for (int o = 0; o < BP_HEADS; ++o) acc[o] = fmaf(dr[o], hv, acc[o]);
  }
  __shared__ float s_acc[BP_HEADS][TC_H];
  if (half == 1) {
#pragma unroll
    for (int o = 0; o < BP_HEADS; ++o) s_acc[o][u] = acc[o];
  }
  __syncthreads();
  if (half == 0) {
    float* gp = a.gw_part + (size_t)blockIdx.x * BP_HEADS * TC_H;
#pragma unroll
    for (int o = 0; o < BP_HEADS; ++o) gp[o * TC_H + u] += acc[o] + s_acc[o][u];
  }
}

// s_t = 2^e with  bound * s_t in (2^13, 2^14]:  |d gate| <= (|dc| + |dh|) * max(1, |c_prev| / 4)
__global__ void bptt_scale_kernel(BpttScalars* sc, int q) {
  const float dh = __uint_as_float(sc->dhmax) + __uint_as_float(sc->hbound[q]);
  const float dc = __uint_as_float(sc->dcmax);
  const float bound = (dh + dc) * fmaxf(1.f, 0.25f * sc->cmax);
  float s = 1.f;
  if (bound > 0.f && isfinite(bound)) {
    int e;
    frexpf(bound, &e);                       // bound = m * 2^e, m in [0.5, 1)
    e = 14 - e;
    e = e > 100 ? 100 : (e < -100 ? -100 : e);
    s = ldexpf(1.f, e);
  }
  sc->scale[q] = s;
  sc->inv_scale[q] = 1.f / s;
  sc->dhmax = 0u;
  sc->dcmax = 0u;
  sc->hbound[q] = 0u;
}

// ------------------------------------------------------------------------------------------------------------------
// gates: forward gate GEMM re-computed + LSTM cell backward in the epilogue
// ------------------------------------------------------------------------------------------------------------------
struct GatesArgs {
  int R, N;
  const float* c_prev;      // [R, H] c_{t-1}
  const uint8_t* fresh;     // [B] step t starts an episode: h_{t-1} = c_{t-1} = 0 and nothing flows further back
  const uint8_t* cut;       // [B] or NULL: (h', c') of step t were detached (trainer.py:56-60): incoming dh, dc are dropped
  const float* dout;        // [R, 8]
  float* dh;                // [R, H] in: d loss / d h'_t from later steps
  float* dc;                // [R, H] in: d loss / d c'_t;  out: d loss / d c_{t-1}
  __half* dg_img;           // d gates image
  BpttScalars* sc;
  int q;                    // t & 1
  int32_t* err;
};

// sigmoid / tanh of the four gates of a hidden unit with the forward's arithmetic (lstm_cell4): same SFU
// approximations, so the re-computed activations are the ones the rollout used.
__device__ __forceinline__ void gates4(const uint32_t (&v)[16], const float* s_bias4, float (&gi)[4], float (&gf)[4],
                                       float (&gg)[4], float (&go)[4]) {
  constexpr float SG = -INV_SCALE * LOG2E;
  constexpr float TMAX = 30.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 b = *reinterpret_cast<const float4*>(s_bias4 + 4 * j);
    const float ai = 1.f + ex2_fast(fminf(fmaf(__uint_as_float(v[4 * j + 0]), SG, b.x), TMAX));
    const float af = 1.f + ex2_fast(fminf(fmaf(__uint_as_float(v[4 * j + 1]), SG, b.y), TMAX));
    const float ag = 1.f + ex2_fast(fminf(fmaf(__uint_as_float(v[4 * j + 2]), 2.f * SG, b.z), TMAX));
    const float ao = 1.f + ex2_fast(fminf(fmaf(__uint_as_float(v[4 * j + 3]), SG, b.w), TMAX));
    const float p1 = ai * af, p2 = ag * ao;
    const float r = rcp_fast(p1 * p2);
    const float r1 = r * p2, r2 = r * p1;
    gi[j] = r1 * af;
    gf[j] = r1 * ai;
    gg[j] = fmaf(2.f, r2 * ao, -1.f);
    go[j] = r2 * ag;
  }
}

__device__ __forceinline__ float tanh_fwd(float c) {      // tanh(c') as the forward computes it
  const float b = 1.f + ex2_fast(fminf(c * (-2.f * LOG2E), 30.f));
  return fmaf(2.f, rcp_fast(b), -1.f);
}

// 8 values -> hi / lo fp16 halves (x * scale = hi + lo).  hi = x * scale truncated to 11 significant bits by an
// integer mask -- exactly representable in fp16, so no conversion back is needed -- and lo = the exact remainder rounded
// to fp16 (|lo| < 2^-10 |hi|): 21-22 significant bits, two values per conversion instruction.
__device__ __forceinline__ uint4 pack8_hi_lo(const float (&x)[8], float scale, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float a = x[2 * j] * scale, b = x[2 * j + 1] * scale;       // power of two: exact
    const float ah = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u), bh = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
    const __half2 hh = __floats2half2_rn(ah, bh);
    const __half2 ll = __floats2half2_rn(a - ah, b - bh);
    h[j] = *reinterpret_cast<const uint32_t*>(&hh);
    l[j] = *reinterpret_cast<const uint32_t*>(&ll);
  }
  lo = make_uint4(l[0], l[1], l[2], l[3]);
  return make_uint4(h[0], h[1], h[2], h[3]);
}

__global__ void __launch_bounds__(TC_P_THREADS, 1) bptt_gates_kernel(GatesArgs g, const __half* __restrict__ a_img,
                                                                    const __half* __restrict__ b_img,
                                                                    const float* __restrict__ bias_cat, int nitems,
                                                                    const float* __restrict__ head_w, int nout) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NSTAGE_P * STAGE_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  float* s_hw = reinterpret_cast<float*>(smem + NSTAGE_P * STAGE_BYTES + 256);   // head weights, unit-major [128][8]
  float* s_bias = s_hw + TC_H * HEAD_PAD;
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + NSTAGE_P);
  const uint32_t bar_tfull = smem_u32(bars + 2 * NSTAGE_P), bar_tempty = smem_u32(bars + 2 * NSTAGE_P + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < NSTAGE_P; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  load_scaled_bias(s_bias, bias_cat);
  for (int idx = threadIdx.x; idx < TC_H * HEAD_PAD; idx += blockDim.x) {
    const int u = idx / HEAD_PAD, o = idx - u * HEAD_PAD;
    s_hw[idx] = o < nout ? __ldg(head_w + (size_t)o * TC_H + u) : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int ncta = gridDim.x;

  if (warp == EPI_WARPS && lane == 0) {
    // ===== producer (as lstm_tc_kernel) =====
    uint32_t li = 0;
    bool ok = true;
    const uint32_t smem_base = smem_u32(smem);
    for (int item = blockIdx.x; item < nitems && ok; item += ncta, ++li) {
      const int tile = item >> 1, nh = item & 1;
      const unsigned char* a_src = reinterpret_cast<const unsigned char*>(a_img) + (size_t)tile * TC_NCHUNK * A_CHUNK_BYTES;
      const unsigned char* b_src = reinterpret_cast<const unsigned char*>(b_img) + (size_t)nh * TC_NCHUNK * B_CHUNK_BYTES;
#pragma unroll
      for (int c = 0; c < TC_NCHUNK; ++c) {
        if (!ok) break;
        const uint32_t s = c % NSTAGE_P;
        ok = mbar_wait(bar_empty + 8 * s, ((li * (TC_NCHUNK / NSTAGE_P) + c / NSTAGE_P) & 1) ^ 1, g.err);
        const uint32_t dst = smem_base + s * STAGE_BYTES;
        mbar_expect_tx(bar_full + 8 * s, STAGE_BYTES);
        bulk_g2s(dst, a_src + (size_t)c * (A_CHUNK_BYTES / 2), A_CHUNK_BYTES / 2, bar_full + 8 * s);
        bulk_g2s(dst + A_CHUNK_BYTES / 2, a_src + A_TILE_HALFS + (size_t)c * (A_CHUNK_BYTES / 2), A_CHUNK_BYTES / 2,
                 bar_full + 8 * s);
        bulk_g2s(dst + A_CHUNK_BYTES, b_src + (size_t)c * B_CHUNK_BYTES, B_CHUNK_BYTES, bar_full + 8 * s);
      }
    }
  } else if (warp == EPI_WARPS + 1 && lane == 0) {
    // ===== MMA issuer (as lstm_tc_kernel) =====
    const uint32_t idesc = (1u << 4) | ((uint32_t)(TC_NH >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
    uint32_t li = 0;
    bool ok = true;
    const uint64_t dA = make_desc(smem_u32(smem), 2048, 128), dB = make_desc(smem_u32(smem) + A_CHUNK_BYTES, 4096, 128);
    for (int item = blockIdx.x; item < nitems && ok; item += ncta, ++li) {
      const uint32_t acc = li & 1;
      ok = mbar_wait(bar_tempty + 8 * acc, ((li >> 1) & 1) ^ 1, g.err);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * TC_NH;
#pragma unroll
      for (int c = 0; c < TC_NCHUNK; ++c) {
        if (!ok) break;
        const uint32_t s = c % NSTAGE_P;
        ok = mbar_wait(bar_full + 8 * s, (li * (TC_NCHUNK / NSTAGE_P) + c / NSTAGE_P) & 1, g.err);
        tc_fence_after();
#pragma unroll
        for (int ks = 0; ks < TC_KC / 16; ++ks) {
          const uint64_t da_hi = dA + ((s * STAGE_BYTES + ks * 4096) >> 4);
          const uint64_t da_lo = dA + ((s * STAGE_BYTES + A_CHUNK_BYTES / 2 + ks * 4096) >> 4);
          const uint64_t db_hi = dB + ((s * STAGE_BYTES + ks * 8192) >> 4);
          const uint64_t db_lo = dB + ((s * STAGE_BYTES + B_CHUNK_BYTES / 2 + ks * 8192) >> 4);
          tc_mma_f16(tmem_d, da_hi, db_hi, idesc, (c | ks) != 0);
          tc_mma_f16(tmem_d, da_lo, db_hi, idesc, 1);
          tc_mma_f16(tmem_d, da_hi, db_lo, idesc, 1);
        }
        tc_commit(bar_empty + 8 * s);
      }
      tc_commit(bar_tfull + 8 * acc);
    }
  } else if (warp < EPI_WARPS) {
    // ===== epilogue: thread = (row of the tile, 16 hidden units) =====
    const int quarter = warp & 3, cq = warp >> 2;
    const float scale = g.sc->scale[g.q];
    uint32_t li = 0;
    bool ok = true;
    float dcm = 0.f;
    for (int item = blockIdx.x; item < nitems; item += ncta, ++li) {
      const int tile = item >> 1, nh = item & 1;
      const uint32_t acc = li & 1;
      const int row = tile * TC_M + quarter * 32 + lane;
      const bool inrange = row < g.R;
      const int ubase = nh * (TC_NH / 4) + cq * 16;
      bool fr = false, ct = false;
      if (inrange) {
        const int e = row / g.N;
        fr = g.fresh && g.fresh[e] != 0;
        ct = g.cut && g.cut[e] != 0;
      }
      float dsum[HEAD_PAD];      // d outputs of this row (value + logits)
      {
        float4 d0 = make_float4(0.f, 0.f, 0.f, 0.f), d1 = d0;
        if (inrange) {
          d0 = *reinterpret_cast<const float4*>(g.dout + (size_t)row * BP_HEADS);
          d1 = *reinterpret_cast<const float4*>(g.dout + (size_t)row * BP_HEADS + 4);
        }
        dsum[0] = d0.x; dsum[1] = d0.y; dsum[2] = d0.z; dsum[3] = d0.w;
        dsum[4] = d1.x; dsum[5] = d1.y; dsum[6] = d1.z; dsum[7] = d1.w;
      }
      // c_{t-1}, dh, dc of the first 4 hidden units: in flight while the MMAs of this item finish
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      const bool ld_c = inrange && !fr, ld_d = inrange && !ct;
      const size_t rbase = (size_t)row * TC_H + ubase;
      float4 cp_n = ld_c ? *reinterpret_cast<const float4*>(g.c_prev + rbase) : z4;
      float4 dh_n = ld_d ? *reinterpret_cast<const float4*>(g.dh + rbase) : z4;
      float4 dc_n = ld_d ? *reinterpret_cast<const float4*>(g.dc + rbase) : z4;
      if (ok) ok = mbar_wait(bar_tfull + 8 * acc, (li >> 1) & 1, g.err);
      tc_fence_after();
      const uint32_t taddr = tmem_base + acc * TC_NH + cq * 64 + ((uint32_t)(quarter * 32) << 16);
      __half* img_row = g.dg_img + (size_t)tile * DG_TILE_HALFS + (size_t)((quarter * 4 + (lane >> 3)) * 64 + (lane & 7) * 8);
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) {        // 4 hidden units (16 accumulator columns = 2 column groups) at a time
        const float4 cp = cp_n, dhv = dh_n, dcv = dc_n;
        if (q4 < 3) {                          // next group's operands: issued before this group's math
          cp_n = ld_c ? *reinterpret_cast<const float4*>(g.c_prev + rbase + (q4 + 1) * 4) : z4;
          dh_n = ld_d ? *reinterpret_cast<const float4*>(g.dh + rbase + (q4 + 1) * 4) : z4;
          dc_n = ld_d ? *reinterpret_cast<const float4*>(g.dc + rbase + (q4 + 1) * 4) : z4;
        }
        uint32_t v[16];
        tmem_ld16(taddr + q4 * 16, v);
        const int u0 = ubase + q4 * 4;
        float dg[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) dg[j] = 0.f;
        if (ok && inrange) {
          float gi[4], gf[4], gg[4], go[4];
          gates4(v, s_bias + 4 * u0, gi, gf, gg, go);
          const float cpa[4] = {cp.x, cp.y, cp.z, cp.w};
          const float dha[4] = {dhv.x, dhv.y, dhv.z, dhv.w};
          const float dca[4] = {dcv.x, dcv.y, dcv.z, dcv.w};
          float dcp[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            // heads: dh += sum_o dout_o W_o[u]
            const float4 w0 = *reinterpret_cast<const float4*>(&s_hw[(u0 + j) * HEAD_PAD]);
            const float4 w1 = *reinterpret_cast<const float4*>(&s_hw[(u0 + j) * HEAD_PAD + 4]);
            float dh = dha[j];
            dh = fmaf(dsum[0], w0.x, dh); dh = fmaf(dsum[1], w0.y, dh); dh = fmaf(dsum[2], w0.z, dh); dh = fmaf(dsum[3], w0.w, dh);
            dh = fmaf(dsum[4], w1.x, dh); dh = fmaf(dsum[5], w1.y, dh); dh = fmaf(dsum[6], w1.z, dh); dh = fmaf(dsum[7], w1.w, dh);
            const float cn = fmaf(gf[j], cpa[j], gi[j] * gg[j]);
            const float tc = tanh_fwd(cn);
            const float dct = fmaf(dh * go[j], 1.f - tc * tc, dca[j]);
            dg[4 * j + 0] = dct * gg[j] * gi[j] * (1.f - gi[j]);
            dg[4 * j + 1] = dct * cpa[j] * gf[j] * (1.f - gf[j]);
            dg[4 * j + 2] = dct * gi[j] * (1.f - gg[j] * gg[j]);
            dg[4 * j + 3] = dh * tc * go[j] * (1.f - go[j]);
            dcp[j] = fr ? 0.f : dct * gf[j];
            dcm = fmaxf(dcm, fabsf(dcp[j]));
          }
          *reinterpret_cast<float4*>(g.dc + (size_t)row * TC_H + u0) = make_float4(dcp[0], dcp[1], dcp[2], dcp[3]);
        }
        // d gates image: column 4u + gate; this thread's 16 columns = column groups cgA, cgA + 1 of its row
        const int cgA = (nh * 256 + cq * 64 + q4 * 16) >> 3;
        const float x0[8] = {dg[0], dg[1], dg[2], dg[3], dg[4], dg[5], dg[6], dg[7]};
        const float x1[8] = {dg[8], dg[9], dg[10], dg[11], dg[12], dg[13], dg[14], dg[15]};
        uint4 lo0, lo1;
        const uint4 hi0 = pack8_hi_lo(x0, scale, lo0), hi1 = pack8_hi_lo(x1, scale, lo1);
        __half* p0 = img_row + (size_t)cgA * 1024;
        *reinterpret_cast<uint4*>(p0) = hi0;
        *reinterpret_cast<uint4*>(p0 + DG_PART_HALFS) = lo0;
        *reinterpret_cast<uint4*>(p0 + 1024) = hi1;
        *reinterpret_cast<uint4*>(p0 + 1024 + DG_PART_HALFS) = lo1;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) dcm = fmaxf(dcm, __shfl_xor_sync(IC3_FULL_MASK, dcm, s));
    if (lane == 0 && dcm > 0.f) atomicMax(&g.sc->dcmax, __float_as_uint(dcm));
  }
  tc_fence_before();
  __syncthreads();
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------------------------
// dgrad: [dS | dh_direct] = d gates . [W_ih C | W_hh]        (M = rows, K = 512 gate columns, N = 256)
// ------------------------------------------------------------------------------------------------------------------
constexpr int DGR_NCHUNK = 16;                       // 512 gate columns / 32
constexpr int DGR_STAGE = A_CHUNK_BYTES + B_CHUNK_BYTES;   // 16 KB (hi + lo of 32 columns x 128 rows) + 32 KB

// weight image of the dgrad GEMM: element (n = S / h feature, k = gate column j) = scaled forward weight
// [W_ih ; W_ih C ; W_hh] (j, 128 + n): [chunk 16][hi, lo][kcore 4][ncore 32][8][8]
__host__ __device__ __forceinline__ size_t w2_img_off(int k, int n, int part) {
  const int c = k >> 5, kk = k & 31;
  return ((((size_t)(c * 2 + part) * 4 + (kk >> 3)) * 32 + (n >> 3)) * 8 + (n & 7)) * 8 + (kk & 7);
}
constexpr size_t W2_IMG_HALFS = (size_t)DGR_NCHUNK * 2 * 4 * 32 * 64;     // 262144 halfs = 512 KB

__global__ void bptt_pack_w2_kernel(const __half* __restrict__ b_img, __half* __restrict__ w2) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;      // (n, j)
  if (idx >= 256 * 512) return;
  const int n = idx >> 9, j = idx & 511;
  const int nh = j >> 8, col = j & 255;
#pragma unroll
  for (int part = 0; part < 2; ++part) w2[w2_img_off(j, n, part)] = b_img[b_img_off(nh, 128 + n, col, part)];
}

struct DgradArgs {
  int R;
  const float* gs;       // [R] g / den
  float* dSs;            // [R, H]  out: gs * dS
  float* dh_direct;      // [R, H]  out
  const BpttScalars* sc;
  int q;
  int32_t* err;
};

__global__ void __launch_bounds__(TC_P_THREADS, 1) bptt_dgrad_kernel(DgradArgs g, const __half* __restrict__ dg_img,
                                                                    const __half* __restrict__ w2_img, int ntiles) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NSTAGE_P * DGR_STAGE);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + NSTAGE_P);
  const uint32_t bar_tfull = smem_u32(bars + 2 * NSTAGE_P), bar_tempty = smem_u32(bars + 2 * NSTAGE_P + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < NSTAGE_P; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int ncta = gridDim.x;
  static_assert(DGR_NCHUNK % NSTAGE_P == 0, "stage index must be a function of the chunk index alone");

  if (warp == EPI_WARPS && lane == 0) {
    uint32_t li = 0;
    bool ok = true;
    const uint32_t smem_base = smem_u32(smem);
    for (int tile = blockIdx.x; tile < ntiles && ok; tile += ncta, ++li) {
      const unsigned char* a_src = reinterpret_cast<const unsigned char*>(dg_img) + (size_t)tile * DG_TILE_HALFS * 2;
      const unsigned char* b_src = reinterpret_cast<const unsigned char*>(w2_img);
#pragma unroll
      for (int c = 0; c < DGR_NCHUNK; ++c) {
        if (!ok) break;
        const uint32_t s = c % NSTAGE_P;
        ok = mbar_wait(bar_empty + 8 * s, ((li * (DGR_NCHUNK / NSTAGE_P) + c / NSTAGE_P) & 1) ^ 1, g.err);
        const uint32_t dst = smem_base + s * DGR_STAGE;
        mbar_expect_tx(bar_full + 8 * s, DGR_STAGE);
        // 32 gate columns = 4 column groups = 8 KB per part, contiguous in the d gates image
        bulk_g2s(dst, a_src + (size_t)c * 8192, 8192, bar_full + 8 * s);
        bulk_g2s(dst + 8192, a_src + (size_t)DG_PART_HALFS * 2 + (size_t)c * 8192, 8192, bar_full + 8 * s);
        bulk_g2s(dst + A_CHUNK_BYTES, b_src + (size_t)c * B_CHUNK_BYTES, B_CHUNK_BYTES, bar_full + 8 * s);
      }
    }
  } else if (warp == EPI_WARPS + 1 && lane == 0) {
    const uint32_t idesc = (1u << 4) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
    uint32_t li = 0;
    bool ok = true;
    const uint64_t dA = make_desc(smem_u32(smem), 2048, 128), dB = make_desc(smem_u32(smem) + A_CHUNK_BYTES, 4096, 128);
    for (int tile = blockIdx.x; tile < ntiles && ok; tile += ncta, ++li) {
      const uint32_t acc = li & 1;
      ok = mbar_wait(bar_tempty + 8 * acc, ((li >> 1) & 1) ^ 1, g.err);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * 256;
#pragma unroll
      for (int c = 0; c < DGR_NCHUNK; ++c) {
        if (!ok) break;
        const uint32_t s = c % NSTAGE_P;
        ok = mbar_wait(bar_full + 8 * s, (li * (DGR_NCHUNK / NSTAGE_P) + c / NSTAGE_P) & 1, g.err);
        tc_fence_after();
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
          const uint64_t da_hi = dA + ((s * DGR_STAGE + ks * 4096) >> 4);
          const uint64_t da_lo = dA + ((s * DGR_STAGE + 8192 + ks * 4096) >> 4);
          const uint64_t db_hi = dB + ((s * DGR_STAGE + ks * 8192) >> 4);
          const uint64_t db_lo = dB + ((s * DGR_STAGE + B_CHUNK_BYTES / 2 + ks * 8192) >> 4);
          tc_mma_f16(tmem_d, da_hi, db_hi, idesc, (c | ks) != 0);
          tc_mma_f16(tmem_d, da_lo, db_hi, idesc, 1);
          tc_mma_f16(tmem_d, da_hi, db_lo, idesc, 1);
        }
        tc_commit(bar_empty + 8 * s);
      }
      tc_commit(bar_tfull + 8 * acc);
    }
  } else if (warp < EPI_WARPS) {
    const int quarter = warp & 3, cq = warp >> 2;
    const float unscale = g.sc->inv_scale[g.q] * (1.f / SCALE_B);
    uint32_t li = 0;
    bool ok = true;
    for (int tile = blockIdx.x; tile < ntiles; tile += ncta, ++li) {
      const uint32_t acc = li & 1;
      const int row = tile * TC_M + quarter * 32 + lane;
      const bool inrange = row < g.R;
      float f = unscale;
      if (cq < 2 && inrange) f *= g.gs[row];
      if (ok) ok = mbar_wait(bar_tfull + 8 * acc, (li >> 1) & 1, g.err);
      tc_fence_after();
      const uint32_t taddr = tmem_base + acc * 256 + cq * 64 + ((uint32_t)(quarter * 32) << 16);
      float* dst = (cq < 2 ? g.dSs : g.dh_direct) + (size_t)row * TC_H + (cq & 1) * 64;
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) {
        uint32_t v[16];
        tmem_ld16(taddr + q4 * 16, v);
        if (ok && inrange) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            *reinterpret_cast<float4*>(dst + q4 * 16 + 4 * j) =
                make_float4(__uint_as_float(v[4 * j]) * f, __uint_as_float(v[4 * j + 1]) * f, __uint_as_float(v[4 * j + 2]) * f,
                            __uint_as_float(v[4 * j + 3]) * f);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------------------------
// comm: backward of S_k = (g_k / den) (sum_j g_j h_j - g_k h_k)  (comm.py:181-205) + the cuts of the recursion
//   dh_{t-1}[j] = keep * (dh_direct[j] + g_j (sum_k dSs[k] - g_j dSs[j])),  dSs = (g / den) dS,  keep = 1 - fresh_t
// One warp per environment, lane = 4 hidden units.
// ------------------------------------------------------------------------------------------------------------------
struct CommArgs {
  int B, N;
  const float* dSs;
  const float* dh_direct;
  const float* gr;          // [R]
  const uint8_t* fresh;     // [B]
  int no_comm;              // comm_mask_zero
  float* dh;                // [R, H] out
  BpttScalars* sc;
};

__global__ void __launch_bounds__(256) bptt_comm_kernel(CommArgs a) {
  const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  float m = 0.f;
  if (e < a.B) {
    const bool fr = a.fresh && a.fresh[e] != 0;
    const size_t base = (size_t)e * a.N;
    float4 tot = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!fr && !a.no_comm) {
      for (int k = 0; k < a.N; ++k) {
        const float4 d = *(reinterpret_cast<const float4*>(a.dSs + (base + k) * TC_H) + lane);
        tot.x += d.x; tot.y += d.y; tot.z += d.z; tot.w += d.w;
      }
    }
    for (int j = 0; j < a.N; ++j) {
      float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
      if (!fr) {
        o = *(reinterpret_cast<const float4*>(a.dh_direct + (base + j) * TC_H) + lane);
        if (!a.no_comm) {
          const float gj = a.gr[base + j];
          if (gj != 0.f) {
            const float4 d = *(reinterpret_cast<const float4*>(a.dSs + (base + j) * TC_H) + lane);
            o.x += gj * (tot.x - gj * d.x); o.y += gj * (tot.y - gj * d.y);
            o.z += gj * (tot.z - gj * d.z); o.w += gj * (tot.w - gj * d.w);
          }
        }
      }
      *(reinterpret_cast<float4*>(a.dh + (base + j) * TC_H) + lane) = o;
      m = fmaxf(m, fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w))));
    }
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) m = fmaxf(m, __shfl_xor_sync(IC3_FULL_MASK, m, s));
  if (lane == 0 && m > 0.f) atomicMax(&a.sc->dhmax, __float_as_uint(m));
}

// ------------------------------------------------------------------------------------------------------------------
// wgrad: G[gate column j][feature n] += sum_rows dgates[row][j] * F[row][n],  F = [x | S | h] (hi/lo) and P (exact)
// Both operands are MN-major views of images written for the other GEMMs; a pipeline stage is a 32-row slab
// gathered by tensor copies (cp.async.bulk.tensor) whose box re-packs it as [group][4 row groups][8][8].
// CTA role = (block of 128 gate columns mb, feature slice sl, row-tile subset): accumulators stay in tensor memory
// for the whole launch and are added into the CTA's private fp32 partial at the end (no atomics; the partials of all
// CTAs are summed in float64 by ic3_bptt_finish).
// ------------------------------------------------------------------------------------------------------------------
constexpr int WG_THREADS = 192;          // 4 epilogue warps (TMEM lanes) + producer warp + MMA warp
constexpr int WG_DG_BYTES = 16 * 4 * 128;       // 8 KB: 16 column groups x 4 row groups, one part
constexpr int WG_A_BYTES = 48 * 4 * 128;        // 24 KB: 48 feature groups x 4 row groups, one part
constexpr int WG_STAGE0 = 2 * WG_DG_BYTES + 2 * WG_A_BYTES;   // 64 KB
constexpr int WG_NSTAGE0 = 3;
constexpr int WG_NSTAGE1 = 4;

struct WgradArgs {
  int ntiles;
  int np;                // columns of P (multiple of 16, <= WG_MAX_NP)
  int j0, j1;            // row-tile subsets of slice 0 / slice 1 (4 * (j0 + j1) CTAs)
  float* partial;        // [ncta][512 columns max][128] fp32, CTA-private
  const BpttScalars* sc;
  int q;
  int32_t* err;
};

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, int c4,
                                            uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

__global__ void __launch_bounds__(WG_THREADS, 1) bptt_wgrad_kernel(WgradArgs g, const __grid_constant__ CUtensorMap map_dg,
                                                                  const __grid_constant__ CUtensorMap map_a,
                                                                  const __grid_constant__ CUtensorMap map_p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t bars[2 * WG_NSTAGE1 + 1];
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // role
  const int per_mb = g.j0 + g.j1;
  const int mb = blockIdx.x / per_mb, rj = blockIdx.x - mb * per_mb;
  const int sl = rj < g.j0 ? 0 : 1;
  const int jj = sl == 0 ? rj : rj - g.j0, jn = sl == 0 ? g.j0 : g.j1;
  const int nstage = sl == 0 ? WG_NSTAGE0 : WG_NSTAGE1;
  const int p_bytes = g.np * 64;                    // np/8 groups x 4 row groups x 128 B
  const int stage_bytes = sl == 0 ? WG_STAGE0 : 2 * WG_DG_BYTES + p_bytes;
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + WG_NSTAGE1), bar_done = smem_u32(bars + 2 * WG_NSTAGE1);
  if (threadIdx.x == 0) {
    for (int s = 0; s < WG_NSTAGE1; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const int nmine = (g.ntiles - jj + jn - 1) / jn;      // tiles jj, jj + jn, ...
  const int nchunks = nmine > 0 ? nmine * 4 : 0;         // 32-row slabs

  if (warp == 4 && lane == 0) {
    // ===== producer =====
    bool ok = true;
    const uint32_t smem_base = smem_u32(smem);
    for (int ch = 0; ch < nchunks && ok; ++ch) {
      const int tile = jj + (ch >> 2) * jn, rc = ch & 3;
      const int s = ch % nstage;
      ok = mbar_wait(bar_empty + 8 * s, ((ch / nstage) & 1) ^ 1, g.err);
      const uint32_t dst = smem_base + s * stage_bytes;
      mbar_expect_tx(bar_full + 8 * s, stage_bytes);
      tma_load_5d(dst, &map_dg, 0, 4 * rc, 16 * mb, 0, tile, bar_full + 8 * s);
      tma_load_5d(dst + WG_DG_BYTES, &map_dg, 0, 4 * rc, 16 * mb, 1, tile, bar_full + 8 * s);
      if (sl == 0) {
        tma_load_5d(dst + 2 * WG_DG_BYTES, &map_a, 0, 4 * rc, 0, 0, tile, bar_full + 8 * s);
        tma_load_5d(dst + 2 * WG_DG_BYTES + WG_A_BYTES, &map_a, 0, 4 * rc, 0, 1, tile, bar_full + 8 * s);
      } else {
        tma_load_4d(dst + 2 * WG_DG_BYTES, &map_p, 0, 4 * rc, 0, tile, bar_full + 8 * s);
      }
    }
  } else if (warp == 5 && lane == 0) {
    // ===== MMA issuer =====
    // D = f32, A = B = f16, both MN-major (bits 15, 16); M = 128 gate columns
    const uint32_t ibase = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(TC_M >> 4) << 24);
    bool ok = true;
    const uint32_t sbase = smem_u32(smem);
    // MN-major no-swizzle: LBO = stride between the two 8-row (K) groups of one MMA = 128 B,
    //                      SBO = stride between 8-element MN groups = 4 row groups x 128 B = 512 B
    for (int ch = 0; ch < nchunks && ok; ++ch) {
      const int s = ch % nstage;
      ok = mbar_wait(bar_full + 8 * s, (ch / nstage) & 1, g.err);
      tc_fence_after();
      const uint32_t st = sbase + s * stage_bytes;
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {               // 16 rows = 2 row groups per MMA
        const uint64_t dg_hi = make_desc(st + ks * 256, 128, 512);
        const uint64_t dg_lo = make_desc(st + WG_DG_BYTES + ks * 256, 128, 512);
        const uint32_t accum = (ch | ks) != 0;
        if (sl == 0) {
          const uint32_t a_hi = st + 2 * WG_DG_BYTES + ks * 256, a_lo = a_hi + WG_A_BYTES;
          const uint32_t i256 = ibase | ((uint32_t)(256 >> 3) << 17), i128 = ibase | ((uint32_t)(128 >> 3) << 17);
          // features 0..255 (x | S) -> columns 0..255; features 256..383 (h) -> columns 256..383
          tc_mma_f16(tmem_base, dg_hi, make_desc(a_hi, 128, 512), i256, accum);
          tc_mma_f16(tmem_base, dg_lo, make_desc(a_hi, 128, 512), i256, 1);
          tc_mma_f16(tmem_base, dg_hi, make_desc(a_lo, 128, 512), i256, 1);
          tc_mma_f16(tmem_base + 256, dg_hi, make_desc(a_hi + 32 * 512, 128, 512), i128, accum);
          tc_mma_f16(tmem_base + 256, dg_lo, make_desc(a_hi + 32 * 512, 128, 512), i128, 1);
          tc_mma_f16(tmem_base + 256, dg_hi, make_desc(a_lo + 32 * 512, 128, 512), i128, 1);
        } else {
          const uint32_t p0 = st + 2 * WG_DG_BYTES + ks * 256;
          const int n0 = g.np > 256 ? 256 : g.np, n1 = g.np - n0;
          const uint32_t in0 = ibase | ((uint32_t)(n0 >> 3) << 17);
          tc_mma_f16(tmem_base, dg_hi, make_desc(p0, 128, 512), in0, accum);
          tc_mma_f16(tmem_base, dg_lo, make_desc(p0, 128, 512), in0, 1);
          if (n1 > 0) {
            const uint32_t in1 = ibase | ((uint32_t)(n1 >> 3) << 17);
            tc_mma_f16(tmem_base + 256, dg_hi, make_desc(p0 + 32 * 512, 128, 512), in1, accum);
            tc_mma_f16(tmem_base + 256, dg_lo, make_desc(p0 + 32 * 512, 128, 512), in1, 1);
          }
        }
      }
      tc_commit(bar_empty + 8 * s);
    }
    tc_commit(bar_done);
  } else if (warp < 4) {
    // ===== flush: TMEM lane = gate column of the block, column = feature =====
    const int ncols = sl == 0 ? 384 : g.np;
    float* part = g.partial + (size_t)blockIdx.x * 512 * 128;
    if (nchunks > 0) {
      const bool ok = mbar_wait(bar_done, 0, g.err);
      tc_fence_after();
      // slice 0: x|S|h products carry SCALE_A * s_t, slice 1 (P exact) only s_t
      const float unscale = g.sc->inv_scale[g.q] * (sl == 0 ? 1.f / SCALE_A : 1.f);
      const int m = warp * 32 + lane;
      for (int c0 = 0; c0 < ncols; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(tmem_base + c0 + ((uint32_t)(warp * 32) << 16), v);
        if (ok) {
#pragma unroll
          for (int j = 0; j < 16; ++j) part[(size_t)(c0 + j) * 128 + m] += __uint_as_float(v[j]) * unscale;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------------------------
// finish
// ------------------------------------------------------------------------------------------------------------------
// G[j][n] = sum over the CTAs of (mb = j / 128, slice(n)) of partial[cta][n_local][j % 128]   (float64)
__global__ void bptt_reduce_partials_kernel(const float* __restrict__ partial, int j0, int j1, int np, double* __restrict__ G,
                                            int ncols_total) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;     // (n, j): j fastest -> coalesced partial reads
  if (idx >= 512 * ncols_total) return;
  const int n = idx >> 9, j = idx & 511;
  const int mb = j >> 7, m = j & 127;
  const int sl = n < 384 ? 0 : 1, nl = sl == 0 ? n : n - 384;
  const int per_mb = j0 + j1;
  const int first = mb * per_mb + (sl == 0 ? 0 : j0), cnt = sl == 0 ? j0 : j1;
  double acc = 0.0;
  for (int c = 0; c < cnt; ++c) acc += (double)partial[((size_t)(first + c) * 512 + nl) * 128 + m];
  G[(size_t)j * ncols_total + n] = acc;
}

// out[m][n] (+)= sum_k A[k * lda + m] * B[k * ldb + n]   (float64, tiny matrices: once per update)
__global__ void small_gemm_tn_kernel(int M, int Nn, int K, const double* __restrict__ A, int lda, const double* __restrict__ Bm,
                                     int ldb, double* __restrict__ out, int ldo, int accumulate) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * Nn) return;
  const int m = idx / Nn, n = idx - m * Nn;
  double acc = 0.0;
  for (int k = 0; k < K; ++k) acc += A[(size_t)k * lda + m] * Bm[(size_t)k * ldb + n];
  if (accumulate) out[(size_t)m * ldo + n] += acc;
  else out[(size_t)m * ldo + n] = acc;
}

struct FinishArgs {
  int O, nheads, atot, npos, np, WW;
  int head_dim[IC3_MAX_HEADS];
  const double* G;          // [512][NC] rows = gate column j = 4u + gate
  int NC;
  const double* Y;          // [128][np]  W_ih^T Q
  const double* GSC;        // [512][128] G_S C^T
  const double* dC;         // [128][128] W_ih^T G_S
  const float* c_b;
  float* g_w_ih; float* g_w_hh; float* g_b_ih; float* g_b_hh; float* g_c_w; float* g_c_b;
  float* g_enc_w; float* g_enc_b; float* g_value_w; float* g_value_b;
  float* g_head_w[IC3_MAX_HEADS]; float* g_head_b[IC3_MAX_HEADS];
  const float* gw_part; const double* gs_part; int nhb;     // heads partials
  double* losses;            // [3] out
  ic3_pp_cfg pp; ic3_tj_cfg tj; int is_tj;
  int ones_col;              // column of P holding the constant 1
};

// LSTM / comm parameter gradients: thread = (LSTM row r = gate * H + u, k)
__global__ void bptt_finish_lstm_kernel(FinishArgs f) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < 512 * TC_H) {
    const int r = idx >> 7, k = idx & 127;
    const int gate = r >> 7, u = r & 127, j = 4 * u + gate;
    const double* Gj = f.G + (size_t)j * f.NC;
    const double g1 = Gj[384 + f.ones_col];                   // sum over rows of d gates (bias gradient)
    f.g_w_hh[idx] += (float)Gj[256 + k];
    f.g_w_ih[idx] += (float)(Gj[k] + f.GSC[(size_t)j * TC_H + k] + g1 * (double)f.c_b[k]);
    if (k == 0) {
      f.g_b_ih[r] += (float)g1;
      f.g_b_hh[r] += (float)g1;
    }
  }
  if (idx < TC_H * TC_H) f.g_c_w[idx] += (float)f.dC[idx];     // [k][m]
}

// encoder / comm-bias / heads gradients
__global__ void bptt_finish_misc_kernel(FinishArgs f) {
  const int ones_col = f.ones_col;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int k = idx & 127;
  if (idx < TC_H) {
    const double y1 = f.Y[(size_t)k * f.np + ones_col];
    f.g_c_b[k] += (float)y1;                   // W_ih^T g1
    f.g_enc_b[k] += (float)y1;
  }
  // encoder weight [H][O]: position one-hot columns -> every window cell's class feature of that position
  const int W = f.is_tj ? 2 * f.tj.vision + 1 : 2 * f.pp.vision + 1;
  const int WW = W * W;
  const int item = idx >> 7;
  if (item < f.npos * WW) {
    const int pos = item / WW, w = item - pos * WW;
    const int dy = w / W, dx = w - dy * W;
    int feat;
    if (!f.is_tj) {
      const int D = f.pp.dim, v = f.pp.vision, V = D * D + 4;
      const int rr = pos / D - v + dy, cc = pos % D - v + dx;
      feat = (rr >= 0 && rr < D && cc >= 0 && cc < D) ? w * V + rr * D + cc : w * V + V - 3;
    } else {
      const int v = f.tj.vision, V = f.tj.vocab;
      const int rr = pos / f.tj.w - v + dy, cc = pos % f.tj.w - v + dx;
      int cls = f.tj.outside_cls;
      if (rr >= 0 && rr < f.tj.h && cc >= 0 && cc < f.tj.w) cls = f.tj.grid[rr * f.tj.w + cc];
      feat = 2 + w * V + cls;
    }
    atomicAdd(&f.g_enc_w[(size_t)k * f.O + feat], (float)f.Y[(size_t)k * f.np + pos]);
  }
  // count / scalar feature columns
  const int nextra = f.is_tj ? WW + 3 : 2 * WW;
  if (item < nextra) {
    int feat;
    double y;
    if (!f.is_tj) {
      const int V = f.pp.dim * f.pp.dim + 4;
      const int w = item >> 1;
      feat = w * V + ((item & 1) ? V - 1 : V - 2);          // predator : prey count
      y = f.Y[(size_t)k * f.np + f.npos + item];
    } else if (item < WW) {
      feat = 2 + item * f.tj.vocab + f.tj.car_cls;
      y = f.Y[(size_t)k * f.np + f.npos + item];
    } else if (item == WW) {
      feat = 0;                                               // last_act
      y = f.Y[(size_t)k * f.np + f.npos + WW];
    } else if (item == WW + 1) {
      feat = 1;                                               // route id ratio: hi + lo columns
      y = f.Y[(size_t)k * f.np + f.npos + WW + 1] + f.Y[(size_t)k * f.np + f.npos + WW + 2];
    } else {
      return;
    }
    atomicAdd(&f.g_enc_w[(size_t)k * f.O + feat], (float)y);
  }
}

__global__ void bptt_finish_heads_kernel(FinishArgs f) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;     // (o, u)
  if (idx < BP_HEADS * TC_H) {
    const int o = idx >> 7, u = idx & 127;
    double acc = 0.0;
    for (int b = 0; b < f.nhb; ++b) acc += (double)f.gw_part[((size_t)b * BP_HEADS + o) * TC_H + u];
    if (o == 0) {
      f.g_value_w[u] += (float)acc;
    } else {
      int off = 1;
      for (int m = 0; m < f.nheads; ++m) {
        if (o < off + f.head_dim[m]) {
          f.g_head_w[m][(size_t)(o - off) * TC_H + u] += (float)acc;
          break;
        }
        off += f.head_dim[m];
      }
    }
  }
  if (idx < BP_HEADS + 3) {
    double acc = 0.0;
    for (int b = 0; b < f.nhb; ++b) acc += f.gs_part[(size_t)b * (BP_HEADS + 3) + idx];
    if (idx >= BP_HEADS) {
      f.losses[idx - BP_HEADS] = acc;
    } else if (idx == 0) {
      f.g_value_b[0] += (float)acc;
    } else {
      int off = 1;
      for (int m = 0; m < f.nheads; ++m) {
        if (idx < off + f.head_dim[m]) {
          f.g_head_b[m][idx - off] += (float)acc;
          break;
        }
        off += f.head_dim[m];
      }
    }
  }
}

// double copies of the fp32 weights the finishing GEMMs need: W_ih in gate-column order [j][k], C [n][k]
__global__ void bptt_weights_f64_kernel(const float* __restrict__ w_ih, const float* __restrict__ c_w, double* __restrict__ wj,
                                        double* __restrict__ cw) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < 512 * TC_H) {
    const int j = idx >> 7, k = idx & 127;
    const int u = j >> 2, gate = j & 3;
    wj[idx] = (double)w_ih[(size_t)(gate * TC_H + u) * TC_H + k];
  }
  if (idx < TC_H * TC_H) cw[idx] = (double)c_w[idx];
}

// G_S C^T: out[j][k] = sum_m G[j][128 + m] * C[k][m]   -> small_gemm_tn wants A[k'][m'] layout; do it directly
__global__ void bptt_gsc_kernel(const double* __restrict__ G, int NC, const double* __restrict__ cw, double* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 512 * TC_H) return;
  const int j = idx >> 7, k = idx & 127;
  double acc = 0.0;
  for (int m = 0; m < TC_H; ++m) acc += G[(size_t)j * NC + 128 + m] * cw[(size_t)k * TC_H + m];
  out[idx] = acc;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// image of core matrices [tile][(part)][group][rg 16][64 halfs]: box = [64][4 row groups][ngroups_box][1]([1])
int make_image_map(CUtensorMap* map, void* base, int ntiles, int nparts, int ngroups, int box_groups) {
  EncodeTiledFn fn = encode_tiled();
  if (!fn) return IC3_E_UNSUPPORTED;
  if (nparts > 0) {
    cuuint64_t dims[5] = {64, 16, (cuuint64_t)ngroups, (cuuint64_t)nparts, (cuuint64_t)ntiles};
    cuuint64_t strides[4] = {128, 2048, (cuuint64_t)ngroups * 2048, (cuuint64_t)nparts * ngroups * 2048};
    cuuint32_t box[5] = {64, 4, (cuuint32_t)box_groups, 1, 1};
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? IC3_OK : IC3_E_RANGE;
  }
  cuuint64_t dims[4] = {64, 16, (cuuint64_t)ngroups, (cuuint64_t)ntiles};
  cuuint64_t strides[3] = {128, 2048, (cuuint64_t)ngroups * 2048};
  cuuint32_t box[4] = {64, 4, (cuuint32_t)box_groups, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? IC3_OK : IC3_E_RANGE;
}

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// Side stream of the weight-gradient kernel + the events that order it against the main stream (IC3_BPTT_OVERLAP=0
// keeps everything on the caller's stream).
struct BpttStreams {
  cudaStream_t side;
  cudaEvent_t gates_done[2], wgrad_done[2], prep_done[2], main_done[2];
  bool overlap;
  int prepared_t[2];         // lock-step index whose heads / operand images occupy buffer set q (-1: none)
};

BpttStreams* bptt_streams() {
  static BpttStreams ss;
  static int state = 0;      // 0 = not created, 1 = ok, -1 = failed
  if (state == 0) {
    const char* e = getenv("IC3_BPTT_OVERLAP");
    ss.overlap = !(e && atoi(e) == 0);
    ss.prepared_t[0] = ss.prepared_t[1] = -1;
    bool ok = cudaStreamCreateWithFlags(&ss.side, cudaStreamNonBlocking) == cudaSuccess;
    for (int k = 0; k < 2 && ok; ++k) {
      ok = cudaEventCreateWithFlags(&ss.gates_done[k], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&ss.wgrad_done[k], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&ss.prep_done[k], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&ss.main_done[k], cudaEventDisableTiming) == cudaSuccess;
    }
    state = ok ? 1 : -1;
  }
  return state == 1 ? &ss : nullptr;
}

// The persistent tensor-core kernels leave ~30 KB of an SM's shared memory unused; with the carve-out pinned to the
// maximum (instead of the smallest configuration that fits the kernel) one CTA of the look-ahead kernels (operand images,
// heads gradient) can be resident beside them.
template <typename K>
cudaError_t prefer_max_smem(K kern) {
  return cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}

// Development aid (IC3_BPTT_TRACE=1): CUDA events after every kernel of the first steps of a compute_grad, on whatever
// stream the kernel ran, dumped by ic3_debug_bptt_trace() as end times on one clock -- shows what overlaps what.
constexpr int TR_STEPS = 16, TR_KERNELS = 7;     // heads, prep, scale, gates, dgrad, comm, wgrad
struct BpttTrace {
  bool on;
  cudaEvent_t base, ev[TR_STEPS][TR_KERNELS];
  bool used[TR_STEPS][TR_KERNELS];
  int t_first;
};
BpttTrace* bptt_trace() {
  static BpttTrace tr;
  static int state = 0;
  if (state == 0) {
    const char* e = getenv("IC3_BPTT_TRACE");
    tr.on = e && atoi(e) != 0;
    if (tr.on) {
      cudaEventCreate(&tr.base);
      for (int i = 0; i < TR_STEPS; ++i)
        for (int k = 0; k < TR_KERNELS; ++k) cudaEventCreate(&tr.ev[i][k]);
    }
    state = 1;
  }
  return &tr;
}
inline void trace_mark(int kernel, int t, cudaStream_t s) {
  BpttTrace* tr = bptt_trace();
  if (!tr->on) return;
  const int i = tr->t_first - t;
  if (i < 0 || i >= TR_STEPS) return;
  cudaEventRecord(tr->ev[i][kernel], s);
  tr->used[i][kernel] = true;
}

struct Layout {         // of the workspace, in bytes
  size_t a_img, p_img, dg_img, img_stride, w2_img, dout, dSs, dh_direct, gs, gr, partial, gw_part, gs_part, sc, G, Y, GSC, dC, wj, cw, losses,
      total;
  int ntiles, np, npos, WW, j0, j1, ncta_wg, nhb;
};

int plan_layout(const ic3_policy_cfg* cfg, int npos, int WW, int is_tj, Layout* L) {
  const long R = (long)cfg->B * cfg->N;
  L->ntiles = (int)((R + TC_M - 1) / TC_M);
  L->npos = npos;
  L->WW = WW;
  const int used = npos + (is_tj ? WW + 4 : 2 * WW + 1);
  L->np = (used + 15) / 16 * 16;
  if (L->np > WG_MAX_NP) return IC3_E_UNSUPPORTED;
  const int per_mb = sm_count() / 4;
  if (per_mb < 2) return IC3_E_UNSUPPORTED;
  // MMA cycles per 16 rows: slice 0 = 3 * (128 + 86), slice 1 = 2 * (n0 + n1 shapes) -> split the CTAs accordingly
  const double c0 = 3.0 * (128 + 86), c1 = 2.0 * (L->np > 256 ? 128 + 0.5 * (L->np - 256) + 22 : 0.5 * L->np + 22);
  int j0 = (int)(per_mb * c0 / (c0 + c1) + 0.5);
  if (j0 < 1) j0 = 1;
  if (j0 > per_mb - 1) j0 = per_mb - 1;
  L->j0 = j0;
  L->j1 = per_mb - j0;
  L->ncta_wg = 4 * per_mb;
  L->nhb = (int)((R + HB_ROWS - 1) / HB_ROWS);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 1023) / 1024 * 1024; return o; };
  // two sets of operand images (step parity): the weight-gradient kernel of step t reads set t & 1 on the side stream
  // while the main stream fills the other set for step t - 1
  L->a_img = take((size_t)L->ntiles * A_TILE_HALFS * 2);
  L->p_img = take((size_t)L->ntiles * (L->np / 8) * 16 * 128);
  L->dg_img = take((size_t)L->ntiles * DG_TILE_HALFS * 2);
  L->img_stride = off;
  take(off);                                   // second set: same sizes, same order
  L->w2_img = take(W2_IMG_HALFS * 2);
  L->dout = take((size_t)2 * L->ntiles * TC_M * BP_HEADS * 4);         // [2]: heads of step t - 1 run while step t reads
  L->dSs = take((size_t)L->ntiles * TC_M * TC_H * 4);
  L->dh_direct = take((size_t)L->ntiles * TC_M * TC_H * 4);
  L->gs = take((size_t)2 * L->ntiles * TC_M * 4);                       // [2] by step parity, like the images
  L->gr = take((size_t)2 * L->ntiles * TC_M * 4);
  L->partial = take((size_t)L->ncta_wg * 512 * 128 * 4);
  L->gw_part = take((size_t)L->nhb * BP_HEADS * TC_H * 4);
  L->gs_part = take((size_t)L->nhb * (BP_HEADS + 3) * 8);
  L->sc = take(sizeof(BpttScalars));
  const int NC = 384 + L->np;
  L->G = take((size_t)512 * NC * 8);
  L->Y = take((size_t)TC_H * L->np * 8);
  L->GSC = take((size_t)512 * TC_H * 8);
  L->dC = take((size_t)TC_H * TC_H * 8);
  L->wj = take((size_t)512 * TC_H * 8);
  L->cw = take((size_t)TC_H * TC_H * 8);
  L->losses = take(3 * 8);
  L->total = off;
  return IC3_OK;
}

int env_geometry(const ic3_bptt_plan* p, int* npos, int* WW, int* is_tj) {
  if (p->pp_env) {
    const int W = 2 * p->pp_env->vision + 1;
    *npos = p->pp_env->dim * p->pp_env->dim;
    *WW = W * W;
    *is_tj = 0;
  } else if (p->tj_env) {
    const int W = 2 * p->tj_env->vision + 1;
    *npos = p->tj_env->h * p->tj_env->w;
    *WW = W * W;
    *is_tj = 1;
  } else {
    return IC3_E_NULL;
  }
  if (*WW > PREP_MAX_WW) return IC3_E_UNSUPPORTED;
  return IC3_OK;
}

}  // namespace

extern "C" uint64_t ic3_bptt_workspace_bytes(const ic3_bptt_plan* p) {
  if (!p || !p->cfg || p->cfg->H != TC_H) return 0;
  int npos, WW, is_tj;
  if (env_geometry(p, &npos, &WW, &is_tj)) return 0;
  Layout L;
  if (plan_layout(p->cfg, npos, WW, is_tj, &L)) return 0;
  int nout = 1;
  for (int k = 0; k < p->cfg->nheads; ++k) nout += p->cfg->head_dim[k];
  if (nout > BP_HEADS) return 0;
  return (uint64_t)L.total;
}

// Start of a compute_grad: zero the accumulators, build the dgrad weight image, set max |c|.
extern "C" int ic3_bptt_begin(const ic3_bptt_plan* p, float cmax, void* stream) {
  if (!p || !p->cfg || !p->w || !p->workspace) return IC3_E_NULL;
  int npos, WW, is_tj;
  int rc = env_geometry(p, &npos, &WW, &is_tj);
  if (rc) return rc;
  Layout L;
  rc = plan_layout(p->cfg, npos, WW, is_tj, &L);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned char* ws = reinterpret_cast<unsigned char*>(p->workspace);
  cudaError_t e = cudaMemsetAsync(ws + L.partial, 0, L.total - L.partial, s);   // partial .. end: all accumulators / scalars
  if (e != cudaSuccess) return (int)e;
  e = cudaMemsetAsync(ws + L.a_img, 0, L.w2_img - L.a_img, s);                  // both image sets
  if (e != cudaSuccess) return (int)e;
  bptt_pack_w2_kernel<<<(256 * 512 + 255) / 256, 256, 0, s>>>(reinterpret_cast<const __half*>(p->w->lstm_img),
                                                              reinterpret_cast<__half*>(ws + L.w2_img));
  IC3_LAUNCH_CHECK();
  BpttStreams* ss = bptt_streams();
  if (!ss) return IC3_E_UNSUPPORTED;
  ss->prepared_t[0] = ss->prepared_t[1] = -1;
  if (BpttTrace* tr = bptt_trace(); tr->on) {
    memset(tr->used, 0, sizeof(tr->used));
    tr->t_first = -1;
    cudaEventRecord(tr->base, s);
  }
  BpttScalars init;
  memset(&init, 0, sizeof(init));
  init.cmax = cmax;
  init.scale[0] = init.scale[1] = 1.f;
  init.inv_scale[0] = init.inv_scale[1] = 1.f;
  e = cudaMemcpyAsync(ws + L.sc, &init, sizeof(init), cudaMemcpyHostToDevice, s);
  if (e != cudaSuccess) return (int)e;
  // the look-ahead kernels of the first two steps (side stream) must see the zeroed accumulators -- and everything the
  // caller enqueued before this call (returns, advantages, the rollout records)
  for (int k = 0; k < 2; ++k) {
    e = cudaEventRecord(ss->main_done[k], s);
    if (e != cudaSuccess) return (int)e;
  }
  return IC3_OK;
}

// Recursion-independent part of a step: d loss / d outputs from the records (heads) and the operand images of the
// step (prep).  Runs on `s` into buffer set q = t & 1.
static int bptt_prepare_on(const ic3_bptt_plan* p, const ic3_bptt_step_io* io, const Layout& L, int npos, int is_tj,
                           cudaStream_t s) {
  const ic3_policy_cfg* cfg = p->cfg;
  unsigned char* ws = reinterpret_cast<unsigned char*>(p->workspace);
  const int R = cfg->B * cfg->N;
  int atot = 0;
  for (int k = 0; k < cfg->nheads; ++k) atot += cfg->head_dim[k];
  BpttScalars* sc = reinterpret_cast<BpttScalars*>(ws + L.sc);
  const int q = io->t & 1;
  const size_t rows_pad = (size_t)L.ntiles * TC_M;
  __half* a_img = reinterpret_cast<__half*>(ws + L.a_img + (size_t)q * L.img_stride);
  __half* p_img = reinterpret_cast<__half*>(ws + L.p_img + (size_t)q * L.img_stride);
  // ---- operand images of step t from the records ----
  ic3_policy_io pio;
  memset(&pio, 0, sizeof(pio));
  pio.h = io->h_prev; pio.c = io->c_prev; pio.comm_action = io->comm; pio.alive = io->alive; pio.fresh = io->fresh;
  pio.err = io->err;
  if (cfg->hard_attn && !io->comm) return IC3_E_NULL;
  PrepSrc src;
  memset(&src, 0, sizeof(src));
  src.wT = p->w->enc_wT; src.bias = p->w->enc_b; src.split = cfg->obs_vocab > 0; src.table = p->x_table;
  src.wflags = p->w->flags;
  if (!src.table || !src.split) return IC3_E_NULL;
  PrepBwd bw;
  bw.p_img = p_img;
  bw.gs = reinterpret_cast<float*>(ws + L.gs) + (size_t)q * rows_pad;
  bw.gr = reinterpret_cast<float*>(ws + L.gr) + (size_t)q * rows_pad;
  bw.npg = L.np / 8;
  bw.npos = npos;
  const int ntiles = L.ntiles;
  if (!is_tj) {
    if (!io->pp_loc) return IC3_E_NULL;
    src.pp = *p->pp_env;
    memset(&src.pps, 0, sizeof(src.pps));
    src.pps.loc = const_cast<int32_t*>(io->pp_loc);
    prep_kernel<XSRC_PP, true, true><<<2 * ntiles, PREP_THREADS, prep_T_bytes(cfg->N), s>>>(*cfg, pio, a_img, src, bw);
    IC3_LAUNCH_CHECK();
    trace_mark(1, io->t, s);
  } else {
    if (!io->tj_loc || !io->tj_alive || !io->tj_last_act || !io->tj_route_id) return IC3_E_NULL;
    src.tj = *p->tj_env;
    memset(&src.tjs, 0, sizeof(src.tjs));
    src.tjs.loc = const_cast<int32_t*>(io->tj_loc);
    src.tjs.alive = const_cast<uint8_t*>(io->tj_alive);
    src.tjs.last_act = const_cast<uint8_t*>(io->tj_last_act);
    src.tjs.route_id = const_cast<int32_t*>(io->tj_route_id);
    prep_kernel<XSRC_TJ, true, true><<<2 * ntiles, PREP_THREADS, prep_T_bytes(cfg->N), s>>>(*cfg, pio, a_img, src, bw);
    IC3_LAUNCH_CHECK();
  }
  // ---- heads ----
  HeadsArgs ha;
  memset(&ha, 0, sizeof(ha));
  ha.R = R; ha.N = cfg->N; ha.nheads = cfg->nheads; ha.atot = atot;
  for (int k = 0; k < IC3_MAX_HEADS; ++k) ha.head_dim[k] = cfg->head_dim[k];
  ha.value_coeff = p->value_coeff; ha.entr = p->entr;
  ha.logp = io->logp; ha.action = io->action; ha.value = io->value; ha.ret = io->ret; ha.adv = io->adv;
  ha.alive_post = io->alive_post; ha.valid = io->valid; ha.h_new = io->h_new; ha.head_w = p->w->head_w;
  ha.dout = reinterpret_cast<float*>(ws + L.dout) + (size_t)q * rows_pad * BP_HEADS;
  ha.gw_part = reinterpret_cast<float*>(ws + L.gw_part);
  ha.gs_part = reinterpret_cast<double*>(ws + L.gs_part);
  ha.sc = sc;
  ha.q = q;
  bptt_heads_kernel<<<L.nhb, 256, 0, s>>>(ha);
  IC3_LAUNCH_CHECK();
  trace_mark(0, io->t, s);
  return IC3_OK;
}

static int bptt_common(const ic3_bptt_plan* p, const ic3_bptt_step_io* io, Layout* L, int* npos, int* is_tj) {
  if (!p || !io || !p->cfg || !p->w || !p->workspace) return IC3_E_NULL;
  if (!io->h_prev || !io->c_prev || !io->h_new || !io->logp || !io->action || !io->value || !io->ret || !io->adv ||
      !io->alive_post || !io->dh || !io->dc)
    return IC3_E_NULL;
  if (p->cfg->H != TC_H) return IC3_E_UNSUPPORTED;
  int WW;
  int rc = env_geometry(p, npos, &WW, is_tj);
  if (rc) return rc;
  rc = plan_layout(p->cfg, *npos, WW, *is_tj, L);
  if (rc) return rc;
  int nout = 1;
  for (int k = 0; k < p->cfg->nheads; ++k) nout += p->cfg->head_dim[k];
  return nout > BP_HEADS ? IC3_E_UNSUPPORTED : IC3_OK;
}

// Optional: launch the recursion-independent kernels of step io->t (heads, operand images) AHEAD of ic3_bptt_step(t),
// on the library's side stream, so that they overlap the tensor-core kernels of step t + 1 (which leave one CTA slot
// per SM free).  `stream` is the stream ic3_bptt_step will be called on.  Without this call (or with
// IC3_BPTT_OVERLAP=0) ic3_bptt_step runs them itself.
extern "C" int ic3_bptt_prepare(const ic3_bptt_plan* p, const ic3_bptt_step_io* io, void* stream) {
  Layout L;
  int npos, is_tj;
  int rc = bptt_common(p, io, &L, &npos, &is_tj);
  if (rc) return rc;
  BpttStreams* ss = bptt_streams();
  if (!ss) return IC3_E_UNSUPPORTED;
  if (BpttTrace* tr = bptt_trace(); tr->on && tr->t_first < 0) tr->t_first = io->t;
  if (!ss->overlap) return IC3_OK;                  // ic3_bptt_step will do it inline
  const int q = io->t & 1;
  // buffer set q was last used by step t + 2: its main-stream kernels (gates / dgrad / comm read A, dout, gs, gr) and
  // its weight-gradient kernel (side stream, already ordered before this call)
  cudaError_t e = cudaStreamWaitEvent(ss->side, ss->main_done[q], 0);
  if (e != cudaSuccess) return (int)e;
  rc = bptt_prepare_on(p, io, L, npos, is_tj, ss->side);
  if (rc) return rc;
  e = cudaEventRecord(ss->prep_done[q], ss->side);
  if (e != cudaSuccess) return (int)e;
  ss->prepared_t[q] = io->t;
  return IC3_OK;
}

extern "C" int ic3_bptt_step(const ic3_bptt_plan* p, const ic3_bptt_step_io* io, void* stream) {
  Layout L;
  int npos, is_tj;
  int rc = bptt_common(p, io, &L, &npos, &is_tj);
  if (rc) return rc;
  const ic3_policy_cfg* cfg = p->cfg;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned char* ws = reinterpret_cast<unsigned char*>(p->workspace);
  const int R = cfg->B * cfg->N;
  int nout = 1;
  for (int k = 0; k < cfg->nheads; ++k) nout += cfg->head_dim[k];
  BpttScalars* sc = reinterpret_cast<BpttScalars*>(ws + L.sc);
  const int q = io->t & 1;
  const size_t rows_pad = (size_t)L.ntiles * TC_M;
  const int ntiles = L.ntiles;
  __half* a_img = reinterpret_cast<__half*>(ws + L.a_img + (size_t)q * L.img_stride);
  __half* dg_img = reinterpret_cast<__half*>(ws + L.dg_img + (size_t)q * L.img_stride);
  BpttStreams* ss = bptt_streams();
  if (!ss) return IC3_E_UNSUPPORTED;
  if (BpttTrace* tr = bptt_trace(); tr->on && tr->t_first < 0) tr->t_first = io->t;
  // buffer set q (images, scale) was last read by the weight-gradient kernel of step t + 2 (side stream)
  cudaError_t se = cudaStreamWaitEvent(s, ss->wgrad_done[q], 0);
  if (se != cudaSuccess) return (int)se;
  if (ss->prepared_t[q] == io->t) {                 // heads + images were launched ahead (ic3_bptt_prepare)
    se = cudaStreamWaitEvent(s, ss->prep_done[q], 0);
    if (se != cudaSuccess) return (int)se;
    ss->prepared_t[q] = -1;
  } else {
    rc = bptt_prepare_on(p, io, L, npos, is_tj, s);
    if (rc) return rc;
  }
  bptt_scale_kernel<<<1, 1, 0, s>>>(sc, q);
  IC3_LAUNCH_CHECK();
  trace_mark(2, io->t, s);

  // ---- gates ----
  {
    static bool cfgd = false;
    const size_t smem = NSTAGE_P * STAGE_BYTES + 256 + TC_H * HEAD_PAD * sizeof(float) + 4 * TC_H * sizeof(float);
    if (!cfgd) {
      cudaError_t e = cudaFuncSetAttribute(bptt_gates_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
      prefer_max_smem(bptt_gates_kernel);
      cfgd = true;
    }
    GatesArgs ga;
    ga.R = R; ga.N = cfg->N; ga.c_prev = io->c_prev; ga.fresh = io->fresh; ga.cut = io->cut;
    ga.dout = reinterpret_cast<const float*>(ws + L.dout) + (size_t)q * rows_pad * BP_HEADS; ga.dh = io->dh; ga.dc = io->dc; ga.dg_img = dg_img; ga.sc = sc;
    ga.q = q;
    ga.err = io->err;
    const int nitems = 2 * ntiles;
    const int grid = nitems < sm_count() ? nitems : sm_count();
    bptt_gates_kernel<<<grid, TC_P_THREADS, smem, s>>>(ga, a_img, reinterpret_cast<const __half*>(p->w->lstm_img),
                                                      (const float*)p->w->bias_cat, nitems, (const float*)p->w->head_w, nout);
    IC3_LAUNCH_CHECK();
    trace_mark(3, io->t, s);
    se = cudaEventRecord(ss->gates_done[q], s);
    if (se != cudaSuccess) return (int)se;
  }
  // ---- dgrad ----
  {
    static bool cfgd = false;
    const size_t smem = NSTAGE_P * DGR_STAGE + 256;
    if (!cfgd) {
      cudaError_t e = cudaFuncSetAttribute(bptt_dgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
      prefer_max_smem(bptt_dgrad_kernel);
      cfgd = true;
    }
    DgradArgs da;
    da.R = R; da.gs = reinterpret_cast<const float*>(ws + L.gs) + (size_t)q * rows_pad; da.dSs = reinterpret_cast<float*>(ws + L.dSs);
    da.dh_direct = reinterpret_cast<float*>(ws + L.dh_direct); da.sc = sc; da.q = q; da.err = io->err;
    const int grid = ntiles < sm_count() ? ntiles : sm_count();
    bptt_dgrad_kernel<<<grid, TC_P_THREADS, smem, s>>>(da, dg_img, reinterpret_cast<const __half*>(ws + L.w2_img), ntiles);
    IC3_LAUNCH_CHECK();
    trace_mark(4, io->t, s);
  }
  // ---- comm backward -> dh_{t-1} ----
  {
    CommArgs ca;
    ca.B = cfg->B; ca.N = cfg->N; ca.dSs = reinterpret_cast<const float*>(ws + L.dSs);
    ca.dh_direct = reinterpret_cast<const float*>(ws + L.dh_direct); ca.gr = reinterpret_cast<const float*>(ws + L.gr) + (size_t)q * rows_pad;
    ca.fresh = io->fresh; ca.no_comm = cfg->comm_mask_zero || cfg->N < 2; ca.dh = io->dh; ca.sc = sc;
    bptt_comm_kernel<<<(cfg->B + 7) / 8, 256, 0, s>>>(ca);
    IC3_LAUNCH_CHECK();
    trace_mark(5, io->t, s);
    se = cudaEventRecord(ss->main_done[q], s);          // buffer set q may be refilled for step t - 2 once wgrad(t) is done too
    if (se != cudaSuccess) return (int)se;
  }
  // ---- weight gradients: on the side stream, overlapping the small kernels of this and the next step ----
  {
    static bool cfgd = false;
    static CUtensorMap map_dg[2], map_a[2], map_p[2];
    static void* key_ws = nullptr;
    static int key_tiles = 0, key_np = 0;
    const size_t smem1 = (size_t)WG_NSTAGE1 * (2 * WG_DG_BYTES + (size_t)L.np * 64);
    const size_t smem = (size_t)WG_NSTAGE0 * WG_STAGE0 > smem1 ? (size_t)WG_NSTAGE0 * WG_STAGE0 : smem1;
    if (!cfgd) {
      cudaError_t e = cudaFuncSetAttribute(bptt_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      if (e != cudaSuccess) return (int)e;
      prefer_max_smem(bptt_wgrad_kernel);
      prefer_max_smem(bptt_heads_kernel);
      prefer_max_smem(bptt_comm_kernel);
      prefer_max_smem(prep_kernel<XSRC_PP, true, true>);
      prefer_max_smem(prep_kernel<XSRC_TJ, true, true>);
      cfgd = true;
    }
    if (smem > 200 * 1024) return IC3_E_UNSUPPORTED;
    if (key_ws != p->workspace || key_tiles != ntiles || key_np != L.np) {
      for (int k = 0; k < 2; ++k) {
        rc = make_image_map(&map_dg[k], ws + L.dg_img + (size_t)k * L.img_stride, ntiles, 2, 64, 16);
        if (rc) return rc;
        rc = make_image_map(&map_a[k], ws + L.a_img + (size_t)k * L.img_stride, ntiles, 2, 48, 48);
        if (rc) return rc;
        rc = make_image_map(&map_p[k], ws + L.p_img + (size_t)k * L.img_stride, ntiles, 0, L.np / 8, L.np / 8);
        if (rc) return rc;
      }
      key_ws = p->workspace; key_tiles = ntiles; key_np = L.np;
    }
    WgradArgs wa;
    wa.ntiles = ntiles; wa.np = L.np; wa.j0 = L.j0; wa.j1 = L.j1;
    wa.partial = reinterpret_cast<float*>(ws + L.partial); wa.sc = sc; wa.q = q; wa.err = io->err;
    cudaStream_t ws_stream = ss->overlap ? ss->side : s;
    if (ss->overlap) {
      se = cudaStreamWaitEvent(ws_stream, ss->gates_done[q], 0);
      if (se != cudaSuccess) return (int)se;
    }
    bptt_wgrad_kernel<<<L.ncta_wg, WG_THREADS, smem, ws_stream>>>(wa, map_dg[q], map_a[q], map_p[q]);
    IC3_LAUNCH_CHECK();
    trace_mark(6, io->t, ws_stream);
    se = cudaEventRecord(ss->wgrad_done[q], ws_stream);
    if (se != cudaSuccess) return (int)se;
  }
  return IC3_OK;
}

// After step 0: fold the accumulators into the parameter gradients (added to what the buffers hold) and return the
// three loss sums (action_loss, value_loss, entropy) in losses[3] (device, float64).
extern "C" int ic3_bptt_finish(const ic3_bptt_plan* p, const ic3_policy_params* params, const ic3_policy_params* grads,
                               double* losses, void* stream) {
  if (!p || !params || !grads || !losses || !p->cfg || !p->workspace) return IC3_E_NULL;
  const ic3_policy_cfg* cfg = p->cfg;
  int npos, WW, is_tj;
  int rc = env_geometry(p, &npos, &WW, &is_tj);
  if (rc) return rc;
  Layout L;
  rc = plan_layout(cfg, npos, WW, is_tj, &L);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned char* ws = reinterpret_cast<unsigned char*>(p->workspace);
  if (BpttStreams* ss = bptt_streams()) {       // the last weight-gradient kernels may still run on the side stream
    for (int k = 0; k < 2; ++k) {
      cudaError_t e = cudaStreamWaitEvent(s, ss->wgrad_done[k], 0);
      if (e != cudaSuccess) return (int)e;
    }
  }
  const int NC = 384 + L.np;
  double* G = reinterpret_cast<double*>(ws + L.G);
  double* Y = reinterpret_cast<double*>(ws + L.Y);
  double* GSC = reinterpret_cast<double*>(ws + L.GSC);
  double* dC = reinterpret_cast<double*>(ws + L.dC);
  double* wj = reinterpret_cast<double*>(ws + L.wj);
  double* cw = reinterpret_cast<double*>(ws + L.cw);
  bptt_reduce_partials_kernel<<<(512 * NC + 255) / 256, 256, 0, s>>>(reinterpret_cast<const float*>(ws + L.partial), L.j0, L.j1,
                                                                     L.np, G, NC);
  IC3_LAUNCH_CHECK();
  bptt_weights_f64_kernel<<<(512 * TC_H + 255) / 256, 256, 0, s>>>(params->w_ih, params->c_w, wj, cw);
  IC3_LAUNCH_CHECK();
  // Y[k][n] = sum_j W_ih[j][k] Q[j][n],  Q = G[:, 384:]
  small_gemm_tn_kernel<<<(TC_H * L.np + 255) / 256, 256, 0, s>>>(TC_H, L.np, 512, wj, TC_H, G + 384, NC, Y, L.np, 0);
  IC3_LAUNCH_CHECK();
  // dC[k][m] = sum_j W_ih[j][k] G_S[j][m]
  small_gemm_tn_kernel<<<(TC_H * TC_H + 255) / 256, 256, 0, s>>>(TC_H, TC_H, 512, wj, TC_H, G + 128, NC, dC, TC_H, 0);
  IC3_LAUNCH_CHECK();
  bptt_gsc_kernel<<<(512 * TC_H + 255) / 256, 256, 0, s>>>(G, NC, cw, GSC);
  IC3_LAUNCH_CHECK();
  FinishArgs f;
  memset(&f, 0, sizeof(f));
  int atot = 0;
  for (int k = 0; k < cfg->nheads; ++k) atot += cfg->head_dim[k];
  f.O = cfg->O; f.nheads = cfg->nheads; f.atot = atot; f.npos = npos; f.np = L.np; f.WW = WW;
  for (int k = 0; k < IC3_MAX_HEADS; ++k) f.head_dim[k] = cfg->head_dim[k];
  f.G = G; f.NC = NC; f.Y = Y; f.GSC = GSC; f.dC = dC; f.c_b = params->c_b;
  f.g_w_ih = const_cast<float*>(grads->w_ih); f.g_w_hh = const_cast<float*>(grads->w_hh);
  f.g_b_ih = const_cast<float*>(grads->b_ih); f.g_b_hh = const_cast<float*>(grads->b_hh);
  f.g_c_w = const_cast<float*>(grads->c_w); f.g_c_b = const_cast<float*>(grads->c_b);
  f.g_enc_w = const_cast<float*>(grads->encoder_w); f.g_enc_b = const_cast<float*>(grads->encoder_b);
  f.g_value_w = const_cast<float*>(grads->value_w); f.g_value_b = const_cast<float*>(grads->value_b);
  for (int k = 0; k < IC3_MAX_HEADS; ++k) {
    f.g_head_w[k] = const_cast<float*>(grads->head_w[k]);
    f.g_head_b[k] = const_cast<float*>(grads->head_b[k]);
  }
  f.gw_part = reinterpret_cast<const float*>(ws + L.gw_part);
  f.gs_part = reinterpret_cast<const double*>(ws + L.gs_part);
  f.nhb = L.nhb;
  f.losses = losses;
  f.is_tj = is_tj;
  if (is_tj) f.tj = *p->tj_env;
  else f.pp = *p->pp_env;
  f.ones_col = npos + (is_tj ? WW + 3 : 2 * WW);     // the constant column of P is its last used column
  bptt_finish_lstm_kernel<<<(512 * TC_H + 255) / 256, 256, 0, s>>>(f);
  IC3_LAUNCH_CHECK();
  const int items = npos * WW > (is_tj ? WW + 3 : 2 * WW) ? npos * WW : (is_tj ? WW + 3 : 2 * WW);
  bptt_finish_misc_kernel<<<(items * 128 + 255) / 256, 256, 0, s>>>(f);
  IC3_LAUNCH_CHECK();
  bptt_finish_heads_kernel<<<(BP_HEADS * TC_H + 255) / 256, 256, 0, s>>>(f);
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}

// Development aid: end time (us after ic3_bptt_begin) of every traced kernel, [TR_STEPS][TR_KERNELS], -1 = not recorded.
// Not part of the C ABI; only meaningful with IC3_BPTT_TRACE=1.
extern "C" int ic3_debug_bptt_trace(float* out) {
  BpttTrace* tr = bptt_trace();
  if (!tr->on) return IC3_E_UNSUPPORTED;
  cudaDeviceSynchronize();
  for (int i = 0; i < TR_STEPS; ++i)
    for (int k = 0; k < TR_KERNELS; ++k) {
      float ms = -1.f;
      if (tr->used[i][k] && cudaEventElapsedTime(&ms, tr->base, tr->ev[i][k]) != cudaSuccess) ms = -1.f;
      out[i * TR_KERNELS + k] = ms < 0.f ? -1.f : ms * 1000.f;
    }
  return IC3_OK;
}
