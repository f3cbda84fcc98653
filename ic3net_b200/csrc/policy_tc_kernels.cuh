// Kernels of the tcgen05 policy path (see policy_tc.cu for the overview).  Included by policy_tc.cu (rollout
// forward) and bptt_tc.cu (backward), each inside its own anonymous namespace.
#pragma once
#include <cuda_fp16.h>

#include <cstdlib>
#include <cstring>

#include "ic3_common.cuh"
#include "policy_internal.h"
#include "tc_common.cuh"

namespace {

constexpr int TC_H = 128;
constexpr int TC_K = 384;               // [x | S | h]
constexpr int TC_KC = 32;               // K per pipeline stage
constexpr int TC_NCHUNK = TC_K / TC_KC; // 12
constexpr int TC_M = 128;               // rows per tile
constexpr int TC_NH = 256;              // gate columns per CTA (64 hidden units x i,f,g,o)
constexpr int A_CHUNK_BYTES = 2 * TC_M * TC_KC * 2;   // hi + lo = 16384
constexpr int B_CHUNK_BYTES = 2 * TC_NH * TC_KC * 2;  // 32768
constexpr int STAGE_BYTES = A_CHUNK_BYTES + B_CHUNK_BYTES;
constexpr int A_TILE_HALFS = TC_NCHUNK * A_CHUNK_BYTES / 2;   // 98304

// ---- image addressing (in halfs) ---------------------------------------------------------
// A image: [tile][part = hi, lo][fg = k >> 3 (48)][rg = r >> 3 (16)][r & 7][k & 7].  Uniform strides in both
// directions (feature group 2048 B, row group 128 B), so the SAME bytes serve as a K-major operand of the
// forward / backward GEMMs that contract over features (a pipeline chunk of 32 features = 4 consecutive feature
// groups = one contiguous 8 KB piece per part) and as an MN-major operand of the weight-gradient GEMM that
// contracts over rows (bptt_tc.cu).
__host__ __device__ __forceinline__ size_t a_img_off(int tile, int k, int r, int part) {
  return (size_t)tile * A_TILE_HALFS + (size_t)part * (A_TILE_HALFS / 2) + ((size_t)(k >> 3) * 16 + (r >> 3)) * 64 + (r & 7) * 8 +
         (k & 7);
}
__host__ __device__ __forceinline__ size_t b_img_off(int nh, int k, int n, int part) {
  const int c = k >> 5, kk = k & 31;
  return ((((((size_t)(nh * TC_NCHUNK + c) * 2 + part) * 4 + (kk >> 3)) * 32 + (n >> 3)) * 8 + (n & 7)) * 8) + (kk & 7);
}

constexpr size_t B_IMG_HALFS = (size_t)2 * TC_NCHUNK * B_CHUNK_BYTES / 2;   // one weight image, in halfs

// ---- weight images (once per optimizer step) ------------------------------------------------
__global__ void pack_tc_kernel(ic3_policy_params p, __half* __restrict__ img, float* __restrict__ bias_cat,
                               int32_t* __restrict__ flags) {
  const int H = TC_H;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;      // (col, k)
  if (idx < 4 * H * TC_K) {
    const int col = idx / TC_K, k = idx - col * TC_K;
    const int u = col >> 2, g = col & 3, row = g * H + u;       // column 4*u+gate <- LSTMCell row g*H+u
    double w;
    if (k < H) {
      w = p.w_ih[(size_t)row * H + k];
    } else if (k < 2 * H) {                                     // (W_ih . C)[row][k-H]
      double acc = 0.0;
      for (int m = 0; m < H; ++m) acc += (double)p.w_ih[(size_t)row * H + m] * (double)p.c_w[(size_t)m * H + (k - H)];
      w = acc;
    } else {
      w = p.w_hh[(size_t)row * H + (k - 2 * H)];
    }
    __half hi, lo;
    split_f16((float)w, SCALE_B, hi, lo);
    if (flags && !(fabs(w) * SCALE_B < 65504.0)) atomicOr(flags, IC3_ERR_FP16_RANGE);   // also catches NaN
    const int nh = col >> 8, n = col & 255;
    img[b_img_off(nh, k, n, 0)] = hi;
    img[b_img_off(nh, k, n, 1)] = lo;
  }
  if (idx < 4 * H) {
    const int u = idx >> 2, g = idx & 3, row = g * H + u;
    double acc = (double)p.b_ih[row] + (double)p.b_hh[row];
    for (int m = 0; m < H; ++m) acc += (double)p.w_ih[(size_t)row * H + m] * (double)p.c_b[m];
    bias_cat[idx] = (float)acc;
  }
}

// ---- operand A image: x | S | h (every step) ---------------------------------------------------
// One CTA per 128-row tile.  Phase 1 forms, per environment touching the tile, the gated sum
// T = sum_j g_j h_j (comm.py:181-205) in shared memory (environments may straddle tiles: their
// other rows are read straight from global memory); phase 2 streams the tile: a warp item is
// 8 rows x 4 float4 columns so every store instruction writes two complete 128-byte core
// matrices, with S_k = g_k (T - h_k) / (n_alive - 1).
constexpr int PREP_ROWS = 64;      // rows per CTA (half a tile): 2 x more CTAs in flight than tiles
constexpr int PREP_THREADS = 160;  // 40 registers x 160 threads -> 10 CTAs/SM: the 1280 half-tile CTAs of a c2 step form ONE wave on 148 SMs (256 threads: 8 CTAs/SM = 1184 slots, a second wave of 96 CTAs)
__host__ __device__ inline size_t prep_T_bytes(int N) { return (size_t)(PREP_ROWS / N + 2) * TC_H * sizeof(float); }
constexpr int PREP_MAX_WW = 25;    // window cells (vision <= 2) the fused index encoder supports
constexpr int PREP_X_BYTES = PREP_ROWS * TC_H * 4;   // shared-memory x tile of the fused index encoder

// Where the encoder output x comes from: a [R,H] fp32 tensor, or -- fused index encoder -- straight from the
// environment state (same sum, same order as *_encoder_index_kernel / encoder_dense_kernel -> bit-identical x).
enum { XSRC_TENSOR = 0, XSRC_PP = 1, XSRC_TJ = 2 };
struct PrepSrc {
  ic3_pp_cfg pp;
  ic3_pp_state pps;
  ic3_tj_cfg tj;
  ic3_tj_state tjs;
  const float* wT;     // encoder.weight^T [O, H]
  const float* bias;   // [H]
  const float* table;  // [positions, H] class part of the sum per agent position (ic3_*_encoder_table) or NULL
  int split;           // ic3_policy_cfg.obs_vocab > 0: class terms and count / scalar terms are summed separately
  const int32_t* wflags;   // ic3_policy_packed.flags (weight range check of the pack kernel) or NULL
};

__device__ __forceinline__ void fma4(float4& a, float v, const float4 w) {
  a.x = fmaf(v, w.x, a.x); a.y = fmaf(v, w.y, a.y); a.z = fmaf(v, w.z, a.z); a.w = fmaf(v, w.w, a.w);
}

// accumulate into `a` when sel, else into `b` (both stay in registers)
__device__ __forceinline__ void fma4_sel(bool sel, float4& a, float4& b, float v, const float4 w) {
  if (sel) fma4(a, v, w);
  else fma4(b, v, w);
}

// TAB: the class part of x comes from the per-position table (src.table); the fused encoder then needs neither
// the x tile in shared memory nor the class feature indices, only the sparse count terms of each row.
// Extra outputs of the operand-preparation kernel when it runs inside the backward pass (bptt_tc.cu):
//   p_img  "feature" operand of the weight-gradient GEMM, [tile][pg = column >> 3][rg 16][8 rows][8 columns] fp16:
//          the NON-ZERO pattern of the observation row as exact small numbers -- one-hot agent position (columns
//          [0, npos)), the count features of the window cells, the scalar features, and a constant 1 (bias column);
//          d(loss)/d(encoder weights) = (d gates)^T . P folded with W_ih afterwards, so the [R, O] observation is
//          never materialised in the backward pass either
//   gs, gr per-row comm gate factors g / den and g of comm.py:181-205 (needed by the comm backward)
struct PrepBwd {
  __half* p_img;
  float* gs;
  float* gr;
  int npg;      // column groups of P (columns padded to a multiple of 16)
  int npos;     // positions (dim*dim or h*w): first column after the one-hot block
};

template <int XSRC, bool TAB, bool BWD = false>
__global__ void __launch_bounds__(256) prep_kernel(ic3_policy_cfg cfg, ic3_policy_io io, __half* __restrict__ img,
                                                   PrepSrc src, PrepBwd bw) {
  static_assert(!(TAB && XSRC == XSRC_TENSOR), "the table belongs to the fused index encoder");
  static_assert(!BWD || TAB, "the backward pass uses the per-position table form of the encoder");
  __shared__ float s_gate[PREP_ROWS + 64];
  __shared__ float s_den[PREP_ROWS + 64];
  // s_T: gated hidden-state sum of every environment touching this CTA's rows, [PREP_ROWS / N + 2][H] floats at the
  // start of the dynamic shared memory (sized by the launcher: a static [34][H] array would cap the kernel at 8 CTAs/SM)
  // fused index encoder: per (row, window cell) the feature index of the one-hot class and the counts
  __shared__ int s_feat[(XSRC == XSRC_TENSOR || TAB) ? 1 : PREP_ROWS * PREP_MAX_WW];
  __shared__ int s_cnt[XSRC == XSRC_TENSOR ? 1 : PREP_ROWS * PREP_MAX_WW];
  __shared__ unsigned s_mask[TAB ? PREP_ROWS : 1];    // window cells of the row that hold a count
  __shared__ int s_pos[TAB ? PREP_ROWS : 1];          // table row of the agent (-1: observation is all zero)
  __shared__ float s_la[XSRC == XSRC_TJ ? PREP_ROWS : 1], s_ri[XSRC == XSRC_TJ ? PREP_ROWS : 1];
  __shared__ int s_live[XSRC == XSRC_TJ ? PREP_ROWS : 1];
  extern __shared__ __align__(16) float s_dyn[];
  float (*s_T)[TC_H] = reinterpret_cast<float (*)[TC_H]>(s_dyn);
  float* s_x = s_dyn + (size_t)(PREP_ROWS / cfg.N + 2) * TC_H;   // [PREP_ROWS][H] encoder output (index sources without table)
  const int N = cfg.N;
  const int R = cfg.B * N;
  const int tile = blockIdx.x >> 1, hb = blockIdx.x & 1;
  const int row0 = tile * TC_M + hb * PREP_ROWS;
  if (TAB) {
    if (threadIdx.x < PREP_ROWS) s_mask[threadIdx.x] = 0u;
    __syncthreads();
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && src.wflags && io.err && *src.wflags) atomicOr(io.err, *src.wflags);
  for (int w = threadIdx.x; w < PREP_ROWS + 64; w += blockDim.x) {
    const int row = row0 - 32 + w;
    float g = 0.f, den = 1.f;
    if (row >= 0 && row < R) {
      const int e = row / N, i = row - e * N;
      const bool fr = io.fresh && io.fresh[e];
      int n_alive = N, al = 1;
      if (io.alive && !fr) {                       // comm.py:102-104
        n_alive = 0;
        for (int j = 0; j < N; ++j) n_alive += io.alive[(size_t)e * N + j] != 0;
        al = io.alive[(size_t)e * N + i] != 0;
      }
      int cm = 1;
      if (cfg.hard_attn) cm = fr ? 0 : (io.comm_action[(size_t)e * N + i] != 0);   // comm.py:171-175
      // episode start: every agent of the env has h = 0 (trainer.py:50-51) -> nothing to send in the first comm pass
      g = (fr && io.pass_index == 0) ? 0.f : (float)(al * cm);
      if (cfg.comm_avg && n_alive > 1) den = (float)(n_alive - 1);                  // comm.py:194-196
    }
    s_gate[w] = g;
    s_den[w] = den;
  }
  if (XSRC == XSRC_PP) {          // predator_prey_env.py:188-210
    const int D = src.pp.dim, v = src.pp.vision, W = 2 * v + 1, WW = W * W, V = D * D + 4;
    const int NP = src.pp.N;      // predators; agent row NP (present with enemy_comm: N == NP + 1) is the prey
    for (int p = threadIdx.x; p < PREP_ROWS * WW; p += blockDim.x) {
      const int rl = p / WW, w = p - rl * WW, row = row0 + rl;
      int feat = 0, cnt = 0;
      if (row < R) {
        const int e = row / N, i = row - e * N;
        const int* l = src.pps.loc + (size_t)e * (NP + 1) * 2;
        const int dy = w / W, dx = w - dy * W;
        const int rr = l[2 * i] - v + dy, cc = l[2 * i + 1] - v + dx;
        if (rr >= 0 && rr < D && cc >= 0 && cc < D) {
          int npred = 0;
          for (int j = 0; j < NP; ++j) npred += (l[2 * j] == rr && l[2 * j + 1] == cc);
          const int nprey = (l[2 * NP] == rr && l[2 * NP + 1] == cc);
          feat = w * V + rr * D + cc;
          cnt = npred | (nprey << 8);
        } else {
          feat = w * V + V - 3;                          // OUTSIDE class
        }
        if (TAB && w == 0) s_pos[rl] = l[2 * i] * D + l[2 * i + 1];
      } else if (TAB && w == 0) {
        s_pos[rl] = -1;
      }
      if (!TAB) s_feat[rl * WW + w] = feat;
      s_cnt[rl * WW + w] = cnt;
      if (TAB && cnt) atomicOr(&s_mask[rl], 1u << w);
    }
  } else if (XSRC == XSRC_TJ) {   // traffic_junction_env.py:321-366
    const int v = src.tj.vision, W = 2 * v + 1, WW = W * W, V = src.tj.vocab;
    for (int rl = threadIdx.x; rl < PREP_ROWS; rl += blockDim.x) {
      const int row = row0 + rl;
      int live = 0;
      float la = 0.f, ri = 0.f;
      if (row < R) {
        live = src.tjs.alive[row] != 0;
        la = (float)src.tjs.last_act[row];
        ri = (float)src.tjs.route_id[row] / (float)(src.tj.npath - 1);
      }
      s_live[rl] = live; s_la[rl] = la; s_ri[rl] = ri;
    }
    for (int p = threadIdx.x; p < PREP_ROWS * WW; p += blockDim.x) {
      const int rl = p / WW, w = p - rl * WW, row = row0 + rl;
      int feat = 0, cnt = 0;
      if (row < R) {
        const int e = row / N;
        const int* l = src.tjs.loc + (size_t)e * N * 2;
        const int i = row - e * N;
        const int dy = w / W, dx = w - dy * W;
        const int rr = l[2 * i] - v + dy, cc = l[2 * i + 1] - v + dx;
        int cls = src.tj.outside_cls;
        if (rr >= 0 && rr < src.tj.h && cc >= 0 && cc < src.tj.w) {
          cls = src.tj.grid[rr * src.tj.w + cc];
          for (int j = 0; j < N; ++j) cnt += (l[2 * j] == rr && l[2 * j + 1] == cc);
        }
        feat = 2 + w * V + cls;
        if (TAB && w == 0) s_pos[rl] = src.tjs.alive[row] ? l[2 * i] * src.tj.w + l[2 * i + 1] : -1;
        if (TAB && !src.tjs.alive[row]) cnt = 0;         // dead car: all-zero observation
      } else if (TAB && w == 0) {
        s_pos[rl] = -1;
      }
      if (!TAB) s_feat[rl * WW + w] = feat;
      s_cnt[rl * WW + w] = cnt;
      if (TAB && cnt) atomicOr(&s_mask[rl], 1u << w);
    }
  }
  __syncthreads();
  if (XSRC != XSRC_TENSOR && !TAB) {
    // comm.py:119 on the one-hot observation, never materialised: warp per row, lane = 4 consecutive hidden
    // units, every weight-row read is one coalesced 512-byte request; x lands in shared memory.
    // xv = bias + class terms, x2 = count / scalar terms when the layout hint asks for separate sums (else they join
    // xv, in feature order).  (With the per-position table this whole phase is skipped: TAB specialisation below.)
    const int gw = threadIdx.x >> 5, gl = threadIdx.x & 31;
    const float4* wq = reinterpret_cast<const float4*>(src.wT) + gl;
    const bool split = src.split != 0;
    for (int rl = gw; rl < PREP_ROWS; rl += (blockDim.x >> 5)) {
      float4 xv = __ldg(reinterpret_cast<const float4*>(src.bias) + gl);
      float4 x2 = make_float4(0.f, 0.f, 0.f, 0.f);
      const int row = row0 + rl;
      if (row < R) {
        if (XSRC == XSRC_PP) {
          const int W = 2 * src.pp.vision + 1, WW = W * W, V = src.pp.dim * src.pp.dim + 4;
          for (int w = 0; w < WW; ++w) {
            const int feat = s_feat[rl * WW + w], cnt = s_cnt[rl * WW + w];
            fma4(xv, 1.f, __ldg(wq + (size_t)feat * (TC_H / 4)));
            if (cnt >> 8) fma4_sel(split, x2, xv, (float)(cnt >> 8), __ldg(wq + (size_t)(w * V + V - 2) * (TC_H / 4)));     // PREY
            if (cnt & 255) fma4_sel(split, x2, xv, (float)(cnt & 255), __ldg(wq + (size_t)(w * V + V - 1) * (TC_H / 4)));  // PREDATOR
          }
        } else if (s_live[rl]) {
          const int W = 2 * src.tj.vision + 1, WW = W * W, V = src.tj.vocab;
          if (s_la[rl] != 0.f) fma4_sel(split, x2, xv, s_la[rl], __ldg(wq));
          if (s_ri[rl] != 0.f) fma4_sel(split, x2, xv, s_ri[rl], __ldg(wq + (TC_H / 4)));
          for (int w = 0; w < WW; ++w) {
            const int feat = s_feat[rl * WW + w], cnt = s_cnt[rl * WW + w];
            fma4(xv, 1.f, __ldg(wq + (size_t)feat * (TC_H / 4)));
            if (cnt) fma4_sel(split, x2, xv, (float)cnt, __ldg(wq + (size_t)(2 + w * V + src.tj.car_cls) * (TC_H / 4)));
          }
        }
      }
      xv.x += x2.x; xv.y += x2.y; xv.z += x2.z; xv.w += x2.w;
      *reinterpret_cast<float4*>(&s_x[rl * TC_H + 4 * gl]) = xv;
    }
  }
  const int e_first = row0 / N;
  const int last_row = min(R, row0 + PREP_ROWS) - 1;
  const bool want_s = !cfg.comm_mask_zero && N >= 2 && last_row >= row0;
  if (want_s) {
    const int nenv = last_row / N - e_first + 1;
    for (int idx = threadIdx.x; idx < nenv * (TC_H / 4); idx += blockDim.x) {
      const int el = idx >> 5, q = idx & 31;
      const int base = (e_first + el) * N;
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int j = 0; j < N; ++j) {
        if (s_gate[base + j - row0 + 32] != 0.f) {
          const float4 o = __ldg(reinterpret_cast<const float4*>(io.h + (size_t)(base + j) * TC_H) + q);
          t.x += o.x; t.y += o.y; t.z += o.z; t.w += o.w;
        }
      }
      *reinterpret_cast<float4*>(&s_T[el][4 * q]) = t;
    }
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (BWD) {
    // row factors of the comm backward
    for (int rl = threadIdx.x; rl < PREP_ROWS; rl += blockDim.x) {
      const int row = row0 + rl;
      if (row < R) {
        bw.gs[row] = s_gate[rl + 32] / s_den[rl + 32];
        bw.gr[row] = s_gate[rl + 32];
      }
    }
    // P image of this CTA's 8 row groups: one core matrix (8 rows x 8 columns, 128 B) per warp iteration,
    // lane = (row r8 = lane >> 2, column pair 2 * (lane & 3)) -> every store instruction writes one whole core matrix
    const int WW = XSRC == XSRC_PP ? (2 * src.pp.vision + 1) * (2 * src.pp.vision + 1)
                                   : (2 * src.tj.vision + 1) * (2 * src.tj.vision + 1);
    const int r8 = lane >> 2, c2 = (lane & 3) * 2;
    for (int cm = warp; cm < bw.npg * 8; cm += (blockDim.x >> 5)) {
      const int pg = cm >> 3, rgl = cm & 7;
      const int rl = rgl * 8 + r8, row = row0 + rl;
      float v[2] = {0.f, 0.f};
      if (row < R) {
        const int pos = s_pos[rl];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int col = pg * 8 + c2 + j;
          if (col < bw.npos) {
            v[j] = (col == pos) ? 1.f : 0.f;
          } else {
            const int idx = col - bw.npos;
            if (XSRC == XSRC_PP) {        // [prey count, predator count] per window cell, then the constant
              if (idx < 2 * WW) {
                const int cnt = s_cnt[rl * WW + (idx >> 1)];
                v[j] = (float)((idx & 1) ? (cnt & 255) : (cnt >> 8));
              } else if (idx == 2 * WW) {
                v[j] = 1.f;
              }
            } else if (XSRC == XSRC_TJ) { // car count per window cell, last_act, route id ratio (hi, lo), the constant
              if (idx < WW) v[j] = pos >= 0 ? (float)s_cnt[rl * WW + idx] : 0.f;
              else if (idx == WW) v[j] = pos >= 0 ? s_la[rl] : 0.f;
              else if (idx == WW + 1) v[j] = pos >= 0 ? __half2float(__float2half_rn(s_ri[rl])) : 0.f;
              else if (idx == WW + 2) v[j] = pos >= 0 ? s_ri[rl] - __half2float(__float2half_rn(s_ri[rl])) : 0.f;
              else if (idx == WW + 3) v[j] = 1.f;
            }
          }
        }
      }
      const size_t off = (((size_t)tile * bw.npg + pg) * 16 + (hb * 8 + rgl)) * 64 + r8 * 8 + c2;
      *reinterpret_cast<__half2*>(bw.p_img + off) = __floats2half2_rn(v[0], v[1]);
    }
  }
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  const size_t tile_base = (size_t)tile * A_TILE_HALFS;
#pragma unroll 2
  for (int item = warp; item < 64; item += (blockDim.x >> 5)) {
    const int rcl = item & 7, qg = item >> 3;
    const int r8 = lane & 7, q = qg * 4 + (lane >> 3);
    const int rl = rcl * 8 + r8;                 // row inside this CTA's 64 rows
    const int rc = hb * 8 + rcl;                 // 8-row group inside the 128-row tile
    const int row = row0 + rl;
    float4 xv = zero4, hv = zero4, sv = zero4;
    if (row < R) {
      const int e = row / N;
      const bool fr = io.fresh && io.fresh[e] && io.pass_index == 0;     // zero state: first comm pass only
      if (XSRC == XSRC_TENSOR) {
        xv = __ldg(reinterpret_cast<const float4*>(io.x + (size_t)row * TC_H) + q);
      } else if (!TAB) {
        xv = *reinterpret_cast<const float4*>(&s_x[rl * TC_H + 4 * q]);
      } else {
        // x = table[position] + (count / scalar terms in feature order): the same additions as the gather above
        const int pos = s_pos[rl];
        xv = __ldg(reinterpret_cast<const float4*>(pos >= 0 ? src.table + (size_t)pos * TC_H : src.bias) + q);
        float4 x2 = zero4;
        const float4* wq = reinterpret_cast<const float4*>(src.wT) + q;
        if (XSRC == XSRC_PP) {
          const int W = 2 * src.pp.vision + 1, WW = W * W, V = src.pp.dim * src.pp.dim + 4;
          for (unsigned m = s_mask[rl]; m; m &= m - 1) {
            const int w = __ffs(m) - 1, cnt = s_cnt[rl * WW + w];
            if (cnt >> 8) fma4(x2, (float)(cnt >> 8), __ldg(wq + (size_t)(w * V + V - 2) * (TC_H / 4)));     // PREY
            if (cnt & 255) fma4(x2, (float)(cnt & 255), __ldg(wq + (size_t)(w * V + V - 1) * (TC_H / 4)));  // PREDATOR
          }
        } else if (pos >= 0) {
          const int W = 2 * src.tj.vision + 1, WW = W * W, V = src.tj.vocab;
          if (s_la[rl] != 0.f) fma4(x2, s_la[rl], __ldg(wq));
          if (s_ri[rl] != 0.f) fma4(x2, s_ri[rl], __ldg(wq + (TC_H / 4)));
          for (unsigned m = s_mask[rl]; m; m &= m - 1) {
            const int w = __ffs(m) - 1;
            fma4(x2, (float)s_cnt[rl * WW + w], __ldg(wq + (size_t)(2 + w * V + src.tj.car_cls) * (TC_H / 4)));
          }
        }
        xv.x += x2.x; xv.y += x2.y; xv.z += x2.z; xv.w += x2.w;
      }
      if (!fr) hv = __ldg(reinterpret_cast<const float4*>(io.h + (size_t)row * TC_H) + q);
      if (want_s && s_gate[rl + 32] != 0.f) {      // gate 1 => own h is part of T
        const float4 t = *reinterpret_cast<const float4*>(&s_T[e - e_first][4 * q]);
        const float inv = 1.f / s_den[rl + 32];
        sv.x = (t.x - hv.x) * inv; sv.y = (t.y - hv.y) * inv; sv.z = (t.z - hv.z) * inv; sv.w = (t.w - hv.w) * inv;
      }
    }
    {   // operand split range (|a| * 16 must stay inside fp16): flag instead of silently saturating to inf
      const float m = fmaxf(fmaxf(fmaxf(fabsf(xv.x), fabsf(xv.y)), fmaxf(fabsf(xv.z), fabsf(xv.w))),
                            fmaxf(fmaxf(fmaxf(fabsf(hv.x), fabsf(hv.y)), fmaxf(fabsf(hv.z), fabsf(hv.w))),
                                  fmaxf(fmaxf(fabsf(sv.x), fabsf(sv.y)), fmaxf(fabsf(sv.z), fabsf(sv.w)))));
      if (!(m * SCALE_A < 65504.f) && io.err) atomicOr(io.err, IC3_ERR_FP16_RANGE);
    }
    // k = sec*128 + 4q  ->  feature group fg = sec*16 + (q >> 1), k & 7 = 4 * (q & 1)
    const size_t cell = tile_base + (size_t)(((q >> 1) * 16 + rc) * 64 + r8 * 8 + (q & 1) * 4);
    constexpr size_t LO = A_TILE_HALFS / 2, SEC = 16 * 1024;      // lo half of the tile; 16 feature groups per section
    store_split4(img, cell + 0 * SEC, cell + 0 * SEC + LO, xv, SCALE_A);
    store_split4(img, cell + 1 * SEC, cell + 1 * SEC + LO, sv, SCALE_A);
    store_split4(img, cell + 2 * SEC, cell + 2 * SEC + LO, hv, SCALE_A);
  }
}

// Gate non-linearities on the SFU, one ex2.approx (2^-22 rel.) + one rcp.approx (1 ulp) each, well inside the
// 1e-5 budget of the hidden state (tests/test_gpu_policy.py, tests/test_gpu_rollout.py).  The epilogue is the
// pacing stage of the kernel, so the forms are chosen for instruction count: the argument arrives already scaled
// by -log2(e) (folded into the accumulator scale and the shared-memory bias copy), and both functions are
// 1 / (1 + 2^t), see lstm_cell4.
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_fast(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr float LOG2E = 1.4426950408889634f;

// Gate biases pre-multiplied like the accumulator scale: (i, f, o) * -log2(e), g * -2 log2(e); [4H] in shared memory.
__device__ __forceinline__ void load_scaled_bias(float* s_bias, const float* __restrict__ bias_cat) {
  for (int idx = threadIdx.x; idx < 4 * TC_H; idx += blockDim.x)
    s_bias[idx] = __ldg(bias_cat + idx) * ((idx & 3) == 2 ? -2.f * LOG2E : -LOG2E);
}

// LSTM cell of 4 hidden units from 16 accumulator columns (column 4*u+gate): LSTMCell semantics of comm.py:194.
// The SFU (16 lanes/clk/SM) is the scarcest pipe of the epilogue, so reciprocals are shared: the four gates of a
// unit are 1/(1+2^t) with ONE rcp of the product of the four denominators (each 1/a recovered with FMA-pipe
// multiplies), and the four tanh(c') of the group share one more -- 6.25 SFU ops per hidden unit instead of 10.
// Exponents are clamped at 30 (denominators <= 2^30+1, products <= 2^121: no overflow); the clamp changes a
// sigmoid by < 1e-9.
__device__ __forceinline__ void lstm_cell4(const uint32_t (&v)[16], const float (&co)[4], const float* s_bias4,
                                           float (&cn)[4], float (&hn)[4]) {
  constexpr float SG = -INV_SCALE * LOG2E;
  constexpr float TMAX = 30.f;
  float go[4], bc[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 b = *reinterpret_cast<const float4*>(s_bias4 + 4 * j);
    const float ai = 1.f + ex2_fast(fminf(fmaf(__uint_as_float(v[4 * j + 0]), SG, b.x), TMAX));
    const float af = 1.f + ex2_fast(fminf(fmaf(__uint_as_float(v[4 * j + 1]), SG, b.y), TMAX));
    const float ag = 1.f + ex2_fast(fminf(fmaf(__uint_as_float(v[4 * j + 2]), 2.f * SG, b.z), TMAX));
    const float ao = 1.f + ex2_fast(fminf(fmaf(__uint_as_float(v[4 * j + 3]), SG, b.w), TMAX));
    const float p1 = ai * af, p2 = ag * ao;
    const float r = rcp_fast(p1 * p2);
    const float r1 = r * p2, r2 = r * p1;              // 1 / (ai af), 1 / (ag ao)
    const float gi = r1 * af, gf = r1 * ai;            // sigmoid(i), sigmoid(f)
    const float gg = fmaf(2.f, r2 * ao, -1.f);         // tanh(g) = 2 sigmoid(2g) - 1
    go[j] = r2 * ag;                                   // sigmoid(o)
    cn[j] = fmaf(gf, co[j], gi * gg);
    bc[j] = 1.f + ex2_fast(fminf(cn[j] * (-2.f * LOG2E), TMAX));
  }
  const float q1 = bc[0] * bc[1], q2 = bc[2] * bc[3];
  const float r = rcp_fast(q1 * q2);
  const float r1 = r * q2, r2 = r * q1;
  hn[0] = go[0] * fmaf(2.f, r1 * bc[1], -1.f);         // o * tanh(c')
  hn[1] = go[1] * fmaf(2.f, r1 * bc[0], -1.f);
  hn[2] = go[2] * fmaf(2.f, r2 * bc[3], -1.f);
  hn[3] = go[3] * fmaf(2.f, r2 * bc[2], -1.f);
}

// ---- the tensor-core kernel -----------------------------------------------------------------------
// Persistent, one CTA per SM, warp-specialised:
//   warp 16 producer   ring of NSTAGE (A 16 KB + B 32 KB) stages filled by cp.async.bulk, running
//                      ahead across work items
//   warp 17 MMA        one thread issues 3 x tcgen05.mma (128 x 256 x 16) per k-step into one of
//                      two 256-column TMEM accumulators
//   warps 0-15 epilogue warp w owns TMEM lanes 32*(w%4).. and columns 64*(w/4)..: LSTM cell of item i
//                      overlaps the MMAs of item i+1
// Work item = (128-row tile, 256-column half); item 2t and 2t+1 share the A tile (second read hits L2).
constexpr int NSTAGE_P = 4;
constexpr int HEAD_PAD = 8;          // outputs (value + action logits) the fused epilogue supports
constexpr int EPI_WARPS = 16;        // 4 warps per TMEM lane quarter, 64 accumulator columns (16 hidden units) each
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int TC_P_THREADS = EPI_THREADS + 64;   // + producer warp + MMA warp
constexpr int NSLOT = 8;             // partial-logit slots per row: (column half of the item) x (column quarter of the warp)

// Two adjacent lanes (rows 2k, 2k+1 of the tile) hold 8 consecutive floats of their own row each (a = first 4,
// b = last 4).  Written directly, every STG.128 of the warp touches 32 half-used 32-byte sectors; after one
// exchange the pair writes row 2k with one instruction and row 2k+1 with the next, 32 contiguous bytes each, so
// L2 sees whole sectors (half the write transactions; the kernel is paced by L2 transactions).
__device__ __forceinline__ void pair_store8(float* pe, float* po, const float (&a)[4], const float (&b)[4], bool ev, bool ov,
                                            bool odd) {
  float r[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) r[j] = __shfl_xor_sync(IC3_FULL_MASK, odd ? a[j] : b[j], 1);
  const float4 x1 = odd ? make_float4(r[0], r[1], r[2], r[3]) : make_float4(a[0], a[1], a[2], a[3]);
  const float4 x2 = odd ? make_float4(b[0], b[1], b[2], b[3]) : make_float4(r[0], r[1], r[2], r[3]);
  if (ev) *reinterpret_cast<float4*>(pe + (odd ? 4 : 0)) = x1;
  if (ov) *reinterpret_cast<float4*>(po + (odd ? 4 : 0)) = x2;
}

// Previous cell state of an epilogue thread's 16 hidden units (zero for a fresh episode).  Independent of the
// MMAs, so the caller issues it before waiting for the accumulator.  (Prefetching it one whole item ahead was
// measured: no gain -- the load is not on the critical path -- and the 16 extra live registers cost 4%.)
__device__ __forceinline__ void load_cold(const ic3_policy_cfg& cfg, const ic3_policy_io& io, int tile, int nh, int quarter,
                                          int cq, int lane, float4 (&cold)[4]) {
  const int R = cfg.B * cfg.N;
  const int row = tile * TC_M + quarter * 32 + lane;
  const bool inrange = row < R;
  bool fr = false;
  if (inrange && io.fresh && io.pass_index == 0) fr = io.fresh[row / cfg.N] != 0;
  const int ubase = nh * (TC_NH / 4) + cq * 16;
#pragma unroll
  for (int cg = 0; cg < 4; ++cg) {
    cold[cg] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (inrange && !fr) cold[cg] = *reinterpret_cast<const float4*>(io.c + (size_t)row * TC_H + ubase + cg * 4);
  }
}

// One work item of an epilogue thread = (row of the tile, 16 hidden units): LSTM cell from the finished
// accumulator, h'/c' stores, partial head logits.
__device__ __forceinline__ void epilogue_item(const ic3_policy_cfg& cfg, const ic3_policy_io& io, const float* s_bias,
                                              const float* s_hw, float* __restrict__ partial, uint32_t tmem_base,
                                              uint32_t bar_tfull, uint32_t bar_tempty, uint32_t li, int tile, int nh,
                                              int quarter, int cq, int lane, const float4 (&cold)[4], bool& ok) {
  const uint32_t acc = li & 1;
  const int R = cfg.B * cfg.N;
  const int row = tile * TC_M + quarter * 32 + lane;       // row parity == lane parity
  const bool odd = lane & 1;
  const bool inrange = row < R;
  const int ubase = nh * (TC_NH / 4) + cq * 16;
  if (ok) ok = mbar_wait(bar_tfull + 8 * acc, (li >> 1) & 1, io.err);
  tc_fence_after();
  const bool valid = ok && inrange;
  const int erow = row & ~1, orow = row | 1;
  const bool ev = ok && erow < R, ov = ok && orow < R;     // validity of the two rows this lane pair writes
  const uint32_t taddr = tmem_base + acc * TC_NH + cq * 64 + ((uint32_t)(quarter * 32) << 16);
  float part[HEAD_PAD];
#pragma unroll
  for (int o = 0; o < HEAD_PAD; ++o) part[o] = 0.f;
#pragma unroll
  for (int cp = 0; cp < 2; ++cp) {          // 8 hidden units (32 accumulator columns) at a time
    uint32_t v0[16], v1[16];
    tmem_ld16(taddr + cp * 32, v0);
    tmem_ld16(taddr + cp * 32 + 16, v1);
    const int u0 = ubase + cp * 8;
    float cn0[4] = {0.f, 0.f, 0.f, 0.f}, hn0[4] = {0.f, 0.f, 0.f, 0.f};
    float cn1[4] = {0.f, 0.f, 0.f, 0.f}, hn1[4] = {0.f, 0.f, 0.f, 0.f};
    if (valid) {
      const float co0[4] = {cold[2 * cp].x, cold[2 * cp].y, cold[2 * cp].z, cold[2 * cp].w};
      const float co1[4] = {cold[2 * cp + 1].x, cold[2 * cp + 1].y, cold[2 * cp + 1].z, cold[2 * cp + 1].w};
      lstm_cell4(v0, co0, s_bias + 4 * u0, cn0, hn0);
      lstm_cell4(v1, co1, s_bias + 4 * (u0 + 4), cn1, hn1);
      if (partial) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float hv = j < 4 ? hn0[j & 3] : hn1[j & 3];
          const float4 w0 = *reinterpret_cast<const float4*>(&s_hw[(u0 + j) * HEAD_PAD]);
          const float4 w1 = *reinterpret_cast<const float4*>(&s_hw[(u0 + j) * HEAD_PAD + 4]);
          part[0] = fmaf(hv, w0.x, part[0]); part[1] = fmaf(hv, w0.y, part[1]);
          part[2] = fmaf(hv, w0.z, part[2]); part[3] = fmaf(hv, w0.w, part[3]);
          part[4] = fmaf(hv, w1.x, part[4]); part[5] = fmaf(hv, w1.y, part[5]);
          part[6] = fmaf(hv, w1.z, part[6]); part[7] = fmaf(hv, w1.w, part[7]);
        }
      }
    }
    pair_store8(io.c_out + (size_t)erow * TC_H + u0, io.c_out + (size_t)orow * TC_H + u0, cn0, cn1, ev, ov, odd);
    pair_store8(io.h_out + (size_t)erow * TC_H + u0, io.h_out + (size_t)orow * TC_H + u0, hn0, hn1, ev, ov, odd);
  }
  tc_fence_before();
  __syncwarp();                              // every lane of the warp is done reading the accumulator:
  if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);        // one arrival per warp
  if (partial) {                             // slot = (column half of the item, column quarter of the warp)
    const size_t so = (size_t)(nh * 4 + cq) * HEAD_PAD;
    const float pa[4] = {part[0], part[1], part[2], part[3]}, pb[4] = {part[4], part[5], part[6], part[7]};
    pair_store8(partial + (size_t)erow * NSLOT * HEAD_PAD + so, partial + (size_t)orow * NSLOT * HEAD_PAD + so, pa, pb, ev,
                ov, odd);
  }
}

__global__ void __launch_bounds__(TC_P_THREADS, 1) lstm_tc_kernel(ic3_policy_cfg cfg, ic3_policy_io io,
                                                                 const __half* __restrict__ a_img,
                                                                 const __half* __restrict__ b_img,
                                                                 const float* __restrict__ bias_cat, int nitems,
                                                                 const float* __restrict__ head_w, int nout,
                                                                 float* __restrict__ partial) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NSTAGE_P * STAGE_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  // head weights, unit-major [128][8] (zero padded): the epilogue folds value/action-head dot products
  // of its 32 hidden units into per-slot partial logits (partial != nullptr  <=>  nout <= 8)
  float* s_hw = reinterpret_cast<float*>(smem + NSTAGE_P * STAGE_BYTES + 256);
  float* s_bias = s_hw + TC_H * HEAD_PAD;
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + NSTAGE_P);
  const uint32_t bar_tfull = smem_u32(bars + 2 * NSTAGE_P), bar_tempty = smem_u32(bars + 2 * NSTAGE_P + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NSTAGE_P; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);         // released by the MMA warp's commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, EPI_WARPS);         // one arrival per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI_WARPS) {   // all 512 TMEM columns: two 128-lane x 256-column fp32 accumulators
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  load_scaled_bias(s_bias, bias_cat);
  if (partial) {
    for (int idx = threadIdx.x; idx < TC_H * HEAD_PAD; idx += blockDim.x) {
      const int u = idx / HEAD_PAD, o = idx - u * HEAD_PAD;
      s_hw[idx] = o < nout ? __ldg(head_w + (size_t)o * TC_H + u) : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == EPI_WARPS && lane == 0) {
    // ===== producer =====
    static_assert(TC_NCHUNK % NSTAGE_P == 0, "stage index must be a function of the chunk index alone");
    uint32_t li = 0;
    bool ok = true;
    const uint32_t smem_base = smem_u32(smem);
    for (int item = blockIdx.x; item < nitems && ok; item += gridDim.x, ++li) {
      const int tile = item >> 1, nh = item & 1;
      const unsigned char* a_src = reinterpret_cast<const unsigned char*>(a_img) + (size_t)tile * TC_NCHUNK * A_CHUNK_BYTES;
      const unsigned char* b_src = reinterpret_cast<const unsigned char*>(b_img) + (size_t)nh * TC_NCHUNK * B_CHUNK_BYTES;
      // TC_NCHUNK is a multiple of the ring depth: chunk c of every item uses stage c % NSTAGE_P, so the stage
      // index (and with it every shared-memory address / descriptor below) is a compile-time constant
#pragma unroll
      for (int c = 0; c < TC_NCHUNK; ++c) {
        if (!ok) break;
        const uint32_t s = c % NSTAGE_P;
        ok = mbar_wait(bar_empty + 8 * s, ((li * (TC_NCHUNK / NSTAGE_P) + c / NSTAGE_P) & 1) ^ 1, io.err);
        const uint32_t dst = smem_base + s * STAGE_BYTES;
        mbar_expect_tx(bar_full + 8 * s, STAGE_BYTES);
        bulk_g2s(dst, a_src + (size_t)c * (A_CHUNK_BYTES / 2), A_CHUNK_BYTES / 2, bar_full + 8 * s);                       // hi
        bulk_g2s(dst + A_CHUNK_BYTES / 2, a_src + A_TILE_HALFS + (size_t)c * (A_CHUNK_BYTES / 2), A_CHUNK_BYTES / 2,   // lo
                 bar_full + 8 * s);
        bulk_g2s(dst + A_CHUNK_BYTES, b_src + (size_t)c * B_CHUNK_BYTES, B_CHUNK_BYTES, bar_full + 8 * s);
      }
    }
  } else if (warp == EPI_WARPS + 1 && lane == 0) {
    // ===== MMA issuer =====
    // instruction descriptor: D = f32 (bits 4-5 = 1), A = B = f16 (0), K-major both, N >> 3 at 17, M >> 4 at 24
    const uint32_t idesc = (1u << 4) | ((uint32_t)(TC_NH >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
    uint32_t li = 0;
    bool ok = true;
    // descriptors of stage 0 / k-step 0; every other one is + (byte offset >> 4) in the address field.
    // A: kcore block = 16 rcores x 128 B = 2048 B; B: 32 ncores x 128 B = 4096 B; lo half follows hi half
    const uint64_t dA = make_desc(smem_u32(smem), 2048, 128), dB = make_desc(smem_u32(smem) + A_CHUNK_BYTES, 4096, 128);
    for (int item = blockIdx.x; item < nitems && ok; item += gridDim.x, ++li) {
      const uint32_t acc = li & 1;
      ok = mbar_wait(bar_tempty + 8 * acc, ((li >> 1) & 1) ^ 1, io.err);   // epilogue drained this accumulator
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * TC_NH;
#pragma unroll
      for (int c = 0; c < TC_NCHUNK; ++c) {
        if (!ok) break;
        const uint32_t s = c % NSTAGE_P;
        ok = mbar_wait(bar_full + 8 * s, (li * (TC_NCHUNK / NSTAGE_P) + c / NSTAGE_P) & 1, io.err);
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
        tc_commit(bar_empty + 8 * s);      // frees the stage when these MMAs have read it
      }
      tc_commit(bar_tfull + 8 * acc);      // accumulator complete
    }
  } else if (warp < EPI_WARPS) {
    // ===== epilogue: thread = (row of the tile, 16 hidden units) =====
    const int quarter = warp & 3, cq = warp >> 2;
    uint32_t li = 0;
    bool ok = true;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++li) {
      const int tile = item >> 1, nh = item & 1;
      float4 cold[4];         // issued before the accumulator wait: overlaps the MMAs of this item
      load_cold(cfg, io, tile, nh, quarter, cq, lane, cold);
      epilogue_item(cfg, io, s_bias, s_hw, partial, tmem_base, bar_tfull, bar_tempty, li, tile, nh, quarter, cq, lane, cold, ok);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ---- heads + sampling from h' (comm.py:228-239, action_utils.py:32-36) -----------------------------
// P lanes per agent row (P = pow2 >= 1 + sum(na)), lane o of a group computes output o as a full
// 128-long dot product (h row broadcast inside the group, weight rows L1-resident), then the
// log-softmax / inverse-CDF sampling runs inside the group with width-P shuffles.
template <int P>
__global__ void __launch_bounds__(256) heads_kernel(ic3_policy_cfg cfg, ic3_policy_packed w, ic3_policy_io io) {
  constexpr int RPW = 32 / P;
  const int lane = threadIdx.x & 31, o = lane % P;
  const long R = (long)cfg.B * cfg.N;
  const long row = ((long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW + lane / P;
  const bool live = row < R;
  int atot = 0;
  for (int k = 0; k < cfg.nheads; ++k) atot += cfg.head_dim[k];
  const int nout = 1 + atot;
  // head weights k-major in shared memory: the P lanes of a group read P consecutive floats,
  // every group reads the same addresses -> one broadcast wavefront per load
  __shared__ float s_w[TC_H * P];
  for (int idx = threadIdx.x; idx < TC_H * P; idx += blockDim.x) {
    const int k = idx / P, oo = idx - k * P;
    s_w[idx] = oo < nout ? __ldg(w.head_w + (size_t)oo * TC_H + k) : 0.f;
  }
  __syncthreads();
  float logit = 0.f;
  if (live) {
    const float4* hp = reinterpret_cast<const float4*>(io.h_out + (size_t)row * TC_H);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
    for (int q = 0; q < TC_H / 4; ++q) {
      const float4 hv = hp[q];
      a0 = fmaf(hv.x, s_w[(4 * q + 0) * P + o], a0);
      a1 = fmaf(hv.y, s_w[(4 * q + 1) * P + o], a1);
      a2 = fmaf(hv.z, s_w[(4 * q + 2) * P + o], a2);
      a3 = fmaf(hv.w, s_w[(4 * q + 3) * P + o], a3);
    }
    logit = (a0 + a1) + (a2 + a3) + (o < nout ? __ldg(w.head_b + o) : 0.f);
  }
  if (live && o == 0) io.value[row] = logit;
  const bool do_sample = io.action != nullptr;
  const int e = live ? (int)(row / cfg.N) : 0, i = live ? (int)(row - (long)e * cfg.N) : 0;
  uint32_t w0 = 0, w1 = 0, w2 = 0, w3 = 0;
  if (do_sample && !io.draws) {
    if (o == 0 && live) {
      const uint4 d = ic3_draw24(cfg.seed, cfg.env_id0 + (uint32_t)e, io.tick ? io.tick[e] : 0u, IC3_STREAM_ACTION, (uint32_t)i);
      w0 = d.x; w1 = d.y; w2 = d.z; w3 = d.w;
    }
    w0 = __shfl_sync(IC3_FULL_MASK, w0, 0, P); w1 = __shfl_sync(IC3_FULL_MASK, w1, 0, P);
    w2 = __shfl_sync(IC3_FULL_MASK, w2, 0, P); w3 = __shfl_sync(IC3_FULL_MASK, w3, 0, P);
  }
  int off = 1;
  for (int k = 0; k < cfg.nheads; ++k) {
    const int na = cfg.head_dim[k];
    float m = -INFINITY;
    for (int a = 0; a < na; ++a) m = fmaxf(m, __shfl_sync(IC3_FULL_MASK, logit, off + a, P));
    float s = 0.f;
    for (int a = 0; a < na; ++a) s += expf(__shfl_sync(IC3_FULL_MASK, logit, off + a, P) - m);
    const float mylogp = logit - (m + logf(s));
    uint32_t u24 = 0;
    if (do_sample) {
      if (io.draws) u24 = live ? io.draws[(size_t)row * cfg.nheads + k] : 0u;
      else u24 = k == 0 ? w0 : (k == 1 ? w1 : (k == 2 ? w2 : w3));
    }
    const float u = (float)u24 * 5.9604644775390625e-08f;
    int act = na - 1;
    if (do_sample) {
      float cdf = 0.f;
      bool found = false;
      for (int a = 0; a < na; ++a) {
        cdf += expf(__shfl_sync(IC3_FULL_MASK, mylogp, off + a, P));
        if (!found && cdf > u) {
          act = a;
          found = true;
        }
      }
    }
    if (live && o >= off && o < off + na) io.logp[(size_t)row * atot + (off - 1) + (o - off)] = mylogp;
    if (live && do_sample && o == 0) io.action[(size_t)row * cfg.nheads + k] = act;
    off += na;
  }
}

// Finishing the heads from the per-slot partial logits of the LSTM epilogue (fixed summation order -> deterministic):
// value, log-softmax per head, inverse-CDF sampling of ONE agent row by ONE thread.
struct HeadsFinish {
  const float* partial;   // [R][NSLOT][HEAD_PAD]
  const float* head_b;    // [1 + sum(na)]
  int nheads;
  int head_dim[IC3_MAX_HEADS];
  uint64_t seed;
  uint32_t env_id0;
  const uint32_t* tick;   // [B] or NULL
  const uint32_t* draws;  // [R, nheads] or NULL
  float* value;           // [R]
  float* logp;            // [R, sum(na)]
  int32_t* action;        // [R, nheads] or NULL (no sampling)
};

__device__ __forceinline__ void heads_finish_row(const HeadsFinish& f, long row, int e, int i) {
  float logit[HEAD_PAD];
  const float4* p4 = reinterpret_cast<const float4*>(f.partial + (size_t)row * NSLOT * HEAD_PAD);
  {
    float4 a = p4[0], b = p4[1];
#pragma unroll
    for (int sl = 1; sl < NSLOT; ++sl) {
      const float4 c = p4[2 * sl], d = p4[2 * sl + 1];
      a.x += c.x; a.y += c.y; a.z += c.z; a.w += c.w;
      b.x += d.x; b.y += d.y; b.z += d.z; b.w += d.w;
    }
    logit[0] = a.x; logit[1] = a.y; logit[2] = a.z; logit[3] = a.w;
    logit[4] = b.x; logit[5] = b.y; logit[6] = b.z; logit[7] = b.w;
  }
  int atot = 0;
  for (int k = 0; k < f.nheads; ++k) atot += f.head_dim[k];
#pragma unroll
  for (int o = 0; o < HEAD_PAD; ++o) logit[o] += (o < 1 + atot) ? __ldg(f.head_b + o) : 0.f;
  f.value[row] = logit[0];
  const bool do_sample = f.action != nullptr;
  uint4 d24 = make_uint4(0, 0, 0, 0);
  if (do_sample && !f.draws)
    d24 = ic3_draw24(f.seed, f.env_id0 + (uint32_t)e, f.tick ? f.tick[e] : 0u, IC3_STREAM_ACTION, (uint32_t)i);
  int off = 1;
  for (int k = 0; k < f.nheads; ++k) {
    const int na = f.head_dim[k];
    float m = -INFINITY;
#pragma unroll
    for (int o = 1; o < HEAD_PAD; ++o)
      if (o >= off && o < off + na) m = fmaxf(m, logit[o]);
    float ssum = 0.f;
#pragma unroll
    for (int o = 1; o < HEAD_PAD; ++o)
      if (o >= off && o < off + na) ssum += expf(logit[o] - m);
    const float lse = m + logf(ssum);
    uint32_t u24 = 0;
    if (do_sample) u24 = f.draws ? f.draws[(size_t)row * f.nheads + k] : ic3_word(d24, k);
    const float u = (float)u24 * 5.9604644775390625e-08f;
    float cdf = 0.f;
    int act = na - 1;
    bool found = false;
#pragma unroll
    for (int o = 1; o < HEAD_PAD; ++o) {
      if (o >= off && o < off + na) {
        const float lp = logit[o] - lse;
        f.logp[(size_t)row * atot + (o - 1)] = lp;
        cdf += expf(lp);
        if (!found && cdf > u) {
          act = o - off;
          found = true;
        }
      }
    }
    if (do_sample) f.action[(size_t)row * f.nheads + k] = act;
    off += na;
  }
}

// Finish the heads from the NSLOT per-slot partial logits (fixed summation order -> deterministic):
// value, log-softmax per head, inverse-CDF sampling.  One thread per agent row.
__global__ void __launch_bounds__(128) heads_finish_kernel(ic3_policy_cfg cfg, ic3_policy_packed w, ic3_policy_io io,
                                                            const float* __restrict__ partial) {
  const long row = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= (long)cfg.B * cfg.N) return;
  HeadsFinish f;
  f.partial = partial; f.head_b = w.head_b; f.nheads = cfg.nheads;
#pragma unroll
  for (int k = 0; k < IC3_MAX_HEADS; ++k) f.head_dim[k] = cfg.head_dim[k];
  f.seed = cfg.seed; f.env_id0 = cfg.env_id0; f.tick = io.tick; f.draws = io.draws;
  f.value = io.value; f.logp = io.logp; f.action = io.action;
  const int e = (int)(row / cfg.N), i = (int)(row - (long)e * cfg.N);
  heads_finish_row(f, row, e, i);
}

}  // namespace
