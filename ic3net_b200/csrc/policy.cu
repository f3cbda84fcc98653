// CommNet / IC3Net policy step (reference: comm.py:134-244, action_utils.py:32-36).
//
// fp32 SIMT implementation ("policy v1"): one CTA owns a tile of whole environments
// (<= 64 agent rows), so the all-to-all hidden-state mean of comm.py:181-205 never
// leaves shared memory.  Per tile:
//   A  stage h (zeroed on episode start) + per-row gate g = alive * comm_action
//   B  S[k] = g[k] * sum_{j != k} g[j] h[j] / (n_alive - 1)            (smem -> smem)
//   C  inp = x + C(S)                    register-tiled GEMM, weights streamed K-major
//   D  gates = [inp | h] . [W_ih ; W_hh]^T, LSTM cell in the epilogue (columns are
//      interleaved 4*u+gate so one thread owns i,f,g,o of a hidden unit)
//   E  value / action heads, log-softmax, inverse-CDF sampling (warp per row)
// Weights are pre-packed K-major by ic3_policy_pack so every weight read is a
// contiguous row; h/c/x/h'/c' move through HBM exactly once per step.
#include <cstring>

#include "ic3_common.cuh"
#include "policy_heads.cuh"
#include "policy_internal.h"

namespace {

constexpr int ROWS = 64;   // agent rows per CTA tile
constexpr int KC = 16;     // K chunk staged in smem
constexpr int NT = 256;    // threads per CTA
constexpr int RPT = ROWS / (NT / 32);  // rows per thread = 8

template <int H>
struct PolicySmem {
  float hs[ROWS][H];
  float ss[ROWS][H];
  float h2[ROWS][H];
  float bs[2][KC][128];
  float gate[ROWS];
  float den[ROWS];
};

// acc[r][c] += sum_k A[r][k] * Bt[k][col0 + tx*CPT + c]   for rows ty*8..ty*8+7
// A = A0 for k < H, A1 for H <= k < K.  Bt is global, K-major, leading dim ldb.
template <int H, int CPT>
__device__ __forceinline__ void gemm_tile(const float (*A0)[H], const float (*A1)[H], int K,
                                          const float* __restrict__ Bt, int ldb, int col0,
                                          float (*bs)[KC][128], float (&acc)[RPT][CPT]) {
  constexpr int BW = 32 * CPT;             // columns staged per chunk
  constexpr int F4 = KC * BW / 4;          // float4 per chunk
  constexpr int PF = (F4 + NT - 1) / NT;   // float4 per thread
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  float4 pf[PF];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int i = 0; i < PF; ++i) {
      const int idx = tid + i * NT;
      if (idx < F4) {
        const int kk = idx / (BW / 4), c4 = idx - kk * (BW / 4);
        pf[i] = __ldg(reinterpret_cast<const float4*>(Bt + (size_t)(k0 + kk) * ldb + col0) + c4);
      }
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int i = 0; i < PF; ++i) {
      const int idx = tid + i * NT;
      if (idx < F4) {
        const int kk = idx / (BW / 4), c4 = idx - kk * (BW / 4);
        *reinterpret_cast<float4*>(&bs[buf][kk][c4 * 4]) = pf[i];
      }
    }
  };
  const int nchunk = K / KC;
  fetch(0);
  for (int kc = 0; kc < nchunk; ++kc) {
    const int buf = kc & 1;
    stash(buf);
    __syncthreads();
    if (kc + 1 < nchunk) fetch((kc + 1) * KC);
    const int k0 = kc * KC;
    const float(*A)[H] = (k0 < H) ? A0 : A1;
    const int ka = (k0 < H) ? k0 : k0 - H;
#pragma unroll
    for (int kk = 0; kk < KC; kk += 4) {
      float4 a[RPT];
#pragma unroll
      for (int r = 0; r < RPT; ++r) a[r] = *reinterpret_cast<const float4*>(&A[ty * RPT + r][ka + kk]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float b[CPT];
#pragma unroll
        for (int c = 0; c < CPT; ++c) b[c] = bs[buf][kk + i][tx * CPT + c];
#pragma unroll
        for (int r = 0; r < RPT; ++r) {
          const float av = i == 0 ? a[r].x : (i == 1 ? a[r].y : (i == 2 ? a[r].z : a[r].w));
#pragma unroll
          for (int c = 0; c < CPT; ++c) acc[r][c] = fmaf(av, b[c], acc[r][c]);
        }
      }
    }
  }
  __syncthreads();
}

__device__ __forceinline__ float sigmoidf_(float v) { return 1.f / (1.f + expf(-v)); }

struct PolicyArgs {
  ic3_policy_cfg cfg;
  ic3_policy_packed w;
  ic3_policy_io io;
};

template <int H>
__global__ void __launch_bounds__(NT) policy_step_kernel(PolicyArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  PolicySmem<H>& sm = *reinterpret_cast<PolicySmem<H>*>(smem_raw);
  const ic3_policy_cfg& cfg = a.cfg;
  const ic3_policy_io& io = a.io;
  const int N = cfg.N, B = cfg.B;
  const int epb = ROWS / N;
  const int e0 = blockIdx.x * epb;
  const int nenv = min(epb, B - e0);
  const int nrows = nenv * N;
  const size_t row0 = (size_t)e0 * N;
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  constexpr int H4 = H / 4;

  // ---- A: stage h, gates ---------------------------------------------------
  // hidden state entering the first comm pass: the recurrent state io.h (zero at an episode start), or -- non-recurrent
  // branch, comm.py:127-129 / models.py:24 -- the encoded observation itself
  for (int idx = tid; idx < ROWS * H4; idx += NT) {
    const int r = idx / H4, q = idx - r * H4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < nrows) {
      const int e = e0 + r / N;
      if (cfg.h_from_x) {
        v = __ldg(reinterpret_cast<const float4*>(io.x + (row0 + r) * H) + q);
        if (cfg.x_tanh) v = make_float4(tanhf(v.x), tanhf(v.y), tanhf(v.z), tanhf(v.w));
      } else if (!(io.fresh && io.fresh[e])) {
        v = __ldg(reinterpret_cast<const float4*>(io.h + (row0 + r) * H) + q);
      }
    }
    *reinterpret_cast<float4*>(&sm.hs[r][q * 4]) = v;
  }
  for (int r = tid; r < ROWS; r += NT) {
    float g = 0.f, den = 1.f;
    if (r < nrows) {
      const int el = r / N, e = e0 + el, i = r - el * N;
      const bool fr = io.fresh && io.fresh[e];
      int n_alive = N;                       // comm.py:105-107 (no alive_mask -> everyone)
      int al = 1;
      if (io.alive && !fr) {                 // comm.py:102-104
        n_alive = 0;
        for (int j = 0; j < N; ++j) n_alive += io.alive[(size_t)e * N + j] != 0;
        al = io.alive[(size_t)e * N + i] != 0;
      }
      int cm = 1;
      if (cfg.hard_attn) cm = fr ? 0 : (io.comm_action[(size_t)e * N + i] != 0);   // comm.py:171-175, trainer.py:45-46
      g = (float)(al * cm);
      if (cfg.comm_avg && n_alive > 1) den = (float)(n_alive - 1);                  // comm.py:194-196
    }
    sm.gate[r] = g;
    sm.den[r] = den;
  }
  __syncthreads();

  const int npass = cfg.passes > 1 ? cfg.passes : 1;
  for (int ps = 0; ps < npass; ++ps) {        // comm passes (comm.py:179)
    if (ps > 0) {                             // the hidden state of the previous pass feeds this one
      for (int idx = tid; idx < ROWS * H4; idx += NT) {
        const int r = idx / H4, q = idx - r * H4;
        *reinterpret_cast<float4*>(&sm.hs[r][q * 4]) = *reinterpret_cast<const float4*>(&sm.h2[r][q * 4]);
      }
      __syncthreads();
    }
    // ---- B: communication vector (comm.py:181-205) -----------------------------
    for (int idx = tid; idx < ROWS * H4; idx += NT) {
      const int r = idx / H4, q = idx - r * H4;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nrows && !cfg.comm_mask_zero && sm.gate[r] != 0.f) {
        const int base = (r / N) * N;
        for (int j = 0; j < N; ++j) {
          if (base + j != r && sm.gate[base + j] != 0.f) {
            const float4 hv = *reinterpret_cast<const float4*>(&sm.hs[base + j][q * 4]);
            acc.x += hv.x; acc.y += hv.y; acc.z += hv.z; acc.w += hv.w;
          }
        }
        const float d = sm.den[r];
        acc.x /= d; acc.y /= d; acc.z /= d; acc.w /= d;
      }
      *reinterpret_cast<float4*>(&sm.ss[r][q * 4]) = acc;
    }
    __syncthreads();

    // ---- C: inp = x + C_i(S) (comm.py:206,211) -----------------------------------
    {
      constexpr int CPT = H / 32;
      float acc[RPT][CPT];
#pragma unroll
      for (int r = 0; r < RPT; ++r)
#pragma unroll
        for (int c = 0; c < CPT; ++c) acc[r][c] = 0.f;
      gemm_tile<H, CPT>(sm.ss, sm.ss, H, a.w.c_wT + (size_t)ps * H * H, H, 0, sm.bs, acc);   // trailing sync: all reads of S done
#pragma unroll
      for (int r = 0; r < RPT; ++r) {
        const int row = ty * RPT + r;
#pragma unroll
        for (int c = 0; c < CPT; ++c) {
          const int col = tx * CPT + c;
          float v = 0.f;
          if (row < nrows) {
            float xv = __ldg(io.x + (row0 + row) * H + col);
            if (cfg.x_tanh) xv = tanhf(xv);
            v = xv + (acc[r][c] + __ldg(a.w.c_b + (size_t)ps * H + col));
          }
          sm.ss[row][col] = v;
        }
      }
    }
    __syncthreads();

    if (cfg.cell == IC3_CELL_TANH) {
      // ---- D': h = tanh(x + f_i(h) + C_i(S)) (comm.py:220-224; models.py:25,84) ----------
      constexpr int CPT = H / 32;
      float acc[RPT][CPT];
#pragma unroll
      for (int r = 0; r < RPT; ++r)
#pragma unroll
        for (int c = 0; c < CPT; ++c) acc[r][c] = 0.f;
      gemm_tile<H, CPT>(sm.hs, sm.hs, H, a.w.f_wT + (size_t)ps * H * H, H, 0, sm.bs, acc);
#pragma unroll
      for (int r = 0; r < RPT; ++r) {
        const int row = ty * RPT + r;
#pragma unroll
        for (int c = 0; c < CPT; ++c) {
          const int col = tx * CPT + c;
          float hn = 0.f;
          if (row < nrows) {
            hn = tanhf(sm.ss[row][col] + (acc[r][c] + __ldg(a.w.f_b + (size_t)ps * H + col)));
            if (ps == npass - 1) io.h_out[(row0 + row) * H + col] = hn;
          }
          sm.h2[row][col] = hn;
        }
      }
    } else {
      // ---- D: LSTM cell (comm.py:213-218; torch.nn.LSTMCell, gates i,f,g,o) -------
      for (int p = 0; p < (4 * H) / 128; ++p) {
        float acc[RPT][4];
#pragma unroll
        for (int r = 0; r < RPT; ++r)
#pragma unroll
          for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
        gemm_tile<H, 4>(sm.ss, sm.hs, 2 * H, a.w.lstm_wT, 4 * H, p * 128, sm.bs, acc);
        const int u = p * 32 + tx;
        const float4 bias = __ldg(reinterpret_cast<const float4*>(a.w.lstm_b) + u);
#pragma unroll
        for (int r = 0; r < RPT; ++r) {
          const int row = ty * RPT + r;
          float hn = 0.f;
          if (row < nrows) {
            const int e = e0 + row / N;
            const bool fr = io.fresh && io.fresh[e];
            // cell state: the recurrent input on the first pass, this thread's own c' of the previous pass afterwards
            const float cold = ps > 0 ? io.c_out[(row0 + row) * H + u] : (fr ? 0.f : __ldg(io.c + (row0 + row) * H + u));
            const float gi = sigmoidf_(acc[r][0] + bias.x);
            const float gf = sigmoidf_(acc[r][1] + bias.y);
            const float gg = tanhf(acc[r][2] + bias.z);
            const float go = sigmoidf_(acc[r][3] + bias.w);
            const float cn = gf * cold + gi * gg;
            hn = go * tanhf(cn);
            io.c_out[(row0 + row) * H + u] = cn;
            if (ps == npass - 1) io.h_out[(row0 + row) * H + u] = hn;
          }
          sm.h2[row][u] = hn;
        }
      }
    }
    __syncthreads();
  }

  // ---- E: heads, log-softmax, sampling (comm.py:228-239, action_utils.py:32-36) --
  const int warp = ty, lane = tx;
  for (int r = warp; r < nrows; r += NT / 32) {
    float hv[H / 32];
#pragma unroll
    for (int m = 0; m < H / 32; ++m) hv[m] = sm.h2[r][lane + 32 * m];
    const int e = e0 + r / N, i = r - (r / N) * N;
    heads_for_row<H>(cfg, a.w.head_w, a.w.head_b, hv, row0 + r, e, i, lane, io.tick, io.draws, io.value, io.logp,
                     io.action);
  }
}

// ---------------------------------------------------------------------------
// select_action alone (action_utils.py:32-36): one thread per (env, agent)
// ---------------------------------------------------------------------------
__global__ void sample_kernel(ic3_policy_cfg cfg, const float* __restrict__ logp, const uint32_t* __restrict__ tick,
                              const uint32_t* __restrict__ draws, int32_t* __restrict__ action) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= cfg.B * cfg.N) return;
  const int e = row / cfg.N, i = row - e * cfg.N;
  int atot = 0;
  for (int k = 0; k < cfg.nheads; ++k) atot += cfg.head_dim[k];
  uint4 w = make_uint4(0, 0, 0, 0);
  if (!draws) w = ic3_draw24(cfg.seed, cfg.env_id0 + (uint32_t)e, tick ? tick[e] : 0u, IC3_STREAM_ACTION, (uint32_t)i);
  int off = 0;
  for (int k = 0; k < cfg.nheads; ++k) {
    const int na = cfg.head_dim[k];
    const uint32_t u24 = draws ? draws[(size_t)row * cfg.nheads + k] : ic3_word(w, k);
    const float u = (float)u24 * 5.9604644775390625e-08f;
    float cdf = 0.f;
    int act = na - 1;
    bool found = false;
    for (int q = 0; q < na; ++q) {
      cdf += expf(logp[(size_t)row * atot + off + q]);
      if (!found && cdf > u) {
        act = q;
        found = true;
      }
    }
    action[(size_t)row * cfg.nheads + k] = act;
    off += na;
  }
}

// ---------------------------------------------------------------------------
// encoder, dense form (comm.py:119): warp per agent row, obs streamed once with
// 16-byte evict-first loads; only non-zero features touch the (L2-resident) W^T.
// ---------------------------------------------------------------------------
template <int CPT>
__device__ __forceinline__ void axpy_row(float (&acc)[CPT], float v, const float* __restrict__ wrow, int lane) {
  if (CPT == 4) {
    const float4 wv = __ldg(reinterpret_cast<const float4*>(wrow) + lane);
    acc[0] = fmaf(v, wv.x, acc[0]); acc[1] = fmaf(v, wv.y, acc[1]);
    acc[2] = fmaf(v, wv.z, acc[2]); acc[3] = fmaf(v, wv.w, acc[3]);
  } else if (CPT == 2) {
    const float2 wv = __ldg(reinterpret_cast<const float2*>(wrow) + lane);
    acc[0] = fmaf(v, wv.x, acc[0]); acc[1] = fmaf(v, wv.y, acc[1]);
  } else {
    acc[0] = fmaf(v, __ldg(wrow + lane), acc[0]);
  }
}

template <int CPT>
__device__ __forceinline__ void store_x(const float (&acc)[CPT], float* __restrict__ xrow, int lane) {
  if (CPT == 4) reinterpret_cast<float4*>(xrow)[lane] = make_float4(acc[0], acc[1], acc[2], acc[3]);
  else if (CPT == 2) reinterpret_cast<float2*>(xrow)[lane] = make_float2(acc[0], acc[1]);
  else xrow[lane] = acc[0];
}

// Observation layout hint of ic3_policy_cfg (obs_off, obs_vocab, obs_ncount): is feature f a one-hot position
// class (first accumulator, may come from a per-position table) or a count / scalar (second accumulator)?
struct ObsLayout {
  int off, V, ncount;
  __device__ __forceinline__ bool is_class(int f) const {
    if (V <= 0) return true;            // no hint: one sum
    if (f < off) return false;
    return ((f - off) % V) < V - ncount;
  }
  // four consecutive features f0 .. f0+3 with ONE integer division (V >= 4, checked by policy_check)
  __device__ __forceinline__ void is_class4(int f0, bool (&c)[4]) const {
    if (V <= 0) {
      c[0] = c[1] = c[2] = c[3] = true;
      return;
    }
    const int r = f0 - off;                 // negative only for the scalar features in front of the cells
    const int m = r >= 0 ? r % V : r;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      int rk = m + k;
      if (rk >= V) rk -= V;
      c[k] = rk >= 0 && rk < V - ncount;
    }
  }
};

template <int CPT>
__device__ __forceinline__ void store_x2(const float (&a)[CPT], const float (&b)[CPT], float* __restrict__ xrow, int lane) {
  float r[CPT];
#pragma unroll
  for (int c = 0; c < CPT; ++c) r[c] = a[c] + b[c];      // x = (bias + class terms) + (other terms)
  store_x<CPT>(r, xrow, lane);
}

template <int H, bool VEC>
__global__ void __launch_bounds__(256) encoder_dense_kernel(const float* __restrict__ obs, const float* __restrict__ wT,
                                                            const float* __restrict__ bias, float* __restrict__ x,
                                                            int rows, int O, ObsLayout lay) {
  constexpr int CPT = H / 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + warp;
  if (row >= rows) return;
  float acc[CPT], acc2[CPT];
#pragma unroll
  for (int c = 0; c < CPT; ++c) {
    acc[c] = __ldg(bias + lane * CPT + c);
    acc2[c] = 0.f;
  }
  const float* orow = obs + (size_t)row * O;
  constexpr int U = 4;
  if (VEC) {
    const float4* o4 = reinterpret_cast<const float4*>(orow);
    const int n4 = O >> 2;
    for (int base = 0; base < n4; base += 32 * U) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int idx = base + u * 32 + lane;
        v[u] = idx < n4 ? ic3_ld_stream(o4 + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        unsigned m = __ballot_sync(IC3_FULL_MASK, v[u].x != 0.f || v[u].y != 0.f || v[u].z != 0.f || v[u].w != 0.f);
        while (m) {
          const int src = __ffs(m) - 1;
          m &= m - 1;
          const float sx = __shfl_sync(IC3_FULL_MASK, v[u].x, src), sy = __shfl_sync(IC3_FULL_MASK, v[u].y, src);
          const float sz = __shfl_sync(IC3_FULL_MASK, v[u].z, src), sw = __shfl_sync(IC3_FULL_MASK, v[u].w, src);
          const int f0 = (base + u * 32 + src) * 4;
          const float* wr = wT + (size_t)f0 * H;
          bool cl[4];
          lay.is_class4(f0, cl);
          if (sx != 0.f) { if (cl[0]) axpy_row<CPT>(acc, sx, wr, lane); else axpy_row<CPT>(acc2, sx, wr, lane); }
          if (sy != 0.f) { if (cl[1]) axpy_row<CPT>(acc, sy, wr + H, lane); else axpy_row<CPT>(acc2, sy, wr + H, lane); }
          if (sz != 0.f) { if (cl[2]) axpy_row<CPT>(acc, sz, wr + 2 * H, lane); else axpy_row<CPT>(acc2, sz, wr + 2 * H, lane); }
          if (sw != 0.f) { if (cl[3]) axpy_row<CPT>(acc, sw, wr + 3 * H, lane); else axpy_row<CPT>(acc2, sw, wr + 3 * H, lane); }
        }
      }
    }
  } else {
    for (int base = 0; base < O; base += 32 * U) {
      float v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int idx = base + u * 32 + lane;
        v[u] = idx < O ? ic3_ld_stream(orow + idx) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        unsigned m = __ballot_sync(IC3_FULL_MASK, v[u] != 0.f);
        while (m) {
          const int src = __ffs(m) - 1;
          m &= m - 1;
          const float s = __shfl_sync(IC3_FULL_MASK, v[u], src);
          const int f = base + u * 32 + src;
          if (lay.is_class(f)) axpy_row<CPT>(acc, s, wT + (size_t)f * H, lane);
          else axpy_row<CPT>(acc2, s, wT + (size_t)f * H, lane);
        }
      }
    }
  }
  store_x2<CPT>(acc, acc2, x + (size_t)row * H, lane);
}

// ---------------------------------------------------------------------------
// encoder, index form: the same sum taken straight from the env state, in the
// same feature order as the dense kernel (bit-identical x), no [B,N,O] tensor.
// ---------------------------------------------------------------------------
template <int H>
__global__ void __launch_bounds__(256) pp_encoder_index_kernel(ic3_pp_cfg env, ic3_pp_state st,
                                                               const float* __restrict__ wT,
                                                               const float* __restrict__ bias, float* __restrict__ x,
                                                               bool split) {
  constexpr int CPT = H / 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + warp;
  const int N = env.N, D = env.dim, v = env.vision, W = 2 * v + 1, V = D * D + 4;
  const int NA = ic3_pp_agents(env);          // agent rows per env: row N = the prey (enemy_comm)
  if (row >= env.B * NA) return;
  const int e = row / NA, i = row - e * NA;
  int lr = -1, lc = -1;
  if (lane <= N) {
    const int* l = st.loc + ((size_t)e * (N + 1) + lane) * 2;
    lr = l[0];
    lc = l[1];
  }
  const int r0 = __shfl_sync(IC3_FULL_MASK, lr, i), c0 = __shfl_sync(IC3_FULL_MASK, lc, i);
  float acc[CPT], acc2[CPT];
#pragma unroll
  for (int c = 0; c < CPT; ++c) {
    acc[c] = __ldg(bias + lane * CPT + c);
    acc2[c] = 0.f;
  }
  for (int w = 0; w < W * W; ++w) {
    const int dy = w / W, dx = w - dy * W;
    const int rr = r0 - v + dy, cc = c0 - v + dx;
    const float* wcell = wT + (size_t)w * V * H;
    const unsigned here = __ballot_sync(IC3_FULL_MASK, lr == rr && lc == cc);
    if (rr >= 0 && rr < D && cc >= 0 && cc < D) {
      const int npred = __popc(here & ((1u << N) - 1u));
      const int nprey = (here >> N) & 1u;
      axpy_row<CPT>(acc, 1.f, wcell + (size_t)(rr * D + cc) * H, lane);
      if (split) {          // counts go to the second sum (ic3_policy_cfg.obs_vocab > 0)
        if (nprey) axpy_row<CPT>(acc2, (float)nprey, wcell + (size_t)(V - 2) * H, lane);
        if (npred) axpy_row<CPT>(acc2, (float)npred, wcell + (size_t)(V - 1) * H, lane);
      } else {
        if (nprey) axpy_row<CPT>(acc, (float)nprey, wcell + (size_t)(V - 2) * H, lane);
        if (npred) axpy_row<CPT>(acc, (float)npred, wcell + (size_t)(V - 1) * H, lane);
      }
    } else {
      axpy_row<CPT>(acc, 1.f, wcell + (size_t)(V - 3) * H, lane);
    }
  }
  store_x2<CPT>(acc, acc2, x + (size_t)row * H, lane);
}

template <int H>
__global__ void __launch_bounds__(256) tj_encoder_index_kernel(ic3_tj_cfg env, ic3_tj_state st,
                                                               const float* __restrict__ wT,
                                                               const float* __restrict__ bias, float* __restrict__ x,
                                                               bool split) {
  constexpr int CPT = H / 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + warp;
  const int N = env.N, v = env.vision, W = 2 * v + 1, V = env.vocab;
  if (row >= env.B * N) return;
  const int e = row / N, i = row - e * N;
  int lr = -1, lc = -1;
  if (lane < N) {
    lr = st.loc[((size_t)e * N + lane) * 2];
    lc = st.loc[((size_t)e * N + lane) * 2 + 1];
  }
  const int r0 = __shfl_sync(IC3_FULL_MASK, lr, i), c0 = __shfl_sync(IC3_FULL_MASK, lc, i);
  float acc[CPT], acc2s[CPT];
#pragma unroll
  for (int c = 0; c < CPT; ++c) {
    acc[c] = __ldg(bias + lane * CPT + c);
    acc2s[c] = 0.f;
  }
  // split (ic3_policy_cfg.obs_vocab > 0): scalars and car counts form the second sum
  if (st.alive[(size_t)e * N + i]) {
    const float la = (float)st.last_act[(size_t)e * N + i];
    const float ri = (float)st.route_id[(size_t)e * N + i] / (float)(env.npath - 1);
    if (split) {
      if (la != 0.f) axpy_row<CPT>(acc2s, la, wT, lane);
      if (ri != 0.f) axpy_row<CPT>(acc2s, ri, wT + H, lane);
    } else {
      if (la != 0.f) axpy_row<CPT>(acc, la, wT, lane);
      if (ri != 0.f) axpy_row<CPT>(acc, ri, wT + H, lane);
    }
    for (int w = 0; w < W * W; ++w) {
      const int dy = w / W, dx = w - dy * W;
      const int rr = r0 - v + dy, cc = c0 - v + dx;
      const float* wcell = wT + (size_t)(2 + w * V) * H;
      const unsigned here = __ballot_sync(IC3_FULL_MASK, lr == rr && lc == cc);
      int cls = env.outside_cls, cnt = 0;
      if (rr >= 0 && rr < env.h && cc >= 0 && cc < env.w) {
        cls = env.grid[rr * env.w + cc];
        cnt = __popc(here);
      }
      // dense order: class index ascending; cls < car_cls always (BASE+2)
      axpy_row<CPT>(acc, 1.f, wcell + (size_t)cls * H, lane);
      if (cnt) {
        if (split) axpy_row<CPT>(acc2s, (float)cnt, wcell + (size_t)env.car_cls * H, lane);
        else axpy_row<CPT>(acc, (float)cnt, wcell + (size_t)env.car_cls * H, lane);
      }
    }
  }
  store_x2<CPT>(acc, acc2s, x + (size_t)row * H, lane);      // acc2s == 0 when not split: x = acc
}

// ---------------------------------------------------------------------------
// class part of the encoder sum per agent position (see ic3_policy_cfg.obs_vocab): thread = hidden unit,
// same sequence of fp32 additions as the kernels above -> the fused encoder that starts from this table is
// bit-identical to them.
// ---------------------------------------------------------------------------
__global__ void pp_encoder_table_kernel(int D, int v, int H, const float* __restrict__ wT, const float* __restrict__ bias,
                                        float* __restrict__ table) {
  const int pos = blockIdx.x, n = threadIdx.x;
  const int r0 = pos / D, c0 = pos - r0 * D, W = 2 * v + 1, V = D * D + 4;
  if (n >= H) return;
  float acc = bias[n];
  for (int w = 0; w < W * W; ++w) {
    const int dy = w / W, dx = w - dy * W;
    const int rr = r0 - v + dy, cc = c0 - v + dx;
    const int cls = (rr >= 0 && rr < D && cc >= 0 && cc < D) ? rr * D + cc : V - 3;
    acc = fmaf(1.f, wT[(size_t)(w * V + cls) * H + n], acc);
  }
  table[(size_t)pos * H + n] = acc;
}

__global__ void tj_encoder_table_kernel(ic3_tj_cfg env, int H, const float* __restrict__ wT, const float* __restrict__ bias,
                                        float* __restrict__ table) {
  const int pos = blockIdx.x, n = threadIdx.x;
  const int r0 = pos / env.w, c0 = pos - r0 * env.w, v = env.vision, W = 2 * v + 1, V = env.vocab;
  if (n >= H) return;
  float acc = bias[n];
  for (int w = 0; w < W * W; ++w) {
    const int dy = w / W, dx = w - dy * W;
    const int rr = r0 - v + dy, cc = c0 - v + dx;
    const int cls = (rr >= 0 && rr < env.h && cc >= 0 && cc < env.w) ? env.grid[rr * env.w + cc] : env.outside_cls;
    acc = fmaf(1.f, wT[(size_t)(2 + w * V + cls) * H + n], acc);
  }
  table[(size_t)pos * H + n] = acc;
}

// ---------------------------------------------------------------------------
// weight packing (state_dict layout -> kernel layout), once per optimizer step
// ---------------------------------------------------------------------------
__global__ void pack_kernel(ic3_policy_cfg cfg, ic3_policy_params p, ic3_policy_packed o) {
  const int H = cfg.H, O = cfg.O;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (size_t idx = t0; idx < (size_t)O * H; idx += stride) {   // enc_wT[j][n] = W_e[n][j]
    const size_t j = idx / H, n = idx - j * H;
    o.enc_wT[idx] = p.encoder_w[n * O + j];
  }
  const int P = cfg.passes > 1 ? cfg.passes : 1;
  for (int ps = 0; ps < P; ++ps) {
    const float* cw = (ps > 0 && p.c_w_pass[ps]) ? p.c_w_pass[ps] : p.c_w;
    const float* cb = (ps > 0 && p.c_b_pass[ps]) ? p.c_b_pass[ps] : p.c_b;
    for (size_t idx = t0; idx < (size_t)H * H; idx += stride) {   // c_wT[ps][k][n] = W_c[n][k]
      const size_t k = idx / H, n = idx - k * H;
      o.c_wT[(size_t)ps * H * H + idx] = cw[n * H + k];
      if (cfg.cell == IC3_CELL_TANH) o.f_wT[(size_t)ps * H * H + idx] = p.f_w_pass[ps][n * H + k];
    }
    for (size_t idx = t0; idx < (size_t)H; idx += stride) {
      if (ps > 0) o.c_b[(size_t)ps * H + idx] = cb[idx];
      if (cfg.cell == IC3_CELL_TANH) o.f_b[(size_t)ps * H + idx] = p.f_b_pass[ps][idx];
    }
  }
  if (cfg.cell == IC3_CELL_LSTM) {
    for (size_t idx = t0; idx < (size_t)2 * H * 4 * H; idx += stride) {  // lstm_wT[k][4u+g]
      const size_t k = idx / (4 * H), col = idx - k * (4 * H);
      const size_t u = col >> 2, g = col & 3;
      o.lstm_wT[idx] = (k < (size_t)H) ? p.w_ih[(g * H + u) * H + k] : p.w_hh[(g * H + u) * H + (k - H)];
    }
    for (size_t idx = t0; idx < (size_t)4 * H; idx += stride) {
      const size_t u = idx >> 2, g = idx & 3;
      o.lstm_b[idx] = p.b_ih[g * H + u] + p.b_hh[g * H + u];
    }
  }
  for (size_t idx = t0; idx < (size_t)H; idx += stride) {
    o.enc_b[idx] = p.encoder_b[idx];
    o.c_b[idx] = p.c_b[idx];
    o.head_w[idx] = p.value_w[idx];
  }
  if (t0 == 0) o.head_b[0] = p.value_b[0];
  int rowoff = 1;
  for (int k = 0; k < cfg.nheads; ++k) {
    const int na = cfg.head_dim[k];
    for (size_t idx = t0; idx < (size_t)na * H; idx += stride) o.head_w[(size_t)rowoff * H + idx] = p.head_w[k][idx];
    for (size_t idx = t0; idx < (size_t)na; idx += stride) o.head_b[rowoff + idx] = p.head_b[k][idx];
    rowoff += na;
  }
}

int policy_check(const ic3_policy_cfg* cfg) {
  if (!cfg) return IC3_E_NULL;
  if (cfg->B <= 0 || cfg->N <= 0 || cfg->N > IC3_MAX_AGENTS || cfg->O <= 0) return IC3_E_RANGE;
  if (cfg->obs_vocab < 0 || cfg->obs_off < 0 || cfg->obs_ncount < 0 ||
      (cfg->obs_vocab > 0 && (cfg->obs_ncount >= cfg->obs_vocab || cfg->obs_vocab < 4)))
    return IC3_E_RANGE;
  if (cfg->H != 32 && cfg->H != 64 && cfg->H != 128) return IC3_E_UNSUPPORTED;
  if (cfg->nheads < 1 || cfg->nheads > IC3_MAX_HEADS) return IC3_E_RANGE;
  int tot = 1;
  for (int k = 0; k < cfg->nheads; ++k) {
    if (cfg->head_dim[k] < 1 || cfg->head_dim[k] > IC3_MAX_HEAD_DIM) return IC3_E_RANGE;
    tot += cfg->head_dim[k];
  }
  if (tot > 32) return IC3_E_RANGE;  // one logit per lane
  if (cfg->cell != IC3_CELL_LSTM && cfg->cell != IC3_CELL_TANH) return IC3_E_RANGE;
  if (cfg->passes < 0 || cfg->passes > IC3_MAX_PASSES) return IC3_E_RANGE;
  return IC3_OK;
}

// tcgen05 path: LSTM cell on the encoded observation, any number of comm passes (policy_tc.cu loops them)
bool policy_tc_capable(const ic3_policy_cfg* cfg) {
  return cfg->cell == IC3_CELL_LSTM && !cfg->x_tanh && !cfg->h_from_x;
}

int packed_check(const ic3_policy_packed* w) {
  if (!w) return IC3_E_NULL;
  if (!w->enc_wT || !w->enc_b || !w->c_wT || !w->c_b || !w->lstm_wT || !w->lstm_b || !w->head_w || !w->head_b)
    return IC3_E_NULL;
  return IC3_OK;
}

template <int H>
int launch_policy(const PolicyArgs& a, cudaStream_t s) {
  const size_t smem = sizeof(PolicySmem<H>);
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(policy_step_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  const int epb = ROWS / a.cfg.N;
  policy_step_kernel<H><<<(a.cfg.B + epb - 1) / epb, NT, smem, s>>>(a);
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}

template <int H>
int launch_encoder_dense(const ic3_policy_cfg* cfg, const ic3_policy_packed* w, const float* obs, float* x,
                         cudaStream_t s) {
  const int rows = cfg->B * cfg->N;
  const bool vec = (cfg->O % 4 == 0) && ((reinterpret_cast<uintptr_t>(obs) & 15) == 0);
  const int grid = (rows + 7) / 8;
  const ObsLayout lay{cfg->obs_off, cfg->obs_vocab, cfg->obs_ncount};
  if (vec) encoder_dense_kernel<H, true><<<grid, 256, 0, s>>>(obs, w->enc_wT, w->enc_b, x, rows, cfg->O, lay);
  else encoder_dense_kernel<H, false><<<grid, 256, 0, s>>>(obs, w->enc_wT, w->enc_b, x, rows, cfg->O, lay);
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}

}  // namespace

#define IC3_DISPATCH_H(Hval, CALL)          \
  switch (Hval) {                           \
    case 32: { constexpr int HH = 32; return CALL; }   \
    case 64: { constexpr int HH = 64; return CALL; }   \
    case 128: { constexpr int HH = 128; return CALL; } \
    default: return IC3_E_UNSUPPORTED;      \
  }

extern "C" int ic3_policy_pack(const ic3_policy_cfg* cfg, const ic3_policy_params* p,
                               const ic3_policy_packed* out, void* stream) {
  int rc = policy_check(cfg);
  if (rc) return rc;
  if (!p) return IC3_E_NULL;
  rc = packed_check(out);
  if (rc) return rc;
  if (!p->encoder_w || !p->encoder_b || !p->c_w || !p->c_b || !p->value_w || !p->value_b) return IC3_E_NULL;
  if (cfg->cell == IC3_CELL_LSTM && (!p->w_ih || !p->w_hh || !p->b_ih || !p->b_hh)) return IC3_E_NULL;
  if (cfg->cell == IC3_CELL_TANH) {
    if (!out->f_wT || !out->f_b) return IC3_E_NULL;
    for (int i = 0; i < (cfg->passes > 1 ? cfg->passes : 1); ++i)
      if (!p->f_w_pass[i] || !p->f_b_pass[i]) return IC3_E_NULL;
  }
  if (!policy_tc_capable(cfg) && (out->lstm_img || out->bias_cat)) return IC3_E_UNSUPPORTED;  // tanh cells: SIMT kernel only
  for (int k = 0; k < cfg->nheads; ++k)
    if (!p->head_w[k] || !p->head_b[k]) return IC3_E_NULL;
  pack_kernel<<<296, 256, 0, (cudaStream_t)stream>>>(*cfg, *p, *out);
  IC3_LAUNCH_CHECK();
  if (out->lstm_img || out->bias_cat) {   // tensor-core operand images
    if (!out->lstm_img || !out->bias_cat) return IC3_E_NULL;
    return ic3_tc_pack(cfg, p, out, (cudaStream_t)stream);
  }
  return IC3_OK;
}

extern "C" uint64_t ic3_policy_workspace_bytes(const ic3_policy_cfg* cfg) { return ic3_tc_workspace_bytes(cfg); }

// the layout hint, when given, must be the environment's own
int ic3_pp_layout_check(const ic3_pp_cfg* env, const ic3_policy_cfg* cfg) {
  if (cfg->obs_vocab == 0) return IC3_OK;
  return (cfg->obs_off == 0 && cfg->obs_vocab == env->dim * env->dim + 4 && cfg->obs_ncount == 2) ? IC3_OK : IC3_E_RANGE;
}
int ic3_tj_layout_check(const ic3_tj_cfg* env, const ic3_policy_cfg* cfg) {
  if (cfg->obs_vocab == 0) return IC3_OK;
  return (cfg->obs_off == 2 && cfg->obs_vocab == env->vocab && cfg->obs_ncount == 1 && env->car_cls == env->vocab - 1)
             ? IC3_OK : IC3_E_RANGE;
}

extern "C" int ic3_pp_encoder_table(const ic3_pp_cfg* env, const ic3_policy_cfg* cfg, const ic3_policy_packed* w,
                                    float* table, void* stream) {
  int rc = policy_check(cfg);
  if (rc) return rc;
  rc = packed_check(w);
  if (rc) return rc;
  if (!env || !table) return IC3_E_NULL;
  const int W = 2 * env->vision + 1;
  if (cfg->O != W * W * (env->dim * env->dim + 4) || cfg->obs_vocab == 0) return IC3_E_RANGE;
  rc = ic3_pp_layout_check(env, cfg);
  if (rc) return rc;
  pp_encoder_table_kernel<<<env->dim * env->dim, cfg->H, 0, (cudaStream_t)stream>>>(env->dim, env->vision, cfg->H, w->enc_wT,
                                                                                   w->enc_b, table);
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}

extern "C" int ic3_tj_encoder_table(const ic3_tj_cfg* env, const ic3_policy_cfg* cfg, const ic3_policy_packed* w,
                                    float* table, void* stream) {
  int rc = policy_check(cfg);
  if (rc) return rc;
  rc = packed_check(w);
  if (rc) return rc;
  if (!env || !env->grid || !table) return IC3_E_NULL;
  const int W = 2 * env->vision + 1;
  if (cfg->O != 2 + W * W * env->vocab || cfg->obs_vocab == 0) return IC3_E_RANGE;
  rc = ic3_tj_layout_check(env, cfg);
  if (rc) return rc;
  tj_encoder_table_kernel<<<env->h * env->w, cfg->H, 0, (cudaStream_t)stream>>>(*env, cfg->H, w->enc_wT, w->enc_b, table);
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}

extern "C" int ic3_encoder_dense(const ic3_policy_cfg* cfg, const ic3_policy_packed* w, const float* obs,
                                 float* x, void* stream) {
  int rc = policy_check(cfg);
  if (rc) return rc;
  rc = packed_check(w);
  if (rc) return rc;
  if (!obs || !x) return IC3_E_NULL;
  IC3_DISPATCH_H(cfg->H, launch_encoder_dense<HH>(cfg, w, obs, x, (cudaStream_t)stream));
}

extern "C" int ic3_pp_encoder_index(const ic3_pp_cfg* env, const ic3_pp_state* st, const ic3_policy_cfg* cfg,
                                    const ic3_policy_packed* w, float* x, void* stream) {
  int rc = policy_check(cfg);
  if (rc) return rc;
  rc = packed_check(w);
  if (rc) return rc;
  if (!env || !st || !st->loc || !x) return IC3_E_NULL;
  if (env->B != cfg->B || ic3_pp_agents(*env) != cfg->N || env->N >= IC3_MAX_AGENTS) return IC3_E_RANGE;
  const int W = 2 * env->vision + 1;
  if (cfg->O != W * W * (env->dim * env->dim + 4)) return IC3_E_RANGE;
  rc = ic3_pp_layout_check(env, cfg);
  if (rc) return rc;
  const bool split = cfg->obs_vocab > 0;
  const int rows = cfg->B * cfg->N, grid = (rows + 7) / 8;
  cudaStream_t s = (cudaStream_t)stream;
  switch (cfg->H) {
    case 32: pp_encoder_index_kernel<32><<<grid, 256, 0, s>>>(*env, *st, w->enc_wT, w->enc_b, x, split); break;
    case 64: pp_encoder_index_kernel<64><<<grid, 256, 0, s>>>(*env, *st, w->enc_wT, w->enc_b, x, split); break;
    case 128: pp_encoder_index_kernel<128><<<grid, 256, 0, s>>>(*env, *st, w->enc_wT, w->enc_b, x, split); break;
    default: return IC3_E_UNSUPPORTED;
  }
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}

extern "C" int ic3_tj_encoder_index(const ic3_tj_cfg* env, const ic3_tj_state* st, const ic3_policy_cfg* cfg,
                                    const ic3_policy_packed* w, float* x, void* stream) {
  int rc = policy_check(cfg);
  if (rc) return rc;
  rc = packed_check(w);
  if (rc) return rc;
  if (!env || !st || !st->loc || !st->alive || !st->last_act || !st->route_id || !env->grid || !x) return IC3_E_NULL;
  if (env->B != cfg->B || env->N != cfg->N) return IC3_E_RANGE;
  const int W = 2 * env->vision + 1;
  if (cfg->O != 2 + W * W * env->vocab) return IC3_E_RANGE;
  rc = ic3_tj_layout_check(env, cfg);
  if (rc) return rc;
  const bool split = cfg->obs_vocab > 0;
  const int rows = cfg->B * cfg->N, grid = (rows + 7) / 8;
  cudaStream_t s = (cudaStream_t)stream;
  switch (cfg->H) {
    case 32: tj_encoder_index_kernel<32><<<grid, 256, 0, s>>>(*env, *st, w->enc_wT, w->enc_b, x, split); break;
    case 64: tj_encoder_index_kernel<64><<<grid, 256, 0, s>>>(*env, *st, w->enc_wT, w->enc_b, x, split); break;
    case 128: tj_encoder_index_kernel<128><<<grid, 256, 0, s>>>(*env, *st, w->enc_wT, w->enc_b, x, split); break;
    default: return IC3_E_UNSUPPORTED;
  }
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}

extern "C" int ic3_policy_step(const ic3_policy_cfg* cfg, const ic3_policy_packed* w, const ic3_policy_io* io,
                               void* stream) {
  int rc = policy_check(cfg);
  if (rc) return rc;
  rc = packed_check(w);
  if (rc) return rc;
  if (!io || !io->h_out || !io->value || !io->logp) return IC3_E_NULL;
  if (!cfg->h_from_x && !io->h) return IC3_E_NULL;
  if (cfg->cell == IC3_CELL_LSTM && (!io->c || !io->c_out)) return IC3_E_NULL;
  if (cfg->hard_attn && !io->comm_action) return IC3_E_NULL;
  if (cfg->N > ROWS) return IC3_E_RANGE;
  if (io->workspace && w->lstm_img) {     // tcgen05 path (policy_tc.cu); otherwise the fp32 SIMT kernel below
    if (!policy_tc_capable(cfg)) return IC3_E_UNSUPPORTED;
    return ic3_tc_policy_step(cfg, w, io, (cudaStream_t)stream);
  }
  if (!io->x) return IC3_E_NULL;
  if (cfg->cell == IC3_CELL_TANH && (!w->f_wT || !w->f_b)) return IC3_E_NULL;
  PolicyArgs a{*cfg, *w, *io};
  IC3_DISPATCH_H(cfg->H, launch_policy<HH>(a, (cudaStream_t)stream));
}

extern "C" int ic3_sample_actions(const ic3_policy_cfg* cfg, const float* logp, const uint32_t* tick,
                                  const uint32_t* draws, int32_t* action, void* stream) {
  int rc = policy_check(cfg);
  if (rc) return rc;
  if (!logp || !action) return IC3_E_NULL;
  const int rows = cfg->B * cfg->N;
  sample_kernel<<<(rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*cfg, logp, tick, draws, action);
  IC3_LAUNCH_CHECK();
  return IC3_OK;
}
