// Fused per-step Sable inference for the rollout: SableNetwork.get_actions (networks/sable_network.py:443-482) for a
// batch of envs in ONE kernel — recurrent encoder over the A agents (utils/sable/encode.py:58-84, sable_network.py:139-156),
// the A autoregressive decoder steps (utils/sable/decode.py:111-153, sable_network.py:219-242,321-343), each followed by the
// distrax gumbel-max sample from the step's threefry key, and the value head. It replaces ~80 short launches per env step.
//
// Mapping: the envs of a rollout never interact, and inside one env the decoder is a chain (agent i's input token is agent
// i-1's sampled action), so one warp runs the whole chain for EPW envs with nothing but warp shuffles between stages:
//   * a 64-wide activation row lives in one float2 per lane (lane l = columns 2l, 2l+1), the same layout the row kernels use;
//   * a dense layer y = x W is 64 broadcast-FMA steps: x_k by shuffle, the k-th weight row from shared memory (256 contiguous
//     bytes per warp, conflict-free). The CTA streams the weight matrices of the step (0.4 MB, L2 resident) through two
//     32 KiB buffers with cp.async, one piece ahead of the arithmetic (the 64 x 256 projections go through as two 64 x 128 column
//     halves), so no weight load is ever waited for; EPW envs (x A tokens in the encoder) share each weight read. With 32 KiB
//     buffers TWO CTAs of 7 warps fit on an SM (80 KB of shared memory, 128 registers per thread each): they drift apart in phase, so
//     one CTA's state stream (HBM) runs under the other's dense layers (FMA) instead of the whole SM alternating between the two;
//   * the 64x64 retention states (3 x 16 KiB per env, the only large HBM stream of the rollout) are read row by row, 256
//     coalesced bytes per row and warp, 8 rows in flight per env. The decoder states are READ once per agent but WRITTEN once
//     per step: with H0 the stored state, lam the step's decay and (k_j, v_j) the tokens added so far,
//         ret_i = q_i (lam H0 + sum_{j<=i} k_j^T v_j) = lam (q_i H0) + sum_{j<=i} (q_i . k_j) v_j,
//     so agents 0..A-2 only read H0 and the last agent's pass also writes lam H0 + sum_j k_j^T v_j. Per env-step the state
//     traffic is 32 + 2 (16 A + 16) KiB instead of 32 (1 + 2 A) KiB.
// All arithmetic is fp32 FMA (no TF32 split on this path). Algorithmic HBM bytes per env-step: state traffic above +
// A (4 d + a + 4) in + 12 A out.
#include <stdlib.h>
#include "kernels.cuh"
#include "params.cuh"
#include "prng.cuh"

namespace magpo {
namespace {

constexpr float kEps = 1e-6f;
// envs per warp: 2 for large batches (every weight read from shared memory serves 2 A rows), 1 for small ones (twice the warps, half
// the dependent work per warp: the RWARE shard of 1024 envs is latency-bound, not bandwidth-bound)
constexpr int SS_WARPS = 8;    // max warps per CTA; two CTAs per SM
constexpr int SS_WBUF = kD * 2 * kD;  // floats of the largest staged piece [64, 128]
constexpr int SS_XROWS = 8;  // rows of the per-warp activation scratch (EPW x A <= 8)
constexpr uint32_t ss_smem(int warps) { return (uint32_t)((2 * SS_WBUF + warps * SS_XROWS * kD) * sizeof(float)); }
constexpr unsigned kFull = 0xffffffffu;

struct StepArgs {
  int B, d, a, max_step, gumbel_rows, dry;
  int keep_l2;               // decoder-state reads before the last agent's pass keep the default L2 policy (MAGPO_STEP_KEEP_L2, default 1)
  float kappa;
  const float* obs;          // [B,A,d]
  const uint8_t* mask;       // [B,A,a]
  const int32_t* step;       // [B,A]
  const uint8_t* prev_done;  // [B] or null
  const uint32_t* keys;      // [A][2] sample keys of this step
  const float* pe;           // [max_step+1, 64]
  const float* dec_tab;      // [(a+1) + (max_step+1), 256]: token rows then step rows of the decoder's first projection
  float *h_enc, *h_self, *h_cross;  // [B,64,64]
  int32_t* action;           // [B,A]
  float *log_prob, *value;   // [B,A]
  float* masked_logits;      // [B,A,a] or null
};

__device__ __forceinline__ float2 ldg2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
__device__ __forceinline__ float2 f2add(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
// ex2.approx / rcp.approx forms (2 ulp each): a fifth of this kernel's instructions were expf + IEEE division + tanhf expansions. The
// logits move at the 1e-7 level, well inside the 1e-6 the gumbel-argmax is already robust to (the oracle sums in another order anyway);
// every action-parity test of the suite runs on this path.
__device__ __forceinline__ float swishf(float x) { return x * __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float gelu_step(float x) {
  const float u = 0.7978845608028654f * (x + 0.044715f * x * x * x);
  const float t = 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * u));
  return 0.5f * x * (1.0f + t);
}
// acc + s * v on both halves with one packed instruction (FFMA2, sm_100: two IEEE fp32 FMAs per lane and issue slot)
__device__ __forceinline__ float2 fma2(float s_, float2 v, float2 acc) { return __ffma2_rn(make_float2(s_, s_), v, acc); }

// y[r][j] (+)= x[r] W[:, 64 j + (2l, 2l+1)]   for R rows sharing every weight load; W row-major [64, ldw]
// The R input rows are parked in the warp's shared scratch `xs` [R][64] and read back four k at a time as broadcast LDS.128
// (one shared-memory instruction per row and 4 k instead of four shuffles).
template <int NB, int R>
__device__ __forceinline__ void dense(const float* __restrict__ W /*shared*/, int ldw, const float2 (&x)[R], float2 (&y)[R][NB],
                                      float* __restrict__ xs, int lane) {
#pragma unroll
  for (int r = 0; r < R; ++r) {
    *reinterpret_cast<float2*>(xs + r * kD + 2 * lane) = x[r];
#pragma unroll
    for (int j = 0; j < NB; ++j) y[r][j] = make_float2(0.f, 0.f);
  }
  __syncwarp();
#pragma unroll 2
  for (int k4 = 0; k4 < 16; ++k4) {
    float4 xv[R];
#pragma unroll
    for (int r = 0; r < R; ++r) xv[r] = *reinterpret_cast<const float4*>(xs + r * kD + 4 * k4);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      float2 w[NB];
#pragma unroll
      for (int j = 0; j < NB; ++j) w[j] = *reinterpret_cast<const float2*>(W + (4 * k4 + kk) * ldw + 64 * j + 2 * lane);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const float xk = kk == 0 ? xv[r].x : (kk == 1 ? xv[r].y : (kk == 2 ? xv[r].z : xv[r].w));
#pragma unroll
        for (int j = 0; j < NB; ++j) y[r][j] = fma2(xk, w[j], y[r][j]);
      }
    }
  }
  __syncwarp();  // the scratch is rewritten by the next layer
}
template <int R>
__device__ __forceinline__ void dense1(const float* __restrict__ W, const float2 (&x)[R], float2 (&y)[R], float* __restrict__ xs,
                                       int lane) {
  float2 t[R][1];
  dense<1, R>(W, kD, x, t, xs, lane);
#pragma unroll
  for (int r = 0; r < R; ++r) y[r] = t[r][0];
}

// Weight pipeline: every thread copies its 16-byte pieces of the next piece — 64 rows x `cols` floats out of a row-major matrix with
// leading dimension `ld` — into the idle buffer (compact: leading dimension `cols`).
__device__ __forceinline__ void stage_issue(float* dst /*shared*/, const float* __restrict__ src, int cols, int ld) {
  const uint32_t d0 = (uint32_t)__cvta_generic_to_shared(dst);
  const int per_row = cols >> 2;  // 16-byte pieces per row
  for (int i = threadIdx.x; i < kD * per_row; i += blockDim.x) {
    const int r = i / per_row, c = (i - r * per_row) << 2;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d0 + (uint32_t)(r * cols + c) * 4u), "l"(src + (size_t)r * ld + c) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}
// the layer issued last has landed for every thread, and every warp is done with the other buffer
__device__ __forceinline__ void stage_wait() {
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
}

// RMSNorm(p) * scale   (flax nn.RMSNorm, eps 1e-6)
__device__ __forceinline__ float2 rmsnorm(float2 p, float2 sc) {
  const float rstd = rsqrtf(warp_sum(p.x * p.x + p.y * p.y) * (1.0f / kD) + kEps);
  return make_float2(p.x * (rstd * sc.x), p.y * (rstd * sc.y));
}
// swish(g) * GroupNorm_1(ret)  (flax fast variance; retention.py:289-295)
__device__ __forceinline__ float2 gn_gate(float2 g, float2 x, float2 sc, float2 bi) {
  const float mean = warp_sum(x.x + x.y) * (1.0f / kD);
  const float m2 = warp_sum(x.x * x.x + x.y * x.y) * (1.0f / kD);
  const float rstd = rsqrtf(fmaxf(0.0f, m2 - mean * mean) + kEps);
  return make_float2(swishf(g.x) * ((x.x - mean) * rstd * sc.x + bi.x), swishf(g.y) * ((x.y - mean) * rstd * sc.y + bi.y));
}
__device__ __forceinline__ float2 pe_row(const float* __restrict__ pe, int step, int max_step, int lane) {
  return ldg2(pe + (size_t)min(max(step, 0), max_step) * kD + 2 * lane);
}
// component r of a row held as float2 per lane
__device__ __forceinline__ float row_elem(float2 v, int r) { return __shfl_sync(kFull, (r & 1) ? v.y : v.x, r >> 1); }

// pull one 16 KiB state towards L2 ahead of its row-by-row read (one bulk prefetch instruction)
__device__ __forceinline__ void prefetch_state(const float* H) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(H), "r"((uint32_t)(kD * kD * sizeof(float))) : "memory");
}

// state rows r0..r0+7 of env state H. KEEP = false: evict-first (the last read of the state in this launch). KEEP = true: default
// policy — a decoder state is read once per agent, and next to evict-first streams the lines of an earlier agent's pass survive in
// L2 longer (tools/step_l2_experiment.sh: RWARE shard, 1024 envs x 4 agents, whose states fit L2: rollout 23.3 -> 22.3 ms in both
// A/B runs; LBF, 8192 envs x 2 agents: 49.8 -> 48.4 ms in one A/B run and no difference in two others, DRAM bytes per launch
// unchanged under ncu; explicit evict_last / evict_normal createpolicy operands and a second L2 prefetch between the passes
// measured no better)
template <bool KEEP = false>
__device__ __forceinline__ void load_rows(float2 (&h)[8], const float* __restrict__ H, int r0, int lane) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float2* src = reinterpret_cast<const float2*>(H + (size_t)(r0 + j) * kD + 2 * lane);
    if (KEEP) {
      float2 x;
      asm volatile("ld.global.v2.f32 {%0, %1}, [%2];" : "=f"(x.x), "=f"(x.y) : "l"(src));
      h[j] = x;
    } else {
      h[j] = __ldcs(src);
    }
  }
}

// Decoder retention of agent i (token-causal): out_e = lam (q_e H0_e) + sum_{j<=i} (q_e . k_ej) v_ej, H0 read-only; the last
// agent's pass also writes lam H0 + sum_j k_j^T v_j. Both envs' rows are in flight together.
template <int A, int EPW>
__device__ __forceinline__ void decoder_retention(int i, float* __restrict__ Hall, const int (&b)[EPW], const bool (&live)[EPW],
                                                  const float (&lam)[EPW], const float2 (&q)[EPW], const float2 (&k)[EPW][A],
                                                  const float2 (&v)[EPW][A], float2 (&out)[EPW], int lane, bool keep_l2) {
  float2 acc[EPW];
#pragma unroll
  for (int e = 0; e < EPW; ++e) acc[e] = make_float2(0.f, 0.f);
  for (int r0 = 0; r0 < kD; r0 += 8) {
    float2 h[EPW][8];
#pragma unroll
    for (int e = 0; e < EPW; ++e) {
      if (i == A - 1 || !keep_l2) load_rows<false>(h[e], Hall + (size_t)b[e] * kD * kD, r0, lane);
      else load_rows<true>(h[e], Hall + (size_t)b[e] * kD * kD, r0, lane);
    }
#pragma unroll
    for (int e = 0; e < EPW; ++e) {
      float* H = Hall + (size_t)b[e] * kD * kD;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        acc[e] = fma2(row_elem(q[e], r0 + j), h[e][j], acc[e]);
        if (i == A - 1 && live[e]) {
          float2 hn = make_float2(h[e][j].x * lam[e], h[e][j].y * lam[e]);
#pragma unroll
          for (int jj = 0; jj < A; ++jj) {
            hn = fma2(row_elem(k[e][jj], r0 + j), v[e][jj], hn);
          }
          __stcs(reinterpret_cast<float2*>(H + (size_t)(r0 + j) * kD + 2 * lane), hn);
        }
      }
    }
  }
#pragma unroll
  for (int e = 0; e < EPW; ++e) {
    acc[e].x *= lam[e]; acc[e].y *= lam[e];
#pragma unroll
    for (int jj = 0; jj < A; ++jj)
      if (jj <= i) {
        const float qk = warp_sum(q[e].x * k[e][jj].x + q[e].y * k[e][jj].y);
        acc[e] = fma2(qk, v[e][jj], acc[e]);
      }
    out[e] = acc[e];
  }
}

template <int A, int KMAX, int EPW>
// two CTAs of <= 8 warps per SM: 128 registers per thread is the ceiling
__global__ void __launch_bounds__(256, 2)
sable_step_kernel(const GuiderP p, const StepArgs s) {
  extern __shared__ __align__(16) float wbuf[];  // two weight buffers of SS_WBUF floats
  float* const w_a = wbuf;
  float* const w_b = wbuf + SS_WBUF;
  float* const xs = wbuf + 2 * SS_WBUF + (threadIdx.x >> 5) * SS_XROWS * kD;  // this warp's activation scratch
  const int lane = threadIdx.x & 31;
  const int64_t pair = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // warps past the batch run dead (no stores)
  stage_issue(w_a, p.qkvg, 2 * kD, 4 * kD);  // [w_q | w_k]
  float* cur_w = w_a;  // buffer of the layer about to be computed
  float* nxt_w = w_b;  // buffer the following layer is prefetched into
  const bool full = !s.dry && s.action;
// the current layer's weights are complete and the other buffer is free: start the next layer's copy, then compute
#define LAYER(next_ptr, next_cols, next_ld)                    \
  stage_wait();                                               \
  if ((next_ptr) != nullptr) stage_issue(nxt_w, (next_ptr), (next_cols), (next_ld));
#define LAYER_DONE()                                          \
  { float* t_ = cur_w; cur_w = nxt_w; nxt_w = t_; }
  int b[EPW];
  bool live[EPW];
  float lam[EPW];
#pragma unroll
  for (int e = 0; e < EPW; ++e) {
    const int64_t be = pair * EPW + e;
    live[e] = be < s.B;
    b[e] = live[e] ? (int)be : s.B - 1;  // a dead slot recomputes the last env and writes nothing
    lam[e] = (s.prev_done && s.prev_done[b[e]]) ? 0.0f : s.kappa;
  }
  constexpr int RE = EPW * A;  // encoder rows of this warp: (env, agent)
  if (lane < EPW) {
    const int bl = lane == 0 ? b[0] : b[EPW - 1];
    prefetch_state(s.h_enc + (size_t)bl * kD * kD);
  }

  // ------------------------------------------------------------------ encoder
  float2 xin[RE], cur[RE];
  int stp[RE];
  if constexpr (KMAX > 0) {
    float2 w[KMAX];
    float sc[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
      w[k] = k < s.d ? ldg2(p.Wobs + (size_t)k * kD + 2 * lane) : make_float2(0.f, 0.f);
      sc[k] = k < s.d ? __ldg(p.obs_scale + k) : 0.f;
    }
    const float2 ln = ldg2(p.ln + 2 * lane);
    const float inv_d = 1.0f / (float)s.d;
#pragma unroll
    for (int r = 0; r < RE; ++r) {
      const int64_t row = (int64_t)b[r / A] * A + (r % A);
      float x[KMAX], ss = 0.f;
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        x[k] = k < s.d ? __ldg(s.obs + row * s.d + k) : 0.f;
        ss = fmaf(x[k], x[k], ss);
      }
      const float rstd0 = rsqrtf(ss * inv_d + kEps);
      float2 z = make_float2(0.f, 0.f);
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        const float o = x[k] * (rstd0 * sc[k]);
        z.x = fmaf(o, w[k].x, z.x);
        z.y = fmaf(o, w[k].y, z.y);
      }
      xin[r] = rmsnorm(make_float2(gelu_step(z.x), gelu_step(z.y)), ln);
      stp[r] = __ldg(s.step + row);
      cur[r] = f2add(xin[r], pe_row(s.pe, stp[r], s.max_step, lane));
    }
  } else {
    // wide observations (RWARE d = 75, the larger LBF scenarios): the embedding runs over chunks of 16 features; the RMSNorm
    // factor of the observation is linear in the projection, so it is applied once after the last chunk
    float2 zacc[RE];
    float ssq[RE];
#pragma unroll
    for (int r = 0; r < RE; ++r) {
      zacc[r] = make_float2(0.f, 0.f);
      ssq[r] = 0.f;
    }
    for (int k0 = 0; k0 < s.d; k0 += 16) {
      float2 w[16];
      float sc[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const int kk = k0 + k;
        w[k] = kk < s.d ? ldg2(p.Wobs + (size_t)kk * kD + 2 * lane) : make_float2(0.f, 0.f);
        sc[k] = kk < s.d ? __ldg(p.obs_scale + kk) : 0.f;
      }
#pragma unroll
      for (int r = 0; r < RE; ++r) {
        const int64_t row = (int64_t)b[r / A] * A + (r % A);
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const float x = (k0 + k) < s.d ? __ldg(s.obs + row * s.d + k0 + k) : 0.f;
          ssq[r] = fmaf(x, x, ssq[r]);
          const float o = x * sc[k];
          zacc[r].x = fmaf(o, w[k].x, zacc[r].x);
          zacc[r].y = fmaf(o, w[k].y, zacc[r].y);
        }
      }
    }
    const float2 ln = ldg2(p.ln + 2 * lane);
    const float inv_d = 1.0f / (float)s.d;
#pragma unroll
    for (int r = 0; r < RE; ++r) {
      const int64_t row = (int64_t)b[r / A] * A + (r % A);
      const float rstd0 = rsqrtf(ssq[r] * inv_d + kEps);
      xin[r] = rmsnorm(make_float2(gelu_step(zacc[r].x * rstd0), gelu_step(zacc[r].y * rstd0)), ln);
      stp[r] = __ldg(s.step + row);
      cur[r] = f2add(xin[r], pe_row(s.pe, stp[r], s.max_step, lane));
    }
  }
  float2 ret[RE], gate[RE];
  {
    float2 qkvg[RE][4];
    {
      float2 half[RE][2];
      LAYER(p.qkvg + 2 * kD, 2 * kD, 4 * kD)  // next: [w_v | w_g]
      dense<2, RE>(cur_w, 2 * kD, cur, half, xs, lane);
      LAYER_DONE()
#pragma unroll
      for (int r = 0; r < RE; ++r) { qkvg[r][0] = half[r][0]; qkvg[r][1] = half[r][1]; }
      LAYER(p.wo, kD, kD)
      dense<2, RE>(cur_w, 2 * kD, cur, half, xs, lane);
      LAYER_DONE()
#pragma unroll
      for (int r = 0; r < RE; ++r) { qkvg[r][2] = half[r][0]; qkvg[r][3] = half[r][1]; }
    }
    // retention: H <- lam H + sum_i k_i^T v_i ; ret_i = q_i H   (all A tokens are added before any output)
#pragma unroll
    for (int r = 0; r < RE; ++r) ret[r] = make_float2(0.f, 0.f);
    for (int r0 = 0; r0 < kD; r0 += 8) {
      float2 h[EPW][8];
#pragma unroll
      for (int e = 0; e < EPW; ++e) load_rows(h[e], s.h_enc + (size_t)b[e] * kD * kD, r0, lane);
#pragma unroll
      for (int e = 0; e < EPW; ++e) {
        float* H = s.h_enc + (size_t)b[e] * kD * kD;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int r = r0 + j;
          float2 hh = make_float2(h[e][j].x * lam[e], h[e][j].y * lam[e]);
#pragma unroll
          for (int i = 0; i < A; ++i) {
            hh = fma2(row_elem(qkvg[e * A + i][1], r), qkvg[e * A + i][2], hh);
          }
          if (!s.dry && live[e]) __stcs(reinterpret_cast<float2*>(H + (size_t)r * kD + 2 * lane), hh);
#pragma unroll
          for (int i = 0; i < A; ++i) {
            ret[e * A + i] = fma2(row_elem(qkvg[e * A + i][0], r), hh, ret[e * A + i]);
          }
        }
      }
    }
#pragma unroll
    for (int r = 0; r < RE; ++r) gate[r] = qkvg[r][3];
    if (full && lane < EPW) {  // the decoder states are needed ~10 layers from now
      const int bl = lane == 0 ? b[0] : b[EPW - 1];
      prefetch_state(s.h_self + (size_t)bl * kD * kD);
      prefetch_state(s.h_cross + (size_t)bl * kD * kD);
    }
  }
  float2 x[RE], xpe[RE];
  {
    const float2 gs = ldg2(p.gn_s + 2 * lane), gb = ldg2(p.gn_b + 2 * lane);
#pragma unroll
    for (int r = 0; r < RE; ++r) cur[r] = gn_gate(gate[r], ret[r], gs, gb);
    float2 o[RE];
    LAYER(p.ffn_gl, 2 * kD, 2 * kD)
    dense1<RE>(cur_w, cur, o, xs, lane);
    LAYER_DONE()
    const float2 ln1 = ldg2(p.ln1 + 2 * lane);
#pragma unroll
    for (int r = 0; r < RE; ++r) xin[r] = rmsnorm(f2add(o[r], xin[r]), ln1);  // x1
    float2 gl[RE][2];
    LAYER(p.ffn_out, kD, kD)
    dense<2, RE>(cur_w, 2 * kD, xin, gl, xs, lane);
    LAYER_DONE()
#pragma unroll
    for (int r = 0; r < RE; ++r) cur[r] = make_float2(swishf(gl[r][0].x) * gl[r][1].x, swishf(gl[r][0].y) * gl[r][1].y);
    LAYER(p.h0_w, kD, kD)
    dense1<RE>(cur_w, cur, o, xs, lane);
    LAYER_DONE()
    const float2 ln2 = ldg2(p.ln2 + 2 * lane);
#pragma unroll
    for (int r = 0; r < RE; ++r) {
      x[r] = rmsnorm(f2add(o[r], xin[r]), ln2);
      xpe[r] = f2add(x[r], pe_row(s.pe, stp[r], s.max_step, lane));
    }
    // value head: Dense(64) -> gelu -> RMSNorm -> Dense(1)
    LAYER(full ? p.wo1 : nullptr, kD, kD)
    dense1<RE>(cur_w, x, o, xs, lane);
    LAYER_DONE()
    const float2 hb = ldg2(p.h0_b + 2 * lane), hs = ldg2(p.h2_s + 2 * lane), hw = ldg2(p.h3_w + 2 * lane);
    const float hb3 = __ldg(p.h3_b);
#pragma unroll
    for (int r = 0; r < RE; ++r) {
      const float2 hn = rmsnorm(make_float2(gelu_step(o[r].x + hb.x), gelu_step(o[r].y + hb.y)), hs);
      const float v = warp_sum(hn.x * hw.x + hn.y * hw.y) + hb3;
      if (lane == 0 && live[r / A]) s.value[(int64_t)b[r / A] * A + (r % A)] = v;
    }
  }
  if (!full) return;

  // ------------------------------------------------------------------ decoder: A autoregressive steps
  float2 k1[EPW][A], v1[EPW][A], k2[EPW][A], v2[EPW][A];  // tokens added to the self / cross states so far
#pragma unroll
  for (int e = 0; e < EPW; ++e)
#pragma unroll
    for (int jj = 0; jj < A; ++jj) k1[e][jj] = v1[e][jj] = k2[e][jj] = v2[e][jj] = make_float2(0.f, 0.f);
  int prev_act[EPW];
#pragma unroll
  for (int e = 0; e < EPW; ++e) prev_act[e] = 0;
  // a real loop (the body is ~2k instructions: unrolling it A times overflows the instruction cache); the per-agent k/v
  // history stays in registers through compile-time indices under runtime predicates
#pragma unroll 1
  for (int i = 0; i < A; ++i) {
    float2 xD[EPW];
    int st[EPW], tokv[EPW];
    {
      const float2 dln = ldg2(p.dln + 2 * lane);
#pragma unroll
      for (int e = 0; e < EPW; ++e) {
        const int tok = i == 0 ? 0 : 1 + prev_act[e];  // start-of-timestep token, else one-hot(previous action)
        tokv[e] = tok;
        const float2 z = ldg2(p.Wa + (size_t)tok * kD + 2 * lane);
        xD[e] = rmsnorm(make_float2(gelu_step(z.x), gelu_step(z.y)), dln);
        st[e] = 0;
#pragma unroll
        for (int jj = 0; jj < A; ++jj)
          if (jj == i) st[e] = stp[e * A + jj];
      }
    }
    // ---- self retention
    float2 r1[EPW], g1[EPW];
    {
      // (xD + pe[step]) W_qkvg1 = xD W + pe[step] W, and xD only depends on the input token (a + 1 values): both terms come
      // from the tables sable_step_tables() builds once per rollout instead of a 64 x 256 layer per agent
      float2 qkvg[EPW][4];
#pragma unroll
      for (int e = 0; e < EPW; ++e) {
        const float* ut = s.dec_tab + (size_t)tokv[e] * 4 * kD;
        const float* pt = s.dec_tab + (size_t)(s.a + 1 + min(max(st[e], 0), s.max_step)) * 4 * kD;
#pragma unroll
        for (int j = 0; j < 4; ++j) qkvg[e][j] = f2add(ldg2(ut + 64 * j + 2 * lane), ldg2(pt + 64 * j + 2 * lane));
      }
#pragma unroll
      for (int e = 0; e < EPW; ++e) {
#pragma unroll
        for (int jj = 0; jj < A; ++jj)
          if (jj == i) { k1[e][jj] = qkvg[e][1]; v1[e][jj] = qkvg[e][2]; }
        g1[e] = qkvg[e][3];
      }
      float2 q1[EPW];
#pragma unroll
      for (int e = 0; e < EPW; ++e) q1[e] = qkvg[e][0];
      decoder_retention<A, EPW>(i, s.h_self, b, live, lam, q1, k1, v1, r1, lane, s.keep_l2 != 0);
    }
    float2 rpe[EPW];
    {
      const float2 gs = ldg2(p.gn1_s + 2 * lane), gb = ldg2(p.gn1_b + 2 * lane), dln1 = ldg2(p.dln1 + 2 * lane);
      float2 t[EPW], o[EPW];
#pragma unroll
      for (int e = 0; e < EPW; ++e) t[e] = gn_gate(g1[e], r1[e], gs, gb);
      LAYER(p.qkvg2, 2 * kD, 4 * kD)  // next: [w_q | w_k] of the cross retention
      dense1<EPW>(cur_w, t, o, xs, lane);
      LAYER_DONE()
#pragma unroll
      for (int e = 0; e < EPW; ++e)
        rpe[e] = f2add(rmsnorm(f2add(o[e], xD[e]), dln1), pe_row(s.pe, st[e], s.max_step, lane));
    }
    // ---- cross retention: key = value = r (+PE), query = obs_rep (+PE)
    float2 yv[EPW];
    {
      float2 q2[EPW], qin[EPW], kvg[EPW][3];
#pragma unroll
      for (int e = 0; e < EPW; ++e) {
        qin[e] = xpe[e * A];
#pragma unroll
        for (int jj = 1; jj < A; ++jj)
          if (jj == i) qin[e] = xpe[e * A + jj];
      }
      {
        float2 t[EPW][1];
        LAYER(p.qkvg2 + 2 * kD, 2 * kD, 4 * kD)  // next: [w_v | w_g]
        dense<1, EPW>(cur_w, 2 * kD, qin, t, xs, lane);
#pragma unroll
        for (int e = 0; e < EPW; ++e) q2[e] = t[e][0];
        dense<1, EPW>(cur_w + kD, 2 * kD, rpe, t, xs, lane);
#pragma unroll
        for (int e = 0; e < EPW; ++e) kvg[e][0] = t[e][0];
        LAYER_DONE()
        float2 vg[EPW][2];
        LAYER(p.wo2, kD, kD)
        dense<2, EPW>(cur_w, 2 * kD, rpe, vg, xs, lane);
        LAYER_DONE()
#pragma unroll
        for (int e = 0; e < EPW; ++e) { kvg[e][1] = vg[e][0]; kvg[e][2] = vg[e][1]; }
      }
      float2 r2[EPW];
#pragma unroll
      for (int e = 0; e < EPW; ++e) {
#pragma unroll
        for (int jj = 0; jj < A; ++jj)
          if (jj == i) { k2[e][jj] = kvg[e][0]; v2[e][jj] = kvg[e][1]; }
      }
      decoder_retention<A, EPW>(i, s.h_cross, b, live, lam, q2, k2, v2, r2, lane, s.keep_l2 != 0);
      const float2 gs = ldg2(p.gn2_s + 2 * lane), gb = ldg2(p.gn2_b + 2 * lane), dln2 = ldg2(p.dln2 + 2 * lane);
      float2 t[EPW], o[EPW];
#pragma unroll
      for (int e = 0; e < EPW; ++e) t[e] = gn_gate(kvg[e][2], r2[e], gs, gb);
      LAYER(p.dffn_gl, 2 * kD, 2 * kD)
      dense1<EPW>(cur_w, t, o, xs, lane);
      LAYER_DONE()
#pragma unroll
      for (int e = 0; e < EPW; ++e) {
        float2 xr = x[e * A];
#pragma unroll
        for (int jj = 1; jj < A; ++jj)
          if (jj == i) xr = x[e * A + jj];
        yv[e] = rmsnorm(f2add(o[e], xr), dln2);
      }
    }
    // ---- SwiGLU FFN, head, sample
    {
      float2 gl[EPW][2], t[EPW], o[EPW];
      LAYER(p.dffn_out, kD, kD)
      dense<2, EPW>(cur_w, 2 * kD, yv, gl, xs, lane);
      LAYER_DONE()
#pragma unroll
      for (int e = 0; e < EPW; ++e) t[e] = make_float2(swishf(gl[e][0].x) * gl[e][1].x, swishf(gl[e][0].y) * gl[e][1].y);
      LAYER(p.dh0_w, kD, kD)
      dense1<EPW>(cur_w, t, o, xs, lane);
      LAYER_DONE()
      const float2 dln3 = ldg2(p.dln3 + 2 * lane);
#pragma unroll
      for (int e = 0; e < EPW; ++e) t[e] = rmsnorm(f2add(o[e], yv[e]), dln3);  // xd
      LAYER(i + 1 < A ? p.wo1 : nullptr, kD, kD)
      dense1<EPW>(cur_w, t, o, xs, lane);
      LAYER_DONE()
      const float2 hb = ldg2(p.dh0_b + 2 * lane), hs = ldg2(p.dh2_s + 2 * lane);
      float2 hn[EPW];
#pragma unroll
      for (int e = 0; e < EPW; ++e) hn[e] = rmsnorm(make_float2(gelu_step(o[e].x + hb.x), gelu_step(o[e].y + hb.y)), hs);
      // logits: lane j < a owns action j
      float lg[EPW];
#pragma unroll
      for (int e = 0; e < EPW; ++e) lg[e] = lane < s.a ? __ldg(p.dh3_b + lane) : 0.f;
      const int jc = lane < s.a ? lane : 0;
#pragma unroll 4
      for (int k2i = 0; k2i < 32; ++k2i) {
        const float wa = __ldg(p.dh3_w + (size_t)(2 * k2i) * s.a + jc), wb = __ldg(p.dh3_w + (size_t)(2 * k2i + 1) * s.a + jc);
#pragma unroll
        for (int e = 0; e < EPW; ++e) {
          lg[e] = fmaf(__shfl_sync(kFull, hn[e].x, k2i), wa, lg[e]);
          lg[e] = fmaf(__shfl_sync(kFull, hn[e].y, k2i), wb, lg[e]);
        }
      }
      // distrax.Categorical(logits=masked).sample_and_log_prob(seed=sample_key)  (decode.py:135-142): noise shape (1,E,1,a)
      const uint32_t key0 = __ldg(s.keys + 2 * i), key1 = __ldg(s.keys + 2 * i + 1);
#pragma unroll
      for (int e = 0; e < EPW; ++e) {
        const int64_t row = (int64_t)b[e] * A + i;
        const bool mine = lane < s.a;
        const bool legal = mine && s.mask[row * s.a + jc];
        const float ml = legal ? lg[e] : kF32Min;
        const float mx = warp_max(mine ? ml : kF32Min);
        const float se = warp_sum(mine ? expf(ml - mx) : 0.f);
        const float lp = ml - (mx + logf(se));
        const uint64_t ctr = (uint64_t)(b[e] % s.gumbel_rows) * (uint64_t)s.a + (uint64_t)jc;
        float sc = mine ? prng_gumbel_from_bits(prng_bits_i(key0, key1, ctr)) + lp : -INFINITY;
        int idx = mine ? lane : 0x7fffffff;
        // argmax, first index on ties (jnp.argmax)
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) {
          const float os = __shfl_xor_sync(kFull, sc, o2);
          const int oi = __shfl_xor_sync(kFull, idx, o2);
          if (os > sc || (os == sc && oi < idx)) { sc = os; idx = oi; }
        }
        const float best_lp = __shfl_sync(kFull, lp, idx);
        prev_act[e] = idx;
        if (live[e]) {
          if (lane == 0) { s.action[row] = idx; s.log_prob[row] = best_lp; }
          if (s.masked_logits && mine) s.masked_logits[row * s.a + lane] = ml;
        }
      }
    }
  }
}

// Row r < a + 1: (RMSNorm(gelu(Wa[r])) * dln) W_qkvg1 (the decoder input token r); row a + 1 + t: pe[t] W_qkvg1.
__global__ void __launch_bounds__(256)
decoder_tables_kernel(const GuiderP p, int a, int max_step, const float* __restrict__ pe, float* __restrict__ tab) {
  __shared__ float x[kD];
  const int r = blockIdx.x, lane = threadIdx.x & 31;
  if (threadIdx.x < 32) {
    float2 v;
    if (r <= a) {
      const float2 z = ldg2(p.Wa + (size_t)r * kD + 2 * lane);
      v = rmsnorm(make_float2(gelu_step(z.x), gelu_step(z.y)), ldg2(p.dln + 2 * lane));
    } else {
      v = ldg2(pe + (size_t)(r - a - 1) * kD + 2 * lane);
    }
    x[2 * lane] = v.x;
    x[2 * lane + 1] = v.y;
  }
  __syncthreads();
  float acc = 0.f;
#pragma unroll 8
  for (int k = 0; k < kD; ++k) acc = fmaf(x[k], __ldg(p.qkvg1 + (size_t)k * 4 * kD + threadIdx.x), acc);
  tab[(size_t)r * 4 * kD + threadIdx.x] = acc;
}

// Warps per CTA. Two CTAs share an SM (296 CTA slots): pick the CTA size whose last wave is fullest; small batches keep >= 6 warps,
// because every CTA streams the step's weights (0.4 MB) through its own shared memory (RWARE shard of 1024 envs, rollout of 128
// steps: 118 ms at 4 warps per CTA, 34.8 ms at 7 — tools/step_warps_experiment.sh).
int pick_warps(int64_t units) {
  static int forced_warps = -1;
  if (forced_warps < 0) {
    const char* e = getenv("MAGPO_STEP_WARPS");
    forced_warps = e ? std::min(std::max(atoi(e), 1), SS_WARPS) : 0;
  }
  if (forced_warps) return forced_warps;
  const int64_t slots = 2 * kNumSMs;
  int best = 7;
  double best_eff = -1.0;
  for (int w = 6; w <= SS_WARPS; ++w) {
    const int64_t ctas = ceil_div(units, w);
    const double eff = (double)units / ((double)ceil_div(ctas, slots) * slots * w);  // useful warps / warp slots over all waves
    if (eff > best_eff + 1e-9) { best_eff = eff; best = w; }
  }
  return best;
}

template <int A, int EPW>
int launch_ae(cudaStream_t st, const GuiderP& p, const StepArgs& s) {
  const int64_t units = ceil_div(s.B, EPW);  // warps of work
  const int warps = pick_warps(units);
  const unsigned grid = (unsigned)ceil_div(units, warps);
  const unsigned threads = (unsigned)warps * 32;
  const uint32_t smem = ss_smem(warps);
  if (once_per_device(ONCE_SABLE_STEP_1 + (A - 1) * 2 + (EPW - 1))) {
    const int cap = (int)ss_smem(SS_WARPS);
    MAGPO_CUDA_OK(cudaFuncSetAttribute(sable_step_kernel<A, 4, EPW>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    MAGPO_CUDA_OK(cudaFuncSetAttribute(sable_step_kernel<A, 8, EPW>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    MAGPO_CUDA_OK(cudaFuncSetAttribute(sable_step_kernel<A, 16, EPW>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    MAGPO_CUDA_OK(cudaFuncSetAttribute(sable_step_kernel<A, 0, EPW>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
  }
  if (s.d <= 4) sable_step_kernel<A, 4, EPW><<<grid, threads, smem, st>>>(p, s);
  else if (s.d <= 8) sable_step_kernel<A, 8, EPW><<<grid, threads, smem, st>>>(p, s);
  else if (s.d <= 16) sable_step_kernel<A, 16, EPW><<<grid, threads, smem, st>>>(p, s);
  else sable_step_kernel<A, 0, EPW><<<grid, threads, smem, st>>>(p, s);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

// envs per warp: 2 when the batch fills the 296 CTA slots anyway, 1 below that (twice the warps, half the chain per warp)
int envs_per_warp(int64_t B) {
  static int forced_epw = -1;
  if (forced_epw < 0) {
    const char* e = getenv("MAGPO_STEP_EPW");
    forced_epw = e ? atoi(e) : 0;
  }
  return (forced_epw == 1 || forced_epw == 2) ? forced_epw : (B <= 2048 ? 1 : 2);
}

template <int A>
int launch_a(cudaStream_t st, const GuiderP& p, const StepArgs& s) {
  return envs_per_warp(s.B) == 1 ? launch_ae<A, 1>(st, p, s) : launch_ae<A, 2>(st, p, s);
}

}  // namespace

bool sable_step_supported(int A, int d, int a) { return A >= 1 && A <= 4 && d >= 1 && d <= 128 && a >= 1 && a <= 32; }

size_t sable_step_table_floats(const MagpoNetCfg* net) { return (size_t)(net->action_dim + 1 + net->max_step_count + 1) * 4 * kD; }

// Once per parameter set (the rollout: once per call): the decoder's first-projection tables read by sable_step().
int sable_step_tables(cudaStream_t st, const MagpoNetCfg* net, const GuiderP& p, const float* pe, float* tab) {
  decoder_tables_kernel<<<net->action_dim + 1 + net->max_step_count + 1, 256, 0, st>>>(p, net->action_dim, net->max_step_count, pe, tab);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

// One SableNetwork.get_actions for B envs. action == nullptr (bootstrap): encoder + value only, states untouched.
int sable_step(cudaStream_t st, const MagpoNetCfg* net, int B, int gumbel_rows, const GuiderP& p, float kappa, const float* agents_view,
               const uint8_t* action_mask, const int32_t* step_count, const uint8_t* prev_done, const uint32_t* sample_keys,
               const float* pe, const float* dec_tab, MagpoSableHState hs, bool dry, int32_t* action, float* log_prob, float* value,
               float* masked_logits) {
  if (B <= 0) return MAGPO_OK;
  const int A = net->n_agents;
  if (!sable_step_supported(A, net->obs_dim, net->action_dim)) return MAGPO_ERR_UNSUPPORTED;
  StepArgs s;
  s.B = B; s.d = net->obs_dim; s.a = net->action_dim; s.max_step = net->max_step_count; s.gumbel_rows = gumbel_rows;
  s.dry = (dry || !action) ? 1 : 0;
  static int keep_l2 = -1;
  if (keep_l2 < 0) {
    const char* e = getenv("MAGPO_STEP_KEEP_L2");
    keep_l2 = e ? (atoi(e) != 0) : 1;
  }
  s.keep_l2 = keep_l2;
  s.kappa = kappa;
  s.obs = agents_view; s.mask = action_mask; s.step = step_count; s.prev_done = prev_done; s.keys = sample_keys; s.pe = pe;
  s.dec_tab = dec_tab;
  s.h_enc = hs.encoder; s.h_self = hs.decoder_self; s.h_cross = hs.decoder_cross;
  s.action = action; s.log_prob = log_prob; s.value = value; s.masked_logits = masked_logits;
  const double state_bytes = s.dry ? 16384.0 : (32768.0 + 2.0 * (16384.0 * A + 16384.0));
  ProfScope ps(PROF_SAMPLE, st, (double)B * (state_bytes + A * (4.0 * s.d + s.a + 4.0) + 12.0 * A));
  switch (A) {
    case 1: return launch_a<1>(st, p, s);
    case 2: return launch_a<2>(st, p, s);
    case 3: return launch_a<3>(st, p, s);
    default: return launch_a<4>(st, p, s);
  }
}

}  // namespace magpo

// Host-only: the envs per warp and warps per CTA the fused step kernel launches with for B envs (tests assert which branch a case
// covers).
extern "C" int magpo_debug_step_plan(int32_t B, int32_t* epw, int32_t* warps) {
  if (B < 1 || !epw || !warps) return MAGPO_ERR_ARG;
  *epw = magpo::envs_per_warp(B);
  *warps = magpo::pick_warps(magpo::ceil_div(B, *epw));
  return MAGPO_OK;
}
