// Fused row chains of the Sable guider's training forward (sable_network.py:111-156,296-343; retention.py:289-295; torsos.py:79-99).
// Retention is the only cross-row operator of the network, so between two retentions every token row runs through a chain of row-local
// layers. Two persistent tcgen05 kernels cover the chains after a retention (building blocks: chain.cuh):
//   chain_gate_kernel   gated = swish(g) * GroupNorm(ret) -> o = gated W_o -> y = RMSNorm(o + res) (+PE)
//                       [-> gl = y [W_gate|W_linear] -> hmid = swish(gl_a) * gl_b]
//   chain_tail_kernel   f = hmid W_out -> x = RMSNorm(f + res) (+PE, [-> q = xpe W_q]) -> zh = x W_h0 + b -> head(gelu, RMSNorm, Dense)
// Each token row is read once, every activation the backward needs is written once, nothing else touches HBM; the GEMMs are 3xTF32
// (x_lo W_hi + x_hi W_lo + x_hi W_hi, fp32 accumulation in tensor memory) exactly as in gemm_tc.cu.
#include <cuda.h>

#include "chain.cuh"
#include "common.cuh"
#include "kernels.cuh"

namespace magpo {
namespace {
using namespace chain;

constexpr float kEps = 1e-6f;

struct Carve {
  uint8_t *sW, *ring, *obuf;
  float* sPar;  // small per-kernel parameter vectors
  uint64_t *in_full, *in_empty, *a_ready, *d_ready, *in_done, *b_ready;
  uint32_t* tmem_ptr;
};

__device__ __forceinline__ Carve carve_smem(uint8_t* smem_raw, const ChainCommon& cc) {
  Carve c;
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  c.sW = base;
  c.ring = c.sW + cc.w_bytes;
  c.obuf = c.ring + (size_t)cc.ring_slots * CH_SLOT;
  c.sPar = reinterpret_cast<float*>(c.obuf + 2 * 2 * CH_SLOT);
  uint64_t* bars = reinterpret_cast<uint64_t*>(c.sPar + cc.par_floats);
  c.in_full = bars;
  c.in_empty = bars + CH_MAX_RING;
  c.a_ready = bars + 2 * CH_MAX_RING;
  c.d_ready = c.a_ready + 2;
  c.in_done = c.d_ready + 2;
  c.b_ready = c.in_done + 2;
  c.tmem_ptr = reinterpret_cast<uint32_t*>(c.b_ready + 1);
  return c;
}
inline uint32_t chain_smem_bytes(uint32_t w_bytes, int ring_slots, int par_floats) {
  return 1024 + w_bytes + (uint32_t)ring_slots * CH_SLOT + 4 * CH_SLOT + (uint32_t)par_floats * 4 + (2 * CH_MAX_RING + 7) * 8 + 16;
}

// barriers + TMEM allocation; every thread of the CTA calls this once
__device__ __forceinline__ uint32_t chain_setup(const Carve& c, const ChainCommon& cc) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < cc.ring_slots; ++i) {
      mbar_init(&c.in_full[i], 1);
      mbar_init(&c.in_empty[i], 4);  // one arrival per warp of the consuming row group
    }
    for (int g = 0; g < 2; ++g) {
      mbar_init(&c.a_ready[g], 4);
      mbar_init(&c.d_ready[g], 1);
      mbar_init(&c.in_done[g], 4);
    }
    mbar_init(c.b_ready, 1);
    fence_barrier_init();
  } else if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(c.tmem_ptr)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return *c.tmem_ptr;
}
__device__ __forceinline__ void chain_teardown(uint32_t tmem_base) {
  tc_fence_before();
  __syncthreads();
  if ((threadIdx.x >> 5) == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// warp 0, one thread: weights once, then the input boxes of this CTA's tiles in consumption order
__device__ __forceinline__ void chain_producer(const Carve& c, const ChainCommon& cc, const ChainMaps& m) {
  mbar_expect_tx(c.b_ready, cc.w_bytes);
  for (int i = 0; i < cc.n_gemm; ++i) {
    const uint32_t chunk = (uint32_t)cc.g_N[i] * 128u, image = 2 * chunk;
    for (int kc = 0; kc < 2; ++kc) {
      tma_load_2d(c.sW + cc.g_boff[i] + kc * chunk, &m.w[2 * i], kc * 32, cc.g_wrow[i], c.b_ready);
      tma_load_2d(c.sW + cc.g_boff[i] + image + kc * chunk, &m.w[2 * i + 1], kc * 32, cc.g_wrow[i], c.b_ready);
    }
  }
  uint32_t it = 0;
  for (int tile = blockIdx.x; tile < cc.num_tiles; tile += gridDim.x) {
    for (int j = 0; j < cc.n_in; ++j, ++it) {
      const uint32_t s = it % (uint32_t)cc.ring_slots, ph = (it / (uint32_t)cc.ring_slots) & 1u;
      mbar_wait(&c.in_empty[s], ph ^ 1u);
      mbar_expect_tx(&c.in_full[s], CH_SLOT);
      tma_load_2d(c.ring + (size_t)s * CH_SLOT, &m.in[cc.in_map[j]], cc.in_col[j], tile * 128, &c.in_full[s]);
    }
  }
}

// warp 1, one thread: the GEMMs of two tiles in flight, interleaved stage by stage
__device__ __forceinline__ void chain_mma(const Carve& c, const ChainCommon& cc, uint32_t tmem_base) {
  mbar_wait(c.b_ready, 0);
  int n_local = 0;
  for (int tile = blockIdx.x; tile < cc.num_tiles; tile += gridDim.x) ++n_local;
  uint32_t uses[2] = {0, 0};
  const uint32_t sW = smem_u32(c.sW);
  for (int t0 = 0; t0 < n_local; t0 += 2) {
    for (int i = 0; i < cc.n_gemm; ++i) {
      const int N = cc.g_N[i];
      const uint32_t idesc = umma_idesc_tf32(N), chunk = (uint32_t)N * 128u, image = 2 * chunk;
      for (int g = 0; g < 2; ++g) {
        if (t0 + g >= n_local) break;
        mbar_wait(&c.a_ready[g], uses[g] & 1u);
        ++uses[g];
        tc_fence_after();
        const uint32_t a_hi = tmem_base + (uint32_t)(g * CH_TM_GROUP), a_lo = a_hi + CH_TM_ALO, d = a_hi + CH_TM_D + (uint32_t)cc.g_dcol[i];
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
          const uint32_t bh = sW + cc.g_boff[i] + (uint32_t)(kk >> 2) * chunk + (uint32_t)(kk & 3) * 32u, bl = bh + image;
          umma_tf32_ts(d, a_lo + kk * 8, umma_desc_k_sw128(bh), idesc, kk ? 1u : 0u);
          umma_tf32_ts(d, a_hi + kk * 8, umma_desc_k_sw128(bl), idesc, 1u);
          umma_tf32_ts(d, a_hi + kk * 8, umma_desc_k_sw128(bh), idesc, 1u);
        }
        umma_commit(&c.d_ready[g]);
      }
    }
  }
}

__device__ __forceinline__ RowCtx row_ctx(const Carve& c, const ChainCommon& cc, uint32_t tmem_base) {
  RowCtx r;
  const int warp = threadIdx.x >> 5;
  r.lane = threadIdx.x & 31;
  r.group = (warp - 4) >> 2;
  r.rt = (warp & 3) * 32 + r.lane;
  r.tm = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(r.group * CH_TM_GROUP);
  r.ring = c.ring;
  r.in_full = c.in_full;
  r.in_empty = c.in_empty;
  r.ring_slots = cc.ring_slots;
  r.n_in = cc.n_in;
  r.in_done_mine = &c.in_done[r.group];
  r.in_done_other = &c.in_done[r.group ^ 1];
  r.in_it = 0;
  r.obuf = c.obuf + (size_t)r.group * 2 * CH_SLOT;
  r.a_ready = &c.a_ready[r.group];
  r.d_ready = &c.d_ready[r.group];
  r.a_uses = r.d_uses = 0;
  return r;
}

// The update needs fp32-faithful, not bit-identical, activations (the rollout, whose sampled actions must not move, never runs these
// kernels): ex2.approx / rcp.approx forms, absolute error ~1e-7, a third of the instructions of expf + IEEE division. A row thread has
// one warp per scheduler pair to hide latency behind, so the instruction count of the activation is what bounds these kernels.
__device__ __forceinline__ float swishf(float x) { return x * __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float gelu_fast(float x) {
  const float u = 0.7978845608028654f * (x + 0.044715f * x * x * x);
  const float t = 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * u));
  return 0.5f * x * (1.0f + t);
}

// x <- RMSNorm(x) * scale (scale: 64 floats in shared memory)
__device__ __forceinline__ void rms64(float (&x)[64], const float* scale) {
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < 64; ++j) ss = fmaf(x[j], x[j], ss);
  const float rstd = rsqrtf(ss * (1.0f / 64) + kEps);
#pragma unroll
  for (int j = 0; j < 64; j += 4) {
    const float4 s4 = *reinterpret_cast<const float4*>(scale + j);
    x[j] *= rstd * s4.x; x[j + 1] *= rstd * s4.y; x[j + 2] *= rstd * s4.z; x[j + 3] *= rstd * s4.w;
  }
}
__device__ __forceinline__ void add_pe64(float (&x)[64], const float* __restrict__ pe_row) {
#pragma unroll
  for (int j = 0; j < 64; j += 4) {
    const float4 e = __ldg(reinterpret_cast<const float4*>(pe_row + j));
    x[j] += e.x; x[j + 1] += e.y; x[j + 2] += e.z; x[j + 3] += e.w;
  }
}

// ------------------------------------------------------------------------------------------------------------------ gate chain
struct GateParams {
  ChainCommon cc;
  const float *gn_s, *gn_b, *ln_s, *pe;
  const int32_t* step;
  int max_step;
  int store_y, store_ype;
};
enum { GO_GATED = 0, GO_O, GO_Y, GO_YPE, GO_GL /* MODE 2: the projection's output */, GO_H };

// MODE 0: ends after the norm; 1: + SwiGLU up-projection; 2: + a [64 -> 192] projection of ype (the decoder's cross-retention k | v | g)
template <int MODE>
__global__ void __launch_bounds__(CH_THREADS, 1)
chain_gate_kernel(const __grid_constant__ ChainMaps maps, const GateParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const Carve c = carve_smem(smem_raw, p.cc);
  for (int i = threadIdx.x; i < 64; i += CH_THREADS) {
    c.sPar[i] = p.gn_s[i];
    c.sPar[64 + i] = p.gn_b[i];
    c.sPar[128 + i] = p.ln_s[i];
  }
  const uint32_t tmem_base = chain_setup(c, p.cc);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) {
    if (lane == 0) chain_producer(c, p.cc, maps);
  } else if (warp == 1) {
    if (lane == 0) chain_mma(c, p.cc, tmem_base);
  } else if (warp >= 4) {
    RowCtx r = row_ctx(c, p.cc, tmem_base);
    const float *gs = c.sPar, *gb = c.sPar + 64, *ls = c.sPar + 128;
    int ti = 0;
    for (int tile = blockIdx.x; tile < p.cc.num_tiles; tile += gridDim.x, ++ti) {
      if ((ti & 1) != r.group) continue;
      in_begin(r, ti);
      const int row0 = tile * 128;
      const int64_t row = (int64_t)row0 + r.rt;
      float x[64];
      // ---- gated = swish(g) * GroupNorm(ret)       (one group: LayerNorm statistics with flax's "fast variance")
      in_take64(r, x);
      {
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int j = 0; j < 64; ++j) { s1 += x[j]; s2 = fmaf(x[j], x[j], s2); }
        const float mean = s1 * (1.0f / 64);
        const float rstd = rsqrtf(fmaxf(0.0f, s2 * (1.0f / 64) - mean * mean) + kEps);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float g[32];
          in_take(r, g);
#pragma unroll
          for (int j = 0; j < 32; ++j) x[32 * h + j] = swishf(g[j]) * ((x[32 * h + j] - mean) * rstd * gs[32 * h + j] + gb[32 * h + j]);
        }
      }
      put_A(r, x);
      stash_input64<64>(r);  // the residual rows wait in the idle half of the accumulator columns: the input ring keeps flowing
      in_end(r);
      out_store64(r, &maps.out[GO_GATED], 0, row0, x);
      // ---- o = gated W_o ; y = RMSNorm(o + res) * scale (+ PE)
      wait_D(r);
      ld_D64<0>(r, x);
      out_store64(r, &maps.out[GO_O], 0, row0, x);
      add_D64<64>(r, x);
      rms64(x, ls);
      if (p.store_y) out_store64(r, &maps.out[GO_Y], 0, row0, x);
      if (p.store_ype) {
        const int st = row < p.cc.R ? min(max(p.step[row], 0), p.max_step) : 0;
        add_pe64(x, p.pe + (size_t)st * 64);
        out_store64(r, &maps.out[GO_YPE], 0, row0, x);
      }
      if (MODE == 2) {
        put_A(r, x);
        wait_D(r);
        ld_D64<0>(r, x);
        out_store64(r, &maps.out[GO_GL], 0, row0, x);
        ld_D64<64>(r, x);
        rearm_A(r);  // the last 64 columns run while the first 128 leave
        out_store64(r, &maps.out[GO_GL], 64, row0, x);
        wait_D(r);
        ld_D64<0>(r, x);
        out_store64(r, &maps.out[GO_GL], 128, row0, x);
      }
      if (MODE == 1) {
        // ---- gl = y [W_gate | W_linear] ; hmid = swish(gl_a) * gl_b
        put_A(r, x);
        wait_D(r);
        ld_D64<0>(r, x);
        out_store64(r, &maps.out[GO_GL], 0, row0, x);
        ld_D64<64>(r, x);
        out_store64(r, &maps.out[GO_GL], 64, row0, x);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float a[32], b[32];
          ld_D32(r, 32 * h, a);
          ld_D32(r, 64 + 32 * h, b);
#pragma unroll
          for (int j = 0; j < 32; ++j) x[32 * h + j] = swishf(a[j]) * b[j];
        }
        out_store64(r, &maps.out[GO_H], 0, row0, x);
      }
    }
    if (r.lane == 0) bulk_wait_all();
  }
  chain_teardown(tmem_base);
}

// ------------------------------------------------------------------------------------------------------------------ tail chain
struct TailParams {
  ChainCommon cc;
  const float *ln_s, *pe, *h_bias, *h2_s, *W3, *b3;
  const int32_t* step;
  int max_step, nout;
  int with_q;   // extra GEMM q = xpe W_q between the norm and the head (cross-retention query of the decoder)
  int store_xpe;
  float* out;   // [R, nout]
};
enum { TO_F = 0, TO_X, TO_XPE, TO_Q, TO_ZH };

__global__ void __launch_bounds__(CH_THREADS, 1)
chain_tail_kernel(const __grid_constant__ ChainMaps maps, const TailParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const Carve c = carve_smem(smem_raw, p.cc);
  const int NP = (p.nout + 3) & ~3;  // W3 rows padded to float4s
  float *ls = c.sPar, *hb = c.sPar + 64, *h2 = c.sPar + 128, *w3 = c.sPar + 192, *b3 = c.sPar + 192 + 64 * 32;
  for (int i = threadIdx.x; i < 64; i += CH_THREADS) {
    ls[i] = p.ln_s[i];
    hb[i] = p.h_bias[i];
    h2[i] = p.h2_s[i];
  }
  for (int i = threadIdx.x; i < 64 * NP; i += CH_THREADS) {
    const int cidx = i / NP, j = i % NP;
    w3[i] = j < p.nout ? p.W3[cidx * p.nout + j] : 0.f;
  }
  for (int i = threadIdx.x; i < 32; i += CH_THREADS) b3[i] = i < p.nout ? p.b3[i] : 0.f;
  const uint32_t tmem_base = chain_setup(c, p.cc);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) {
    if (lane == 0) chain_producer(c, p.cc, maps);
  } else if (warp == 1) {
    if (lane == 0) chain_mma(c, p.cc, tmem_base);
  } else if (warp >= 4) {
    RowCtx r = row_ctx(c, p.cc, tmem_base);
    int ti = 0;
    for (int tile = blockIdx.x; tile < p.cc.num_tiles; tile += gridDim.x, ++ti) {
      if ((ti & 1) != r.group) continue;
      in_begin(r, ti);
      const int row0 = tile * 128;
      const int64_t row = (int64_t)row0 + r.rt;
      float x[64];
      // ---- f = hmid W_out
      in_take64(r, x);
      put_A(r, x);
      stash_input64<64>(r);
      in_end(r);
      wait_D(r);
      ld_D64<0>(r, x);
      out_store64(r, &maps.out[TO_F], 0, row0, x);
      // ---- x = RMSNorm(f + res) * scale
      add_D64<64>(r, x);
      rms64(x, ls);
      put_A(r, x);  // zh = x W_h0 -> accumulator columns [0, 64)
      out_store64(r, &maps.out[TO_X], 0, row0, x);
      if (p.store_xpe) {
        const int st = row < p.cc.R ? min(max(p.step[row], 0), p.max_step) : 0;
        add_pe64(x, p.pe + (size_t)st * 64);
        out_store64(r, &maps.out[TO_XPE], 0, row0, x);
      }
      wait_D(r);
      if (p.with_q) put_A(r, x);  // q = xpe W_q -> accumulator columns [64, 128)
      // ---- zh + b
      ld_D64<0>(r, x);
#pragma unroll
      for (int j = 0; j < 64; ++j) x[j] += hb[j];
      out_store64(r, &maps.out[TO_ZH], 0, row0, x);
      // ---- head: out = RMSNorm(gelu(zh)) * scale @ W3 + b3
#pragma unroll
      for (int j = 0; j < 64; ++j) x[j] = gelu_fast(x[j]);
      rms64(x, h2);
      if (row < p.cc.R) {
        for (int jb = 0; jb < NP; jb += 4) {
          float4 acc = make_float4(b3[jb], b3[jb + 1], b3[jb + 2], b3[jb + 3]);
#pragma unroll
          for (int k = 0; k < 64; ++k) {
            const float4 w = *reinterpret_cast<const float4*>(w3 + k * NP + jb);
            acc.x = fmaf(x[k], w.x, acc.x); acc.y = fmaf(x[k], w.y, acc.y);
            acc.z = fmaf(x[k], w.z, acc.z); acc.w = fmaf(x[k], w.w, acc.w);
          }
          float* o = p.out + row * p.nout + jb;
          if (jb + 0 < p.nout) o[0] = acc.x;
          if (jb + 1 < p.nout) o[1] = acc.y;
          if (jb + 2 < p.nout) o[2] = acc.z;
          if (jb + 3 < p.nout) o[3] = acc.w;
        }
      }
      if (p.with_q) {
        wait_D(r);
        ld_D64<64>(r, x);
        out_store64(r, &maps.out[TO_Q], 0, row0, x);
      }
    }
    if (r.lane == 0) bulk_wait_all();
  }
  chain_teardown(tmem_base);
}

// ------------------------------------------------------------------------------------------------------------------ front chain
// The rows entering the first retention of each network:
//   OBS   on = RMSNorm_d(obs) * obs_scale -> z0 = on W_obs -> x = RMSNorm(gelu(z0)) * ln -> xpe = x + PE -> qkvg = xpe [w_q|w_k|w_v|w_g]
//   !OBS  token = shifted action -> x = RMSNorm(gelu(W_a[token])) * ln (a per-CTA table) -> xpe = x + PE -> qkvg = xpe [w_q|w_k|w_v|w_g]
struct FrontParams {
  ChainCommon cc;
  int d, A, a, max_step;
  const float *obs, *obs_scale, *Wobs, *Wa, *ln_s, *pe;
  const int32_t *action, *step;
};
enum { FO_Z0 = 0, FO_X, FO_XPE, FO_Q };

template <bool OBS>
__global__ void __launch_bounds__(CH_THREADS, 1)
chain_front_kernel(const __grid_constant__ ChainMaps maps, const FrontParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const Carve c = carve_smem(smem_raw, p.cc);
  float *ls = c.sPar, *osc = c.sPar + 64, *tab = c.sPar + 80;  // tab: W_obs [d][64] or the token table [(a+1)][64]
  for (int i = threadIdx.x; i < 64; i += CH_THREADS) ls[i] = p.ln_s[i];
  if (OBS) {
    for (int i = threadIdx.x; i < 16; i += CH_THREADS) osc[i] = i < p.d ? p.obs_scale[i] : 0.f;
    for (int i = threadIdx.x; i < p.d * 64; i += CH_THREADS) tab[i] = p.Wobs[i];
  }
  __syncthreads();
  if (!OBS && threadIdx.x <= p.a) {  // x of every token value, once per CTA
    float v[64];
#pragma unroll
    for (int j = 0; j < 64; ++j) v[j] = gelu_fast(p.Wa[threadIdx.x * 64 + j]);
    rms64(v, ls);
#pragma unroll
    for (int j = 0; j < 64; ++j) tab[threadIdx.x * 64 + j] = v[j];
  }
  const uint32_t tmem_base = chain_setup(c, p.cc);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) {
    if (lane == 0) chain_producer(c, p.cc, maps);
  } else if (warp == 1) {
    if (lane == 0) chain_mma(c, p.cc, tmem_base);
  } else if (warp >= 4) {
    RowCtx r = row_ctx(c, p.cc, tmem_base);
    int ti = 0;
    for (int tile = blockIdx.x; tile < p.cc.num_tiles; tile += gridDim.x, ++ti) {
      if ((ti & 1) != r.group) continue;
      const int row0 = tile * 128;
      const int64_t row = (int64_t)row0 + r.rt;
      const bool live = row < p.cc.R;
      float x[64];
      if (OBS) {
        float ob[16];
        float ss = 0.f;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          ob[k] = (live && k < p.d) ? __ldg(p.obs + row * p.d + k) : 0.f;
          ss = fmaf(ob[k], ob[k], ss);
        }
        const float rstd0 = rsqrtf(ss / (float)p.d + kEps);
#pragma unroll
        for (int j = 0; j < 64; ++j) x[j] = 0.f;
        for (int k = 0; k < p.d; ++k) {
          float okv = 0.f;
#pragma unroll
          for (int kk = 0; kk < 16; ++kk) okv = kk == k ? ob[kk] : okv;
          okv *= rstd0 * osc[k];
          const float* wr = tab + k * 64;
#pragma unroll
          for (int j = 0; j < 64; j += 4) {
            const float4 w = *reinterpret_cast<const float4*>(wr + j);
            x[j] = fmaf(okv, w.x, x[j]); x[j + 1] = fmaf(okv, w.y, x[j + 1]);
            x[j + 2] = fmaf(okv, w.z, x[j + 2]); x[j + 3] = fmaf(okv, w.w, x[j + 3]);
          }
        }
        out_store64(r, &maps.out[FO_Z0], 0, row0, x);
#pragma unroll
        for (int j = 0; j < 64; ++j) x[j] = gelu_fast(x[j]);
        rms64(x, ls);
      } else {
        int tok = 0;
        if (live && (row % p.A) != 0) tok = 1 + p.action[row - 1];
        const float* tr = tab + tok * 64;
#pragma unroll
        for (int j = 0; j < 64; j += 4) {
          const float4 t = *reinterpret_cast<const float4*>(tr + j);
          x[j] = t.x; x[j + 1] = t.y; x[j + 2] = t.z; x[j + 3] = t.w;
        }
      }
      out_store64(r, &maps.out[FO_X], 0, row0, x);
      const int st = live ? min(max(p.step[row], 0), p.max_step) : 0;
      add_pe64(x, p.pe + (size_t)st * 64);
      put_A(r, x);
      out_store64(r, &maps.out[FO_XPE], 0, row0, x);
      // ---- the four 64-wide projections, 128 columns per pass
      wait_D(r);
      ld_D64<0>(r, x);
      out_store64(r, &maps.out[FO_Q], 0, row0, x);
      ld_D64<64>(r, x);
      rearm_A(r);
      out_store64(r, &maps.out[FO_Q], 64, row0, x);
      wait_D(r);
      ld_D64<0>(r, x);
      out_store64(r, &maps.out[FO_Q], 128, row0, x);
      ld_D64<64>(r, x);
      out_store64(r, &maps.out[FO_Q], 192, row0, x);
    }
    if (r.lane == 0) bulk_wait_all();
  }
  chain_teardown(tmem_base);
}

// ---------------------------------------------------------------- host side
bool g_chain_enabled = true;  // magpo_set_chain_kernels: tests compare the chain kernels with the layer-by-layer path

bool act_map(CUtensorMap* tm, const float* ptr, int64_t R, int cols, int ld) { return tc_make_map(tm, ptr, R, cols, ld, 128); }
// outputs leave per warp: boxes of 32 rows
bool out_map(CUtensorMap* tm, const float* ptr, int64_t R, int cols, int ld) { return tc_make_map(tm, ptr, R, cols, ld, 32); }

// B operand images of a [N, 64] transposed weight registered with tc_prepare_region
bool weight_maps(ChainMaps* m, int i, const float* wt, int N, int ld, int box_rows = 0) {
  const float *hi, *lo;
  if (!tc_lookup(wt, &hi, &lo)) return false;
  if (!box_rows) box_rows = N;
  return tc_make_map(&m->w[2 * i], hi, N, 64, ld, box_rows) && tc_make_map(&m->w[2 * i + 1], lo, N, 64, ld, box_rows);
}

void add_gemm(ChainCommon* cc, int N, int dcol = 0, int wrow = 0) {
  const int i = cc->n_gemm++;
  cc->g_N[i] = N;
  cc->g_dcol[i] = dcol;
  cc->g_wrow[i] = wrow;
  cc->g_boff[i] = cc->w_bytes;
  cc->w_bytes += 2u * 2u * (uint32_t)N * 128u;  // hi + lo, two 32-wide k chunks each
}
void add_input(ChainCommon* cc, int map) {
  for (int h = 0; h < 2; ++h) {
    cc->in_map[cc->n_in] = map;
    cc->in_col[cc->n_in++] = 32 * h;
  }
}
bool finish_plan(ChainCommon* cc, int64_t R, int par_floats, uint32_t* smem) {
  cc->R = R;
  cc->num_tiles = (int)ceil_div(R, 128);
  cc->par_floats = par_floats;
  int slots = cc->n_in ? CH_MAX_RING : 0;
  while (slots >= 2 && chain_smem_bytes(cc->w_bytes, slots, par_floats) > CH_SMEM_LIMIT) --slots;
  if (cc->n_in ? slots < 2 : chain_smem_bytes(cc->w_bytes, 0, par_floats) > CH_SMEM_LIMIT) return false;
  cc->ring_slots = slots;
  *smem = chain_smem_bytes(cc->w_bytes, slots, par_floats);
  return true;
}

}  // namespace

void chain_set_enabled(bool on) { g_chain_enabled = on; }
bool chain_supported(int64_t R) { return g_chain_enabled && R >= 256 && R < (int64_t)1 << 31; }

int chain_gate_fwd(cudaStream_t s, int64_t R, const float* g, int ldg, const float* ret, const float* res, const float* gn_s,
                   const float* gn_b, const float* ln_s, const float* pe, const int32_t* step, int max_step, const float* W1T,
                   const float* W2T, const float* WpT, float* gated, float* o, float* y, float* ype, float* gl, float* hmid, float* proj,
                   int ldproj) {
  ChainMaps m;
  GateParams p{};
  const int mode = W2T ? 1 : (WpT ? 2 : 0);
  add_input(&p.cc, 0);  // ret
  add_input(&p.cc, 1);  // g
  add_input(&p.cc, 2);  // res
  add_gemm(&p.cc, 64);
  if (mode == 1) add_gemm(&p.cc, 128);
  if (mode == 2) {
    add_gemm(&p.cc, 128, 0, 0);
    add_gemm(&p.cc, 64, 0, 128);
  }
  uint32_t smem;
  if (!finish_plan(&p.cc, R, 192, &smem)) return MAGPO_ERR_UNSUPPORTED;
  bool ok = act_map(&m.in[0], ret, R, 64, 64) && act_map(&m.in[1], g, R, 64, ldg) && act_map(&m.in[2], res, R, 64, 64) &&
            out_map(&m.out[GO_GATED], gated, R, 64, 64) && out_map(&m.out[GO_O], o, R, 64, 64) && weight_maps(&m, 0, W1T, 64, 64);
  if (y) ok = ok && out_map(&m.out[GO_Y], y, R, 64, 64);
  if (ype) ok = ok && out_map(&m.out[GO_YPE], ype, R, 64, 64);
  if (mode == 1) ok = ok && out_map(&m.out[GO_GL], gl, R, 128, 128) && out_map(&m.out[GO_H], hmid, R, 64, 64) && weight_maps(&m, 1, W2T, 128, 64);
  if (mode == 2)
    ok = ok && ype && out_map(&m.out[GO_GL], proj, R, 192, ldproj) && weight_maps(&m, 1, WpT, 192, 64, 128) && weight_maps(&m, 2, WpT, 192, 64, 64);
  if (!ok) return MAGPO_ERR_ARG;
  p.gn_s = gn_s; p.gn_b = gn_b; p.ln_s = ln_s; p.pe = pe; p.step = step; p.max_step = max_step;
  p.store_y = y != nullptr;
  p.store_ype = ype != nullptr;
  const unsigned grid = (unsigned)std::min(p.cc.num_tiles, kNumSMs);
  const double units = 3 + 2 + (y ? 1 : 0) + (ype ? 1 : 0) + (mode ? 3 : 0);
  ProfScope ps(PROF_CHAIN, s, 2.0 * R * 64 * (64 + (mode == 1 ? 128 : mode == 2 ? 192 : 0)), units * 256.0 * R);
#define LAUNCH_GATE(MODE, ONCE)                                                                                                    \
  {                                                                                                                                \
    if (once_per_device(ONCE))                                                                                                     \
      MAGPO_CUDA_OK(cudaFuncSetAttribute(chain_gate_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_SMEM_LIMIT)); \
    chain_gate_kernel<MODE><<<grid, CH_THREADS, smem, s>>>(m, p);                                                                  \
  }
  if (mode == 1) LAUNCH_GATE(1, ONCE_CHAIN_GATE_FFN) else if (mode == 2) LAUNCH_GATE(2, ONCE_CHAIN_GATE_PROJ) else LAUNCH_GATE(0, ONCE_CHAIN_GATE)
#undef LAUNCH_GATE
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

int chain_front_fwd(cudaStream_t s, int64_t R, int d, const float* obs, const float* obs_scale, const float* Wobs, int A, int a,
                    const int32_t* action, const float* Wa, const float* ln_s, const float* pe, const int32_t* step, int max_step,
                    const float* WqT, float* z0, float* x, float* xpe, float* qkvg) {
  ChainMaps m;
  FrontParams p{};
  const bool obs_mode = obs != nullptr;
  if (obs_mode ? (d < 1 || d > 16) : (a < 1 || a > 32)) return MAGPO_ERR_UNSUPPORTED;
  add_gemm(&p.cc, 128, 0, 0);
  add_gemm(&p.cc, 128, 0, 128);
  uint32_t smem;
  if (!finish_plan(&p.cc, R, 64 + 16 + 33 * 64, &smem)) return MAGPO_ERR_UNSUPPORTED;
  bool ok = out_map(&m.out[FO_X], x, R, 64, 64) && out_map(&m.out[FO_XPE], xpe, R, 64, 64) && out_map(&m.out[FO_Q], qkvg, R, 256, 256) &&
            weight_maps(&m, 0, WqT, 256, 64, 128) && weight_maps(&m, 1, WqT, 256, 64, 128);
  if (obs_mode) ok = ok && out_map(&m.out[FO_Z0], z0, R, 64, 64);
  if (!ok) return MAGPO_ERR_ARG;
  p.d = d; p.obs = obs; p.obs_scale = obs_scale; p.Wobs = Wobs; p.A = A; p.a = a; p.action = action; p.Wa = Wa; p.ln_s = ln_s;
  p.pe = pe; p.step = step; p.max_step = max_step;
  const unsigned grid = (unsigned)std::min(p.cc.num_tiles, kNumSMs);
  ProfScope ps(PROF_CHAIN, s, 2.0 * R * 64 * 256, ((obs_mode ? 7 : 6) * 256.0 + (obs_mode ? 4.0 * d : 4.0)) * R);
  if (obs_mode) {
    if (once_per_device(ONCE_CHAIN_FRONT_OBS))
      MAGPO_CUDA_OK(cudaFuncSetAttribute(chain_front_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_SMEM_LIMIT));
    chain_front_kernel<true><<<grid, CH_THREADS, smem, s>>>(m, p);
  } else {
    if (once_per_device(ONCE_CHAIN_FRONT_EMB))
      MAGPO_CUDA_OK(cudaFuncSetAttribute(chain_front_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_SMEM_LIMIT));
    chain_front_kernel<false><<<grid, CH_THREADS, smem, s>>>(m, p);
  }
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

int chain_tail_fwd(cudaStream_t s, int64_t R, const float* hmid, const float* res, const float* ln_s, const float* pe,
                   const int32_t* step, int max_step, const float* W1T, const float* WqT, int ldwq, const float* WhT, const float* h_bias,
                   const float* h2_s, const float* W3, const float* b3, int nout, float* f, float* x, float* xpe, float* q, int ldq,
                   float* zh, float* out) {
  ChainMaps m;
  TailParams p{};
  if (nout < 1 || nout > 32) return MAGPO_ERR_UNSUPPORTED;
  add_input(&p.cc, 0);  // hmid
  add_input(&p.cc, 1);  // res
  add_gemm(&p.cc, 64);          // ffn_out
  add_gemm(&p.cc, 64);          // h0
  if (q) add_gemm(&p.cc, 64, 64);  // q
  uint32_t smem;
  if (!finish_plan(&p.cc, R, 192 + 64 * 32 + 32, &smem)) return MAGPO_ERR_UNSUPPORTED;
  bool ok = act_map(&m.in[0], hmid, R, 64, 64) && act_map(&m.in[1], res, R, 64, 64) && out_map(&m.out[TO_F], f, R, 64, 64) &&
            out_map(&m.out[TO_X], x, R, 64, 64) && out_map(&m.out[TO_ZH], zh, R, 64, 64) && weight_maps(&m, 0, W1T, 64, 64);
  if (xpe) ok = ok && out_map(&m.out[TO_XPE], xpe, R, 64, 64);
  ok = ok && weight_maps(&m, 1, WhT, 64, 64);
  if (q) ok = ok && xpe && out_map(&m.out[TO_Q], q, R, 64, ldq) && weight_maps(&m, 2, WqT, 64, ldwq);
  if (!ok) return MAGPO_ERR_ARG;
  p.ln_s = ln_s; p.pe = pe; p.step = step; p.max_step = max_step; p.h_bias = h_bias; p.h2_s = h2_s; p.W3 = W3; p.b3 = b3;
  p.nout = nout; p.with_q = q != nullptr; p.store_xpe = xpe != nullptr; p.out = out;
  const unsigned grid = (unsigned)std::min(p.cc.num_tiles, kNumSMs);
  const double units = 2 + 3 + (xpe ? 1 : 0) + (q ? 1 : 0);
  ProfScope ps(PROF_CHAIN, s, 2.0 * R * 64 * 64 * (q ? 3 : 2), (units * 256.0 + 4.0 * nout) * R);
  if (once_per_device(ONCE_CHAIN_TAIL))
    MAGPO_CUDA_OK(cudaFuncSetAttribute(chain_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_SMEM_LIMIT));
  chain_tail_kernel<<<grid, CH_THREADS, smem, s>>>(m, p);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

}  // namespace magpo

extern "C" int magpo_set_chain_kernels(int on) {
  magpo::chain_set_enabled(on != 0);
  return MAGPO_OK;
}
