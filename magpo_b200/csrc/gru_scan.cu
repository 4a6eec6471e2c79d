// Persistent tensor-core GRU scans for the learner's update (ScannedRNN over T steps, networks/base.py:124-142, flax
// GRUCell of SURVEY.md Appendix A8; BPTT per Appendix G).
//
// The recurrence is independent per (env, agent) row, so one CTA owns a tile of 128 rows for the whole sequence:
//   * the hidden state never leaves the SM: it lives in registers (exact fp32) and, split into TF32 hi/lo images, in TENSOR MEMORY
//     as the A operand of tcgen05.mma (A-from-TMEM form; round 2: it used to be a 128 KiB shared-memory operand — the tensor core
//     re-read it on every K = 8 step, and publishing it cost an STS pass + fence.proxy.async per timestep). The gate threads write
//     their 4 x 2 patches with tcgen05.st in the same 16x256b shape they read the accumulators with;
//   * W_h (hi/lo images, 384 KiB) does not fit in shared memory, so it is streamed from L2 every timestep through a TMA ring
//     (8 stages of the 16 pieces of a step now that the A operand is gone from shared memory);
//   * accumulators live in tensor memory; the gate math runs straight out of tcgen05.ld registers, fused with the loads of
//     the batched input-side pre-activations and the stores of everything the backward needs. The gate warps read TMEM with
//     the 16x256b fragment shape; their inputs and (forward) outputs travel through TMA-loaded / bulk-stored staging boxes in shared
//     memory instead of 8-rows-x-32-B global accesses (the lg_throttle of round 1); a service warp issues the loads one block ahead.
// Per timestep and tile the forward issues 16 pieces x 12 MMAs (M=128, N=96: the r|z|n columns of one block of 32 hidden
// units, so that the gates of block jb run while the tensor core works on block jb+1), the backward 12 pieces x 12 MMAs
// (N=128; the contraction index is ordered (block, gate) so that the MMAs of a block start as soon as its dgh is written).
// 3xTF32 throughout (fp32-faithful). warps 0-15: gates, warp 16: TMA producer of W_h, warp 17: MMA issuer, warp 18: TMA loader of the gate inputs
// (warp 19 only donates its registers to the gate warps through setmaxnreg).
#include <cuda.h>
#include <stdlib.h>

#include "actor.cuh"
#include "tc_ptx.cuh"

namespace magpo {
using namespace tcp;
namespace {

constexpr int GS_GATE_WARPS = 16;
constexpr int GS_GATE_THREADS = GS_GATE_WARPS * 32;
constexpr int GS_THREADS = GS_GATE_THREADS + 128;  // + one warpgroup of service warps
constexpr int GS_CHUNK = 128 * 128;            // bytes of one [128 rows x 32 floats] operand chunk
constexpr int GS_STAGES = 4;       // backward ring
constexpr int GS_FWD_STAGES = 3;   // forward ring (24 KiB pieces)
constexpr int GS_IN_BOXES = 3;     // staging of one block's input pre-activations (r, z, n columns): 3 x [128 rows x 32 floats]
constexpr int GS_OUT_BOXES = 6;    // staging of one block's saved activations: 6 x [128 rows x 32 floats]
// forward TMEM columns: A hi [0,128), A lo [128,256), two accumulators of 96 at 256 / 352
constexpr uint32_t GS_F_ALO = 128, GS_F_ACC = 256;
// backward TMEM columns: A slots (gate r, z, n of a block) hi [0,96), lo [96,192), two carry accumulators of 128 at 192 / 320
constexpr uint32_t GS_B_ALO = 96, GS_B_ACC = 192;
constexpr int GS_FWD_STAGE = 2 * 96 * 128;     // [96 x 32] hi + lo
constexpr int GS_BWD_STAGE = 2 * GS_CHUNK;     // [128 x 32] hi + lo
constexpr uint32_t GS_SMEM = 227 * 1024;

// tcgen05.ld 16x256b.x1: 16 lanes x 8 columns; lane l of the warp receives r[2h + e] = (row l/4 + 8h, column 2(l%4) + e)
// (probed with tools/probes/tmem_layout_probe.cu).
__device__ __forceinline__ void tmem_ld_frag_nowait(uint32_t taddr, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.16x256b.x1.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// the mirror image: thread values r[2h + e] -> (row l/4 + 8h, column 2(l%4) + e) of a 16-lane x 8-column patch
__device__ __forceinline__ void tmem_st_frag(uint32_t taddr, const uint32_t* v) {
  asm volatile("tcgen05.st.sync.aligned.16x256b.x1.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// an 8-value patch as the TF32 hi / lo images of an A operand in tensor memory (hi = truncation, lo = exact remainder)
__device__ __forceinline__ void tmem_st_patch_split(uint32_t taddr_hi, uint32_t taddr_lo, const float* v) {
  uint32_t hi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    hi[i] = __float_as_uint(v[i]) & 0xFFFFE000u;
    lo[i] = __float_as_uint(v[i] - __uint_as_float(hi[i]));
  }
  tmem_st_frag(taddr_hi, hi);
  tmem_st_frag(taddr_hi + (16u << 16), hi + 4);
  tmem_st_frag(taddr_lo, lo);
  tmem_st_frag(taddr_lo + (16u << 16), lo + 4);
}
// D[tmem] (+)= A[tmem] . B[smem], kind::tf32
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
// both 16-lane halves of the warp's sub-partition: v[4 half + 2h + e]
__device__ __forceinline__ void tmem_ld_patch_nowait(uint32_t taddr, uint32_t* v) {
  tmem_ld_frag_nowait(taddr, v);
  tmem_ld_frag_nowait(taddr + (16u << 16), v + 4);
}

// A gate warp owns 32 rows x 8 of every 32 hidden units; a thread the 4 x 2 patch rows {rr = 2 half + h} x columns {2m + e}.
// Value index inside an 8-vector: 4 (rr >> 1) + 2 (rr & 1) + e.
struct GateGeom {
  int m;             // lane % 4
  int row[4];        // row inside the 128-row tile
  int64_t grow[4];   // global row
  bool valid[4];
};
__device__ __forceinline__ int vidx(int rr, int e) { return (rr >> 1) * 4 + 2 * (rr & 1) + e; }

__device__ __forceinline__ GateGeom make_geom(int sp, int lane, int64_t tile_row0, int64_t Rs, int rpt) {
  GateGeom gg;
  gg.m = lane & 3;
#pragma unroll
  for (int rr = 0; rr < 4; ++rr) {
    gg.row[rr] = sp * 32 + (rr >> 1) * 16 + (rr & 1) * 8 + (lane >> 2);
    gg.grow[rr] = tile_row0 + gg.row[rr];
    gg.valid[rr] = gg.row[rr] < rpt && gg.grow[rr] < Rs;
  }
  return gg;
}
// 8 values of the patch from a row-major [rows, width] slab (col = first column of the warp's 8-column slab)
__device__ __forceinline__ void load_patch(float* v, const float* slab, int width, int col, const GateGeom& gg) {
#pragma unroll
  for (int rr = 0; rr < 4; ++rr) {
    float2 x = make_float2(0.f, 0.f);
    if (gg.valid[rr]) x = __ldg(reinterpret_cast<const float2*>(slab + gg.grow[rr] * width + col + 2 * gg.m));
    v[vidx(rr, 0)] = x.x;
    v[vidx(rr, 1)] = x.y;
  }
}
__device__ __forceinline__ void store_patch(const float* v, float* slab, int width, int col, const GateGeom& gg) {
#pragma unroll
  for (int rr = 0; rr < 4; ++rr)
    if (gg.valid[rr])
      *reinterpret_cast<float2*>(slab + gg.grow[rr] * width + col + 2 * gg.m) = make_float2(v[vidx(rr, 0)], v[vidx(rr, 1)]);
}
// the patch into a 128B-swizzled [rows x 32 floats] staging box (c0 = first column of the warp's slab inside the box): the layout a TMA
// store of the box expects. The gate warps' patches touch 8 rows x 32 B per global store instruction; staged, a block's six output
// tensors leave as six bulk stores issued by one thread.
__device__ __forceinline__ void stage_patch(uint8_t* box, int c0, const float* v, const GateGeom& gg) {
#pragma unroll
  for (int rr = 0; rr < 4; ++rr)
    if (gg.valid[rr]) {
      const int row = gg.row[rr];
      const int unit = ((c0 >> 2) + (gg.m >> 1)) ^ (row & 7);
      *reinterpret_cast<float2*>(box + row * 128 + unit * 16 + (gg.m & 1) * 8) = make_float2(v[vidx(rr, 0)], v[vidx(rr, 1)]);
    }
}
// ... and back: the patch out of a staging box a TMA load filled
__device__ __forceinline__ void unstage_patch(float* v, const uint8_t* box, int c0, const GateGeom& gg) {
#pragma unroll
  for (int rr = 0; rr < 4; ++rr) {
    float2 x = make_float2(0.f, 0.f);
    if (gg.valid[rr]) {
      const int row = gg.row[rr];
      const int unit = ((c0 >> 2) + (gg.m >> 1)) ^ (row & 7);
      x = *reinterpret_cast<const float2*>(box + row * 128 + unit * 16 + (gg.m & 1) * 8);
    }
    v[vidx(rr, 0)] = x.x;
    v[vidx(rr, 1)] = x.y;
  }
}

// The update only needs fp32-faithful (not bit-identical) gates: ex2.approx-based forms, abs error ~1e-7
__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_fast(float x) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x)); }


__device__ __forceinline__ void regs_gate_warps() { asm volatile("setmaxnreg.inc.sync.aligned.u32 112;"); }
__device__ __forceinline__ void regs_service_warps() { asm volatile("setmaxnreg.dec.sync.aligned.u32 32;"); }

__device__ __forceinline__ uint32_t idesc_tf32(int n) {  // kind::tf32, fp32 accumulate, A and B K-major, M = 128
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

__device__ __forceinline__ uint64_t gtimer() {
  uint64_t t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// timeline probe (GRU_TIMELINE=1 tools/diag_gru.py): CTA 0 records %globaltimer at the hand-over points of the first steps
#define GS_STAMP(role, idx)                                                                     \
  do {                                                                                          \
    if (p.dbg && blockIdx.x == 0 && (idx) < 1024) p.dbg[(role) * 1024 + (idx)] = gtimer();      \
  } while (0)

struct GruOutMaps {  // [T(+1), Rs, cols] tensors, boxes of [1, rpt, 32]
  CUtensorMap gi, rzn, ghn, Y, HU;
};

struct GruFwdArgs {
  unsigned long long* dbg;
  int T, N, A;
  int64_t Rs;
  int rpt;              // rows per CTA
  const float* gi;      // [T, Rs, 384]  x @ Wi + bi
  const float* bhn;     // [128]
  const uint8_t* done;  // [T, N]
  float* rzn;           // [T, Rs, 384]
  float* ghn;           // [T, Rs, 128]
  float* Y;             // [T, Rs, 128]
  float* HU;            // [T+1, Rs, 128]; HU[0] is the (masked) initial state
};

__global__ void __launch_bounds__(GS_THREADS, 1)
gru_scan_fwd_kernel(const __grid_constant__ CUtensorMap tmWh, const __grid_constant__ CUtensorMap tmWl,
                    const __grid_constant__ GruOutMaps om, const GruFwdArgs p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sB = base;                        // GS_FWD_STAGES x {hi 12K, lo 12K}
  uint8_t* sOut = sB + GS_FWD_STAGES * GS_FWD_STAGE;  // 6 staging boxes (r, z, n, gh_n, y, h) of the block being finished (1 KiB-aligned)
  uint8_t* sIn = sOut + GS_OUT_BOXES * GS_CHUNK;  // 3 staging boxes: the next block's gi columns, loaded while this block is computed
  uint64_t* bars = reinterpret_cast<uint64_t*>(sIn + GS_IN_BOXES * GS_CHUNK);
  uint64_t* b_full = bars;
  uint64_t* b_empty = bars + GS_FWD_STAGES;
  uint64_t* acc_full = bars + 2 * GS_FWD_STAGES;  // 2 accumulators
  uint64_t* acc_empty = acc_full + 2;
  uint64_t* a_ready = acc_empty + 2;
  uint64_t* in_full = a_ready + 1;
  uint64_t* in_empty = in_full + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(in_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int T = p.T;
  // a CTA owns p.rpt (32, 64 or 128) rows of its 128-row MMA tile: with few rows, spreading them over more SMs divides the
  // per-SM stream of saved activations; the unused rows of the tile are zero operands
  const int64_t tile_row0 = (int64_t)blockIdx.x * p.rpt;

  if (warp == GS_GATE_WARPS + 1 && lane == 0) {
    for (int i = 0; i < GS_FWD_STAGES; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], GS_GATE_WARPS);
    }
    mbar_init(a_ready, GS_GATE_WARPS);
    mbar_init(in_full, 1);
    mbar_init(in_empty, GS_GATE_WARPS);
    fence_barrier_init();
  } else if (warp == GS_GATE_WARPS) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp >= GS_GATE_WARPS) {
    regs_service_warps();
    if (warp == GS_GATE_WARPS) {
      // ===================== TMA producer: W_h^T pieces, the same 16 every timestep =====================
      if (lane == 0) {
        uint32_t it = 0;
        for (int t = 0; t < T; ++t)
          for (int jb = 0; jb < 4; ++jb)
            for (int kc = 0; kc < 4; ++kc, ++it) {
              const int s = it % GS_FWD_STAGES;
              mbar_wait(&b_empty[s], ((it / GS_FWD_STAGES) & 1) ^ 1);
              GS_STAMP(0, it);
              mbar_expect_tx(&b_full[s], GS_FWD_STAGE);
              uint8_t* st = sB + (size_t)s * GS_FWD_STAGE;
#pragma unroll
              for (int g = 0; g < 3; ++g) {
                tma_load_2d(st + g * 4096, &tmWh, kc * 32, g * kH + 32 * jb, &b_full[s]);
                tma_load_2d(st + GS_FWD_STAGE / 2 + g * 4096, &tmWl, kc * 32, g * kH + 32 * jb, &b_full[s]);
              }
            }
      }
    } else if (warp == GS_GATE_WARPS + 1) {
      // ===================== MMA issuer =====================
      if (lane == 0) {
        const uint32_t idesc = idesc_tf32(96);
        uint32_t it = 0;
        for (int t = 0; t < T; ++t) {
          mbar_wait(a_ready, t & 1);
          tc_fence_after();
          GS_STAMP(1, t * 16);
          for (int jb = 0; jb < 4; ++jb) {
            const int acc = jb & 1;
            const uint32_t use = (uint32_t)t * 2 + (jb >> 1);  // uses of this accumulator so far
            if (use > 0) {  // the gate warps have read the block that last occupied it
              mbar_wait(&acc_empty[acc], (use - 1) & 1);
              tc_fence_after();
            }
            const uint32_t tmem_d = tmem_base + GS_F_ACC + (uint32_t)(acc * 96);
            for (int kc = 0; kc < 4; ++kc, ++it) {
              const int s = it % GS_FWD_STAGES;
              mbar_wait(&b_full[s], (it / GS_FWD_STAGES) & 1);
              tc_fence_after();
              if (kc == 0) GS_STAMP(1, t * 16 + 1 + jb * 2);
              const uint32_t a_hi = tmem_base + (uint32_t)(kc * 32), a_lo = a_hi + GS_F_ALO;
              const uint32_t b_hi = smem_u32(sB + (size_t)s * GS_FWD_STAGE), b_lo = b_hi + GS_FWD_STAGE / 2;
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t ko = k * 32;
                umma_tf32_ts(tmem_d, a_lo + k * 8, umma_desc_k_sw128(b_hi + ko), idesc, (kc | k) ? 1u : 0u);
                umma_tf32_ts(tmem_d, a_hi + k * 8, umma_desc_k_sw128(b_lo + ko), idesc, 1u);
                umma_tf32_ts(tmem_d, a_hi + k * 8, umma_desc_k_sw128(b_hi + ko), idesc, 1u);
              }
              umma_commit(&b_empty[s]);
            }
            umma_commit(&acc_full[acc]);
            GS_STAMP(1, t * 16 + 2 + jb * 2);
          }
        }
      }
    } else if (warp == GS_GATE_WARPS + 2) {
      // ============ TMA loader of the input pre-activations: the gi columns of block (t, jb + 1) land while block (t, jb) is computed ====
      if (lane == 0) {
        for (int n = 0; n < 4 * T; ++n) {
          const int t = n >> 2, jb = n & 3;
          mbar_wait(in_empty, ((uint32_t)n & 1u) ^ 1u);
          mbar_expect_tx(in_full, 3u * (uint32_t)p.rpt * 128u);
#pragma unroll
          for (int g = 0; g < 3; ++g) tma_load_3d(sIn + g * GS_CHUNK, &om.gi, g * kH + 32 * jb, (int)tile_row0, t, in_full);
        }
      }
    }
  } else {
    regs_gate_warps();
    // ===================== gates: warp = (32 rows, 8 of every 32 hidden units), thread = 4 x 2 patch =====================
    const int sp = warp & 3, cq = warp >> 2;
    const GateGeom gg = make_geom(sp, lane, tile_row0, p.Rs, p.rpt);
    const uint32_t tmem_lane = tmem_base + ((uint32_t)(sp * 32) << 16);
    const bool grp_live = 32 * sp < p.rpt && tile_row0 + 32 * sp < p.Rs;  // this warp's 32 rows hold rows of the tile
    const bool grp_leader = cq == 0 && lane == 0;
    float h[32];  // masked previous state: block jb at [8 jb, 8 jb + 8)
    float bh[8];
#pragma unroll
    for (int jb = 0; jb < 4; ++jb) {
      load_patch(&h[8 * jb], p.HU, kH, 32 * jb + 8 * cq, gg);
      tmem_st_patch_split(tmem_lane + (uint32_t)(32 * jb + 8 * cq), tmem_lane + GS_F_ALO + (uint32_t)(32 * jb + 8 * cq), &h[8 * jb]);
      bh[2 * jb] = p.bhn[32 * jb + 8 * cq + 2 * gg.m];
      bh[2 * jb + 1] = p.bhn[32 * jb + 8 * cq + 2 * gg.m + 1];
    }
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(a_ready);

    for (int t = 0; t < T; ++t) {
      bool keep[4];  // row is live and not reset before the next step
#pragma unroll
      for (int rr = 0; rr < 4; ++rr)
        keep[rr] = gg.valid[rr] && !((t + 1 < T) && p.done[(int64_t)(t + 1) * p.N + gg.grow[rr] / p.A]);
#pragma unroll
      for (int jb = 0; jb < 4; ++jb) {
        float gi_r[8], gi_z[8], gi_n[8];
        mbar_wait(in_full, (uint32_t)(t * 4 + jb) & 1u);
        unstage_patch(gi_r, sIn + 0 * GS_CHUNK, 8 * cq, gg);
        unstage_patch(gi_z, sIn + 1 * GS_CHUNK, 8 * cq, gg);
        unstage_patch(gi_n, sIn + 2 * GS_CHUNK, 8 * cq, gg);
        __syncwarp();
        if (lane == 0) mbar_arrive(in_empty);  // the loader may fetch the next block's columns
        if (threadIdx.x == 0) GS_STAMP(2, (t * 4 + jb) * 6 + 0);
        mbar_wait(&acc_full[jb & 1], (uint32_t)(t * 2 + (jb >> 1)) & 1u);
        tc_fence_after();
        if (threadIdx.x == 0) GS_STAMP(2, (t * 4 + jb) * 6 + 1);
        uint32_t ar[8], az[8], an[8];
        const uint32_t tcol = tmem_lane + GS_F_ACC + (uint32_t)((jb & 1) * 96 + 8 * cq);
        tmem_ld_patch_nowait(tcol, ar);
        tmem_ld_patch_nowait(tcol + 32, az);
        tmem_ld_patch_nowait(tcol + 64, an);
        tmem_ld_wait();
        tc_fence_before();  // this warp's part of the accumulator is in registers: hand the buffer back
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[jb & 1]);
        if (threadIdx.x == 0) GS_STAMP(2, (t * 4 + jb) * 6 + 2);
        float y_[8];
#pragma unroll
        for (int rr = 0; rr < 4; ++rr)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int i = vidx(rr, e);
            const float r = sigmoid_fast(gi_r[i] + __uint_as_float(ar[i]));
            const float z = sigmoid_fast(gi_z[i] + __uint_as_float(az[i]));
            const float ghn = __uint_as_float(an[i]) + bh[2 * jb + e];
            const float n = tanh_fast(gi_n[i] + r * ghn);
            const float hn = (1.0f - z) * n + z * h[8 * jb + i];
            gi_r[i] = r; gi_z[i] = z; gi_n[i] = n;  // reuse as output registers
            ar[i] = __float_as_uint(ghn);
            y_[i] = hn;
            h[8 * jb + i] = keep[rr] ? hn : 0.0f;
          }
        if (threadIdx.x == 0) GS_STAMP(2, (t * 4 + jb) * 6 + 3);
        // staging + bulk stores per group of the 4 warps that share 32 rows (sub-boxes of [32 rows x 32 floats]): the groups do not wait
        // for each other, a 128-thread barrier instead of a 512-thread one
        if (grp_live) {
          if (grp_leader) bulk_wait_read<0>();  // the previous block's bulk stores of this group have read its sub-boxes
          named_bar_sync(1 + sp, 128);
          stage_patch(sOut + 0 * GS_CHUNK, 8 * cq, gi_r, gg);
          stage_patch(sOut + 1 * GS_CHUNK, 8 * cq, gi_z, gg);
          stage_patch(sOut + 2 * GS_CHUNK, 8 * cq, gi_n, gg);
          stage_patch(sOut + 3 * GS_CHUNK, 8 * cq, reinterpret_cast<const float*>(ar), gg);
          stage_patch(sOut + 4 * GS_CHUNK, 8 * cq, y_, gg);
          stage_patch(sOut + 5 * GS_CHUNK, 8 * cq, &h[8 * jb], gg);
          fence_proxy_async();
          named_bar_sync(1 + sp, 128);
          if (grp_leader) {
            const int r0 = (int)tile_row0 + 32 * sp;
            const uint8_t* src = sOut + sp * 4096;
            tma_store_3d(&om.rzn, src + 0 * GS_CHUNK, 32 * jb, r0, t);
            tma_store_3d(&om.rzn, src + 1 * GS_CHUNK, kH + 32 * jb, r0, t);
            tma_store_3d(&om.rzn, src + 2 * GS_CHUNK, 2 * kH + 32 * jb, r0, t);
            tma_store_3d(&om.ghn, src + 3 * GS_CHUNK, 32 * jb, r0, t);
            tma_store_3d(&om.Y, src + 4 * GS_CHUNK, 32 * jb, r0, t);
            tma_store_3d(&om.HU, src + 5 * GS_CHUNK, 32 * jb, r0, t + 1);
            bulk_commit();
          }
        }
        if (threadIdx.x == 0) GS_STAMP(2, (t * 4 + jb) * 6 + 4);
      }
      if (t + 1 < T) {
        // every MMA of this step has completed (the last block's acc_full was observed): the A operand may be replaced
#pragma unroll
        for (int jb = 0; jb < 4; ++jb)
          tmem_st_patch_split(tmem_lane + (uint32_t)(32 * jb + 8 * cq), tmem_lane + GS_F_ALO + (uint32_t)(32 * jb + 8 * cq), &h[8 * jb]);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(a_ready);  // one arrival per warp: 512 serialized shared-memory arrivals cost microseconds
        if (threadIdx.x == 0) GS_STAMP(2, (t * 4 + 3) * 6 + 5);
      }
    }
  }
  if (threadIdx.x < GS_GATE_THREADS && (threadIdx.x >> 5) < 4 && (threadIdx.x & 31) == 0) bulk_wait_all();  // the group leaders
  tc_fence_before();
  __syncthreads();
  if (warp == GS_GATE_WARPS) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

struct GruBwdMaps {  // [T(+1), Rs, cols] saved activations, boxes of [1, rpt, 32]
  CUtensorMap dY, rzn, ghn, HU;
};

struct GruBwdArgs {
  int T, N, A;
  int64_t Rs;
  int rpt;              // rows per CTA
  const float* dY;      // [T, Rs, 128]
  const float* rzn;     // [T, Rs, 384]
  const float* ghn;     // [T, Rs, 128]
  const float* HU;      // [T+1, Rs, 128]
  const uint8_t* done;  // [T, N]
  float* dgi;           // [T, Rs, 384]  [da_r, da_z, da_n]
  float* dgh;           // [T, Rs, 384]  [da_r, da_z, da_n * r]
  float* dbi;           // [384] += column sums of dgi (the input-side bias gradient), optional
  float* dbhn;          // [128] += column sums of da_n * r (the hidden-side bias gradient of the candidate gate), optional
};

__global__ void __launch_bounds__(GS_THREADS, 1)
gru_scan_bwd_kernel(const __grid_constant__ CUtensorMap tmWh, const __grid_constant__ CUtensorMap tmWl,
                    const __grid_constant__ GruBwdMaps im, const GruBwdArgs p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sB = base;                         // GS_STAGES x {hi 16K, lo 16K}
  uint8_t* sIn = sB + GS_STAGES * GS_BWD_STAGE;  // 6 staging boxes: dY, r, z, n, gh_n, hu columns of the next block (TMA-loaded)
  float* sCol = reinterpret_cast<float*>(sIn + 6 * GS_CHUNK);  // [4][128] column sums of da_r, da_z, da_n, da_n * r over this CTA's rows
  uint64_t* bars = reinterpret_cast<uint64_t*>(sCol + 4 * kH);
  uint64_t* b_full = bars;
  uint64_t* b_empty = bars + GS_STAGES;
  uint64_t* a_full = bars + 2 * GS_STAGES;   // the three A slots of a block (tensor memory) are handed over together
  uint64_t* a_empty = a_full + 1;
  uint64_t* acc_full = a_empty + 1;
  uint64_t* in_full = acc_full + 1;
  uint64_t* in_empty = in_full + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(in_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int T = p.T;
  // a CTA owns p.rpt (32, 64 or 128) rows of its 128-row MMA tile: with few rows, spreading them over more SMs divides the
  // per-SM stream of saved activations; the unused rows of the tile are zero operands
  const int64_t tile_row0 = (int64_t)blockIdx.x * p.rpt;

  if (warp == GS_GATE_WARPS + 1 && lane == 0) {
    for (int i = 0; i < GS_STAGES; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    mbar_init(a_full, GS_GATE_WARPS);
    mbar_init(a_empty, 1);
    mbar_init(acc_full, 1);
    mbar_init(in_full, 1);
    mbar_init(in_empty, GS_GATE_WARPS);
    fence_barrier_init();
  }
  if (threadIdx.x < 4 * kH) sCol[threadIdx.x] = 0.f;
  // the layout fills the 227 KiB to the last kilobyte: it relies on the (declared) 1 KiB alignment of the dynamic shared window
  if (reinterpret_cast<uint8_t*>(tmem_ptr + 1) > smem_raw + GS_SMEM) __trap();
  if (warp == GS_GATE_WARPS) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp >= GS_GATE_WARPS) {
    regs_service_warps();
    if (warp == GS_GATE_WARPS) {
      // ============ TMA producer: W_h pieces [128 outputs x 32 contraction columns], order (block, gate) ============
      if (lane == 0) {
        uint32_t it = 0;
        for (int si = 0; si + 1 < T; ++si)
          for (int jb = 0; jb < 4; ++jb)
            for (int g = 0; g < 3; ++g, ++it) {
              const int s = it % GS_STAGES;
              mbar_wait(&b_empty[s], ((it / GS_STAGES) & 1) ^ 1);
              mbar_expect_tx(&b_full[s], GS_BWD_STAGE);
              uint8_t* st = sB + (size_t)s * GS_BWD_STAGE;
              tma_load_2d(st, &tmWh, g * kH + 32 * jb, 0, &b_full[s]);
              tma_load_2d(st + GS_CHUNK, &tmWl, g * kH + 32 * jb, 0, &b_full[s]);
            }
      }
    } else if (warp == GS_GATE_WARPS + 1) {
      // ===================== MMA issuer: carry[128 rows, 128] = dgh_t @ W_h^T =====================
      if (lane == 0) {
        const uint32_t idesc = idesc_tf32(128);
        uint32_t it = 0;
        for (int si = 0; si + 1 < T; ++si) {
          const uint32_t tmem_d = tmem_base + GS_B_ACC + (uint32_t)((si & 1) * 128);
          for (int jb = 0; jb < 4; ++jb) {
            const uint32_t n = (uint32_t)si * 4 + jb;
            mbar_wait(a_full, n & 1);
            for (int g = 0; g < 3; ++g, ++it) {
              const int s = it % GS_STAGES;
              mbar_wait(&b_full[s], (it / GS_STAGES) & 1);
              tc_fence_after();
              const uint32_t a_hi = tmem_base + (uint32_t)(g * 32), a_lo = a_hi + GS_B_ALO;
              const uint32_t b_hi = smem_u32(sB + (size_t)s * GS_BWD_STAGE), b_lo = b_hi + GS_CHUNK;
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t ko = k * 32;
                umma_tf32_ts(tmem_d, a_lo + k * 8, umma_desc_k_sw128(b_hi + ko), idesc, (jb | g | k) ? 1u : 0u);
                umma_tf32_ts(tmem_d, a_hi + k * 8, umma_desc_k_sw128(b_lo + ko), idesc, 1u);
                umma_tf32_ts(tmem_d, a_hi + k * 8, umma_desc_k_sw128(b_hi + ko), idesc, 1u);
              }
              umma_commit(&b_empty[s]);
            }
            umma_commit(a_empty);
          }
          umma_commit(acc_full);
        }
      }
    } else if (warp == GS_GATE_WARPS + 2) {
      // ============ TMA loader of the saved activations: the six column blocks of (step, jb + 1) land while (step, jb) is computed ======
      if (lane == 0) {
        for (int n = 0; n < 4 * T; ++n) {
          const int t = T - 1 - (n >> 2), jb = n & 3;
          mbar_wait(in_empty, ((uint32_t)n & 1u) ^ 1u);
          mbar_expect_tx(in_full, 6u * (uint32_t)p.rpt * 128u);
          const int r0 = (int)tile_row0;
          tma_load_3d(sIn + 0 * GS_CHUNK, &im.dY, 32 * jb, r0, t, in_full);
          tma_load_3d(sIn + 1 * GS_CHUNK, &im.rzn, 32 * jb, r0, t, in_full);
          tma_load_3d(sIn + 2 * GS_CHUNK, &im.rzn, kH + 32 * jb, r0, t, in_full);
          tma_load_3d(sIn + 3 * GS_CHUNK, &im.rzn, 2 * kH + 32 * jb, r0, t, in_full);
          tma_load_3d(sIn + 4 * GS_CHUNK, &im.ghn, 32 * jb, r0, t, in_full);
          tma_load_3d(sIn + 5 * GS_CHUNK, &im.HU, 32 * jb, r0, t, in_full);
        }
      }
    }
  } else {
    regs_gate_warps();
    // ============ gate backward: warp = (32 rows, 8 of every 32 hidden units), thread = 4 x 2 patch ============
    const int sp = warp & 3, cq = warp >> 2;
    const GateGeom gg = make_geom(sp, lane, tile_row0, p.Rs, p.rpt);
    const uint32_t tmem_lane = tmem_base + ((uint32_t)(sp * 32) << 16);
    float cz[32];  // dh_{t+1} * z_{t+1}
#pragma unroll
    for (int i = 0; i < 32; ++i) cz[i] = 0.0f;

    for (int si = 0; si < T; ++si) {
      const int t = T - 1 - si;
      const int64_t slab = (int64_t)t * p.Rs;
      const bool has_carry = si > 0;
      bool use_carry[4];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr)
        use_carry[rr] = has_carry && gg.valid[rr] && !p.done[(int64_t)(t + 1) * p.N + gg.grow[rr] / p.A];
      const uint32_t tmem_acc = tmem_lane + GS_B_ACC + (uint32_t)(((si + 1) & 1) * 128);  // written by the MMAs of step si-1
      const bool feed = t > 0;  // the carry of step 0 goes nowhere
#pragma unroll
      for (int jb = 0; jb < 4; ++jb) {
        const int j0 = 32 * jb + 8 * cq;
        float dy[8], r_[8], z_[8], n_[8], gh_[8], hu[8];
        mbar_wait(in_full, (uint32_t)(si * 4 + jb) & 1u);
        unstage_patch(dy, sIn + 0 * GS_CHUNK, 8 * cq, gg);
        unstage_patch(r_, sIn + 1 * GS_CHUNK, 8 * cq, gg);
        unstage_patch(z_, sIn + 2 * GS_CHUNK, 8 * cq, gg);
        unstage_patch(n_, sIn + 3 * GS_CHUNK, 8 * cq, gg);
        unstage_patch(gh_, sIn + 4 * GS_CHUNK, 8 * cq, gg);
        unstage_patch(hu, sIn + 5 * GS_CHUNK, 8 * cq, gg);
        __syncwarp();
        if (lane == 0) mbar_arrive(in_empty);  // the loader may fetch the next block's columns
        uint32_t acc[8];
        if (has_carry) {
          if (jb == 0) {
            mbar_wait(acc_full, (si - 1) & 1);
            tc_fence_after();
          }
          tmem_ld_patch_nowait(tmem_acc + (uint32_t)j0, acc);
          tmem_ld_wait();
        }
#pragma unroll
        for (int rr = 0; rr < 4; ++rr)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int i = vidx(rr, e);
            float dh = dy[i];
            if (use_carry[rr]) dh += cz[8 * jb + i] + __uint_as_float(acc[i]);
            const float r = r_[i], z = z_[i], n = n_[i];
            const float dan = dh * (1.0f - z) * (1.0f - n * n);
            const float daz = dh * (hu[i] - n) * z * (1.0f - z);
            const float dar = dan * gh_[i] * r * (1.0f - r);
            cz[8 * jb + i] = dh * z;
            r_[i] = dar; z_[i] = daz; n_[i] = dan; gh_[i] = dan * r;  // reuse as output registers
          }
        if (p.dbi) {
          // bias gradients: this thread's 4 rows in registers, the 8 lanes that share its two columns by shuffles, one shared-memory
          // add per column and warp (the column sums of dgi / dgh used to be two more passes over 2 GB)
          float cs[8];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            cs[e] = r_[vidx(0, e)] + r_[vidx(1, e)] + r_[vidx(2, e)] + r_[vidx(3, e)];
            cs[2 + e] = z_[vidx(0, e)] + z_[vidx(1, e)] + z_[vidx(2, e)] + z_[vidx(3, e)];
            cs[4 + e] = n_[vidx(0, e)] + n_[vidx(1, e)] + n_[vidx(2, e)] + n_[vidx(3, e)];
            cs[6 + e] = gh_[vidx(0, e)] + gh_[vidx(1, e)] + gh_[vidx(2, e)] + gh_[vidx(3, e)];
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            cs[i] += __shfl_xor_sync(0xffffffffu, cs[i], 4);
            cs[i] += __shfl_xor_sync(0xffffffffu, cs[i], 8);
            cs[i] += __shfl_xor_sync(0xffffffffu, cs[i], 16);
          }
          if (lane < 4) {
#pragma unroll
            for (int i = 0; i < 8; ++i) atomicAdd(&sCol[(i >> 1) * kH + j0 + 2 * lane + (i & 1)], cs[i]);
          }
        }
        store_patch(r_, p.dgi + slab * (3 * kH), 3 * kH, j0, gg);
        store_patch(z_, p.dgi + slab * (3 * kH), 3 * kH, kH + j0, gg);
        store_patch(n_, p.dgi + slab * (3 * kH), 3 * kH, 2 * kH + j0, gg);
        store_patch(r_, p.dgh + slab * (3 * kH), 3 * kH, j0, gg);
        store_patch(z_, p.dgh + slab * (3 * kH), 3 * kH, kH + j0, gg);
        store_patch(gh_, p.dgh + slab * (3 * kH), 3 * kH, 2 * kH + j0, gg);
        if (feed) {
          const uint32_t n = (uint32_t)si * 4 + jb;
          mbar_wait(a_empty, (n & 1) ^ 1);
          tc_fence_after();
          tmem_st_patch_split(tmem_lane + (uint32_t)(8 * cq), tmem_lane + GS_B_ALO + (uint32_t)(8 * cq), r_);
          tmem_st_patch_split(tmem_lane + (uint32_t)(32 + 8 * cq), tmem_lane + GS_B_ALO + (uint32_t)(32 + 8 * cq), z_);
          tmem_st_patch_split(tmem_lane + (uint32_t)(64 + 8 * cq), tmem_lane + GS_B_ALO + (uint32_t)(64 + 8 * cq), gh_);
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(a_full);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (p.dbi && threadIdx.x < 4 * kH) {
    const float v = sCol[threadIdx.x];
    if (threadIdx.x < 3 * kH) atomicAdd(p.dbi + threadIdx.x, v);
    else if (p.dbhn) atomicAdd(p.dbhn + (threadIdx.x - 3 * kH), v);
  }
  if (warp == GS_GATE_WARPS) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

}  // namespace

unsigned long long* g_gru_dbg = nullptr;

// Rows per CTA. Measured on B200 (tools/gru_rpt_experiment.sh): the per-timestep chain of a scan CTA shortens when it owns fewer
// rows (RWARE shard, 2048 rows: 57.6 / 41.2 / 33.7 ms per step of 8 minibatches at 128 / 64 / 32 rows), but the scans run on a
// forked stream beside the guider's persistent kernels and a scan CTA fills its SM (227 KB of shared memory): more than ~64 scan
// CTAs starve the guider and the step gets slower (LBF, 8192 rows: GRU 63 -> 45 ms but the step 284 -> 289 ms at 64 rows). So: the
// fewest rows per CTA that keep the scan on at most 64 SMs. MAGPO_GRU_RPT overrides, for experiments.
static int gru_rows_per_tile(int64_t Rs) {
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("MAGPO_GRU_RPT");
    const int v = e ? atoi(e) : 0;
    forced = (v >= 8 && v <= 128) ? v : 0;
  }
  if (forced) return forced;
  if (ceil_div(Rs, 32) <= 64) return 32;
  if (ceil_div(Rs, 64) <= 64) return 64;
  return 128;
}

// HU[0] must already hold the masked initial state. WhT_hi/lo: TF32 images of W_h^T [384, 128].
int gru_scan_fwd(cudaStream_t s, int T, int N, int A, const float* gi, const float* WhT_hi, const float* WhT_lo, const float* bhn,
                 const uint8_t* done, float* rzn, float* ghn, float* Y, float* HU) {
  const int64_t Rs = (int64_t)N * A;
  CUtensorMap tmh, tml;
  if (!tc_make_map(&tmh, WhT_hi, 3 * kH, kH, kH, 32) || !tc_make_map(&tml, WhT_lo, 3 * kH, kH, kH, 32)) return MAGPO_ERR_ARG;
  if (once_per_device(ONCE_GRU_FWD))
    MAGPO_CUDA_OK(cudaFuncSetAttribute(gru_scan_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GS_SMEM));
  const int rpt = gru_rows_per_tile(Rs);
  GruOutMaps om;
  const int ob = std::min(rpt, 32);  // the outputs leave per group of 32 rows
  if (!tc_make_map3(&om.gi, gi, T, Rs, 3 * kH, rpt) || !tc_make_map3(&om.rzn, rzn, T, Rs, 3 * kH, ob) || !tc_make_map3(&om.ghn, ghn, T, Rs, kH, ob) ||
      !tc_make_map3(&om.Y, Y, T, Rs, kH, ob) || !tc_make_map3(&om.HU, HU, T + 1, Rs, kH, ob))
    return MAGPO_ERR_ARG;
  GruFwdArgs a{g_gru_dbg, T, N, A, Rs, rpt, gi, bhn, done, rzn, ghn, Y, HU};
  // per row and step: 3xTF32 MMAs are the pipe work; bytes: gi 1536 read, rzn+ghn+Y+HU 3072 written
  ProfScope ps(PROF_GRU, s, 4608.0 * (double)Rs * T);
  gru_scan_fwd_kernel<<<(unsigned)ceil_div(Rs, rpt), GS_THREADS, GS_SMEM, s>>>(tmh, tml, om, a);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

// Wh_hi/lo: TF32 images of W_h [128, 384] (un-transposed).
int gru_scan_bwd(cudaStream_t s, int T, int N, int A, const float* dY, const float* rzn, const float* ghn, const float* HU,
                 const uint8_t* done, const float* Wh_hi, const float* Wh_lo, float* dgi, float* dgh, float* dbi, float* dbhn) {
  const int64_t Rs = (int64_t)N * A;
  CUtensorMap tmh, tml;
  if (!tc_make_map(&tmh, Wh_hi, kH, 3 * kH, 3 * kH, 128) || !tc_make_map(&tml, Wh_lo, kH, 3 * kH, 3 * kH, 128)) return MAGPO_ERR_ARG;
  if (once_per_device(ONCE_GRU_BWD))
    MAGPO_CUDA_OK(cudaFuncSetAttribute(gru_scan_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GS_SMEM));
  const int rpt = gru_rows_per_tile(Rs);
  GruBwdMaps im;
  if (!tc_make_map3(&im.dY, dY, T, Rs, kH, rpt) || !tc_make_map3(&im.rzn, rzn, T, Rs, 3 * kH, rpt) || !tc_make_map3(&im.ghn, ghn, T, Rs, kH, rpt) ||
      !tc_make_map3(&im.HU, HU, T + 1, Rs, kH, rpt))
    return MAGPO_ERR_ARG;
  GruBwdArgs a{T, N, A, Rs, rpt, dY, rzn, ghn, HU, done, dgi, dgh, dbi, dbhn};
  ProfScope ps(PROF_GRU, s, 6144.0 * (double)Rs * T);
  gru_scan_bwd_kernel<<<(unsigned)ceil_div(Rs, rpt), GS_THREADS, GS_SMEM, s>>>(tmh, tml, im, a);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

}  // namespace magpo

// GRU_TIMELINE=1 tools/diag_gru.py: device buffer of 3 x 1024 uint64 %globaltimer stamps written by CTA 0 of the forward scan
extern "C" int magpo_debug_gru_timeline(unsigned long long* buf) {
  magpo::g_gru_dbg = buf;
  return MAGPO_OK;
}

// Host-only: the rows per CTA both scans launch with for Rs = N * A rows (tests assert which tile branch a case covers).
extern "C" int magpo_debug_gru_rows_per_tile(int64_t Rs) { return magpo::gru_rows_per_tile(Rs); }
