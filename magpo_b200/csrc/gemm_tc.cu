// Tensor-core GEMM for the update path:  Y[M,N] (+)= X[M,K] @ B^T (+ bias) (relu),  B given as [N,K] (K-major).
// fp32 in / fp32 out with fp32-faithful accuracy through the 3xTF32 split
//     x = x_hi + x_lo  (both exactly representable in TF32, round-to-nearest):   X.B ~= Xhi.Bhi + Xlo.Bhi + Xhi.Blo
// (dropped term ~2^-22 relative), accumulated in fp32 in tensor memory.
//
// Blackwell-native structure (sm_100a): persistent CTAs, one per SM, warp-specialised:
//   warp 0      TMA producer: X tiles [128 rows x 32 floats] (one 128B-swizzle atom) into an smem ring; B (hi, lo) is loaded
//               once per CTA and stays resident in shared memory
//   warps 8-11  converters: split each landed X chunk in place into hi (+ a second buffer for lo), fence to the async proxy
//   warp 1      MMA issuer: one thread issues tcgen05.mma.kind::tf32 (M=128, N=BN, K=8) x3 per k-step into TMEM;
//               tcgen05.commit releases the smem stage / publishes the accumulator
//   warps 4-7   epilogue: tcgen05.ld (thread = row) -> bias/relu -> 128B-swizzled smem slab -> TMA store
//               (or TMA reduce-add for Y += ...), double-buffered; TMEM accumulators are double-buffered too.
// The tensor core re-reads its shared-memory operands on every K = 8 step, so with three MMAs per step the operand reads (not the
// flops, not HBM) are what a narrow GEMM saturates first (measured: ~70 % of the shared-memory bandwidth at N = 64). For N tiles <= 128
// the hi and lo images of B therefore sit side by side and the two products that share A_hi run as ONE MMA of width 2 BN:
//     D[:, 0:BN] += A_hi B_hi,  D[:, BN:2BN] += A_hi B_lo   (one instruction),      D[:, 0:BN] += A_lo B_hi
// and the epilogue adds the two halves. A is read twice per step instead of three times.
// Every mbarrier wait is bounded and traps instead of hanging.
#include <cuda.h>

#include <stdlib.h>

#include <vector>

#include "common.cuh"
#include "kernels.cuh"
#include "tc_ptx.cuh"

namespace magpo {
namespace {

using tcp::TC_BM;
constexpr int TC_KC = 32;
constexpr int TC_CHUNK_BYTES = TC_BM * TC_KC * 4;  // 16 KiB
constexpr int TC_CONV_THREADS = 256;               // warps 8..15
constexpr int TC_THREADS = 256 + TC_CONV_THREADS;
constexpr int TC_MAX_STAGES = 6;
constexpr int kTnMaxRows = 8192;  // rows one gemm_tc_tn accumulator reduces (see gemm_tc_tn)
constexpr uint32_t TC_SMEM_LIMIT = 227 * 1024;

struct TcParams {
  int M, N, K, BN, kchunks, stages, flags, num_row_tiles, tmem_cols, stacked /* B hi | lo as one operand of width 2 BN */;
  const float* bias;
};

using namespace tcp;

__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmBh,
               const __grid_constant__ CUtensorMap tmBl, const __grid_constant__ CUtensorMap tmY, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve (everything TMA touches is 1024-byte aligned)
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int b_chunk_bytes = p.BN * 128;
  uint8_t* sBh = base;                                             // per k chunk: [hi rows | lo rows]
  uint8_t* sBl = sBh + b_chunk_bytes;
  uint8_t* sA = sBh + (size_t)p.kchunks * 2 * b_chunk_bytes;       // stages x {hi 16K, lo 16K}
  uint8_t* sOut = sA + (size_t)p.stages * 2 * TC_CHUNK_BYTES;      // 2 x 16K
  float* sBias = reinterpret_cast<float*>(sOut + 2 * TC_CHUNK_BYTES);  // 256 floats
  uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + 256);
  uint64_t* full_raw = bars;
  uint64_t* full_conv = bars + TC_MAX_STAGES;
  uint64_t* empty = bars + 2 * TC_MAX_STAGES;
  uint64_t* tmem_full = bars + 3 * TC_MAX_STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* b_ready = tmem_empty + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(b_ready + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.y * p.BN;

  if (warp == 1 && lane == 0) {
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&full_raw[i], 1);
      mbar_init(&full_conv[i], TC_CONV_THREADS / 32);  // one arrival per converter warp
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 4);  // one arrival per epilogue warp
    }
    mbar_init(b_ready, 1);
    fence_barrier_init();
  } else if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"((uint32_t)p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x >= 128 && threadIdx.x < 256) {  // epilogue threads stage the bias slice
    const int j = threadIdx.x - 128;
    for (int c = j; c < p.BN; c += 128) sBias[c] = p.bias ? p.bias[n0 + c] : 0.0f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_expect_tx(b_ready, 2u * p.kchunks * b_chunk_bytes);
      for (int c = 0; c < p.kchunks; ++c) {
        tma_load_2d(sBh + (size_t)c * 2 * b_chunk_bytes, &tmBh, c * TC_KC, n0, b_ready);
        tma_load_2d(sBl + (size_t)c * 2 * b_chunk_bytes, &tmBl, c * TC_KC, n0, b_ready);
      }
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < p.num_row_tiles; tile += gridDim.x) {
        for (int c = 0; c < p.kchunks; ++c, ++it) {
          const int s = it % p.stages;
          mbar_wait(&empty[s], ((it / p.stages) & 1) ^ 1);
          mbar_expect_tx(&full_raw[s], TC_CHUNK_BYTES);
          tma_load_2d(sA + (size_t)s * 2 * TC_CHUNK_BYTES, &tmX, c * TC_KC, tile * TC_BM, &full_raw[s]);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_tf32(p.BN), idesc2 = umma_idesc_tf32(2 * p.BN);
      const int acc_cols = p.stacked ? 2 * p.BN : p.BN;
      mbar_wait(b_ready, 0);
      uint32_t it = 0, ti = 0;
      for (int tile = blockIdx.x; tile < p.num_row_tiles; tile += gridDim.x, ++ti) {
        const int acc = ti & 1;
        mbar_wait(&tmem_empty[acc], ((ti >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * acc_cols);
        for (int c = 0; c < p.kchunks; ++c, ++it) {
          const int s = it % p.stages;
          mbar_wait(&full_conv[s], (it / p.stages) & 1);
          tc_fence_after();
          const uint32_t a_hi = smem_u32(sA + (size_t)s * 2 * TC_CHUNK_BYTES);
          const uint32_t a_lo = a_hi + TC_CHUNK_BYTES;
          const uint32_t b_hi = smem_u32(sBh + (size_t)c * 2 * b_chunk_bytes);
          const uint32_t b_lo = smem_u32(sBl + (size_t)c * 2 * b_chunk_bytes);
#pragma unroll
          for (int k = 0; k < TC_KC / 8; ++k) {
            const uint32_t ko = k * 32;  // 8 tf32 = 32 bytes along K inside the swizzle atom
            if (p.stacked) {
              umma_tf32(tmem_d, umma_desc_k_sw128(a_hi + ko), umma_desc_k_sw128(b_hi + ko), idesc2, (c | k) ? 1u : 0u);
              umma_tf32(tmem_d, umma_desc_k_sw128(a_lo + ko), umma_desc_k_sw128(b_hi + ko), idesc, 1u);
            } else {
              umma_tf32(tmem_d, umma_desc_k_sw128(a_lo + ko), umma_desc_k_sw128(b_hi + ko), idesc, (c | k) ? 1u : 0u);
              umma_tf32(tmem_d, umma_desc_k_sw128(a_hi + ko), umma_desc_k_sw128(b_lo + ko), idesc, 1u);
              umma_tf32(tmem_d, umma_desc_k_sw128(a_hi + ko), umma_desc_k_sw128(b_hi + ko), idesc, 1u);
            }
          }
          umma_commit(&empty[s]);  // stage reusable once these MMAs have read it
        }
        umma_commit(&tmem_full[acc]);
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ===================== epilogue =====================
    const int sub = warp & 3;             // TMEM sub-partition of this warp: lanes [32*sub, 32*sub+32)
    const bool relu = p.flags & GEMM_RELU, accumulate = p.flags & GEMM_ACCUMULATE;
    const int nslab = p.BN / 32;
    const int acc_cols = p.stacked ? 2 * p.BN : p.BN;
    uint32_t ti = 0, slab_it = 0;
    for (int tile = blockIdx.x; tile < p.num_row_tiles; tile += gridDim.x, ++ti) {
      const int acc = ti & 1;
      mbar_wait(&tmem_full[acc], (ti >> 1) & 1);
      tc_fence_after();
      for (int sl = 0; sl < nslab; ++sl, ++slab_it) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(acc * acc_cols + sl * 32), v);
        if (p.stacked) {  // + the A_hi B_lo half
          uint32_t w[32];
          tmem_ld32(tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(acc * acc_cols + p.BN + sl * 32), w);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(w[j]));
        }
        if (sl == nslab - 1) {  // accumulator fully read: hand it back to the MMA warp (one arrival per warp: hundreds of
          tc_fence_before();    // arrivals on one mbarrier serialise in shared memory and cost a large part of a microsecond)
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[acc]);
        }
        // every warp stages and stores its own 32 rows ([32 x 32 floats] boxes): no barrier between the epilogue warps
        uint8_t* buf = sOut + (size_t)(slab_it & 1) * TC_CHUNK_BYTES + (size_t)sub * 4096;
        if (lane == 0) bulk_wait_read<1>();  // the store that last used this buffer has finished reading it
        __syncwarp();
        float4* dst_row = reinterpret_cast<float4*>(buf + (size_t)lane * 128);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float4 o;
          o.x = __uint_as_float(v[4 * j + 0]) + sBias[sl * 32 + 4 * j + 0];
          o.y = __uint_as_float(v[4 * j + 1]) + sBias[sl * 32 + 4 * j + 1];
          o.z = __uint_as_float(v[4 * j + 2]) + sBias[sl * 32 + 4 * j + 2];
          o.w = __uint_as_float(v[4 * j + 3]) + sBias[sl * 32 + 4 * j + 3];
          if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
          dst_row[j ^ (lane & 7)] = o;  // 128B swizzle: 16-byte chunk index XOR (row mod 8)
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          if (accumulate) tma_reduce_add_2d(&tmY, buf, n0 + sl * 32, tile * TC_BM + sub * 32);
          else tma_store_2d(&tmY, buf, n0 + sl * 32, tile * TC_BM + sub * 32);
          bulk_commit();
        }
      }
    }
    if (lane == 0) bulk_wait_all();
  } else if (warp >= 8) {
    // ===================== converters: lo = x - tf32_trunc(x) =====================
    // The landed fp32 chunk is itself the hi operand: kind::tf32 reads the top 19 bits of each word, i.e. truncates. Only the
    // residual is written (exact in fp32; the tensor core truncates it to TF32 in turn: relative error <= 2^-20).
    const int ct = threadIdx.x - 256;  // 0..TC_CONV_THREADS-1
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < p.num_row_tiles; tile += gridDim.x) {
      for (int c = 0; c < p.kchunks; ++c, ++it) {
        const int s = it % p.stages;
        mbar_wait(&full_raw[s], (it / p.stages) & 1);
        const float4* hi = reinterpret_cast<const float4*>(sA + (size_t)s * 2 * TC_CHUNK_BYTES);
        float4* lo = reinterpret_cast<float4*>(sA + (size_t)s * 2 * TC_CHUNK_BYTES + TC_CHUNK_BYTES);
#pragma unroll
        for (int i = 0; i < TC_CHUNK_BYTES / 16 / TC_CONV_THREADS; ++i) {
          const int idx = ct + i * TC_CONV_THREADS;
          lo[idx] = tf32_residual4(hi[idx]);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full_conv[s]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}


// =====================================================================================================================
// Weight-gradient GEMM on the tensor cores:  dW[K,N] += X[M,K]^T @ dY[M,N]   (K in {64,128}; reduction over the rows).
// Both operands are activations and are consumed exactly as they lie in memory: a [32 rows x 32 floats] TMA box is an
// MN-major (M/N contiguous) 128B-swizzled UMMA operand whose 8-row groups are the K=8 steps of kind::tf32. Both operands are
// split into TF32 hi/lo by the converter warps. Each CTA reduces a contiguous slab of at most kTnMaxRows rows into one TMEM
// accumulator and adds it to dW with a TMA reduce-add, so the cross-CTA reduction needs no extra pass.
// rows per pipeline stage: 32, or 64 where the stage stays small (narrow K and N): the per-stage hand-overs (barrier round trips of the
// producer / converter / MMA roles) cost the same for 16 KiB as for 48 KiB, and the narrow GEMMs were bound by them

struct TnParams {
  int K, BN, stages, tmem_cols, rc /* rows per stage */;
  int64_t M, rows_per_cta;
};

__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t saddr, uint32_t box_bytes) {
  // 32-bit MN-major operands must use the 128B swizzle with a 32-byte base (UMMA layout type SWIZZLE_128B_BASE32B,
  // TMA CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): the atom is 4 K-rows x 128 B, a K=8 step spans two atoms.
  // LBO = stride between 32-float column blocks (one TMA box), SBO = stride between 4-row groups.
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(box_bytes >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)1 << 61);
}

__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_tn_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDY,
                  const __grid_constant__ CUtensorMap tmDW, const TnParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int TN_RC = p.rc, TN_BOX = TN_RC * 128;  // one [rc rows x 32 floats] box
  const int x_bytes = (p.K / 32) * TN_BOX, y_bytes = (p.BN / 32) * TN_BOX;
  const int raw_bytes = x_bytes + y_bytes;  // per stage: [X hi | dY hi | X lo | dY lo]
  uint8_t* sStage = base;
  uint8_t* sOut = sStage + (size_t)p.stages * 2 * raw_bytes;  // 2 x 16 KiB
  uint64_t* bars = reinterpret_cast<uint64_t*>(sOut + 2 * TC_CHUNK_BYTES);
  uint64_t* full_raw = bars;
  uint64_t* full_conv = bars + TC_MAX_STAGES;
  uint64_t* empty = bars + 2 * TC_MAX_STAGES;
  uint64_t* tmem_full = bars + 3 * TC_MAX_STAGES;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.y * p.BN;
  const int64_t row_begin = (int64_t)blockIdx.x * p.rows_per_cta;
  const int64_t row_end = row_begin + p.rows_per_cta < p.M ? row_begin + p.rows_per_cta : p.M;
  const int nchunks = row_begin < row_end ? (int)((row_end - row_begin + TN_RC - 1) / TN_RC) : 0;

  if (warp == 1 && lane == 0) {
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&full_raw[i], 1);
      mbar_init(&full_conv[i], TC_CONV_THREADS / 32);  // one arrival per converter warp
      mbar_init(&empty[i], 1);
    }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
  } else if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"((uint32_t)p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (nchunks > 0) {
    if (warp == 0) {
      if (lane == 0) {
        for (int it = 0; it < nchunks; ++it) {
          const int s = it % p.stages;
          mbar_wait(&empty[s], ((it / p.stages) & 1) ^ 1);
          mbar_expect_tx(&full_raw[s], (uint32_t)raw_bytes);
          uint8_t* st = sStage + (size_t)s * 2 * raw_bytes;
          const int r0 = (int)(row_begin + (int64_t)it * TN_RC);
          for (int kb = 0; kb < p.K / 32; ++kb) tma_load_2d(st + kb * TN_BOX, &tmX, kb * 32, r0, &full_raw[s]);
          for (int nb = 0; nb < p.BN / 32; ++nb) tma_load_2d(st + x_bytes + nb * TN_BOX, &tmDY, n0 + nb * 32, r0, &full_raw[s]);
        }
      }
    } else if (warp == 1) {
      if (lane == 0) {
        // kind::tf32, fp32 accumulate, A and B MN-major, M = K (of the GEMM), N = BN
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(p.BN >> 3) << 17) |
                               ((uint32_t)(p.K >> 4) << 24);
        for (int it = 0; it < nchunks; ++it) {
          const int s = it % p.stages;
          mbar_wait(&full_conv[s], (it / p.stages) & 1);
          tc_fence_after();
          const uint32_t x_hi = smem_u32(sStage + (size_t)s * 2 * raw_bytes);
          const uint32_t y_hi = x_hi + x_bytes, x_lo = x_hi + raw_bytes, y_lo = y_hi + raw_bytes;
          for (int g = 0; g < TN_RC / 8; ++g) {
            const uint32_t go = g * 1024;  // next 8-row group = next K=8 step
            umma_tf32(tmem_base, umma_desc_mn_sw128(x_lo + go, TN_BOX), umma_desc_mn_sw128(y_hi + go, TN_BOX), idesc, (it | g) ? 1u : 0u);
            umma_tf32(tmem_base, umma_desc_mn_sw128(x_hi + go, TN_BOX), umma_desc_mn_sw128(y_lo + go, TN_BOX), idesc, 1u);
            umma_tf32(tmem_base, umma_desc_mn_sw128(x_hi + go, TN_BOX), umma_desc_mn_sw128(y_hi + go, TN_BOX), idesc, 1u);
          }
          umma_commit(&empty[s]);
        }
        umma_commit(tmem_full);
      }
    } else if (warp >= 4 && warp < 8) {
      const int et = threadIdx.x - 128;
      const int sub = warp & 3;
      // M = 128: lane l of sub-partition s holds row 32 s + l.  M = 64: rows 16 s + l live in lanes l < 16.
      const bool m64 = p.K == 64;
      const int row = m64 ? sub * 16 + lane : sub * 32 + lane;
      const bool active = !m64 || lane < 16;
      mbar_wait(tmem_full, 0);
      tc_fence_after();
      const int nslab = p.BN / 32;
      for (int sl = 0; sl < nslab; ++sl) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(sl * 32), v);
        uint8_t* buf = sOut + (size_t)(sl & 1) * TC_CHUNK_BYTES;
        if (et == 0) bulk_wait_read<1>();
        named_bar_sync(1, 128);
        if (active) {
          float4* dst_row = reinterpret_cast<float4*>(buf + (size_t)row * 128);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            dst_row[j ^ (row & 7)] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                                 __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        }
        fence_proxy_async();
        named_bar_sync(1, 128);
        if (et == 0) {
          tma_reduce_add_2d(&tmDW, buf, n0 + sl * 32, 0);
          bulk_commit();
        }
      }
      if (et == 0) bulk_wait_all();
    } else if (warp >= 8) {
      // converters: the landed chunks are the hi operands as they are (the tensor core truncates to TF32); write the residuals
      const int ct = threadIdx.x - 256;
      const int nvec = raw_bytes / 16;
      for (int it = 0; it < nchunks; ++it) {
        const int s = it % p.stages;
        mbar_wait(&full_raw[s], (it / p.stages) & 1);
        const float4* hi = reinterpret_cast<const float4*>(sStage + (size_t)s * 2 * raw_bytes);
        float4* lo = reinterpret_cast<float4*>(sStage + (size_t)s * 2 * raw_bytes + raw_bytes);
        for (int idx = ct; idx < nvec; idx += TC_CONV_THREADS) lo[idx] = tf32_residual4(hi[idx]);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full_conv[s]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}

__global__ void __launch_bounds__(256)
split_region_kernel(int64_t n, const float* __restrict__ x, float* __restrict__ hi, float* __restrict__ lo) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float h, l;
    split_tf32(x[i], h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

// ---------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// row-major [rows, cols] fp32 matrix with leading dimension ld; box = [box_rows, 32 floats], 128B swizzle
bool make_map(CUtensorMap* tm, const float* ptr, int64_t rows, int cols, int ld, int box_rows,
              CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {(cuuint32_t)TC_KC, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

bool tc_make_map(void* tensor_map, const float* ptr, int64_t rows, int cols, int ld, int box_rows) {
  return make_map(static_cast<CUtensorMap*>(tensor_map), ptr, rows, cols, ld, box_rows);
}
// [T, rows, cols] fp32 tensor (contiguous), boxes of [1, box_rows, 32 floats], 128B swizzle: per-timestep slabs whose row tiles clip at
// `rows` (the GRU scans' saved activations)
bool tc_make_map3(void* tensor_map, const float* ptr, int64_t T, int64_t rows, int cols, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t gdim[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)T};
  cuuint64_t gstride[2] = {(cuuint64_t)cols * 4, (cuuint64_t)rows * cols * 4};
  cuuint32_t box[3] = {(cuuint32_t)TC_KC, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(static_cast<CUtensorMap*>(tensor_map), CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(ptr), gdim, gstride, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Split a weight region into TF32 hi/lo copies and remember the mapping so that GEMMs on any sub-matrix find them.
int tc_prepare_region(cudaStream_t s, const float* base, int64_t n, float* hi, float* lo) {
  if (n <= 0) return MAGPO_OK;
  split_region_kernel<<<(unsigned)std::min<int64_t>(ceil_div(n, 256), 4 * kNumSMs), 256, 0, s>>>(n, base, hi, lo);
  MAGPO_LAUNCH_OK();
  // Workspaces are re-planned between calls (rollout vs. update, different T/N): drop every older registration whose
  // source range touches memory this one claims (its source or its hi/lo images) — a stale range must never match.
  auto overlaps = [](const float* a, int64_t na, const float* b, int64_t nb) { return a < b + nb && b < a + na; };
  std::vector<TcRegion>& g_regions = ctx().regions;
  for (size_t i = 0; i < g_regions.size();) {
    const TcRegion& r = g_regions[i];
    if (overlaps(r.base, r.n, base, n) || overlaps(r.base, r.n, hi, n) || overlaps(r.base, r.n, lo, n) ||
        overlaps(r.hi, r.n, base, n) || overlaps(r.lo, r.n, base, n))
      g_regions.erase(g_regions.begin() + (long)i);
    else
      ++i;
  }
  g_regions.push_back(TcRegion{base, n, hi, lo});
  return MAGPO_OK;
}

bool tc_lookup(const float* w, const float** hi, const float** lo) {
  const std::vector<TcRegion>& g_regions = ctx().regions;
  for (auto it = g_regions.rbegin(); it != g_regions.rend(); ++it) {
    const TcRegion& r = *it;
    if (w >= r.base && w < r.base + r.n) {
      *hi = r.hi + (w - r.base);
      *lo = r.lo + (w - r.base);
      return true;
    }
  }
  return false;
}

// Pick the N tile and ring depth; false when the shape does not fit the kernel.
static bool tc_plan(int64_t M, int N, int K, TcParams* p, uint32_t* smem_bytes) {
  if (K % TC_KC || K < TC_KC || N % 32 || M < 1) return false;
  const int cands[] = {256, 192, 128, 96, 64, 32};
  for (int bn : cands) {
    if (N % bn) continue;
    const uint32_t b_bytes = (uint32_t)K * bn * 8;
    const uint32_t fixed = b_bytes + 2 * TC_CHUNK_BYTES + 256 * 4 + 256 + 1024 /*alignment slack*/;
    if (fixed + 2 * 2 * TC_CHUNK_BYTES > TC_SMEM_LIMIT) continue;
    int stages = (int)((TC_SMEM_LIMIT - fixed) / (2 * TC_CHUNK_BYTES));
    stages = std::min(stages, TC_MAX_STAGES);
    p->BN = bn;
    p->kchunks = K / TC_KC;
    p->stages = stages;
    p->stacked = bn <= 128 ? 1 : 0;
    int cols = 32;
    while (cols < (p->stacked ? 4 : 2) * bn) cols <<= 1;
    p->tmem_cols = cols;
    *smem_bytes = fixed + (uint32_t)stages * 2 * TC_CHUNK_BYTES;
    return true;
  }
  return false;
}

bool tc_supported(int64_t M, int N, int K, const float* X, int ldx, const float* Y, int ldy, int ldb) {
  if (!get_encode()) return false;
  if ((ldx & 3) || (ldy & 3) || (ldb & 3)) return false;
  if ((reinterpret_cast<uintptr_t>(X) & 15) || (reinterpret_cast<uintptr_t>(Y) & 15)) return false;
  TcParams p;
  uint32_t smem;
  return M >= 256 && tc_plan(M, N, K, &p, &smem);
}

// Y[M,N] (+)= X[M,K] @ B^T with B = Bhi + Blo given as [N,K] row-major (leading dimension ldb).
int gemm_tc(cudaStream_t s, int64_t M, int N, int K, const float* X, int ldx, const float* Bhi, const float* Blo, int ldb,
            const float* bias, float* Y, int ldy, int flags) {
  TcParams p;
  uint32_t smem;
  if (!tc_plan(M, N, K, &p, &smem)) return MAGPO_ERR_UNSUPPORTED;
  if ((flags & GEMM_ACCUMULATE) && ((flags & GEMM_RELU) || bias)) return MAGPO_ERR_UNSUPPORTED;
  p.M = (int)M; p.N = N; p.K = K; p.flags = flags; p.bias = bias;
  p.num_row_tiles = (int)ceil_div(M, TC_BM);
  CUtensorMap tmX, tmBh, tmBl, tmY;
  if (!make_map(&tmX, X, M, K, ldx, TC_BM) || !make_map(&tmBh, Bhi, N, K, ldb, p.BN) || !make_map(&tmBl, Blo, N, K, ldb, p.BN) ||
      !make_map(&tmY, Y, M, N, ldy, 32))
    return MAGPO_ERR_ARG;
  if (once_per_device(ONCE_GEMM_TC))
    MAGPO_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_LIMIT));
  const int n_tiles = N / p.BN;
  dim3 grid((unsigned)std::max(1, std::min(p.num_row_tiles, kNumSMs / n_tiles)), (unsigned)n_tiles);
  ProfScope ps(M < 65536 ? PROF_GEMM_SMALL : PROF_GEMM_NN, s, 2.0 * (double)M * N * K, 4.0 * (double)M * (K + N + ((flags & GEMM_ACCUMULATE) ? N : 0)));
  gemm_tc_kernel<<<grid, TC_THREADS, smem, s>>>(tmX, tmBh, tmBl, tmY, p);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}


static bool tn_plan(int N, int K, TnParams* p, uint32_t* smem_bytes) {
  if ((K != 64 && K != 128) || N % 32) return false;
  const int cands[] = {256, 192, 128, 96, 64, 32};
  for (int bn : cands) {
    if (N % bn) continue;
    const int rc = (K / 32 + bn / 32) <= 4 ? 64 : 32;
    const uint32_t raw = (uint32_t)(K / 32 + bn / 32) * (uint32_t)rc * 128u;
    const uint32_t fixed = 2 * TC_CHUNK_BYTES + 256 + 1024;
    if (fixed + 2 * 2 * raw > TC_SMEM_LIMIT) continue;
    p->K = K;
    p->BN = bn;
    p->rc = rc;
    p->stages = std::min<int>(TC_MAX_STAGES, (int)((TC_SMEM_LIMIT - fixed) / (2 * raw)));
    int cols = 32;
    while (cols < bn) cols <<= 1;
    p->tmem_cols = cols;
    *smem_bytes = fixed + (uint32_t)p->stages * 2 * raw;
    return true;
  }
  return false;
}

bool tc_tn_supported(int64_t M, int N, int K, const float* X, int ldx, const float* dY, int ldy, const float* dW, int ldw) {
  if (!get_encode()) return false;
  if ((ldx & 3) || (ldy & 3) || (ldw & 3)) return false;
  if ((reinterpret_cast<uintptr_t>(X) & 15) || (reinterpret_cast<uintptr_t>(dY) & 15) || (reinterpret_cast<uintptr_t>(dW) & 15)) return false;
  TnParams p;
  uint32_t smem;
  return M >= 256 && tn_plan(N, K, &p, &smem);
}

// dW[K,N] += X[M,K]^T @ dY[M,N]
int gemm_tc_tn(cudaStream_t s, int64_t M, int N, int K, const float* X, int ldx, const float* dY, int ldy, float* dW, int ldw) {
  TnParams p;
  uint32_t smem;
  if (!tn_plan(N, K, &p, &smem)) return MAGPO_ERR_UNSUPPORTED;
  p.M = M;
  const int n_tiles = N / p.BN;
  const int TN_RC = p.rc;
  const int64_t chunks = ceil_div(M, TN_RC);
  // A TMEM accumulator takes at most kTnMaxRows rows: the tensor core's fp32 accumulation error grows with the length of the chain (one
  // slab of 65 k rows put CoordSum's GRU weight gradients 2.7e-4 from float64), so long reductions run as several full waves of slabs.
  const int64_t per_wave = std::max(1, kNumSMs / n_tiles);
  const int64_t waves = ceil_div(chunks, per_wave * (kTnMaxRows / TN_RC));
  const int gx = (int)std::max<int64_t>(1, std::min<int64_t>(chunks, per_wave * waves));
  p.rows_per_cta = ceil_div(chunks, gx) * TN_RC;
  CUtensorMap tmX, tmDY, tmDW;
  // boxes of [32 rows x 32 floats] for the operands; the accumulator slab is [K rows x 32 floats]
  if (!make_map(&tmX, X, M, K, ldx, TN_RC, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) ||
      !make_map(&tmDY, dY, M, N, ldy, TN_RC, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) || !make_map(&tmDW, dW, K, N, ldw, K))
    return MAGPO_ERR_ARG;
  if (once_per_device(ONCE_GEMM_TN))
    MAGPO_CUDA_OK(cudaFuncSetAttribute(gemm_tc_tn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_LIMIT));
  ProfScope ps(PROF_GEMM_TN, s, 2.0 * (double)M * N * K, 4.0 * (double)M * (K + N));
  gemm_tc_tn_kernel<<<dim3((unsigned)gx, (unsigned)n_tiles), TC_THREADS, smem, s>>>(tmX, tmDY, tmDW, p);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

}  // namespace magpo

using namespace magpo;

// Test hook: Y = X @ W (+bias) through the tensor-core path. WT is W^T [N,K] row-major; scratch holds 2*N*K floats.
extern "C" int magpo_test_gemm_tc(magpo_stream_t s_, int64_t M, int N, int K, const float* X, int ldx, const float* WT,
                                  float* scratch, const float* bias, float* Y, int ldy, int flags) {
  cudaStream_t s = as_stream(s_);
  if (!tc_supported(M, N, K, X, ldx, Y, ldy, K)) return MAGPO_ERR_UNSUPPORTED;
  MAGPO_TRY(tc_prepare_region(s, WT, (int64_t)N * K, scratch, scratch + (int64_t)N * K));
  return gemm_tc(s, M, N, K, X, ldx, scratch, scratch + (int64_t)N * K, K, bias, Y, ldy, flags);
}

extern "C" int magpo_test_gemm_tc_tn(magpo_stream_t s_, int64_t M, int N, int K, const float* X, int ldx, const float* dY, int ldy,
                                     float* dW, int ldw) {
  if (!tc_tn_supported(M, N, K, X, ldx, dY, ldy, dW, ldw)) return MAGPO_ERR_UNSUPPORTED;
  return gemm_tc_tn(as_stream(s_), M, N, K, X, ldx, dY, ldy, dW, ldw);
}
