// Chunkwise retention for the training pass (T > 1), forward and backward, on the tensor cores.
// Reference: networks/retention.py:66-100 (SimpleRetention chunkwise), :117-213 (decay matrix / xi).
//
// One CTA per env sequence walks the rollout in chunks of Lc = 32 / A timesteps (<= 32 token rows). With
//   lam_t = done_t ? 0 : kappa,   c[tl] = prod_{s<=tl} lam,   e[tl] = prod_{s>tl} lam   (inside the chunk),
//   D[n,m] = [order(n,m)] prod_{tl(m) < s <= tl(n)} lam_s     (order: n >= m for the decoder, tl(n) >= tl(m) for the encoder)
// the chunk is four small GEMMs (this is the reference's own formulation, with the state carried between chunks):
//   P = D * (Q K^T)            O  = P V + diag(c) Q Hp          Hn = c_L Hp + (diag(e) K)^T V
// and the backward, with G = dL/dHn carried in reverse, W = D * (dO V^T):
//   dQ = W K + diag(c) dO Hp^T      dK = W^T Q + diag(e) V G^T      dV = P^T dO + diag(e) K G      dHp = c_L G + (diag(c) Q)^T dO
// Only the state entering each chunk is saved for the backward (T/Lc x 16 KiB per env instead of T x 16 KiB).
// All products run as warp-level m16n8k8 TF32 MMAs with the 3xTF32 split (x = hi + lo by truncation, hi*hi + hi*lo + lo*hi, fp32
// accumulate), operands staged once per chunk in shared memory; the running state (H forward, G backward) lives in
// accumulator fragments for the whole sequence. Tiles are 32x64x64 at most, far below what a tcgen05 instruction (M >= 64,
// operands through descriptors, accumulator in TMEM) is built for, so the warp-level instruction is the right size here.
#include "common.cuh"
#include "kernels.cuh"

namespace magpo {
namespace {

constexpr int RC_ROWS = 32;  // token rows per chunk (padded)
constexpr int LDA = 68;      // operand read as A rows or as B^T: ld % 32 == 4 -> conflict-free fragment loads
constexpr int LDB = 72;      // operand read as B[k][n] or as A^T: ld % 32 == 8
constexpr int LDP = 36;      // [32][32] chunk matrices read as A rows
constexpr int LDPT = 40;     // [32][32] chunk matrices read as A^T

struct Frag {
  uint32_t h[4], l[4];
};
struct FragB {
  uint32_t h[2], l[2];
};

// x = hi + lo: hi = x truncated to TF32 (what the tensor core reads of the fp32 word anyway), lo = x - hi exact in fp32 and
// truncated to TF32 by the tensor core in turn (relative error of the 3-term product <= 2^-20). Two ALU ops per element.
__device__ __forceinline__ void split(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xFFFFE000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}

__device__ __forceinline__ void mma8(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ void mma3(float (&c)[4], const Frag& a, const FragB& b) {
  mma8(c, a.l, b.h);
  mma8(c, a.h, b.l);
  mma8(c, a.h, b.h);
}

// ldmatrix moves 8 x 16-byte rows per matrix: for fp32 data that is an 8 x 4 tile whose word (row r, col c) lands in lane 4 r + c —
// exactly the m16n8k8 TF32 fragment layout (a: row g, col tq). One instruction replaces the 4 (A) or 2 (B) scalar LDS of a
// K-contiguous fragment; rows are 16-byte aligned (ld % 4 == 0, k0 % 4 == 0) and ld % 32 == 4 keeps the 8 rows on distinct banks.
__device__ __forceinline__ void ldsm_x4(const float* p, uint32_t (&r)[4]) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a) : "memory");
}
__device__ __forceinline__ void ldsm_x2(const float* p, uint32_t (&r)[2]) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(a) : "memory");
}
__device__ __forceinline__ void split_u(uint32_t x, uint32_t& hi, uint32_t& lo) {
  hi = x & 0xFFFFE000u;
  lo = __float_as_uint(__uint_as_float(x) - __uint_as_float(hi));
}

// A[m][k] = X[m][k]  (16 x 8 tile at (m0, k0)); matrices: (rows 0-7, k 0-3), (rows 8-15, k 0-3), (rows 0-7, k 4-7), (rows 8-15, k 4-7)
__device__ __forceinline__ Frag lda_row(const float* X, int ld, int m0, int k0, int g, int tq) {
  const int lane = 4 * g + tq;
  uint32_t r[4];
  ldsm_x4(X + (m0 + (lane & 7) + ((lane >> 3) & 1) * 8) * ld + k0 + (lane >> 4) * 4, r);
  Frag f;
#pragma unroll
  for (int i = 0; i < 4; ++i) split_u(r[i], f.h[i], f.l[i]);
  return f;
}
// A[m][k] = X[k][m]
__device__ __forceinline__ Frag lda_tr(const float* X, int ld, int m0, int k0, int g, int tq) {
  Frag f;
  split(X[(k0 + tq) * ld + m0 + g], f.h[0], f.l[0]);
  split(X[(k0 + tq) * ld + m0 + g + 8], f.h[1], f.l[1]);
  split(X[(k0 + tq + 4) * ld + m0 + g], f.h[2], f.l[2]);
  split(X[(k0 + tq + 4) * ld + m0 + g + 8], f.h[3], f.l[3]);
  return f;
}
// B[k][n] = Y[k][n]  (8 x 8 tile at (k0, n0))
__device__ __forceinline__ FragB ldb(const float* Y, int ld, int k0, int n0, int g, int tq) {
  FragB f;
  split(Y[(k0 + tq) * ld + n0 + g], f.h[0], f.l[0]);
  split(Y[(k0 + tq + 4) * ld + n0 + g], f.h[1], f.l[1]);
  return f;
}
// B[k][n] = Y[n][k]; matrices: (rows n0..n0+7, k 0-3), (same rows, k 4-7)
__device__ __forceinline__ FragB ldb_tr(const float* Y, int ld, int k0, int n0, int g, int tq) {
  const int lane = 4 * g + tq;
  uint32_t r[2];
  ldsm_x2(Y + (n0 + (lane & 7)) * ld + k0 + ((lane >> 3) & 1) * 4, r);
  FragB f;
  split_u(r[0], f.h[0], f.l[0]);
  split_u(r[1], f.h[1], f.l[1]);
  return f;
}

__device__ __forceinline__ void zero4(float (&c)[4]) { c[0] = c[1] = c[2] = c[3] = 0.f; }

// Per-chunk decay bookkeeping, identical in every warp: lane l holds cd = number of dones in timesteps t0..t0+l.
struct ChunkDecay {
  int cd_lane;  // this lane's cumulative done count (lanes >= L repeat the last value)
  __device__ __forceinline__ void init(const uint8_t* done, int t0, int L, int N, int n, int lane) {
    const bool d = done && lane < L && done[(int64_t)(t0 + lane) * N + n];
    const unsigned m = __ballot_sync(0xffffffffu, d);
    cd_lane = __popc(m & (0xffffffffu >> (31 - lane)));
  }
  __device__ __forceinline__ int cd(int tl) const { return __shfl_sync(0xffffffffu, cd_lane, tl); }
};

// smem tables shared by the two kernels
struct Tables {
  float* kpow;       // [40] kappa^j
  int* cds;          // [32] cumulative done count per chunk timestep
  uint8_t* row_tl;   // [32] timestep of a token row (row / A)
};

// D[n][m] of the chunk (rows/cols beyond the valid range give 0 because their operands are zero)
template <bool CAUSAL>
__device__ __forceinline__ float decay_nm(const Tables& tb, int n, int m) {
  const int tn = tb.row_tl[n], tm = tb.row_tl[m];
  const bool order = CAUSAL ? (n >= m) : (tn >= tm);
  if (!order || tb.cds[tn] != tb.cds[tm]) return 0.f;
  return tb.kpow[tn - tm];
}

// ------------------------------------------------------------------------------------------------ forward
template <bool CAUSAL>
__global__ void __launch_bounds__(256, 2)
retention_chunk_fwd_kernel(int T, int N, int A, int Lc, float kappa, const float* __restrict__ q, const float* __restrict__ k,
                           const float* __restrict__ v, int ld, const float* __restrict__ H0, const uint8_t* __restrict__ done,
                           float* __restrict__ ret, float* __restrict__ Hck, float* __restrict__ Hout) {
  extern __shared__ __align__(16) float sm[];
  float* Hp = sm;                 // [64][LDB]   state entering the chunk            (B of Q Hp)
  float* Qs = Hp + 64 * LDB;      // [32][LDA]                                        (A of Q K^T, A of Q Hp)
  float* Ks = Qs + RC_ROWS * LDA; // [32][LDA]                                        (B^T of Q K^T)
  float* Kt = Ks + RC_ROWS * LDA; // [32][LDB]   diag(e) K                            (A^T of the state update)
  float* Vs = Kt + RC_ROWS * LDB; // [32][LDB]                                        (B of P V and of the state update)
  float* Ps = Vs + RC_ROWS * LDB; // [32][LDP]                                        (A of P V)
  Tables tb;
  tb.kpow = Ps + RC_ROWS * LDP;
  tb.cds = reinterpret_cast<int*>(tb.kpow + 40);
  tb.row_tl = reinterpret_cast<uint8_t*>(tb.cds + 32);

  const int n = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tq = lane & 3;
  if (tid == 0) {
    float p = 1.f;
    for (int j = 0; j < 40; ++j) { tb.kpow[j] = p; p *= kappa; }
  }
  if (tid < 32) tb.row_tl[tid] = (uint8_t)(tid / A);
  // zero the operand tiles once: rows beyond the chunk's valid rows stay zero unless a longer chunk wrote them,
  // in which case the per-chunk stores below overwrite them with zeros again
  for (int i = tid; i < RC_ROWS * LDP; i += 256) Ps[i] = 0.f;

  // running state in accumulator fragments: warp owns rows 16*mt.., column tiles 8*(nt0+j)..
  const int mt = warp & 3, nt0 = (warp >> 2) * 4;
  float Hacc[4][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int r = 16 * mt + g, c = 8 * (nt0 + j) + 2 * tq;
    float2 lo2 = make_float2(0.f, 0.f), hi2 = make_float2(0.f, 0.f);
    if (H0) {
      lo2 = *reinterpret_cast<const float2*>(H0 + ((int64_t)n * 64 + r) * 64 + c);
      hi2 = *reinterpret_cast<const float2*>(H0 + ((int64_t)n * 64 + r + 8) * 64 + c);
    }
    Hacc[j][0] = lo2.x; Hacc[j][1] = lo2.y; Hacc[j][2] = hi2.x; Hacc[j][3] = hi2.y;
  }

  const int nchunks = (T + Lc - 1) / Lc;
  float pq[8], pk[8], pv[8];
  auto fetch = [&](int ch) {
    const int t0 = ch * Lc, L = min(Lc, T - t0), rows = L * A;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int idx = tid + j * 256, row = idx >> 6, col = idx & 63;
      pq[j] = pk[j] = pv[j] = 0.f;
      if (row < rows) {
        const int tl = tb.row_tl[row];
        const int64_t grow = ((int64_t)(t0 + tl) * N + n) * A + (row - tl * A);
        pq[j] = q[grow * ld + col]; pk[j] = k[grow * ld + col]; pv[j] = v[grow * ld + col];
      }
    }
  };
  __syncthreads();  // row_tl / kpow visible
  fetch(0);

  for (int ch = 0; ch < nchunks; ++ch) {
    const int t0 = ch * Lc, L = min(Lc, T - t0), rows = L * A;
    ChunkDecay cdk;
    cdk.init(done, t0, L, N, n, lane);
    const int cd_last = cdk.cd(L - 1);
    if (warp == 0) tb.cds[lane] = cdk.cd_lane;
    // state entering the chunk -> smem (+ checkpoint for the backward)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = 16 * mt + g, c = 8 * (nt0 + j) + 2 * tq;
      *reinterpret_cast<float2*>(Hp + r * LDB + c) = make_float2(Hacc[j][0], Hacc[j][1]);
      *reinterpret_cast<float2*>(Hp + (r + 8) * LDB + c) = make_float2(Hacc[j][2], Hacc[j][3]);
      if (Hck) {
        float* dst = Hck + (((int64_t)ch * N + n) * 64) * 64;
        *reinterpret_cast<float2*>(dst + r * 64 + c) = make_float2(Hacc[j][0], Hacc[j][1]);
        *reinterpret_cast<float2*>(dst + (r + 8) * 64 + c) = make_float2(Hacc[j][2], Hacc[j][3]);
      }
    }
    // operands
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int idx = tid + j * 256, row = idx >> 6, col = idx & 63;
      const int tl = tb.row_tl[row];
      const int cdt = cdk.cd(tl);  // warp-uniform row: every lane takes part in the shuffle
      const float e = (row < rows && cdt == cd_last) ? tb.kpow[L - 1 - tl] : 0.f;
      Qs[row * LDA + col] = pq[j];
      Ks[row * LDA + col] = pk[j];
      Kt[row * LDB + col] = pk[j] * e;
      Vs[row * LDB + col] = pv[j];
    }
    __syncthreads();  // A: operands, tables, Hp ready
    if (ch + 1 < nchunks) fetch(ch + 1);

    // ---- phase 1: P = D * (Q K^T)  (one 16x8 tile per warp)  and  O2 = Q Hp  (column tile `warp`, both row tiles)
    float o2[2][4];
    zero4(o2[0]); zero4(o2[1]);
    {
      const int mi = warp >> 2, ni = warp & 3;
      float s[4];
      zero4(s);
#pragma unroll
      for (int k0 = 0; k0 < 64; k0 += 8) {
        const Frag a0 = lda_row(Qs, LDA, 0, k0, g, tq);
        const Frag a1 = lda_row(Qs, LDA, 16, k0, g, tq);
        const FragB bk = ldb_tr(Ks, LDA, k0, 8 * ni, g, tq);
        mma3(s, mi ? a1 : a0, bk);
        const FragB bh = ldb(Hp, LDB, k0, 8 * warp, g, tq);
        mma3(o2[0], a0, bh);
        mma3(o2[1], a1, bh);
      }
      const int r = 16 * mi + g, c = 8 * ni + 2 * tq;
      Ps[r * LDP + c] = s[0] * decay_nm<CAUSAL>(tb, r, c);
      Ps[r * LDP + c + 1] = s[1] * decay_nm<CAUSAL>(tb, r, c + 1);
      Ps[(r + 8) * LDP + c] = s[2] * decay_nm<CAUSAL>(tb, r + 8, c);
      Ps[(r + 8) * LDP + c + 1] = s[3] * decay_nm<CAUSAL>(tb, r + 8, c + 1);
    }
    __syncthreads();  // B: P ready; every read of Hp is done

    // ---- phase 2: O = P V + diag(c) O2 ;  H <- c_L H + Kt^T V
    {
      float o1[2][4];
      zero4(o1[0]); zero4(o1[1]);
#pragma unroll
      for (int k0 = 0; k0 < RC_ROWS; k0 += 8) {
        const FragB bv = ldb(Vs, LDB, k0, 8 * warp, g, tq);
        mma3(o1[0], lda_row(Ps, LDP, 0, k0, g, tq), bv);
        mma3(o1[1], lda_row(Ps, LDP, 16, k0, g, tq), bv);
      }
#pragma unroll
      for (int mi = 0; mi < 2; ++mi)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int row = 16 * mi + g + 8 * h;
          if (row < rows) {
            const int tl = tb.row_tl[row];
            const float cc = (tb.cds[tl] == 0) ? tb.kpow[tl + 1] : 0.f;
            const int64_t grow = ((int64_t)(t0 + tl) * N + n) * A + (row - tl * A);
            *reinterpret_cast<float2*>(ret + grow * 64 + 8 * warp + 2 * tq) =
                make_float2(o1[mi][2 * h] + cc * o2[mi][2 * h], o1[mi][2 * h + 1] + cc * o2[mi][2 * h + 1]);
          }
        }
    }
    {
      const float cL = (cd_last == 0) ? tb.kpow[L] : 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int x = 0; x < 4; ++x) Hacc[j][x] *= cL;
#pragma unroll
      for (int k0 = 0; k0 < RC_ROWS; k0 += 8) {
        const Frag a = lda_tr(Kt, LDB, 16 * mt, k0, g, tq);
#pragma unroll
        for (int j = 0; j < 4; ++j) mma3(Hacc[j], a, ldb(Vs, LDB, k0, 8 * (nt0 + j), g, tq));
      }
    }
    __syncthreads();  // C: all reads of this chunk's operands are done
  }
  if (Hout) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = 16 * mt + g, c = 8 * (nt0 + j) + 2 * tq;
      float* dst = Hout + (int64_t)n * 64 * 64;
      *reinterpret_cast<float2*>(dst + r * 64 + c) = make_float2(Hacc[j][0], Hacc[j][1]);
      *reinterpret_cast<float2*>(dst + (r + 8) * 64 + c) = make_float2(Hacc[j][2], Hacc[j][3]);
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward
template <bool CAUSAL>
__global__ void __launch_bounds__(256, 2)
retention_chunk_bwd_kernel(int T, int N, int A, int Lc, float kappa, const float* __restrict__ q, const float* __restrict__ k,
                           const float* __restrict__ v, int ld, const uint8_t* __restrict__ done,
                           const float* __restrict__ Hck, const float* __restrict__ dret, float* __restrict__ dq,
                           float* __restrict__ dk, float* __restrict__ dv, int ldd) {
  extern __shared__ __align__(16) float sm[];
  float* Hp = sm;                   // [64][LDA]  state entering the chunk      (B^T of dO Hp^T)
  float* Gs = Hp + 64 * LDA;        // [64][LDA]  G = dL/d(state leaving)       (B^T of V G^T)
  float* Gt = Gs + 64 * LDA;        // [64][LDA]  G^T                           (B^T of K G)
  float* Qs = Gt + 64 * LDA;        // [32][LDA]  A of Q K^T ; B of W^T Q
  float* Ks = Qs + RC_ROWS * LDA;   // [32][LDA]  B^T of Q K^T ; B of W K ; A of K G
  float* Vs = Ks + RC_ROWS * LDA;   // [32][LDA]  B^T of dO V^T ; A of V G^T
  float* Ds = Vs + RC_ROWS * LDA;   // [32][LDA]  dO: A of dO V^T, dO Hp^T ; B of P^T dO, (cQ)^T dO
  float* Qc = Ds + RC_ROWS * LDA;   // [32][LDB]  diag(c) Q                     (A^T of the G update)
  float* Ps = Qc + RC_ROWS * LDB;   // [32][LDPT] P                             (A^T of P^T dO)
  float* Ws = Ps + RC_ROWS * LDPT;  // [32][LDP]  W                             (A of W K ; A^T of W^T Q)
  Tables tb;
  tb.kpow = Ws + RC_ROWS * LDP;
  tb.cds = reinterpret_cast<int*>(tb.kpow + 40);
  tb.row_tl = reinterpret_cast<uint8_t*>(tb.cds + 32);

  const int n = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tq = lane & 3;
  if (tid == 0) {
    float p = 1.f;
    for (int j = 0; j < 40; ++j) { tb.kpow[j] = p; p *= kappa; }
  }
  if (tid < 32) tb.row_tl[tid] = (uint8_t)(tid / A);

  const int mt = warp & 3, nt0 = (warp >> 2) * 4;
  float Gacc[4][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) zero4(Gacc[j]);

  const int nchunks = (T + Lc - 1) / Lc;
  float pq[8], pk[8], pv[8], pd[8];
  auto fetch = [&](int ch) {
    const int t0 = ch * Lc, L = min(Lc, T - t0), rows = L * A;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int idx = tid + j * 256, row = idx >> 6, col = idx & 63;
      pq[j] = pk[j] = pv[j] = pd[j] = 0.f;
      if (row < rows) {
        const int tl = tb.row_tl[row];
        const int64_t grow = ((int64_t)(t0 + tl) * N + n) * A + (row - tl * A);
        pq[j] = q[grow * ld + col]; pk[j] = k[grow * ld + col]; pv[j] = v[grow * ld + col];
        pd[j] = dret[grow * 64 + col];
      }
    }
  };
  __syncthreads();
  fetch(nchunks - 1);

  for (int ch = nchunks - 1; ch >= 0; --ch) {
    const int t0 = ch * Lc, L = min(Lc, T - t0), rows = L * A;
    ChunkDecay cdk;
    cdk.init(done, t0, L, N, n, lane);
    const int cd_last = cdk.cd(L - 1);
    if (warp == 0) tb.cds[lane] = cdk.cd_lane;
    // G (and its transpose) -> smem
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = 16 * mt + g, c = 8 * (nt0 + j) + 2 * tq;
      *reinterpret_cast<float2*>(Gs + r * LDA + c) = make_float2(Gacc[j][0], Gacc[j][1]);
      *reinterpret_cast<float2*>(Gs + (r + 8) * LDA + c) = make_float2(Gacc[j][2], Gacc[j][3]);
      Gt[c * LDA + r] = Gacc[j][0];
      Gt[(c + 1) * LDA + r] = Gacc[j][1];
      Gt[c * LDA + r + 8] = Gacc[j][2];
      Gt[(c + 1) * LDA + r + 8] = Gacc[j][3];
    }
    // state that entered this chunk
    {
      const float4* src = reinterpret_cast<const float4*>(Hck + ((int64_t)ch * N + n) * 64 * 64);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int idx = tid + j * 256;  // float4 index: 16 per row
        const float4 h = src[idx];
        *reinterpret_cast<float4*>(Hp + (idx >> 4) * LDA + (idx & 15) * 4) = h;
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int idx = tid + j * 256, row = idx >> 6, col = idx & 63;
      const int tl = tb.row_tl[row];
      const int cdt = cdk.cd(tl);  // warp-uniform row: every lane takes part in the shuffle
      const float cc = (row < rows && cdt == 0) ? tb.kpow[tl + 1] : 0.f;
      Qs[row * LDA + col] = pq[j];
      Ks[row * LDA + col] = pk[j];
      Vs[row * LDA + col] = pv[j];
      Ds[row * LDA + col] = pd[j];
      Qc[row * LDB + col] = pq[j] * cc;
    }
    __syncthreads();  // A
    if (ch > 0) fetch(ch - 1);

    // ---- phase 1: P = D*(Q K^T), W = D*(dO V^T) (one tile per warp); state products for column tile `warp`
    float dq2[2][4], dk2[2][4], dv2[2][4];
    zero4(dq2[0]); zero4(dq2[1]); zero4(dk2[0]); zero4(dk2[1]); zero4(dv2[0]); zero4(dv2[1]);
    {
      const int mi = warp >> 2, ni = warp & 3;
      float s[4], w[4];
      zero4(s); zero4(w);
#pragma unroll
      for (int k0 = 0; k0 < 64; k0 += 8) {
        {
          const Frag a = lda_row(Qs, LDA, 16 * mi, k0, g, tq);
          mma3(s, a, ldb_tr(Ks, LDA, k0, 8 * ni, g, tq));
        }
        const Frag d0 = lda_row(Ds, LDA, 0, k0, g, tq);
        const Frag d1 = lda_row(Ds, LDA, 16, k0, g, tq);
        mma3(w, mi ? d1 : d0, ldb_tr(Vs, LDA, k0, 8 * ni, g, tq));
        {  // dq2[n][r] = sum_c dO[n][c] Hp[r][c]
          const FragB b = ldb_tr(Hp, LDA, k0, 8 * warp, g, tq);
          mma3(dq2[0], d0, b);
          mma3(dq2[1], d1, b);
        }
        {  // dk2[m][r] = sum_c V[m][c] G[r][c]
          const FragB b = ldb_tr(Gs, LDA, k0, 8 * warp, g, tq);
          mma3(dk2[0], lda_row(Vs, LDA, 0, k0, g, tq), b);
          mma3(dk2[1], lda_row(Vs, LDA, 16, k0, g, tq), b);
        }
        {  // dv2[m][c] = sum_r K[m][r] G[r][c] = sum_r K[m][r] Gt[c][r]
          const FragB b = ldb_tr(Gt, LDA, k0, 8 * warp, g, tq);
          mma3(dv2[0], lda_row(Ks, LDA, 0, k0, g, tq), b);
          mma3(dv2[1], lda_row(Ks, LDA, 16, k0, g, tq), b);
        }
      }
      const int r = 16 * mi + g, c = 8 * ni + 2 * tq;
      const float d00 = decay_nm<CAUSAL>(tb, r, c), d01 = decay_nm<CAUSAL>(tb, r, c + 1);
      const float d10 = decay_nm<CAUSAL>(tb, r + 8, c), d11 = decay_nm<CAUSAL>(tb, r + 8, c + 1);
      Ps[r * LDPT + c] = s[0] * d00; Ps[r * LDPT + c + 1] = s[1] * d01;
      Ps[(r + 8) * LDPT + c] = s[2] * d10; Ps[(r + 8) * LDPT + c + 1] = s[3] * d11;
      Ws[r * LDP + c] = w[0] * d00; Ws[r * LDP + c + 1] = w[1] * d01;
      Ws[(r + 8) * LDP + c] = w[2] * d10; Ws[(r + 8) * LDP + c + 1] = w[3] * d11;
    }
    __syncthreads();  // B

    // ---- phase 2: dQ = W K + c dq2 ; dK = W^T Q + e dk2 ; dV = P^T dO + e dv2 ; G <- c_L G + Qc^T dO
    {
      float dq1[2][4], dk1[2][4], dv1[2][4];
      zero4(dq1[0]); zero4(dq1[1]); zero4(dk1[0]); zero4(dk1[1]); zero4(dv1[0]); zero4(dv1[1]);
#pragma unroll
      for (int k0 = 0; k0 < RC_ROWS; k0 += 8) {
        {
          const FragB b = ldb(Ks, LDA, k0, 8 * warp, g, tq);
          mma3(dq1[0], lda_row(Ws, LDP, 0, k0, g, tq), b);
          mma3(dq1[1], lda_row(Ws, LDP, 16, k0, g, tq), b);
        }
        {
          const FragB b = ldb(Qs, LDA, k0, 8 * warp, g, tq);
          mma3(dk1[0], lda_tr(Ws, LDP, 0, k0, g, tq), b);
          mma3(dk1[1], lda_tr(Ws, LDP, 16, k0, g, tq), b);
        }
        {
          const FragB b = ldb(Ds, LDA, k0, 8 * warp, g, tq);
          mma3(dv1[0], lda_tr(Ps, LDPT, 0, k0, g, tq), b);
          mma3(dv1[1], lda_tr(Ps, LDPT, 16, k0, g, tq), b);
        }
      }
#pragma unroll
      for (int mi = 0; mi < 2; ++mi)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int row = 16 * mi + g + 8 * h;
          if (row < rows) {
            const int tl = tb.row_tl[row];
            const int cdt = tb.cds[tl];
            const float cc = (cdt == 0) ? tb.kpow[tl + 1] : 0.f;
            const float ee = (cdt == cd_last) ? tb.kpow[L - 1 - tl] : 0.f;
            const int64_t grow = ((int64_t)(t0 + tl) * N + n) * A + (row - tl * A);
            const int col = 8 * warp + 2 * tq;
            *reinterpret_cast<float2*>(dq + grow * ldd + col) =
                make_float2(dq1[mi][2 * h] + cc * dq2[mi][2 * h], dq1[mi][2 * h + 1] + cc * dq2[mi][2 * h + 1]);
            *reinterpret_cast<float2*>(dk + grow * ldd + col) =
                make_float2(dk1[mi][2 * h] + ee * dk2[mi][2 * h], dk1[mi][2 * h + 1] + ee * dk2[mi][2 * h + 1]);
            *reinterpret_cast<float2*>(dv + grow * ldd + col) =
                make_float2(dv1[mi][2 * h] + ee * dv2[mi][2 * h], dv1[mi][2 * h + 1] + ee * dv2[mi][2 * h + 1]);
          }
        }
    }
    {
      const float cL = (cd_last == 0) ? tb.kpow[L] : 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int x = 0; x < 4; ++x) Gacc[j][x] *= cL;
#pragma unroll
      for (int k0 = 0; k0 < RC_ROWS; k0 += 8) {
        const Frag a = lda_tr(Qc, LDB, 16 * mt, k0, g, tq);
#pragma unroll
        for (int j = 0; j < 4; ++j) mma3(Gacc[j], a, ldb(Ds, LDA, k0, 8 * (nt0 + j), g, tq));
      }
    }
    __syncthreads();  // C
  }
}

constexpr size_t kFwdSmem = (size_t)(64 * LDB + 2 * RC_ROWS * LDA + 2 * RC_ROWS * LDB + RC_ROWS * LDP + 40 + 32 + 8) * sizeof(float);
constexpr size_t kBwdSmem =
    (size_t)(3 * 64 * LDA + 4 * RC_ROWS * LDA + RC_ROWS * LDB + RC_ROWS * LDPT + RC_ROWS * LDP + 40 + 32 + 8) * sizeof(float);

template <typename Kern>
int set_smem(Kern kern, size_t bytes) {
  MAGPO_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return MAGPO_OK;
}

}  // namespace

int retention_chunk_len(int A) { return std::max(1, RC_ROWS / A); }
int retention_num_chunks(int T, int A) { return (T + retention_chunk_len(A) - 1) / retention_chunk_len(A); }

int retention_chunk_fwd(cudaStream_t s, int T, int N, int A, float kappa, bool causal, const float* q, const float* k,
                        const float* v, int ld, const float* H0, const uint8_t* done, float* ret, float* Hck, float* Hout) {
  const int Lc = retention_chunk_len(A);
  if (once_per_device(ONCE_RET_FWD)) {
    MAGPO_TRY(set_smem(retention_chunk_fwd_kernel<true>, kFwdSmem));
    MAGPO_TRY(set_smem(retention_chunk_fwd_kernel<false>, kFwdSmem));
  }
  ProfScope ps(PROF_RET_FWD, s, 4.0 * 256.0 * (double)T * N * A);
  if (causal)
    retention_chunk_fwd_kernel<true><<<N, 256, kFwdSmem, s>>>(T, N, A, Lc, kappa, q, k, v, ld, H0, done, ret, Hck, Hout);
  else
    retention_chunk_fwd_kernel<false><<<N, 256, kFwdSmem, s>>>(T, N, A, Lc, kappa, q, k, v, ld, H0, done, ret, Hck, Hout);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

int retention_chunk_bwd(cudaStream_t s, int T, int N, int A, float kappa, bool causal, const float* q, const float* k,
                        const float* v, int ld, const uint8_t* done, const float* Hck, const float* dret, float* dq,
                        float* dk, float* dv, int ldd) {
  const int Lc = retention_chunk_len(A);
  if (once_per_device(ONCE_RET_BWD)) {
    MAGPO_TRY(set_smem(retention_chunk_bwd_kernel<true>, kBwdSmem));
    MAGPO_TRY(set_smem(retention_chunk_bwd_kernel<false>, kBwdSmem));
  }
  ProfScope ps(PROF_RET_BWD, s, 7.0 * 256.0 * (double)T * N * A);
  if (causal)
    retention_chunk_bwd_kernel<true><<<N, 256, kBwdSmem, s>>>(T, N, A, Lc, kappa, q, k, v, ld, done, Hck, dret, dq, dk, dv, ldd);
  else
    retention_chunk_bwd_kernel<false><<<N, 256, kBwdSmem, s>>>(T, N, A, Lc, kappa, q, k, v, ld, done, Hck, dret, dq, dk, dv, ldd);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

}  // namespace magpo

// Host-only: timesteps per chunk the chunkwise kernels launch with for A agents (tests assert which chunk geometry a case covers).
extern "C" int magpo_debug_retention_chunk_len(int A) { return magpo::retention_chunk_len(A); }
