// Retention in its recurrent form, forward and backward, one CTA per env sequence.
// Reference: networks/retention.py:66-115 (SimpleRetention chunkwise + recurrent), :117-213 (decay matrix / xi).
// The chunkwise form the reference trains with, ret = ((Q K^T) * D) V + (Q h0) * xi, with
//   D[n,m] = kappa^(t(n)-t(m)) [t(n)>=t(m)] [no done in (t(m), t(n)]]   (block-full over agents for the
//   encoder, lower-triangular over tokens for the decoder),  xi[t] = kappa^(t+1) [t < first done],
// is algebraically the scan   H <- lam_t * H (lam_t = 0 if done_t else kappa);  H <- H + k_i^T v_i;  o_i = q_i H
// (encoder: all A tokens of the timestep are added before any output; decoder: token by token), which is
// also exactly what SableNetwork.get_actions runs at inference (sable_network.py:457, retention.py:102-115).
// The scan costs 2*64*64 MAC per token instead of 2*64*C and never materialises the [N,C,C] decay matrix.
// State layout: the 64x64 state lives in registers, a 4x4 block per thread (16x16 threads); sums over
// columns use 16-lane shuffles, sums over rows go through shared memory. The backward walks time in
// reverse with G = dL/dH in registers and re-reads the per-timestep states the forward saved
// (within a timestep the per-token states are recovered by exact rank-1 down-dates).
#include "common.cuh"
#include "kernels.cuh"

namespace magpo {
namespace {

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float half_warp_sum(float v) {
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <bool CAUSAL>
__global__ void __launch_bounds__(256)
retention_fwd_kernel(int T, int N, int A, float kappa, const float* __restrict__ q, const float* __restrict__ k,
                     const float* __restrict__ v, int ld, const float* __restrict__ H0,
                     const uint8_t* __restrict__ done, float* __restrict__ ret, float* __restrict__ Hsave,
                     float* __restrict__ Hout) {
  extern __shared__ __align__(16) float sm[];
  float* qs = sm;
  float* ks = qs + A * 64;
  float* vs = ks + A * 64;
  float* part = vs + A * 64;  // [A][16][64]
  const int n = blockIdx.x, tid = threadIdx.x;
  const int tr = tid >> 4, tc = tid & 15, r0 = tr * 4, c0 = tc * 4;
  float H[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
    if (H0) h = ld4(H0 + ((int64_t)n * 64 + r0 + a) * 64 + c0);
    H[a][0] = h.x; H[a][1] = h.y; H[a][2] = h.z; H[a][3] = h.w;
  }
  // software pipeline: the q,k,v rows of step t+1 are fetched into registers while step t is computed
  float pq[2], pk[2], pv[2];
  auto fetch = [&](int t) {
    const int64_t b0 = ((int64_t)t * N + n) * A;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int idx = tid + j * 256;
      if (idx < A * 64) {
        const int64_t off = (b0 + (idx >> 6)) * ld + (idx & 63);
        pq[j] = q[off]; pk[j] = k[off]; pv[j] = v[off];
      }
    }
  };
  fetch(0);
  for (int t = 0; t < T; ++t) {
    const float lam = (done && done[(int64_t)t * N + n]) ? 0.0f : kappa;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) H[a][b] *= lam;
    const int64_t base = ((int64_t)t * N + n) * A;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int idx = tid + j * 256;
      if (idx < A * 64) { qs[idx] = pq[j]; ks[idx] = pk[j]; vs[idx] = pv[j]; }
    }
    __syncthreads();
    if (t + 1 < T) fetch(t + 1);
    if (!CAUSAL) {
      for (int i = 0; i < A; ++i) {
        const float4 kr = ld4(ks + i * 64 + r0), vc = ld4(vs + i * 64 + c0);
        const float ka[4] = {kr.x, kr.y, kr.z, kr.w}, vb[4] = {vc.x, vc.y, vc.z, vc.w};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) H[a][b] = fmaf(ka[a], vb[b], H[a][b]);
      }
    }
    for (int i = 0; i < A; ++i) {
      if (CAUSAL) {
        const float4 kr = ld4(ks + i * 64 + r0), vc = ld4(vs + i * 64 + c0);
        const float ka[4] = {kr.x, kr.y, kr.z, kr.w}, vb[4] = {vc.x, vc.y, vc.z, vc.w};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) H[a][b] = fmaf(ka[a], vb[b], H[a][b]);
      }
      const float4 qr = ld4(qs + i * 64 + r0);
      const float qa[4] = {qr.x, qr.y, qr.z, qr.w};
      float p[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) p[b] = fmaf(qa[a], H[a][b], p[b]);
      st4(part + (i * 16 + tr) * 64 + c0, make_float4(p[0], p[1], p[2], p[3]));
    }
    __syncthreads();
    for (int idx = tid; idx < A * 64; idx += 256) {
      const int i = idx >> 6, c = idx & 63;
      float s = 0.f;
#pragma unroll
      for (int r = 0; r < 16; ++r) s += part[(i * 16 + r) * 64 + c];
      ret[(base + i) * 64 + c] = s;
    }
    if (Hsave) {
#pragma unroll
      for (int a = 0; a < 4; ++a)
        st4(Hsave + (((int64_t)t * N + n) * 64 + r0 + a) * 64 + c0, make_float4(H[a][0], H[a][1], H[a][2], H[a][3]));
    }
    __syncthreads();
  }
  if (Hout) {
#pragma unroll
    for (int a = 0; a < 4; ++a)
      st4(Hout + ((int64_t)n * 64 + r0 + a) * 64 + c0, make_float4(H[a][0], H[a][1], H[a][2], H[a][3]));
  }
}

template <bool CAUSAL>
__global__ void __launch_bounds__(256)
retention_bwd_kernel(int T, int N, int A, float kappa, const float* __restrict__ q, const float* __restrict__ k,
                     const float* __restrict__ v, int ld, const uint8_t* __restrict__ done,
                     const float* __restrict__ Hsave, const float* __restrict__ dret, float* __restrict__ dq,
                     float* __restrict__ dk, float* __restrict__ dv, int ldd) {
  extern __shared__ __align__(16) float sm[];
  float* qs = sm;
  float* ks = qs + A * 64;
  float* vs = ks + A * 64;
  float* ds = vs + A * 64;
  float* part = ds + A * 64;  // [A][16][64]
  const int n = blockIdx.x, tid = threadIdx.x;
  const int tr = tid >> 4, tc = tid & 15, r0 = tr * 4, c0 = tc * 4;
  float G[4][4], H[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) G[a][b] = 0.f;
  // software pipeline: rows and the saved state of step t-1 are fetched while step t is processed
  float pq[2], pk[2], pv[2], pd[2];
  float4 ph[4];
  auto fetch = [&](int t) {
    const int64_t b0 = ((int64_t)t * N + n) * A;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int idx = tid + j * 256;
      if (idx < A * 64) {
        const int64_t row = b0 + (idx >> 6);
        const int c = idx & 63;
        pq[j] = q[row * ld + c]; pk[j] = k[row * ld + c]; pv[j] = v[row * ld + c]; pd[j] = dret[row * 64 + c];
      }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) ph[a] = ld4(Hsave + (((int64_t)t * N + n) * 64 + r0 + a) * 64 + c0);
  };
  fetch(T - 1);
  for (int t = T - 1; t >= 0; --t) {
    const int64_t base = ((int64_t)t * N + n) * A;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int idx = tid + j * 256;
      if (idx < A * 64) { qs[idx] = pq[j]; ks[idx] = pk[j]; vs[idx] = pv[j]; ds[idx] = pd[j]; }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) { H[a][0] = ph[a].x; H[a][1] = ph[a].y; H[a][2] = ph[a].z; H[a][3] = ph[a].w; }
    __syncthreads();
    if (t > 0) fetch(t - 1);
    if (!CAUSAL) {
      for (int i = 0; i < A; ++i) {
        const float4 qr = ld4(qs + i * 64 + r0), dc = ld4(ds + i * 64 + c0);
        const float qa[4] = {qr.x, qr.y, qr.z, qr.w}, db[4] = {dc.x, dc.y, dc.z, dc.w};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) G[a][b] = fmaf(qa[a], db[b], G[a][b]);
      }
    }
    for (int ii = 0; ii < A; ++ii) {
      const int i = CAUSAL ? (A - 1 - ii) : ii;
      const float4 dc = ld4(ds + i * 64 + c0), vc = ld4(vs + i * 64 + c0), kr = ld4(ks + i * 64 + r0);
      const float db[4] = {dc.x, dc.y, dc.z, dc.w}, vb[4] = {vc.x, vc.y, vc.z, vc.w}, ka[4] = {kr.x, kr.y, kr.z, kr.w};
      if (CAUSAL) {
        const float4 qr = ld4(qs + i * 64 + r0);
        const float qa[4] = {qr.x, qr.y, qr.z, qr.w};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) G[a][b] = fmaf(qa[a], db[b], G[a][b]);
      }
      float dqp[4], dkp[4], dvp[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        float sq = 0.f, sk = 0.f;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          sq = fmaf(db[b], H[a][b], sq);
          sk = fmaf(G[a][b], vb[b], sk);
          dvp[b] = fmaf(ka[a], G[a][b], dvp[b]);
        }
        dqp[a] = half_warp_sum(sq);
        dkp[a] = half_warp_sum(sk);
      }
      if (tc == 0) {
        st4(dq + (base + i) * ldd + r0, make_float4(dqp[0], dqp[1], dqp[2], dqp[3]));
        st4(dk + (base + i) * ldd + r0, make_float4(dkp[0], dkp[1], dkp[2], dkp[3]));
      }
      st4(part + (i * 16 + tr) * 64 + c0, make_float4(dvp[0], dvp[1], dvp[2], dvp[3]));
      if (CAUSAL) {
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) H[a][b] = fmaf(-ka[a], vb[b], H[a][b]);
      }
    }
    __syncthreads();
    for (int idx = tid; idx < A * 64; idx += 256) {
      const int i = idx >> 6, c = idx & 63;
      float s = 0.f;
#pragma unroll
      for (int r = 0; r < 16; ++r) s += part[(i * 16 + r) * 64 + c];
      dv[(base + i) * ldd + c] = s;
    }
    const float lam = (done && done[(int64_t)t * N + n]) ? 0.0f : kappa;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) G[a][b] *= lam;
    __syncthreads();
  }
}

template <typename Kern>
int set_smem(Kern kern, size_t bytes) {
  if (bytes > 48 * 1024) MAGPO_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return MAGPO_OK;
}

}  // namespace

// retention_chunk.cu
int retention_chunk_fwd(cudaStream_t s, int T, int N, int A, float kappa, bool causal, const float* q, const float* k,
                        const float* v, int ld, const float* H0, const uint8_t* done, float* ret, float* Hck, float* Hout);
int retention_chunk_bwd(cudaStream_t s, int T, int N, int A, float kappa, bool causal, const float* q, const float* k,
                        const float* v, int ld, const uint8_t* done, const float* Hck, const float* dret, float* dq,
                        float* dk, float* dv, int ldd);

int retention_fwd(cudaStream_t s, int T, int N, int A, float kappa, bool causal, const float* q, const float* k,
                  const float* v, int ld, const float* H0, const uint8_t* done, float* ret, float* Hsave,
                  float* Hout) {
  if (T <= 0 || N <= 0) return MAGPO_OK;
  if (A < 1 || A > kMaxAgents || (ld & 3)) return MAGPO_ERR_UNSUPPORTED;
  // sequences (the update) run chunkwise on the tensor cores; a single step (the rollout) keeps the register scan
  if (T > 1) return retention_chunk_fwd(s, T, N, A, kappa, causal, q, k, v, ld, H0, done, ret, Hsave, Hout);
  const size_t smem = (size_t)(3 * A * 64 + A * 16 * 64) * sizeof(float);
  ProfScope ps(PROF_RET_FWD, s, 4.0 * 4096.0 * (double)T * N * A);
  if (causal) {
    MAGPO_TRY(set_smem(retention_fwd_kernel<true>, smem));
    retention_fwd_kernel<true><<<N, 256, smem, s>>>(T, N, A, kappa, q, k, v, ld, H0, done, ret, Hsave, Hout);
  } else {
    MAGPO_TRY(set_smem(retention_fwd_kernel<false>, smem));
    retention_fwd_kernel<false><<<N, 256, smem, s>>>(T, N, A, kappa, q, k, v, ld, H0, done, ret, Hsave, Hout);
  }
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

int retention_bwd(cudaStream_t s, int T, int N, int A, float kappa, bool causal, const float* q, const float* k,
                  const float* v, int ld, const float* H0, const uint8_t* done, const float* Hsave,
                  const float* dret, float* dq, float* dk, float* dv, int ldd) {
  (void)H0;
  if (T <= 0 || N <= 0) return MAGPO_OK;
  if (A < 1 || A > kMaxAgents || (ld & 3) || (ldd & 3)) return MAGPO_ERR_UNSUPPORTED;
  if (T > 1) return retention_chunk_bwd(s, T, N, A, kappa, causal, q, k, v, ld, done, Hsave, dret, dq, dk, dv, ldd);
  const size_t smem = (size_t)(4 * A * 64 + A * 16 * 64) * sizeof(float);
  ProfScope ps(PROF_RET_BWD, s, 10.0 * 4096.0 * (double)T * N * A);
  if (causal) {
    MAGPO_TRY(set_smem(retention_bwd_kernel<true>, smem));
    retention_bwd_kernel<true><<<N, 256, smem, s>>>(T, N, A, kappa, q, k, v, ld, done, Hsave, dret, dq, dk, dv, ldd);
  } else {
    MAGPO_TRY(set_smem(retention_bwd_kernel<false>, smem));
    retention_bwd_kernel<false><<<N, 256, smem, s>>>(T, N, A, kappa, q, k, v, ld, done, Hsave, dret, dq, dk, dv, ldd);
  }
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

}  // namespace magpo

using namespace magpo;

// Test hook: retention forward/backward on caller buffers (q,k,v packed with row stride ld).
extern "C" int magpo_test_retention(magpo_stream_t s, int bwd, int T, int N, int A, float kappa, int causal,
                                    const float* q, const float* k, const float* v, int ld, const float* H0,
                                    const uint8_t* done, float* ret, float* Hsave, float* Hout, const float* dret,
                                    float* dq, float* dk, float* dv, int ldd) {
  if (!bwd) return retention_fwd(as_stream(s), T, N, A, kappa, causal != 0, q, k, v, ld, H0, done, ret, Hsave, Hout);
  return retention_bwd(as_stream(s), T, N, A, kappa, causal != 0, q, k, v, ld, H0, done, Hsave, dret, dq, dk, dv, ldd);
}
