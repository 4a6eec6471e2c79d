// Learner policy: RecurrentActor = MLPTorso -> ScannedRNN(GRUCell, reset on done) -> MLPTorso -> DiscreteActionHead.
// Reference: networks/base.py:121-184, networks/torsos.py:24-47, networks/heads.py:26-63, flax 0.10.3 GRUCell
// (SURVEY.md Appendix A8); backward per Appendix G (BPTT).  The input-side GEMMs are batched over all T
// timesteps; only h @ [W_hr|W_hz|W_hn] (and its transpose in the backward) is sequential in T.
#include "actor.cuh"

namespace magpo {
namespace {

// One thread per (row, j): gates of flax GRUCell. gi = x@Wi + bi [rows,384], gh = hu@Wh [rows,384].
__global__ void __launch_bounds__(256)
gru_gate_fwd_kernel(int64_t rows, int A, const float* __restrict__ gi, const float* __restrict__ gh,
                    const float* __restrict__ bhn, const float* __restrict__ hu, const uint8_t* __restrict__ done_next,
                    float* __restrict__ rzn, float* __restrict__ ghn_out, float* __restrict__ y,
                    float* __restrict__ hu_next, const uint8_t* __restrict__ done_cur) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * kH) return;
  const int64_t row = idx / kH;
  const int j = (int)(idx % kH);
  const float* gir = gi + row * 3 * kH;
  const float* ghr = gh + row * 3 * kH;
  // done_cur: `hu` / `gh` come from the un-masked carry; a row mask commutes with the right-multiplication by W_h, so
  // resetting the carry (base.py:136-139) is zeroing the row's gh and h here
  const float keep = (done_cur && done_cur[row / A]) ? 0.0f : 1.0f;
  const float r = sigmoid_precise(gir[j] + keep * ghr[j]);
  const float z = sigmoid_precise(gir[kH + j] + keep * ghr[kH + j]);
  const float ghn = keep * ghr[2 * kH + j] + bhn[j];
  const float n = tanhf(gir[2 * kH + j] + r * ghn);
  const float hprev = keep * hu[idx];
  const float h = (1.0f - z) * n + z * hprev;
  if (rzn) {
    float* o = rzn + row * 3 * kH;
    o[j] = r; o[kH + j] = z; o[2 * kH + j] = n;
  }
  if (ghn_out) ghn_out[idx] = ghn;
  if (y) y[idx] = h;
  if (hu_next) hu_next[idx] = (done_next && done_next[row / A]) ? 0.0f : h;
}

// dh = dy + (done_next ? 0 : carry); writes dGI = [da_r, da_z, da_n], dGH = [da_r, da_z, da_n * r], carry_out = dh * z
__global__ void __launch_bounds__(256)
gru_gate_bwd_kernel(int64_t rows, int A, const float* __restrict__ dy, const float* __restrict__ carry,
                    const uint8_t* __restrict__ done_next, const float* __restrict__ rzn,
                    const float* __restrict__ ghn, const float* __restrict__ hu, float* __restrict__ dgi,
                    float* __restrict__ dgh, float* __restrict__ carry_out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * kH) return;
  const int64_t row = idx / kH;
  const int j = (int)(idx % kH);
  float dh = dy[idx];
  if (carry && !(done_next && done_next[row / A])) dh += carry[idx];
  const float* g = rzn + row * 3 * kH;
  const float r = g[j], z = g[kH + j], n = g[2 * kH + j];
  const float dn = dh * (1.0f - z);
  const float dz = dh * (hu[idx] - n);
  const float dan = dn * (1.0f - n * n);
  const float daz = dz * z * (1.0f - z);
  const float dr = dan * ghn[idx];
  const float dar = dr * r * (1.0f - r);
  float* o1 = dgi + row * 3 * kH;
  float* o2 = dgh + row * 3 * kH;
  o1[j] = dar; o1[kH + j] = daz; o1[2 * kH + j] = dan;
  o2[j] = dar; o2[kH + j] = daz; o2[2 * kH + j] = dan * r;
  carry_out[idx] = dh * z;
}

__global__ void __launch_bounds__(256)
mask_rows_kernel(int64_t rows, int A, const float* __restrict__ h, const uint8_t* __restrict__ done,
                 float* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * kH) return;
  out[idx] = (done && done[(idx / kH) / A]) ? 0.0f : h[idx];
}

__global__ void __launch_bounds__(256)
relu_bwd_kernel(int64_t n, const float* __restrict__ act, float* __restrict__ d) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < n && !(act[idx] > 0.0f)) d[idx] = 0.0f;
}

inline unsigned g256(int64_t n) { return (unsigned)ceil_div(n, 256); }

}  // namespace

void ActorT::plan(Arena& ar, int a) {
  WiT = ar.get<float>(3 * kH * kH);
  WhT = ar.get<float>(3 * kH * kH);
  postT = ar.get<float>(kH * kH);
  headT = ar.get<float>((size_t)a * kH);
  region_n = (int64_t)(reinterpret_cast<uintptr_t>(headT) + (size_t)a * kH * sizeof(float) - reinterpret_cast<uintptr_t>(WiT)) / 4;
  region_hi = ar.get<float>((size_t)region_n);
  region_lo = ar.get<float>((size_t)region_n);
}

int actor_transpose(cudaStream_t s, const ActorP& p, const ActorT& t, int a) {
  MAGPO_TRY(transpose(s, kH, 3 * kH, p.Wi, t.WiT));
  MAGPO_TRY(transpose(s, kH, 3 * kH, p.Wh, t.WhT));
  MAGPO_TRY(transpose(s, kH, kH, p.post_w, t.postT));
  MAGPO_TRY(transpose(s, kH, a, p.head_w, t.headT));
  MAGPO_TRY(tc_prepare_region(s, t.WiT, t.region_n, t.region_hi, t.region_lo));
  return MAGPO_OK;
}

void ActorActs::plan(Arena& ar, int64_t R, int64_t Rs, int a, bool with_backward) {
  const size_t rH = (size_t)R * kH;
  e = ar.get<float>(rH);
  gi = ar.get<float>(3 * rH);
  gh = ar.get<float>((size_t)Rs * 3 * kH);
  HU = ar.get<float>(rH + (size_t)Rs * kH);  // one extra step: hu_next of the last timestep
  Y = ar.get<float>(rH);
  post = ar.get<float>(rH);
  if (with_backward) {
    rzn = ar.get<float>(3 * rH);
    ghn = ar.get<float>(rH);
    dgh = ar.get<float>(3 * rH);
    dA = ar.get<float>(rH);
    dB = ar.get<float>(rH);
    carry = ar.get<float>((size_t)Rs * kH);
  } else {
    rzn = ghn = dgh = dA = dB = carry = nullptr;
  }
}

// RecurrentActor.apply over T steps (base.py:161-184): masked=false raw logits [T*Rs, a].
int actor_forward(cudaStream_t s, const ActorP& p, const ActorT* pt, int T, int N, int A, int d, int a, const float* agents_view,
                  const uint8_t* done, const float* h0, const ActorActs& w, float* logits, float* h_out) {
  const int64_t Rs = (int64_t)N * A, R = Rs * T;
  if (thin_k_ok(d, kH, kH, p.pre_w, w.e, kH)) MAGPO_TRY(thin_k_fwd(s, R, d, kH, agents_view, d, p.pre_w, kH, p.pre_b, w.e, kH, 1));
  else MAGPO_TRY(gemm_nn(s, R, kH, d, agents_view, d, wref(p.pre_w, kH), p.pre_b, w.e, kH, GEMM_RELU));
  MAGPO_TRY(gemm_nn(s, R, 3 * kH, kH, w.e, kH, wref(p.Wi, 3 * kH, pt ? pt->WiT : nullptr, kH), p.bi, w.gi, 3 * kH, 0));
  // inference (no backward buffers, T = 1: the rollout's state push): the reset mask is applied inside the gate kernel
  const bool mask_in_gate = !w.rzn && T == 1;
  if (!mask_in_gate) {
    mask_rows_kernel<<<g256(Rs * kH), 256, 0, s>>>(Rs, A, h0, done, w.HU);
    MAGPO_LAUNCH_OK();
  }
  const float *wh_hi = nullptr, *wh_lo = nullptr;
  const bool scan = T > 1 && w.rzn && pt && tc_lookup(pt->WhT, &wh_hi, &wh_lo);
  if (scan) MAGPO_TRY(gru_scan_fwd(s, T, N, A, w.gi, wh_hi, wh_lo, p.bhn, done, w.rzn, w.ghn, w.Y, w.HU));
  for (int t = 0; t < T && !scan; ++t) {
    const float* hu = mask_in_gate ? h0 : w.HU + (size_t)t * Rs * kH;
    MAGPO_TRY(gemm_nn(s, Rs, 3 * kH, kH, hu, kH, wref(p.Wh, 3 * kH, pt ? pt->WhT : nullptr, kH), nullptr, w.gh, 3 * kH, 0));
    const uint8_t* dn = (t + 1 < T) ? done + (size_t)(t + 1) * N : nullptr;
    ProfScope ps(PROF_GRU, s, 4.0 * kH * 13 * (double)Rs);
    gru_gate_fwd_kernel<<<g256(Rs * kH), 256, 0, s>>>(
        Rs, A, w.gi + (size_t)t * Rs * 3 * kH, w.gh, p.bhn, hu, dn, w.rzn ? w.rzn + (size_t)t * Rs * 3 * kH : nullptr,
        w.ghn ? w.ghn + (size_t)t * Rs * kH : nullptr, w.Y + (size_t)t * Rs * kH, w.HU + (size_t)(t + 1) * Rs * kH,
        mask_in_gate ? done : nullptr);
    MAGPO_LAUNCH_OK();
  }
  if (h_out) MAGPO_CUDA_OK(cudaMemcpyAsync(h_out, w.Y + (size_t)(T - 1) * Rs * kH, (size_t)Rs * kH * sizeof(float),
                                           cudaMemcpyDeviceToDevice, s));
  if (logits) {
    MAGPO_TRY(gemm_nn(s, R, kH, kH, w.Y, kH, wref(p.post_w, kH, pt ? pt->postT : nullptr, kH), p.post_b, w.post, kH, GEMM_RELU));
    if (thin_n_ok(kH, a, w.post, kH)) MAGPO_TRY(thin_n_fwd(s, R, kH, a, w.post, kH, p.head_w, a, p.head_b, logits, a));
    else MAGPO_TRY(gemm_nn(s, R, a, kH, w.post, kH, wref(p.head_w, a), p.head_b, logits, a, 0));
  }
  return MAGPO_OK;
}

// BPTT given dL/dlogits [R,a]; grads accumulate into g. agents_view is data (no input gradient).
int actor_backward(cudaStream_t s, const ActorP& p, const ActorT& pt, int T, int N, int A, int d, int a,
                   const float* agents_view, const uint8_t* done, const ActorActs& w, const float* dlogits,
                   const ActorP& g) {
  const int64_t Rs = (int64_t)N * A, R = Rs * T;
  // head + post torso
  if (thin_n_ok(kH, a, w.post, kH)) {  // dW, db, dX and the relu mask of the post torso in one pass
    MAGPO_TRY(thin_n_bwd(s, R, kH, a, w.post, kH, dlogits, a, p.head_w, a, 1, w.dA, kH, g.head_w, a, g.head_b, g.post_b));
  } else {
    MAGPO_TRY(gemm_tn(s, R, a, kH, w.post, kH, dlogits, a, g.head_w, a));
    MAGPO_TRY(colsum(s, R, a, dlogits, a, g.head_b));
    MAGPO_TRY(gemm_nn(s, R, kH, a, dlogits, a, wref(pt.headT, kH), nullptr, w.dA, kH, 0));
    relu_bwd_kernel<<<g256(R * kH), 256, 0, s>>>(R * kH, w.post, w.dA);
    MAGPO_LAUNCH_OK();
    MAGPO_TRY(colsum(s, R, kH, w.dA, kH, g.post_b));
  }
  MAGPO_TRY(gemm_tn(s, R, kH, kH, w.Y, kH, w.dA, kH, g.post_w, kH));
  MAGPO_TRY(gemm_nn(s, R, kH, kH, w.dA, kH, wref(pt.postT, kH, p.post_w, kH), nullptr, w.dB, kH, 0));  // dB = dL/dY
  // reverse scan; dgi reuses the gi buffer (dead after the forward)
  float* dgi = w.gi;
  const float *wh_hi = nullptr, *wh_lo = nullptr;
  const bool scan = T > 1 && tc_lookup(p.Wh, &wh_hi, &wh_lo);
  if (scan) MAGPO_TRY(gru_scan_bwd(s, T, N, A, w.dB, w.rzn, w.ghn, w.HU, done, wh_hi, wh_lo, dgi, w.dgh, g.bi, g.bhn));  // bias sums inside
  for (int t = T - 1; t >= 0 && !scan; --t) {
    const size_t o1 = (size_t)t * Rs * kH, o3 = (size_t)t * Rs * 3 * kH;
    const bool last = (t == T - 1);
    {
    ProfScope ps(PROF_GRU, s, 4.0 * kH * 14 * (double)Rs);
    gru_gate_bwd_kernel<<<g256(Rs * kH), 256, 0, s>>>(Rs, A, w.dB + o1, last ? nullptr : w.carry,
                                                      last ? nullptr : done + (size_t)(t + 1) * N, w.rzn + o3,
                                                      w.ghn + o1, w.HU + o1, dgi + o3, w.dgh + o3, w.carry);
    }
    MAGPO_LAUNCH_OK();
    if (t > 0)  // carry += dGH @ Wh^T  (gradient w.r.t. hu_t; masked by done_t when consumed at t-1)
      MAGPO_TRY(gemm_nn(s, Rs, kH, 3 * kH, w.dgh + o3, 3 * kH, wref(pt.WhT, kH, p.Wh, 3 * kH), nullptr, w.carry, kH, GEMM_ACCUMULATE));
  }
  MAGPO_TRY(gemm_tn(s, R, 3 * kH, kH, w.HU, kH, w.dgh, 3 * kH, g.Wh, 3 * kH));
  if (!scan) MAGPO_TRY(colsum(s, R, kH, w.dgh + 2 * kH, 3 * kH, g.bhn));
  MAGPO_TRY(gemm_tn(s, R, 3 * kH, kH, w.e, kH, dgi, 3 * kH, g.Wi, 3 * kH));
  if (!scan) MAGPO_TRY(colsum(s, R, 3 * kH, dgi, 3 * kH, g.bi));
  MAGPO_TRY(gemm_nn(s, R, kH, 3 * kH, dgi, 3 * kH, wref(pt.WiT, kH, p.Wi, 3 * kH), nullptr, w.dA, kH, 0));  // dA = dL/de (pre-relu mask next)
  if (thin_k_ok(d, kH, kH, w.dA, w.dA, kH)) {  // relu mask of the pre torso applied on the fly
    MAGPO_TRY(thin_k_bwd(s, R, d, kH, agents_view, d, w.dA, kH, w.e, g.pre_w, kH, g.pre_b));
  } else {
    relu_bwd_kernel<<<g256(R * kH), 256, 0, s>>>(R * kH, w.e, w.dA);
    MAGPO_LAUNCH_OK();
    MAGPO_TRY(gemm_tn(s, R, kH, d, agents_view, d, w.dA, kH, g.pre_w, kH));
    MAGPO_TRY(colsum(s, R, kH, w.dA, kH, g.pre_b));
  }
  return MAGPO_OK;
}

}  // namespace magpo

// Test hook: the persistent GRU scans on caller buffers, set up as actor_forward / actor_backward set them up.
//   gi [T, Rs, 384] (x @ Wi + bi), Wh [128, 384], bhn [128], done [T, N], h0 [Rs, 128], dY [T, Rs, 128]; Rs = N * A.
//   scratch: 3 * 128 * 384 floats (W_h^T and the TF32 hi / lo images).
//   bwd == 0: HU[0] = h0 masked by done[0], then rzn [T, Rs, 384], ghn / Y [T, Rs, 128], HU [T+1, Rs, 128].
//   bwd != 0: from the forward's rzn / ghn / HU: dgi, dgh [T, Rs, 384]; dbi [384] and dbhn [128] are accumulated into.
// There is no stepwise fallback here: MAGPO_ERR_UNSUPPORTED when T < 2.
extern "C" int magpo_test_gru_scan(magpo_stream_t s_, int bwd, int T, int N, int A, const float* gi, const float* Wh,
                                   const float* bhn, const uint8_t* done, const float* h0, const float* dY, float* scratch,
                                   float* rzn, float* ghn, float* Y, float* HU, float* dgi, float* dgh, float* dbi, float* dbhn) {
  using namespace magpo;
  if (T < 2) return MAGPO_ERR_UNSUPPORTED;
  if (N < 1 || A < 1 || !gi || !Wh || !done || !scratch || !rzn || !ghn || !HU) return MAGPO_ERR_ARG;
  cudaStream_t s = as_stream(s_);
  const int64_t Rs = (int64_t)N * A, n = 3 * kH * kH;
  float *hi = scratch + n, *lo = scratch + 2 * n;
  if (!bwd) {
    if (!bhn || !h0 || !Y) return MAGPO_ERR_ARG;
    mask_rows_kernel<<<g256(Rs * kH), 256, 0, s>>>(Rs, A, h0, done, HU);
    MAGPO_LAUNCH_OK();
    MAGPO_TRY(transpose(s, kH, 3 * kH, Wh, scratch));
    MAGPO_TRY(tc_prepare_region(s, scratch, n, hi, lo));
    return gru_scan_fwd(s, T, N, A, gi, hi, lo, bhn, done, rzn, ghn, Y, HU);
  }
  if (!dY || !dgi || !dgh) return MAGPO_ERR_ARG;
  MAGPO_TRY(tc_prepare_region(s, Wh, n, hi, lo));
  return gru_scan_bwd(s, T, N, A, dY, rzn, ghn, HU, done, hi, lo, dgi, dgh, dbi, dbhn);
}
