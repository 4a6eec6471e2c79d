// Sable guider sequencers: training forward + hand-derived backward, and the building blocks the
// rollout uses for SableNetwork.get_actions.  Reference: networks/sable_network.py:40-482,
// networks/utils/sable/{encode,decode}.py, networks/retention.py:265-323.  Backward: SURVEY.md Appendix G.
#include <stdlib.h>

#include "sable.cuh"
#include "update.cuh"

namespace magpo {

void GuiderT::plan(Arena& ar, int d) {
  WobsT = ar.get<float>((size_t)kD * d);
  qkvgT = ar.get<float>(4 * kD * kD);
  woT = ar.get<float>(kD * kD);
  ffn_glT = ar.get<float>(2 * kD * kD);
  ffn_outT = ar.get<float>(kD * kD);
  h0T = ar.get<float>(kD * kD);
  qkvg1T = ar.get<float>(4 * kD * kD);
  wo1T = ar.get<float>(kD * kD);
  qkvg2T = ar.get<float>(4 * kD * kD);
  wo2T = ar.get<float>(kD * kD);
  dffn_glT = ar.get<float>(2 * kD * kD);
  dffn_outT = ar.get<float>(kD * kD);
  dh0T = ar.get<float>(kD * kD);
  // TF32 hi/lo images of the whole transposed-weight region (tensor-core B operands); integer arithmetic because the
  // arena is also planned with a null base when sizing the workspace
  region_n = (int64_t)(reinterpret_cast<uintptr_t>(dh0T) + kD * kD * sizeof(float) - reinterpret_cast<uintptr_t>(WobsT)) / 4;
  region_hi = ar.get<float>((size_t)region_n);
  region_lo = ar.get<float>((size_t)region_n);
}

int guider_transpose(cudaStream_t s, const GuiderP& p, const GuiderT& t, int d) {
  MAGPO_TRY(transpose(s, d, kD, p.Wobs, t.WobsT));
  MAGPO_TRY(transpose(s, kD, 4 * kD, p.qkvg, t.qkvgT));
  MAGPO_TRY(transpose(s, kD, kD, p.wo, t.woT));
  MAGPO_TRY(transpose(s, kD, 2 * kD, p.ffn_gl, t.ffn_glT));
  MAGPO_TRY(transpose(s, kD, kD, p.ffn_out, t.ffn_outT));
  MAGPO_TRY(transpose(s, kD, kD, p.h0_w, t.h0T));
  MAGPO_TRY(transpose(s, kD, 4 * kD, p.qkvg1, t.qkvg1T));
  MAGPO_TRY(transpose(s, kD, kD, p.wo1, t.wo1T));
  MAGPO_TRY(transpose(s, kD, 4 * kD, p.qkvg2, t.qkvg2T));
  MAGPO_TRY(transpose(s, kD, kD, p.wo2, t.wo2T));
  MAGPO_TRY(transpose(s, kD, 2 * kD, p.dffn_gl, t.dffn_glT));
  MAGPO_TRY(transpose(s, kD, kD, p.dffn_out, t.dffn_outT));
  MAGPO_TRY(transpose(s, kD, kD, p.dh0_w, t.dh0T));
  MAGPO_TRY(tc_prepare_region(s, t.WobsT, t.region_n, t.region_hi, t.region_lo));
  return MAGPO_OK;
}

void SableActs::plan(Arena& ar, int64_t R, int64_t TN, int d, bool with_backward) {
  const size_t r64 = (size_t)R * kD;
  on = ar.get<float>((size_t)R * d);
  z0 = ar.get<float>(r64); xin = ar.get<float>(r64); kqv = ar.get<float>(r64);
  qkvg = ar.get<float>(4 * r64); ret = ar.get<float>(r64); gated = ar.get<float>(r64); o = ar.get<float>(r64);
  x1 = ar.get<float>(r64); gl = ar.get<float>(2 * r64); hmid = ar.get<float>(r64); f = ar.get<float>(r64);
  x = ar.get<float>(r64); xpe = ar.get<float>(r64); zh = ar.get<float>(r64);
  xD = ar.get<float>(r64); xpeD = ar.get<float>(r64); qkvg1 = ar.get<float>(4 * r64); ret1 = ar.get<float>(r64);
  gated1 = ar.get<float>(r64); o1 = ar.get<float>(r64); rpe = ar.get<float>(r64); qkvg2 = ar.get<float>(4 * r64);
  ret2 = ar.get<float>(r64); gated2 = ar.get<float>(r64); o2 = ar.get<float>(r64); y = ar.get<float>(r64);
  glD = ar.get<float>(2 * r64); hmidD = ar.get<float>(r64); fD = ar.get<float>(r64); xd = ar.get<float>(r64);
  zhD = ar.get<float>(r64);
  if (with_backward) {
    const size_t hs = (size_t)TN * kD * kD;
    Hs_enc = ar.get<float>(hs); Hs_self = ar.get<float>(hs); Hs_cross = ar.get<float>(hs);
    tA = ar.get<float>(r64); tB = ar.get<float>(r64); tC = ar.get<float>(r64); tD = ar.get<float>(r64);
    tE = ar.get<float>(r64); tQ = ar.get<float>(4 * r64); tG = ar.get<float>(2 * r64);
    t_d = ar.get<float>((size_t)R * d);
  } else {
    Hs_enc = Hs_self = Hs_cross = nullptr;
    tA = tB = tC = tD = tE = tQ = tG = t_d = nullptr;
  }
}

// ----------------------------------------------------------------------------- forward pieces
// Encoder over R = T*N*A rows (Encoder.__call__/recurrent, sable_network.py:121-156).
int sable_encoder_forward(cudaStream_t s, const GuiderP& p, const GuiderT* pt, int T, int N, int A, int d, int max_step,
                          const float* agents_view, const int32_t* step, const uint8_t* done, const float* H0,
                          float kappa, const float* pe, const SableActs& w, float* value, float* Hsave, float* Hout, bool chain, float* dec_q) {
  const int64_t R = (int64_t)T * N * A;
  const bool chained = chain && pt && chain_supported(R);
  if (chained && obs_embed_ok(d)) {
    MAGPO_TRY(chain_front_fwd(s, R, d, agents_view, p.obs_scale, p.Wobs, A, 0, nullptr, nullptr, p.ln, pe, step, max_step, pt->qkvgT, w.z0,
                              w.xin, w.kqv, w.qkvg));
  } else if (obs_embed_ok(d)) {
    MAGPO_TRY(obs_embed_fwd(s, R, d, agents_view, p.obs_scale, p.Wobs, p.ln, pe, step, max_step, w.on, w.z0, w.xin, w.kqv));
  } else {
    MAGPO_TRY(rms_general_fwd(s, R, d, agents_view, p.obs_scale, w.on));
    MAGPO_TRY(gemm_nn(s, R, kD, d, w.on, d, wref(p.Wobs, kD), nullptr, w.z0, kD, 0));
    MAGPO_TRY(act_rms_fwd(s, R, w.z0, nullptr, p.ln, ROW_GELU, pe, step, max_step, w.xin, w.kqv));
  }
  if (!(chained && obs_embed_ok(d)))
    MAGPO_TRY(gemm_nn(s, R, 4 * kD, kD, w.kqv, kD, wref(p.qkvg, 4 * kD, pt ? pt->qkvgT : nullptr, kD), nullptr, w.qkvg, 4 * kD, 0));
  MAGPO_TRY(retention_fwd(s, T, N, A, kappa, false, w.qkvg, w.qkvg + kD, w.qkvg + 2 * kD, 4 * kD, H0, done, w.ret,
                          Hsave, Hout));
  if (chained) {
    // the two row chains after the retention, one persistent kernel each (chain_fwd.cu); dec_q: the decoder's cross-retention query
    MAGPO_TRY(chain_gate_fwd(s, R, w.qkvg + 3 * kD, 4 * kD, w.ret, w.xin, p.gn_s, p.gn_b, p.ln1, nullptr, nullptr, 0, pt->woT, pt->ffn_glT,
                             nullptr, w.gated, w.o, w.x1, nullptr, w.gl, w.hmid, nullptr, 0));
    MAGPO_TRY(chain_tail_fwd(s, R, w.hmid, w.x1, p.ln2, pe, step, max_step, pt->ffn_outT, dec_q ? pt->qkvg2T : nullptr, kD, pt->h0T, p.h0_b,
                             p.h2_s, p.h3_w, p.h3_b, 1, w.f, w.x, w.xpe, dec_q, 4 * kD, w.zh, value));
    return MAGPO_OK;
  }
  if (dec_q) return MAGPO_ERR_ARG;
  MAGPO_TRY(gn_gate_fwd(s, R, w.qkvg + 3 * kD, 4 * kD, w.ret, p.gn_s, p.gn_b, w.gated));
  MAGPO_TRY(gemm_nn(s, R, kD, kD, w.gated, kD, wref(p.wo, kD, pt ? pt->woT : nullptr, kD), nullptr, w.o, kD, 0));
  MAGPO_TRY(act_rms_fwd(s, R, w.o, w.xin, p.ln1, 0, nullptr, nullptr, 0, w.x1, nullptr));
  MAGPO_TRY(gemm_nn(s, R, 2 * kD, kD, w.x1, kD, wref(p.ffn_gl, 2 * kD, pt ? pt->ffn_glT : nullptr, kD), nullptr, w.gl, 2 * kD, 0));
  MAGPO_TRY(swiglu_fwd(s, R, w.gl, w.hmid));
  MAGPO_TRY(gemm_nn(s, R, kD, kD, w.hmid, kD, wref(p.ffn_out, kD, pt ? pt->ffn_outT : nullptr, kD), nullptr, w.f, kD, 0));
  MAGPO_TRY(act_rms_fwd(s, R, w.f, w.x1, p.ln2, 0, pe, step, max_step, w.x, w.xpe));
  MAGPO_TRY(gemm_nn(s, R, kD, kD, w.x, kD, wref(p.h0_w, kD, pt ? pt->h0T : nullptr, kD), p.h0_b, w.zh, kD, 0));
  MAGPO_TRY(head_fwd(s, R, w.zh, p.h2_s, p.h3_w, p.h3_b, 1, value));
  return MAGPO_OK;
}

// Decoder over R rows (Decoder.__call__/recurrent, sable_network.py:296-343). `embed_A`: agents per timestep for
// the shifted-action tokens (>0 training; 0: action[] holds the previous agent's action; <0: start tokens).
// `ret_A`: tokens per timestep seen by the retention scans. x_rep / x_rep_pe: encoder output (+PE) rows.
// phase 1: the part that does not depend on the encoder (token embedding, self retention, the key / value / gate projections of the
// cross retention); phase 2: the rest; phase 0: both.
static int decoder_forward_phase(int phase, bool q_done, cudaStream_t s, const GuiderP& p, const GuiderT* pt, int T, int N, int ret_A, int embed_A, int a,
                                 int max_step, const int32_t* action, const float* x_rep, const float* x_rep_pe,
                                 const int32_t* step, const uint8_t* done, const float* Hself0, const float* Hcross0,
                                 float kappa, const float* pe, const SableActs& w, float* logits, float* Hs_self,
                                 float* Hs_cross, float* Hself_out, float* Hcross_out) {
  const int64_t R = (int64_t)T * N * ret_A;
  const bool chained = pt && embed_A > 0 && !Hself_out && chain_supported(R);  // training forward only: the rollout keeps its kernels
  if (phase != 2) {
    if (chained) {
      MAGPO_TRY(chain_front_fwd(s, R, 0, nullptr, nullptr, nullptr, embed_A, a, action, p.Wa, p.dln, pe, step, max_step, pt->qkvg1T, nullptr,
                                w.xD, w.xpeD, w.qkvg1));
    } else {
      MAGPO_TRY(embed_fwd(s, R, embed_A, action, p.Wa, p.dln, pe, step, max_step, w.xD, w.xpeD));
      MAGPO_TRY(gemm_nn(s, R, 4 * kD, kD, w.xpeD, kD, wref(p.qkvg1, 4 * kD, pt ? pt->qkvg1T : nullptr, kD), nullptr, w.qkvg1, 4 * kD, 0));
    }
    MAGPO_TRY(retention_fwd(s, T, N, ret_A, kappa, true, w.qkvg1, w.qkvg1 + kD, w.qkvg1 + 2 * kD, 4 * kD, Hself0, done,
                            w.ret1, Hs_self, Hself_out));
    if (chained) {
      // ... and the key / value / gate projections of the cross retention in the same kernel
      MAGPO_TRY(chain_gate_fwd(s, R, w.qkvg1 + 3 * kD, 4 * kD, w.ret1, w.xD, p.gn1_s, p.gn1_b, p.dln1, pe, step, max_step, pt->wo1T, nullptr,
                               pt->qkvg2T + kD * kD, w.gated1, w.o1, nullptr, w.rpe, nullptr, nullptr, w.qkvg2 + kD, 4 * kD));
    } else {
      MAGPO_TRY(gn_gate_fwd(s, R, w.qkvg1 + 3 * kD, 4 * kD, w.ret1, p.gn1_s, p.gn1_b, w.gated1));
      MAGPO_TRY(gemm_nn(s, R, kD, kD, w.gated1, kD, wref(p.wo1, kD, pt ? pt->wo1T : nullptr, kD), nullptr, w.o1, kD, 0));
      MAGPO_TRY(act_rms_fwd(s, R, w.o1, w.xD, p.dln1, 0, pe, step, max_step, nullptr, w.rpe));
    }
    // cross retention: key = value = r (+PE), query = obs_rep (+PE); gate input is the PE-added key
    if (!chained) MAGPO_TRY(gemm_nn(s, R, 3 * kD, kD, w.rpe, kD, wref(p.qkvg2 + kD, 4 * kD, pt ? pt->qkvg2T + kD * kD : nullptr, kD), nullptr, w.qkvg2 + kD, 4 * kD, 0));
  }
  if (phase == 1) return MAGPO_OK;
  if (!q_done) MAGPO_TRY(gemm_nn(s, R, kD, kD, x_rep_pe, kD, wref(p.qkvg2, 4 * kD, pt ? pt->qkvg2T : nullptr, kD), nullptr, w.qkvg2, 4 * kD, 0));
  MAGPO_TRY(retention_fwd(s, T, N, ret_A, kappa, true, w.qkvg2, w.qkvg2 + kD, w.qkvg2 + 2 * kD, 4 * kD, Hcross0, done,
                          w.ret2, Hs_cross, Hcross_out));
  if (chained) {
    MAGPO_TRY(chain_gate_fwd(s, R, w.qkvg2 + 3 * kD, 4 * kD, w.ret2, x_rep, p.gn2_s, p.gn2_b, p.dln2, nullptr, nullptr, 0, pt->wo2T, pt->dffn_glT,
                             nullptr, w.gated2, w.o2, w.y, nullptr, w.glD, w.hmidD, nullptr, 0));
    MAGPO_TRY(chain_tail_fwd(s, R, w.hmidD, w.y, p.dln3, nullptr, nullptr, 0, pt->dffn_outT, nullptr, 0, pt->dh0T, p.dh0_b, p.dh2_s, p.dh3_w,
                             p.dh3_b, a, w.fD, w.xd, nullptr, nullptr, 0, w.zhD, logits));
    return MAGPO_OK;
  }
  MAGPO_TRY(gn_gate_fwd(s, R, w.qkvg2 + 3 * kD, 4 * kD, w.ret2, p.gn2_s, p.gn2_b, w.gated2));
  MAGPO_TRY(gemm_nn(s, R, kD, kD, w.gated2, kD, wref(p.wo2, kD, pt ? pt->wo2T : nullptr, kD), nullptr, w.o2, kD, 0));
  MAGPO_TRY(act_rms_fwd(s, R, w.o2, x_rep, p.dln2, 0, nullptr, nullptr, 0, w.y, nullptr));
  MAGPO_TRY(gemm_nn(s, R, 2 * kD, kD, w.y, kD, wref(p.dffn_gl, 2 * kD, pt ? pt->dffn_glT : nullptr, kD), nullptr, w.glD, 2 * kD, 0));
  MAGPO_TRY(swiglu_fwd(s, R, w.glD, w.hmidD));
  MAGPO_TRY(gemm_nn(s, R, kD, kD, w.hmidD, kD, wref(p.dffn_out, kD, pt ? pt->dffn_outT : nullptr, kD), nullptr, w.fD, kD, 0));
  MAGPO_TRY(act_rms_fwd(s, R, w.fD, w.y, p.dln3, 0, nullptr, nullptr, 0, w.xd, nullptr));
  MAGPO_TRY(gemm_nn(s, R, kD, kD, w.xd, kD, wref(p.dh0_w, kD, pt ? pt->dh0T : nullptr, kD), p.dh0_b, w.zhD, kD, 0));
  MAGPO_TRY(head_fwd(s, R, w.zhD, p.dh2_s, p.dh3_w, p.dh3_b, a, logits));
  return MAGPO_OK;
}

int sable_decoder_forward(cudaStream_t s, const GuiderP& p, const GuiderT* pt, int T, int N, int ret_A, int embed_A, int a,
                          int max_step, const int32_t* action, const float* x_rep, const float* x_rep_pe,
                          const int32_t* step, const uint8_t* done, const float* Hself0, const float* Hcross0,
                          float kappa, const float* pe, const SableActs& w, float* logits, float* Hs_self,
                          float* Hs_cross, float* Hself_out, float* Hcross_out) {
  return decoder_forward_phase(0, false, s, p, pt, T, N, ret_A, embed_A, a, max_step, action, x_rep, x_rep_pe, step, done, Hself0, Hcross0,
                               kappa, pe, w, logits, Hs_self, Hs_cross, Hself_out, Hcross_out);
}

// The decoder's encoder-independent prefix runs beside the encoder on the context's `dec` stream: both are chains of kernels that sit
// at 0.3-0.7 of the HBM roofline each, so together they use the memory system better than one after the other.
int sable_train_forward(cudaStream_t s, const GuiderP& p, const GuiderT* pt, const SableBatch& b, const SableActs& w,
                        float* value, float* logits, bool save_states) {
  const bool overlap = nets_overlap_enabled();
  float* hs_self = save_states ? w.Hs_self : nullptr;
  float* hs_cross = save_states ? w.Hs_cross : nullptr;
  ForkJoin& g_dec = ctx().dec;
  if (overlap) {
    MAGPO_CUDA_OK(cudaEventRecord(g_dec.fork, s));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(g_dec.s, g_dec.fork, 0));
    MAGPO_TRY(decoder_forward_phase(1, false, g_dec.s, p, pt, b.T, b.N, b.A, b.A, b.a, b.max_step, b.action, w.x, w.xpe, b.step_count,
                                    b.done, b.h_self, b.h_cross, b.kappa, b.pe, w, logits, hs_self, hs_cross, nullptr, nullptr));
  }
  // with the fused chains the encoder's tail kernel also projects the decoder's cross-retention query (q = (x + PE) W_q of retn2)
  const bool fuse_q = pt && chain_supported((int64_t)b.T * b.N * b.A);
  MAGPO_TRY(sable_encoder_forward(s, p, pt, b.T, b.N, b.A, b.d, b.max_step, b.agents_view, b.step_count, b.done, b.h_enc,
                                  b.kappa, b.pe, w, value, save_states ? w.Hs_enc : nullptr, nullptr, true, fuse_q ? w.qkvg2 : nullptr));
  if (overlap) {
    MAGPO_CUDA_OK(cudaEventRecord(g_dec.join, g_dec.s));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(s, g_dec.join, 0));
  }
  MAGPO_TRY(decoder_forward_phase(overlap ? 2 : 0, fuse_q, s, p, pt, b.T, b.N, b.A, b.A, b.a, b.max_step, b.action, w.x, w.xpe, b.step_count,
                                  b.done, b.h_self, b.h_cross, b.kappa, b.pe, w, logits, hs_self, hs_cross, nullptr, nullptr));
  return MAGPO_OK;
}

// ----------------------------------------------------------------------------- backward
// dense layer y = x @ W (+ b): dW += x^T dy, db += colsum(dy), dx = dy @ W^T
// W [K,N] (leading dimension ldw) is the layer's weight, WT its transposed copy [N,K]
static int dense_bwd(cudaStream_t s, int64_t R, int K, int N, const float* x, int ldx, const float* dy, int lddy,
                     const float* WT, const float* W, int ldw, float* dW, int lddw, float* db, float* dx, int lddx,
                     int dx_flags) {
  if (dW) MAGPO_TRY(gemm_tn(s, R, N, K, x, ldx, dy, lddy, dW, lddw));
  if (db) MAGPO_TRY(colsum(s, R, N, dy, lddy, db));
  if (dx) MAGPO_TRY(gemm_nn(s, R, K, N, dy, lddy, wref(WT, K, W, ldw), nullptr, dx, lddx, dx_flags));
  return MAGPO_OK;
}

int sable_train_backward(cudaStream_t s, const GuiderP& p, const GuiderT& pt, const SableBatch& b, const SableActs& w,
                         const float* dlogits, const float* dvalue, const GuiderP& g) {
  const int T = b.T, N = b.N, A = b.A, a = b.a, d = b.d;
  const int64_t R = (int64_t)T * N * A;
  const int Q = 4 * kD;
  // ---- decoder
  MAGPO_TRY(head_bwd(s, R, w.zhD, p.dh2_s, p.dh3_w, a, dlogits, w.tA, g.dh2_s, g.dh3_w, g.dh3_b, g.dh0_b));
  MAGPO_TRY(dense_bwd(s, R, kD, kD, w.xd, kD, w.tA, kD, pt.dh0T, p.dh0_w, kD, g.dh0_w, kD, nullptr, w.tB, kD, 0));
  MAGPO_TRY(act_rms_bwd(s, R, w.fD, w.y, p.dln3, 0, w.tB, nullptr, nullptr, w.tA, g.dln3));       // tA = d(fD) = d(y) residual
  MAGPO_TRY(dense_bwd(s, R, kD, kD, w.hmidD, kD, w.tA, kD, pt.dffn_outT, p.dffn_out, kD, g.dffn_out, kD, nullptr, w.tB, kD, 0));
  MAGPO_TRY(swiglu_bwd(s, R, w.glD, w.tB, w.tG));
  MAGPO_TRY(dense_bwd(s, R, kD, 2 * kD, w.y, kD, w.tG, 2 * kD, pt.dffn_glT, p.dffn_gl, 2 * kD, g.dffn_gl, 2 * kD, nullptr, w.tB, kD, 0));
  MAGPO_TRY(act_rms_bwd(s, R, w.o2, w.x, p.dln2, 0, w.tA, w.tB, nullptr, w.tD, g.dln2));          // tD = d(o2) = d(obs_rep) #1
  MAGPO_TRY(dense_bwd(s, R, kD, kD, w.gated2, kD, w.tD, kD, pt.wo2T, p.wo2, kD, g.wo2, kD, nullptr, w.tA, kD, 0));
  MAGPO_TRY(gn_gate_bwd(s, R, w.qkvg2 + 3 * kD, Q, w.ret2, p.gn2_s, p.gn2_b, w.tA, w.tQ + 3 * kD, Q, w.tB, g.gn2_s,
                        g.gn2_b));
  MAGPO_TRY(retention_bwd(s, T, N, A, b.kappa, true, w.qkvg2, w.qkvg2 + kD, w.qkvg2 + 2 * kD, Q, b.h_cross, b.done,
                          w.Hs_cross, w.tB, w.tQ, w.tQ + kD, w.tQ + 2 * kD, Q));
  // query path -> obs_rep (+PE); key/value/gate path -> r (+PE)
  MAGPO_TRY(dense_bwd(s, R, kD, kD, w.xpe, kD, w.tQ, Q, pt.qkvg2T, p.qkvg2, Q, g.qkvg2, Q, nullptr, w.tE, kD, 0));  // tE = d(obs_rep) #2
  MAGPO_TRY(dense_bwd(s, R, kD, 3 * kD, w.rpe, kD, w.tQ + kD, Q, pt.qkvg2T + kD * kD, p.qkvg2 + kD, Q, g.qkvg2 + kD, Q, nullptr, w.tA,
                      kD, 0));                                                                     // tA = d(r)
  MAGPO_TRY(act_rms_bwd(s, R, w.o1, w.xD, p.dln1, 0, w.tA, nullptr, nullptr, w.tB, g.dln1));      // tB = d(o1) = d(xD) residual
  MAGPO_TRY(dense_bwd(s, R, kD, kD, w.gated1, kD, w.tB, kD, pt.wo1T, p.wo1, kD, g.wo1, kD, nullptr, w.tA, kD, 0));
  MAGPO_TRY(gn_gate_bwd(s, R, w.qkvg1 + 3 * kD, Q, w.ret1, p.gn1_s, p.gn1_b, w.tA, w.tQ + 3 * kD, Q, w.tC, g.gn1_s,
                        g.gn1_b));
  MAGPO_TRY(retention_bwd(s, T, N, A, b.kappa, true, w.qkvg1, w.qkvg1 + kD, w.qkvg1 + 2 * kD, Q, b.h_self, b.done,
                          w.Hs_self, w.tC, w.tQ, w.tQ + kD, w.tQ + 2 * kD, Q));
  MAGPO_TRY(dense_bwd(s, R, kD, Q, w.xpeD, kD, w.tQ, Q, pt.qkvg1T, p.qkvg1, Q, g.qkvg1, Q, nullptr, w.tA, kD, 0));  // tA = d(xpeD)
  MAGPO_TRY(embed_bwd(s, R, A, a, b.action, p.Wa, p.dln, w.tB, w.tA, g.Wa, g.dln));
  // ---- encoder: d(obs_rep) = head path + tD + tE
  MAGPO_TRY(head_bwd(s, R, w.zh, p.h2_s, p.h3_w, 1, dvalue, w.tA, g.h2_s, g.h3_w, g.h3_b, g.h0_b));
  MAGPO_TRY(dense_bwd(s, R, kD, kD, w.x, kD, w.tA, kD, pt.h0T, p.h0_w, kD, g.h0_w, kD, nullptr, w.tB, kD, 0));
  MAGPO_TRY(act_rms_bwd(s, R, w.f, w.x1, p.ln2, 0, w.tB, w.tD, w.tE, w.tA, g.ln2));               // tA = d(f) = d(x1) residual
  MAGPO_TRY(dense_bwd(s, R, kD, kD, w.hmid, kD, w.tA, kD, pt.ffn_outT, p.ffn_out, kD, g.ffn_out, kD, nullptr, w.tB, kD, 0));
  MAGPO_TRY(swiglu_bwd(s, R, w.gl, w.tB, w.tG));
  MAGPO_TRY(dense_bwd(s, R, kD, 2 * kD, w.x1, kD, w.tG, 2 * kD, pt.ffn_glT, p.ffn_gl, 2 * kD, g.ffn_gl, 2 * kD, nullptr, w.tB, kD, 0));
  MAGPO_TRY(act_rms_bwd(s, R, w.o, w.xin, p.ln1, 0, w.tA, w.tB, nullptr, w.tD, g.ln1));           // tD = d(o) = d(xin) residual
  MAGPO_TRY(dense_bwd(s, R, kD, kD, w.gated, kD, w.tD, kD, pt.woT, p.wo, kD, g.wo, kD, nullptr, w.tA, kD, 0));
  MAGPO_TRY(gn_gate_bwd(s, R, w.qkvg + 3 * kD, Q, w.ret, p.gn_s, p.gn_b, w.tA, w.tQ + 3 * kD, Q, w.tB, g.gn_s, g.gn_b));
  MAGPO_TRY(retention_bwd(s, T, N, A, b.kappa, false, w.qkvg, w.qkvg + kD, w.qkvg + 2 * kD, Q, b.h_enc, b.done,
                          w.Hs_enc, w.tB, w.tQ, w.tQ + kD, w.tQ + 2 * kD, Q));
  MAGPO_TRY(dense_bwd(s, R, kD, Q, w.kqv, kD, w.tQ, Q, pt.qkvgT, p.qkvg, Q, g.qkvg, Q, nullptr, w.tA, kD, 0));  // tA = d(kqv)
  MAGPO_TRY(act_rms_bwd(s, R, w.z0, nullptr, p.ln, ROW_GELU, w.tD, w.tA, nullptr, w.tB, g.ln));   // tB = d(z0)
  if (obs_embed_ok(d)) {
    MAGPO_TRY(obs_embed_bwd(s, R, d, b.agents_view, p.obs_scale, p.Wobs, w.tB, g.Wobs, g.obs_scale));
  } else {
    MAGPO_TRY(dense_bwd(s, R, d, kD, w.on, d, w.tB, kD, pt.WobsT, p.Wobs, kD, g.Wobs, kD, nullptr, w.t_d, d, 0));
    MAGPO_TRY(rms_general_bwd_scale(s, R, d, b.agents_view, w.t_d, g.obs_scale));
  }
  return MAGPO_OK;
}

}  // namespace magpo
