// The general Sable guider (generic.cuh): training forward + hand-derived backward and the per-timestep inference path for any
// (embed_dim, n_head, n_block) of net_shape_ok(), as sequences of GEMMs (gemm.cu / gemm_tc.cu), the row kernels of generic_rows.cu and the
// per-(env, head) retention scan. Structure and quirks follow networks/sable_network.py: the encoder applies its ONE shared `ln` in front of
// every block (:128-133), the decoder normalises the action embedding once (:305-306), every decoder block reads the same obs_rep
// (:309-311), MultiScaleRetention adds the positional encoding to key / query / value and gates on the PE-added key (retention.py:278-295).
#include <stdlib.h>

#include <string>

#include "generic.cuh"

namespace magpo {

// ----------------------------------------------------------------------------- parameters
GuiderG GuiderG::bind(float* base, const NetShape& s) {
  GuiderG p;
  int64_t off = 0;
  auto take = [&](int64_t n) {
    float* r = base ? base + off : nullptr;
    off += align4(n);
    return r;
  };
  auto retn = [&](RetnG& r) {
    r.qkvg = take((int64_t)s.D * 4 * s.D);
    r.wo = take((int64_t)s.D * s.D);
    r.gn_s = take(s.hs);
    r.gn_b = take(s.hs);
  };
  const int D = s.D;
  p.obs_scale = take(s.d); p.Wobs = take((int64_t)s.d * D); p.ln = take(D);
  for (int b = 0; b < s.nb; ++b) {
    EncBlockG& e = p.enc[b];
    e.ln1 = take(D); e.ln2 = take(D);
    retn(e.r);
    e.ffn_gl = take((int64_t)D * 2 * D); e.ffn_out = take((int64_t)D * D);
  }
  p.h0_w = take((int64_t)D * D); p.h0_b = take(D); p.h2_s = take(D); p.h3_w = take(D); p.h3_b = take(1);
  p.Wa = take((int64_t)(s.a + 1) * D); p.dln = take(D);
  for (int b = 0; b < s.nb; ++b) {
    DecBlockG& e = p.dec[b];
    e.ln1 = take(D); e.ln2 = take(D); e.ln3 = take(D);
    retn(e.r1);
    retn(e.r2);
    e.ffn_gl = take((int64_t)D * 2 * D); e.ffn_out = take((int64_t)D * D);
  }
  p.dh0_w = take((int64_t)D * D); p.dh0_b = take(D); p.dh2_s = take(D); p.dh3_w = take((int64_t)D * s.a); p.dh3_b = take(s.a);
  p.total = off;
  return p;
}

void guider_table_g(const NetShape& s, std::vector<ParamEntryG>* out) {
  GuiderG p = GuiderG::bind(reinterpret_cast<float*>(sizeof(float)), s);  // fake base: pointer arithmetic -> offsets
  auto off = [](const float* q) { return (int64_t)(reinterpret_cast<uintptr_t>(q) / sizeof(float)) - 1; };
  auto add = [&](const std::string& name, const float* q, int64_t extra, int r, int c, int ld) {
    ParamEntryG e;
    snprintf(e.name, sizeof(e.name), "%s", name.c_str());
    e.offset = off(q) + extra; e.dim0 = r; e.dim1 = c; e.ld = ld;
    out->push_back(e);
  };
  const int D = s.D, hs = s.hs;
  auto retn = [&](const std::string& pre, const RetnG& r) {
    for (int h = 0; h < s.nh; ++h) {
      const std::string hp = pre + "/retention_heads_" + std::to_string(h);
      add(hp + "/w_q", r.qkvg, h * hs, D, hs, 4 * D);
      add(hp + "/w_k", r.qkvg, D + h * hs, D, hs, 4 * D);
      add(hp + "/w_v", r.qkvg, 2 * D + h * hs, D, hs, 4 * D);
    }
    add(pre + "/w_g", r.qkvg, 3 * D, D, D, 4 * D);
    add(pre + "/w_o", r.wo, 0, D, D, D);
    add(pre + "/group_norm/scale", r.gn_s, 0, hs, 0, 1);
    add(pre + "/group_norm/bias", r.gn_b, 0, hs, 0, 1);
  };
  add("encoder/obs_encoder/layers_0/scale", p.obs_scale, 0, s.d, 0, 1);
  add("encoder/obs_encoder/layers_1/kernel", p.Wobs, 0, s.d, D, D);
  add("encoder/ln/scale", p.ln, 0, D, 0, 1);
  for (int b = 0; b < s.nb; ++b) {
    const std::string pre = "encoder/encoder_block_" + std::to_string(b);
    add(pre + "/ln1/scale", p.enc[b].ln1, 0, D, 0, 1);
    add(pre + "/ln2/scale", p.enc[b].ln2, 0, D, 0, 1);
    retn(pre + "/retn", p.enc[b].r);
    add(pre + "/ffn/W_gate", p.enc[b].ffn_gl, 0, D, D, 2 * D);
    add(pre + "/ffn/W_linear", p.enc[b].ffn_gl, D, D, D, 2 * D);
    add(pre + "/ffn/W_output", p.enc[b].ffn_out, 0, D, D, D);
  }
  add("encoder/head/layers_0/kernel", p.h0_w, 0, D, D, D);
  add("encoder/head/layers_0/bias", p.h0_b, 0, D, 0, 1);
  add("encoder/head/layers_2/scale", p.h2_s, 0, D, 0, 1);
  add("encoder/head/layers_3/kernel", p.h3_w, 0, D, 1, 1);
  add("encoder/head/layers_3/bias", p.h3_b, 0, 1, 0, 1);
  add("decoder/action_encoder/layers_0/kernel", p.Wa, 0, s.a + 1, D, D);
  add("decoder/ln/scale", p.dln, 0, D, 0, 1);
  for (int b = 0; b < s.nb; ++b) {
    const std::string pre = "decoder/decoder_block_" + std::to_string(b);
    add(pre + "/ln1/scale", p.dec[b].ln1, 0, D, 0, 1);
    add(pre + "/ln2/scale", p.dec[b].ln2, 0, D, 0, 1);
    add(pre + "/ln3/scale", p.dec[b].ln3, 0, D, 0, 1);
    retn(pre + "/retn1", p.dec[b].r1);
    retn(pre + "/retn2", p.dec[b].r2);
    add(pre + "/ffn/W_gate", p.dec[b].ffn_gl, 0, D, D, 2 * D);
    add(pre + "/ffn/W_linear", p.dec[b].ffn_gl, D, D, D, 2 * D);
    add(pre + "/ffn/W_output", p.dec[b].ffn_out, 0, D, D, D);
  }
  add("decoder/head/layers_0/kernel", p.dh0_w, 0, D, D, D);
  add("decoder/head/layers_0/bias", p.dh0_b, 0, D, 0, 1);
  add("decoder/head/layers_2/scale", p.dh2_s, 0, D, 0, 1);
  add("decoder/head/layers_3/kernel", p.dh3_w, 0, D, s.a, s.a);
  add("decoder/head/layers_3/bias", p.dh3_b, 0, s.a, 0, 1);
}

namespace {

using Kap = HeadKappas;

// ----------------------------------------------------------------------------- workspace
struct EncActs {
  float *xn, *kqv, *qkvg, *ret, *gated, *o, *x1, *gl, *hmid, *f, *xout, *xpe, *Hs;
};
struct DecActs {
  float *xin, *xpe, *qkvg1, *ret1, *gated1, *o1, *r, *rpe, *qkvg2, *ret2, *gated2, *o2, *y, *gl, *hmid, *f, *xd, *Hs1, *Hs2;
};
// transposed weights (dX = dY W^T on the GEMM kernels that take [K, N] operands) + TF32 hi / lo images for the tensor-core path
struct RetnT {
  float *qkvgT, *woT;
};
struct Ws {
  float *on, *z0, *zh, *hn, *xD, *zhD, *hnD, *pe;
  EncActs enc[3];
  DecActs dec[3];
  float *WobsT, *h0T, *h3T, *dh0T, *dh3T;
  RetnT et[3], dt1[3], dt2[3];
  float *e_glT[3], *e_outT[3], *d_glT[3], *d_outT[3];
  float *t_hi, *t_lo, *p_hi, *p_lo;
  int64_t t_n;
  // backward scratch
  float *tA, *tB, *tC, *tD, *tE, *tX, *tQ, *tG, *t_d, *t_a, *dxrep;
  void plan(Arena& ar, const NetShape& s, int T, int N, int rows_per_step, bool bwd) {
    const int D = s.D;
    const int64_t R = (int64_t)T * N * rows_per_step;
    const size_t rD = (size_t)R * D;
    on = ar.get<float>((size_t)R * s.d); z0 = ar.get<float>(rD); zh = ar.get<float>(rD); hn = ar.get<float>(rD);
    xD = ar.get<float>(rD); zhD = ar.get<float>(rD); hnD = ar.get<float>(rD);
    pe = ar.get<float>((size_t)(s.max_step + 1) * D);
    const size_t hsave = bwd ? (size_t)T * N * s.nh * s.hs * s.hs : 0;
    for (int b = 0; b < s.nb; ++b) {
      EncActs& e = enc[b];
      e.xn = ar.get<float>(rD); e.kqv = ar.get<float>(rD); e.qkvg = ar.get<float>(4 * rD); e.ret = ar.get<float>(rD);
      e.gated = ar.get<float>(rD); e.o = ar.get<float>(rD); e.x1 = ar.get<float>(rD); e.gl = ar.get<float>(2 * rD);
      e.hmid = ar.get<float>(rD); e.f = ar.get<float>(rD); e.xout = ar.get<float>(rD); e.xpe = ar.get<float>(rD);
      e.Hs = hsave ? ar.get<float>(hsave) : nullptr;
      DecActs& c = dec[b];
      c.xin = b == 0 ? xD : dec[b - 1].xd;
      c.xpe = ar.get<float>(rD); c.qkvg1 = ar.get<float>(4 * rD); c.ret1 = ar.get<float>(rD); c.gated1 = ar.get<float>(rD);
      c.o1 = ar.get<float>(rD); c.r = ar.get<float>(rD); c.rpe = ar.get<float>(rD); c.qkvg2 = ar.get<float>(4 * rD);
      c.ret2 = ar.get<float>(rD); c.gated2 = ar.get<float>(rD); c.o2 = ar.get<float>(rD); c.y = ar.get<float>(rD);
      c.gl = ar.get<float>(2 * rD); c.hmid = ar.get<float>(rD); c.f = ar.get<float>(rD); c.xd = ar.get<float>(rD);
      c.Hs1 = hsave ? ar.get<float>(hsave) : nullptr;
      c.Hs2 = hsave ? ar.get<float>(hsave) : nullptr;
    }
    // transposed weights: one contiguous region
    float* t0 = ar.get<float>(0);
    WobsT = ar.get<float>((size_t)D * s.d); h0T = ar.get<float>((size_t)D * D); h3T = ar.get<float>(D);
    dh0T = ar.get<float>((size_t)D * D); dh3T = ar.get<float>((size_t)s.a * D);
    for (int b = 0; b < s.nb; ++b) {
      et[b].qkvgT = ar.get<float>((size_t)4 * D * D); et[b].woT = ar.get<float>((size_t)D * D);
      dt1[b].qkvgT = ar.get<float>((size_t)4 * D * D); dt1[b].woT = ar.get<float>((size_t)D * D);
      dt2[b].qkvgT = ar.get<float>((size_t)4 * D * D); dt2[b].woT = ar.get<float>((size_t)D * D);
      e_glT[b] = ar.get<float>((size_t)2 * D * D); e_outT[b] = ar.get<float>((size_t)D * D);
      d_glT[b] = ar.get<float>((size_t)2 * D * D); d_outT[b] = ar.get<float>((size_t)D * D);
    }
    float* t1 = ar.get<float>(0);
    t_n = (int64_t)(reinterpret_cast<uintptr_t>(t1) - reinterpret_cast<uintptr_t>(t0)) / 4;
    t_hi = ar.get<float>((size_t)t_n); t_lo = ar.get<float>((size_t)t_n);
    const int64_t n_p = GuiderG::bind(nullptr, s).total;
    p_hi = ar.get<float>((size_t)n_p); p_lo = ar.get<float>((size_t)n_p);
    if (bwd) {
      tA = ar.get<float>(rD); tB = ar.get<float>(rD); tC = ar.get<float>(rD); tD = ar.get<float>(rD); tE = ar.get<float>(rD);
      tX = ar.get<float>(rD); tQ = ar.get<float>(4 * rD); tG = ar.get<float>(2 * rD); t_d = ar.get<float>((size_t)R * s.d);
      t_a = ar.get<float>((size_t)R * s.a); dxrep = ar.get<float>(rD);
    } else {
      tA = tB = tC = tD = tE = tX = tQ = tG = t_d = t_a = dxrep = nullptr;
    }
  }
};

int transposes(cudaStream_t s, const NetShape& sh, const GuiderG& p, const Ws& w) {
  const int D = sh.D;
  MAGPO_TRY(transpose(s, sh.d, D, p.Wobs, w.WobsT));
  MAGPO_TRY(transpose(s, D, D, p.h0_w, w.h0T));
  MAGPO_TRY(transpose(s, D, 1, p.h3_w, w.h3T));
  MAGPO_TRY(transpose(s, D, D, p.dh0_w, w.dh0T));
  MAGPO_TRY(transpose(s, D, sh.a, p.dh3_w, w.dh3T));
  for (int b = 0; b < sh.nb; ++b) {
    MAGPO_TRY(transpose(s, D, 4 * D, p.enc[b].r.qkvg, w.et[b].qkvgT));
    MAGPO_TRY(transpose(s, D, D, p.enc[b].r.wo, w.et[b].woT));
    MAGPO_TRY(transpose(s, D, 4 * D, p.dec[b].r1.qkvg, w.dt1[b].qkvgT));
    MAGPO_TRY(transpose(s, D, D, p.dec[b].r1.wo, w.dt1[b].woT));
    MAGPO_TRY(transpose(s, D, 4 * D, p.dec[b].r2.qkvg, w.dt2[b].qkvgT));
    MAGPO_TRY(transpose(s, D, D, p.dec[b].r2.wo, w.dt2[b].woT));
    MAGPO_TRY(transpose(s, D, 2 * D, p.enc[b].ffn_gl, w.e_glT[b]));
    MAGPO_TRY(transpose(s, D, D, p.enc[b].ffn_out, w.e_outT[b]));
    MAGPO_TRY(transpose(s, D, 2 * D, p.dec[b].ffn_gl, w.d_glT[b]));
    MAGPO_TRY(transpose(s, D, D, p.dec[b].ffn_out, w.d_outT[b]));
  }
  MAGPO_TRY(tc_prepare_region(s, w.WobsT, w.t_n, w.t_hi, w.t_lo));
  MAGPO_TRY(tc_prepare_region(s, p.obs_scale, p.total, w.p_hi, w.p_lo));
  return MAGPO_OK;
}

// y = x @ W (+ b): W [K, N] (leading dimension ldw), WT its transposed copy
int dense_fwd(cudaStream_t s, int64_t R, int K, int N, const float* x, int ldx, const float* W, int ldw, const float* WT, const float* b, float* y,
              int ldy) {
  return gemm_nn(s, R, N, K, x, ldx, wref(W, ldw, WT, K), b, y, ldy, 0);
}
// dW += x^T dy, db += colsum(dy), dx = dy @ W^T
int dense_bwd(cudaStream_t s, int64_t R, int K, int N, const float* x, int ldx, const float* dy, int lddy, const float* WT, const float* W,
              int ldw, float* dW, int lddw, float* db, float* dx, int lddx) {
  if (dW) MAGPO_TRY(gemm_tn(s, R, N, K, x, ldx, dy, lddy, dW, lddw));
  if (db) MAGPO_TRY(colsum(s, R, N, dy, lddy, db));
  if (dx) MAGPO_TRY(gemm_nn(s, R, K, N, dy, lddy, wref(WT, K, W, ldw), nullptr, dx, lddx, 0));
  return MAGPO_OK;
}

Kap kappas_of(const MagpoNetCfg* net, bool ones) {
  Kap k;
  for (int h = 0; h < 4; ++h) k.k[h] = ones ? 1.0f : (h < net->n_head ? head_kappa(net, h) : 0.f);
  return k;
}

// MultiScaleRetention of one block from the PE-added input rows `in_kvg` (key = value = gate input) and `in_q` (query; == in_kvg for the
// self retentions): qkvg projection(s), per-head scan, GroupNorm * swish gate, output projection. T, N, rps: the scan's geometry.
int msr_fwd(cudaStream_t s, const NetShape& sh, const Kap& kap, int blk, int T, int N, int rps, bool causal, const float* in_q, const float* in_kvg,
            const RetnG& r, const RetnT& rt, const uint8_t* done, const float* H0, float* qkvg, float* ret, float* gated, float* o, float* Hsave,
            float* Hout) {
  const int D = sh.D, Q = 4 * D;
  const int64_t R = (int64_t)T * N * rps;
  if (in_q == in_kvg) {
    MAGPO_TRY(dense_fwd(s, R, D, Q, in_kvg, D, r.qkvg, Q, rt.qkvgT, nullptr, qkvg, Q));
  } else {
    MAGPO_TRY(dense_fwd(s, R, D, D, in_q, D, r.qkvg, Q, rt.qkvgT, nullptr, qkvg, Q));
    MAGPO_TRY(dense_fwd(s, R, D, 3 * D, in_kvg, D, r.qkvg + D, Q, rt.qkvgT + (size_t)D * D, nullptr, qkvg + D, Q));
  }
  MAGPO_TRY(g_retention_fwd(s, sh, kap, blk, T, N, rps, causal, qkvg, qkvg + D, qkvg + 2 * D, Q, H0, done, ret, D, Hsave, Hout));
  MAGPO_TRY(g_gn_gate_fwd(s, D, sh.nh, R, qkvg + 3 * D, Q, ret, r.gn_s, r.gn_b, gated));
  MAGPO_TRY(dense_fwd(s, R, D, D, gated, D, r.wo, D, rt.woT, nullptr, o, D));
  return MAGPO_OK;
}
// backward of msr_fwd given d(o) in `d_o`: parameter gradients into gr, d(in_q) -> d_in_q (written), d(in_kvg) -> d_in_kvg (written);
// when in_q == in_kvg both receive the single input gradient through d_in_kvg. scratch: tQ [R, 4D], t1, t2 [R, D].
int msr_bwd(cudaStream_t s, const NetShape& sh, const Kap& kap, int T, int N, int rps, bool causal, const float* in_q, const float* in_kvg,
            const RetnG& r, const RetnT& rt, const RetnG& gr, const uint8_t* done, const float* qkvg, const float* ret, const float* gated,
            const float* Hsave, const float* d_o, float* d_in_q, float* d_in_kvg, float* tQ, float* t1, float* t2) {
  const int D = sh.D, Q = 4 * D;
  const int64_t R = (int64_t)T * N * rps;
  MAGPO_TRY(dense_bwd(s, R, D, D, gated, D, d_o, D, rt.woT, r.wo, D, gr.wo, D, nullptr, t1, D));  // t1 = d(gated)
  MAGPO_TRY(g_gn_gate_bwd(s, D, sh.nh, R, qkvg + 3 * D, Q, ret, r.gn_s, r.gn_b, t1, tQ + 3 * D, Q, t2, gr.gn_s, gr.gn_b));  // t2 = d(ret)
  MAGPO_TRY(g_retention_bwd(s, sh, kap, T, N, rps, causal, qkvg, qkvg + D, qkvg + 2 * D, Q, done, Hsave, t2, D, tQ, tQ + D, tQ + 2 * D, Q));
  if (in_q == in_kvg) {
    MAGPO_TRY(dense_bwd(s, R, D, Q, in_kvg, D, tQ, Q, rt.qkvgT, r.qkvg, Q, gr.qkvg, Q, nullptr, d_in_kvg, D));
  } else {
    MAGPO_TRY(dense_bwd(s, R, D, D, in_q, D, tQ, Q, rt.qkvgT, r.qkvg, Q, gr.qkvg, Q, nullptr, d_in_q, D));
    MAGPO_TRY(dense_bwd(s, R, D, 3 * D, in_kvg, D, tQ + D, Q, rt.qkvgT + (size_t)D * D, r.qkvg + D, Q, gr.qkvg + D, Q, nullptr, d_in_kvg, D));
  }
  return MAGPO_OK;
}

// head: zh = x @ W0 + b0; hn = RMSNorm(gelu(zh)) * s2; out = hn @ W3 + b3
int head_fwd_g(cudaStream_t s, const NetShape& sh, int64_t R, const float* x, const float* W0, const float* W0T, const float* b0, const float* s2,
               const float* W3, const float* W3T, const float* b3, int nout, float* zh, float* hn, float* out) {
  const int D = sh.D;
  MAGPO_TRY(dense_fwd(s, R, D, D, x, D, W0, D, W0T, b0, zh, D));
  MAGPO_TRY(g_act_rms_fwd(s, D, R, zh, nullptr, s2, ROW_GELU, nullptr, nullptr, 0, hn, nullptr));
  MAGPO_TRY(gemm_nn(s, R, nout, D, hn, D, wref(W3, nout), b3, out, nout, 0));
  return MAGPO_OK;
}
// d(x) -> dx (written); scratch t1, t2 [R, D]
int head_bwd_g(cudaStream_t s, const NetShape& sh, int64_t R, const float* x, const float* W0, const float* W0T, const float* s2, const float* W3,
               const float* W3T, int nout, const float* zh, const float* hn, const float* dout, float* gW0, float* gb0, float* gs2, float* gW3,
               float* gb3, float* dx, float* t1, float* t2) {
  const int D = sh.D;
  MAGPO_TRY(gemm_tn(s, R, nout, D, hn, D, dout, nout, gW3, nout));
  MAGPO_TRY(colsum(s, R, nout, dout, nout, gb3));
  MAGPO_TRY(gemm_nn(s, R, D, nout, dout, nout, wref(W3T, D), nullptr, t1, D, 0));  // t1 = d(hn)
  MAGPO_TRY(g_act_rms_bwd(s, D, R, zh, nullptr, s2, ROW_GELU, t1, nullptr, nullptr, t2, gs2));  // t2 = d(zh)
  MAGPO_TRY(dense_bwd(s, R, D, D, x, D, t2, D, W0T, W0, D, gW0, D, gb0, dx, D));
  return MAGPO_OK;
}

// Encoder over R = T * N * A rows (Encoder.__call__ / .recurrent, sable_network.py:121-156).
int encoder_fwd(cudaStream_t s, const MagpoNetCfg* net, const NetShape& sh, const GuiderG& p, const Ws& w, int T, int N, const float* agents_view,
                const int32_t* step, const uint8_t* done, const float* H0, float* value, bool save, float* Hout) {
  const int D = sh.D, A = sh.A;
  const int64_t R = (int64_t)T * N * A;
  const Kap kap = kappas_of(net, false);
  MAGPO_TRY(rms_general_fwd(s, R, sh.d, agents_view, p.obs_scale, w.on));
  MAGPO_TRY(gemm_nn(s, R, D, sh.d, w.on, sh.d, wref(p.Wobs, D), nullptr, w.z0, D, 0));
  for (int b = 0; b < sh.nb; ++b) {
    const EncActs& e = w.enc[b];
    const float* xprev = b == 0 ? w.z0 : w.enc[b - 1].xout;
    MAGPO_TRY(g_act_rms_fwd(s, D, R, xprev, nullptr, p.ln, b == 0 ? ROW_GELU : 0, w.pe, step, sh.max_step, e.xn, e.kqv));
    MAGPO_TRY(msr_fwd(s, sh, kap, b, T, N, A, false, e.kqv, e.kqv, p.enc[b].r, w.et[b], done, H0, e.qkvg, e.ret, e.gated, e.o, save ? e.Hs : nullptr,
                      Hout));
    MAGPO_TRY(g_act_rms_fwd(s, D, R, e.o, e.xn, p.enc[b].ln1, 0, nullptr, nullptr, 0, e.x1, nullptr));
    MAGPO_TRY(dense_fwd(s, R, D, 2 * D, e.x1, D, p.enc[b].ffn_gl, 2 * D, w.e_glT[b], nullptr, e.gl, 2 * D));
    MAGPO_TRY(g_swiglu_fwd(s, D, R, e.gl, e.hmid));
    MAGPO_TRY(dense_fwd(s, R, D, D, e.hmid, D, p.enc[b].ffn_out, D, w.e_outT[b], nullptr, e.f, D));
    MAGPO_TRY(g_act_rms_fwd(s, D, R, e.f, e.x1, p.enc[b].ln2, 0, w.pe, step, sh.max_step, e.xout, e.xpe));
  }
  const EncActs& last = w.enc[sh.nb - 1];
  MAGPO_TRY(head_fwd_g(s, sh, R, last.xout, p.h0_w, w.h0T, p.h0_b, p.h2_s, p.h3_w, w.h3T, p.h3_b, 1, w.zh, w.hn, value));
  return MAGPO_OK;
}

// Decoder over R = T * N * rps rows (Decoder.__call__ / .recurrent, :296-343). embed_A as in rowops' embed_fwd (> 0: training tokens shifted per
// timestep; 0: action[] is the previous agent's action; < 0: start tokens). x_rep / x_rep_pe: encoder output (+PE) rows.
int decoder_fwd(cudaStream_t s, const MagpoNetCfg* net, const NetShape& sh, const GuiderG& p, const Ws& w, int T, int N, int rps, int embed_A,
                const int32_t* action, const float* x_rep, const float* x_rep_pe, const int32_t* step, const uint8_t* done, const float* Hself0,
                const float* Hcross0, bool decay, float* logits, bool save, float* Hself_out, float* Hcross_out) {
  const int D = sh.D;
  const int64_t R = (int64_t)T * N * rps;
  const Kap kap = kappas_of(net, !decay);
  MAGPO_TRY(g_embed_fwd(s, D, R, embed_A, action, p.Wa, p.dln, w.pe, step, sh.max_step, w.xD, w.dec[0].xpe));
  for (int b = 0; b < sh.nb; ++b) {
    const DecActs& c = w.dec[b];
    const DecBlockG& pb = p.dec[b];
    // block input (+PE): the previous block wrote xd and its PE-added copy into this block's xpe
    MAGPO_TRY(msr_fwd(s, sh, kap, b, T, N, rps, true, c.xpe, c.xpe, pb.r1, w.dt1[b], done, Hself0, c.qkvg1, c.ret1, c.gated1, c.o1,
                      save ? c.Hs1 : nullptr, Hself_out));
    MAGPO_TRY(g_act_rms_fwd(s, D, R, c.o1, c.xin, pb.ln1, 0, w.pe, step, sh.max_step, c.r, c.rpe));
    MAGPO_TRY(msr_fwd(s, sh, kap, b, T, N, rps, true, x_rep_pe, c.rpe, pb.r2, w.dt2[b], done, Hcross0, c.qkvg2, c.ret2, c.gated2, c.o2,
                      save ? c.Hs2 : nullptr, Hcross_out));
    MAGPO_TRY(g_act_rms_fwd(s, D, R, c.o2, x_rep, pb.ln2, 0, nullptr, nullptr, 0, c.y, nullptr));
    MAGPO_TRY(dense_fwd(s, R, D, 2 * D, c.y, D, pb.ffn_gl, 2 * D, w.d_glT[b], nullptr, c.gl, 2 * D));
    MAGPO_TRY(g_swiglu_fwd(s, D, R, c.gl, c.hmid));
    MAGPO_TRY(dense_fwd(s, R, D, D, c.hmid, D, pb.ffn_out, D, w.d_outT[b], nullptr, c.f, D));
    float* next_pe = b + 1 < sh.nb ? w.dec[b + 1].xpe : nullptr;
    MAGPO_TRY(g_act_rms_fwd(s, D, R, c.f, c.y, pb.ln3, 0, next_pe ? w.pe : nullptr, step, sh.max_step, c.xd, next_pe));
  }
  MAGPO_TRY(head_fwd_g(s, sh, R, w.dec[sh.nb - 1].xd, p.dh0_w, w.dh0T, p.dh0_b, p.dh2_s, p.dh3_w, w.dh3T, p.dh3_b, sh.a, w.zhD, w.hnD, logits));
  return MAGPO_OK;
}

// rows of agent i out of [B, A, width] -> [B, width]
__global__ void gather_agent_k(int64_t B, int A, int i, int width, const float* __restrict__ src, float* __restrict__ dst) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * width) return;
  const int64_t b = idx / width;
  dst[idx] = src[(b * A + i) * width + idx % width];
}
__global__ void gather_agent_i32_k(int64_t B, int A, int i, const int32_t* __restrict__ src, int32_t* __restrict__ dst) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) dst[b] = src[b * A + i];
}
inline unsigned g256(int64_t n) { return (unsigned)ceil_div(n, 256); }

}  // namespace

// rollout.cu: distrax.Categorical(logits=masked).sample_and_log_prob of agent i (decode.py:135-142)
int sample_agent(cudaStream_t s, int64_t B, int A, int i, int a, int gumbel_rows, const float* logits, const uint8_t* mask, const uint32_t* key,
                 int32_t* action, float* log_prob, int32_t* prev_action, float* masked_logits);

size_t sable_g_workspace_bytes(const NetShape& s, int T, int N, bool with_backward) {
  Arena ar(nullptr, SIZE_MAX);
  Ws w;
  w.plan(ar, s, T, N, s.A, with_backward);
  return ar.off;
}

int sable_g_train_forward(cudaStream_t st, const MagpoNetCfg* net, const float* guider, int T, int N, const float* agents_view,
                          const int32_t* step_count, const uint8_t* done, const int32_t* action, const float* h_enc, const float* h_self,
                          const float* h_cross, float* value, float* logits, void* ws, size_t ws_bytes, bool with_backward) {
  const NetShape sh = NetShape::of(net);
  Arena ar(ws, ws_bytes);
  Ws w;
  w.plan(ar, sh, T, N, sh.A, with_backward);
  if (ar.overflow) return MAGPO_ERR_WORKSPACE;
  const GuiderG p = GuiderG::bind(const_cast<float*>(guider), sh);
  MAGPO_TRY(g_pe_table(st, sh.D, sh.max_step, w.pe, net->timestep_pe != 0));
  MAGPO_TRY(transposes(st, sh, p, w));
  MAGPO_TRY(encoder_fwd(st, net, sh, p, w, T, N, agents_view, step_count, done, h_enc, value, with_backward, nullptr));
  const EncActs& last = w.enc[sh.nb - 1];
  MAGPO_TRY(decoder_fwd(st, net, sh, p, w, T, N, sh.A, sh.A, action, last.xout, last.xpe, step_count, done, h_self, h_cross, true, logits,
                        with_backward, nullptr, nullptr));
  return MAGPO_OK;
}

int sable_g_train_backward(cudaStream_t st, const MagpoNetCfg* net, const float* guider, int T, int N, const float* agents_view,
                           const int32_t* step_count, const uint8_t* done, const int32_t* action, const float* h_enc, const float* h_self,
                           const float* h_cross, const float* dlogits, const float* dvalue, float* gflat, void* ws, size_t ws_bytes) {
  (void)step_count; (void)h_enc; (void)h_self; (void)h_cross;
  const NetShape sh = NetShape::of(net);
  const int D = sh.D, A = sh.A;
  const int64_t R = (int64_t)T * N * A;
  Arena ar(ws, ws_bytes);
  Ws w;
  w.plan(ar, sh, T, N, A, true);
  if (ar.overflow) return MAGPO_ERR_WORKSPACE;
  const GuiderG p = GuiderG::bind(const_cast<float*>(guider), sh);
  const GuiderG g = GuiderG::bind(gflat, sh);
  const Kap kap = kappas_of(net, false);
  const EncActs& elast = w.enc[sh.nb - 1];
  // ---- decoder; d(obs_rep) accumulates in dxrep over the blocks (ln2 residual + cross-retention query path)
  MAGPO_CUDA_OK(cudaMemsetAsync(w.dxrep, 0, sizeof(float) * (size_t)R * D, st));
  MAGPO_TRY(head_bwd_g(st, sh, R, w.dec[sh.nb - 1].xd, p.dh0_w, w.dh0T, p.dh2_s, p.dh3_w, w.dh3T, sh.a, w.zhD, w.hnD, dlogits, g.dh0_w, g.dh0_b,
                       g.dh2_s, g.dh3_w, g.dh3_b, w.tX, w.tA, w.tB));  // tX = d(xd of the last block)
  for (int b = sh.nb - 1; b >= 0; --b) {
    const DecActs& c = w.dec[b];
    const DecBlockG& pb = p.dec[b];
    const DecBlockG& gb = g.dec[b];
    // tX = d(xd_b) [for b < nb - 1 it already includes the PE-added copy's gradient: both are the same tensor up to a constant]
    MAGPO_TRY(g_act_rms_bwd(st, D, R, c.f, c.y, pb.ln3, 0, w.tX, nullptr, nullptr, w.tA, gb.ln3));   // tA = d(f) = d(y) residual
    MAGPO_TRY(dense_bwd(st, R, D, D, c.hmid, D, w.tA, D, w.d_outT[b], pb.ffn_out, D, gb.ffn_out, D, nullptr, w.tB, D));
    MAGPO_TRY(g_swiglu_bwd(st, D, R, c.gl, w.tB, w.tG));
    MAGPO_TRY(dense_bwd(st, R, D, 2 * D, c.y, D, w.tG, 2 * D, w.d_glT[b], pb.ffn_gl, 2 * D, gb.ffn_gl, 2 * D, nullptr, w.tB, D));
    MAGPO_TRY(g_act_rms_bwd(st, D, R, c.o2, elast.xout, pb.ln2, 0, w.tA, w.tB, nullptr, w.tD, gb.ln2));  // tD = d(o2) = d(obs_rep) via the residual
    MAGPO_TRY(g_add_rows(st, R * D, w.dxrep, w.tD, w.dxrep));
    // cross retention: query <- obs_rep (+PE), key / value / gate <- r (+PE)
    MAGPO_TRY(msr_bwd(st, sh, kap, T, N, A, true, elast.xpe, c.rpe, pb.r2, w.dt2[b], gb.r2, done, c.qkvg2, c.ret2, c.gated2, c.Hs2, w.tD, w.tE, w.tA,
                      w.tQ, w.tB, w.tC));  // tE = d(obs_rep) via the query, tA = d(r)
    MAGPO_TRY(g_add_rows(st, R * D, w.dxrep, w.tE, w.dxrep));
    MAGPO_TRY(g_act_rms_bwd(st, D, R, c.o1, c.xin, pb.ln1, 0, w.tA, nullptr, nullptr, w.tB, gb.ln1));  // tB = d(o1) = d(xin) residual
    MAGPO_TRY(msr_bwd(st, sh, kap, T, N, A, true, c.xpe, c.xpe, pb.r1, w.dt1[b], gb.r1, done, c.qkvg1, c.ret1, c.gated1, c.Hs1, w.tB, nullptr, w.tA,
                      w.tQ, w.tC, w.tD));  // tA = d(xin + PE)
    MAGPO_TRY(g_add_rows(st, R * D, w.tA, w.tB, w.tX));  // tX = d(block input) = d(xd of block b - 1) or d(xD)
  }
  MAGPO_TRY(g_embed_bwd(st, D, R, A, action, p.Wa, p.dln, w.tX, nullptr, g.Wa, g.dln));
  // ---- encoder: d(obs_rep) = head path + dxrep
  MAGPO_TRY(head_bwd_g(st, sh, R, elast.xout, p.h0_w, w.h0T, p.h2_s, p.h3_w, w.h3T, 1, w.zh, w.hn, dvalue, g.h0_w, g.h0_b, g.h2_s, g.h3_w, g.h3_b,
                       w.tX, w.tA, w.tB));
  MAGPO_TRY(g_add_rows(st, R * D, w.tX, w.dxrep, w.tX));  // tX = d(xout of the last block)
  for (int b = sh.nb - 1; b >= 0; --b) {
    const EncActs& e = w.enc[b];
    const EncBlockG& pb = p.enc[b];
    const EncBlockG& gb = g.enc[b];
    MAGPO_TRY(g_act_rms_bwd(st, D, R, e.f, e.x1, pb.ln2, 0, w.tX, nullptr, nullptr, w.tA, gb.ln2));   // tA = d(f) = d(x1) residual
    MAGPO_TRY(dense_bwd(st, R, D, D, e.hmid, D, w.tA, D, w.e_outT[b], pb.ffn_out, D, gb.ffn_out, D, nullptr, w.tB, D));
    MAGPO_TRY(g_swiglu_bwd(st, D, R, e.gl, w.tB, w.tG));
    MAGPO_TRY(dense_bwd(st, R, D, 2 * D, e.x1, D, w.tG, 2 * D, w.e_glT[b], pb.ffn_gl, 2 * D, gb.ffn_gl, 2 * D, nullptr, w.tB, D));
    MAGPO_TRY(g_act_rms_bwd(st, D, R, e.o, e.xn, pb.ln1, 0, w.tA, w.tB, nullptr, w.tD, gb.ln1));       // tD = d(o) = d(xn) residual
    MAGPO_TRY(msr_bwd(st, sh, kap, T, N, A, false, e.kqv, e.kqv, pb.r, w.et[b], gb.r, done, e.qkvg, e.ret, e.gated, e.Hs, w.tD, nullptr, w.tA, w.tQ,
                      w.tB, w.tC));  // tA = d(kqv) = d(xn) via the retention
    const float* xprev = b == 0 ? w.z0 : w.enc[b - 1].xout;
    MAGPO_TRY(g_act_rms_bwd(st, D, R, xprev, nullptr, p.ln, b == 0 ? ROW_GELU : 0, w.tD, w.tA, nullptr, w.tX, g.ln));  // tX = d(xprev)
  }
  // tX = d(z0)
  MAGPO_TRY(gemm_tn(st, R, D, sh.d, w.on, sh.d, w.tX, D, g.Wobs, D));
  MAGPO_TRY(gemm_nn(st, R, sh.d, D, w.tX, D, wref(w.WobsT, sh.d), nullptr, w.t_d, sh.d, 0));
  MAGPO_TRY(rms_general_bwd_scale(st, R, sh.d, agents_view, w.t_d, g.obs_scale));
  return MAGPO_OK;
}

// ----------------------------------------------------------------------------- inference (SableNetwork.get_actions, :443-482)
namespace {
struct StepWs {
  Ws w;
  float *xrep_i, *xrep_pe_i, *logits_i;
  int32_t *step_i, *prev_action;
  void plan(Arena& ar, const NetShape& s, int B) {
    w.plan(ar, s, 1, B, s.A, false);
    xrep_i = ar.get<float>((size_t)B * s.D);
    xrep_pe_i = ar.get<float>((size_t)B * s.D);
    logits_i = ar.get<float>((size_t)B * s.a);
    step_i = ar.get<int32_t>(B);
    prev_action = ar.get<int32_t>(B);
  }
};
}  // namespace

int sable_g_prepare(cudaStream_t st, const MagpoNetCfg* net, int B, const float* guider, void* ws, size_t ws_bytes) {
  const NetShape sh = NetShape::of(net);
  Arena ar(ws, ws_bytes);
  StepWs sw;
  sw.plan(ar, sh, B);
  if (ar.overflow) return MAGPO_ERR_WORKSPACE;
  const GuiderG p = GuiderG::bind(const_cast<float*>(guider), sh);
  MAGPO_TRY(g_pe_table(st, sh.D, sh.max_step, sw.w.pe, net->timestep_pe != 0));
  return transposes(st, sh, p, sw.w);
}

size_t sable_g_step_workspace_bytes(const NetShape& s, int B) {
  Arena ar(nullptr, SIZE_MAX);
  StepWs w;
  w.plan(ar, s, B);
  return ar.off;
}

int sable_g_get_actions(cudaStream_t st, const MagpoNetCfg* net, int B, int gumbel_rows, const float* guider, const float* agents_view,
                        const uint8_t* action_mask, const int32_t* step_count, const uint8_t* prev_done, const uint32_t* sample_keys,
                        MagpoSableHState hs, bool dry, int32_t* action, float* log_prob, float* value, float* masked_logits, void* ws,
                        size_t ws_bytes, bool prepare) {
  const NetShape sh = NetShape::of(net);
  Arena ar(ws, ws_bytes);
  StepWs sw;
  sw.plan(ar, sh, B);
  if (ar.overflow) return MAGPO_ERR_WORKSPACE;
  const Ws& w = sw.w;
  const GuiderG p = GuiderG::bind(const_cast<float*>(guider), sh);
  const int A = sh.A, D = sh.D;
  if (prepare) MAGPO_TRY(sable_g_prepare(st, net, B, guider, ws, ws_bytes));
  MAGPO_TRY(encoder_fwd(st, net, sh, p, w, 1, B, agents_view, step_count, prev_done, hs.encoder, value, false, dry ? nullptr : hs.encoder));
  if (!action) return MAGPO_OK;
  const EncActs& last = w.enc[sh.nb - 1];
  for (int i = 0; i < A; ++i) {
    gather_agent_k<<<g256((int64_t)B * D), 256, 0, st>>>(B, A, i, D, last.xout, sw.xrep_i);
    MAGPO_LAUNCH_OK();
    gather_agent_k<<<g256((int64_t)B * D), 256, 0, st>>>(B, A, i, D, last.xpe, sw.xrep_pe_i);
    MAGPO_LAUNCH_OK();
    gather_agent_i32_k<<<g256(B), 256, 0, st>>>(B, A, i, step_count, sw.step_i);
    MAGPO_LAUNCH_OK();
    // the once-per-timestep decay (and the reset on done) is applied when the first agent's token arrives
    MAGPO_TRY(decoder_fwd(st, net, sh, p, w, 1, B, 1, i == 0 ? -1 : 0, sw.prev_action, sw.xrep_i, sw.xrep_pe_i, sw.step_i, i == 0 ? prev_done : nullptr,
                          hs.decoder_self, hs.decoder_cross, i == 0, sw.logits_i, false, dry ? nullptr : hs.decoder_self,
                          dry ? nullptr : hs.decoder_cross));
    MAGPO_TRY(sample_agent(st, B, A, i, sh.a, gumbel_rows, sw.logits_i, action_mask, sample_keys + 2 * i, action, log_prob, sw.prev_action,
                           masked_logits));
  }
  return MAGPO_OK;
}

}  // namespace magpo
