// Internal launchers shared by the host-side sequencers (sable.cu, actor.cu, rollout.cu, update.cu).
// Everything works on row-major fp32 activations [rows, C]; a "row" is one token (t, env, agent).
#pragma once
#include "common.cuh"

namespace magpo {

constexpr int kD = 64;   // Sable embed_dim supported by the kernels (configs/network/magpo.yaml:4)
constexpr int kH = 128;  // learner hidden_state_dim / torso width (magpo.yaml:19-31)
constexpr int kMaxActions = 32;
constexpr int kMaxAgents = 8;

enum { GEMM_ACCUMULATE = 1, GEMM_RELU = 2 };

// A weight operand: `w` is [K,N] row-major (leading dimension ldw) for the fp32 SIMT kernel; `wt` (optional) is the
// same matrix transposed, [N,K] row-major (ldwt), whose TF32 hi/lo split has been registered with
// tc_prepare_region() — when present and the shape fits, the GEMM runs on the tcgen05 tensor-core kernel.
struct Wref {
  const float* w;
  int ldw;
  const float* wt;
  int ldwt;
};
inline Wref wref(const float* w, int ldw, const float* wt = nullptr, int ldwt = 0) { return Wref{w, ldw, wt, ldwt}; }

// ---- gemm.cu
int gemm_nn(cudaStream_t s, int64_t M, int N, int K, const float* X, int ldx, Wref W, const float* bias, float* Y,
            int ldy, int flags);
// ---- gemm_tc.cu (tcgen05 + TMA, 3xTF32)
int tc_prepare_region(cudaStream_t s, const float* base, int64_t n, float* hi, float* lo);
bool tc_lookup(const float* w, const float** hi, const float** lo);
bool tc_supported(int64_t M, int N, int K, const float* X, int ldx, const float* Y, int ldy, int ldb);
int gemm_tc(cudaStream_t s, int64_t M, int N, int K, const float* X, int ldx, const float* Bhi, const float* Blo, int ldb,
            const float* bias, float* Y, int ldy, int flags);
bool tc_tn_supported(int64_t M, int N, int K, const float* X, int ldx, const float* dY, int ldy, const float* dW, int ldw);
int gemm_tc_tn(cudaStream_t s, int64_t M, int N, int K, const float* X, int ldx, const float* dY, int ldy, float* dW, int ldw);
// TMA map (CUtensorMap*) of a row-major fp32 [rows, cols] matrix (leading dimension ld): boxes of [box_rows x 32 floats], 128B swizzle
bool tc_make_map(void* tensor_map, const float* ptr, int64_t rows, int cols, int ld, int box_rows);
// the same for a contiguous [T, rows, cols] tensor: boxes of [1, box_rows, 32 floats] that clip at `rows`
bool tc_make_map3(void* tensor_map, const float* ptr, int64_t T, int64_t rows, int cols, int box_rows);
int gemm_tn(cudaStream_t s, int64_t M, int N, int K, const float* X, int ldx, const float* dY, int ldy, float* dW,
            int ldw);
// ---- chain_fwd.cu: fused row chains of the guider's training forward (persistent tcgen05 kernels, A operands in tensor memory)
void chain_set_enabled(bool on);
bool chain_supported(int64_t R);
// gated = swish(g) * GroupNorm(ret); o = gated W1; y = RMSNorm(o + res) * ln_s; ype = y + pe[step] (y / ype optional);
// with W2T: gl = y W2 [R,128]; hmid = swish(gl[:, :64]) * gl[:, 64:].  W1T [64,64], W2T [128,64]: transposed weights with registered images
int chain_gate_fwd(cudaStream_t s, int64_t R, const float* g, int ldg, const float* ret, const float* res, const float* gn_s,
                   const float* gn_b, const float* ln_s, const float* pe, const int32_t* step, int max_step, const float* W1T,
                   const float* W2T, const float* WpT, float* gated, float* o, float* y, float* ype, float* gl, float* hmid, float* proj,
                   int ldproj);
// with WpT [192,64] (instead of W2T): proj[R,192] (row stride ldproj) = ype Wp
// The rows entering the first retention: obs != null: z0 = (RMSNorm_d(obs) * obs_scale) Wobs (d <= 16), x = RMSNorm(gelu(z0)) * ln_s;
// obs == null: x = RMSNorm(gelu(Wa[shifted action token])) * ln_s (A agents per timestep); then xpe = x + pe[step], qkvg[R,256] = xpe Wq
int chain_front_fwd(cudaStream_t s, int64_t R, int d, const float* obs, const float* obs_scale, const float* Wobs, int A, int a,
                    const int32_t* action, const float* Wa, const float* ln_s, const float* pe, const int32_t* step, int max_step,
                    const float* WqT, float* z0, float* x, float* xpe, float* qkvg);
// f = hmid W1; x = RMSNorm(f + res) * ln_s; xpe = x + pe[step] (optional); q = xpe Wq (optional, row stride ldq); zh = x Wh + h_bias;
// out[R,nout] = RMSNorm(gelu(zh)) * h2_s @ W3 + b3
int chain_tail_fwd(cudaStream_t s, int64_t R, const float* hmid, const float* res, const float* ln_s, const float* pe,
                   const int32_t* step, int max_step, const float* W1T, const float* WqT, int ldwq, const float* WhT, const float* h_bias,
                   const float* h2_s, const float* W3, const float* b3, int nout, float* f, float* x, float* xpe, float* q, int ldq,
                   float* zh, float* out);
// ---- gru_scan.cu: persistent tcgen05 GRU scans over T steps (one CTA per 128 rows, W_h streamed through a TMA ring)
int gru_scan_fwd(cudaStream_t s, int T, int N, int A, const float* gi, const float* WhT_hi, const float* WhT_lo, const float* bhn,
                 const uint8_t* done, float* rzn, float* ghn, float* Y, float* HU);
int gru_scan_bwd(cudaStream_t s, int T, int N, int A, const float* dY, const float* rzn, const float* ghn, const float* HU,
                 const uint8_t* done, const float* Wh_hi, const float* Wh_lo, float* dgi, float* dgh, float* dbi /* [384] += colsum(dgi), optional */,
                 float* dbhn /* [128] += colsum(dgh[:, 256:]), optional */);
int colsum(cudaStream_t s, int64_t M, int N, const float* dY, int ldy, float* db);
int transpose(cudaStream_t s, int R, int Cc, const float* in, float* out);

// ---- thin.cu: dense layers with a thin side (K <= 16 or N <= 16), HBM-bound streaming kernels
bool thin_k_ok(int K, int N, int ldw, const float* W, const float* Y, int ldy);
bool thin_n_ok(int K, int N, const float* X, int ldx);
bool obs_embed_ok(int d);
int thin_k_fwd(cudaStream_t s, int64_t R, int K, int N, const float* X, int ldx, const float* W, int ldw, const float* bias,
               float* Y, int ldy, int relu);
int thin_k_bwd(cudaStream_t s, int64_t R, int K, int N, const float* X, int ldx, const float* dY, int lddy, const float* relu_out,
               float* dW, int lddw, float* db);
int thin_n_fwd(cudaStream_t s, int64_t R, int K, int N, const float* X, int ldx, const float* W, int ldw, const float* bias,
               float* Y, int ldy);
// dbx (optional): column sums of the (masked) dX, i.e. the bias gradient of the relu layer that produced X
int thin_n_bwd(cudaStream_t s, int64_t R, int K, int N, const float* X, int ldx, const float* dY, int lddy, const float* W, int ldw,
               int relu_mask, float* dX, int lddx, float* dW, int lddw, float* db, float* dbx);
int obs_embed_fwd(cudaStream_t s, int64_t R, int d, const float* obs, const float* obs_scale, const float* Wobs,
                  const float* ln_scale, const float* pe, const int32_t* step, int max_step, float* on, float* z0, float* xin,
                  float* kqv);
int obs_embed_bwd(cudaStream_t s, int64_t R, int d, const float* obs, const float* obs_scale, const float* Wobs, const float* dz0,
                  float* dWobs, float* dscale);

// ---- rowops.cu (all on 64-wide rows unless noted)
enum { ROW_GELU = 1 };
// on = RMSNorm_d(x) * scale, general width C (the obs encoder's first layer, sable_network.py:93-101)
int rms_general_fwd(cudaStream_t s, int64_t R, int C, const float* x, const float* scale, float* y);
// dscale[c] += sum_r dy[r,c] * x[r,c] * rstd_r   (x is data: no dx)
int rms_general_bwd_scale(cudaStream_t s, int64_t R, int C, const float* x, const float* dy, float* dscale);
// y = RMSNorm((gelu?)(z) + res) * scale ; ype = y + pe[step[row]]   (res, ype, pe optional)
int act_rms_fwd(cudaStream_t s, int64_t R, const float* z, const float* res, const float* scale, int flags,
                const float* pe, const int32_t* step, int max_step, float* y, float* ype);
// dpre from dy = dy1+dy2+dy3 (nullable); out = gelu ? dpre * gelu'(z) : dpre ; dscale accumulated
int act_rms_bwd(cudaStream_t s, int64_t R, const float* z, const float* res, const float* scale, int flags,
                const float* dy1, const float* dy2, const float* dy3, float* dout, float* dscale);
// gated = swish(g) * LayerNorm(ret) (flax GroupNorm with one group, retention.py:289-295). g has row stride ldg.
int gn_gate_fwd(cudaStream_t s, int64_t R, const float* g, int ldg, const float* ret, const float* gn_scale,
                const float* gn_bias, float* gated);
int gn_gate_bwd(cudaStream_t s, int64_t R, const float* g, int ldg, const float* ret, const float* gn_scale,
                const float* gn_bias, const float* dgated, float* dg, int lddg, float* dret, float* dgn_scale,
                float* dgn_bias);
// SwiGLU middle: h = swish(gl[:, :64]) * gl[:, 64:]  (torsos.py:96-99)
int swiglu_fwd(cudaStream_t s, int64_t R, const float* gl, float* h);
int swiglu_bwd(cudaStream_t s, int64_t R, const float* gl, const float* dh, float* dgl);
// out[r, :nout] = RMSNorm(gelu(zh)) * scale @ W3[64,nout] + b3     (head layers 1..3, sable_network.py:102-109,274-283)
int head_fwd(cudaStream_t s, int64_t R, const float* zh, const float* scale, const float* W3, const float* b3,
             int nout, float* out);
// dbz (optional): column sums of dzh, i.e. the bias gradient of the Dense(64) that produced zh
int head_bwd(cudaStream_t s, int64_t R, const float* zh, const float* scale, const float* W3, int nout,
             const float* dout, float* dzh, float* dscale, float* dW3, float* db3, float* dbz);
// decoder input: x = RMSNorm(gelu(Wa[token])) * scale, token = start (0) for the first agent of a timestep else
// 1 + action of the previous token (decode.py:86-108); xpe = x + pe
int embed_fwd(cudaStream_t s, int64_t R, int A, const int32_t* action, const float* Wa, const float* scale,
              const float* pe, const int32_t* step, int max_step, float* x, float* xpe);
int embed_bwd(cudaStream_t s, int64_t R, int A, int a, const int32_t* action, const float* Wa, const float* scale,
              const float* dy1, const float* dy2, float* dWa, float* dscale);
// y = x + pe[step]
int add_pe(cudaStream_t s, int64_t R, const float* x, const float* pe, const int32_t* step, int max_step, float* y);
// enabled == false (memory_config.timestep_positional_encoding: False, retention.py:278,304): an all-zero table, x + 0 = x exactly
int build_pe_table(cudaStream_t s, int max_step, float* pe, bool enabled = true);
int fill_f32(cudaStream_t s, float* p, int64_t n, float v);

// ---- retention.cu : recurrent-form retention over per-env sequences, rows ordered (t, env, agent)
// q,k,v: column blocks of a packed buffer with row stride ld. H0 [N,64,64] initial state (un-decayed,
// as stored in the learner state); done [T,N] resets. Hsave (optional) [T,N,64,64] = state after each timestep.
// Hout (optional) [N,64,64] final state. causal: decoder (masked=True) vs encoder (block-full over agents).
// For T > 1 the chunkwise tensor-core kernels (retention_chunk.cu) run instead of the scan and Hsave holds only the
// state entering each chunk: [retention_num_chunks(T, A), N, 64, 64].
int retention_chunk_len(int A);
int retention_num_chunks(int T, int A);
int retention_fwd(cudaStream_t s, int T, int N, int A, float kappa, bool causal, const float* q, const float* k,
                  const float* v, int ld, const float* H0, const uint8_t* done, float* ret, float* Hsave,
                  float* Hout);
int retention_bwd(cudaStream_t s, int T, int N, int A, float kappa, bool causal, const float* q, const float* k,
                  const float* v, int ld, const float* H0, const uint8_t* done, const float* Hsave,
                  const float* dret, float* dq, float* dk, float* dv, int ldd);

}  // namespace magpo
