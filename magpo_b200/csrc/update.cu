// The update step of rec_magpo.py:214-499 behind the C ABI: per-epoch shuffle indices, minibatch gather,
// guider + learner forward/backward with the MAGPO losses.  All U update-batch slots of a minibatch are
// processed as one batch: the per-slot losses are means over equally many tokens, so the mean over slots of
// the per-slot gradients (the pmean over "batch", :395-405) is the gradient of the token mean over all slots;
// only the advantage normalisation is per slot (:283,356).
#include <stdlib.h>
#include "update.cuh"

#include <string.h>

#include "actor.cuh"
#include "generic.cuh"
#include "prng.cuh"
#include "sable.cuh"

extern "C" int magpo_prng_permutation(magpo_stream_t s, const uint32_t* key, int32_t n, int32_t* out, uint32_t* scratch);

namespace magpo {
namespace {

// key, batch_key, agent_key, entropy_key = split(key, 4)   (rec_magpo.py:439)
__global__ void split4_kernel(uint32_t* __restrict__ key, uint32_t* __restrict__ sub /*[2][2]: batch, agent*/) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const uint32_t k0 = key[0], k1 = key[1];
  uint32_t n0, n1;
  prng_split_i(k0, k1, 0u, n0, n1);
  prng_split_i(k0, k1, 1u, sub[0], sub[1]);
  prng_split_i(k0, k1, 2u, sub[2], sub[3]);
  key[0] = n0;
  key[1] = n1;
}

// env_index / hs_index / env_slot for every minibatch of the epoch, laid out [M][U][N].
__global__ void epoch_index_kernel(int E, int U, int M, const int32_t* __restrict__ batch_perm,
                                   int32_t* __restrict__ hs_perm, int first_epoch, int32_t* __restrict__ hs_perm_new,
                                   int32_t* __restrict__ env_index, int32_t* __restrict__ hs_index,
                                   int32_t* __restrict__ env_slot) {
  const int N = E / M;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * U * N) return;
  const int j = idx % N, u = (idx / N) % U, m = idx / (N * U);
  const int pos = m * N + j;
  const int bp = batch_perm[pos];
  // prev_hstates carries every earlier epoch's permutation (rec_magpo.py:447,471): new[i] = old[batch_perm[i]]
  const int hp = first_epoch ? bp : hs_perm[bp];
  env_index[idx] = u * E + bp;
  hs_index[idx] = u * E + hp;
  env_slot[idx] = u;
  if (u == 0) hs_perm_new[pos] = hp;
}

// One warp per output row (t, n, i): gathers env env_index[n], agent agent_perm[i] of the trajectory.
__global__ void __launch_bounds__(256)
pack_rows_kernel(int T, int B, int A, int d, int a, int n_env, MagpoTrajectory tr, const float* __restrict__ adv,
                 const float* __restrict__ tgt, const int32_t* __restrict__ env_index,
                 const int32_t* __restrict__ agent_perm, float* __restrict__ o_view, uint8_t* __restrict__ o_mask,
                 int32_t* __restrict__ o_step, uint8_t* __restrict__ o_done, int32_t* __restrict__ o_action,
                 float* __restrict__ o_value, float* __restrict__ o_logp, float* __restrict__ o_adv,
                 float* __restrict__ o_tgt) {
  const int lane = threadIdx.x & 31;
  const int64_t R = (int64_t)T * n_env * A;
  const int64_t wstride = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < R; row += wstride) {
    const int i = (int)(row % A);
    const int n = (int)((row / A) % n_env);
    const int t = (int)(row / ((int64_t)A * n_env));
    const int b = env_index[n], ai = agent_perm ? agent_perm[i] : i;
    const int64_t src = ((int64_t)t * B + b) * A + ai;
    for (int c = lane; c < d; c += 32) o_view[row * d + c] = tr.agents_view[src * d + c];
    for (int c = lane; c < a; c += 32) o_mask[row * a + c] = tr.action_mask[src * a + c];
    if (lane == 0) {
      o_step[row] = tr.step_count[src];
      o_action[row] = tr.action[src];
      o_value[row] = tr.value[src];
      o_logp[row] = tr.log_prob[src];
      o_adv[row] = adv[src];
      o_tgt[row] = tgt[src];
      if (i == 0) o_done[(int64_t)t * n_env + n] = tr.done[(int64_t)t * B + b];
    }
  }
}

// Same gather with one thread per output row, for narrow observations (d <= 16): all 32 lanes issue the per-row scalars and
// the 4d-byte observation, so consecutive rows (the agents of one env, then the next env of the minibatch) coalesce.
__global__ void __launch_bounds__(256)
pack_rows_narrow_kernel(int T, int B, int A, int d, int a, int n_env, MagpoTrajectory tr, const float* __restrict__ adv,
                        const float* __restrict__ tgt, const int32_t* __restrict__ env_index,
                        const int32_t* __restrict__ agent_perm, float* __restrict__ o_view, uint8_t* __restrict__ o_mask,
                        int32_t* __restrict__ o_step, uint8_t* __restrict__ o_done, int32_t* __restrict__ o_action,
                        float* __restrict__ o_value, float* __restrict__ o_logp, float* __restrict__ o_adv,
                        float* __restrict__ o_tgt) {
  const int64_t R = (int64_t)T * n_env * A;
  for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < R; row += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(row % A);
    const int n = (int)((row / A) % n_env);
    const int t = (int)(row / ((int64_t)A * n_env));
    const int b = __ldg(env_index + n), ai = agent_perm ? __ldg(agent_perm + i) : i;
    const int64_t src = ((int64_t)t * B + b) * A + ai;
    const int32_t st = tr.step_count[src], ac = tr.action[src];
    const float va = tr.value[src], lp = tr.log_prob[src], ad = adv[src], tg = tgt[src];
    if ((d & 3) == 0) {
      for (int c = 0; c < d; c += 4)
        *reinterpret_cast<float4*>(o_view + row * d + c) = *reinterpret_cast<const float4*>(tr.agents_view + src * d + c);
    } else {
      for (int c = 0; c < d; ++c) o_view[row * d + c] = tr.agents_view[src * d + c];
    }
    for (int c = 0; c < a; ++c) o_mask[row * a + c] = tr.action_mask[src * a + c];
    o_step[row] = st; o_action[row] = ac; o_value[row] = va; o_logp[row] = lp; o_adv[row] = ad; o_tgt[row] = tg;
    if (i == 0) o_done[(int64_t)t * n_env + n] = tr.done[(int64_t)t * B + b];
  }
}

__global__ void __launch_bounds__(256)
pack_hidden_kernel(int A, int n_env, int quads /* float4 per env state */, const float* __restrict__ policy_h0, const float* __restrict__ h_enc,
                   const float* __restrict__ h_self, const float* __restrict__ h_cross,
                   const int32_t* __restrict__ env_index, const int32_t* __restrict__ hs_index,
                   const int32_t* __restrict__ agent_perm, float* __restrict__ o_h0, float* __restrict__ o_enc,
                   float* __restrict__ o_self, float* __restrict__ o_cross) {
  const int n = blockIdx.x;
  const int b = env_index[n], hb = hs_index[n];
  for (int idx = threadIdx.x; idx < A * kH; idx += blockDim.x) {
    const int i = idx / kH, c = idx % kH;
    o_h0[((int64_t)n * A + i) * kH + c] = policy_h0[((int64_t)b * A + agent_perm[i]) * kH + c];
  }
  const float4* se = reinterpret_cast<const float4*>(h_enc) + (int64_t)hb * quads;
  const float4* ss = reinterpret_cast<const float4*>(h_self) + (int64_t)hb * quads;
  const float4* sc = reinterpret_cast<const float4*>(h_cross) + (int64_t)hb * quads;
  float4* de = reinterpret_cast<float4*>(o_enc) + (int64_t)n * quads;
  float4* ds = reinterpret_cast<float4*>(o_self) + (int64_t)n * quads;
  float4* dc = reinterpret_cast<float4*>(o_cross) + (int64_t)n * quads;
  for (int idx = threadIdx.x; idx < quads; idx += blockDim.x) {
    de[idx] = se[idx];
    ds[idx] = ss[idx];
    dc[idx] = sc[idx];
  }
}

struct UpdateWs {
  GuiderT gt;
  ActorT at;
  SableActs sa;
  ActorActs aa;
  float *pe, *lg, *ll, *value, *dlg, *dll, *dvalue;
  float *g_hi, *g_lo, *a_hi, *a_lo;  // TF32 hi/lo images of the two flat parameter buffers (dX operands)
  void* gws;  // general guider shapes (generic.cuh): the workspace of sable_g_train_forward / backward
  size_t gws_bytes;
  void plan(Arena& ar, const MagpoNetCfg* net, int T, int N, bool with_backward) {
    const int A = net->n_agents, a = net->action_dim, d = net->obs_dim;
    const int64_t Rs = (int64_t)N * A, R = Rs * T;
    const NetShape shape = NetShape::of(net);
    gws = nullptr; gws_bytes = 0;
    const int64_t n_a = ActorP::bind(nullptr, d, a).total;
    if (shape.is_default()) {  // (the forward-only and the backward plan agree on every offset up to the backward-only buffers)
      gt.plan(ar, d);
      at.plan(ar, a);
      const int64_t n_g = GuiderP::bind(nullptr, d, a).total;
      g_hi = ar.get<float>((size_t)n_g); g_lo = ar.get<float>((size_t)n_g);
      a_hi = ar.get<float>((size_t)n_a); a_lo = ar.get<float>((size_t)n_a);
      sa.plan(ar, R, (int64_t)T * N, d, with_backward);
      aa.plan(ar, R, Rs, a, with_backward);
    } else {
      at.plan(ar, a);
      a_hi = ar.get<float>((size_t)n_a); a_lo = ar.get<float>((size_t)n_a);
      aa.plan(ar, R, Rs, a, with_backward);
      g_hi = g_lo = nullptr;
      gws_bytes = sable_g_workspace_bytes(shape, T, N, with_backward);
      gws = ar.get<char>(gws_bytes);
    }
    pe = ar.get<float>((size_t)(net->max_step_count + 1) * kD);
    lg = ar.get<float>((size_t)R * a);
    ll = ar.get<float>((size_t)R * a);
    value = ar.get<float>(R);
    if (with_backward) {
      dlg = ar.get<float>((size_t)R * a);
      dll = ar.get<float>((size_t)R * a);
      dvalue = ar.get<float>(R);
    } else {
      dlg = dll = dvalue = nullptr;
    }
  }
};

SableBatch make_batch(const MagpoNetCfg* net, const MagpoMinibatch& mb, const float* pe) {
  SableBatch b;
  b.T = mb.T; b.N = mb.N; b.A = net->n_agents; b.d = net->obs_dim; b.a = net->action_dim;
  b.max_step = net->max_step_count;
  b.agents_view = mb.agents_view; b.step_count = mb.step_count; b.done = mb.done; b.action = mb.action;
  b.h_enc = mb.sable_h0.encoder; b.h_self = mb.sable_h0.decoder_self; b.h_cross = mb.sable_h0.decoder_cross;
  b.pe = pe;
  b.kappa = net_kappa(net);
  return b;
}

int check_mb(const MagpoMinibatch& mb) {
  if (mb.T < 1 || mb.N < 1 || !mb.agents_view || !mb.action_mask || !mb.step_count || !mb.done || !mb.action ||
      !mb.sable_h0.encoder || !mb.sable_h0.decoder_self || !mb.sable_h0.decoder_cross)
    return MAGPO_ERR_ARG;
  return MAGPO_OK;
}

__global__ void mask_logits_kernel(int64_t n, const uint8_t* __restrict__ mask, float* __restrict__ logits) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && !mask[i]) logits[i] = kF32Min;
}

}  // namespace

int epoch_index(cudaStream_t s, int E, int U, int M, const int32_t* batch_perm, int32_t* hs_perm, int first_epoch, int32_t* hs_perm_new,
                int32_t* env_index, int32_t* hs_index, int32_t* env_slot) {
  const int total = M * U * (E / M);
  epoch_index_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(E, U, M, batch_perm, hs_perm, first_epoch, hs_perm_new, env_index,
                                                                   hs_index, env_slot);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

int pack_rows(cudaStream_t s, const MagpoNetCfg* net, const MagpoSysCfg* sys, const MagpoTrajectory& traj, const float* advantages,
              const float* targets, const int32_t* env_index, const int32_t* agent_perm, int n_env, const MagpoMinibatch& out) {
  const int A = net->n_agents, T = sys->rollout_length, B = sys->update_batch_size * sys->num_envs;
  const int64_t R = (int64_t)T * n_env * A;
  const bool narrow = net->obs_dim <= 16;
  (narrow ? pack_rows_narrow_kernel : pack_rows_kernel)<<<(unsigned)std::min<int64_t>(ceil_div(R, narrow ? 256 : 8), (int64_t)kNumSMs * 16), 256, 0, s>>>(
      T, B, A, net->obs_dim, net->action_dim, n_env, traj, advantages, targets, env_index, agent_perm,
      const_cast<float*>(out.agents_view), const_cast<uint8_t*>(out.action_mask), const_cast<int32_t*>(out.step_count),
      const_cast<uint8_t*>(out.done), const_cast<int32_t*>(out.action), const_cast<float*>(out.value),
      const_cast<float*>(out.log_prob), const_cast<float*>(out.advantages), const_cast<float*>(out.targets));
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

}  // namespace magpo

using namespace magpo;

extern "C" {

int magpo_epoch_indices(magpo_stream_t s_, const MagpoSysCfg* sys, int32_t A, uint32_t* key, int32_t* hs_perm,
                        int32_t first_epoch, int32_t* batch_perm, int32_t* agent_perm, int32_t* env_index,
                        int32_t* hs_index, int32_t* env_slot, uint32_t* scratch) {
  if (!sys || !key || !hs_perm || !batch_perm || !agent_perm || !env_index || !hs_index || !env_slot || !scratch)
    return MAGPO_ERR_ARG;
  const int E = sys->num_envs, U = sys->update_batch_size, M = sys->num_minibatches;
  if (E < 1 || M < 1 || E % M || A < 1) return MAGPO_ERR_ARG;
  cudaStream_t s = as_stream(s_);
  uint32_t* sub = scratch;                      // [4]
  uint32_t* pscr = scratch + 4;                 // [2*max(E,A)]
  int32_t* hs_new = reinterpret_cast<int32_t*>(scratch + 4 + 2 * (size_t)max(E, A));  // [E]
  split4_kernel<<<1, 32, 0, s>>>(key, sub);
  MAGPO_LAUNCH_OK();
  MAGPO_TRY(magpo_prng_permutation(s_, sub, E, batch_perm, pscr));
  MAGPO_TRY(magpo_prng_permutation(s_, sub + 2, A, agent_perm, pscr));
  MAGPO_TRY(epoch_index(s, E, U, M, batch_perm, hs_perm, first_epoch, hs_new, env_index, hs_index, env_slot));
  MAGPO_CUDA_OK(cudaMemcpyAsync(hs_perm, hs_new, sizeof(int32_t) * E, cudaMemcpyDeviceToDevice, s));
  return MAGPO_OK;
}

int magpo_adv_stats(magpo_stream_t s_, int32_t T, int32_t B, int32_t A, const float* advantages,
                    const int32_t* env_index, int32_t n_env, int32_t U, void* scratch, float* stats) {
  if (!advantages || !env_index || !scratch || !stats) return MAGPO_ERR_ARG;
  return adv_stats(as_stream(s_), T, B, A, advantages, env_index, n_env, U, static_cast<double*>(scratch), stats);
}

int magpo_pack_minibatch(magpo_stream_t s_, const MagpoNetCfg* net, const MagpoSysCfg* sys, MagpoTrajectory traj,
                         const float* advantages, const float* targets, const int32_t* env_index,
                         const int32_t* hs_index, const int32_t* agent_perm, int32_t n_env, MagpoMinibatch out) {
  MAGPO_TRY(check_net(net));
  if (!sys || !advantages || !targets || !env_index || !hs_index || !agent_perm || n_env < 1) return MAGPO_ERR_ARG;
  if (out.T != sys->rollout_length || out.N != n_env) return MAGPO_ERR_ARG;
  cudaStream_t s = as_stream(s_);
  const int A = net->n_agents, T = sys->rollout_length;
  const int64_t R = (int64_t)T * n_env * A;
  ProfScope ps(PROF_PACK, s, 2.0 * (double)R * (4.0 * net->obs_dim + net->action_dim + 24.0) + 2.0 * n_env * (3 * 16384.0 + 512.0 * A));
  MAGPO_TRY(pack_rows(s, net, sys, traj, advantages, targets, env_index, agent_perm, n_env, out));
  pack_hidden_kernel<<<n_env, 256, 0, s>>>(A, n_env, (int)(NetShape::of(net).state_elems() / 4), traj.policy_h0, traj.sable_h0.encoder, traj.sable_h0.decoder_self,
                                           traj.sable_h0.decoder_cross, env_index, hs_index, agent_perm,
                                           const_cast<float*>(out.policy_h0), out.sable_h0.encoder,
                                           out.sable_h0.decoder_self, out.sable_h0.decoder_cross);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

size_t magpo_update_workspace_bytes(const MagpoNetCfg* net, int32_t T, int32_t N) {
  if (check_net(net) != MAGPO_OK || T < 1 || N < 1) return 0;
  Arena ar(nullptr, SIZE_MAX);
  UpdateWs w;
  w.plan(ar, net, T, N, true);
  return ar.off;
}

namespace {
// The guider and the learner are independent until the losses (which need both logits) and again after them. The learner's
// persistent GRU scans are latency chains on <= 96 of the 148 SMs, so its forward / backward run on the context's `side` stream and
// the guider's streaming kernels fill the idle SMs and HBM bandwidth meanwhile.
bool g_overlap_nets = true;
}  // namespace

}  // extern "C"
namespace magpo {
bool nets_overlap_enabled() { return g_overlap_nets; }
}  // namespace magpo
extern "C" {

int magpo_debug_set_overlap(int on) {
  g_overlap_nets = on != 0;
  return MAGPO_OK;
}

int magpo_minibatch_grads(MagpoContext* ctx_, magpo_stream_t s_, const MagpoNetCfg* net, const MagpoSysCfg* sys, const float* guider,
                          const float* actor, MagpoMinibatch mb, const int32_t* env_slot, const float* adv_stats_,
                          float inv_tokens, float* grads, int32_t reduce_grads, void* workspace, size_t workspace_bytes) {
  MAGPO_CTX(ctx_);
  MAGPO_TRY(check_net(net));
  MAGPO_TRY(check_mb(mb));
  if (!sys || !guider || !actor || !env_slot || !adv_stats_ || !grads || !workspace || !mb.value || !mb.log_prob ||
      !mb.advantages || !mb.targets || !mb.policy_h0)
    return MAGPO_ERR_ARG;
  cudaStream_t s = as_stream(s_);
  const int A = net->n_agents, a = net->action_dim, d = net->obs_dim, T = mb.T, N = mb.N;
  const int64_t R = (int64_t)T * N * A;
  Arena ar(workspace, workspace_bytes);
  UpdateWs w;
  w.plan(ar, net, T, N, true);
  if (ar.overflow) return MAGPO_ERR_WORKSPACE;
  const NetShape shape = NetShape::of(net);
  const bool general = !shape.is_default();
  GuiderP gp = GuiderP::bind(const_cast<float*>(guider), d, a);
  if (general) gp.total = GuiderG::bind(nullptr, shape).total;  // the general layout's length; the default structs are not used then
  const ActorP ap = ActorP::bind(const_cast<float*>(actor), d, a);
  const GuiderP gg = GuiderP::bind(grads, d, a);
  const ActorP ag = ActorP::bind(grads + gp.total, d, a);
  float* loss_sums = grads + gp.total + ap.total;
  MAGPO_TRY(actor_transpose(s, ap, w.at, a));
  if (!general) {
    MAGPO_TRY(build_pe_table(s, net->max_step_count, w.pe, net->timestep_pe != 0));
    MAGPO_TRY(guider_transpose(s, gp, w.gt, d));
  }
  if (!general) MAGPO_TRY(tc_prepare_region(s, guider, gp.total, w.g_hi, w.g_lo));
  MAGPO_TRY(tc_prepare_region(s, actor, ap.total, w.a_hi, w.a_lo));
  const SableBatch b = make_batch(net, mb, w.pe);
  const bool sable_only = sys->sable_only != 0;
  const bool overlap = g_overlap_nets && !sable_only;
  cudaStream_t s2 = s, sg = s;  // learner stream, guider stream
  ForkJoin& g_side = ctx().side;
  if (overlap) {
    s2 = g_side.s;
    MAGPO_CUDA_OK(cudaEventRecord(g_side.fork, s));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(g_side.s, g_side.fork, 0));
  }
  if (!sable_only)
    MAGPO_TRY(actor_forward(s2, ap, &w.at, T, N, A, d, a, mb.agents_view, mb.done, mb.policy_h0, w.aa, w.ll, nullptr));
  if (general)
    MAGPO_TRY(sable_g_train_forward(sg, net, guider, T, N, mb.agents_view, mb.step_count, mb.done, mb.action, mb.sable_h0.encoder,
                                    mb.sable_h0.decoder_self, mb.sable_h0.decoder_cross, w.value, w.lg, w.gws, w.gws_bytes, true));
  else
    MAGPO_TRY(sable_train_forward(sg, gp, &w.gt, b, w.sa, w.value, w.lg, true));
  if (overlap) {
    MAGPO_CUDA_OK(cudaEventRecord(g_side.join, g_side.s));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(s, g_side.join, 0));
  }
  // rec_sable: the learner's masked logits are the guider's own (constants to the gradient): the guidance KL vanishes and the
  // double clip of the MAGPO ratio collapses to the PPO clip (rec_sable.py:196-226)
  MAGPO_TRY(magpo_losses(s, R, N, A, a, sys, inv_tokens, w.lg, sable_only ? w.lg : w.ll, mb.action_mask, mb.action, mb.log_prob,
                         mb.advantages, w.value, mb.value, mb.targets, env_slot, adv_stats_, w.dlg, w.dll, w.dvalue,
                         loss_sums));
  if (overlap) {
    MAGPO_CUDA_OK(cudaEventRecord(g_side.fork, s));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(g_side.s, g_side.fork, 0));
  }
  if (!sable_only) MAGPO_TRY(actor_backward(s2, ap, w.at, T, N, A, d, a, mb.agents_view, mb.done, w.aa, w.dll, ag));
  // pmean over "device" (rec_magpo.py:399-409), issued where the gradients are produced: the learner's half (+ the 8 loss sums, which
  // lie behind it) as soon as the learner's backward is done — on its own stream, under the guider's remaining backward — and the
  // guider's half at the end. Every rank issues the two all-reduces in this order.
  MagpoComm* comm = reduce_grads ? ctx().comm : nullptr;
  if (comm) MAGPO_TRY(comm_allreduce(comm, s2, grads + gp.total, ap.total + 8, 0));
  if (general)
    MAGPO_TRY(sable_g_train_backward(sg, net, guider, T, N, mb.agents_view, mb.step_count, mb.done, mb.action, mb.sable_h0.encoder,
                                     mb.sable_h0.decoder_self, mb.sable_h0.decoder_cross, w.dlg, w.dvalue, grads, w.gws, w.gws_bytes));
  else
    MAGPO_TRY(sable_train_backward(sg, gp, w.gt, b, w.sa, w.dlg, w.dvalue, gg));
  if (comm) MAGPO_TRY(comm_allreduce(comm, sg, grads, gp.total, 0));
  if (overlap) {
    MAGPO_CUDA_OK(cudaEventRecord(g_side.join, g_side.s));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(s, g_side.join, 0));
  }
  return MAGPO_OK;
}

int magpo_guider_forward(MagpoContext* ctx_, magpo_stream_t s_, const MagpoNetCfg* net, const float* guider, MagpoMinibatch mb,
                         float* value, float* logits, void* workspace, size_t workspace_bytes) {
  MAGPO_CTX(ctx_);
  MAGPO_TRY(check_net(net));
  MAGPO_TRY(check_mb(mb));
  if (!guider || !value || !logits || !workspace) return MAGPO_ERR_ARG;
  cudaStream_t s = as_stream(s_);
  Arena ar(workspace, workspace_bytes);
  UpdateWs w;
  w.plan(ar, net, mb.T, mb.N, false);
  if (ar.overflow) return MAGPO_ERR_WORKSPACE;
  if (w.gws) {
    MAGPO_TRY(sable_g_train_forward(s, net, guider, mb.T, mb.N, mb.agents_view, mb.step_count, mb.done, mb.action, mb.sable_h0.encoder,
                                    mb.sable_h0.decoder_self, mb.sable_h0.decoder_cross, value, logits, w.gws, w.gws_bytes, false));
  } else {
    const GuiderP gp = GuiderP::bind(const_cast<float*>(guider), net->obs_dim, net->action_dim);
    MAGPO_TRY(build_pe_table(s, net->max_step_count, w.pe, net->timestep_pe != 0));
    const SableBatch b = make_batch(net, mb, w.pe);
    MAGPO_TRY(sable_train_forward(s, gp, nullptr, b, w.sa, value, logits, false));
  }
  const int64_t n = (int64_t)mb.T * mb.N * net->n_agents * net->action_dim;
  mask_logits_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(n, mb.action_mask, logits);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

int magpo_actor_forward(MagpoContext* ctx_, magpo_stream_t s_, const MagpoNetCfg* net, const float* actor, MagpoMinibatch mb,
                        float* logits, void* workspace, size_t workspace_bytes) {
  MAGPO_CTX(ctx_);
  MAGPO_TRY(check_net(net));
  if (!actor || !logits || !workspace || !mb.agents_view || !mb.done || !mb.policy_h0 || !mb.action_mask)
    return MAGPO_ERR_ARG;
  cudaStream_t s = as_stream(s_);
  Arena ar(workspace, workspace_bytes);
  UpdateWs w;
  w.plan(ar, net, mb.T, mb.N, false);
  if (ar.overflow) return MAGPO_ERR_WORKSPACE;
  const ActorP ap = ActorP::bind(const_cast<float*>(actor), net->obs_dim, net->action_dim);
  MAGPO_TRY(actor_forward(s, ap, nullptr, mb.T, mb.N, net->n_agents, net->obs_dim, net->action_dim, mb.agents_view, mb.done,
                          mb.policy_h0, w.aa, logits, nullptr));
  const int64_t n = (int64_t)mb.T * mb.N * net->n_agents * net->action_dim;
  mask_logits_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(n, mb.action_mask, logits);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

// Test hook: byte offset inside the update workspace of a saved activation (same plan as magpo_minibatch_grads),
// so that parity tests can compare intermediates with the oracle after a call. Returns -1 for unknown names.
int64_t magpo_debug_buffer_offset(const MagpoNetCfg* net, int32_t T, int32_t N, const char* name) {
  if (check_net(net) != MAGPO_OK || !name || !NetShape::of(net).is_default()) return -1;
  Arena ar(nullptr, SIZE_MAX);
  UpdateWs w;
  w.plan(ar, net, T, N, true);
  struct { const char* n; const void* p; } tab[] = {
      {"on", w.sa.on}, {"z0", w.sa.z0}, {"xin", w.sa.xin}, {"kqv", w.sa.kqv}, {"qkvg", w.sa.qkvg}, {"ret", w.sa.ret},
      {"gated", w.sa.gated}, {"o", w.sa.o}, {"x1", w.sa.x1}, {"gl", w.sa.gl}, {"hmid", w.sa.hmid}, {"f", w.sa.f},
      {"x", w.sa.x}, {"xpe", w.sa.xpe}, {"zh", w.sa.zh}, {"xD", w.sa.xD}, {"xpeD", w.sa.xpeD}, {"qkvg1", w.sa.qkvg1},
      {"ret1", w.sa.ret1}, {"gated1", w.sa.gated1}, {"o1", w.sa.o1}, {"rpe", w.sa.rpe}, {"qkvg2", w.sa.qkvg2},
      {"ret2", w.sa.ret2}, {"gated2", w.sa.gated2}, {"o2", w.sa.o2}, {"y", w.sa.y}, {"glD", w.sa.glD},
      {"hmidD", w.sa.hmidD}, {"fD", w.sa.fD}, {"xd", w.sa.xd}, {"zhD", w.sa.zhD}, {"Hs_enc", w.sa.Hs_enc},
      {"Hs_self", w.sa.Hs_self}, {"Hs_cross", w.sa.Hs_cross}, {"e", w.aa.e}, {"HU", w.aa.HU}, {"Y", w.aa.Y},
      {"post", w.aa.post}, {"rzn", w.aa.rzn}, {"ghn", w.aa.ghn}, {"lg", w.lg}, {"ll", w.ll}, {"value", w.value},
      {"dlg", w.dlg}, {"dll", w.dll}, {"dvalue", w.dvalue}, {"pe", w.pe}};
  for (auto& e : tab)
    if (strcmp(e.n, name) == 0) return (int64_t)reinterpret_cast<uintptr_t>(e.p);
  return -1;
}

// ------------------------------------------------------------------ parameter table (flax tree paths)
struct ParamEntry {
  const char* name;
  int64_t offset;
  int32_t dim0, dim1, ld;
};

static int guider_table(const MagpoNetCfg* net, ParamEntry* out) {
  const int d = net->obs_dim, a = net->action_dim;
  GuiderP p = GuiderP::bind(reinterpret_cast<float*>(sizeof(float)), d, a);  // fake base: pointer arithmetic -> offsets
  auto off = [](const float* q) { return (int64_t)(reinterpret_cast<uintptr_t>(q) / sizeof(float)) - 1; };
  int n = 0;
  auto add = [&](const char* name, const float* q, int64_t extra, int r, int c, int ld) {
    if (out) out[n] = ParamEntry{name, off(q) + extra, r, c, ld};
    ++n;
  };
  add("encoder/obs_encoder/layers_0/scale", p.obs_scale, 0, d, 0, 1);
  add("encoder/obs_encoder/layers_1/kernel", p.Wobs, 0, d, kD, kD);
  add("encoder/ln/scale", p.ln, 0, kD, 0, 1);
  add("encoder/encoder_block_0/ln1/scale", p.ln1, 0, kD, 0, 1);
  add("encoder/encoder_block_0/ln2/scale", p.ln2, 0, kD, 0, 1);
  add("encoder/encoder_block_0/retn/retention_heads_0/w_q", p.qkvg, 0, kD, kD, 4 * kD);
  add("encoder/encoder_block_0/retn/retention_heads_0/w_k", p.qkvg, kD, kD, kD, 4 * kD);
  add("encoder/encoder_block_0/retn/retention_heads_0/w_v", p.qkvg, 2 * kD, kD, kD, 4 * kD);
  add("encoder/encoder_block_0/retn/w_g", p.qkvg, 3 * kD, kD, kD, 4 * kD);
  add("encoder/encoder_block_0/retn/w_o", p.wo, 0, kD, kD, kD);
  add("encoder/encoder_block_0/retn/group_norm/scale", p.gn_s, 0, kD, 0, 1);
  add("encoder/encoder_block_0/retn/group_norm/bias", p.gn_b, 0, kD, 0, 1);
  add("encoder/encoder_block_0/ffn/W_gate", p.ffn_gl, 0, kD, kD, 2 * kD);
  add("encoder/encoder_block_0/ffn/W_linear", p.ffn_gl, kD, kD, kD, 2 * kD);
  add("encoder/encoder_block_0/ffn/W_output", p.ffn_out, 0, kD, kD, kD);
  add("encoder/head/layers_0/kernel", p.h0_w, 0, kD, kD, kD);
  add("encoder/head/layers_0/bias", p.h0_b, 0, kD, 0, 1);
  add("encoder/head/layers_2/scale", p.h2_s, 0, kD, 0, 1);
  add("encoder/head/layers_3/kernel", p.h3_w, 0, kD, 1, 1);
  add("encoder/head/layers_3/bias", p.h3_b, 0, 1, 0, 1);
  add("decoder/action_encoder/layers_0/kernel", p.Wa, 0, a + 1, kD, kD);
  add("decoder/ln/scale", p.dln, 0, kD, 0, 1);
  add("decoder/decoder_block_0/ln1/scale", p.dln1, 0, kD, 0, 1);
  add("decoder/decoder_block_0/ln2/scale", p.dln2, 0, kD, 0, 1);
  add("decoder/decoder_block_0/ln3/scale", p.dln3, 0, kD, 0, 1);
  add("decoder/decoder_block_0/retn1/retention_heads_0/w_q", p.qkvg1, 0, kD, kD, 4 * kD);
  add("decoder/decoder_block_0/retn1/retention_heads_0/w_k", p.qkvg1, kD, kD, kD, 4 * kD);
  add("decoder/decoder_block_0/retn1/retention_heads_0/w_v", p.qkvg1, 2 * kD, kD, kD, 4 * kD);
  add("decoder/decoder_block_0/retn1/w_g", p.qkvg1, 3 * kD, kD, kD, 4 * kD);
  add("decoder/decoder_block_0/retn1/w_o", p.wo1, 0, kD, kD, kD);
  add("decoder/decoder_block_0/retn1/group_norm/scale", p.gn1_s, 0, kD, 0, 1);
  add("decoder/decoder_block_0/retn1/group_norm/bias", p.gn1_b, 0, kD, 0, 1);
  add("decoder/decoder_block_0/retn2/retention_heads_0/w_q", p.qkvg2, 0, kD, kD, 4 * kD);
  add("decoder/decoder_block_0/retn2/retention_heads_0/w_k", p.qkvg2, kD, kD, kD, 4 * kD);
  add("decoder/decoder_block_0/retn2/retention_heads_0/w_v", p.qkvg2, 2 * kD, kD, kD, 4 * kD);
  add("decoder/decoder_block_0/retn2/w_g", p.qkvg2, 3 * kD, kD, kD, 4 * kD);
  add("decoder/decoder_block_0/retn2/w_o", p.wo2, 0, kD, kD, kD);
  add("decoder/decoder_block_0/retn2/group_norm/scale", p.gn2_s, 0, kD, 0, 1);
  add("decoder/decoder_block_0/retn2/group_norm/bias", p.gn2_b, 0, kD, 0, 1);
  add("decoder/decoder_block_0/ffn/W_gate", p.dffn_gl, 0, kD, kD, 2 * kD);
  add("decoder/decoder_block_0/ffn/W_linear", p.dffn_gl, kD, kD, kD, 2 * kD);
  add("decoder/decoder_block_0/ffn/W_output", p.dffn_out, 0, kD, kD, kD);
  add("decoder/head/layers_0/kernel", p.dh0_w, 0, kD, kD, kD);
  add("decoder/head/layers_0/bias", p.dh0_b, 0, kD, 0, 1);
  add("decoder/head/layers_2/scale", p.dh2_s, 0, kD, 0, 1);
  add("decoder/head/layers_3/kernel", p.dh3_w, 0, kD, a, a);
  add("decoder/head/layers_3/bias", p.dh3_b, 0, a, 0, 1);
  return n;
}

// which 1: the learner's RecurrentActor; which 2: rec_ippo's critic, RecurrentValueNet (networks/base.py:187-226): the same torsos and
// GRU with a Dense(1) head and no action mask (the actor's layout at a = 1)
static int actor_table(const MagpoNetCfg* net, ParamEntry* out, int which) {
  const int d = net->obs_dim, a = which == 2 ? 1 : net->action_dim;
  ActorP p = ActorP::bind(reinterpret_cast<float*>(sizeof(float)), d, a);
  auto off = [](const float* q) { return (int64_t)(reinterpret_cast<uintptr_t>(q) / sizeof(float)) - 1; };
  int n = 0;
  auto add = [&](const char* name, const float* q, int64_t extra, int r, int c, int ld) {
    if (out) out[n] = ParamEntry{name, off(q) + extra, r, c, ld};
    ++n;
  };
  add("pre_torso/Dense_0/kernel", p.pre_w, 0, d, kH, kH);
  add("pre_torso/Dense_0/bias", p.pre_b, 0, kH, 0, 1);
  add("ScannedRNN_0/GRUCell_0/ir/kernel", p.Wi, 0, kH, kH, 3 * kH);
  add("ScannedRNN_0/GRUCell_0/iz/kernel", p.Wi, kH, kH, kH, 3 * kH);
  add("ScannedRNN_0/GRUCell_0/in/kernel", p.Wi, 2 * kH, kH, kH, 3 * kH);
  add("ScannedRNN_0/GRUCell_0/ir/bias", p.bi, 0, kH, 0, 1);
  add("ScannedRNN_0/GRUCell_0/iz/bias", p.bi, kH, kH, 0, 1);
  add("ScannedRNN_0/GRUCell_0/in/bias", p.bi, 2 * kH, kH, 0, 1);
  add("ScannedRNN_0/GRUCell_0/hr/kernel", p.Wh, 0, kH, kH, 3 * kH);
  add("ScannedRNN_0/GRUCell_0/hz/kernel", p.Wh, kH, kH, kH, 3 * kH);
  add("ScannedRNN_0/GRUCell_0/hn/kernel", p.Wh, 2 * kH, kH, kH, 3 * kH);
  add("ScannedRNN_0/GRUCell_0/hn/bias", p.bhn, 0, kH, 0, 1);
  add("post_torso/Dense_0/kernel", p.post_w, 0, kH, kH, kH);
  add("post_torso/Dense_0/bias", p.post_b, 0, kH, 0, 1);
  // the critic's head is created directly in RecurrentValueNet's compact body, so its flax path is the bare auto-name (from memory)
  const bool critic = which == 2;
  add(critic ? "Dense_0/kernel" : "action_head/Dense_0/kernel", p.head_w, 0, kH, a, a);
  add(critic ? "Dense_0/bias" : "action_head/Dense_0/bias", p.head_b, 0, a, 0, 1);
  return n;
}

// the general guider's table (generic.cuh); names live in a per-thread cache so that the returned pointers stay valid
static const std::vector<ParamEntryG>& general_table(const MagpoNetCfg* net) {
  static thread_local std::vector<ParamEntryG> tab;
  tab.clear();
  guider_table_g(NetShape::of(net), &tab);
  return tab;
}

int64_t magpo_param_count(const MagpoNetCfg* net, int which) {
  if (check_net(net) != MAGPO_OK) return -1;
  if (which == 0 && !NetShape::of(net).is_default()) return GuiderG::bind(nullptr, NetShape::of(net)).total;
  return which == 0 ? GuiderP::bind(nullptr, net->obs_dim, net->action_dim).total
                    : ActorP::bind(nullptr, net->obs_dim, which == 2 ? 1 : net->action_dim).total;
}

int32_t magpo_param_num_tensors(const MagpoNetCfg* net, int which) {
  if (check_net(net) != MAGPO_OK) return -1;
  if (which == 0 && !NetShape::of(net).is_default()) return (int32_t)general_table(net).size();
  return which == 0 ? guider_table(net, nullptr) : actor_table(net, nullptr, which);
}

int magpo_param_tensor(const MagpoNetCfg* net, int which, int32_t index, const char** name, int64_t* offset,
                       int32_t* dim0, int32_t* dim1, int32_t* ld) {
  MAGPO_TRY(check_net(net));
  if (which == 0 && !NetShape::of(net).is_default()) {
    const std::vector<ParamEntryG>& t = general_table(net);
    if (index < 0 || index >= (int32_t)t.size() || !name || !offset || !dim0 || !dim1 || !ld) return MAGPO_ERR_ARG;
    *name = t[index].name;  // valid until the next table query on this thread
    *offset = t[index].offset; *dim0 = t[index].dim0; *dim1 = t[index].dim1; *ld = t[index].ld;
    return MAGPO_OK;
  }
  ParamEntry tab[64];
  const int n = which == 0 ? guider_table(net, tab) : actor_table(net, tab, which);
  if (index < 0 || index >= n || !name || !offset || !dim0 || !dim1 || !ld) return MAGPO_ERR_ARG;
  *name = tab[index].name;
  *offset = tab[index].offset;
  *dim0 = tab[index].dim0;
  *dim1 = tab[index].dim1;
  *ld = tab[index].ld;
  return MAGPO_OK;
}

}  // extern "C"
