// rec_ippo (mava/systems/ppo/anakin/rec_ippo.py): recurrent IPPO with a GRU actor and a GRU critic on the learner's kernels.
// The critic (RecurrentValueNet, networks/base.py:187-226) is the learner's RecurrentActor with a 1-wide head and no action mask, so
// both networks run through actor_forward / actor_backward (the critic at a = 1, its flat layout ActorP::bind(p, d, 1)). The loss is
// rec_sable's clipped PPO + clipped value loss, evaluated by magpo_losses on the pair (actor logits, critic values): with the same
// logits passed as the guider's and the learner's, the guidance KL is 0 and the double clip is the PPO clip (as for rec_sable).
// Every entry point sizes its own workspace: with workspace == NULL it writes the byte count to *workspace_bytes and returns.
#include "actor.cuh"
#include "envs.cuh"
#include "prng.cuh"
#include "update.cuh"

extern "C" int magpo_prng_permutation(magpo_stream_t s, const uint32_t* key, int32_t n, int32_t* out, uint32_t* scratch);

namespace magpo {
namespace {

// key, policy_key = split(key) per rollout step (rec_ippo.py `_env_step`); keys [T][2]; the bootstrap value consumes no key, so the
// key advances by exactly T splits.
__global__ void ippo_keys_kernel(uint32_t* __restrict__ key, int steps, uint32_t* __restrict__ keys) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  uint32_t k0 = key[0], k1 = key[1];
  for (int t = 0; t < steps; ++t) {
    uint32_t n0, n1;
    prng_split_i(k0, k1, 0u, n0, n1);
    prng_split_i(k0, k1, 1u, keys[2 * t], keys[2 * t + 1]);
    k0 = n0; k1 = n1;
  }
  key[0] = k0;
  key[1] = k1;
}

// Categorical(masked logits).sample(seed=key) and its log_prob for all agents at once, one thread per (env, agent) row: masked
// log-softmax, gumbel-max with tfp's noise layout (noise tensor (1, E, A, a): element (e, i, j) uses counter (e*A + i)*a + j, e = b mod
// gumbel_rows, so every update-batch slot draws the same noise), log_prob = the log-softmax at the chosen action.
__global__ void __launch_bounds__(128)
ippo_sample_kernel(int64_t BA, int A, int a, int gumbel_rows, const float* __restrict__ logits /*[B,A,a]*/,
                   const uint8_t* __restrict__ mask /*[B,A,a]*/, const uint32_t* __restrict__ key, int32_t* __restrict__ action,
                   float* __restrict__ log_prob) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= BA) return;
  const float* l = logits + row * a;
  const uint8_t* m = mask + row * a;
  float mx = kF32Min;
  for (int j = 0; j < a; ++j) mx = fmaxf(mx, m[j] ? l[j] : kF32Min);
  float se = 0.f;
  for (int j = 0; j < a; ++j) se += expf((m[j] ? l[j] : kF32Min) - mx);
  const float lse = mx + logf(se);
  const int64_t b = row / A, i = row % A;
  const uint64_t base = ((uint64_t)(b % gumbel_rows) * (uint64_t)A + (uint64_t)i) * (uint64_t)a;
  const uint32_t k0 = key[0], k1 = key[1];
  float best = 0.f, best_lp = 0.f;
  int best_j = -1;
  for (int j = 0; j < a; ++j) {
    const float lp = (m[j] ? l[j] : kF32Min) - lse;
    const float sc = prng_gumbel_from_bits(prng_bits_i(k0, k1, base + j)) + lp;
    if (best_j < 0 || sc > best) { best = sc; best_j = j; best_lp = lp; }
  }
  action[row] = best_j;
  log_prob[row] = best_lp;
}

// key, shuffle_key, _ = split(key, 3) (rec_ippo.py `_update_epoch`, from memory); sub [2] = shuffle_key
__global__ void split3_kernel(uint32_t* __restrict__ key, uint32_t* __restrict__ sub) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const uint32_t k0 = key[0], k1 = key[1];
  uint32_t n0, n1;
  prng_split_i(k0, k1, 0u, n0, n1);
  prng_split_i(k0, k1, 1u, sub[0], sub[1]);
  key[0] = n0;
  key[1] = n1;
}

// the stored t = 0 hidden states of the minibatch's envs: [n_env, A, H] from [B, A, H], both networks
__global__ void __launch_bounds__(256)
ippo_pack_h0_kernel(int A, const float* __restrict__ policy_h0, const float* __restrict__ critic_h0, const int32_t* __restrict__ env_index,
                    float* __restrict__ o_policy, float* __restrict__ o_critic) {
  const int n = blockIdx.x;
  const int64_t src = (int64_t)env_index[n] * A * kH, dst = (int64_t)n * A * kH;
  const int q = A * kH / 4;
  for (int idx = threadIdx.x; idx < q; idx += blockDim.x) {
    reinterpret_cast<float4*>(o_policy + dst)[idx] = reinterpret_cast<const float4*>(policy_h0 + src)[idx];
    reinterpret_cast<float4*>(o_critic + dst)[idx] = reinterpret_cast<const float4*>(critic_h0 + src)[idx];
  }
}

inline unsigned g128(int64_t n) { return (unsigned)ceil_div(n, 128); }

// workspace answer of the CUB-style size query: 0 when the caller asked for the size (and it was written), else whether it fits
int ws_check(const Arena& ar, void* workspace, size_t* workspace_bytes, bool* query) {
  *query = workspace == nullptr;
  if (*query) {
    *workspace_bytes = ar.off;
    return MAGPO_OK;
  }
  return ar.overflow ? MAGPO_ERR_WORKSPACE : MAGPO_OK;
}

struct IppoRolloutWs {
  ActorActs aa, ca;  // actor / critic activations of one step (inference plan)
  ActorT at, ct;     // transposed weights + TF32 images of both networks
  float* logits;     // [B, A, a]
  uint32_t* keys;    // [T][2] policy keys
  void plan(Arena& ar, const MagpoNetCfg* net, int B, int T) {
    const int64_t R = (int64_t)B * net->n_agents;
    aa.plan(ar, R, R, net->action_dim, false);
    ca.plan(ar, R, R, 1, false);
    at.plan(ar, net->action_dim);
    ct.plan(ar, 1);
    logits = ar.get<float>((size_t)R * net->action_dim);
    keys = ar.get<uint32_t>((size_t)2 * (T > 0 ? T : 1));
  }
};

struct IppoUpdateWs {
  ActorT at, ct;
  ActorActs aa, ca;
  float *a_hi, *a_lo, *c_hi, *c_lo;  // TF32 images of the two flat parameter buffers (the backward's dX operands)
  float *logits, *value, *dlogits, *dll, *dvalue;
  void plan(Arena& ar, const MagpoNetCfg* net, int T, int N) {
    const int A = net->n_agents, a = net->action_dim, d = net->obs_dim;
    const int64_t Rs = (int64_t)N * A, R = Rs * T;
    at.plan(ar, a);
    ct.plan(ar, 1);
    const int64_t n_a = ActorP::bind(nullptr, d, a).total, n_c = ActorP::bind(nullptr, d, 1).total;
    a_hi = ar.get<float>((size_t)n_a); a_lo = ar.get<float>((size_t)n_a);
    c_hi = ar.get<float>((size_t)n_c); c_lo = ar.get<float>((size_t)n_c);
    aa.plan(ar, R, Rs, a, true);
    ca.plan(ar, R, Rs, 1, true);
    logits = ar.get<float>((size_t)R * a);
    value = ar.get<float>((size_t)R);
    dlogits = ar.get<float>((size_t)R * a);
    dll = ar.get<float>((size_t)R * a);  // magpo_losses' second logits gradient: the same policy's, unused here
    dvalue = ar.get<float>((size_t)R);
  }
};

}  // namespace
}  // namespace magpo

using namespace magpo;

extern "C" {

int magpo_ippo_rollout(MagpoContext* ctx_, magpo_stream_t s_, const MagpoNetCfg* net, const MagpoSysCfg* sys, int env_kind,
                       const void* env_cfg, void* env_state, MagpoTimeStep ts, const float* actor, const float* critic, uint32_t* key,
                       float* policy_h, float* critic_h, MagpoTrajectory traj, float* critic_h0, int32_t carry_over, void* workspace,
                       size_t* workspace_bytes) {
  MAGPO_TRY(check_net(net));
  if (!sys || !workspace_bytes || sys->num_envs < 1 || sys->update_batch_size < 1 || sys->rollout_length < 1) return MAGPO_ERR_ARG;
  const int A = net->n_agents, d = net->obs_dim, a = net->action_dim;
  const int T = sys->rollout_length, E = sys->num_envs;
  const int B = sys->update_batch_size * E;
  const int64_t BA = (int64_t)B * A;
  Arena ar(workspace, workspace ? *workspace_bytes : SIZE_MAX);
  IppoRolloutWs w;
  w.plan(ar, net, B, T);
  bool query;
  MAGPO_TRY(ws_check(ar, workspace, workspace_bytes, &query));
  if (query) return MAGPO_OK;
  MAGPO_CTX(ctx_);
  if (!env_cfg || !env_state || !actor || !critic || !key || !policy_h || !critic_h || !critic_h0 || !traj.policy_h0 || !traj.done ||
      !traj.agents_view || !traj.action_mask || !traj.action || !traj.value || !traj.log_prob || !traj.reward || !traj.last_value)
    return MAGPO_ERR_ARG;
  if (env_kind != MAGPO_ENV_COORDSUM && env_kind != MAGPO_ENV_LBF && env_kind != MAGPO_ENV_RWARE) return MAGPO_ERR_UNSUPPORTED;
  cudaStream_t s = as_stream(s_);
  const ActorP ap = ActorP::bind(const_cast<float*>(actor), d, a);
  const ActorP cp = ActorP::bind(const_cast<float*>(critic), d, 1);
  MAGPO_TRY(actor_transpose(s, ap, w.at, a));
  MAGPO_TRY(actor_transpose(s, cp, w.ct, 1));
  if (carry_over) {  // LearnerState.timestep of the previous call becomes observation slot 0
    MAGPO_CUDA_OK(cudaMemcpyAsync(traj.done, traj.done + (size_t)T * B, B, cudaMemcpyDeviceToDevice, s));
    MAGPO_CUDA_OK(cudaMemcpyAsync(traj.agents_view, traj.agents_view + (size_t)T * BA * d, BA * d * sizeof(float),
                                  cudaMemcpyDeviceToDevice, s));
    MAGPO_CUDA_OK(cudaMemcpyAsync(traj.action_mask, traj.action_mask + (size_t)T * BA * a, BA * a, cudaMemcpyDeviceToDevice, s));
    MAGPO_CUDA_OK(cudaMemcpyAsync(traj.step_count, traj.step_count + (size_t)T * BA, BA * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
  }
  // the hidden states before the first step are the ones the update starts from (stored without the reset: the networks apply it
  // from done[0], as for rec_magpo's policy_h0)
  MAGPO_CUDA_OK(cudaMemcpyAsync(traj.policy_h0, policy_h, BA * kH * sizeof(float), cudaMemcpyDeviceToDevice, s));
  MAGPO_CUDA_OK(cudaMemcpyAsync(critic_h0, critic_h, BA * kH * sizeof(float), cudaMemcpyDeviceToDevice, s));
  ippo_keys_kernel<<<1, 32, 0, s>>>(key, T, w.keys);
  MAGPO_LAUNCH_OK();

  // The critic's step needs only the step's observation: it runs on the context's forked rollout stream beside the actor, the
  // sampler and the env step.
  const bool overlap = nets_overlap_enabled();
  ForkJoin& side = ctx().rside;
  cudaStream_t s2 = overlap ? side.s : s;
  for (int t = 0; t < T; ++t) {
    const float* obs = traj.agents_view + (size_t)t * BA * d;
    const uint8_t* prev_done = traj.done + (size_t)t * B;
    int32_t* act = traj.action + (size_t)t * BA;
    if (overlap) {  // observation slot t and done[t] are complete on `s` here
      MAGPO_CUDA_OK(cudaEventRecord(side.fork, s));
      MAGPO_CUDA_OK(cudaStreamWaitEvent(s2, side.fork, 0));
    }
    MAGPO_TRY(actor_forward(s2, cp, &w.ct, 1, B, A, d, 1, obs, prev_done, critic_h, w.ca, traj.value + (size_t)t * BA, critic_h));
    MAGPO_TRY(actor_forward(s, ap, &w.at, 1, B, A, d, a, obs, prev_done, policy_h, w.aa, w.logits, policy_h));
    {
      ProfScope ps(PROF_SAMPLE, s, (double)BA * (5.0 * a + 12.0));
      ippo_sample_kernel<<<g128(BA), 128, 0, s>>>(BA, A, a, E, w.logits, traj.action_mask + (size_t)t * BA * a, w.keys + 2 * t, act,
                                                  traj.log_prob + (size_t)t * BA);
      MAGPO_LAUNCH_OK();
    }
    MagpoTimeStep o = ts;
    o.reward = traj.reward + (size_t)t * BA;
    o.agents_view = traj.agents_view + (size_t)(t + 1) * BA * d;
    o.action_mask = traj.action_mask + (size_t)(t + 1) * BA * a;
    o.step_count = traj.step_count + (size_t)(t + 1) * BA;
    o.episode_return = traj.episode_return + (size_t)t * B;
    o.episode_length = traj.episode_length + (size_t)t * B;
    o.is_terminal_step = traj.is_terminal_step + (size_t)t * B;
    uint8_t* done_next = traj.done + (size_t)(t + 1) * B;
    if (env_kind == MAGPO_ENV_RWARE)
      MAGPO_TRY(rware_step_launch(s, static_cast<const MagpoRwareCfg*>(env_cfg), B, act, *static_cast<MagpoRwareState*>(env_state), o,
                                  done_next));
    else if (env_kind == MAGPO_ENV_LBF)
      MAGPO_TRY(lbf_step_launch(s, static_cast<const MagpoLbfCfg*>(env_cfg), B, act, *static_cast<MagpoLbfState*>(env_state), o, done_next));
    else
      MAGPO_TRY(coordsum_step_launch(s, static_cast<const MagpoCoordSumCfg*>(env_cfg), B, act,
                                     *static_cast<MagpoCoordSumState*>(env_state), o, done_next));
  }
  if (overlap) {
    MAGPO_CUDA_OK(cudaEventRecord(side.join, s2));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(s, side.join, 0));
  }
  // bootstrap value: the critic on the final observation with the final critic state and last done; its new state is discarded
  return actor_forward(s, cp, &w.ct, 1, B, A, d, 1, traj.agents_view + (size_t)T * BA * d, traj.done + (size_t)T * B, critic_h, w.ca,
                       traj.last_value, nullptr);
}

int magpo_ippo_epoch_indices(magpo_stream_t s_, const MagpoSysCfg* sys, uint32_t* key, int32_t* perm, int32_t* env_index,
                             int32_t* env_slot, void* workspace, size_t* workspace_bytes) {
  if (!sys || !workspace_bytes) return MAGPO_ERR_ARG;
  const int E = sys->num_envs, U = sys->update_batch_size, M = sys->num_minibatches;
  if (E < 1 || U < 1 || M < 1 || E % M) return MAGPO_ERR_ARG;
  Arena ar(workspace, workspace ? *workspace_bytes : SIZE_MAX);
  uint32_t* sub = ar.get<uint32_t>(2);
  uint32_t* pscr = ar.get<uint32_t>(2 * (size_t)E);
  int32_t* hs_perm = ar.get<int32_t>(E);
  int32_t* hs_index = ar.get<int32_t>((size_t)U * E);
  bool query;
  MAGPO_TRY(ws_check(ar, workspace, workspace_bytes, &query));
  if (query) return MAGPO_OK;
  if (!key || !perm || !env_index || !env_slot) return MAGPO_ERR_ARG;
  cudaStream_t s = as_stream(s_);
  split3_kernel<<<1, 32, 0, s>>>(key, sub);
  MAGPO_LAUNCH_OK();
  MAGPO_TRY(magpo_prng_permutation(s_, sub, E, perm, pscr));
  // every epoch gathers the stored t = 0 states of its envs afresh: no permutation accumulates across epochs (first_epoch = 1)
  return epoch_index(s, E, U, M, perm, hs_perm, 1, hs_perm, env_index, hs_index, env_slot);
}

int magpo_ippo_pack_minibatch(magpo_stream_t s_, const MagpoNetCfg* net, const MagpoSysCfg* sys, MagpoTrajectory traj,
                              const float* critic_h0, const float* advantages, const float* targets, const int32_t* env_index, int32_t n_env,
                              MagpoMinibatch out, float* out_critic_h0) {
  MAGPO_TRY(check_net(net));
  if (!sys || !critic_h0 || !advantages || !targets || !env_index || n_env < 1 || !out_critic_h0 || !traj.policy_h0 || !out.policy_h0)
    return MAGPO_ERR_ARG;
  if (out.T != sys->rollout_length || out.N != n_env) return MAGPO_ERR_ARG;
  cudaStream_t s = as_stream(s_);
  const int A = net->n_agents;
  const int64_t R = (int64_t)out.T * n_env * A;
  ProfScope ps(PROF_PACK, s, 2.0 * (double)R * (4.0 * net->obs_dim + net->action_dim + 24.0) + 2.0 * n_env * 1024.0 * A);
  MAGPO_TRY(pack_rows(s, net, sys, traj, advantages, targets, env_index, nullptr, n_env, out));
  ippo_pack_h0_kernel<<<n_env, 256, 0, s>>>(A, traj.policy_h0, critic_h0, env_index, const_cast<float*>(out.policy_h0), out_critic_h0);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}

int magpo_ippo_minibatch_grads(MagpoContext* ctx_, magpo_stream_t s_, const MagpoNetCfg* net, const MagpoSysCfg* sys, const float* actor,
                               const float* critic, MagpoMinibatch mb, const float* critic_h0, const int32_t* env_slot,
                               const float* adv_stats, float inv_tokens, float* grads, int32_t reduce_grads, void* workspace,
                               size_t* workspace_bytes) {
  MAGPO_TRY(check_net(net));
  if (!sys || !workspace_bytes || mb.T < 1 || mb.N < 1) return MAGPO_ERR_ARG;
  const int A = net->n_agents, a = net->action_dim, d = net->obs_dim, T = mb.T, N = mb.N;
  const int64_t R = (int64_t)T * N * A;
  Arena ar(workspace, workspace ? *workspace_bytes : SIZE_MAX);
  IppoUpdateWs w;
  w.plan(ar, net, T, N);
  bool query;
  MAGPO_TRY(ws_check(ar, workspace, workspace_bytes, &query));
  if (query) return MAGPO_OK;
  MAGPO_CTX(ctx_);
  if (!actor || !critic || !critic_h0 || !env_slot || !adv_stats || !grads || !mb.agents_view || !mb.action_mask || !mb.done ||
      !mb.action || !mb.value || !mb.log_prob || !mb.advantages || !mb.targets || !mb.policy_h0)
    return MAGPO_ERR_ARG;
  cudaStream_t s = as_stream(s_);
  const ActorP ap = ActorP::bind(const_cast<float*>(actor), d, a);
  const ActorP cp = ActorP::bind(const_cast<float*>(critic), d, 1);
  const ActorP ag = ActorP::bind(grads, d, a);
  const ActorP cg = ActorP::bind(grads + ap.total, d, 1);
  float* loss_sums = grads + ap.total + cp.total;
  MAGPO_TRY(actor_transpose(s, ap, w.at, a));
  MAGPO_TRY(actor_transpose(s, cp, w.ct, 1));
  MAGPO_TRY(tc_prepare_region(s, actor, ap.total, w.a_hi, w.a_lo));
  MAGPO_TRY(tc_prepare_region(s, critic, cp.total, w.c_hi, w.c_lo));
  // The actor and the critic are independent until the loss and again after it: the actor runs on the context's side stream, the
  // critic on the caller's, and their persistent GRU scans share the SMs.
  const bool overlap = nets_overlap_enabled();
  ForkJoin& side = ctx().side;
  cudaStream_t s2 = overlap ? side.s : s;
  if (overlap) {
    MAGPO_CUDA_OK(cudaEventRecord(side.fork, s));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(s2, side.fork, 0));
  }
  MAGPO_TRY(actor_forward(s2, ap, &w.at, T, N, A, d, a, mb.agents_view, mb.done, mb.policy_h0, w.aa, w.logits, nullptr));
  MAGPO_TRY(actor_forward(s, cp, &w.ct, T, N, A, d, 1, mb.agents_view, mb.done, critic_h0, w.ca, w.value, nullptr));
  if (overlap) {
    MAGPO_CUDA_OK(cudaEventRecord(side.join, s2));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(s, side.join, 0));
  }
  // rec_sable's path through the MAGPO loss: identical logits as guider and learner make the guidance ratio exactly 1 and the KL 0, so
  // clip_gpo only has to exceed 1 and alpha scales a gradient that is discarded
  MagpoSysCfg ls = *sys;
  ls.clip_gpo = 2.0;
  ls.alpha = 1.0;
  MAGPO_TRY(magpo_losses(s, R, N, A, a, &ls, inv_tokens, w.logits, w.logits, mb.action_mask, mb.action, mb.log_prob, mb.advantages,
                         w.value, mb.value, mb.targets, env_slot, adv_stats, w.dlogits, w.dll, w.dvalue, loss_sums));
  if (overlap) {
    MAGPO_CUDA_OK(cudaEventRecord(side.fork, s));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(s2, side.fork, 0));
  }
  MAGPO_TRY(actor_backward(s2, ap, w.at, T, N, A, d, a, mb.agents_view, mb.done, w.aa, w.dlogits, ag));
  MAGPO_TRY(actor_backward(s, cp, w.ct, T, N, A, d, 1, mb.agents_view, mb.done, w.ca, w.dvalue, cg));
  if (overlap) {
    MAGPO_CUDA_OK(cudaEventRecord(side.join, s2));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(s, side.join, 0));
  }
  // the pmean over "device": one sum all-reduce of [actor grads | critic grads | loss sums]; the 1/Nd is the optimiser's grad_scale
  MagpoComm* comm = reduce_grads ? ctx().comm : nullptr;
  if (comm) MAGPO_TRY(comm_allreduce(comm, s, grads, ap.total + cp.total + 8, 0));
  return MAGPO_OK;
}

}  // extern "C"
