// Rollout: lax.scan(_env_step, length=T) + bootstrap value of rec_magpo.py:126-208 for B = U*E envs.
// Per step: SableNetwork.get_actions (sable_network.py:443-482: decay, recurrent encoder over the A agents,
// A autoregressive decoder steps each followed by a distrax gumbel-max sample from the step's threefry key),
// the learner's GRU push (rec_magpo.py:146-159), then vmap(env.step) (rec_magpo.py:162).
// The PRNG key chain is data-independent, so all T+1 policy keys and their per-agent sample keys are derived
// by one tiny kernel up front (rec_magpo.py:135,202; decode.py:140).
#include "actor.cuh"
#include "envs.cuh"
#include "generic.cuh"
#include "prng.cuh"
#include "sable.cuh"
#include "update.cuh"

namespace magpo {

// sable.cu
int sable_encoder_forward(cudaStream_t s, const GuiderP& p, const GuiderT* pt, int T, int N, int A, int d, int max_step,
                          const float* agents_view, const int32_t* step, const uint8_t* done, const float* H0,
                          float kappa, const float* pe, const SableActs& w, float* value, float* Hsave, float* Hout, bool chain = false,
                          float* dec_q = nullptr);
int sable_decoder_forward(cudaStream_t s, const GuiderP& p, const GuiderT* pt, int T, int N, int ret_A, int embed_A, int a,
                          int max_step, const int32_t* action, const float* x_rep, const float* x_rep_pe,
                          const int32_t* step, const uint8_t* done, const float* Hself0, const float* Hcross0,
                          float kappa, const float* pe, const SableActs& w, float* logits, float* Hs_self,
                          float* Hs_cross, float* Hself_out, float* Hcross_out);

// sable_step.cu: the whole get_actions of a step as one kernel (A <= 4, obs_dim <= 16)
bool sable_step_supported(int A, int d, int a);
size_t sable_step_table_floats(const MagpoNetCfg* net);
int sable_step_tables(cudaStream_t st, const MagpoNetCfg* net, const GuiderP& p, const float* pe, float* tab);
int sable_step(cudaStream_t st, const MagpoNetCfg* net, int B, int gumbel_rows, const GuiderP& p, float kappa, const float* agents_view,
               const uint8_t* action_mask, const int32_t* step_count, const uint8_t* prev_done, const uint32_t* sample_keys,
               const float* pe, const float* dec_tab, MagpoSableHState hs, bool dry, int32_t* action, float* log_prob, float* value,
               float* masked_logits);

namespace {

// keys: [T+1][A][2] sample keys; key advanced in place by T+1 splits.
__global__ void rollout_keys_kernel(uint32_t* __restrict__ key, int steps, int A, uint32_t* __restrict__ sample_keys) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  uint32_t k0 = key[0], k1 = key[1];
  for (int t = 0; t < steps; ++t) {
    uint32_t n0, n1, p0, p1;
    prng_split_i(k0, k1, 0u, n0, n1);  // key, policy_key = split(key)
    prng_split_i(k0, k1, 1u, p0, p1);
    k0 = n0; k1 = n1;
    for (int i = 0; i < A; ++i) {
      uint32_t q0, q1, s0, s1;
      prng_split_i(p0, p1, 0u, q0, q1);  // key, sample_key = split(key)   (decode.py:140)
      prng_split_i(p0, p1, 1u, s0, s1);
      p0 = q0; p1 = q1;
      sample_keys[((size_t)t * A + i) * 2] = s0;
      sample_keys[((size_t)t * A + i) * 2 + 1] = s1;
    }
  }
  key[0] = k0;
  key[1] = k1;
}

// rows of agent i out of [B, A, width] -> [B, width]
__global__ void gather_agent_kernel(int64_t B, int A, int i, int width, const float* __restrict__ src,
                                    float* __restrict__ dst) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * width) return;
  const int64_t b = idx / width;
  dst[idx] = src[(b * A + i) * width + idx % width];
}
__global__ void gather_agent_i32_kernel(int64_t B, int A, int i, const int32_t* __restrict__ src, int32_t* __restrict__ dst) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) dst[b] = src[b * A + i];
}

// distrax.Categorical(logits=masked).sample_and_log_prob(seed=sample_key)  (decode.py:135-142, Appendix A3):
// noise tensor shape (1, E, 1, a) -> element (e, j) uses counter e*a + j; every update-batch slot shares the key.
__global__ void __launch_bounds__(128)
sample_kernel(int64_t B, int A, int i, int a, int gumbel_rows, const float* __restrict__ logits /*[B,a]*/,
              const uint8_t* __restrict__ mask /*[B,A,a]*/, const uint32_t* __restrict__ key,
              int32_t* __restrict__ action /*[B,A]*/, float* __restrict__ log_prob /*[B,A]*/,
              int32_t* __restrict__ prev_action /*[B]*/, float* __restrict__ masked_logits /*[B,A,a] or null*/) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float* l = logits + b * a;
  const uint8_t* m = mask + (b * A + i) * a;
  float mx = kF32Min;
  for (int j = 0; j < a; ++j) mx = fmaxf(mx, m[j] ? l[j] : kF32Min);
  float se = 0.f;
  for (int j = 0; j < a; ++j) se += expf((m[j] ? l[j] : kF32Min) - mx);
  const float lse = mx + logf(se);
  const uint32_t k0 = key[0], k1 = key[1];
  const uint64_t e = (uint64_t)(b % gumbel_rows);
  float best = 0.f, best_lp = 0.f;
  int best_j = -1;
  for (int j = 0; j < a; ++j) {
    const float ml = m[j] ? l[j] : kF32Min;
    const float lp = ml - lse;
    const float g = prng_gumbel_from_bits(prng_bits_i(k0, k1, e * (uint64_t)a + j));
    const float sc = g + lp;
    if (best_j < 0 || sc > best) { best = sc; best_j = j; best_lp = lp; }
    if (masked_logits) masked_logits[(b * A + i) * a + j] = ml;
  }
  action[b * A + i] = best_j;
  log_prob[b * A + i] = best_lp;
  prev_action[b] = best_j;
}

// dst[b] = done[b] ? 0 : src[b]  for [B, n_head, n_block, hs, hs] states
__global__ void copy_zero_done_kernel(int64_t B, int64_t quads /* float4 per env state */, const float* __restrict__ src,
                                      const uint8_t* __restrict__ done, float* __restrict__ dst) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * quads) return;
  const int64_t b = idx / quads;
  float4 v = reinterpret_cast<const float4*>(src)[idx];
  if (done && done[b]) v = make_float4(0.f, 0.f, 0.f, 0.f);
  reinterpret_cast<float4*>(dst)[idx] = v;
}

inline unsigned g256(int64_t n) { return (unsigned)ceil_div(n, 256); }

struct RolloutWs {
  SableActs sa;
  ActorActs aa;
  GuiderT gt;  // transposed weights + TF32 hi/lo images: the rollout GEMMs run on the tensor cores as well
  ActorT at;
  float *pe, *dec_tab, *xrep_i, *xrep_pe_i, *logits_i;
  int32_t *step_i, *prev_action;
  uint32_t* sample_keys;
  void* gws;  // general guider shapes (generic.cuh): the step workspace of sable_g_get_actions instead of the default path's buffers
  size_t gws_bytes;
  void plan(Arena& ar, const MagpoNetCfg* net, int B, int T) {
    const int64_t R = (int64_t)B * net->n_agents;
    aa.plan(ar, R, R, net->action_dim, false);
    at.plan(ar, net->action_dim);
    sample_keys = ar.get<uint32_t>((size_t)(T + 1) * net->n_agents * 2);
    gws = nullptr; gws_bytes = 0;
    const NetShape shape = NetShape::of(net);
    if (!shape.is_default()) {
      gws_bytes = sable_g_step_workspace_bytes(shape, B);
      gws = ar.get<char>(gws_bytes);
      pe = dec_tab = xrep_i = xrep_pe_i = logits_i = nullptr;
      step_i = prev_action = nullptr;
      return;
    }
    sa.plan(ar, R, B, net->obs_dim, false);
    gt.plan(ar, net->obs_dim);
    pe = ar.get<float>((size_t)(net->max_step_count + 1) * kD);
    dec_tab = ar.get<float>(sable_step_table_floats(net));
    xrep_i = ar.get<float>((size_t)B * kD);
    xrep_pe_i = ar.get<float>((size_t)B * kD);
    logits_i = ar.get<float>((size_t)B * net->action_dim);
    step_i = ar.get<int32_t>(B);
    prev_action = ar.get<int32_t>(B);
  }
};

// One SableNetwork.get_actions over B envs (T=1 recurrent step). hs updated in place unless `dry` (bootstrap).
int get_actions(cudaStream_t s, const MagpoNetCfg* net, int B, int gumbel_rows, const GuiderP& gp, const GuiderT* gt, float kappa,
                const float* agents_view, const uint8_t* action_mask, const int32_t* step_count,
                const uint8_t* prev_done, const uint32_t* sample_keys, MagpoSableHState hs, bool dry,
                int32_t* action, float* log_prob, float* value, float* masked_logits, const RolloutWs& w) {
  const int A = net->n_agents, d = net->obs_dim, a = net->action_dim, ms = net->max_step_count;
  if (w.gws)  // general (embed_dim, n_head, n_block): layer by layer (the caller prepared the workspace once: sable_g_prepare)
    return sable_g_get_actions(s, net, B, gumbel_rows, gp.obs_scale, agents_view, action_mask, step_count, prev_done, sample_keys, hs, dry,
                               action, log_prob, value, masked_logits, w.gws, w.gws_bytes, false);
  if (sable_step_supported(A, d, a))
    return sable_step(s, net, B, gumbel_rows, gp, kappa, agents_view, action_mask, step_count, prev_done, sample_keys, w.pe, w.dec_tab,
                      hs, dry, action, log_prob, value, masked_logits);
  MAGPO_TRY(sable_encoder_forward(s, gp, gt, 1, B, A, d, ms, agents_view, step_count, prev_done, hs.encoder, kappa, w.pe,
                                  w.sa, value, nullptr, dry ? nullptr : hs.encoder));
  if (!action) return MAGPO_OK;
  for (int i = 0; i < A; ++i) {
    {
      ProfScope ps(PROF_MISC, s, 4.0 * 256.0 * B);
      gather_agent_kernel<<<g256((int64_t)B * kD), 256, 0, s>>>(B, A, i, kD, w.sa.x, w.xrep_i);
      MAGPO_LAUNCH_OK();
      gather_agent_kernel<<<g256((int64_t)B * kD), 256, 0, s>>>(B, A, i, kD, w.sa.xpe, w.xrep_pe_i);
      MAGPO_LAUNCH_OK();
      gather_agent_i32_kernel<<<g256(B), 256, 0, s>>>(B, A, i, step_count, w.step_i);
      MAGPO_LAUNCH_OK();
    }
    // the once-per-timestep decay (and the reset on done) is applied when the first agent's token arrives
    MAGPO_TRY(sable_decoder_forward(s, gp, gt, 1, B, 1, i == 0 ? -1 : 0, a, ms, w.prev_action, w.xrep_i, w.xrep_pe_i,
                                    w.step_i, i == 0 ? prev_done : nullptr, hs.decoder_self, hs.decoder_cross,
                                    i == 0 ? kappa : 1.0f, w.pe, w.sa, w.logits_i, nullptr, nullptr,
                                    dry ? nullptr : hs.decoder_self, dry ? nullptr : hs.decoder_cross));
    ProfScope ps(PROF_SAMPLE, s, (double)B * (5.0 * a + 12.0));
    sample_kernel<<<(unsigned)ceil_div(B, 128), 128, 0, s>>>(B, A, i, a, gumbel_rows, w.logits_i, action_mask,
                                                            sample_keys + 2 * i, action, log_prob, w.prev_action,
                                                            masked_logits);
    MAGPO_LAUNCH_OK();
  }
  return MAGPO_OK;
}

}  // namespace

int sample_agent(cudaStream_t s, int64_t B, int A, int i, int a, int gumbel_rows, const float* logits, const uint8_t* mask, const uint32_t* key,
                 int32_t* action, float* log_prob, int32_t* prev_action, float* masked_logits) {
  ProfScope ps(PROF_SAMPLE, s, (double)B * (5.0 * a + 12.0));
  sample_kernel<<<(unsigned)ceil_div(B, 128), 128, 0, s>>>(B, A, i, a, gumbel_rows, logits, mask, key, action, log_prob, prev_action, masked_logits);
  MAGPO_LAUNCH_OK();
  return MAGPO_OK;
}
}  // namespace magpo

using namespace magpo;

extern "C" {

size_t magpo_rollout_workspace_bytes(const MagpoNetCfg* net, int32_t B, int32_t T) {
  if (check_net(net) != MAGPO_OK || B < 0 || T < 0) return 0;
  Arena ar(nullptr, SIZE_MAX);
  RolloutWs w;
  w.plan(ar, net, B, T);
  return ar.off;
}

int magpo_sable_get_actions(MagpoContext* ctx_, magpo_stream_t s_, const MagpoNetCfg* net, int32_t B, int32_t gumbel_rows,
                            const float* guider, const float* agents_view, const uint8_t* action_mask,
                            const int32_t* step_count, const uint8_t* prev_done, const uint32_t* sample_keys,
                            MagpoSableHState hs, int32_t* action, float* log_prob, float* value, float* logits,
                            void* workspace, size_t workspace_bytes) {
  MAGPO_CTX(ctx_);
  MAGPO_TRY(check_net(net));
  if (B <= 0 || !guider || !agents_view || !step_count || !value || !workspace) return MAGPO_ERR_ARG;
  if (action && (!action_mask || !sample_keys || !log_prob || gumbel_rows < 1)) return MAGPO_ERR_ARG;
  cudaStream_t s = as_stream(s_);
  Arena ar(workspace, workspace_bytes);
  RolloutWs w;
  w.plan(ar, net, B, 0);
  if (ar.overflow) return MAGPO_ERR_WORKSPACE;
  if (w.gws)
    return sable_g_get_actions(s, net, B, gumbel_rows, guider, agents_view, action_mask, step_count, prev_done, sample_keys, hs, false, action,
                               log_prob, value, logits, w.gws, w.gws_bytes, true);
  MAGPO_TRY(build_pe_table(s, net->max_step_count, w.pe, net->timestep_pe != 0));
  if (sable_step_supported(net->n_agents, net->obs_dim, net->action_dim))
    MAGPO_TRY(sable_step_tables(s, net, GuiderP::bind(const_cast<float*>(guider), net->obs_dim, net->action_dim), w.pe, w.dec_tab));
  const GuiderP gp = GuiderP::bind(const_cast<float*>(guider), net->obs_dim, net->action_dim);
  return get_actions(s, net, B, gumbel_rows, gp, nullptr, net_kappa(net), agents_view, action_mask, step_count, prev_done,
                     sample_keys, hs, false, action, log_prob, value, logits, w);
}

int magpo_actor_step(MagpoContext* ctx_, magpo_stream_t s_, const MagpoNetCfg* net, int32_t B, const float* actor,
                     const float* agents_view, const uint8_t* done, float* policy_h, void* workspace,
                     size_t workspace_bytes) {
  MAGPO_CTX(ctx_);
  MAGPO_TRY(check_net(net));
  if (B <= 0 || !actor || !agents_view || !policy_h || !workspace) return MAGPO_ERR_ARG;
  Arena ar(workspace, workspace_bytes);
  RolloutWs w;
  w.plan(ar, net, B, 0);
  if (ar.overflow) return MAGPO_ERR_WORKSPACE;
  const ActorP ap = ActorP::bind(const_cast<float*>(actor), net->obs_dim, net->action_dim);
  return actor_forward(as_stream(s_), ap, nullptr, 1, B, net->n_agents, net->obs_dim, net->action_dim, agents_view, done,
                       policy_h, w.aa, nullptr, policy_h);
}

int magpo_rollout(MagpoContext* ctx_, magpo_stream_t s_, const MagpoNetCfg* net, const MagpoSysCfg* sys, int env_kind,
                  const void* env_cfg, void* env_state, MagpoTimeStep ts, const float* guider, const float* actor,
                  uint32_t* key, MagpoSableHState hs, float* policy_h, MagpoTrajectory traj, int32_t carry_over,
                  void* workspace, size_t workspace_bytes) {
  MAGPO_CTX(ctx_);
  MAGPO_TRY(check_net(net));
  if (!sys || !env_cfg || !env_state || !guider || !actor || !key || !policy_h || !workspace) return MAGPO_ERR_ARG;
  if (env_kind != MAGPO_ENV_COORDSUM && env_kind != MAGPO_ENV_LBF && env_kind != MAGPO_ENV_RWARE) return MAGPO_ERR_UNSUPPORTED;
  cudaStream_t s = as_stream(s_);
  const int A = net->n_agents, d = net->obs_dim, a = net->action_dim;
  const int T = sys->rollout_length, E = sys->num_envs;
  const int B = sys->update_batch_size * E;
  const int64_t BA = (int64_t)B * A;
  Arena ar(workspace, workspace_bytes);
  RolloutWs w;
  w.plan(ar, net, B, T);
  if (ar.overflow) return MAGPO_ERR_WORKSPACE;
  const NetShape shape = NetShape::of(net);
  GuiderP gp = GuiderP::bind(const_cast<float*>(guider), d, a);
  const ActorP ap = ActorP::bind(const_cast<float*>(actor), d, a);
  const float kappa = net_kappa(net);
  const GuiderT* gtp = nullptr;
  const ActorT* atp = nullptr;
  if (w.gws) {  // general guider shape: PE table, transposed weights and their TF32 images once per rollout
    gp.obs_scale = const_cast<float*>(guider);  // get_actions hands the flat buffer to the general path
    MAGPO_TRY(sable_g_prepare(s, net, B, guider, w.gws, w.gws_bytes));
    MAGPO_TRY(actor_transpose(s, ap, w.at, a));
    atp = &w.at;
  } else {
    MAGPO_TRY(build_pe_table(s, net->max_step_count, w.pe, net->timestep_pe != 0));
    if (sable_step_supported(net->n_agents, net->obs_dim, net->action_dim))
      MAGPO_TRY(sable_step_tables(s, net, GuiderP::bind(const_cast<float*>(guider), net->obs_dim, net->action_dim), w.pe, w.dec_tab));
    // parameters are constant during the rollout: one transpose + TF32 split up front
    MAGPO_TRY(guider_transpose(s, gp, w.gt, d));
    MAGPO_TRY(actor_transpose(s, ap, w.at, a));
    gtp = &w.gt;
    atp = &w.at;
  }
  if (carry_over) {  // LearnerState.timestep of the previous call becomes observation slot 0
    MAGPO_CUDA_OK(cudaMemcpyAsync(traj.done, traj.done + (size_t)T * B, B, cudaMemcpyDeviceToDevice, s));
    MAGPO_CUDA_OK(cudaMemcpyAsync(traj.agents_view, traj.agents_view + (size_t)T * BA * d, BA * d * sizeof(float),
                                  cudaMemcpyDeviceToDevice, s));
    MAGPO_CUDA_OK(cudaMemcpyAsync(traj.action_mask, traj.action_mask + (size_t)T * BA * a, BA * a,
                                  cudaMemcpyDeviceToDevice, s));
    MAGPO_CUDA_OK(cudaMemcpyAsync(traj.step_count, traj.step_count + (size_t)T * BA, BA * sizeof(int32_t),
                                  cudaMemcpyDeviceToDevice, s));
  }
  // hidden states the update will start from (rec_magpo.py:190-192, 244-248)
  MAGPO_CUDA_OK(cudaMemcpyAsync(traj.policy_h0, policy_h, BA * kH * sizeof(float), cudaMemcpyDeviceToDevice, s));
  const int64_t quads = shape.state_elems() / 4;
  const unsigned gz = g256((int64_t)B * quads);
  copy_zero_done_kernel<<<gz, 256, 0, s>>>(B, quads, hs.encoder, traj.done, traj.sable_h0.encoder);
  MAGPO_LAUNCH_OK();
  copy_zero_done_kernel<<<gz, 256, 0, s>>>(B, quads, hs.decoder_self, traj.done, traj.sable_h0.decoder_self);
  MAGPO_LAUNCH_OK();
  copy_zero_done_kernel<<<gz, 256, 0, s>>>(B, quads, hs.decoder_cross, traj.done, traj.sable_h0.decoder_cross);
  MAGPO_LAUNCH_OK();
  rollout_keys_kernel<<<1, 32, 0, s>>>(key, T + 1, A, w.sample_keys);
  MAGPO_LAUNCH_OK();

  const bool overlap = nets_overlap_enabled() && !sys->sable_only;
  cudaStream_t s2 = s;
  // The learner's GRU push of a step (rec_magpo.py:146-159) depends only on the step's observation, not on the guider's actions: it
  // trails along on the context's forked stream and fills the SMs the fused guider kernel and the env step kernel leave idle.
  ForkJoin& g_rside = ctx().rside;
  if (overlap) s2 = g_rside.s;
  for (int t = 0; t < T; ++t) {
    const float* obs = traj.agents_view + (size_t)t * BA * d;
    const uint8_t* mask = traj.action_mask + (size_t)t * BA * a;
    const int32_t* stepc = traj.step_count + (size_t)t * BA;
    const uint8_t* prev_done = traj.done + (size_t)t * B;
    int32_t* act = traj.action + (size_t)t * BA;
    if (overlap) {  // observation slot t and done[t] are complete on `s` here
      MAGPO_CUDA_OK(cudaEventRecord(g_rside.fork, s));
      MAGPO_CUDA_OK(cudaStreamWaitEvent(s2, g_rside.fork, 0));
    }
    if (!sys->sable_only) MAGPO_TRY(actor_forward(s2, ap, atp, 1, B, A, d, a, obs, prev_done, policy_h, w.aa, nullptr, policy_h));
    MAGPO_TRY(get_actions(s, net, B, E, gp, gtp, kappa, obs, mask, stepc, prev_done, w.sample_keys + (size_t)t * A * 2, hs,
                          false, act, traj.log_prob + (size_t)t * BA, traj.value + (size_t)t * BA, nullptr, w));
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
    MAGPO_CUDA_OK(cudaEventRecord(g_rside.join, s2));
    MAGPO_CUDA_OK(cudaStreamWaitEvent(s, g_rside.join, 0));
  }
  // bootstrap value (rec_magpo.py:202-208): a full get_actions of which only the value is kept
  MAGPO_TRY(get_actions(s, net, B, E, gp, gtp, kappa, traj.agents_view + (size_t)T * BA * d, nullptr,
                        traj.step_count + (size_t)T * BA, traj.done + (size_t)T * B, nullptr, hs, true, nullptr, nullptr,
                        traj.last_value, nullptr, w));
  return MAGPO_OK;
}

}  // extern "C"
