/* magpo_b200.h — C ABI of libmagpo_b200.so: hand-written sm_100a CUDA kernels for the
 * rec_magpo Anakin hot path (rollout + GAE + update).
 *
 * The reference (liyheng/MAGPO, 100% Python/JAX) has no FFI/operator registry; the boundary it
 * offers is the Python calling convention inside mava/systems/gpo/anakin/rec_magpo.py.  Each
 * entry point below cites the reference code it replaces.  Conventions (shaped so that an
 * XLA-FFI handler `XLA_FFI_Error* h(XLA_FFI_CallFrame*)` can wrap each op 1:1):
 *   - the CUDA stream (cudaStream_t passed as void*) comes first, after the per-device MagpoContext* for the entry points that
 *     need one (see below); all work is enqueued on that stream (forked context streams are joined back before the call
 *     returns), nothing synchronises, nothing allocates: every buffer is a caller-owned DEVICE pointer, scratch is passed
 *     explicitly and sized by the matching *_workspace_bytes(); there is no process-global state on the product path (the
 *     benchmark / test hooks magpo_prof_*, magpo_debug_set_overlap and magpo_set_chain_kernels are process-wide; it never sets them);
 *   - POD attribute structs by const pointer; no torch / C++ types in any signature;
 *   - return 0 on success, a negative MAGPO_ERR_* otherwise (no exceptions cross the ABI);
 *   - single host thread per device (the reference path is single-threaded).
 * All floating-point tensors are float32, row-major, innermost dimension last.
 */
#ifndef MAGPO_B200_H_
#define MAGPO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* magpo_stream_t; /* cudaStream_t */

enum {
  MAGPO_OK = 0,
  MAGPO_ERR_ARG = -1,         /* bad / inconsistent argument */
  MAGPO_ERR_UNSUPPORTED = -2, /* configuration outside what the kernels implement */
  MAGPO_ERR_CUDA = -3,        /* a CUDA runtime call failed (see magpo_last_cuda_error) */
  MAGPO_ERR_WORKSPACE = -4    /* workspace too small */
};

const char* magpo_version(void);

/* cudaGetLastError() text of the most recent MAGPO_ERR_CUDA on this thread. */
const char* magpo_last_cuda_error(void);

/* ------------------------------------------------------------------ context
 * Per-device context, created by the caller and passed to every entry point that needs more than its arguments: the entry points that
 * fork work onto side streams (rollout, minibatch_grads, guider_forward) or that look up the TF32 images of weight matrices they
 * prepared in the caller's workspace (all GEMM users). It owns three non-blocking streams with their fork / join events and a
 * host-side table of prepared weight regions; nothing the product path uses is process-global (only the benchmark / test hooks
 * magpo_prof_*, magpo_debug_set_overlap and magpo_set_chain_kernels are, and it never sets them), so several learners — on the same device
 * or on different ones — can be driven from one process and interleaved freely. A context is bound to the device it was created
 * on: calling with another device current returns MAGPO_ERR_ARG. One host thread at a time per context. The remaining entry points
 * (PRNG, envs, GAE, shuffle / pack, clip+Adam) are stateless and take no context. */
typedef struct MagpoContext MagpoContext;
int magpo_context_create(int32_t device /* CUDA ordinal, < 0: the current device */, MagpoContext** out);
int magpo_context_destroy(MagpoContext* ctx);

/* ------------------------------------------------------------------ configuration */

/* Network shapes: configs/network/magpo.yaml + env dims (rec_magpo.py:541-578). */
typedef struct MagpoNetCfg {
  int32_t n_agents;   /* A */
  int32_t obs_dim;    /* d, includes the agent-id one-hot (wrappers/observation.py:42-54) */
  int32_t action_dim; /* a */
  int32_t embed_dim;  /* D  (net_config.embed_dim, 64) */
  int32_t n_head;     /* net_config.n_head (1) */
  int32_t n_block;    /* net_config.n_block (1) */
  int32_t hidden;     /* H  (hidden_state_dim == torso width, 128) */
  int32_t timestep_pe;/* memory_config.timestep_positional_encoding */
  float decay_scaling_factor; /* memory_config.decay_scaling_factor (0.8) */
  int32_t max_step_count; /* largest Observation.step_count the env emits (= time_limit): size of the PE table */
} MagpoNetCfg;

/* Hyper-parameters read on the path: configs/system/gpo/rec_magpo.yaml:12-25. */
typedef struct MagpoSysCfg {
  int32_t num_envs;          /* E  arch.num_envs (per device per update-batch slot) */
  int32_t update_batch_size; /* U */
  int32_t rollout_length;    /* T */
  int32_t ppo_epochs;        /* P */
  int32_t num_minibatches;   /* M */
  /* Python floats in the reference (weak-typed f64 constants); rounded to f32 where JAX would. */
  double gamma, gae_lambda, clip_eps, ent_coef, vf_coef, max_grad_norm, clip_gpo, alpha, lr;
  /* 0: rec_magpo (guider + learner). 1: rec_sable (mava/systems/sable/anakin/rec_sable.py): the Sable network alone under the
   * clipped PPO objective — no learner push in the rollout, no learner pass in the update; the MAGPO guider loss with the
   * learner's log-probs replaced by the guider's own is exactly rec_sable's loss (KL term 0, double clip = PPO clip). */
  int32_t sable_only;
} MagpoSysCfg;

/* ------------------------------------------------------------------ parameters
 * Parameters of one network live in ONE flat float32 buffer; the tensors are laid out in the
 * canonical order reported here, named by their flax tree path (SURVEY.md Appendix A8/A9),
 * e.g. "encoder/encoder_block_0/retn/retention_heads_0/w_q".  which: 0 = guider (SableNetwork,
 * networks/sable_network.py:346), 1 = learner (RecurrentActor, networks/base.py:152), 2 = rec_ippo's critic
 * (RecurrentValueNet, networks/base.py:187-226: the learner's layout at action_dim 1, head "Dense_0"). */
int64_t magpo_param_count(const MagpoNetCfg* cfg, int which);
int32_t magpo_param_num_tensors(const MagpoNetCfg* cfg, int which);
/* name -> static string; shape: up to 2 dims (dim1 == 0 for vectors); ld = row stride in floats: tensors that
 * always enter one GEMM together (retention w_q|w_k|w_v|w_g, SwiGLU W_gate|W_linear, the GRU's ir|iz|in and
 * hr|hz|hn) are stored packed side by side, so a flax tensor is a strided view of the flat buffer. Offsets are
 * 16-byte aligned; padding elements are zero and stay zero. */
int magpo_param_tensor(const MagpoNetCfg* cfg, int which, int32_t index, const char** name,
                       int64_t* offset, int32_t* dim0, int32_t* dim1, int32_t* ld);

/* ------------------------------------------------------------------ PRNG (jax.random, threefry2x32)
 * jax 0.6.0 semantics with jax_threefry_partitionable=True (SURVEY.md Appendix A1-A5). Keys are
 * raw uint32[2].  Replaces jax.random.{split,randint,permutation,...} call sites
 * rec_magpo.py:135,202,373,439,443,450,642,660,699. */
int magpo_prng_split(magpo_stream_t s, const uint32_t* key, int32_t num, uint32_t* out /*[num,2]*/);
int magpo_prng_random_bits(magpo_stream_t s, const uint32_t* key, int64_t n, uint32_t* out /*[n]*/);
int magpo_prng_randint(magpo_stream_t s, const uint32_t* key, int64_t n, int32_t minval,
                       int32_t maxval, int32_t* out /*[n]*/);
int magpo_prng_gumbel(magpo_stream_t s, const uint32_t* key, int64_t n, float* out /*[n]*/);
/* jax.random.normal / truncated_normal(key, (n,), float32) — the draws behind flax's normal / lecun_normal / orthogonal initialisers
 * (sable_network.py:97-107, retention.py:50-64, flax GRUCell): uniform from the threefry bits, sqrt(2) * erf_inv with XLA's
 * single-precision expansion. fold_in is a host function (flax derives each parameter's key from the module path on the host). */
int magpo_prng_normal(magpo_stream_t s, const uint32_t* key, int64_t n, float* out /*[n]*/);
int magpo_prng_truncated_normal(magpo_stream_t s, const uint32_t* key, int64_t n, float lower, float upper, float* out /*[n]*/);
int magpo_prng_fold_in_host(const uint32_t* key /*host [2]*/, uint32_t data, uint32_t* out /*host [2]*/);
/* jax.random.permutation(key, n): rounds of stable sort by random bits. scratch: 2n uint32. */
int magpo_prng_permutation(magpo_stream_t s, const uint32_t* key, int32_t n, int32_t* out,
                           uint32_t* scratch);

/* ------------------------------------------------------------------ environments (B envs, SoA)
 * TimeStep + extras of the training wrapper stack
 * RecordEpisodeMetrics(AutoResetWrapper(AgentIDWrapper(<Env>Wrapper(env)))) — utils/make_env.py:90-104. */
typedef struct MagpoTimeStep {
  int8_t* step_type;        /* [B]      jumanji StepType FIRST=0 MID=1 LAST=2 */
  float* reward;            /* [B,A] */
  float* discount;          /* [B,A] */
  float* agents_view;       /* [B,A,d]  float32 image of Observation.agents_view */
  uint8_t* action_mask;     /* [B,A,a] */
  int32_t* step_count;      /* [B,A] */
  float* next_agents_view;  /* [B,A,d]  extras["real_next_obs"] (auto_reset_wrapper.py:52-58) */
  int32_t* next_step_count; /* [B,A] */
  float* episode_return;    /* [B]      extras["episode_metrics"] (episode_metrics.py:98-102) */
  int32_t* episode_length;  /* [B] */
  uint8_t* is_terminal_step;/* [B] */
} MagpoTimeStep;

/* CoordSum (mava/coordsum/env.py:39-139; scenarios coordsum/__init__.py:6-45). */
typedef struct MagpoCoordSumCfg {
  int32_t num_agents, num_actions, time_limit, maxval;
} MagpoCoordSumCfg;

/* RecordEpisodeMetricsState(env_state = CoordSum State) — episode_metrics.py:34-44, coordsum/env.py:17-26. */
typedef struct MagpoCoordSumState {
  int32_t* step_count;      /* [B] */
  int32_t* target;          /* [B, time_limit+1] */
  int32_t* record;          /* [B, num_actions, time_limit] */
  uint32_t* key;            /* [B,2]  CoordSum State.key */
  uint32_t* metrics_key;    /* [B,2]  RecordEpisodeMetricsState.key */
  float* running_return;    /* [B] */
  int32_t* running_length;  /* [B] */
  float* episode_return;    /* [B] */
  int32_t* episode_length;  /* [B] */
} MagpoCoordSumState;

/* vmap(env.reset)(keys) — rec_magpo.py:645-647. keys [B,2]. */
int magpo_coordsum_reset(magpo_stream_t s, const MagpoCoordSumCfg* cfg, int32_t B,
                         const uint32_t* keys, MagpoCoordSumState st, MagpoTimeStep ts);
/* vmap(env.step)(state, action) — rec_magpo.py:162. action [B,A]. In place on `st`; `ts` is the output. */
int magpo_coordsum_step(magpo_stream_t s, const MagpoCoordSumCfg* cfg, int32_t B,
                        const int32_t* action, MagpoCoordSumState st, MagpoTimeStep ts);

/* LevelBasedForaging (jumanji 1.1.0 @ 9ced6b8 `environments/routing/lbf`, un-vendored third-party dependency, restated — see
 * oracle/lbf.py; built by mava/utils/make_env.py:107-135 from configs/env/scenario/{2s-8x8-2p-2f-coop,...}.yaml task_config) under
 * RecordEpisodeMetrics(AutoResetWrapper(AgentIDWrapper(LbfWrapper(env)))) — mava/wrappers/jumanji.py:171-208.
 * obs_dim d = num_agents + 3*(num_food+num_agents), action_dim 6. Limits: grid_size <= 16, num_agents <= 8, num_food <= 8. */
typedef struct MagpoLbfCfg {
  int32_t grid_size, fov, num_agents, num_food, max_agent_level, force_coop, time_limit;
  int32_t agent_mask_rows; /* 1: generator's agent mask clears whole rows (`mask.at[food_positions]`), 0: food cells only */
} MagpoLbfCfg;

/* RecordEpisodeMetricsState(env_state = lbf State(agents, food_items, step_count, key)). Positions are (row, col). */
typedef struct MagpoLbfState {
  int32_t* agent_pos;       /* [B,A,2] */
  int32_t* agent_level;     /* [B,A] */
  uint8_t* agent_loading;   /* [B,A] */
  int32_t* food_pos;        /* [B,F,2] */
  int32_t* food_level;      /* [B,F] */
  uint8_t* food_eaten;      /* [B,F] */
  int32_t* step_count;      /* [B] */
  uint32_t* key;            /* [B,2]  lbf State.key */
  uint32_t* metrics_key;    /* [B,2]  RecordEpisodeMetricsState.key */
  float* running_return;    /* [B] */
  int32_t* running_length;  /* [B] */
  float* episode_return;    /* [B] */
  int32_t* episode_length;  /* [B] */
} MagpoLbfState;

/* vmap(env.reset)(keys) / vmap(env.step)(state, action) for the LBF stack; same contract as the CoordSum pair. */
int magpo_lbf_reset(magpo_stream_t s, const MagpoLbfCfg* cfg, int32_t B, const uint32_t* keys,
                    MagpoLbfState st, MagpoTimeStep ts);
int magpo_lbf_step(magpo_stream_t s, const MagpoLbfCfg* cfg, int32_t B, const int32_t* action,
                   MagpoLbfState st, MagpoTimeStep ts);

/* RobotWarehouse (jumanji 1.1.0 @ 9ced6b8 `environments/routing/robot_warehouse`, un-vendored third-party dependency, restated — see
 * oracle/rware.py; built by mava/utils/make_env.py:107-135 from configs/env/scenario/{tiny-4ag,small-4ag,...}.yaml task_config) under
 * RecordEpisodeMetrics(AutoResetWrapper(AgentIDWrapper(RwareWrapper(env)))) — mava/wrappers/jumanji.py:137-168.
 * H = (column_height+1)*shelf_rows+2, W = 3*shelf_columns+1, S = number of non-highway cells, obs_dim d = num_agents + 8 +
 * 7*(2*sensor_range+1)^2, action_dim 5. Limits: H*W <= 1024, num_agents <= 8, request_queue_size <= 16, sensor_range <= 2. */
typedef struct MagpoRwareCfg {
  int32_t column_height, shelf_rows, shelf_columns, num_agents, sensor_range, request_queue_size, time_limit;
} MagpoRwareCfg;

/* RecordEpisodeMetricsState(env_state = robot_warehouse State(grid, agents, shelves, request_queue, step_count, action_mask, key)).
 * Positions are (x, y) = (row, col). */
typedef struct MagpoRwareState {
  int32_t* grid;            /* [B,2,H,W]  channel 0: shelf id + 1, channel 1: agent id + 1 */
  int32_t* agent_pos;       /* [B,A,2] */
  int32_t* agent_dir;       /* [B,A]     UP 0, RIGHT 1, DOWN 2, LEFT 3 */
  uint8_t* agent_carry;     /* [B,A] */
  int32_t* shelf_pos;       /* [B,S,2] */
  uint8_t* shelf_req;       /* [B,S] */
  int32_t* request_queue;   /* [B,Q] */
  int32_t* step_count;      /* [B] */
  uint8_t* action_mask;     /* [B,A,5] */
  uint32_t* key;            /* [B,2] */
  uint32_t* metrics_key;    /* [B,2]  RecordEpisodeMetricsState.key */
  float* running_return;    /* [B] */
  int32_t* running_length;  /* [B] */
  float* episode_return;    /* [B] */
  int32_t* episode_length;  /* [B] */
} MagpoRwareState;

/* Number of shelves S of a layout (for sizing shelf_pos / shelf_req); negative error code on a bad config. */
int32_t magpo_rware_num_shelves(const MagpoRwareCfg* cfg);
/* vmap(env.reset)(keys) / vmap(env.step)(state, action) for the RWARE stack; same contract as the CoordSum pair. */
int magpo_rware_reset(magpo_stream_t s, const MagpoRwareCfg* cfg, int32_t B, const uint32_t* keys,
                      MagpoRwareState st, MagpoTimeStep ts);
int magpo_rware_step(magpo_stream_t s, const MagpoRwareCfg* cfg, int32_t B, const int32_t* action,
                     MagpoRwareState st, MagpoTimeStep ts);

/* ------------------------------------------------------------------ GAE
 * calculate_gae — mava/utils/multistep.py:24-68. Layout [T,B,A] (time-major), `done` is per env
 * [T,B] (Transition.done is constant over agents, rec_magpo.py:172), last_done [B]. */
int magpo_gae(magpo_stream_t s, int32_t T, int32_t B, int32_t A, const float* reward,
              const float* value, const uint8_t* done, const float* last_value,
              const uint8_t* last_done, double gamma, double gae_lambda, float* advantages,
              float* targets);

/* ------------------------------------------------------------------ rollout
 * Sable hidden states (systems/gpo/types.py:48-53): three arrays [B, n_head, n_block, hs, hs]. */
typedef struct MagpoSableHState {
  float* encoder;
  float* decoder_self;
  float* decoder_cross;
} MagpoSableHState;

/* The trajectory batch (GPOTransition, systems/gpo/types.py:74-83) plus the observation slots the
 * rollout ping-pongs through: slot t holds the observation acted on at step t; slot T is the
 * bootstrap observation (= LearnerState.timestep after the rollout). */
typedef struct MagpoTrajectory {
  uint8_t* done;        /* [T+1,B]     Transition.done (= previous step's done), per env */
  float* agents_view;   /* [T+1,B,A,d] */
  uint8_t* action_mask; /* [T+1,B,A,a] */
  int32_t* step_count;  /* [T+1,B,A] */
  int32_t* action;      /* [T,B,A] */
  float* value;         /* [T,B,A] */
  float* reward;        /* [T,B,A] */
  float* log_prob;      /* [T,B,A] */
  float* policy_h0;     /* [B,A,H]   Transition.hstates.policy_hidden_state[0] (rec_magpo.py:244-248) */
  MagpoSableHState sable_h0; /* prev_sable_hstates (rec_magpo.py:190-192) */
  float* episode_return;     /* [T,B] */
  int32_t* episode_length;   /* [T,B] */
  uint8_t* is_terminal_step; /* [T,B] */
  float* last_value;    /* [B,A]  bootstrap value (rec_magpo.py:202-208) */
} MagpoTrajectory;

enum { MAGPO_ENV_COORDSUM = 0, MAGPO_ENV_LBF = 1, MAGPO_ENV_RWARE = 2 };

size_t magpo_rollout_workspace_bytes(const MagpoNetCfg* net, int32_t B, int32_t T);

/* lax.scan(_env_step, length=T) + the bootstrap value — rec_magpo.py:126-208 — for B = U*E envs
 * (slot-major: b = u*E + e; every slot runs the same key stream, rec_magpo.py:660-673).
 *   guider/actor : flat parameter buffers;
 *   key          : uint32[2] LearnerState.key, advanced in place (T+1 splits);
 *   env_state    : Magpo<Env>State* matching env_kind; ts : timestep scratch/outputs (reward etc. of
 *                  the LAST step remain there; observation slots live in `traj`);
 *   hs / policy_h: recurrent state in/out ([B,A,H] for the learner GRU);
 *   On entry slot 0 of traj.{done,agents_view,action_mask,step_count} holds the current observation
 *   (carry_over == 0), or slot T does and is first copied to slot 0 (carry_over != 0: the LearnerState.timestep
 *   left by the previous call).  The Sable states in `hs` are stored WITHOUT the reset of rec_magpo.py:165-169;
 *   the reset is applied from traj.done when they are next read (and when they are copied to traj.sable_h0), so
 *   the reference's hstates are `where(done[T], 0, hs)`. */
int magpo_rollout(MagpoContext* ctx, magpo_stream_t s, const MagpoNetCfg* net, const MagpoSysCfg* sys, int env_kind,
                  const void* env_cfg, void* env_state, MagpoTimeStep ts, const float* guider,
                  const float* actor, uint32_t* key, MagpoSableHState hs, float* policy_h,
                  MagpoTrajectory traj, int32_t carry_over, void* workspace, size_t workspace_bytes);

/* SableNetwork.get_actions (networks/sable_network.py:443-482) for B envs, one timestep.
 * sample_keys [A,2]: the per-agent `sample_key`s of discrete_autoregressive_act (decode.py:140);
 * gumbel_rows E: noise index of env b is (b % E)*a + j.  Updates hs in place (decay included).
 * Any of action/log_prob/logits may be NULL; with action==NULL only the encoder/value runs. */
int magpo_sable_get_actions(MagpoContext* ctx, magpo_stream_t s, const MagpoNetCfg* net, int32_t B, int32_t gumbel_rows,
                            const float* guider, const float* agents_view, const uint8_t* action_mask,
                            const int32_t* step_count, const uint8_t* prev_done /*[B] or NULL*/,
                            const uint32_t* sample_keys, MagpoSableHState hs, int32_t* action,
                            float* log_prob, float* value, float* logits /*[B,A,a] masked*/,
                            void* workspace, size_t workspace_bytes);

/* RecurrentActor.apply with a length-1 time axis (rec_magpo.py:146-159): h <- GRU(h, obs, done). */
int magpo_actor_step(MagpoContext* ctx, magpo_stream_t s, const MagpoNetCfg* net, int32_t B, const float* actor,
                     const float* agents_view, const uint8_t* done /*[B]*/, float* policy_h,
                     void* workspace, size_t workspace_bytes);

/* ------------------------------------------------------------------ update
 * One minibatch in time-major layout [T, N, A, ...] (N = U * E/M envs, slot-major). This is the
 * reference's (N, T*A, ...) minibatch (rec_magpo.py:453-462) with the time axis outermost. */
typedef struct MagpoMinibatch {
  int32_t T, N;
  const float* agents_view;   /* [T,N,A,d] */
  const uint8_t* action_mask; /* [T,N,A,a] */
  const int32_t* step_count;  /* [T,N,A] */
  const uint8_t* done;        /* [T,N] */
  const int32_t* action;      /* [T,N,A] */
  const float* value;         /* [T,N,A]  old values */
  const float* log_prob;      /* [T,N,A]  old log-probs */
  const float* advantages;    /* [T,N,A]  un-normalised */
  const float* targets;       /* [T,N,A] */
  const float* policy_h0;     /* [N,A,H] */
  MagpoSableHState sable_h0;  /* [N,...] each */
} MagpoMinibatch;

/* Per-epoch shuffle of _update_epoch (rec_magpo.py:439-451), all on device:
 *   key, batch_key, agent_key, _ = split(key, 4) (key advanced in place); batch_perm = permutation(batch_key, E);
 *   agent_perm = permutation(agent_key, A); then for every minibatch m, slot u, position j (layout [M][U][N],
 *   N = E/M):  env_index = u*E + batch_perm[m*N+j],  env_slot = u,  hs_index = u*E + hs_perm'[m*N+j] where
 *   hs_perm' = hs_perm[batch_perm] accumulates over epochs — the reference feeds the already permuted
 *   prev_hstates back into the next epoch (:447,471), so from epoch 2 on the stored Sable states are gathered
 *   through the composition of all permutations so far. hs_perm [E] in/out (ignored on input if first_epoch).
 *   scratch: 4 + 2*max(E,A) + E uint32. */
int magpo_epoch_indices(magpo_stream_t s, const MagpoSysCfg* sys, int32_t A, uint32_t* key, int32_t* hs_perm,
                        int32_t first_epoch, int32_t* batch_perm, int32_t* agent_perm, int32_t* env_index,
                        int32_t* hs_index, int32_t* env_slot, uint32_t* scratch);

/* Mean and population std (jnp.std) of the advantages of each slot's share of a minibatch (:283,356).
 * env_index [n_env] slot-major (n_env/U per slot); scratch: 2*U doubles; stats [U][2] = (mean, std). */
int magpo_adv_stats(magpo_stream_t s, int32_t T, int32_t B, int32_t A, const float* advantages,
                    const int32_t* env_index, int32_t n_env, int32_t U, void* scratch, float* stats);

/* Gathers n_env envs of the trajectory (take(axis=1) by env, take(axis=2) by agent, :445-451) into `out`
 * (time-major [T, n_env, A, ...], out.T == rollout_length, out.N == n_env). A minibatch may be gathered and
 * differentiated in several env chunks; gradients add up. */
int magpo_pack_minibatch(magpo_stream_t s, const MagpoNetCfg* net, const MagpoSysCfg* sys,
                         MagpoTrajectory traj, const float* advantages, const float* targets,
                         const int32_t* env_index, const int32_t* hs_index, const int32_t* agent_perm,
                         int32_t n_env, MagpoMinibatch out);

size_t magpo_update_workspace_bytes(const MagpoNetCfg* net, int32_t T, int32_t N);

/* guider_grad_fn + actor_grad_fn of _update_minibatch (rec_magpo.py:222-391) for the envs held in `mb`.
 *   env_slot [mb.N]: update-batch slot of each env; adv_stats [U][2]: magpo_adv_stats of the whole minibatch;
 *   inv_tokens = 1 / (U * (E/M) * T * A): weight of one token in the slot-averaged mean losses (:395-405).
 *   grads : [n_guider + n_actor + 8] flat, ACCUMULATED into (zero it per optimiser step): guider grads |
 *           learner grads | {-, guider_loss, entropy, value_loss, kl_loss, -, actor_loss, actor_kl}
 *           — the buffer that is all-reduced over devices (the pmean over "device", :399-409): with reduce_grads != 0 and a
 *           communicator attached to the context (magpo_context_set_comm) this call does it itself — sum over ranks, the learner's
 *           half + loss sums on the learner's stream under the guider's remaining backward, the guider's half at the end; pass
 *           reduce_grads only with the LAST env chunk of a minibatch. Otherwise the caller reduces (magpo_comm_allreduce_sum). */
int magpo_minibatch_grads(MagpoContext* ctx, magpo_stream_t s, const MagpoNetCfg* net, const MagpoSysCfg* sys,
                          const float* guider, const float* actor, MagpoMinibatch mb, const int32_t* env_slot,
                          const float* adv_stats, float inv_tokens, float* grads, int32_t reduce_grads,
                          void* workspace, size_t workspace_bytes);

/* Forward-only pieces of the above, exposed for parity tests:
 * SableNetwork.__call__ (sable_network.py:412-441): value [T,N,A], masked logits [T,N,A,a]. */
int magpo_guider_forward(MagpoContext* ctx, magpo_stream_t s, const MagpoNetCfg* net, const float* guider,
                         MagpoMinibatch mb, float* value, float* logits, void* workspace,
                         size_t workspace_bytes);
/* RecurrentActor.apply over T steps (rec_magpo.py:243-250): masked logits [T,N,A,a]. */
int magpo_actor_forward(MagpoContext* ctx, magpo_stream_t s, const MagpoNetCfg* net, const float* actor,
                        MagpoMinibatch mb, float* logits, void* workspace, size_t workspace_bytes);

/* optax.chain(clip_by_global_norm(max_norm), adam(lr, eps=1e-5)) + apply_updates
 * (rec_magpo.py:581-589,412-423; optax 0.2.4). grads are multiplied by grad_scale first (1/Nd
 * after a sum all-reduce). count: device int32 scalar, incremented. scratch: >= 1024 floats. */
int magpo_clip_adam(magpo_stream_t s, int64_t n, float* params, const float* grads, float* mu,
                    float* nu, int32_t* count, float grad_scale, float lr, float max_norm,
                    float* scratch);
/* The same with make_learning_rate's `decay_learning_rates` schedule (mava/utils/training.py:30-64; rec_magpo.py:581):
 * lr_t = lr * (1 - (count // decay_period) / num_updates), decay_period = ppo_epochs * num_minibatches, evaluated on the
 * device from the optimiser count before it is incremented (optax scale_by_schedule). decay_period == 0: constant lr. */
int magpo_clip_adam_sched(magpo_stream_t s, int64_t n, float* params, const float* grads, float* mu,
                          float* nu, int32_t* count, float grad_scale, float lr, int32_t decay_period,
                          int32_t num_updates, float max_norm, float* scratch);

/* ------------------------------------------------------------------ rec_ippo
 * mava/systems/ppo/anakin/rec_ippo.py: recurrent IPPO, the learner's GRU actor (parameters `which` 1) beside a GRU critic (RecurrentValueNet,
 * parameters `which` 2), trained with rec_sable's clipped PPO + clipped value loss. The same conventions as above; each entry point sizes its
 * own workspace (CUB style): with workspace == NULL it writes the bytes it needs to *workspace_bytes and returns MAGPO_OK, otherwise
 * *workspace_bytes is the capacity of `workspace`. The update between these calls is magpo_gae, magpo_adv_stats and magpo_clip_adam_sched. */

/* lax.scan(_env_step, length=T) + the bootstrap value for B = U*E envs (slot-major, every slot on the same key), per step:
 * key, policy_key = split(key); actor and critic each take (obs_t, last_done) and reset their own carry where last_done is set; the action
 * is Categorical(masked logits).sample(seed=policy_key) with tfp's noise layout (element (e, agent, j) uses counter (e*A + agent)*a + j,
 * e = b mod E); env.step. The bootstrap value is the critic on the final observation, final critic state and last done (its new state
 * discarded, no key consumed): `key` advances by exactly T splits. traj.value gets the critic's values, traj.sable_h0 is not used;
 * traj.policy_h0 / critic_h0 [B,A,H] receive the actor's / critic's state before the first step. policy_h / critic_h [B,A,H] in/out.
 * Observation slots and carry_over as for magpo_rollout. */
int magpo_ippo_rollout(MagpoContext* ctx, magpo_stream_t s, const MagpoNetCfg* net, const MagpoSysCfg* sys, int env_kind,
                       const void* env_cfg, void* env_state, MagpoTimeStep ts, const float* actor, const float* critic, uint32_t* key,
                       float* policy_h, float* critic_h, MagpoTrajectory traj, float* critic_h0, int32_t carry_over, void* workspace,
                       size_t* workspace_bytes);

/* Per-epoch shuffle: key, shuffle_key, _ = split(key, 3) (key advanced in place); perm = permutation(shuffle_key, E); for every minibatch
 * m, slot u, position j (layout [M][U][N], N = E/M): env_index = u*E + perm[m*N + j], env_slot = u. No agent shuffle and no permutation
 * carried across epochs. */
int magpo_ippo_epoch_indices(magpo_stream_t s, const MagpoSysCfg* sys, uint32_t* key, int32_t* perm /*[E]*/, int32_t* env_index,
                             int32_t* env_slot, void* workspace, size_t* workspace_bytes);

/* Gathers n_env envs of the trajectory, agents in order, into `out` (out.sable_h0 unused) and both stored t = 0 hidden states by
 * env_index: traj.policy_h0 -> out.policy_h0, critic_h0 [B,A,H] -> out_critic_h0 [n_env,A,H]. */
int magpo_ippo_pack_minibatch(magpo_stream_t s, const MagpoNetCfg* net, const MagpoSysCfg* sys, MagpoTrajectory traj,
                              const float* critic_h0, const float* advantages, const float* targets, const int32_t* env_index, int32_t n_env,
                              MagpoMinibatch out, float* out_critic_h0);

/* actor_grad_fn + critic_grad_fn for the envs held in `mb` (critic_h0 [mb.N,A,H]); env_slot / adv_stats / inv_tokens as for
 * magpo_minibatch_grads. grads [n_actor + n_critic + 8], ACCUMULATED into: actor grads | critic grads | {-, actor_loss, entropy,
 * value_loss, 0, -, actor_loss, 0} (the slots of magpo_minibatch_grads with rec_sable's values). With reduce_grads != 0 and a communicator
 * attached to the context, the whole buffer is sum-all-reduced over the ranks at the end. */
int magpo_ippo_minibatch_grads(MagpoContext* ctx, magpo_stream_t s, const MagpoNetCfg* net, const MagpoSysCfg* sys, const float* actor,
                               const float* critic, MagpoMinibatch mb, const float* critic_h0, const int32_t* env_slot,
                               const float* adv_stats, float inv_tokens, float* grads, int32_t reduce_grads, void* workspace,
                               size_t* workspace_bytes);

/* ------------------------------------------------------------------ data-parallel exchange
 * `jax.lax.pmean(..., "device")` (rec_magpo.py:399-409) as NCCL all-reduces over NVLink / NVSwitch, one process per GPU. libnccl.so.2
 * is resolved with dlopen at first use (no link-time dependency). Bootstrap: rank 0 calls magpo_comm_unique_id, the 128 bytes reach
 * the other ranks by any host channel (the launcher's key-value store), every rank calls magpo_comm_init with its device current.
 * The reductions are sums; the mean's 1/Nd is magpo_clip_adam's grad_scale. */
typedef struct MagpoComm MagpoComm;
int magpo_comm_available(void); /* 1 if libnccl could be loaded */
int magpo_comm_version(void);   /* ncclGetVersion code, 0 if unavailable */
int magpo_comm_unique_id(void* id128 /* out: 128 bytes */);
int magpo_comm_init(int32_t nranks, int32_t rank, const void* id128, MagpoComm** out);
int magpo_comm_destroy(MagpoComm* comm);
int magpo_comm_allreduce_sum(MagpoComm* comm, magpo_stream_t s, float* buf, int64_t n); /* in place, enqueued on s */
int magpo_comm_allreduce_max(MagpoComm* comm, magpo_stream_t s, float* buf, int64_t n);
/* Attach (or with NULL detach) the communicator magpo_minibatch_grads reduces through. The context does not own it. */
int magpo_context_set_comm(MagpoContext* ctx, MagpoComm* comm);

#ifdef __cplusplus
}
#endif
#endif /* MAGPO_B200_H_ */
