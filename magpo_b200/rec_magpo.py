"""System entry of the B200 path, with the calling convention of `mava/systems/gpo/anakin/rec_magpo.py`:

    learn, actor_network, learner_state = learner_setup(env, (key, actor_net_key, net_key), config)
    out = learn(learner_state)        # ExperimentOutput(learner_state, episode_metrics, train_metrics)

`learner_setup` follows rec_magpo.py:533-685 (network / optimiser / env-state / key construction), `get_learner_fn`
rec_magpo.py:91-104,501-530 (`num_updates_per_eval` consecutive `_update_step`s per call). One process drives one GPU: the
reference's device axis Nd is the process group, so every leaf of the learner state carries the leading `[1, U, ...]` of this
rank's device (Appendix B of SURVEY.md lists the pytree). The leaves are views of the learner's device buffers; `learn`
adopts whatever state it is given (copying leaves that are not its own views), runs on the GPU through libmagpo_b200.so and
returns views again. There is no CPU fallback: without a CUDA device `learner_setup` raises.

    python -m magpo_b200.rec_magpo env=coordsum arch.num_envs=1024 system.num_updates=8 arch.num_evaluation=2
"""
from __future__ import annotations

import ctypes as C
import sys
import time
from typing import Any, Callable, Dict, NamedTuple, Tuple

import numpy as np
import torch

from . import _lib as L
from . import init as minit
from .config import Config, check_total_timesteps, compose
from .learner import CoordSumVec, LbfVec, RwareVec, MagpoLearner, NetworkConfig, SystemConfig, param_views


# ----------------------------------------------------------------------------- types (systems/gpo/types.py:25-83, mava/types.py:199-207)
class Params(NamedTuple):
    guider_params: Dict[str, torch.Tensor]
    actor_params: Dict[str, torch.Tensor]


class EmptyState(NamedTuple):  # optax.EmptyState: clip_by_global_norm and the constant-lr scale carry nothing
    pass


class ScaleByAdamState(NamedTuple):  # optax.ScaleByAdamState
    count: torch.Tensor
    mu: Dict[str, torch.Tensor]
    nu: Dict[str, torch.Tensor]


class ScaleByScheduleState(NamedTuple):  # optax.ScaleByScheduleState (only with system.decay_learning_rates)
    count: torch.Tensor


AdamState = ScaleByAdamState  # the name this module used before the optax-shaped tree


def optax_state(adam: ScaleByAdamState, scheduled: bool) -> tuple:
    """The state tree of `optax.chain(optax.clip_by_global_norm(.), optax.adam(lr, eps=1e-5))` (rec_magpo.py:582-589, optax 0.2.4):
    `(EmptyState(), (ScaleByAdamState(count, mu, nu), EmptyState() | ScaleByScheduleState(count)))` — adam itself is
    chain(scale_by_adam, scale_by_learning_rate), whose second state is a schedule counter only when lr is a callable."""
    return (EmptyState(), (adam, ScaleByScheduleState(adam.count) if scheduled else EmptyState()))


def adam_of(opt_state) -> ScaleByAdamState:
    """The ScaleByAdamState inside an optax-shaped optimiser state (or the bare state itself)."""
    if isinstance(opt_state, ScaleByAdamState):
        return opt_state
    return opt_state[1][0]


class OptStates(NamedTuple):
    guider_opt_state: tuple
    actor_opt_state: tuple


class SableHiddenStates(NamedTuple):
    encoder: torch.Tensor
    decoder_self_retn: torch.Tensor
    decoder_cross_retn: torch.Tensor


class HiddenStates(NamedTuple):
    sable_hidden_state: SableHiddenStates
    policy_hidden_state: torch.Tensor


class Observation(NamedTuple):
    agents_view: torch.Tensor
    action_mask: torch.Tensor
    step_count: torch.Tensor


class TimeStep(NamedTuple):  # jumanji.types.TimeStep field order
    step_type: torch.Tensor
    reward: torch.Tensor
    discount: torch.Tensor
    observation: Observation
    extras: Dict[str, Any]


class GPOLearnerState(NamedTuple):
    params: Params
    opt_states: OptStates
    key: torch.Tensor
    env_state: Dict[str, torch.Tensor]
    timestep: TimeStep
    dones: torch.Tensor
    hstates: HiddenStates


class ExperimentOutput(NamedTuple):
    learner_state: GPOLearnerState
    episode_metrics: Dict[str, torch.Tensor]
    train_metrics: Dict[str, torch.Tensor]


LearnerFn = Callable[[GPOLearnerState], ExperimentOutput]


# jumanji registrations of the CoordSum scenarios (mava/coordsum/__init__.py:6-45): task_name -> constructor kwargs
COORDSUM_REGISTRY = {
    "5x20-80-v0": dict(num_agents=5, num_actions=20, time_limit=100, maxval=80),
    "3x30-50-v0": dict(num_agents=3, num_actions=30, time_limit=100, maxval=50),
    "3x10-30-v0": dict(num_agents=3, num_actions=10, time_limit=100, maxval=30),
    "8x15-100-v0": dict(num_agents=8, num_actions=15, time_limit=100, maxval=100),
}


def make_env(config: Config):
    """mava/utils/make_env.py:90-135,202-218: CoordSum (dynamics in the reference tree), LevelBasedForaging and RobotWarehouse (jumanji 1.1.0
    `RandomGenerator(**scenario.task_config)` + `{**env.kwargs, **scenario.env_kwargs}`). The training wrapper stack
    RecordEpisodeMetrics(AutoResetWrapper(AgentIDWrapper(<Env>Wrapper))) is part of the env-step kernel."""
    name = config.env.env_name
    if name == "CoordSum":
        kw = dict(COORDSUM_REGISTRY.get(config.env.scenario.task_name, {}))
        kw.update(config.env.scenario.get("task_config", {}))
        kw.update(config.env.get("kwargs", {}))
        return CoordSumVec(num_agents=kw["num_agents"], num_actions=kw["num_actions"], time_limit=kw.get("time_limit", 100),
                           maxval=kw.get("maxval"))
    if name == "LevelBasedForaging":
        kw = dict(config.env.scenario.task_config)
        env_kw = {**dict(config.env.get("kwargs", {})), **dict(config.env.scenario.get("env_kwargs", {}) or {})}
        unknown = set(env_kw) - {"time_limit"}
        if unknown:
            raise NotImplementedError(f"LevelBasedForaging kwargs {sorted(unknown)}: only the VectorObserver defaults are built")
        return LbfVec(**kw, time_limit=int(env_kw.get("time_limit", 100)))
    if name == "RobotWarehouse":
        env_kw = {**dict(config.env.get("kwargs", {})), **dict(config.env.scenario.get("env_kwargs", {}) or {})}
        unknown = set(env_kw) - {"time_limit"}
        if unknown:
            raise NotImplementedError(f"RobotWarehouse kwargs {sorted(unknown)} are not built")
        return RwareVec(**dict(config.env.scenario.task_config), time_limit=int(env_kw.get("time_limit", 500)))
    raise NotImplementedError(f"{name}: only CoordSum, LevelBasedForaging and RobotWarehouse dynamics are built")


def check_torsos(network, which: str, hidden: int) -> None:
    """`network.<which>.{pre,post}_torso` must be the default MLPTorso the GRU kernels are built for; anything else raises."""
    an = network.get(which)
    if an is None:
        return
    for name in ("pre_torso", "post_torso"):
        t = an.get(name)
        if t is None:
            continue
        if [int(x) for x in t.layer_sizes] != [hidden] or bool(t.get("use_layer_norm", False)) or t.get("activation", "relu") != "relu":
            raise NotImplementedError(f"network.{which}.{name}: only one Dense({hidden}) + relu layer without layer norm is built "
                                      "(RecurrentActor of configs/network/magpo.yaml:19-31)")


def _network_config(config: Config, env) -> NetworkConfig:
    """`config.network` (configs/network/magpo.yaml) + env dims -> the shapes the kernels are built for. Everything the reference
    reads is read here; a value the kernels do not cover raises instead of being silently ignored (the library's own
    check_net returns MAGPO_ERR_UNSUPPORTED for the same shapes)."""
    n = config.network
    nc, mc = n.net_config, n.memory_config
    if not bool(config.system.get("add_agent_id", True)):
        raise NotImplementedError("system.add_agent_id=False: the env kernels emit the AgentIDWrapper observation only")
    hidden = int(n.get("hidden_state_dim", 128))
    check_torsos(n, "actor_network", hidden)
    # memory_config.timestep_chunk_size: chunking the sequence is mathematically exact (tests/test_oracle.py
    # ::test_timestep_chunking_is_exact), the kernels always run their own chunked scan, so any value is accepted.
    net = NetworkConfig(env.num_agents, env.obs_dim, env.action_dim, env.time_limit, embed_dim=int(nc.embed_dim), n_head=int(nc.n_head),
                        n_block=int(nc.n_block), hidden=hidden, timestep_pe=bool(mc.get("timestep_positional_encoding", True)),
                        decay_scaling_factor=float(mc.get("decay_scaling_factor", 0.8)))
    c = net.c_struct()
    if L.lib().magpo_param_count(C.byref(c), 0) < 0:
        raise NotImplementedError(f"network configuration outside what the kernels implement: {net} (built: embed_dim 32 / 64 / 128, "
                                  "n_head 1 / 2 / 4 with head_size divisible by n_head, n_block 1..3, hidden_state_dim=128, <= 8 agents)")
    return net


def _system_config(config: Config) -> SystemConfig:
    s = config.system
    decay = bool(s.get("decay_learning_rates", False))
    return SystemConfig(decay_learning_rates=decay, num_updates=int(s.get("num_updates") or 0) if decay else 0,
                        num_envs=int(config.arch.num_envs), update_batch_size=int(s.update_batch_size),
                        rollout_length=int(s.rollout_length), ppo_epochs=int(s.ppo_epochs),
                        num_minibatches=int(s.num_minibatches), gamma=float(s.gamma), gae_lambda=float(s.gae_lambda),
                        clip_eps=float(s.clip_eps), ent_coef=float(s.ent_coef), vf_coef=float(s.vf_coef),
                        max_grad_norm=float(s.max_grad_norm), clip_gpo=float(s.clip_gpo), alpha=float(s.alpha),
                        actor_lr=float(s.actor_lr), chunk_envs=int(config.arch.get("chunk_envs", 0)))


class ActorNetwork:
    """`actor_network.apply(params, hstate, (observation, done)) -> (hstate, logits)` of RecurrentActor
    (networks/base.py:161-184) for the evaluator hook (rec_magpo.py:709): masked logits [T, N, A, a]."""

    def __init__(self, lrn: MagpoLearner):
        self.lrn = lrn

    def apply(self, actor_flat: torch.Tensor, hstate: torch.Tensor, observation_done: Tuple[Observation, torch.Tensor]):
        """`RecurrentActor.__call__(policy_hidden_state, (observation, done))` (networks/base.py:161-165): observation leaves
        [T, N, A, ...], done [T, N] (or [T, N, A]: constant over agents), hstate [N, A, 128]. Returns (carry, logits [T, N, A, a]
        with illegal actions at finfo.min). The carry is returned for T == 1 (the evaluator's per-step call); else None."""
        observation, done = observation_done
        if done.dim() == 3:
            done = done[..., 0]
        lrn = self.lrn
        T, N, A = observation.agents_view.shape[:3]
        a, dev = lrn.net.action_dim, lrn.dev
        z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=dev)
        mb = dict(agents_view=observation.agents_view.to(torch.float32).contiguous(),
                  action_mask=observation.action_mask.to(torch.uint8).contiguous(),
                  step_count=observation.step_count.to(torch.int32).contiguous(), done=done.to(torch.uint8).contiguous(),
                  action=z(T, N, A, dt=torch.int32), value=z(T, N, A), log_prob=z(T, N, A), advantages=z(T, N, A),
                  targets=z(T, N, A), policy_h0=hstate.to(torch.float32).contiguous())
        s = L.struct_of(L.Minibatch, **mb)
        s.sable_h0 = L.struct_of(L.SableHState, **{k: z(N, *lrn.net.state_shape) for k in ("encoder", "decoder_self", "decoder_cross")})
        s.T, s.N = T, N
        lib = L.lib()
        lib.magpo_update_workspace_bytes.restype = C.c_size_t
        lib.magpo_rollout_workspace_bytes.restype = C.c_size_t
        nbytes = max(int(lib.magpo_update_workspace_bytes(C.byref(lrn.c_net), T, N)),
                     int(lib.magpo_rollout_workspace_bytes(C.byref(lrn.c_net), N, 0)))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        logits = z(T, N, A, a)
        L.call("magpo_actor_forward", lrn.ctx, L.stream_ptr(), C.byref(lrn.c_net), L.ptr(actor_flat), s, L.ptr(logits), L.ptr(ws),
               C.c_size_t(nbytes))
        carry = None
        if T == 1:
            carry = mb["policy_h0"].clone()
            L.call("magpo_actor_step", lrn.ctx, L.stream_ptr(), C.byref(lrn.c_net), N, L.ptr(actor_flat), L.ptr(mb["agents_view"]),
                   L.ptr(mb["done"]), L.ptr(carry), L.ptr(ws), C.c_size_t(nbytes))
        torch.cuda.current_stream().synchronize()  # the temporaries above must outlive the launches
        return carry, logits

    def initialize_carry(self, n_envs: int) -> torch.Tensor:
        """ScannedRNN.initialize_carry (networks/base.py:144-149)."""
        return torch.zeros(n_envs, self.lrn.net.n_agents, self.lrn.net.hidden, device=self.lrn.dev)


def _cur_slot(lrn: MagpoLearner) -> int:
    """Observation / done slot of the trajectory buffers that holds LearnerState.timestep: T after a rollout, 0 after reset."""
    return 0 if lrn.first_rollout else lrn.sys.rollout_length


def _replicated_views(lrn: MagpoLearner) -> Tuple[Params, OptStates, torch.Tensor]:
    """(params, opt_states, key): the leaves every slot shares, as [1, U, ...] broadcast views of the flat device buffers."""
    U = lrn.sys.update_batch_size
    rep = lambda t: t.reshape(1, 1, *t.shape).expand(1, U, *t.shape)
    tree = lambda flat, table: {k_: rep(v) for k_, v in param_views(flat, table).items()}
    params = Params(tree(lrn.guider, lrn.g_table), tree(lrn.actor, lrn.a_table))
    sched = bool(lrn.sys.decay_learning_rates)
    opt = OptStates(optax_state(ScaleByAdamState(rep(lrn.g_count[0]), tree(lrn.g_mu, lrn.g_table), tree(lrn.g_nu, lrn.g_table)), sched),
                    optax_state(ScaleByAdamState(rep(lrn.a_count[0]), tree(lrn.a_mu, lrn.a_table), tree(lrn.a_nu, lrn.a_table)), sched))
    return params, opt, rep(lrn.key)


def _state_views(lrn: MagpoLearner) -> GPOLearnerState:
    """The learner's device buffers as the reference's pytree (systems/gpo/types.py:25-83), every leaf with the leading
    [1, U, ...] of this device. Leaves are views of the device buffers wherever the reference's dtype and value allow it; the
    leaves that need a conversion (CoordSum's int32 `agents_view`, `dones` as bool[E, A], the Sable states with the post-step reset
    applied) are materialised copies, remembered in `lrn._exported` so that `_adopt` recognises them when they come back."""
    U, E, A = lrn.sys.update_batch_size, lrn.sys.num_envs, lrn.net.n_agents
    k = _cur_slot(lrn)
    lead = lambda t: t.reshape(1, U, E, *t.shape[1:])          # per-env leaves [U*E, ...] -> [1, U, E, ...]
    params, opt, key = _replicated_views(lrn)
    exported = {}
    view = lrn.traj["agents_view"][k]
    nview = lrn.ts["next_agents_view"]
    if lrn.env.kind == L.ENV_COORDSUM:  # AgentIDWrapper keeps the wrapped env's dtype: int32 for CoordSum (wrappers/observation.py:47-52)
        view = exported["agents_view"] = view.to(torch.int32)
        nview = nview.to(torch.int32)
    mask = exported["action_mask"] = lrn.traj["action_mask"][k].bool()
    obs = Observation(lead(view), lead(mask), lead(lrn.traj["step_count"][k]))
    # extras of the wrapper stack (episode_metrics.py:98-102, auto_reset_wrapper.py:52-58, wrappers/{matrax,jumanji}.py): the real next
    # observation's action mask is not materialised (nothing on this path reads extras["real_next_obs"])
    extras = {"episode_metrics": {"episode_return": lead(lrn.ts["episode_return"]), "episode_length": lead(lrn.ts["episode_length"]),
                                  "is_terminal_step": lead(lrn.ts["is_terminal_step"]).bool()},
              "env_metrics": {},
              "real_next_obs": Observation(lead(nview), None, lead(lrn.ts["next_step_count"]))}
    ts = TimeStep(lead(lrn.ts["step_type"]), lead(lrn.ts["reward"]), lead(lrn.ts["discount"]), obs, extras)
    done_env = lrn.traj["done"][k]
    dones = exported["dones"] = lead(done_env)[..., None].expand(1, U, E, A).bool()
    sable = lrn.sable_hidden_state() if not lrn.first_rollout else lrn.hs
    for name in ("encoder", "decoder_self", "decoder_cross"):
        exported["sable/" + name] = sable[name]
    hs = HiddenStates(SableHiddenStates(*(lead(sable[n_]).reshape(1, U, E, *lrn.net.state_shape)
                                          for n_ in ("encoder", "decoder_self", "decoder_cross"))), lead(lrn.policy_h))
    lrn._exported = exported
    return GPOLearnerState(params, opt, key, {k_: lead(v) for k_, v in lrn.env_state.items()}, ts, dones, hs)


def _flatten(x, prefix=""):
    if isinstance(x, torch.Tensor):
        yield prefix, x
    elif isinstance(x, dict):
        for k in x:
            yield from _flatten(x[k], f"{prefix}/{k}")
    elif isinstance(x, tuple):
        names = getattr(x, "_fields", range(len(x)))
        for n, v in zip(names, x):
            yield from _flatten(v, f"{prefix}/{n}")


def _adopt(lrn: MagpoLearner, state: GPOLearnerState) -> None:
    """Make the learner's buffers hold `state` (systems/gpo/types.py:62-71: params, opt_states, key, env_state, timestep, dones,
    hstates). Leaves that are the learner's own views / exports (the state `learn` returned last) cost nothing; anything else — a
    restored checkpoint, a state edited by the caller — is copied in. `timestep.step_type / reward / discount` are outputs of the
    env step only (`_env_step`, rec_magpo.py:126-187, reads `observation` and `last()`, which `dones` carries) and are copied too;
    `extras` are per-step outputs and are not adopted. A component given as None is left as it is (rec_sable has no learner half)."""
    exported = getattr(lrn, "_exported", {})  # keeps the copies handed out last alive, so a pointer match is an identity match
    U, E = lrn.sys.update_batch_size, lrn.sys.num_envs
    params, opt, key = _replicated_views(lrn)
    # replicated leaves: slot 0 of the foreign state is the value (identical across U, rec_magpo.py:660-673)
    pairs = [(params.guider_params, state.params.guider_params), (params.actor_params, state.params.actor_params), (key, state.key)]
    for m_opt, t_opt in zip(opt, state.opt_states):
        pairs.append((adam_of(m_opt), None if t_opt is None else adam_of(t_opt)))
    for m_tree, t_tree in pairs:
        if t_tree is None:
            continue
        theirs = dict(_flatten(t_tree))
        for name, dst in _flatten(m_tree):
            src = theirs[name]
            if src.data_ptr() != dst.data_ptr():
                dst[0, 0].copy_(src[0, 0].to(dst.dtype))
    # per-env leaves: [1, U, E, ...] -> the learner's [U*E, ...] buffers
    flat = lambda t: t.reshape(U * E, *t.shape[3:])

    def take(dst: torch.Tensor, src, key_: str | None = None) -> None:
        if src is None:
            return
        if key_ in exported and src.data_ptr() == exported[key_].data_ptr() and src.dtype == exported[key_].dtype:
            return  # the copy this learner exported, unchanged
        if src.data_ptr() == dst.data_ptr() and src.dtype == dst.dtype:
            return  # a view of the buffer itself
        dst.copy_(flat(src).reshape(dst.shape).to(dst.dtype))

    theirs_env = dict(state.env_state)
    for name, dst in lrn.env_state.items():
        take(dst, theirs_env[name])
    k = _cur_slot(lrn)
    ob = state.timestep.observation
    take(lrn.traj["agents_view"][k], ob.agents_view, "agents_view")
    take(lrn.traj["action_mask"][k], ob.action_mask, "action_mask")
    take(lrn.traj["step_count"][k], ob.step_count)
    for name in ("step_type", "reward", "discount"):
        take(lrn.ts[name], getattr(state.timestep, name))
    if state.dones is not None:
        if not ("dones" in exported and state.dones.data_ptr() == exported["dones"].data_ptr()):
            lrn.traj["done"][k].copy_(flat(state.dones)[:, 0].to(torch.uint8))
    elif state.timestep.step_type.data_ptr() != lrn.ts["step_type"].data_ptr():  # rec_sable's state has no `dones`: timestep.last()
        lrn.traj["done"][k].copy_((flat(state.timestep.step_type) == 2).to(torch.uint8))
    sh = state.hstates.sable_hidden_state
    for name, src in (("encoder", sh.encoder), ("decoder_self", sh.decoder_self_retn), ("decoder_cross", sh.decoder_cross_retn)):
        ex = exported.get("sable/" + name)
        if (ex is None or src.data_ptr() != ex.data_ptr()) and src.data_ptr() != lrn.hs[name].data_ptr():
            lrn.hs[name].copy_(src.reshape(U * E, *lrn.net.state_shape).to(torch.float32))
    take(lrn.policy_h, state.hstates.policy_hidden_state)


def get_learner_fn(lrn: MagpoLearner, config: Config) -> LearnerFn:
    """rec_magpo.py:91-104,501-530: `learn` = num_updates_per_eval x `_update_step`, metrics stacked like scan∘vmap∘scan."""
    n_upd = int(config.system.num_updates_per_eval)
    U, E = lrn.sys.update_batch_size, lrn.sys.num_envs

    def learn(learner_state: GPOLearnerState) -> ExperimentOutput:
        _adopt(lrn, learner_state)
        ep = {k: [] for k in ("episode_return", "episode_length", "is_terminal_step")}
        tr = []
        for _ in range(n_upd):
            metrics, losses = lrn.update_step()
            for k in ep:  # [T, U*E] -> [U, T, E]
                ep[k].append(metrics[k].reshape(-1, U, E).permute(1, 0, 2).clone())
            tr.append(losses.clone())
        episode_metrics = {k: torch.stack(v)[None] for k, v in ep.items()}            # [1, updates, U, T, E]
        episode_metrics["is_terminal_step"] = episode_metrics["is_terminal_step"].bool()
        info = MagpoLearner.loss_info(torch.stack(tr), lrn.sys)                        # [updates, P, M]
        train_metrics = {k: v[None, :, None].expand(1, n_upd, U, *v.shape[1:]) for k, v in info.items()}
        return ExperimentOutput(_state_views(lrn), episode_metrics, train_metrics)

    return learn


def shard_env_keys(all_keys: np.ndarray, world_size: int, rank: int, U: int, E: int) -> np.ndarray:
    """The reference reshapes the Nd*U*E reset keys to (Nd, U, E) (rec_magpo.py:648-653): global env index -> (device, slot,
    env). Returns this rank's [U*E, 2] block, slot-major."""
    all_keys = np.asarray(all_keys, np.uint32)
    assert all_keys.shape == (world_size * U * E, 2), all_keys.shape
    return all_keys.reshape(world_size, U * E, 2)[rank]


def mean_over_devices(flat: torch.Tensor, world_size: int) -> torch.Tensor:
    """`jax.lax.pmean(..., "device")` of the flat (guider grads | learner grads | loss sums) buffer (rec_magpo.py:399-409):
    one sum all-reduce; the 1/Nd factor is applied where the buffer is consumed (magpo_clip_adam's grad_scale, the loss read-out).
    This helper is the host-side statement of that contract (used by the CPU tests with the gloo backend)."""
    import torch.distributed as dist

    if world_size > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    return flat * (1.0 / world_size)


def learner_setup(env: CoordSumVec, keys: Tuple[Any, Any, Any], config: Config, device=None, allreduce=None, rank: int = 0,
                  world_size: int = 1, comm=None) -> Tuple[LearnerFn, ActorNetwork, GPOLearnerState]:
    """rec_magpo.py:533-685. keys = (key, actor_net_key, net_key) as raw uint32[2] arrays (jax.random.PRNGKey layout)."""
    if not torch.cuda.is_available():
        raise RuntimeError("magpo_b200 runs on CUDA devices only (no CPU fallback)")
    device = torch.device(device or f"cuda:{torch.cuda.current_device()}")
    key, actor_net_key, net_key = keys
    config.system.num_agents = env.num_agents  # rec_magpo.py:541-543
    config.system.num_actions = env.action_dim
    lrn = MagpoLearner(env, _system_config(config), device=device, allreduce=allreduce, world_size=world_size,
                       net=_network_config(config, env))
    if comm is not None:  # comm.NcclComm: magpo_minibatch_grads reduces the gradients itself (the pmean over "device", :399-409)
        comm.attach(lrn)
    # parameters: flax's initialisers from the two net keys (rec_magpo.py:596-606) — per-parameter keys folded from the module path,
    # jax.random.normal / truncated_normal draws from the library's threefry kernels, Householder QR for the orthogonal ones
    lrn.set_params(minit.flax_init_guider(np.asarray(net_key, np.uint32), env.num_agents, env.obs_dim, env.action_dim, lrn.dev,
                                          lrn.net.embed_dim, lrn.net.n_head, lrn.net.n_block),
                   minit.flax_init_actor(np.asarray(actor_net_key, np.uint32), env.obs_dim, env.action_dim, lrn.dev))
    U, E = lrn.sys.update_batch_size, lrn.sys.num_envs
    # key, *env_keys = split(key, Nd*U*E + 1); reset_key = split(key)[1] is the step key of every device and slot (:642-673)
    allk = minit.split(np.asarray(key, np.uint32), world_size * U * E + 1, device)
    step_key = minit.split(allk[0], 2, device)[1]
    lrn.reset(shard_env_keys(allk[1:], world_size, rank, U, E), step_key)
    return get_learner_fn(lrn, config), ActorNetwork(lrn), _state_views(lrn)


def run_experiment(config: Config, device=None, log=print) -> float:
    """rec_magpo.py:688-831 (console / JSON logger and an npz checkpointer instead of the TensorBoard / Neptune / orbax back-ends): `num_evaluation` calls of `learn`, each
    `num_updates_per_eval` updates, reporting steps per second and the mean return of the episodes that ended."""
    import os

    # one process per GPU (the reference's device axis): launched under torchrun, the ranks exchange gradients through the library's
    # own NCCL communicator (magpo_b200/comm.py)
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    comm = None
    if world > 1:
        from .comm import NcclComm
        comm = NcclComm.from_env(device)
    config = check_total_timesteps(config, world)
    config.system.num_updates_per_eval = config.system.num_updates // config.arch.num_evaluation
    env = make_env(config)
    key, key_e, actor_net_key, net_key = minit.split(minit.prng_key(int(config.system.seed)), 4, device or "cuda:0")
    learn, actor_network, state = learner_setup(env, (key, actor_net_key, net_key), config, device=device, comm=comm,
                                                rank=rank, world_size=world)
    lrn = actor_network.lrn
    # evaluator of the learner policy (rec_magpo.py:706-710): episodes sharded over the devices, no collective (evaluator.py:163)
    from . import evaluator as mev

    evaluator = mev.get_eval_fn(env, actor_network, config, absolute_metric=False, n_devices=world)
    steps_per_rollout = (world * config.system.num_updates_per_eval * config.system.rollout_length *
                         config.system.update_batch_size * config.arch.num_envs)

    def world_mean(x: torch.Tensor) -> float:
        m = x.float().mean().reshape(1).to(lrn.dev)
        if comm is not None:
            comm.allreduce_sum(m)
            m /= world
        return float(m)

    # logger and checkpointer (rec_magpo.py:729-741); rank 0 logs, as the reference's single process does
    from .checkpointing import Checkpointer, unreplicate_n_dims
    from .logger import LogEvent, MavaLogger

    config.logger.system_name = "rec_magpo"
    logger = MavaLogger(config, console_sink=log) if rank == 0 else None
    if logger:
        logger.log_config(config.to_dict())
    save_checkpoint = bool(config.logger.checkpointing.save_model) and rank == 0
    if save_checkpoint:
        checkpointer = Checkpointer(metadata=config, model_name=config.logger.system_name,
                                    **{k: v for k, v in config.logger.checkpointing.save_args.to_dict().items()})

    max_episode_return, best_params, eval_performance = float("-inf"), None, float("nan")
    for ev in range(int(config.arch.num_evaluation)):
        t0 = time.perf_counter()
        out = learn(state)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        state = out.learner_state
        t = int(steps_per_rollout * (ev + 1))
        # rec_magpo.py:756-767: steps per second, the metrics of the episodes that ended, the mean losses
        term = out.episode_metrics["is_terminal_step"].bool()
        if logger:
            logger.log({"timestep": t}, t, ev, LogEvent.MISC)
            if bool(term.any()):  # get_final_step_metrics (utils/training / logger): only completed episodes are reported
                act = {k: v[term] for k, v in out.episode_metrics.items() if k != "is_terminal_step"}
                act["steps_per_second"] = steps_per_rollout / dt
                logger.log(act, t, ev, LogEvent.ACT)
            logger.log(dict(out.train_metrics), t, ev, LogEvent.TRAIN)
        # rec_magpo.py:770-777: key_e, *eval_keys = split(key_e, n_devices + 1); evaluator(trained_params, eval_keys, ...)
        ks = minit.split(key_e, world + 1, device or "cuda:0")
        key_e, eval_key = ks[0], ks[1 + rank]
        eval_metrics = evaluator(lrn.actor, eval_key)
        eval_performance = world_mean(eval_metrics[config.env.eval_metric])
        if logger:
            logger.log(dict(eval_metrics), t, ev, LogEvent.EVAL)
        if save_checkpoint:  # rec_magpo.py:779-786
            checkpointer.save(timestep=t, unreplicated_learner_state=unreplicate_n_dims(state), episode_return=eval_performance)
        if config.arch.absolute_metric and max_episode_return <= eval_performance:  # rec_magpo.py:787-789
            best_params, max_episode_return = lrn.actor.clone(), eval_performance
    if config.arch.absolute_metric and best_params is not None:  # rec_magpo.py:798-812: 10x episodes with the best parameters
        abs_evaluator = mev.get_eval_fn(env, actor_network, config, absolute_metric=True, n_devices=world)
        ks = minit.split(key_e, world + 1, device or "cuda:0")
        abs_metrics = abs_evaluator(best_params, ks[1 + rank])
        world_mean(abs_metrics[config.env.eval_metric])
        if logger:
            logger.log(dict(abs_metrics), int(steps_per_rollout * int(config.arch.num_evaluation)), int(config.arch.num_evaluation) - 1,
                       LogEvent.ABSOLUTE)
    if logger:
        logger.stop()
    return eval_performance


def main(argv=None) -> float:
    return run_experiment(compose("default/rec_magpo", list(sys.argv[1:] if argv is None else argv)))


if __name__ == "__main__":
    main()
