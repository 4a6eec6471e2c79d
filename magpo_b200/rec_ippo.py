"""System entry mirroring `mava/systems/ppo/anakin/rec_ippo.py`: recurrent IPPO, the learner's GRU actor beside a GRU critic
(RecurrentValueNet, networks/base.py:187-226), both on the learner's kernels (libmagpo_b200.so, `magpo_ippo_*`).

`learner_setup(env, (key, actor_net_key, critic_net_key), config) -> (learn, actor_network, init_learner_state)`, `RNNLearnerState(params,
opt_states, key, env_state, timestep, dones, hstates)` with every leaf leading `[1, U, ...]`, `learn` returning `ExperimentOutput` with the
four train metrics of rec_ippo. The loss is rec_sable's (clipped PPO - entropy bonus + clipped value loss), evaluated by the MAGPO loss
kernel on (actor logits, critic values) exactly as rec_sable feeds it; oracle/ippo.py restates it independently.

    python -m magpo_b200.rec_ippo env=lbf arch.num_envs=1024 system.num_updates=8 arch.num_evaluation=2
"""
from __future__ import annotations

import ctypes as C
import sys
import time
from dataclasses import dataclass
from typing import Any, Dict, NamedTuple, Tuple

import numpy as np
import torch

from . import _lib as L
from . import init as minit
from . import rec_magpo as rm
from .config import Config, check_total_timesteps, compose
from .learner import NetworkConfig, SystemConfig, alloc_timestep, param_table, param_views, load_params


@dataclass
class IppoSystemConfig(SystemConfig):
    """configs/system/ppo/rec_ippo.yaml: rec_magpo's hyper-parameters plus the critic's learning rate."""
    critic_lr: float = 2.5e-4


class Params(NamedTuple):
    actor_params: Dict[str, torch.Tensor]
    critic_params: Dict[str, torch.Tensor]


class OptStates(NamedTuple):
    actor_opt_state: tuple
    critic_opt_state: tuple


class HiddenStates(NamedTuple):
    policy_hidden_state: torch.Tensor
    critic_hidden_state: torch.Tensor


class RNNLearnerState(NamedTuple):
    params: Params
    opt_states: OptStates
    key: torch.Tensor
    env_state: Dict[str, torch.Tensor]
    timestep: rm.TimeStep
    dones: torch.Tensor
    hstates: HiddenStates


class IppoLearner:
    """All device buffers of one rank + `update_step()` (rollout, GAE, P epochs x M minibatches) of rec_ippo. The rollout is replayed
    from one CUDA graph after its first (eager) call, as MagpoLearner's is. `.dev`, `.net`, `.c_net` and `.ctx` serve the learner-policy
    evaluator (evaluator.get_eval_fn through rec_magpo.ActorNetwork)."""

    def __init__(self, env, sys: IppoSystemConfig, device="cuda:0", world_size: int = 1, graph_rollout: bool = True):
        self.env, self.sys, self.dev = env, sys, torch.device(device)
        if sys.decay_learning_rates and sys.num_updates < 1:
            raise ValueError("decay_learning_rates needs system.num_updates >= 1 (utils/training.py:38-44)")
        T, E, U, M = sys.rollout_length, sys.num_envs, sys.update_batch_size, sys.num_minibatches
        if E % M:
            raise ValueError("num_envs must be divisible by num_minibatches")
        self.ctx = L.create_context(self.dev)
        self.graph_rollout, self._rollout_graph, self._rollout_graph_launches = graph_rollout, None, 0
        self.world_size, self.comm = world_size, None
        self.net = NetworkConfig(env.num_agents, env.obs_dim, env.action_dim, env.time_limit)
        self.c_net, self.c_sys = self.net.c_struct(), sys.c_struct()
        dev, f32, i32, u8 = self.dev, torch.float32, torch.int32, torch.uint8
        A, d, a, H = self.net.n_agents, self.net.obs_dim, self.net.action_dim, self.net.hidden
        B = self.B = U * E
        self.a_table, self.n_a = param_table(self.net, 1)
        self.c_table, self.n_c = param_table(self.net, 2)
        z = lambda *s, dt=f32: torch.zeros(*s, dtype=dt, device=dev)
        self.actor, self.critic = z(self.n_a), z(self.n_c)
        self.a_mu, self.a_nu, self.c_mu, self.c_nu = z(self.n_a), z(self.n_a), z(self.n_c), z(self.n_c)
        self.a_count, self.c_count = z(1, dt=i32), z(1, dt=i32)
        self.grads = z(self.n_a + self.n_c + 8)
        self.key = z(2, dt=i32)
        self.env_state = env.alloc_state(B, dev)
        self.ts = alloc_timestep(B, A, d, a, dev)
        self.policy_h, self.critic_h = z(B, A, H), z(B, A, H)
        self.traj = dict(done=z(T + 1, B, dt=u8), agents_view=z(T + 1, B, A, d), action_mask=z(T + 1, B, A, a, dt=u8),
                         step_count=z(T + 1, B, A, dt=i32), action=z(T, B, A, dt=i32), value=z(T, B, A), reward=z(T, B, A),
                         log_prob=z(T, B, A), policy_h0=z(B, A, H), episode_return=z(T, B), episode_length=z(T, B, dt=i32),
                         is_terminal_step=z(T, B, dt=u8), last_value=z(B, A))
        self.critic_h0 = z(B, A, H)
        self.adv, self.targets = z(T, B, A), z(T, B, A)
        Nmb = self.Nmb = U * (E // M)
        self.chunk = Nmb if sys.chunk_envs <= 0 else min(sys.chunk_envs, Nmb)
        n = self.chunk
        self.mb = dict(agents_view=z(T, n, A, d), action_mask=z(T, n, A, a, dt=u8), step_count=z(T, n, A, dt=i32), done=z(T, n, dt=u8),
                       action=z(T, n, A, dt=i32), value=z(T, n, A), log_prob=z(T, n, A), advantages=z(T, n, A), targets=z(T, n, A),
                       policy_h0=z(n, A, H))
        self.mb_critic_h0 = z(n, A, H)
        self.perm, self.env_index, self.env_slot = z(E, dt=i32), z(M * Nmb, dt=i32), z(M * Nmb, dt=i32)
        self.stats, self.stats_scratch = z(U, 2), z(2 * U, dt=torch.float64)
        self.adam_scratch = z(1024)
        cn, cs = C.byref(self.c_net), C.byref(self.c_sys)
        wr = L.workspace_bytes("magpo_ippo_rollout", None, None, cn, cs, env.kind, None, None, L.TimeStep(), None, None, None, None, None,
                               L.Trajectory(), None, 0)
        wi = L.workspace_bytes("magpo_ippo_epoch_indices", None, cs, None, None, None, None)
        mbs = self._mb_struct(n)
        wu = L.workspace_bytes("magpo_ippo_minibatch_grads", None, None, cn, cs, None, None, mbs, None, None, None, C.c_float(0), None, 0)
        self.ws_bytes = max(wr, wi, wu)
        self.workspace = torch.empty(self.ws_bytes, dtype=u8, device=dev)
        self.first_rollout = True

    def __del__(self):
        try:
            torch.cuda.synchronize(self.dev)
            L.destroy_context(self.ctx)
        except Exception:
            pass

    # ------------------------------------------------------------------ structs
    def _traj_struct(self):
        return L.struct_of(L.Trajectory, **self.traj)

    def _mb_struct(self, n):
        s = L.struct_of(L.Minibatch, **self.mb)
        s.T, s.N = self.sys.rollout_length, n
        return s

    # ------------------------------------------------------------------ setup
    def set_params(self, actor: dict, critic: dict) -> None:
        load_params(self.actor, self.a_table, actor)
        load_params(self.critic, self.c_table, critic)

    def set_opt_state(self, actor_opt: dict, critic_opt: dict) -> None:
        """Both Adam states: dicts with `count`, `mu`, `nu` (the moments keyed like the parameters)."""
        for opt, table, mu, nu, cnt in ((actor_opt, self.a_table, self.a_mu, self.a_nu, self.a_count),
                                        (critic_opt, self.c_table, self.c_mu, self.c_nu, self.c_count)):
            load_params(mu, table, opt["mu"])
            load_params(nu, table, opt["nu"])
            cnt.fill_(int(opt["count"]))

    def get_params(self):
        return ({k: v.clone() for k, v in param_views(self.actor, self.a_table).items()},
                {k: v.clone() for k, v in param_views(self.critic, self.c_table).items()})

    def reset(self, env_keys, step_key) -> None:
        """vmap(env.reset)(env_keys) for this rank's U*E envs + the shared step key, zero hidden states."""
        B = self.B
        keys = torch.as_tensor(np.asarray(env_keys, dtype=np.uint32).view(np.int32).reshape(B, 2)).to(self.dev)
        self.key.copy_(torch.as_tensor(np.asarray(step_key, dtype=np.uint32).view(np.int32)))
        ts = dict(self.ts)
        ts.update(agents_view=self.traj["agents_view"][0], action_mask=self.traj["action_mask"][0], step_count=self.traj["step_count"][0])
        L.call(self.env.reset_fn, L.stream_ptr(), C.byref(self.env.cfg), B, L.ptr(keys), self.env.state_struct(self.env_state),
               L.struct_of(L.TimeStep, **ts))
        self.traj["done"][0].zero_()
        self.policy_h.zero_()
        self.critic_h.zero_()
        self.first_rollout = True
        torch.cuda.current_stream().synchronize()  # `keys` must outlive the launch

    # ------------------------------------------------------------------ the step
    def _rollout_call(self, carry_over: int) -> None:
        n = C.c_size_t(self.ws_bytes)
        L.call("magpo_ippo_rollout", self.ctx, L.stream_ptr(), C.byref(self.c_net), C.byref(self.c_sys), self.env.kind,
               C.byref(self.env.cfg), C.byref(self.env.state_struct(self.env_state)), L.struct_of(L.TimeStep, **self.ts), L.ptr(self.actor),
               L.ptr(self.critic), L.ptr(self.key), L.ptr(self.policy_h), L.ptr(self.critic_h), self._traj_struct(), L.ptr(self.critic_h0),
               carry_over, L.ptr(self.workspace), C.byref(n))

    def rollout(self) -> None:
        if self.first_rollout or not self.graph_rollout:
            self._rollout_call(0 if self.first_rollout else 1)
            self.first_rollout = False
            return
        lib = L.lib()
        if self._rollout_graph is None:
            lib.magpo_launch_count.restype = C.c_int64
            n0 = lib.magpo_launch_count()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self._rollout_call(1)
            self._rollout_graph_launches = int(lib.magpo_launch_count() - n0)
            lib.magpo_launch_count_add(C.c_int64(-self._rollout_graph_launches))  # capturing launched nothing
            self._rollout_graph = g
        self._rollout_graph.replay()
        lib.magpo_launch_count_add(C.c_int64(self._rollout_graph_launches))

    def gae(self) -> None:
        T, B, A = self.sys.rollout_length, self.B, self.net.n_agents
        L.call("magpo_gae", L.stream_ptr(), T, B, A, L.ptr(self.traj["reward"]), L.ptr(self.traj["value"]), L.ptr(self.traj["done"]),
               L.ptr(self.traj["last_value"]), L.ptr(self.traj["done"][T]), C.c_double(self.sys.gamma), C.c_double(self.sys.gae_lambda),
               L.ptr(self.adv), L.ptr(self.targets))

    def epoch_indices(self) -> None:
        n = C.c_size_t(self.ws_bytes)
        L.call("magpo_ippo_epoch_indices", L.stream_ptr(), C.byref(self.c_sys), L.ptr(self.key), L.ptr(self.perm), L.ptr(self.env_index),
               L.ptr(self.env_slot), L.ptr(self.workspace), C.byref(n))

    def minibatch_grads(self, m: int) -> None:
        """Zeroes self.grads and accumulates the slot-averaged gradients + loss sums of minibatch m."""
        sysc, s, Nmb = self.sys, L.stream_ptr(), self.Nmb
        T, A = sysc.rollout_length, self.net.n_agents
        env_index = self.env_index[m * Nmb:(m + 1) * Nmb]
        env_slot = self.env_slot[m * Nmb:(m + 1) * Nmb]
        self.grads.zero_()
        L.call("magpo_adv_stats", s, T, self.B, A, L.ptr(self.adv), L.ptr(env_index), Nmb, sysc.update_batch_size, L.ptr(self.stats_scratch),
               L.ptr(self.stats))
        inv_tokens = 1.0 / (Nmb * T * A)
        for c0 in range(0, Nmb, self.chunk):
            n = min(self.chunk, Nmb - c0)
            mbs = self._mb_struct(n)
            L.call("magpo_ippo_pack_minibatch", s, C.byref(self.c_net), C.byref(self.c_sys), self._traj_struct(), L.ptr(self.critic_h0),
                   L.ptr(self.adv), L.ptr(self.targets), L.ptr(env_index[c0:c0 + n]), n, mbs, L.ptr(self.mb_critic_h0))
            last = c0 + n >= Nmb  # the attached communicator reduces once the whole minibatch has been accumulated
            ws = C.c_size_t(self.ws_bytes)
            L.call("magpo_ippo_minibatch_grads", self.ctx, s, C.byref(self.c_net), C.byref(self.c_sys), L.ptr(self.actor), L.ptr(self.critic),
                   mbs, L.ptr(self.mb_critic_h0), L.ptr(env_slot[c0:c0 + n]), L.ptr(self.stats), C.c_float(inv_tokens), L.ptr(self.grads),
                   1 if (last and self.comm is not None) else 0, L.ptr(self.workspace), C.byref(ws))

    def apply_grads(self) -> None:
        sysc, s = self.sys, L.stream_ptr()
        scale = 1.0 / self.world_size
        period = sysc.ppo_epochs * sysc.num_minibatches if sysc.decay_learning_rates else 0
        g_a, g_c = self.grads[:self.n_a], self.grads[self.n_a:self.n_a + self.n_c]
        # each network has its own clip_by_global_norm + adam on its own learning rate, both on the same schedule
        for n, p, g, mu, nu, cnt, lr, scr in ((self.n_a, self.actor, g_a, self.a_mu, self.a_nu, self.a_count, sysc.actor_lr, self.adam_scratch),
                                              (self.n_c, self.critic, g_c, self.c_mu, self.c_nu, self.c_count, sysc.critic_lr,
                                               self.adam_scratch[512:])):
            L.call("magpo_clip_adam_sched", s, C.c_int64(n), L.ptr(p), L.ptr(g), L.ptr(mu), L.ptr(nu), L.ptr(cnt), C.c_float(scale),
                   C.c_float(lr), period, int(sysc.num_updates), C.c_float(sysc.max_grad_norm), L.ptr(scr))

    def update_step(self):
        """One `_update_step`. Returns (episode metrics dict of [T,B] tensors (views), loss tensor [P,M,8])."""
        sysc = self.sys
        self.rollout()
        self.gae()
        losses = torch.empty(sysc.ppo_epochs, sysc.num_minibatches, 8, device=self.dev)
        for p in range(sysc.ppo_epochs):
            self.epoch_indices()
            for m in range(sysc.num_minibatches):
                self.minibatch_grads(m)
                self.apply_grads()
                losses[p, m] = self.grads[self.n_a + self.n_c:] * (1.0 / self.world_size)
        metrics = dict(episode_return=self.traj["episode_return"], episode_length=self.traj["episode_length"],
                       is_terminal_step=self.traj["is_terminal_step"])
        return metrics, losses

    @staticmethod
    def loss_info(losses: torch.Tensor, sys: SystemConfig) -> dict:
        """The four train metrics of rec_ippo from the [.., 8] loss sums (the slots rec_sable reads): total = actor total + critic total."""
        al, ent, vl = losses[..., 1], losses[..., 2], losses[..., 3]
        return dict(total_loss=al - sys.ent_coef * ent + sys.vf_coef * vl, value_loss=vl, actor_loss=al, entropy=ent)


# ----------------------------------------------------------------------------- the pytree
def _cur_slot(lrn: IppoLearner) -> int:
    return 0 if lrn.first_rollout else lrn.sys.rollout_length


def _replicated_views(lrn: IppoLearner):
    U = lrn.sys.update_batch_size
    rep = lambda t: t.reshape(1, 1, *t.shape).expand(1, U, *t.shape)
    tree = lambda flat, table: {k: rep(v) for k, v in param_views(flat, table).items()}
    sched = bool(lrn.sys.decay_learning_rates)
    params = Params(tree(lrn.actor, lrn.a_table), tree(lrn.critic, lrn.c_table))
    opt = OptStates(rm.optax_state(rm.ScaleByAdamState(rep(lrn.a_count[0]), tree(lrn.a_mu, lrn.a_table), tree(lrn.a_nu, lrn.a_table)), sched),
                    rm.optax_state(rm.ScaleByAdamState(rep(lrn.c_count[0]), tree(lrn.c_mu, lrn.c_table), tree(lrn.c_nu, lrn.c_table)), sched))
    return params, opt, rep(lrn.key)


def _state_views(lrn: IppoLearner) -> RNNLearnerState:
    """The learner's device buffers as rec_ippo's RNNLearnerState, every leaf with the leading [1, U, ...] of this device; the leaves
    that need a conversion (CoordSum's int32 observation, boolean masks and dones) are copies remembered in `lrn._exported`."""
    U, E, A = lrn.sys.update_batch_size, lrn.sys.num_envs, lrn.net.n_agents
    k = _cur_slot(lrn)
    lead = lambda t: t.reshape(1, U, E, *t.shape[1:])
    params, opt, key = _replicated_views(lrn)
    exported = {}
    view = lrn.traj["agents_view"][k]
    if lrn.env.kind == L.ENV_COORDSUM:
        view = exported["agents_view"] = view.to(torch.int32)
    mask = exported["action_mask"] = lrn.traj["action_mask"][k].bool()
    obs = rm.Observation(lead(view), lead(mask), lead(lrn.traj["step_count"][k]))
    extras = {"episode_metrics": {"episode_return": lead(lrn.ts["episode_return"]), "episode_length": lead(lrn.ts["episode_length"]),
                                  "is_terminal_step": lead(lrn.ts["is_terminal_step"]).bool()}, "env_metrics": {}}
    ts = rm.TimeStep(lead(lrn.ts["step_type"]), lead(lrn.ts["reward"]), lead(lrn.ts["discount"]), obs, extras)
    dones = exported["dones"] = lead(lrn.traj["done"][k])[..., None].expand(1, U, E, A).bool()
    lrn._exported = exported
    return RNNLearnerState(params, opt, key, {n: lead(v) for n, v in lrn.env_state.items()}, ts, dones,
                           HiddenStates(lead(lrn.policy_h), lead(lrn.critic_h)))


def _adopt(lrn: IppoLearner, state: RNNLearnerState) -> None:
    """Make the learner's buffers hold `state`: its own views / exports cost nothing, anything else is copied in."""
    exported = getattr(lrn, "_exported", {})
    U, E = lrn.sys.update_batch_size, lrn.sys.num_envs
    params, opt, key = _replicated_views(lrn)
    pairs = [(params.actor_params, state.params.actor_params), (params.critic_params, state.params.critic_params), (key, state.key)]
    pairs += [(rm.adam_of(m), rm.adam_of(t)) for m, t in zip(opt, state.opt_states)]
    for m_tree, t_tree in pairs:
        theirs = dict(rm._flatten(t_tree))
        for name, dst in rm._flatten(m_tree):
            src = theirs[name]
            if src.data_ptr() != dst.data_ptr():
                dst[0, 0].copy_(src[0, 0].to(dst.dtype))
    flat = lambda t: t.reshape(U * E, *t.shape[3:])

    def take(dst: torch.Tensor, src, key_: str | None = None) -> None:
        if key_ in exported and src.data_ptr() == exported[key_].data_ptr() and src.dtype == exported[key_].dtype:
            return
        if src.data_ptr() == dst.data_ptr() and src.dtype == dst.dtype:
            return
        dst.copy_(flat(src).reshape(dst.shape).to(dst.dtype))

    for name, dst in lrn.env_state.items():
        take(dst, state.env_state[name])
    k = _cur_slot(lrn)
    ob = state.timestep.observation
    take(lrn.traj["agents_view"][k], ob.agents_view, "agents_view")
    take(lrn.traj["action_mask"][k], ob.action_mask, "action_mask")
    take(lrn.traj["step_count"][k], ob.step_count)
    for name in ("step_type", "reward", "discount"):
        take(lrn.ts[name], getattr(state.timestep, name))
    if not ("dones" in exported and state.dones.data_ptr() == exported["dones"].data_ptr()):
        lrn.traj["done"][k].copy_(flat(state.dones)[:, 0].to(torch.uint8))
    take(lrn.policy_h, state.hstates.policy_hidden_state)
    take(lrn.critic_h, state.hstates.critic_hidden_state)


def get_learner_fn(lrn: IppoLearner, config: Config):
    """rec_ippo's learner_fn: `learn` = num_updates_per_eval x `_update_step`, metrics stacked like scan∘vmap∘scan."""
    n_upd = int(config.system.num_updates_per_eval)
    U, E = lrn.sys.update_batch_size, lrn.sys.num_envs

    def learn(learner_state: RNNLearnerState) -> rm.ExperimentOutput:
        _adopt(lrn, learner_state)
        ep = {k: [] for k in ("episode_return", "episode_length", "is_terminal_step")}
        tr = []
        for _ in range(n_upd):
            metrics, losses = lrn.update_step()
            for k in ep:  # [T, U*E] -> [U, T, E]
                ep[k].append(metrics[k].reshape(-1, U, E).permute(1, 0, 2).clone())
            tr.append(losses.clone())
        episode_metrics = {k: torch.stack(v)[None] for k, v in ep.items()}  # [1, updates, U, T, E]
        episode_metrics["is_terminal_step"] = episode_metrics["is_terminal_step"].bool()
        info = IppoLearner.loss_info(torch.stack(tr), lrn.sys)  # [updates, P, M]
        train_metrics = {k: v[None, :, None].expand(1, n_upd, U, *v.shape[1:]) for k, v in info.items()}
        return rm.ExperimentOutput(_state_views(lrn), episode_metrics, train_metrics)

    return learn


# ----------------------------------------------------------------------------- configuration
def _system_config(config: Config) -> IppoSystemConfig:
    s = config.system
    if not bool(s.get("add_agent_id", True)):
        raise NotImplementedError("system.add_agent_id=False: the env kernels emit the AgentIDWrapper observation only")
    chunk = s.get("recurrent_chunk_size")
    if chunk is not None and int(chunk) != int(s.rollout_length):
        raise NotImplementedError(f"system.recurrent_chunk_size={chunk}: only null or rollout_length (the whole rollout per sequence) is built")
    decay = bool(s.get("decay_learning_rates", False))
    return IppoSystemConfig(decay_learning_rates=decay, num_updates=int(s.get("num_updates") or 0) if decay else 0,
                            num_envs=int(config.arch.num_envs), update_batch_size=int(s.update_batch_size),
                            rollout_length=int(s.rollout_length), ppo_epochs=int(s.ppo_epochs), num_minibatches=int(s.num_minibatches),
                            gamma=float(s.gamma), gae_lambda=float(s.gae_lambda), clip_eps=float(s.clip_eps), ent_coef=float(s.ent_coef),
                            vf_coef=float(s.vf_coef), max_grad_norm=float(s.max_grad_norm), actor_lr=float(s.actor_lr),
                            critic_lr=float(s.critic_lr), chunk_envs=int(config.arch.get("chunk_envs", 0)))


def _check_network(config: Config) -> None:
    """configs/network/rnn.yaml: only the default recurrent actor and critic are built."""
    n = config.network
    hidden = int(n.get("hidden_state_dim", 128))
    if hidden != 128:
        raise NotImplementedError(f"network.hidden_state_dim={hidden}: the GRU kernels are built for 128")
    for which in ("actor_network", "critic_network"):
        rm.check_torsos(n, which, hidden)


def learner_setup(env, keys: Tuple[Any, Any, Any], config: Config, device=None, rank: int = 0, world_size: int = 1, comm=None):
    """rec_ippo's learner_setup. keys = (key, actor_net_key, critic_net_key) as raw uint32[2] arrays."""
    if not torch.cuda.is_available():
        raise RuntimeError("magpo_b200 runs on CUDA devices only (no CPU fallback)")
    device = torch.device(device or f"cuda:{torch.cuda.current_device()}")
    key, actor_net_key, critic_net_key = keys
    sysc = _system_config(config)
    _check_network(config)
    lrn = IppoLearner(env, sysc, device=device, world_size=world_size)
    if comm is not None:  # comm.NcclComm: magpo_ippo_minibatch_grads reduces the gradients itself
        comm.attach(lrn)
    lrn.set_params(minit.flax_init_actor(np.asarray(actor_net_key, np.uint32), env.obs_dim, env.action_dim, lrn.dev),
                   minit.flax_init_critic(np.asarray(critic_net_key, np.uint32), env.obs_dim, lrn.dev))
    U, E = sysc.update_batch_size, sysc.num_envs
    # key, *env_keys = split(key, Nd*U*E + 1); the reset key's split is the step key of every device and slot (as in rec_magpo)
    allk = minit.split(np.asarray(key, np.uint32), world_size * U * E + 1, device)
    step_key = minit.split(allk[0], 2, device)[1]
    lrn.reset(rm.shard_env_keys(allk[1:], world_size, rank, U, E), step_key)
    return get_learner_fn(lrn, config), rm.ActorNetwork(lrn), _state_views(lrn)


def run_experiment(config: Config, device=None, log=print) -> float:
    """rec_ippo's run_experiment: `num_evaluation` x (`learn`, evaluation of the actor), logging MISC / ACT / TRAIN / EVAL events,
    optional checkpoints, the absolute metric with the best actor parameters at the end. Under torchrun one process drives one GPU."""
    import os

    from . import evaluator as mev
    from .checkpointing import Checkpointer, unreplicate_n_dims
    from .logger import LogEvent, MavaLogger

    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    comm = None
    if world > 1:
        from .comm import NcclComm
        comm = NcclComm.from_env(device)
    config = check_total_timesteps(config, world)
    config.system.num_updates_per_eval = config.system.num_updates // config.arch.num_evaluation
    env = rm.make_env(config)
    key, key_e, actor_net_key, critic_net_key = minit.split(minit.prng_key(int(config.system.seed)), 4, device or "cuda:0")
    learn, actor_network, state = learner_setup(env, (key, actor_net_key, critic_net_key), config, device=device, comm=comm, rank=rank,
                                                world_size=world)
    lrn = actor_network.lrn
    evaluator = mev.get_eval_fn(env, actor_network, config, absolute_metric=False, n_devices=world)
    config.logger.system_name = "rec_ippo"
    logger = MavaLogger(config, console_sink=log) if rank == 0 else None
    if logger:
        logger.log_config(config.to_dict())
    save_checkpoint = bool(config.logger.checkpointing.save_model) and rank == 0
    if save_checkpoint:
        checkpointer = Checkpointer(metadata=config, model_name=config.logger.system_name, **config.logger.checkpointing.save_args.to_dict())
    steps = world * config.system.num_updates_per_eval * config.system.rollout_length * config.system.update_batch_size * config.arch.num_envs

    def world_mean(x: torch.Tensor) -> float:
        m = x.float().mean().reshape(1).to(lrn.dev)
        if comm is not None:
            comm.allreduce_sum(m)
            m /= world
        return float(m)

    max_episode_return, best_params, eval_performance = float("-inf"), None, float("nan")
    for ev in range(int(config.arch.num_evaluation)):
        t0 = time.perf_counter()
        out = learn(state)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        state = out.learner_state
        t = int(steps * (ev + 1))
        term = out.episode_metrics["is_terminal_step"].bool()
        if logger:
            logger.log({"timestep": t}, t, ev, LogEvent.MISC)
            if bool(term.any()):
                act = {k: v[term] for k, v in out.episode_metrics.items() if k != "is_terminal_step"}
                act["steps_per_second"] = steps / dt
                logger.log(act, t, ev, LogEvent.ACT)
            logger.log(dict(out.train_metrics), t, ev, LogEvent.TRAIN)
        ks = minit.split(key_e, world + 1, device or "cuda:0")
        key_e, eval_key = ks[0], ks[1 + rank]
        eval_metrics = evaluator(lrn.actor, eval_key)
        eval_performance = world_mean(eval_metrics[config.env.eval_metric])
        if logger:
            logger.log(dict(eval_metrics), t, ev, LogEvent.EVAL)
        if save_checkpoint:
            checkpointer.save(timestep=t, unreplicated_learner_state=unreplicate_n_dims(state), episode_return=eval_performance)
        if config.arch.absolute_metric and max_episode_return <= eval_performance:
            best_params, max_episode_return = lrn.actor.clone(), eval_performance
    if config.arch.absolute_metric and best_params is not None:
        abs_evaluator = mev.get_eval_fn(env, actor_network, config, absolute_metric=True, n_devices=world)
        ks = minit.split(key_e, world + 1, device or "cuda:0")
        abs_metrics = abs_evaluator(best_params, ks[1 + rank])
        world_mean(abs_metrics[config.env.eval_metric])
        if logger:
            logger.log(dict(abs_metrics), int(steps * int(config.arch.num_evaluation)), int(config.arch.num_evaluation) - 1, LogEvent.ABSOLUTE)
    if logger:
        logger.stop()
    return eval_performance


def main(argv=None) -> float:
    return run_experiment(compose("default/rec_ippo", list(sys.argv[1:] if argv is None else argv)))


if __name__ == "__main__":
    main()
