"""The rec_ippo Anakin learner (recurrent IPPO: GRU actor + GRU critic) restated on CPU — oracle only.

Restates `mava/systems/ppo/anakin/rec_ippo.py` (the reference file is not in this tree, so this restatement is the specification; the
conventions marked "from memory" below each live in exactly one place here):
  * rollout: per step `key, policy_key = split(key)`; actor and critic each reset their carry where `last_done` is set;
    `Categorical(masked logits).sample(seed=policy_key)` with tfp's noise layout; `env.step`; the transition keeps the hidden states
    before the step; bootstrap value = the critic on the final observation (its new state discarded, no key consumed);
  * GAE as rec_magpo (`learner.gae`);
  * epoch: `key, shuffle_key, _ = split(key, 3)`, `perm = permutation(shuffle_key, E)`, minibatch m = envs perm[m*N:(m+1)*N] over the
    whole rollout, agents in order, starting from the stored t = 0 hidden states;
  * losses: actor -mean(min(r A, clip(r) A)) - ent_coef mean(H), critic vf_coef * 0.5 mean(max((v-R)^2, (v_clip-R)^2)); A normalised per
    (slot, minibatch); gradients averaged over slots; one clip_by_global_norm + adam per network (actor_lr / critic_lr, same schedule).
Network math in torch on the CPU (autograd mirrors jax.value_and_grad), built on `nets.actor_apply` for both networks.
"""
from __future__ import annotations

import dataclasses
from dataclasses import dataclass

import numpy as np
import torch

from . import coordsum, learner, nets, prng

# RecurrentValueNet's output layer is created directly in its compact body, so flax names it "Dense_0" (from memory).
CRITIC_HEAD = "Dense_0"


@dataclass
class SysCfg(learner.SysCfg):
    critic_lr: float = 2.5e-4


def init_critic_params(cfg: nets.NetCfg, seed: int = 2) -> dict:
    """RecurrentValueNet's parameters: the actor's torsos and GRU, a Dense(1) head with orthogonal(1.0)."""
    p = nets.init_actor_params(dataclasses.replace(cfg, action_dim=1), seed)
    del p["action_head/Dense_0/kernel"], p["action_head/Dense_0/bias"]
    p[f"{CRITIC_HEAD}/kernel"] = nets._orthogonal(np.random.default_rng(seed + 1000), (cfg.hidden, 1), 1.0)
    p[f"{CRITIC_HEAD}/bias"] = np.zeros(1, np.float32)
    return p


def critic_apply(p, cfg: nets.NetCfg, h, obs, done):
    """RecurrentValueNet.__call__: `nets.actor_apply` with the critic's head read under its own name and no action mask.
    h [E,A,H]; obs [T,E,A,d]; done bool[T,E,A]. Returns (h_T, value [T,E,A])."""
    q = {k: v for k, v in p.items() if not k.startswith(CRITIC_HEAD + "/")}
    q["action_head/Dense_0/kernel"], q["action_head/Dense_0/bias"] = p[f"{CRITIC_HEAD}/kernel"], p[f"{CRITIC_HEAD}/bias"]
    h, v = nets.actor_apply(q, cfg, h, obs, done, torch.ones(*obs.shape[:3], 1, dtype=torch.bool, device=obs.device))
    return h, v[..., 0]


# ----------------------------------------------------------------------------- rollout
def rollout(spec, ncfg: nets.NetCfg, sys: SysCfg, ap_np, cp_np, slot):
    """T steps of `_env_step` + the bootstrap value for one update-batch slot. Mutates `slot` (key, env_state, timestep, dones,
    hstates) and returns (trajectory dict [T,E,...], episode metrics, last_value [E,A])."""
    ap, cp = nets.to_torch(ap_np), nets.to_torch(cp_np)
    T, A = sys.rollout_length, ncfg.n_agents
    traj = {k: [] for k in ("done", "action", "value", "reward", "log_prob", "obs", "action_mask", "step_count")}
    metrics = {k: [] for k in ("episode_return", "episode_length", "is_terminal_step")}
    traj_h0 = dict(policy_h0=slot["hstates"]["policy"].copy(), critic_h0=slot["hstates"]["critic"].copy())
    with torch.no_grad():
        for _ in range(T):
            ks = prng.split(slot["key"])
            slot["key"], policy_key = ks[0], ks[1]
            ob = slot["timestep"]["observation"]
            obs = torch.tensor(ob["agents_view"].astype(np.float32))[None]
            last_done = torch.tensor(slot["dones"])[None]
            ph, logits = nets.actor_apply(ap, ncfg, torch.tensor(slot["hstates"]["policy"]), obs, last_done, torch.tensor(ob["action_mask"])[None])
            ch, value = critic_apply(cp, ncfg, torch.tensor(slot["hstates"]["critic"]), obs, last_done)
            action, logp, _ = prng.categorical_distrax(policy_key, logits[0].numpy())
            env_state, new_ts = learner.env_module(spec).step(spec, slot["env_state"], action)
            done = new_ts["step_type"] == coordsum.STEP_LAST
            traj["done"].append(slot["dones"].copy())
            traj["action"].append(action)
            traj["value"].append(value[0].numpy().astype(np.float32))
            traj["reward"].append(new_ts["reward"])
            traj["log_prob"].append(logp)
            traj["obs"].append(ob["agents_view"])
            traj["action_mask"].append(ob["action_mask"])
            traj["step_count"].append(ob["step_count"])
            for k in metrics:
                metrics[k].append(new_ts["extras"]["episode_metrics"][k])
            slot["env_state"], slot["timestep"] = env_state, new_ts
            slot["dones"] = np.repeat(done[:, None], A, axis=1)
            slot["hstates"] = dict(policy=ph.numpy().astype(np.float32), critic=ch.numpy().astype(np.float32))
        ob = slot["timestep"]["observation"]
        _, last_val = critic_apply(cp, ncfg, torch.tensor(slot["hstates"]["critic"]), torch.tensor(ob["agents_view"].astype(np.float32))[None],
                                   torch.tensor(slot["dones"])[None])
    traj = {k: np.stack(v) for k, v in traj.items()}
    traj.update(traj_h0)
    return traj, {k: np.stack(v) for k, v in metrics.items()}, last_val[0].numpy().astype(np.float32)


# ----------------------------------------------------------------------------- update
def epoch_perm(key, E: int):
    """`key, shuffle_key, _ = split(key, 3)` (from memory) and the env permutation of one epoch. Returns (new key, perm)."""
    k3 = prng.split(key, 3)
    return k3[0], prng.permutation(k3[1], E)


def make_minibatches(traj, adv, targets, perm, M):
    """Minibatch m: envs perm[m*N:(m+1)*N] of the whole rollout, agents in order, time-major [T, N, A, ...]; the stored t = 0 hidden
    states of the same envs."""
    N = perm.shape[0] // M
    full = dict(traj, adv=adv, targets=targets)
    out = []
    for m in range(M):
        envs = perm[m * N:(m + 1) * N]
        mb = {k: np.take(full[k], envs, axis=1) for k in ("done", "action", "value", "log_prob", "obs", "action_mask", "adv", "targets")}
        mb["policy_h0"], mb["critic_h0"] = traj["policy_h0"][envs], traj["critic_h0"][envs]
        out.append(mb)
    return out


def losses(logits, value, mb, sys: SysCfg):
    """rec_ippo's `_actor_loss_fn` / `_critic_loss_fn` bodies after the network calls. logits masked [..., a], value [...]; mb torch
    tensors. Returns (actor_total, critic_total, (actor_loss, entropy, value_loss))."""
    logp_all = nets.log_softmax(logits)
    logp = logp_all.gather(-1, mb["action"].to(torch.int64)[..., None])[..., 0]
    ratio = torch.exp(logp - mb["log_prob"])
    adv = (mb["adv"] - mb["adv"].mean()) / (mb["adv"].std(unbiased=False) + 1e-8)
    actor_loss = -torch.minimum(ratio * adv, torch.clamp(ratio, 1.0 - sys.clip_eps, 1.0 + sys.clip_eps) * adv).mean()
    pr = torch.exp(logp_all)
    entropy = (-(torch.where(pr == 0, torch.zeros_like(pr), logp_all) * pr).sum(-1)).mean()
    v_clip = mb["value"] + (value - mb["value"]).clamp(-sys.clip_eps, sys.clip_eps)
    value_loss = 0.5 * torch.maximum((value - mb["targets"]) ** 2, (v_clip - mb["targets"]) ** 2).mean()
    return actor_loss - sys.ent_coef * entropy, sys.vf_coef * value_loss, (actor_loss, entropy, value_loss)


def minibatch_losses_and_grads(ap_np, cp_np, mb_np, ncfg: nets.NetCfg, sys: SysCfg, dtype=torch.float32):
    """One slot's actor and critic gradients on one minibatch. Returns (actor grads, critic grads, info dict)."""
    ap = nets.to_torch(ap_np, dtype, requires_grad=True)
    cp = nets.to_torch(cp_np, dtype, requires_grad=True)
    mb = {k: torch.tensor(v, dtype=dtype) if v.dtype.kind == "f" else torch.tensor(v) for k, v in mb_np.items()}
    obs = mb["obs"].to(dtype)
    _, logits = nets.actor_apply(ap, ncfg, mb["policy_h0"], obs, mb["done"], mb["action_mask"])
    _, value = critic_apply(cp, ncfg, mb["critic_h0"], obs, mb["done"])
    tot_a, tot_c, (al, ent, vl) = losses(logits, value, mb, sys)
    ga = torch.autograd.grad(tot_a, list(ap.values()))
    gc = torch.autograd.grad(tot_c, list(cp.values()))
    npf = np.float64 if dtype == torch.float64 else np.float32
    a_grads = {k: g.detach().numpy().astype(npf) for k, g in zip(ap, ga)}
    c_grads = {k: g.detach().numpy().astype(npf) for k, g in zip(cp, gc)}
    info = dict(total_loss=float(tot_a.detach()) + float(tot_c.detach()), value_loss=float(vl.detach()), actor_loss=float(al.detach()),
                entropy=float(ent.detach()))
    return a_grads, c_grads, info


def learner_setup(spec, ncfg: nets.NetCfg, sys: SysCfg, seed: int = 42, param_seed: int = 0):
    """Keys, env resets and the replicated state of one device, with the key plumbing of rec_magpo's setup."""
    ks = prng.split(prng.prng_key(seed), 4)
    U, E = sys.update_batch_size, sys.num_envs
    all_keys = prng.split(ks[0], U * E + 1)
    step_key = prng.split(all_keys[0])[1]
    env_keys = all_keys[1:].reshape(U, E, 2)
    ap = nets.init_actor_params(ncfg, param_seed + 1)
    cp = init_critic_params(ncfg, param_seed + 2)
    slots = []
    for u in range(U):
        env_state, ts = learner.env_module(spec).reset(spec, env_keys[u])
        z = np.zeros((E, ncfg.n_agents, ncfg.hidden), np.float32)
        slots.append(dict(key=step_key.copy(), env_state=env_state, timestep=ts, dones=np.zeros((E, ncfg.n_agents), bool),
                          hstates=dict(policy=z.copy(), critic=z.copy())))
    return dict(actor_params=ap, critic_params=cp, actor_opt=learner.init_opt(ap), critic_opt=learner.init_opt(cp), slots=slots)


def update_step(state, spec, ncfg: nets.NetCfg, sys: SysCfg, record=None, dtype=torch.float32):
    """One `_update_step` for the U slots of one device. `record` (dict) collects the trajectories for parity tests."""
    f = np.float64 if dtype == torch.float64 else np.float32
    lr_a = learner.make_learning_rate(sys, f)
    lr_c = learner.make_learning_rate(dataclasses.replace(sys, actor_lr=sys.critic_lr), f)
    U, P, M, E = sys.update_batch_size, sys.ppo_epochs, sys.num_minibatches, sys.num_envs
    trajs, advs, tgts, mets = [], [], [], []
    for slot in state["slots"]:
        traj, met, last_val = rollout(spec, ncfg, sys, state["actor_params"], state["critic_params"], slot)
        adv, tgt = learner.gae(traj["done"], traj["value"], traj["reward"], last_val, slot["dones"], sys.gamma, sys.gae_lambda)
        trajs.append(traj); advs.append(adv); tgts.append(tgt); mets.append(met)
    if record is not None:
        record.update(traj=trajs, adv=advs, targets=tgts)
    infos = []
    keys = [slot["key"] for slot in state["slots"]]
    for _ in range(P):
        mbs = []
        for u in range(U):
            keys[u], perm = epoch_perm(keys[u], E)
            mbs.append(make_minibatches(trajs[u], advs[u], tgts[u], perm, M))
        for m in range(M):
            asum, csum, slot_infos = None, None, []
            for u in range(U):
                ga, gc, info = minibatch_losses_and_grads(state["actor_params"], state["critic_params"], mbs[u][m], ncfg, sys, dtype)
                asum = ga if asum is None else {k: asum[k] + ga[k] for k in ga}
                csum = gc if csum is None else {k: csum[k] + gc[k] for k in gc}
                slot_infos.append(info)
            learner.clip_adam_step(state["actor_params"], {k: (v / f(U)).astype(f) for k, v in asum.items()}, state["actor_opt"], lr_a,
                                   sys.max_grad_norm, f=f)
            learner.clip_adam_step(state["critic_params"], {k: (v / f(U)).astype(f) for k, v in csum.items()}, state["critic_opt"], lr_c,
                                   sys.max_grad_norm, f=f)
            infos.append({k: float(np.mean([i[k] for i in slot_infos])) for k in slot_infos[0]})
    for u, slot in enumerate(state["slots"]):
        slot["key"] = keys[u]
    return mets, infos
