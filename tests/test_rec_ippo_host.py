"""CPU tests of rec_ippo: config composition and the configurations it refuses, the critic's parameter table, and the oracle's losses
(float64 finite differences, and term by term against rec_sable's loss, which the library evaluates for both systems)."""
import dataclasses

import numpy as np
import pytest
import torch

from magpo_b200 import rec_ippo as ri
from magpo_b200.config import compose
from magpo_b200.learner import NetworkConfig, param_table
from oracle import ippo as oippo
from oracle import learner as olr
from oracle import nets as onets


def test_config_composition_and_overrides():
    c = compose("default/rec_ippo", ["env=lbf", "arch.num_envs=64", "system.rollout_length=32", "system.critic_lr=1e-3",
                                     "system.decay_learning_rates=True", "system.num_updates=8"])
    assert c.env.env_name == "LevelBasedForaging" and c.network.hidden_state_dim == 128
    s = ri._system_config(c)
    assert (s.num_envs, s.rollout_length, s.ppo_epochs, s.num_minibatches, s.update_batch_size) == (64, 32, 4, 2, 2)
    assert s.actor_lr == 2.5e-4 and s.critic_lr == 1e-3 and s.decay_learning_rates and s.num_updates == 8
    assert (s.clip_eps, s.ent_coef, s.vf_coef, s.max_grad_norm, s.gamma, s.gae_lambda) == (0.2, 0.01, 0.5, 0.5, 0.99, 0.95)
    d = compose("default/rec_ippo", [])
    assert d.env.env_name == "RobotWarehouse" and d.system.recurrent_chunk_size is None and ri._system_config(d).critic_lr == 2.5e-4
    ri._check_network(d)
    ri._system_config(compose("default/rec_ippo", ["system.recurrent_chunk_size=128"]))  # = rollout_length: the whole rollout


@pytest.mark.parametrize("override", ["system.recurrent_chunk_size=16", "network.hidden_state_dim=64",
                                      "network.critic_network.pre_torso.layer_sizes=[64,64]",
                                      "network.actor_network.post_torso.use_layer_norm=True",
                                      "network.critic_network.post_torso.activation=tanh", "system.add_agent_id=False"])
def test_unbuilt_configurations_raise(override):
    c = compose("default/rec_ippo", [override])
    with pytest.raises(NotImplementedError):
        ri._system_config(c)
        ri._check_network(c)


def test_critic_parameter_table():
    for A, d, a in ((2, 14, 6), (4, 75, 5), (3, 4, 10)):
        net = NetworkConfig(A, d, a, 100)
        actor, n_a = param_table(net, 1)
        critic, n_c = param_table(net, 2)
        assert n_c == param_table(NetworkConfig(A, d, 1, 100), 1)[1]  # the actor's layout at a = 1
        names = [t[0] for t in critic]
        assert names[-2:] == [f"{oippo.CRITIC_HEAD}/kernel", f"{oippo.CRITIC_HEAD}/bias"]
        assert names[:-2] == [t[0] for t in actor][:-2]
        shapes = {t[0]: (t[2], t[3]) for t in critic}
        assert shapes[f"{oippo.CRITIC_HEAD}/kernel"] == (128, 1) and shapes[f"{oippo.CRITIC_HEAD}/bias"] == (1, 0)
        assert shapes["pre_torso/Dense_0/kernel"] == (d, 128) and shapes["ScannedRNN_0/GRUCell_0/hn/kernel"] == (128, 128)
        assert all(off % 4 == 0 for _, off, *_ in critic)  # 16-byte aligned
        end = max(off + (d0 * ld if d1 else d0) for _, off, d0, d1, ld in critic)
        assert end <= n_c
        p = oippo.init_critic_params(onets.NetCfg(A, d, a))
        assert set(p) == set(names) and all(p[n].shape == ((s[0],) if s[1] == 0 else s) for n, s in shapes.items())


def _case(dtype=torch.float64, seed=0):
    rng = np.random.default_rng(seed)
    T, N, A, d, a = 5, 3, 2, 6, 4
    ncfg = onets.NetCfg(A, d, a)
    sysc = oippo.SysCfg(rollout_length=T, ent_coef=0.05)
    ap, cp = onets.init_actor_params(ncfg, 1), oippo.init_critic_params(ncfg, 2)
    mask = rng.random((T, N, A, a)) < 0.7
    mask[..., 0] = True
    action = np.stack([[[rng.choice(np.flatnonzero(mask[t, n, i])) for i in range(A)] for n in range(N)] for t in range(T)]).astype(np.int32)
    done = np.repeat((rng.random((T, N)) < 0.2)[..., None], A, axis=2)
    mb = dict(obs=rng.standard_normal((T, N, A, d)).astype(np.float32), action_mask=mask, action=action, done=done,
              log_prob=(rng.standard_normal((T, N, A)) * 0.3 - 1.3).astype(np.float32), adv=rng.standard_normal((T, N, A)).astype(np.float32),
              value=(rng.standard_normal((T, N, A)) * 0.1).astype(np.float32), targets=rng.standard_normal((T, N, A)).astype(np.float32),
              policy_h0=(rng.standard_normal((N, A, 128)) * 0.3).astype(np.float32),
              critic_h0=(rng.standard_normal((N, A, 128)) * 0.3).astype(np.float32))
    return ncfg, sysc, ap, cp, mb


def _loss64(ap, cp, mb, ncfg, sysc, which):
    t = {k: torch.tensor(v, dtype=torch.float64) if v.dtype.kind == "f" else torch.tensor(v) for k, v in mb.items()}
    apt, cpt = onets.to_torch(ap, torch.float64), onets.to_torch(cp, torch.float64)
    _, logits = onets.actor_apply(apt, ncfg, t["policy_h0"], t["obs"], t["done"], t["action_mask"])
    _, value = oippo.critic_apply(cpt, ncfg, t["critic_h0"], t["obs"], t["done"])
    ta, tc, _ = oippo.losses(logits, value, t, sysc)
    return float(ta if which == "actor" else tc)


def test_oracle_loss_gradients_match_float64_finite_differences():
    ncfg, sysc, ap, cp, mb = _case()
    ga, gc, _ = oippo.minibatch_losses_and_grads(ap, cp, mb, ncfg, sysc, torch.float64)
    rng = np.random.default_rng(5)
    ap64 = {k: v.astype(np.float64) for k, v in ap.items()}
    cp64 = {k: v.astype(np.float64) for k, v in cp.items()}
    checked = 0
    for which, params, grads in (("actor", ap64, ga), ("critic", cp64, gc)):
        for name in params:
            for _ in range(2):
                idx = tuple(rng.integers(0, s) for s in params[name].shape)
                eps = 1e-6
                plus = {k: v.copy() for k, v in params.items()}
                minus = {k: v.copy() for k, v in params.items()}
                plus[name][idx] += eps
                minus[name][idx] -= eps
                args = (plus, cp64) if which == "actor" else (ap64, plus)
                margs = (minus, cp64) if which == "actor" else (ap64, minus)
                fd = (_loss64(*args, mb, ncfg, sysc, which) - _loss64(*margs, mb, ncfg, sysc, which)) / (2 * eps)
                g = grads[name][idx]
                assert abs(fd - g) <= 1e-6 + 1e-4 * abs(fd), (which, name, idx, fd, g)
                checked += 1
    assert checked == 2 * (len(ap) + len(cp))


def test_oracle_losses_equal_rec_sable_loss_term_by_term():
    """The library evaluates rec_ippo's loss with rec_sable's path through the MAGPO loss kernel: on the same (logits, values) the two
    restatements agree in every term, and rec_ippo's total is rec_sable's."""
    ncfg, sysc, ap, cp, mb = _case(seed=3)
    t = {k: torch.tensor(v, dtype=torch.float64) if v.dtype.kind == "f" else torch.tensor(v) for k, v in mb.items()}
    _, logits = onets.actor_apply(onets.to_torch(ap, torch.float64), ncfg, t["policy_h0"], t["obs"], t["done"], t["action_mask"])
    _, value = oippo.critic_apply(onets.to_torch(cp, torch.float64), ncfg, t["critic_h0"], t["obs"], t["done"])
    ta, tc, (al, ent, vl) = oippo.losses(logits, value, t, sysc)
    logp_all = onets.log_softmax(logits)
    pr = torch.exp(logp_all)
    g_ent = -(torch.where(pr == 0, torch.zeros_like(pr), logp_all) * pr).sum(-1)
    total, (s_al, s_ent, s_vl) = olr.sable_ppo_loss(logits, value, g_ent, t, dataclasses.replace(sysc))
    for ours, theirs in ((al, s_al), (ent, s_ent), (vl, s_vl), (ta + tc, total)):
        assert abs(float(ours) - float(theirs)) <= 1e-12 * max(1.0, abs(float(theirs))), (float(ours), float(theirs))
