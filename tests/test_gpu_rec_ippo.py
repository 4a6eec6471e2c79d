"""-m gpu: rec_ippo (recurrent IPPO, GRU actor + GRU critic) on the B200 kernels against oracle/ippo.py: the rollout, the sampler at the
bench size, full update steps, the critic's GRU at the bench's minibatch shape against float64 autograd, and the system entry."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

from magpo_b200 import _lib as L
from magpo_b200 import init as minit
from magpo_b200 import rec_ippo as ri
from magpo_b200.config import compose
from magpo_b200.learner import CoordSumVec, LbfVec, RwareVec
from oracle import coordsum as ocs
from oracle import ippo as oippo
from oracle import lbf as olbf
from oracle import nets as onets
from oracle import prng as oprng
from oracle import rware as orw

from gpu_util import as_u32, dt, rel_err, sync

pytestmark = pytest.mark.gpu


def _env(name):
    if name == "coordsum":
        kw = ocs.SCENARIOS["3x10-30-v0"]
        return ocs.CoordSumSpec(**kw), CoordSumVec(**kw)
    if name == "lbf":
        kw = olbf.SCENARIOS["2s-8x8-2p-2f-coop"]
        return olbf.LbfSpec(**kw), LbfVec(**kw)
    kw = orw.SCENARIOS["tiny-4ag"]
    return orw.RwareSpec(**kw), RwareVec(**kw)


def _case(name, dev, E, U, T, P=2, M=2, seed=7, **kw):
    spec, vec = _env(name)
    ncfg = onets.NetCfg(spec.num_agents, spec.obs_dim, spec.action_dim)
    osys = oippo.SysCfg(num_envs=E, update_batch_size=U, rollout_length=T, ppo_epochs=P, num_minibatches=M, critic_lr=1e-3, **kw)
    state = oippo.learner_setup(spec, ncfg, osys, seed=seed)
    lrn = ri.IppoLearner(vec, ri.IppoSystemConfig(num_envs=E, update_batch_size=U, rollout_length=T, ppo_epochs=P, num_minibatches=M,
                                                  critic_lr=1e-3, **kw), device=dev)
    lrn.set_params(state["actor_params"], state["critic_params"])
    ks = oprng.split(oprng.prng_key(seed), 4)
    allk = oprng.split(ks[0], U * E + 1)
    lrn.reset(allk[1:], oprng.split(allk[0])[1])
    return spec, ncfg, osys, state, lrn


@pytest.mark.parametrize("env_name", ["coordsum", "lbf", "rware"])
def test_rollout_matches_oracle(dev, env_name):
    E, U, T = 6, 2, 16
    spec, ncfg, osys, state, lrn = _case(env_name, dev, E, U, T)
    lrn.rollout()
    sync()
    for u, slot in enumerate(state["slots"]):
        traj, _, last_val = oippo.rollout(spec, ncfg, osys, state["actor_params"], state["critic_params"], slot)
        sl = slice(u * E, (u + 1) * E)
        g = lambda k: lrn.traj[k].cpu().numpy()[:, sl]
        assert (g("action") == traj["action"]).all(), (env_name, u, "actions")
        assert (g("reward") == traj["reward"]).all(), (env_name, u, "rewards")
        assert (g("done")[:T] == traj["done"][..., 0]).all() and (g("done")[T] == slot["dones"][:, 0]).all(), (env_name, u, "dones")
        assert rel_err(g("log_prob"), traj["log_prob"]) < 1e-4
        assert rel_err(g("value"), traj["value"]) < 1e-4
        assert rel_err(lrn.traj["last_value"].cpu().numpy()[sl], last_val) < 1e-4
        assert rel_err(lrn.policy_h.cpu().numpy()[sl], slot["hstates"]["policy"]) < 1e-4
        assert rel_err(lrn.critic_h.cpu().numpy()[sl], slot["hstates"]["critic"]) < 1e-4
        assert (as_u32(lrn.key) == slot["key"]).all()  # T splits, the bootstrap takes none


@pytest.mark.parametrize("env_name", ["lbf", "rware"])
def test_sampler_at_bench_size(dev, env_name):
    """B = 8192 rows per agent with E = 4096: the gumbel rows wrap once. Every action is the float64 argmax of gumbel + log-softmax of
    the actor's logits, and log_prob is that log-softmax; the logits are recomputed by magpo_actor_forward (a separate forward), so a
    row whose two best scores are within 1e-4 may go either way."""
    E, U, T = 4096, 2, 1
    spec, vec = _env(env_name)
    lrn = ri.IppoLearner(vec, ri.IppoSystemConfig(num_envs=E, update_batch_size=U, rollout_length=T, ppo_epochs=1, num_minibatches=1),
                         device=dev)
    ncfg = onets.NetCfg(spec.num_agents, spec.obs_dim, spec.action_dim)
    ap = onets.init_actor_params(ncfg, 3)
    ap["action_head/Dense_0/kernel"] = ap["action_head/Dense_0/kernel"] * 100  # spread the logits so the argmax is not just the noise's
    lrn.set_params(ap, oippo.init_critic_params(ncfg, 4))
    key = oprng.prng_key(11)
    lrn.reset(oprng.split(key, U * E), oprng.split(key)[1])
    h0 = torch.randn(U * E, spec.num_agents, 128, device=dev) * 0.5
    lrn.policy_h.copy_(h0)
    lrn.rollout()
    B, A, a = U * E, spec.num_agents, spec.action_dim
    net = ri.rm.ActorNetwork(lrn)
    obs = lrn.traj["agents_view"][:1]
    _, logits = net.apply(lrn.actor, h0, (ri.rm.Observation(obs, lrn.traj["action_mask"][:1], lrn.traj["step_count"][:1]),
                                          lrn.traj["done"][:1]))
    lg = logits[0].double().cpu().numpy()
    norm = lg - np.log(np.exp(lg - lg.max(-1, keepdims=True)).sum(-1, keepdims=True)) - lg.max(-1, keepdims=True)
    policy_key = oprng.split(oprng.split(key)[1])[1]
    g = oprng.gumbel(policy_key, (E, A, a)).astype(np.float64)
    sc = np.concatenate([g, g]) + norm
    ref = sc.argmax(-1)
    top2 = np.sort(sc, -1)[..., -2:]
    got = lrn.traj["action"][0].cpu().numpy()
    bad = (got != ref) & (top2[..., 1] - top2[..., 0] > 1e-4)
    assert not bad.any(), f"{int(bad.sum())} of {bad.size} rows"
    assert (got != ref).mean() < 1e-3
    lp = np.take_along_axis(norm, got[..., None], -1)[..., 0]
    assert np.abs(lrn.traj["log_prob"][0].cpu().numpy() - lp).max() < 1e-3 * max(1.0, np.abs(lp).max())


@pytest.mark.parametrize("env_name,decay", [("lbf", False), ("coordsum", False), ("lbf", True)])
def test_update_matches_oracle(dev, env_name, decay):
    E, U, T, P, M = 6, 2, 20, 2, 2
    kw = dict(decay_learning_rates=True, num_updates=3) if decay else {}
    spec, ncfg, osys, state, lrn = _case(env_name, dev, E, U, T, P, M, **kw)
    for it in range(2):
        rec = {}
        _, infos = oippo.update_step(state, spec, ncfg, osys, record=rec)
        _, losses = lrn.update_step()
        sync()
        for u in range(U):
            sl = slice(u * E, (u + 1) * E)
            assert (lrn.traj["action"].cpu().numpy()[:, sl] == rec["traj"][u]["action"]).all(), (it, "actions")
        li = ri.IppoLearner.loss_info(losses.cpu(), lrn.sys)
        k = 0
        for p in range(P):
            for m in range(M):
                for name in ("total_loss", "value_loss", "actor_loss", "entropy"):
                    ref, got = infos[k][name], float(li[name][p, m])
                    assert abs(got - ref) <= 1e-4 * max(1.0, abs(ref)), (it, p, m, name, got, ref)
                k += 1
        worst = {}
        for flat, table, ref_p, opt, mu, nu, cnt in (
                (lrn.actor, lrn.a_table, state["actor_params"], state["actor_opt"], lrn.a_mu, lrn.a_nu, lrn.a_count),
                (lrn.critic, lrn.c_table, state["critic_params"], state["critic_opt"], lrn.c_mu, lrn.c_nu, lrn.c_count)):
            assert int(cnt) == opt["count"]
            for buf, refs, what in ((flat, ref_p, "param"), (mu, opt["mu"], "mu"), (nu, opt["nu"], "nu")):
                views = ri.param_views(buf, table)
                for name, r in refs.items():
                    e = float(np.abs(views[name].cpu().numpy() - r).max() / max(np.abs(r).max(), 1e-3 if what == "param" else 1e-30))
                    if e > worst.get(what, (0.0, ""))[0]:
                        worst[what] = (e, name)
        print(f"  {env_name} decay={decay} update {it}: worst per-tensor max-norm rel. error {worst}")
        for what, (e, name) in worst.items():
            assert e <= 1e-4, (it, what, name, e)
        assert (as_u32(lrn.key) == state["slots"][0]["key"]).all()


def test_critic_at_bench_minibatch_shape(dev):
    """The LBF bench size's minibatch: N = U*E/M = 4096 envs x A = 2 agents (Rs = 8192 GRU rows, the 128-row persistent tile) over
    T = 128, forward and backward through magpo_ippo_minibatch_grads, against float64 autograd of the same losses. Bound as in
    test_gpu_production_paths.py: max(fixed, 4 x the float32 reference's own error), fixed 5e-4 — every weight gradient is a reduction over
    R = 1,048,576 token rows, and the critic's value-error terms of both signs cancel in it (measured on a B200: at most 2.5e-4, in the
    critic's GRU kernels; the actor's gradients sit within 2.5x of the float32 reference's own error)."""
    T, N, A, d, a = 128, 4096, 2, 14, 6
    lib = L.lib()
    assert lib.magpo_debug_gru_rows_per_tile(C.c_int64(N * A)) == 128
    spec, vec = _env("lbf")
    sysc = ri.IppoSystemConfig(num_envs=N, update_batch_size=1, rollout_length=T, ppo_epochs=1, num_minibatches=1)
    lrn = ri.IppoLearner(vec, sysc, device=dev)
    ncfg = onets.NetCfg(A, d, a)
    ap, cp = onets.init_actor_params(ncfg, 5), oippo.init_critic_params(ncfg, 6)
    lrn.set_params(ap, cp)
    rng = np.random.default_rng(0)
    mask = rng.random((T, N, A, a)) < 0.8
    mask[..., 0] = True
    action = np.where(mask, rng.random((T, N, A, a)), -1).argmax(-1).astype(np.int32)
    done = rng.random((T, N)) < 0.02
    mb = dict(obs=rng.standard_normal((T, N, A, d)).astype(np.float32), action_mask=mask, action=action,
              done=np.repeat(done[..., None], A, 2), log_prob=(rng.standard_normal((T, N, A)) * 0.2 - 1.7).astype(np.float32),
              adv=rng.standard_normal((T, N, A)).astype(np.float32), value=(rng.standard_normal((T, N, A)) * 0.1).astype(np.float32),
              targets=rng.standard_normal((T, N, A)).astype(np.float32), policy_h0=(rng.standard_normal((N, A, 128)) * 0.3).astype(np.float32),
              critic_h0=(rng.standard_normal((N, A, 128)) * 0.3).astype(np.float32))
    m = lrn.mb
    m["agents_view"].copy_(dt(mb["obs"], dev)); m["action_mask"].copy_(dt(mask, dev, torch.uint8)); m["action"].copy_(dt(action, dev))
    m["done"].copy_(dt(done, dev, torch.uint8)); m["log_prob"].copy_(dt(mb["log_prob"], dev)); m["advantages"].copy_(dt(mb["adv"], dev))
    m["value"].copy_(dt(mb["value"], dev)); m["targets"].copy_(dt(mb["targets"], dev)); m["policy_h0"].copy_(dt(mb["policy_h0"], dev))
    lrn.mb_critic_h0.copy_(dt(mb["critic_h0"], dev))
    lrn.env_slot.zero_()
    adv64 = mb["adv"].astype(np.float64)
    lrn.stats.copy_(torch.tensor([[adv64.mean(), adv64.std()]], dtype=torch.float32, device=dev))
    lrn.grads.zero_()
    ws = C.c_size_t(lrn.ws_bytes)
    L.call("magpo_ippo_minibatch_grads", lrn.ctx, L.stream_ptr(), C.byref(lrn.c_net), C.byref(lrn.c_sys), L.ptr(lrn.actor), L.ptr(lrn.critic),
           lrn._mb_struct(N), L.ptr(lrn.mb_critic_h0), L.ptr(lrn.env_slot[:N]), L.ptr(lrn.stats), C.c_float(1.0 / (N * T * A)),
           L.ptr(lrn.grads), 0, L.ptr(lrn.workspace), C.byref(ws))
    sync()
    got_a = ri.param_views(lrn.grads[:lrn.n_a], lrn.a_table)
    got_c = ri.param_views(lrn.grads[lrn.n_a:lrn.n_a + lrn.n_c], lrn.c_table)

    def ref(dtype):
        t = {k: torch.tensor(v, dtype=dtype, device=dev) if v.dtype.kind == "f" else torch.tensor(v, device=dev) for k, v in mb.items()}
        apt = {k: torch.tensor(v, dtype=dtype, device=dev, requires_grad=True) for k, v in ap.items()}
        cpt = {k: torch.tensor(v, dtype=dtype, device=dev, requires_grad=True) for k, v in cp.items()}
        _, logits = onets.actor_apply(apt, ncfg, t["policy_h0"], t["obs"], t["done"], t["action_mask"])
        _, value = oippo.critic_apply(cpt, ncfg, t["critic_h0"], t["obs"], t["done"])
        ta, tc, _ = oippo.losses(logits, value, t, sysc)
        ga = torch.autograd.grad(ta, list(apt.values()))
        gc = torch.autograd.grad(tc, list(cpt.values()))
        return {k: g.double().cpu().numpy() for k, g in zip(apt, ga)}, {k: g.double().cpu().numpy() for k, g in zip(cpt, gc)}

    a64, c64 = ref(torch.float64)
    a32, c32 = ref(torch.float32)
    fails = []
    for what, got, r64, r32 in (("critic", got_c, c64, c32), ("actor", got_a, a64, a32)):
        for name in r64:
            e = rel_err(got[name].cpu().numpy(), r64[name])
            bound = max(5e-4, 4 * rel_err(r32[name], r64[name]))
            print(f"  {what} {name:36s} cuda vs f64 {e:.2e}   bound {bound:.1e}")
            if not e <= bound:
                fails.append(f"{what} {name}: {e:.3e} > {bound:.1e}")
    assert not fails, fails


def _setup(dev, extra=()):
    cfg = compose("default/rec_ippo", ["env=lbf", "arch.num_envs=6", "system.rollout_length=10", "system.ppo_epochs=2",
                                       "system.num_updates=4", "arch.num_evaluation=2", *extra])
    cfg.system.num_updates_per_eval = 2
    env = ri.rm.make_env(cfg)
    key, _, ak, ck = minit.split(minit.prng_key(42), 4, dev)
    return cfg, env, ri.learner_setup(env, (key, ak, ck), cfg, device=dev)


def test_system_entry_pytree_adoption_and_graph_replay(dev):
    cfg, env, (learn, actor_network, state) = _setup(dev)
    U, E, A, T, P, M = 2, 6, 2, 10, 2, 2
    assert state._fields == ("params", "opt_states", "key", "env_state", "timestep", "dones", "hstates")
    assert state.params._fields == ("actor_params", "critic_params") and state.hstates._fields == ("policy_hidden_state", "critic_hidden_state")
    assert state.params.critic_params["Dense_0/kernel"].shape == (1, U, 128, 1)
    assert state.params.actor_params["action_head/Dense_0/kernel"].shape == (1, U, 128, 6)
    assert state.hstates.critic_hidden_state.shape == (1, U, E, A, 128) and state.dones.shape == (1, U, E, A) and state.key.shape == (1, U, 2)
    assert ri.rm.adam_of(state.opt_states.critic_opt_state).mu["Dense_0/bias"].shape == (1, U, 1)
    out = learn(state)
    assert set(out.train_metrics) == {"total_loss", "value_loss", "actor_loss", "entropy"}
    for v in out.train_metrics.values():
        assert v.shape == (1, 2, U, P, M) and torch.isfinite(v).all()
    assert out.episode_metrics["episode_return"].shape == (1, 2, U, T, E)
    assert int(ri.rm.adam_of(out.learner_state.opt_states.critic_opt_state).count[0, 0]) == 2 * P * M
    # a deep copy adopted by a second learner reproduces the next update: its rollout bit for bit; the update's cross-CTA fp32
    # reductions (atomics) are order-dependent in the last bits, as for rec_magpo
    snap = copy.deepcopy(out.learner_state)
    _, _, (learn2, an2, _) = _setup(dev)
    o1, o2 = learn(out.learner_state), learn2(snap)
    for k in o1.episode_metrics:
        assert torch.equal(o1.episode_metrics[k], o2.episode_metrics[k]), k
    l1, l2 = actor_network.lrn, an2.lrn
    for k in ("action", "reward", "done", "agents_view"):
        assert torch.equal(l1.traj[k], l2.traj[k]), k
    for k, v in o1.train_metrics.items():
        assert torch.allclose(v, o2.train_metrics[k], rtol=1e-5, atol=1e-6), k
    for a, b in ((l1.actor, l2.actor), (l1.critic, l2.critic)):
        assert float((a - b).abs().max()) <= 2e-6 * max(float(a.abs().max()), 1e-3)
    assert torch.equal(o1.learner_state.key, o2.learner_state.key)
    # the graph-replayed rollout against the eager one, from the same state with the same parameters: identical bits
    _, _, _, _, eager = _case("lbf", dev, 6, 2, 10)
    _, _, _, _, graphed = _case("lbf", dev, 6, 2, 10)
    eager.graph_rollout = False
    for it in range(3):
        eager.rollout()
        graphed.rollout()
        sync()
        for k in ("action", "value", "log_prob", "reward", "done", "agents_view", "last_value", "policy_h0"):
            assert torch.equal(eager.traj[k], graphed.traj[k]), (it, k)
        for k in ("policy_h", "critic_h", "critic_h0", "key"):
            assert torch.equal(getattr(eager, k), getattr(graphed, k)), (it, k)
    assert graphed._rollout_graph is not None and eager._rollout_graph is None


def test_run_experiment_trains_evaluates_and_checkpoints(dev, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    lines = []
    perf = ri.run_experiment(compose("default/rec_ippo", ["env=lbf", "arch.num_envs=8", "system.rollout_length=8", "system.num_updates=2",
                                                          "arch.num_evaluation=2", "arch.num_eval_episodes=4",
                                                          "arch.num_absolute_metric_eval_episodes=8", "logger.checkpointing.save_model=True"]),
                             device=dev, log=lines.append)
    kinds = [ln.split(" - ")[0] for ln in lines]
    assert kinds.count("TRAINER") == 2 and kinds.count("EVALUATOR") == 2 and kinds.count("ABSOLUTE") == 1 and np.isfinite(perf)
    assert list((tmp_path / "checkpoints" / "rec_ippo").rglob("metadata.json")), "no checkpoint written"
    assert len([p for p in (tmp_path / "checkpoints" / "rec_ippo").rglob("*") if p.is_file()]) > 2
