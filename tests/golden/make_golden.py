"""Generates tests/golden/*.json|npz from the CPU oracle.

The reference ships no golden vectors and cannot be imported here (JAX is absent, SURVEY.md F3/F5), so these
fixtures pin the ORACLE's current outputs (regression anchors shared by the CPU and the GPU tests); the
published Random123 / jax.random KATs are asserted separately in tests/test_oracle.py.
Run from the repo root:  python tests/golden/make_golden.py

    python tests/golden/make_golden.py --reference <liyheng/MAGPO checkout>
rewrites only reference_configs.json: the reference's env and scenario YAML fields that the in-tree config tree
(magpo_b200/configs/env) and the oracle's scenario tables must carry.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import coordsum as ocs  # noqa: E402
from oracle import lbf as olbf  # noqa: E402
from oracle import prng  # noqa: E402
from oracle import rware as orw  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    key = prng.prng_key(42)
    gold = dict(seed=42, split4=prng.split(key, 4).tolist(), bits8=prng.random_bits(key, (8,)).tolist(),
                randint8_0_30=prng.randint(key, (8,), 0, 30).tolist(), perm16=prng.permutation(key, 16).tolist())
    with open(os.path.join(HERE, "prng.json"), "w") as f:
        json.dump(gold, f, indent=1)
    # CoordSum trace: 4 envs, 105 steps (through one auto-reset) with a fixed action stream
    spec = ocs.CoordSumSpec(**ocs.SCENARIOS["3x10-30-v0"])
    keys = prng.split(prng.prng_key(5), 4)
    st, ts = ocs.reset(spec, keys)
    rng = np.random.default_rng(0)
    acts, rewards, views, steps = [], [], [ts["observation"]["agents_view"].copy()], []
    for _ in range(105):
        a = rng.integers(0, 10, (4, 3)).astype(np.int32)
        st, ts = ocs.step(spec, st, a)
        acts.append(a); rewards.append(ts["reward"].copy()); views.append(ts["observation"]["agents_view"].copy())
        steps.append(ts["step_type"].copy())
    np.savez_compressed(os.path.join(HERE, "coordsum_trace.npz"), keys=keys, actions=np.stack(acts), rewards=np.stack(rewards),
                        agents_view=np.stack(views), step_type=np.stack(steps), final_target=st["env_state"]["target"],
                        final_key=st["env_state"]["key"], episode_return=st["episode_return"])
    # LBF / RWARE traces: 6 envs, a fixed stream of (mostly legal) actions through several auto-resets
    for name, mod, spec, n_steps in (("lbf", olbf, olbf.LbfSpec(**olbf.SCENARIOS["2s-8x8-2p-2f-coop"]), 230),
                                     ("rware", orw, orw.RwareSpec(**dict(orw.SCENARIOS["tiny-4ag"], time_limit=70)), 160)):
        np.savez_compressed(os.path.join(HERE, f"{name}_trace.npz"), **env_trace(mod, spec, n_steps))
    # one whole `_update_step` of the oracle on the two in-tree env families: sampled actions, rewards, losses, parameter sums
    with open(os.path.join(HERE, "update_step.json"), "w") as f:
        json.dump({name: update_fixture(spec, **kw) for name, spec, kw in UPDATE_CASES()}, f, indent=1)


def UPDATE_CASES():
    return [("coordsum_3x10-30", ocs.CoordSumSpec(**ocs.SCENARIOS["3x10-30-v0"]), dict(E=4, U=1, T=8, P=2, M=2, seed=42)),
            ("lbf_2s-8x8-2p-2f-coop", olbf.LbfSpec(**olbf.SCENARIOS["2s-8x8-2p-2f-coop"]), dict(E=4, U=2, T=8, P=2, M=2, seed=42))]


def update_fixture(spec, E, U, T, P, M, seed):
    from oracle import learner as olr, nets as onets

    ncfg = onets.NetCfg(spec.num_agents, spec.obs_dim, spec.action_dim)
    osys = olr.SysCfg(num_envs=E, update_batch_size=U, rollout_length=T, ppo_epochs=P, num_minibatches=M)
    state = olr.learner_setup(spec, ncfg, osys, seed=seed)
    rec = {}
    _, infos = olr.update_step(state, spec, ncfg, osys, record=rec)
    names = ("value_loss", "actor_loss", "guider_loss", "kl_loss", "entropy", "total_loss")
    return dict(cfg=dict(E=E, U=U, T=T, P=P, M=M, seed=seed),
                actions=[rec["traj"][u]["action"].tolist() for u in range(U)],
                reward_sum=[float(rec["traj"][u]["reward"].sum()) for u in range(U)],
                losses=[{n: i[n] for n in names} for i in infos],
                guider_param_abs_sum={k: float(np.abs(v).sum(dtype=np.float64)) for k, v in state["guider_params"].items()},
                actor_param_abs_sum={k: float(np.abs(v).sum(dtype=np.float64)) for k, v in state["actor_params"].items()},
                final_key=state["slots"][0]["key"].tolist())


def env_trace(mod, spec, n_steps, n_envs=6, seed=9):
    keys = prng.split(prng.prng_key(seed), n_envs)
    st, ts = mod.reset(spec, keys)
    rng = np.random.default_rng(1)
    a_dim = spec.action_dim
    acts, rewards, views, masks, steps, rets = [], [], [ts["observation"]["agents_view"].copy()], [ts["observation"]["action_mask"].copy()], [], []
    for _ in range(n_steps):
        m = ts["observation"]["action_mask"]
        a = rng.integers(0, a_dim, (n_envs, spec.num_agents)).astype(np.int32)
        legal = np.take_along_axis(m, a[..., None].astype(np.int64), -1)[..., 0]
        a = np.where(legal | (rng.random(a.shape) < 0.1), a, 0).astype(np.int32)
        if a_dim == 6:  # LBF: load whenever possible, most of the time
            a = np.where(m[..., 5] & (rng.random(a.shape) < 0.6), 5, a).astype(np.int32)
        st, ts = mod.step(spec, st, a)
        acts.append(a); rewards.append(ts["reward"].copy()); views.append(ts["observation"]["agents_view"].copy())
        masks.append(ts["observation"]["action_mask"].copy()); steps.append(ts["step_type"].copy())
        rets.append(ts["extras"]["episode_metrics"]["episode_return"].copy())
    return dict(keys=keys, actions=np.stack(acts), rewards=np.stack(rewards), agents_view=np.stack(views).astype(np.float32),
                action_mask=np.stack(masks), step_type=np.stack(steps), episode_return=np.stack(rets),
                final_key=st["env_state"]["key"])


def reference_configs(env_dir):
    """{"env": {family: env_name / kwargs / defaults}, "scenario": {file stem: name / task_name / task_config}} of a
    mava/configs/env tree."""
    import glob

    import yaml

    env = {}
    for fam in ("coordsum", "lbf", "rware"):
        with open(os.path.join(env_dir, f"{fam}.yaml")) as f:
            y = yaml.safe_load(f)
        env[fam] = {k: y[k] for k in ("env_name", "kwargs", "defaults")}
    scenario = {}
    for path in sorted(glob.glob(os.path.join(env_dir, "scenario", "*.yaml"))):
        with open(path) as f:
            y = yaml.safe_load(f)
        scenario[os.path.basename(path)[:-len(".yaml")]] = {k: y[k] for k in ("name", "task_name", "task_config")}
    return {"env": env, "scenario": scenario}


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--reference":
        with open(os.path.join(HERE, "reference_configs.json"), "w") as f:
            json.dump(reference_configs(os.path.join(sys.argv[2], "mava", "configs", "env")), f, indent=1)
            f.write("\n")
    else:
        main()
