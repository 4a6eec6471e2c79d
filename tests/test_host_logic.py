"""CPU tests of the host-side mirror of the reference's system entry (magpo_b200/rec_magpo.py, config.py): config composition,
the env registry, env-key sharding across ranks and the gradient mean over a 2-process gloo group (the N>1 path's host logic)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from magpo_b200 import rec_magpo as rm
from magpo_b200.config import check_total_timesteps, compose
from oracle import coordsum as ocs
from oracle import prng as oprng


def test_config_composition_and_overrides():
    c = compose("default/rec_magpo", ["env/scenario=5x20-80", "arch.num_envs=64", "system.rollout_length=32", "system.num_updates=8",
                                      "arch.num_evaluation=2", "system.total_timesteps=~"])
    assert c.env.scenario.task_name == "5x20-80-v0" and c.arch.num_envs == 64 and c.system.rollout_length == 32
    c = check_total_timesteps(c, 2)
    assert c.system.total_timesteps == 2 * 32 * c.system.update_batch_size * 64 * 8
    sysc = rm._system_config(c)
    assert (sysc.num_envs, sysc.rollout_length, sysc.ppo_epochs, sysc.num_minibatches) == (64, 32, 4, 2)
    assert sysc.clip_gpo == 1.5 and sysc.alpha == 1.0 and abs(sysc.actor_lr - 2.5e-4) < 1e-12


def test_env_registry_matches_reference_registrations():
    assert rm.COORDSUM_REGISTRY == ocs.SCENARIOS
    for name in ("3x10-30", "3x30-50", "5x20-80", "8x15-100"):
        c = compose("default/rec_magpo", [f"env/scenario={name}"])
        env = rm.make_env(c)
        kw = ocs.SCENARIOS[c.env.scenario.task_name]
        assert (env.num_agents, env.num_actions, env.time_limit, env.maxval) == (kw["num_agents"], kw["num_actions"], 100, kw["maxval"])
        assert env.obs_dim == env.num_agents + 1 and env.action_dim == env.num_actions


def test_env_key_sharding_is_the_reference_reshape():
    U, E, world = 2, 5, 4
    allk = oprng.split(oprng.prng_key(7), world * U * E + 1)[1:]
    parts = [rm.shard_env_keys(allk, world, r, U, E) for r in range(world)]
    assert (np.concatenate(parts) == allk).all()
    # (device, slot, env) order: env e of slot u on device r is global index (r*U + u)*E + e
    assert (parts[3].reshape(U, E, 2)[1, 2] == allk[(3 * U + 1) * E + 2]).all()


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        U, E = 2, 3
        # every rank derives the same key chain (replicated step key) and takes its own block of reset keys
        allk = oprng.split(oprng.prng_key(42), world * U * E + 1)
        step_key = oprng.split(allk[0])[1]
        mine = rm.shard_env_keys(allk[1:], world, rank, U, E)
        gathered = [torch.zeros(U * E, 2, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(gathered, torch.as_tensor(mine.astype(np.int64)))
        keys = [torch.zeros(2, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(keys, torch.as_tensor(step_key.astype(np.int64)))
        # per-rank gradients: the device mean is one sum all-reduce + a 1/Nd scale
        g = torch.arange(10, dtype=torch.float32) * (rank + 1)
        m = rm.mean_over_devices(g.clone(), world)
        if rank == 0:
            out.put(dict(all=torch.cat(gathered).numpy().astype(np.uint32), ref=allk[1:], keys=[k.numpy() for k in keys],
                         mean=m.numpy(), expect=(torch.arange(10, dtype=torch.float32) * (1 + 2) / 2).numpy()))
    finally:
        dist.destroy_process_group()


def test_two_process_gloo_sharding_and_gradient_mean():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = out.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert (res["all"] == res["ref"]).all()          # the ranks' blocks tile the global key array in order
    assert (res["keys"][0] == res["keys"][1]).all()  # identical step key on every device
    assert np.allclose(res["mean"], res["expect"])


def test_logger_describes_and_writes_marl_eval_json(tmp_path):
    """MavaLogger.log semantics of mava/utils/logger.py:126-150 and the marl-eval JSON layout of JsonLogger (:300-346)."""
    import json

    import numpy as np

    from magpo_b200.config import compose
    from magpo_b200.logger import LogEvent, MavaLogger, describe

    assert describe(np.array([1.0, 3.0])) == {"mean": 2.0, "std": 1.0, "min": 1.0, "max": 3.0} and describe(np.float32(2)) == 2.0
    cfg = compose("default/rec_magpo", ["env=lbf", "logger.use_json=True"])
    cfg.logger.base_exp_path = str(tmp_path)
    lines = []
    lg = MavaLogger(cfg, console_sink=lines.append)
    lg.log({"episode_return": np.array([0.5, 1.0]), "is_terminal_step": np.array([1, 1]), "steps_per_second": 10.0}, 100, 0, LogEvent.ACT)
    lg.log({"total_loss": np.ones((1, 2, 2, 4, 2)), "entropy": np.full((1, 2, 2, 4, 2), 0.5)}, 100, 0, LogEvent.TRAIN)
    lg.log({"episode_return": np.array([0.5, 1.0]), "steps_per_second": 9.0}, 100, 0, LogEvent.EVAL)
    lg.log({"episode_return": np.array([1.0, 1.0])}, 200, 1, LogEvent.ABSOLUTE)
    assert lines[0].startswith("ACTOR - ") and "Episode return mean: 0.750" in lines[0] and "terminal" not in lines[0]
    assert lines[1] == "TRAINER - Entropy: 0.500 | Total loss: 1.000"
    files = list(tmp_path.rglob("metrics.json"))
    run = json.load(open(files[0]))["LevelBasedForaging"]["2s-8x8-2p-2f-coop"]["rec_magpo"]["seed_42"]
    assert run["step_0"] == {"step_count": 100, "mean_episode_return": [0.75], "steps_per_second": [9.0]}
    assert run["absolute_metrics"] == {"mean_episode_return": [1.0]}


def test_checkpointer_keeps_the_best_and_restores(tmp_path, monkeypatch):
    """Checkpointer surface of mava/utils/checkpointing.py:34-215: best_fn = episode_return (max), max_to_keep, keep_period."""
    from collections import namedtuple

    import numpy as np

    from magpo_b200.checkpointing import Checkpointer, unreplicate_n_dims

    monkeypatch.chdir(tmp_path)
    P = namedtuple("Params", "guider_params actor_params")
    H = namedtuple("HiddenStates", "sable_hidden_state policy_hidden_state")
    S = namedtuple("State", "params key hstates")
    st = S(P({"enc/w": np.ones((1, 2, 3, 4))}, {"head/b": np.zeros((1, 2, 5))}), np.zeros((1, 2, 2), np.uint32),
           H({"encoder": np.ones((1, 2, 7))}, np.full((1, 2, 6), 2.0)))
    un = unreplicate_n_dims(st)
    assert un.params.guider_params["enc/w"].shape == (3, 4) and un.key.shape == (2,)
    ck = Checkpointer("rec_magpo", metadata={"system": {"seed": 42}}, checkpoint_uid="u", max_to_keep=1, keep_period=40)
    assert ck.save(10, un, 0.5) and ck.save(20, un, 0.2) and ck.save(30, un, 0.9) and ck.save(40, un, 0.1)
    assert sorted(ck._index) == ["30", "40"]  # the best, plus the one protected by keep_period
    ck2 = Checkpointer("rec_magpo", checkpoint_uid="u")
    params, hs = ck2.restore_params(un.params, timestep=30, restore_hstates=True, THiddenState=H)
    assert params.guider_params["enc/w"].shape == (3, 4) and hs.policy_hidden_state.shape == (6,) and hs.sable_hidden_state["encoder"].shape == (7,)
    assert ck2.get_cfg()["checkpointer_version"] == 1.0 and ck2.get_cfg()["system"]["seed"] == 42


def test_env_scenario_files_match_the_reference_configs():
    """Every LBF / RWARE / CoordSum scenario file shipped here carries the reference's `task_config` (mava/configs/env/scenario/*.yaml);
    the reference's values are stored in tests/golden/reference_configs.json (make_golden.py --reference)."""
    import glob
    import json
    import os

    import yaml

    tests = os.path.dirname(os.path.abspath(__file__))
    with open(os.path.join(tests, "golden", "reference_configs.json")) as f:
        gold = json.load(f)
    here = os.path.join(os.path.dirname(tests), "magpo_b200", "configs", "env", "scenario")
    checked = 0
    for path in glob.glob(os.path.join(here, "*.yaml")):
        mine = yaml.safe_load(open(path))
        ref = gold["scenario"][os.path.basename(path)[:-len(".yaml")]]
        assert mine["task_name"] == ref["task_name"] and mine["name"] == ref["name"], path
        for k, v in ref["task_config"].items():
            assert mine["task_config"][k] == v, (path, k)
        checked += 1
    assert checked >= 20
    for env in ("lbf", "rware", "coordsum"):
        mine = yaml.safe_load(open(os.path.join(os.path.dirname(here), f"{env}.yaml")))
        ref = gold["env"][env]
        assert mine["env_name"] == ref["env_name"] and mine["kwargs"] == ref["kwargs"] and mine["defaults"] == ref["defaults"], env


def test_make_env_builds_every_family_from_config():
    from magpo_b200 import rec_magpo as rm
    from magpo_b200.config import compose
    from magpo_b200.evaluator import get_num_eval_envs

    cases = {("lbf", "15x15-4p-5f"): (4, 31, 6, 100), ("lbf", "2s-8x8-2p-2f-coop"): (2, 14, 6, 100), ("rware", "tiny-4ag"): (4, 75, 5, 500),
             ("rware", "small-4ag"): (4, 75, 5, 500), ("rware", "medium-6ag"): (6, 77, 5, 500), ("coordsum", "5x20-80"): (5, 6, 20, 100)}
    for (env, sc), (A, d, a, tl) in cases.items():
        e = rm.make_env(compose("default/rec_magpo", [f"env={env}", f"env/scenario={sc}"]))
        assert (e.num_agents, e.obs_dim, e.action_dim, e.time_limit) == (A, d, a, tl), (env, sc)
    cfg = compose("default/rec_magpo", ["arch.num_envs=16"])
    assert get_num_eval_envs(cfg, absolute_metric=False) == 16  # 32 episodes > 16 envs -> num_envs (evaluator.py:66-80)
    assert get_num_eval_envs(compose("default/rec_magpo", ["arch.num_envs=64"]), absolute_metric=False) == 32
    assert get_num_eval_envs(compose("default/rec_magpo", ["arch.num_envs=64"]), absolute_metric=False, n_devices=4) == 8


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """No CPU fallback: without the built shared library the first call into the product raises."""
    import pytest

    from magpo_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "libmagpo_b200.so"))
    with pytest.raises(_lib.MagpoError, match="no CPU fallback"):
        _lib.lib()
    with pytest.raises(_lib.MagpoError):
        _lib.call("magpo_gae")


def test_ffi_shim_declares_a_handler_for_every_entry_point_and_compiles():
    """ffi/magpo_ffi.cc: one XLA-FFI handler per compute entry point of include/magpo_b200.h (host-only queries excepted), and the
    file's own code — every magpo_* call's arguments — compiles (syntax-only, against the compile-only stand-in for jaxlib's
    xla/ffi/api/ffi.h under tests/mock_xla_ffi; the real header is not installable here)."""
    import re
    import shutil
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "magpo_b200.h")).read()
    shim = open(os.path.join(root, "ffi", "magpo_ffi.cc")).read()
    declared = set(re.findall(r"^(?:int|int32_t|int64_t|size_t|const char\*)\s+(magpo_\w+)\(", header, flags=re.M))
    host_only = {"magpo_version", "magpo_last_cuda_error", "magpo_context_create", "magpo_context_destroy", "magpo_context_set_comm",
                 "magpo_param_count", "magpo_param_num_tensors", "magpo_param_tensor", "magpo_rware_num_shelves",
                 "magpo_rollout_workspace_bytes", "magpo_update_workspace_bytes", "magpo_comm_available", "magpo_comm_version",
                 "magpo_comm_unique_id", "magpo_comm_init", "magpo_comm_destroy", "magpo_comm_allreduce_max", "magpo_prng_fold_in_host",
                 "magpo_clip_adam"}  # magpo_clip_adam is magpo_clip_adam_sched with decay_period 0: one handler serves both
    called = set(re.findall(r"\b(magpo_\w+)\(", shim))
    missing = sorted(n for n in declared - host_only if n not in called)
    assert not missing, f"no FFI handler calls {missing}"
    handlers = re.findall(r"XLA_FFI_DEFINE_HANDLER_SYMBOL\((magpo_ffi_\w+),", shim)
    assert len(handlers) == len(set(handlers)) >= len(declared - host_only)
    gxx = shutil.which("g++")
    assert gxx, "g++ is part of the image"
    cmd = [gxx, "-std=c++17", "-fsyntax-only", "-Wall", "-Wno-comment", "-I", os.path.join(root, "tests", "mock_xla_ffi"), "-I",
           os.path.join(root, "include"), "-I", "/usr/local/cuda/include", os.path.join(root, "ffi", "magpo_ffi.cc")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    # without the FFI header on the include path the translation unit is empty and still compiles
    res = subprocess.run([gxx, "-std=c++17", "-fsyntax-only", "-I", os.path.join(root, "include"), os.path.join(root, "ffi", "magpo_ffi.cc")],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
