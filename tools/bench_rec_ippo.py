#!/usr/bin/env python
"""Throughput of rec_ippo's update step (rollout + GAE + P epochs x M minibatches) on one GPU, with the rollout / update split (CUDA
events around each phase, every step from the state the previous one left). Sizes: LBF 2s-8x8-2p-2f-coop with 4096 envs x 2 slots and
T = 128 (rec_magpo's bench workload), and RWARE tiny-4ag with 1024 envs x 1 slot. The GPU's name and power limit are read in the same run.
Usage: python tools/bench_rec_ippo.py [--steps 5] [--warmup 2] [--out profiles/r3_rec_ippo_bench.json]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from magpo_b200 import init as minit  # noqa: E402
from magpo_b200 import rec_ippo as ri  # noqa: E402
from magpo_b200.config import compose  # noqa: E402

CASES = {"lbf_2s-8x8-2p-2f-coop_4096x2_T128": ["env=lbf", "env/scenario=2s-8x8-2p-2f-coop", "arch.num_envs=4096", "system.update_batch_size=2"],
         "rware_tiny-4ag_1024x1_T128": ["env=rware", "env/scenario=tiny-4ag", "arch.num_envs=1024", "system.update_batch_size=1"]}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip() or torch.cuda.get_device_name(0)


def bench(overrides, steps, warmup):
    cfg = compose("default/rec_ippo", overrides + ["system.num_updates=1000", "arch.num_evaluation=1"])
    cfg.system.num_updates_per_eval = 1
    env = ri.rm.make_env(cfg)
    key, _, ak, ck = minit.split(minit.prng_key(42), 4, "cuda:0")
    _, actor_network, _ = ri.learner_setup(env, (key, ak, ck), cfg, device="cuda:0")
    lrn = actor_network.lrn
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    roll, upd = [], []
    for i in range(warmup + steps):
        ev[0].record()
        lrn.rollout()
        ev[1].record()
        lrn.gae()
        for p in range(lrn.sys.ppo_epochs):
            lrn.epoch_indices()
            for m in range(lrn.sys.num_minibatches):
                lrn.minibatch_grads(m)
                lrn.apply_grads()
        ev[2].record()
        torch.cuda.synchronize()
        if i >= warmup:
            roll.append(ev[0].elapsed_time(ev[1]))
            upd.append(ev[1].elapsed_time(ev[2]))
    s = lrn.sys
    agent_steps = s.rollout_length * s.update_batch_size * s.num_envs * lrn.net.n_agents
    step_ms = [r + u for r, u in zip(roll, upd)]
    med = sorted(step_ms)[len(step_ms) // 2]
    return dict(step_ms=step_ms, step_ms_median=med, rollout_ms=roll, update_ms=upd, agent_steps_per_step=agent_steps,
                agent_steps_per_s=agent_steps / (med / 1e3), finite_params=bool(torch.isfinite(lrn.actor).all() and torch.isfinite(lrn.critic).all()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    res = dict(gpu=gpu_info(), steps=args.steps, warmup=args.warmup, cases={})
    for name, ov in CASES.items():
        res["cases"][name] = bench(ov, args.steps, args.warmup)
        c = res["cases"][name]
        print(f"{name}: {c['step_ms_median']:.1f} ms/update step (rollout {sorted(c['rollout_ms'])[len(c['rollout_ms']) // 2]:.1f} ms), "
              f"{c['agent_steps_per_s']:.3g} agent-steps/s", flush=True)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
