#!/usr/bin/env python
"""bench.py — end-to-end training throughput of the rec_magpo hot path (rollout + GAE + update).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torch.distributed.run)
    python bench.py --impl reference --steps K --warmup W    (CPU oracle port on the host cores)

A step = one `_update_step` (rec_magpo.py:106-499): T env steps of U*E envs through guider + learner + env,
GAE, then P epochs x M minibatches of guider/learner forward+backward, the gradient all-reduce and clip+Adam.
Metric: agent-env-steps/s = n_gpus * U * E * T * A / step time (whole job). Weak scaling: E per GPU is fixed.
Every warm-up and timed step starts from the same seeded learner state, restored before the step and outside its timed span: the
update sums gradients with float atomics, so the parameters of consecutive steps drift apart between runs in the last bits, and the
next rollout's sampling turns that into different trajectories. From one state, two runs compute the same step up to rounding.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs[1]: `rec_magpo.py env=lbf` default scenario (configs/env/lbf.yaml:4 -> 2s-8x8-2p-2f-coop), num_envs=4096 on
# one B200. `--env coordsum` selects the configs[4] sweep point (CoordSum 3x10-30, coordsum/__init__.py:26-35).
WORKLOADS = {
    "lbf": dict(kw=dict(grid_size=8, fov=2, num_agents=2, num_food=2, max_agent_level=2, force_coop=True, time_limit=100),
                label="LevelBasedForaging 2s-8x8-2p-2f-coop (A=2, a=6, d=14; BASELINE configs[1]; dynamics restated from jumanji "
                      "1.1.0, see oracle/lbf.py)"),
    "rware": dict(kw=dict(column_height=8, shelf_rows=1, shelf_columns=3, num_agents=4, sensor_range=1, request_queue_size=4,
                          time_limit=500),
                  label="RobotWarehouse tiny-4ag (A=4, a=5, d=75; BASELINE configs[2], 8192 envs / 8 GPUs = --num-envs 1024 "
                        "--update-batch-size 1 per GPU; dynamics restated from jumanji 1.1.0, see oracle/rware.py)"),
    "rware-small": dict(kw=dict(column_height=8, shelf_rows=2, shelf_columns=3, num_agents=4, sensor_range=1, request_queue_size=4,
                                time_limit=500),
                        label="RobotWarehouse small-4ag (A=4, a=5, d=75; BASELINE configs[3]: run with a long --rollout-length, "
                              "BPTT-heavy update; dynamics restated from jumanji 1.1.0, see oracle/rware.py)"),
    "coordsum": dict(kw=dict(num_agents=3, num_actions=10, time_limit=100, maxval=30),
                     label="CoordSum 3x10-30 (A=3, a=10, d=4; BASELINE configs[4] sweep point)"),
}
METRIC, UNIT = "end_to_end_training_agent_env_steps_per_sec", "agent-steps/s"
PROF_CATS = ["gemm_nn", "gemm_tn", "colsum", "rowops", "retention_fwd", "retention_bwd", "gru_pointwise", "loss", "pack",
             "optim", "env_step", "sample", "gae", "misc", "gemm_rollout", "chain"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--env", default="lbf", choices=sorted(WORKLOADS))
    ap.add_argument("--num-envs", type=int, default=4096, help="arch.num_envs per GPU per update-batch slot")
    ap.add_argument("--update-batch-size", type=int, default=2)
    ap.add_argument("--rollout-length", type=int, default=128)
    ap.add_argument("--chunk-envs", type=int, default=4096)
    ap.add_argument("--ref-num-envs", type=int, default=16, help="envs per slot of the CPU reference arm's bounded sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--quick", action="store_true", help="1 warm-up step, no e2e loop (for runs under ncu only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (episode metrics, loss sums) and the learner state it left "
                         "(parameters, step key, hidden states) as DIR/<name>.npy; arrays above 2^20 elements are replaced by "
                         "the same seeded sample of 2^20 of them on every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def workload_config(args, n_gpus):
    return {"workload": f"rec_magpo {WORKLOADS[args.env]['label']}, num_envs={args.num_envs}/GPU/slot, "
                        f"update_batch_size={args.update_batch_size}, rollout_length={args.rollout_length}, ppo_epochs=4, "
                        f"num_minibatches=2, Sable D=64 + GRU H=128",
            "env": args.env, "num_envs": args.num_envs, "update_batch_size": args.update_batch_size, "rollout_length": args.rollout_length,
            "ppo_epochs": 4, "num_minibatches": 2, "parallelism": f"dp{n_gpus}", "collective": "magpo_comm_allreduce_sum (NCCL via the C ABI), issued inside magpo_minibatch_grads" if n_gpus > 1 else None,
            "l2": "working set per step (>10 GB of activations + 400 MB of Sable state) exceeds the 126 MB L2"}


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
                time.sleep(0.1)
        except Exception as e:  # NVML missing: report that instead of clocks
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def run_reference(args, as_baseline=False):
    """The CPU restatement (oracle/) of the same step on the host cores: the reference itself is JAX-only and
    cannot be installed here (no jax/flax/optax/jumanji wheels, SURVEY.md F3), so kind = "port"."""
    import torch
    from oracle import coordsum as ocs, lbf as olbf, learner as olr, nets as onets, rware as orw

    # physical cores, at most 16: the sample's GEMMs are tiny and more threads only oversubscribe (32 logical threads ran 2.2x slower
    # than 16 in round 1's SCALE run)
    try:
        import psutil
        cores = psutil.cpu_count(logical=False) or os.cpu_count() or 1
    except Exception:
        cores = os.cpu_count() or 1
    cores = max(1, min(cores, 16))
    torch.set_num_threads(cores)
    E = min(args.ref_num_envs, args.num_envs)  # bounded sample of the workload: E of the envs per slot, everything else as configured
    spec = {"lbf": olbf.LbfSpec, "rware": orw.RwareSpec, "rware-small": orw.RwareSpec, "coordsum": ocs.CoordSumSpec}[args.env](**WORKLOADS[args.env]["kw"])
    ncfg = onets.NetCfg(spec.num_agents, spec.obs_dim, spec.action_dim)
    osys = olr.SysCfg(num_envs=E, update_batch_size=args.update_batch_size, rollout_length=args.rollout_length)
    state = olr.learner_setup(spec, ncfg, osys, seed=42)
    steps, warm = (1, 0) if as_baseline else (max(1, args.steps), max(0, min(args.warmup, 1)))  # ~7 s per step: one warm-up step
    for _ in range(warm):
        olr.update_step(state, spec, ncfg, osys)
    t0 = time.perf_counter()
    for _ in range(steps):
        olr.update_step(state, spec, ncfg, osys)
    dt = (time.perf_counter() - t0) / steps
    per_step = osys.update_batch_size * E * osys.rollout_length * spec.num_agents
    val = per_step / dt
    sample = (f"oracle update_step on {E} envs/slot (of the workload's {args.num_envs}) x U={osys.update_batch_size} x T={osys.rollout_length} "
              f"(same nets, P=4, M=2), torch CPU fp32 with {cores} threads, {warm} warm-up + {steps} timed step(s) of {dt:.1f} s")
    return val, dt, cores, sample, E, warm


DUMP_MAX_ELEMENTS = 1 << 20  # 4 MB per array: the 11 arrays of step_outputs stay under 64 MB at any size


def learner_snapshot(lrn):
    """(buffer, saved copy) pairs of everything an update step reads that an earlier step wrote: parameters, Adam state, step key,
    env state and timestep, recurrent states, and the trajectory's last observation slot, which the next rollout carries over into
    slot 0. Taken right after `reset`, that slot gets the reset observation of slot 0."""
    T = lrn.sys.rollout_length
    pairs = [(t, t.clone()) for t in (lrn.guider, lrn.actor, lrn.g_mu, lrn.g_nu, lrn.a_mu, lrn.a_nu, lrn.g_count, lrn.a_count,
                                      lrn.key, lrn.policy_h, *lrn.env_state.values(), *lrn.ts.values(), *lrn.hs.values())]
    pairs += [(lrn.traj[k][T], lrn.traj[k][0].clone()) for k in ("done", "agents_view", "action_mask", "step_count")]
    return pairs


def step_outputs(lrn, metrics, losses):
    """Host copies of what one `update_step` hands its caller: the episode metrics and loss sums it returns, and the learner
    state it leaves (flat parameter buffers, step key, recurrent states). float32, the key as float64 (uint32 values)."""
    import numpy as np
    import torch

    arrays = {**metrics, "losses": losses, "guider_params": lrn.guider, "actor_params": lrn.actor, "policy_hidden_state": lrn.policy_h,
              **{f"sable_hidden_state_{k}": v for k, v in lrn.sable_hidden_state().items()}}
    out = {}
    for name, t in arrays.items():
        if t.numel() > DUMP_MAX_ELEMENTS:  # a flat, seeded sample: the same elements on every run with the same arguments
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMENTS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        out[name] = t.float().cpu().numpy()
    out["key"] = lrn.key.cpu().numpy().view(np.uint32).astype(np.float64)
    return out


def main():
    # stdout carries exactly ONE line (the JSON): everything else that native libraries print there (e.g. NCCL's version
    # banner) is routed to stderr while the benchmark runs
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        line = run()
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    if line is not None:
        print(line, flush=True)


def run():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank != 0:
            return
        val, dt, cores, sample, e_ref, warm = run_reference(args)
        cfg = workload_config(args, args.gpus)
        # the arm runs a bounded sample: say so in the structured fields, not only in the free text
        cfg.update(num_envs=e_ref, workload_num_envs=args.num_envs, same_num_envs=(e_ref == args.num_envs),
                   workload=cfg["workload"].replace(f"num_envs={args.num_envs}/GPU/slot", f"num_envs={e_ref}/slot (CPU sample of the "
                                                    f"GPU arm's {args.num_envs}/GPU/slot)"))
        return json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
                          "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
                          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})

    import numpy as np
    import torch

    from magpo_b200 import _lib as L
    from magpo_b200 import init as minit
    from magpo_b200.learner import CoordSumVec, LbfVec, MagpoLearner, RwareVec, SystemConfig

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    comm = None
    if world > 1:  # one process per GPU; the gradient exchange is the library's own NCCL all-reduce (magpo_comm_*, include/magpo_b200.h)
        from magpo_b200.comm import NcclComm
        comm = NcclComm.from_env(dev)

    env = {"lbf": LbfVec, "rware": RwareVec, "rware-small": RwareVec, "coordsum": CoordSumVec}[args.env](**WORKLOADS[args.env]["kw"])
    sysc = SystemConfig(num_envs=args.num_envs, update_batch_size=args.update_batch_size, rollout_length=args.rollout_length,
                        chunk_envs=args.chunk_envs)
    lrn = MagpoLearner(env, sysc, device=dev, world_size=world)
    if comm is not None:
        comm.attach(lrn)  # magpo_minibatch_grads reduces the gradients itself, the learner's half under the guider's backward
    lrn.set_params(minit.init_guider(env.num_agents, env.obs_dim, env.action_dim, 0), minit.init_actor(env.obs_dim, env.action_dim, 1))
    env_keys, step_key, _ = minit.setup_keys(42, world, sysc.update_batch_size, sysc.num_envs, dev)
    lrn.reset(env_keys[rank], step_key)
    A, T = env.num_agents, sysc.rollout_length
    per_step = world * sysc.update_batch_size * sysc.num_envs * T * A
    lib = L.lib()
    lib.magpo_launch_count.restype = C.c_int64

    def barrier():
        if comm is not None:
            comm.barrier()
        torch.cuda.synchronize()

    snapshot = learner_snapshot(lrn)

    def restore():
        for buf, saved in snapshot:
            buf.copy_(saved)

    def timed(fn, k):
        """(ms per call, what the last call returned); the learner state is restored before each call, outside its span"""
        barrier()
        spans = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        for e0, e1 in spans:
            restore()
            e0.record()
            last = fn()
            e1.record()
        barrier()
        ms = torch.tensor([sum(e0.elapsed_time(e1) for e0, e1 in spans)], device=dev)
        if comm is not None:
            comm.allreduce_max(ms)
        return float(ms.item()) / k, last

    for _ in range(1 if args.quick else max(3, args.warmup)):
        restore()
        lrn.update_step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    n0 = lib.magpo_launch_count()
    ms, last = timed(lrn.update_step, args.steps)
    launches = lib.magpo_launch_count() - n0
    # the steps below overwrite the learner's buffers: copy the last timed step's outputs out first
    dump = step_outputs(lrn, *last) if args.dump_outputs and rank == 0 else None

    # end to end through the public call, host buffers: per step the step key goes up from pinned memory and the
    # metrics the experiment loop consumes (episode metrics [T,B], the [P,M,8] loss sums, the new key) come back.
    B = lrn.B
    key_host = torch.zeros(2, dtype=torch.int32).pin_memory()
    key_host.copy_(lrn.key.cpu())
    out_host = {k: torch.zeros_like(v, device="cpu").pin_memory() for k, v in
                dict(episode_return=lrn.traj["episode_return"], episode_length=lrn.traj["episode_length"],
                     is_terminal_step=lrn.traj["is_terminal_step"]).items()}
    loss_host = torch.zeros(sysc.ppo_epochs, sysc.num_minibatches, 8).pin_memory()
    h2d = key_host.numel() * 4
    d2h = sum(v.numel() * v.element_size() for v in out_host.values()) + loss_host.numel() * 4 + 8

    def e2e_step():
        lrn.key.copy_(key_host, non_blocking=True)
        metrics, losses = lrn.update_step()
        for k, v in out_host.items():
            v.copy_(metrics[k], non_blocking=True)
        loss_host.copy_(losses, non_blocking=True)
        key_host.copy_(lrn.key, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the host reads the metrics every step

    ms_e2e = ms if args.quick else timed(e2e_step, args.steps)[0]
    sampler.stop_flag = True
    sampler.join(timeout=2)

    out = {"metric": METRIC, "value": per_step / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
           "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": workload_config(args, world), "clocks": sampler.summary(),
           "e2e": {"value": per_step / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
           "gpu_launches": int(launches)}

    # phase split of one more step (CUDA events on the launching stream)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    restore()
    torch.cuda.synchronize()
    ev[0].record(); lrn.rollout(); ev[1].record(); lrn.gae(); ev[2].record()
    for p_ in range(sysc.ppo_epochs):
        lrn.epoch_indices(p_ == 0)
        for m_ in range(sysc.num_minibatches):
            lrn.minibatch_grads(m_)
            lrn.apply_grads()
    ev[3].record()
    torch.cuda.synchronize()
    out["phase_ms"] = {"rollout_and_bootstrap": round(ev[0].elapsed_time(ev[1]), 3), "gae": round(ev[1].elapsed_time(ev[2]), 3),
                       "update": round(ev[2].elapsed_time(ev[3]), 3)}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    if not args.no_profile:
        # one more step with per-category CUDA events on the launching stream (bench-only instrumentation)
        lib.magpo_prof_enable(1 if rank == 0 else 0)
        lrn.graph_rollout = False  # the per-category events are recorded by eager launches, not by a graph replay
        lib.magpo_debug_set_overlap(0)  # ... and kernel by kernel: no guider/learner stream overlap inside this step
        restore()
        lrn.update_step()
        torch.cuda.synchronize()
        lib.magpo_debug_set_overlap(1)
        lrn.graph_rollout = True
        lib.magpo_prof_enable(0)
        if rank == 0:
            brk, total = {}, 0.0
            for i, name in enumerate(PROF_CATS):
                msv, work, cnt = C.c_double(), C.c_double(), C.c_int64()
                lib.magpo_prof_read(i, C.byref(msv), C.byref(work), C.byref(cnt))
                brk[name] = {"ms": round(msv.value, 3), "launch_scopes": cnt.value, "work": work.value}
                total += msv.value
            for v in brk.values():
                v["share"] = round(v["ms"] / total, 4) if total else 0.0
            out["breakdown_ms_per_step"] = brk
            # dominant kernel class: the tcgen05 3xTF32 GEMMs Y[M,N] = X[M,K] W (forward and dX; M = token rows, K, N in 64..384).
            # At 16..64 flop/byte (x3 MMAs per product) they sit on the HBM side of the ridge: the roofline is bandwidth.
            g = brk["gemm_nn"]
            gbytes = C.c_double()
            lib.magpo_prof_read_bytes(PROF_CATS.index("gemm_nn"), C.byref(gbytes))
            hb = peaks.get("hbm_gbs", 6650.0)
            gbs = gbytes.value / (g["ms"] * 1e-3) / 1e9 if g["ms"] else 0.0
            tf = g["work"] / (g["ms"] * 1e-3) / 1e12 if g["ms"] else 0.0
            traffic = None
            try:  # DRAM bytes per launch of the same kernel from the committed ncu launch list (profiles/)
                prof = json.load(open(os.path.join(ROOT, "profiles", "r2_lbf_minibatch_launches.json" if args.env == "lbf" else
                                                  "r1_minibatch_launches.json")))
                k = prof["kernels"]["gemm_tc_kernel"]
                traffic = k["dram_bytes"] / k["launches"]
                if args.env == "lbf" and args.num_envs == 4096:
                    # time-weighted whole-update line: the ncu DRAM bytes of ONE minibatch (committed launch list) x the P*M minibatches of
                    # a step over the live, overlapped update time of this run
                    mb_bytes = sum(v["dram_bytes"] for v in prof["kernels"].values())
                    n_mb = sysc.ppo_epochs * sysc.num_minibatches
                    tokens = sysc.rollout_length * (sysc.num_envs * sysc.update_batch_size // sysc.num_minibatches) * lrn.net.n_agents
                    upd_ms = out["phase_ms"]["update"]
                    out["roofline_update"] = {
                        "dram_bytes_per_minibatch": mb_bytes, "launches_per_minibatch": sum(v["launches"] for v in prof["kernels"].values()),
                        "dram_bytes_per_token_and_pass": mb_bytes / tokens, "update_ms": upd_ms,
                        "achieved_GBps": mb_bytes * n_mb / (upd_ms * 1e-3) / 1e9, "frac_of_measured_hbm": mb_bytes * n_mb / (upd_ms * 1e-3) / 1e9 / hb,
                        "source": "profiles/r2_lbf_minibatch_launches.json (ncu dram__bytes_{read,write}.sum of one minibatch) / live update time"}
            except Exception:
                pass
            out["roofline"] = {"kernel": "gemm_tc_kernel (tcgen05.mma kind::tf32 x3, TMA-fed; all forward and dX GEMMs of both networks)",
                               "bound": "hbm", "achieved": gbs, "peak": hb, "unit": "GB/s", "frac": gbs / hb, "traffic": traffic,
                               "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                               "launches": g["launch_scopes"],
                               "algorithmic_bytes_per_launch": gbytes.value / max(1, g["launch_scopes"]),
                               "avg_launch_ms": g["ms"] / max(1, g["launch_scopes"]),
                               "tensor_side": {"achieved_tflops_fp32_equivalent": tf, "mma_per_product": 3,
                                               "peak_bf16_tflops_sustained": peaks.get("bf16_tflops_sustained", 1400.0)},
                               "note": "share of the profiled step: %.2f; bytes = 4*M*(K+N) per launch (+4*M*N when accumulating), "
                                       "summed over the update's GEMM launches (M = T*N*A rows) and divided by their summed CUDA-event time; "
                                       "the rollout's launch-latency-bound small GEMMs (M = U*E*A rows) are the gemm_rollout class" % g["share"]}
            hb = peaks.get("hbm_gbs", 6650.0)
            out["roofline_hbm_kernels"] = {
                k: {"achieved_GBps": round(brk[k]["work"] / (brk[k]["ms"] * 1e-3) / 1e9, 1) if brk[k]["ms"] else None,
                    "frac_of_measured_hbm": round(brk[k]["work"] / (brk[k]["ms"] * 1e-3) / 1e9 / hb, 4) if brk[k]["ms"] else None}
                for k in ("gae", "env_step", "rowops", "loss", "optim", "pack", "sample")}
            cb = C.c_double()
            lib.magpo_prof_read_bytes(PROF_CATS.index("chain"), C.byref(cb))
            if brk["chain"]["ms"]:  # the fused row-chain kernels of the guider's forward: algorithmic bytes = saved activations + inputs
                out["roofline_hbm_kernels"]["chain"] = {"achieved_GBps": round(cb.value / (brk["chain"]["ms"] * 1e-3) / 1e9, 1),
                                                        "frac_of_measured_hbm": round(cb.value / (brk["chain"]["ms"] * 1e-3) / 1e9 / hb, 4)}
            # "sample" is the rollout's fused per-step Sable kernel (encoder + decoder + sampling): its bytes are the retention
            # state stream (160 KiB per env-step at A = 3) plus observations / actions
            out["roofline_hbm_kernels"]["sable_step"] = out["roofline_hbm_kernels"].pop("sample")

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        val, dt, cores, sample, _, _ = run_reference(args, as_baseline=True)
        out["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
    if comm is not None:
        comm.barrier()
        comm.close()
    return json.dumps(out) if rank == 0 else None


if __name__ == "__main__":
    main()
