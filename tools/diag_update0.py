#!/usr/bin/env python
"""First-update deviation at a BASELINE config (tools/tolerance_control.py): per optimiser step of update 0, the learner's gradient
against the fp32 oracle's and its parameters against the oracle's optimiser. Usage (GPU box): python tools/diag_update0.py [coordsum|lbf]"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from gpu_util import baseline_case  # noqa: E402
from magpo_b200.learner import param_views  # noqa: E402
from oracle import learner as olr  # noqa: E402

env = sys.argv[1] if len(sys.argv) > 1 else "coordsum"
torch.set_num_threads(os.cpu_count() or 1)
dev = torch.device("cuda:0")
spec, ncfg, osys, state, _ = baseline_case(env, dev)
rec32 = {}
olr.update_step(state, spec, ncfg, osys, record=rec32)

# every optimiser step of update 0: gradient of step k (CUDA vs the fp32 oracle's), then the parameters after the step against the
# oracle's optimiser replayed on the oracle's recorded gradients from the same initial parameters
print("=== per optimiser step of update 0")
spec, ncfg, osys, state0, lrn = baseline_case(env, dev)
o_params = {k: v.copy() for k, v in state0["actor_params"].items()}
o_opt = olr.init_opt(o_params)
lrn.rollout(); lrn.gae()
k = 0
for p_ in range(osys.ppo_epochs):
    lrn.epoch_indices(p_ == 0)
    for m_ in range(osys.num_minibatches):
        lrn.minibatch_grads(m_)
        torch.cuda.synchronize()
        g = lrn.grads.clone()
        av = param_views(g[lrn.n_g:lrn.n_g + lrn.n_a], lrn.a_table)
        ref = rec32["grads"][k][1]
        rows = sorted(((float(np.abs(av[n].cpu().numpy() - r).max()) / max(float(np.abs(r).max()), 1e-30), float(np.abs(r).max()), n)
                       for n, r in ref.items()), reverse=True)
        lrn.apply_grads()
        torch.cuda.synchronize()
        olr.clip_adam_step(o_params, ref, o_opt, osys.actor_lr, osys.max_grad_norm)
        _, ap = lrn.get_params()
        prow = sorted(((float(np.abs(ap[n].cpu().numpy() - r).max()) / osys.actor_lr, n) for n, r in o_params.items()), reverse=True)
        print(f"  step {k}: grad dev (rel to max|g|, max|g|, tensor): " + "; ".join("%.1e %.1e %s" % r for r in rows[:3]))
        print(f"          param dev in units of lr: " + "; ".join("%.3f %s" % r for r in prow[:3]))
        n = prow[0][1]
        d = np.abs(ap[n].cpu().numpy() - o_params[n])
        idx = np.unravel_index(int(d.argmax()), d.shape)
        print(f"          worst element {n}{list(idx)}: p_cuda {float(ap[n].cpu().numpy()[idx]):.9g} p_oracle {float(o_params[n][idx]):.9g} "
              f"g_cuda {float(av[n].cpu().numpy()[idx]):.6g} g_oracle {float(ref[n][idx]):.6g} count {int(lrn.a_count.item())}")
        k += 1
