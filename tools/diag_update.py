"""Diagnostic: one update step (E=8,U=2,T=16,P=2,M=2) CUDA vs oracle.
Prints the six losses per (epoch, minibatch) and, per parameter tensor, |cuda - oracle| / |update|."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch

from magpo_b200.learner import MagpoLearner
from oracle import learner as olr
from test_gpu_learner import build


def run(chunk: int):
    spec, ncfg, osys, state, lrn = build(torch.device("cuda:0"), E=8, U=2, T=16, P=2, M=2, chunk=chunk)
    g0 = {k: v.copy() for k, v in state["guider_params"].items()}
    a0 = {k: v.copy() for k, v in state["actor_params"].items()}
    rec = {}
    _, infos = olr.update_step(state, spec, ncfg, osys, record=rec)
    _, losses = lrn.update_step()
    torch.cuda.synchronize()
    li = MagpoLearner.loss_info(losses.cpu(), lrn.sys)
    print(f"==== chunk={chunk}")
    k = 0
    for p in range(2):
        for m in range(2):
            row = []
            for name in ("value_loss", "actor_loss", "guider_loss", "kl_loss", "entropy"):
                row.append(f"{name}={float(li[name][p, m]):+.6f}/{infos[k][name]:+.6f}")
            print(p, m, " ".join(row))
            k += 1
    gp, ap = lrn.get_params()
    for new, ref, old in ((gp, state["guider_params"], g0), (ap, state["actor_params"], a0)):
        for name, r in ref.items():
            got = new[name].cpu().numpy()
            step = np.abs(r - old[name]).max()
            err = np.abs(got - r).max()
            if step > 0 and err / step > 0.01:
                print(f"   {name:60s} err/step={err / step:.4f} err={err:.3e} step={step:.3e}")


if __name__ == "__main__":
    for chunk in (0, 3):
        run(chunk)
