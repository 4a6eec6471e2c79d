"""The update's minibatch gradient pass (magpo_minibatch_grads, csrc/update.cu) against the float64 oracle at the minibatch each
bench.py workload differentiates in one pass (T = 128, net (64, 1, 1), chunk_envs >= the minibatch):

    lbf       A = 2, d = 14, a = 6    N = 2 x 2048   R = 1 048 576   (the bench default, BASELINE configs[1])
    coordsum  A = 3, d = 4,  a = 10   N = 2 x 2048   R = 1 572 864   (--env coordsum)
    rware     A = 4, d = 75, a = 5    N = 1 x 512    R =   262 144   (--env rware --num-envs 1024 --update-batch-size 1)

At these sizes the persistent chain kernels run ~55 tiles per CTA, the row kernels run their grid-stride loops, and the tensor-core GEMMs
split M into slabs; the smaller parity tests reach none of that. The networks are independent per env and every loss is a mean over rows,
so the oracle runs in env chunks with each slot's advantage statistics held fixed, and its gradients are the weighted sum of the chunks'.
Every chunk compares every saved forward tensor and the per-row loss gradients on every row, then the parameter gradients and the loss
sums are compared once. The float32 oracle run of the same chunk is the yardstick (DESIGN.md section 5): at 1 M random tokens some hit
the ill-conditioned GroupNorm case that test_gpu_networks.py documents, and any float32 implementation is far from float64 there.

The workspace starts as NaN, the gradient buffer as a known non-zero vector followed by a sentinel; the LBF case also runs once from a
dirty workspace and once on the layer-by-layer path, which must differ in its bits (the fused chain kernels did run)."""
import ctypes as C
import math
import sys
from contextlib import contextmanager
from dataclasses import dataclass

import numpy as np
import pytest
import torch

from magpo_b200 import _lib as L
from magpo_b200.learner import CoordSumVec, LbfVec, RwareVec, SystemConfig, param_views
from oracle import learner as olr
from oracle import nets as onets

import test_gpu_networks as tgn
from gpu_util import dt, from_time_major, rel_err, sync

T = 128
NUM_SMS = 148  # B200: the persistent chain kernels launch min(tiles, 148) CTAs
CHUNK = 256  # envs per oracle chunk (the float64 oracle needs ~6 GB of host memory for 256 LBF envs)


@dataclass(frozen=True)
class Case:
    env: str
    A: int
    d: int
    a: int
    num_envs: int  # bench.py --num-envs
    U: int  # bench.py --update-batch-size
    M: int = 2  # SystemConfig.num_minibatches

    @property
    def Ns(self):  # envs per slot in one minibatch
        return self.num_envs // self.M

    @property
    def N(self):
        return self.U * self.Ns

    @property
    def R(self):
        return T * self.N * self.A

    @property
    def tiles(self):  # 128-row tiles of one chain-kernel launch
        return -(-self.R // 128)

    def chunks(self):
        """env ranges of the oracle chunks: each inside one slot"""
        return [(u * self.Ns + c, u * self.Ns + min(c + CHUNK, self.Ns)) for u in range(self.U) for c in range(0, self.Ns, CHUNK)]


CASES = {"lbf": Case("lbf", 2, 14, 6, 4096, 2), "coordsum": Case("coordsum", 3, 4, 10, 4096, 2), "rware": Case("rware", 4, 75, 5, 1024, 1)}
VECS = {"lbf": LbfVec, "coordsum": CoordSumVec, "rware": RwareVec}

DONE_KINDS = ("p=0.15", "p=0.01", "never", "every step", "t=0 only")


def done_pattern(rng, N):
    """done [N, T]: env n gets DONE_KINDS[n % 5]"""
    kind = np.arange(N) % len(DONE_KINDS)
    r = rng.random((N, T))
    done = np.where(kind[:, None] == 0, r < 0.15, r < 0.01)
    done[kind >= 2] = False
    done[kind == 3] = True
    done[kind == 4, 0] = True
    return done


def mask_pattern(rng, mask, action):
    """~10 % of the rows get exactly one legal action (the taken one), ~10 % all legal; the rest keep make_case's random mask"""
    kind = rng.integers(0, 10, mask.shape[:2])
    mask = mask.copy()
    mask[kind == 0] = False
    mask[kind == 1] = True
    n, c = np.nonzero(kind == 0)
    mask[n, c, action[n, c]] = True
    return mask


def make_bench_case(case: Case, seed):
    A, a, N = case.A, case.a, case.N
    mb = tgn.make_case(seed, case.U, case.Ns, T, A, case.d, a)
    rng = np.random.default_rng(seed + 100)
    mb["done"] = np.repeat(done_pattern(rng, N), A, 1)
    mb["action_mask"] = mask_pattern(rng, mb["action_mask"], mb["action"])
    adv = rng.standard_normal((N, T * A))
    for u in range(1, case.U):  # slot u: (u + 1) N(0, 1) + 3 u — a slot / env_slot mix-up in the loss kernel shows
        adv[u * case.Ns:(u + 1) * case.Ns] = (u + 1) * adv[u * case.Ns:(u + 1) * case.Ns] + 3 * u
    mb["adv"] = adv.astype(np.float32)
    # old log-probs around a uniform policy's, spread so that both PPO clip branches are taken on many rows
    n_legal = mb["action_mask"].sum(-1)
    mb["log_prob"] = (-np.log(n_legal) + 0.5 * rng.standard_normal((N, T * A))).astype(np.float32)
    return mb


def slot_stats(case, mb):
    """[U, 2] mean and population std of each slot's advantages (what magpo_adv_stats computes), as float32"""
    adv = mb["adv"].astype(np.float64).reshape(case.U, -1)
    return np.stack([adv.mean(1), adv.std(1)], 1).astype(np.float32)


# ----------------------------------------------------------------------------- saved buffers and their oracle counterparts
ENC, DEC = "encoder/encoder_block_0", "decoder/decoder_block_0"


def _qkvg(rec, pre):
    h = f"{pre}/retention_heads_0"
    return np.concatenate([rec[f"{h}/q"], rec[f"{h}/k"], rec[f"{h}/v"], rec[f"{pre}/g"]], -1)


# name -> (width, oracle record -> [n, T*A, width])
FORWARD = {
    "on": (None, lambda r: r["enc/on"]),
    "z0": (64, lambda r: r["enc/z0"]),
    "xin": (64, lambda r: r["enc/xin"]),
    "kqv": (64, lambda r: r[f"{ENC}/retn/key"]),
    "qkvg": (256, lambda r: _qkvg(r, f"{ENC}/retn")),
    "ret": (64, lambda r: r[f"{ENC}/retn/ret"]),
    "gated": (64, lambda r: r[f"{ENC}/retn/gated"]),
    "o": (64, lambda r: r[f"{ENC}/retn/out"]),
    "x1": (64, lambda r: r["enc/x1"]),
    "gl": (128, lambda r: np.concatenate([r[f"{ENC}/ffn/gate"], r[f"{ENC}/ffn/linear"]], -1)),
    "hmid": (64, lambda r: r[f"{ENC}/ffn/hmid"]),
    "f": (64, lambda r: r[f"{ENC}/ffn/out"]),
    "x": (64, lambda r: r["enc/x"]),
    "xpe": (64, lambda r: r[f"{DEC}/retn2/query"]),
    "zh": (64, lambda r: r["encoder/head/zh"]),
    "xD": (64, lambda r: r["dec/xD"]),
    "xpeD": (64, lambda r: r[f"{DEC}/retn1/key"]),
    "qkvg1": (256, lambda r: _qkvg(r, f"{DEC}/retn1")),
    "ret1": (64, lambda r: r[f"{DEC}/retn1/ret"]),
    "gated1": (64, lambda r: r[f"{DEC}/retn1/gated"]),
    "o1": (64, lambda r: r[f"{DEC}/retn1/out"]),
    "rpe": (64, lambda r: r[f"{DEC}/retn2/key"]),
    "qkvg2": (256, lambda r: _qkvg(r, f"{DEC}/retn2")),
    "ret2": (64, lambda r: r[f"{DEC}/retn2/ret"]),
    "gated2": (64, lambda r: r[f"{DEC}/retn2/gated"]),
    "o2": (64, lambda r: r[f"{DEC}/retn2/out"]),
    "y": (64, lambda r: r["dec/y"]),
    "glD": (128, lambda r: np.concatenate([r[f"{DEC}/ffn/gate"], r[f"{DEC}/ffn/linear"]], -1)),
    "hmidD": (64, lambda r: r[f"{DEC}/ffn/hmid"]),
    "fD": (64, lambda r: r[f"{DEC}/ffn/out"]),
    "xd": (64, lambda r: r["dec/xd"]),
    "zhD": (64, lambda r: r["decoder/head/zh"]),
}
LOSS_GRADS = ("dlg", "dll", "dvalue")
# The decoder's cross-retention GroupNorm (retn2) amplifies the rounding of ret2 on its worst-conditioned tokens, and the CUDA path's
# ret2 (3xTF32, chunkwise) rounds differently from the float32 oracle's. Measured on a B200 (1000 W), LBF, over all 1 M rows, as a
# fraction of the 4x bound: gated2 1.36, o2 1.25, y 1.30, glD 1.08, hmidD 1.34, fD 1.21, xd 1.16, zhD 1.39, lg 1.04, with ret2 itself
# within 7e-6 of float64. Those forward tensors are held to 8x the float32 yardstick. So are the gradients of the parameters upstream of
# that GroupNorm's backward (RWARE, as a fraction of the 2x bound: retn2 w_k 2.34, w_q 2.09, decoder/ln 2.13, action_encoder 1.92,
# ln1 1.92, retn1 w_v 1.43, w_g 1.23, group_norm/bias 1.58); every other gradient keeps 2x.
CROSS_GN = ("gated2", "o2", "y", "glD", "hmidD", "fD", "xd", "zhD", "lg")
CROSS_GN_GRADS = ("decoder/action_encoder/", "decoder/ln/", f"{DEC}/ln1/", f"{DEC}/retn1/", f"{DEC}/retn2/retention_heads_0/")
LOSS_SLOTS = ((1, "guider_loss"), (2, "entropy"), (3, "value_loss"), (4, "kl_loss"), (6, "actor_loss"), (7, "actor_kl"))


def forward_names(case):
    """the chained encoder front (d <= 16) does not write `on`; the un-chained one (RWARE, d = 75) does"""
    return [k for k in FORWARD if k != "on" or case.d > 16]


def widths(case):
    w = {k: (case.d if k == "on" else FORWARD[k][0]) for k in forward_names(case)}
    w.update(value=1, lg=case.a, ll=case.a, dlg=case.a, dll=case.a, dvalue=1)
    return w


def device_buffers(ws, net, case):
    """name -> [T, N, A, width] (width 1: [T, N, A]) views of the workspace"""
    lib = L.lib()
    lib.magpo_debug_buffer_offset.restype = C.c_int64
    out = {}
    for name, w in widths(case).items():
        off = lib.magpo_debug_buffer_offset(C.byref(net.c_struct()), T, case.N, name.encode())
        assert off >= 0 and off % 4 == 0, name
        shape = (T, case.N, case.A) + ((w,) if w > 1 else ())
        out[name] = ws[off // 4:off // 4 + int(np.prod(shape))].view(shape)
    return out


def locate(case, n0, idx_env_c, what):
    """`what` at oracle-layout index (env within the chunk, c = t * A + agent): env, t, agent, its 128-row tile and chain-kernel CTA"""
    nl, c = idx_env_c
    env, t, i = n0 + nl, c // case.A, c % case.A
    row = (t * case.N + env) * case.A + i
    tile = row // 128
    return f"{what}: env {env}, t {t}, agent {i}, row {row}, tile {tile}, chain CTA {tile % min(case.tiles, NUM_SMS)}"


def worst_at(got, ref):
    d = np.abs(np.asarray(got, np.float64) - ref)
    return np.unravel_index(int(np.argmax(d)), d.shape)


@contextmanager
def fixed_adv_stats(mean, std):
    """olr._norm_adv with a slot's whole-minibatch statistics instead of the chunk's own"""
    keep = olr._norm_adv
    olr._norm_adv = lambda adv: (adv - float(mean)) / (float(std) + 1e-8)
    try:
        yield
    finally:
        olr._norm_adv = keep


def loss_row_grads(lg, ll, value, part, mask, sysc, weight, dtype):
    """per-row dL/d(guider logits), dL/d(learner logits), dL/d(value) of the chunk's losses, taken at the CUDA path's own logits and
    values (so that only the loss is compared), scaled by the chunk's share of the minibatch's rows"""
    F32_MIN = torch.tensor(onets.F32_MIN, dtype=dtype)
    m = torch.tensor(mask)
    g = torch.where(m, torch.tensor(lg, dtype=dtype), F32_MIN).requires_grad_(True)
    a = torch.where(m, torch.tensor(ll, dtype=dtype), F32_MIN).requires_grad_(True)
    v = torch.tensor(value, dtype=dtype, requires_grad=True)
    mb = {k: torch.tensor(part[k], dtype=dtype if part[k].dtype.kind == "f" else None) for k in ("action", "log_prob", "adv", "value", "targets")}
    logp = onets.log_softmax(g)
    pr = torch.exp(logp)
    ent = -(torch.where(pr == 0, torch.zeros_like(pr), logp) * pr).sum(-1)
    tot_g, _ = olr.guider_loss(g, v, ent, a, mb, sysc)
    tot_a, _ = olr.actor_loss(a, g, mb, sysc)
    dg, dv = torch.autograd.grad(tot_g, (g, v))
    (da,) = torch.autograd.grad(tot_a, (a,))
    return {"dlg": weight * dg.numpy(), "dll": weight * da.numpy(), "dvalue": weight * dv.numpy()}


def branch_edge_rows(lg, ll, value, part, mask, mean, std, sysc, eps=1e-5):
    """rows whose loss sits within eps of a clip / max / min switch (float64 at the CUDA path's inputs): the gradient jumps there, so the
    float32 kernel and a float64 reference may legitimately take different branches. Also: how often each branch is taken."""
    f = np.float64
    lgm, llm = np.where(mask, lg.astype(f), -np.inf), np.where(mask, ll.astype(f), -np.inf)
    lse_g = np.log(np.exp(lgm - lgm.max(-1, keepdims=True)).sum(-1)) + lgm.max(-1)
    lse_l = np.log(np.exp(llm - llm.max(-1, keepdims=True)).sum(-1)) + llm.max(-1)
    act = part["action"].astype(np.int64)[..., None]
    lgp = np.take_along_axis(lgm, act, -1)[..., 0] - lse_g
    llp = np.take_along_axis(llm, act, -1)[..., 0] - lse_l
    value, vold, tgt = value.astype(f), part["value"].astype(f), part["targets"].astype(f)
    lold, advn = part["log_prob"].astype(f), (part["adv"].astype(f) - float(mean)) / (float(std) + 1e-8)
    lo, hi, ce = math.log(1 / sysc.clip_gpo), math.log(sysc.clip_gpo), sysc.clip_eps
    diff, ratio = lgp - llp, np.exp(lgp - lold)
    cr = np.exp(np.clip(diff, lo, hi) + llp - lold)
    ra = np.exp(llp - lold)
    l1, l2 = ratio * advn, np.clip(cr, 1 - ce, 1 + ce) * advn
    dv = value - vold
    e1, e2 = value - tgt, vold + np.clip(dv, -ce, ce) - tgt
    margins = [np.abs(diff - lo), np.abs(diff - hi), np.abs(cr - (1 - ce)), np.abs(cr - (1 + ce)), np.abs(ra - (1 - ce)),
               np.abs(ra - (1 + ce)), np.abs(dv - ce), np.abs(dv + ce), np.where(np.abs(dv) < ce, np.inf, np.abs(np.abs(e1) - np.abs(e2))),
               np.where(np.abs(l1 - l2) == 0, np.inf, np.abs(l1 - l2) / (np.abs(advn) + 1e-30))]
    edge = np.min(margins, axis=0) < eps
    taken = dict(double_clip_mask=int(((diff < lo) | (diff > hi)).sum()), ratio_clipped_low=int((ra < 1 - ce).sum()),
                 ratio_clipped_high=int((ra > 1 + ce).sum()), guider_clipped_branch=int((l2 < l1).sum()), value_clipped=int((np.abs(dv) > ce).sum()))
    return edge, taken


# ----------------------------------------------------------------------------- the GPU side
class Pass:
    """one network setup + workspace; `run` is one magpo_minibatch_grads call"""

    def __init__(self, case, dev):
        self.case, self.dev = case, dev
        self.cfg, self.net, self.gp, self.ap, (self.gt, self.ng, self.gflat), (self.at, self.na, self.aflat) = tgn.setup_nets(
            case.A, case.d, case.a, dev)
        lib = L.lib()
        lib.magpo_update_workspace_bytes.restype = C.c_size_t
        self.nbytes = int(lib.magpo_update_workspace_bytes(C.byref(self.net.c_struct()), T, case.N))
        print(f"{case.env}: R = {case.R}, magpo_update_workspace_bytes = {self.nbytes} ({self.nbytes / 2**30:.1f} GiB)")
        self.ws = torch.full((-(-self.nbytes // 4),), float("nan"), device=dev)  # the whole workspace starts as NaN
        self.bufs = device_buffers(self.ws, self.net, case)
        rng = np.random.default_rng(11)
        n = self.ng + self.na + 8
        self.g0 = dt(rng.integers(-8, 9, n) * 2.0 ** -6, dev, torch.float32)  # far above the gradients: an overwrite cannot hide
        self.sentinel = dt(rng.integers(-2**31, 2**31, 1024, dtype=np.int64).astype(np.int32), dev)  # 4 KiB of arbitrary bits, NaNs included
        self.csys = SystemConfig(num_envs=case.num_envs, update_batch_size=case.U, rollout_length=T, num_minibatches=case.M).c_struct()

    def run(self, mb, stats, g0=None):
        """the gradient buffer starts as `g0` (default zeros); returns it after the call"""
        case = self.case
        mbs, keep = tgn.device_minibatch(mb, T, case.A, self.dev)
        env_slot = dt(np.repeat(np.arange(case.U), case.Ns).astype(np.int32), self.dev)
        st = dt(stats, self.dev)
        n = self.ng + self.na + 8
        grads = torch.empty(n + 1024, device=self.dev)
        grads[:n] = 0.0 if g0 is None else g0
        grads[n:].view(torch.int32).copy_(self.sentinel)
        L.call("magpo_minibatch_grads", L.context(), L.stream_ptr(), C.byref(self.net.c_struct()), C.byref(self.csys), L.ptr(self.gflat),
               L.ptr(self.aflat), mbs, L.ptr(env_slot), L.ptr(st), C.c_float(1.0 / case.R), L.ptr(grads), 0, L.ptr(self.ws),
               C.c_size_t(self.nbytes))
        sync()
        del keep
        assert torch.equal(grads[n:].view(torch.int32), self.sentinel), "the 4 KiB past the gradient buffer changed"
        return grads[:n]

    def snapshot(self):
        return {k: v.clone() for k, v in self.bufs.items()}


def bits_equal(a, b):
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def run_oracle_chunks(case, p, mb, stats, report):
    """every chunk: forward buffers and per-row loss gradients against float64 (float32 yardstick); returns the chunk-weighted float64
    and float32 parameter gradients and loss values"""
    A, a = case.A, case.a
    sysc = olr.SysCfg(num_envs=CHUNK, update_batch_size=1, rollout_length=T, num_minibatches=1)
    names = forward_names(case)
    ref = {torch.float64: {}, torch.float32: {}}
    loss_ref = {torch.float64: {}, torch.float32: {}}
    edges = 0
    for n0, n1 in case.chunks():
        u = n0 // case.Ns
        weight = (n1 - n0) / case.N
        part = {k: (tuple(h[n0:n1] for h in v) if k == "prev_hstates" else v[n0:n1]) for k, v in mb.items()}
        rec, aux = {}, {}
        with fixed_adv_stats(*stats[u]):
            for dtype in (torch.float64, torch.float32):
                onets.RECORD = rec[dtype] = {}
                try:
                    gg, ga, info, aux[dtype] = olr.minibatch_losses_and_grads(p.gp, p.ap, part, p.cfg, sysc, dtype=dtype)
                finally:
                    onets.RECORD = None
                gg.update(ga)
                for k, g in gg.items():
                    ref[dtype][k] = ref[dtype].get(k, 0.0) + weight * g.astype(np.float64)
                for _, k in LOSS_SLOTS:
                    loss_ref[dtype][k] = loss_ref[dtype].get(k, 0.0) + weight * info[k]
        got = {k: from_time_major(v[:, n0:n1].cpu().numpy()) for k, v in p.bufs.items()}
        legal = part["action_mask"]
        fails = []

        def check(name, g, r64, r32, floor=1e-4):
            e, e32 = rel_err(g, r64), rel_err(r32, r64)
            bound = max(floor, (8 if name in CROSS_GN else 4) * e32)
            worst = report.get(name, (0.0, 0.0))
            report[name] = (max(worst[0], e), max(worst[1], e / bound))
            if not e <= bound:
                fails.append(f"{name}: rel err {e:.3e} > bound {bound:.3e} (float32 oracle {e32:.3e}); worst "
                             + locate(case, n0, worst_at(g, r64)[:2], name))

        o64 = {k: v.detach().numpy() for k, v in rec[torch.float64].items()}
        o32 = {k: v.detach().numpy() for k, v in rec[torch.float32].items()}
        for name in names:
            check(name, got[name], FORWARD[name][1](o64), FORWARD[name][1](o32))
        check("value", got["value"], aux[torch.float64]["value"], aux[torch.float32]["value"])
        # logits: legal entries (the illegal ones are masked in the oracle); mask both to the legal entries, same layout for the locator
        for name, key in (("lg", "g_logits"), ("ll", "a_logits")):
            r64, r32 = aux[torch.float64][key], aux[torch.float32][key]
            check(name, np.where(legal, got[name], 0.0), np.where(legal, r64, 0.0), np.where(legal, r32, 0.0))
        # per-row loss gradients at the CUDA path's own logits and values
        mean, std = stats[u]
        edge, taken = branch_edge_rows(got["lg"], got["ll"], got["value"], part, legal, mean, std, olr.SysCfg())
        edges += int(edge.sum())
        assert edge.mean() < 1e-3, f"{edge.sum()} rows on a branch edge"
        for k, v in taken.items():
            report["taken/" + k] = report.get("taken/" + k, 0) + v
        with fixed_adv_stats(mean, std):
            rg = {dtype: loss_row_grads(got["lg"], got["ll"], got["value"], part, legal, olr.SysCfg(), weight, dtype)
                  for dtype in (torch.float64, torch.float32)}
        keep = ~edge
        for name in LOSS_GRADS:
            g = np.where(keep[..., None] if name != "dvalue" else keep, got[name], 0.0)
            r64 = np.where(keep[..., None] if name != "dvalue" else keep, rg[torch.float64][name], 0.0)
            r32 = np.where(keep[..., None] if name != "dvalue" else keep, rg[torch.float32][name], 0.0)
            check(name, g, r64, r32)
        print(f"{case.env} envs [{n0}, {n1}): {len(fails)} failures", flush=True)
        assert not fails, f"{case.env}, envs [{n0}, {n1}):\n" + "\n".join(fails)
    report["rows on a branch edge (excluded from dlg/dll/dvalue)"] = edges
    for k in taken:  # every branch of the losses is taken on many rows
        assert report["taken/" + k] >= 1000, (k, report["taken/" + k])
    return ref, loss_ref


def compare_params(case, p, grads, ref, loss_ref, report):
    gv, av = param_views(grads[:p.ng], p.gt), param_views(grads[p.ng:p.ng + p.na], p.at)
    fails = []
    for name, r64 in ref[torch.float64].items():
        got = (gv if name in gv else av)[name].cpu().numpy()
        e, e32 = rel_err(got, r64), rel_err(ref[torch.float32][name], r64)
        bound = max(2e-4, (8 if name.startswith(CROSS_GN_GRADS) else 2) * e32)
        worst = report.get("grad", (0.0, 0.0))
        report["grad"] = (max(worst[0], e), max(worst[1], e / bound))
        print(f"  grad {name}: rel err {e:.3e}, float32 oracle {e32:.3e}, {e / bound:.2f} of the bound")
        if not e <= bound:
            fails.append(f"grad {name}: rel err {e:.3e} > {bound:.3e} (float32 oracle {e32:.3e})")
    ls = grads[p.ng + p.na:].cpu().numpy()
    assert ls[0] == 0 and ls[5] == 0, "unused loss slots were written"
    for i, k in LOSS_SLOTS:
        r = loss_ref[torch.float64][k]
        e = abs(float(ls[i]) - r) / (abs(r) + 1e-6)
        worst = report.get("loss_sums", (0.0, 0.0))
        report["loss_sums"] = (max(worst[0], e), max(worst[1], e / 1e-4))
        if not e <= 1e-4:
            fails.append(f"loss sum {k}: {ls[i]:.7f} vs float64 {r:.7f}")
    assert not fails, f"{case.env}:\n" + "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("env", list(CASES))
def test_minibatch_grads_at_bench_shape(dev, env):
    case = CASES[env]
    mb = make_bench_case(case, seed=5)
    stats = slot_stats(case, mb)
    p = Pass(case, dev)
    report = {}
    try:
        grads = p.run(mb, stats)
        for k, v in p.bufs.items():
            assert bool(torch.isfinite(v).all()), f"{k} has non-finite entries (read from the NaN-filled workspace?)"
        assert bool(torch.isfinite(grads).all())
        # accumulate semantics (chunked updates rely on them): from G0 the call leaves G0 + the gradients
        acc = p.run(mb, stats, p.g0)
        slack = 1e-5 * float(grads.abs().max()) + 2.0 ** -16 * float(p.g0.abs().max())  # atomics' order + the adds' rounding at G0
        assert float((acc - (p.g0 + grads)).abs().max()) <= slack, "the gradients were not added to the buffer's contents"
        del acc
        if env == "lbf":
            base, base_grads = p.snapshot(), grads.clone()
            # the layer-by-layer path must give different bits: the fused chain kernels are what ran above
            lib = L.lib()
            lib.magpo_set_chain_kernels(0)
            try:
                p.run(mb, stats)
            finally:
                lib.magpo_set_chain_kernels(1)
            differ = [k for k in base if not bits_equal(p.bufs[k], base[k])]
            print("buffers the layer path changes:", differ)
            assert len(differ) >= 10, differ
            # a dirty workspace: another minibatch's pass, then the test minibatch again without clearing
            other = make_bench_case(case, seed=6)
            p.run(other, slot_stats(case, other))
            grads = p.run(mb, stats)
            for k in base:
                assert bits_equal(p.bufs[k], base[k]), f"{k} depends on what the workspace held before the call"
            scale = float(base_grads.abs().max())
            assert float((grads - base_grads).abs().max()) <= 1e-5 * scale  # atomics: the summation order only
            del base, base_grads
        ref, loss_ref = run_oracle_chunks(case, p, mb, stats, report)
        compare_params(case, p, grads, ref, loss_ref, report)
    finally:
        print(f"{env}: worst (error, fraction of bound):")
        for k, v in report.items():
            print(f"  {k}: {v}")
        del p
        torch.cuda.empty_cache()


@pytest.mark.gpu
def test_adv_stats_at_bench_shape(dev):
    """magpo_adv_stats at the LBF bench shape: B = 8192 trajectories of T = 128, 2 minibatches of 2 x 2048 envs, a random env_index"""
    E, U, M, A = 4096, 2, 2, 2
    B, Nmb = U * E, U * E // M
    rng = np.random.default_rng(3)
    adv = rng.standard_normal((T, B, A))
    adv[:, E:] = 2 * adv[:, E:] + 3
    adv = adv.astype(np.float32)
    perm = rng.permutation(E)
    env_index = np.stack([u * E + perm for u in range(U)])  # [U, E]: slot u's envs
    adv_d = dt(adv, dev)
    for m in range(M):
        idx = env_index[:, m * (E // M):(m + 1) * (E // M)].reshape(-1).astype(np.int32)
        scratch, stats = torch.zeros(2 * U, dtype=torch.float64, device=dev), torch.zeros(U, 2, device=dev)
        L.call("magpo_adv_stats", L.stream_ptr(), T, B, A, L.ptr(adv_d), L.ptr(dt(idx, dev)), Nmb, U, L.ptr(scratch), L.ptr(stats))
        got = stats.cpu().numpy()
        for u in range(U):
            x = adv[:, idx[u * (Nmb // U):(u + 1) * (Nmb // U)]].astype(np.float64)
            mean, std = x.mean(), x.std()
            print(f"minibatch {m} slot {u}: mean {got[u, 0]} vs {mean}, std {got[u, 1]} vs {std}")
            assert abs(got[u, 0] - mean) <= 1e-6 * std and abs(got[u, 1] - std) <= 1e-6 * std, (m, u, got[u], mean, std)


def test_case_table_matches_bench_defaults(monkeypatch):
    """the cases are the workloads bench.py runs: shapes, minibatch size and rows per chain launch; the oracle chunks partition each
    minibatch inside its slots; the inputs contain every done and mask pattern they claim"""
    import bench

    monkeypatch.setattr(sys, "argv", ["bench.py"])
    args = bench.parse()
    assert (args.num_envs, args.update_batch_size, args.rollout_length, args.chunk_envs) == (4096, 2, T, 4096)
    M = SystemConfig().num_minibatches
    expect = {"lbf": (1_048_576, 8192), "coordsum": (1_572_864, 12288), "rware": (262_144, 2048)}
    for env, case in CASES.items():
        vec = VECS[env](**bench.WORKLOADS[env]["kw"])
        assert (vec.num_agents, vec.obs_dim, vec.action_dim) == (case.A, case.d, case.a), env
        assert case.M == M
        num_envs, U = (1024, 1) if env == "rware" else (args.num_envs, args.update_batch_size)
        assert (case.num_envs, case.U) == (num_envs, U)
        assert case.N == U * num_envs // M and case.N <= args.chunk_envs  # one pass differentiates the whole minibatch
        assert (case.R, case.tiles) == expect[env] and case.tiles > NUM_SMS
        covered = np.concatenate([np.arange(n0, n1) for n0, n1 in case.chunks()])
        assert np.array_equal(covered, np.arange(case.N))
        assert all(n0 // case.Ns == (n1 - 1) // case.Ns for n0, n1 in case.chunks())
    rng = np.random.default_rng(0)
    done = done_pattern(rng, 40)
    per_env = {tuple(r) for r in done.astype(int)}
    assert (done.all(1).any() and (~done.any(1)).any() and (done[:, 0] & ~done[:, 1:].any(1)).any())
    rate = done[np.arange(40) % 5 == 0].mean()
    assert 0.05 < rate < 0.3 and len(per_env) >= 4
    case = CASES["coordsum"]
    mb = tgn.make_case(0, 1, 8, T, case.A, case.d, case.a)
    mask = mask_pattern(rng, mb["action_mask"], mb["action"])
    n_legal = mask.sum(-1)
    assert (n_legal == 1).any() and (n_legal == case.a).any() and ((n_legal > 1) & (n_legal < case.a)).any()
    assert np.take_along_axis(mask, mb["action"][..., None].astype(np.int64), -1).all()
