"""Sable guider + GRU learner restated in torch (CPU, fp32 or fp64) — oracle only.

Follows, layer by layer:
  * `mava/networks/sable_network.py:40-482`  EncodeBlock/Encoder/DecodeBlock/Decoder/SableNetwork
  * `mava/networks/retention.py:33-323`      SimpleRetention (chunkwise + recurrent), MultiScaleRetention
  * `mava/networks/utils/sable/encode.py:27-84`, `decode.py:36-153`, `positional_encoding.py:24-58`
  * `mava/networks/base.py:121-184`          ScannedRNN / RecurrentActor
  * `mava/networks/torsos.py:24-47,79-99`    MLPTorso, SwiGLU;  `heads.py:26-63` DiscreteActionHead
and the flax/distrax arithmetic of SURVEY.md Appendix A7-A10 (flax 0.10.3, distrax 0.1.5 are
pinned deps not under /root/reference).  Parameters are flat dicts keyed by the flax tree
path ("encoder/encoder_block_0/retn/retention_heads_0/w_q", ...).  torch is used so that
`jax.value_and_grad` can be mirrored by autograd.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F

from . import prng

F32_MIN = float(np.finfo(np.float32).min)

# Optional tap for parity debugging: when set to a dict, forward passes store named intermediates in it
# (tests compare them with the CUDA path's saved activations).
RECORD: dict | None = None


def _rec(name, t):
    if RECORD is not None:
        RECORD[name] = t
    return t


@dataclass
class NetCfg:
    n_agents: int
    obs_dim: int
    action_dim: int
    embed_dim: int = 64
    n_head: int = 1
    n_block: int = 1
    decay_scaling_factor: float = 0.8
    timestep_pe: bool = True
    hidden: int = 128  # learner hidden_state_dim == pre/post torso width
    timestep_chunk_size: int | None = None

    @property
    def head_size(self):
        return self.embed_dim // self.n_head

    def kappas(self):
        # retention.py:231-234 / sable_network.py:366-369 (float32 arithmetic)
        k = 1 - np.exp(np.linspace(np.log(np.float32(1 / 32)), np.log(np.float32(1 / 512)), self.n_head, dtype=np.float32))
        return (k.astype(np.float32) * np.float32(self.decay_scaling_factor)).astype(np.float32)


# ----------------------------------------------------------------------------- init
def _orthogonal(rng, shape, gain):
    rows, cols = shape
    a = rng.standard_normal((max(rows, cols), min(rows, cols)))
    q, r = np.linalg.qr(a)
    q = q * np.sign(np.diag(r))
    if rows < cols:
        q = q.T
    return (gain * q[:rows, :cols]).astype(np.float32)


def _retention_params(rng, D, hs, n_head, prefix, out):
    sd = 1.0 / D
    out[f"{prefix}/w_g"] = (rng.standard_normal((D, D)) * sd).astype(np.float32)
    out[f"{prefix}/w_o"] = (rng.standard_normal((D, D)) * sd).astype(np.float32)
    out[f"{prefix}/group_norm/scale"] = np.ones(hs, np.float32)
    out[f"{prefix}/group_norm/bias"] = np.zeros(hs, np.float32)
    for h in range(n_head):
        for w in ("w_q", "w_k", "w_v"):
            out[f"{prefix}/retention_heads_{h}/{w}"] = (rng.standard_normal((D, hs)) * sd).astype(np.float32)


def init_guider_params(cfg: NetCfg, seed: int = 0, ffn_zero: bool = True) -> dict:
    """Same distributions as the flax initialisers (SURVEY Appendix A7/A9); NOT the same bits as
    jax.random (QR-based orthogonal init cannot be reproduced without JAX)."""
    rng = np.random.default_rng(seed)
    D, hs, d, a = cfg.embed_dim, cfg.head_size, cfg.obs_dim, cfg.action_dim
    p: dict = {}
    p["encoder/obs_encoder/layers_0/scale"] = np.ones(d, np.float32)
    p["encoder/obs_encoder/layers_1/kernel"] = _orthogonal(rng, (d, D), math.sqrt(2))
    p["encoder/ln/scale"] = np.ones(D, np.float32)
    for b in range(cfg.n_block):
        pre = f"encoder/encoder_block_{b}"
        p[f"{pre}/ln1/scale"] = np.ones(D, np.float32)
        p[f"{pre}/ln2/scale"] = np.ones(D, np.float32)
        _retention_params(rng, D, hs, cfg.n_head, f"{pre}/retn", p)
        for w, shp in (("W_linear", (D, D)), ("W_gate", (D, D)), ("W_output", (D, D))):
            p[f"{pre}/ffn/{w}"] = np.zeros(shp, np.float32) if ffn_zero else (rng.standard_normal(shp) / D).astype(np.float32)
    p["encoder/head/layers_0/kernel"] = _orthogonal(rng, (D, D), math.sqrt(2))
    p["encoder/head/layers_0/bias"] = np.zeros(D, np.float32)
    p["encoder/head/layers_2/scale"] = np.ones(D, np.float32)
    p["encoder/head/layers_3/kernel"] = _orthogonal(rng, (D, 1), 0.01)
    p["encoder/head/layers_3/bias"] = np.zeros(1, np.float32)
    p["decoder/action_encoder/layers_0/kernel"] = _orthogonal(rng, (a + 1, D), math.sqrt(2))
    p["decoder/ln/scale"] = np.ones(D, np.float32)
    for b in range(cfg.n_block):
        pre = f"decoder/decoder_block_{b}"
        for ln in ("ln1", "ln2", "ln3"):
            p[f"{pre}/{ln}/scale"] = np.ones(D, np.float32)
        _retention_params(rng, D, hs, cfg.n_head, f"{pre}/retn1", p)
        _retention_params(rng, D, hs, cfg.n_head, f"{pre}/retn2", p)
        for w, shp in (("W_linear", (D, D)), ("W_gate", (D, D)), ("W_output", (D, D))):
            p[f"{pre}/ffn/{w}"] = np.zeros(shp, np.float32) if ffn_zero else (rng.standard_normal(shp) / D).astype(np.float32)
    p["decoder/head/layers_0/kernel"] = _orthogonal(rng, (D, D), math.sqrt(2))
    p["decoder/head/layers_0/bias"] = np.zeros(D, np.float32)
    p["decoder/head/layers_2/scale"] = np.ones(D, np.float32)
    p["decoder/head/layers_3/kernel"] = _orthogonal(rng, (D, a), 0.01)
    p["decoder/head/layers_3/bias"] = np.zeros(a, np.float32)
    return p


def init_actor_params(cfg: NetCfg, seed: int = 1) -> dict:
    rng = np.random.default_rng(seed)
    H, d, a = cfg.hidden, cfg.obs_dim, cfg.action_dim
    p: dict = {}
    p["pre_torso/Dense_0/kernel"] = _orthogonal(rng, (d, H), math.sqrt(2))
    p["pre_torso/Dense_0/bias"] = np.zeros(H, np.float32)
    g = "ScannedRNN_0/GRUCell_0"
    for n in ("ir", "iz", "in"):  # lecun_normal + bias (Appendix A8)
        p[f"{g}/{n}/kernel"] = (rng.standard_normal((H, H)) / math.sqrt(H)).astype(np.float32)
        p[f"{g}/{n}/bias"] = np.zeros(H, np.float32)
    for n in ("hr", "hz", "hn"):
        p[f"{g}/{n}/kernel"] = _orthogonal(rng, (H, H), 1.0)
    p[f"{g}/hn/bias"] = np.zeros(H, np.float32)
    p["post_torso/Dense_0/kernel"] = _orthogonal(rng, (H, H), math.sqrt(2))
    p["post_torso/Dense_0/bias"] = np.zeros(H, np.float32)
    p["action_head/Dense_0/kernel"] = _orthogonal(rng, (H, a), 0.01)
    p["action_head/Dense_0/bias"] = np.zeros(a, np.float32)
    return p


def to_torch(p: dict, dtype=torch.float32, requires_grad=False) -> dict:
    return {k: torch.tensor(np.asarray(v), dtype=dtype, requires_grad=requires_grad) for k, v in p.items()}


# ----------------------------------------------------------------------------- primitives
def rmsnorm(x, scale, eps=1e-6):  # flax nn.RMSNorm (Appendix A9): y = x * (rsqrt(mean(x^2)+eps) * scale)
    return x * (torch.rsqrt((x * x).mean(-1, keepdim=True) + eps) * scale)


def groupnorm_rows(x, scale, bias, num_groups, eps=1e-6):
    """flax nn.GroupNorm on [rows, feat] (retention.py:289-291): stats per row per group, fast variance."""
    rows, feat = x.shape
    xg = x.reshape(rows, num_groups, feat // num_groups)
    mean = xg.mean(-1, keepdim=True)
    var = torch.clamp((xg * xg).mean(-1, keepdim=True) - mean * mean, min=0.0)
    y = (xg - mean) * torch.rsqrt(var + eps)
    return y.reshape(rows, feat) * scale + bias


def gelu(x):  # flax nn.gelu default approximate=True
    return F.gelu(x, approximate="tanh")


def swish(x):
    return x * torch.sigmoid(x)


def pos_encoding(step_count, D, dtype):
    """positional_encoding.py:24-58: pe[...,0::2]=sin(pos*div), pe[...,1::2]=cos(pos*div)."""
    div = torch.exp(torch.arange(0, D, 2, dtype=torch.float32) * (-math.log(10000.0) / D)).to(dtype)
    x = step_count.to(dtype)[..., None] * div
    pe = torch.zeros(*step_count.shape, D, dtype=dtype)
    pe[..., 0::2] = torch.sin(x)
    pe[..., 1::2] = torch.cos(x)
    return pe


def swiglu(p, pre, x):  # torsos.py:79-99
    gate, linear = _rec(f"{pre}/gate", x @ p[f"{pre}/W_gate"]), _rec(f"{pre}/linear", x @ p[f"{pre}/W_linear"])
    return _rec(f"{pre}/out", _rec(f"{pre}/hmid", swish(gate) * linear) @ p[f"{pre}/W_output"])


# ----------------------------------------------------------------------------- retention
def _decay_matrix(ts_dones, kappa, n_agents, masked, dtype):
    """retention.py:117-187. ts_dones bool[B,T] -> D float[B, T*A, T*A]."""
    B, T = ts_dones.shape
    n = torch.arange(T)[:, None]
    m = torch.arange(T)[None, :]
    base = torch.where(n >= m, torch.pow(torch.tensor(float(kappa), dtype=dtype), (n - m).clamp(min=0).to(dtype)), torch.zeros((), dtype=dtype))
    cs = torch.cumsum(ts_dones.to(torch.int64), dim=1)  # done in (m, n]  <=>  cs[n]-cs[m] > 0
    blocked = (cs[:, :, None] - cs[:, None, :]) > 0
    blocked = blocked & (n > m)[None]
    D = base[None] * (~blocked).to(dtype)
    D = D.repeat_interleave(n_agents, dim=1).repeat_interleave(n_agents, dim=2)
    if masked:
        C = T * n_agents
        D = D * torch.tril(torch.ones(C, C, dtype=dtype))[None]
    return D


def _xi(ts_dones, kappa, n_agents, dtype):
    """retention.py:189-213: xi[t] = kappa^(t+1) * [t < first_done]."""
    B, T = ts_dones.shape
    any_done = ts_dones.any(dim=1, keepdim=True)
    first = torch.where(any_done, ts_dones.to(torch.int64).argmax(dim=1, keepdim=True), torch.full((B, 1), T))
    t = torch.arange(T)[None, :]
    xi = torch.pow(torch.tensor(float(kappa), dtype=dtype), (t + 1).to(dtype)) * (t < first).to(dtype)
    return xi.repeat_interleave(n_agents, dim=1)[..., None]


def simple_retention_chunk(p, pre, key, query, value, hstate, dones, kappa, n_agents, masked):
    """SimpleRetention.__call__ (retention.py:66-100), rec_sable branch."""
    B, C, _ = value.shape
    q = _rec(f"{pre}/q", query @ p[f"{pre}/w_q"])
    k = _rec(f"{pre}/k", key @ p[f"{pre}/w_k"])
    v = _rec(f"{pre}/v", value @ p[f"{pre}/w_v"])
    kT = k.transpose(1, 2)
    ts_dones = dones[:, ::n_agents]
    D = _decay_matrix(ts_dones, kappa, n_agents, masked, value.dtype)
    xi = _xi(ts_dones, kappa, n_agents, value.dtype)
    chunk_decay = float(kappa) ** (C // n_agents)
    delta = (~ts_dones.any(dim=1))[:, None, None].to(value.dtype)
    next_h = kT @ (v * D[:, -1].reshape(B, C, 1)) + hstate * chunk_decay * delta
    cross = (q @ hstate) * xi
    inner = ((q @ kT) * D) @ v
    return inner + cross, next_h


def simple_retention_recurrent(p, pre, key, query, value, hstate):
    """SimpleRetention.recurrent (retention.py:102-115)."""
    q = query @ p[f"{pre}/w_q"]
    k = key @ p[f"{pre}/w_k"]
    v = value @ p[f"{pre}/w_v"]
    new_h = hstate + k.transpose(1, 2) @ v
    return q @ new_h, new_h


def msr(p, pre, cfg: NetCfg, key, query, value, hstate, step_count, masked, dones=None):
    """MultiScaleRetention.__call__ (dones given) / .recurrent (dones None). retention.py:265-323.
    hstate [B, n_head, hs, hs]."""
    B, S, D = value.shape
    if cfg.timestep_pe:
        pe = pos_encoding(step_count, D, value.dtype)
        key, query, value = key + pe, query + pe, value + pe
    _rec(f"{pre}/key", key)
    _rec(f"{pre}/query", query)
    outs, new_hs = [], []
    kap = cfg.kappas()
    for h in range(cfg.n_head):
        hp = f"{pre}/retention_heads_{h}"
        if dones is None:
            y, nh = simple_retention_recurrent(p, hp, key, query, value, hstate[:, h])
        else:
            y, nh = simple_retention_chunk(p, hp, key, query, value, hstate[:, h], dones, kap[h], cfg.n_agents, masked)
        outs.append(y)
        new_hs.append(nh)
    ret = torch.cat(outs, dim=-1)
    _rec(f"{pre}/ret", ret)
    ret = groupnorm_rows(ret.reshape(-1, cfg.head_size), p[f"{pre}/group_norm/scale"], p[f"{pre}/group_norm/bias"], cfg.n_head).reshape(ret.shape)
    gated = _rec(f"{pre}/gated", swish(_rec(f"{pre}/g", key @ p[f"{pre}/w_g"])) * ret)
    out = _rec(f"{pre}/out", gated @ p[f"{pre}/w_o"])
    return out, torch.stack(new_hs, dim=1)


# ----------------------------------------------------------------------------- encoder / decoder
def _head(p, pre, x):
    h = gelu(_rec(f"{pre}/zh", x @ p[f"{pre}/layers_0/kernel"] + p[f"{pre}/layers_0/bias"]))
    h = rmsnorm(h, p[f"{pre}/layers_2/scale"])
    return h @ p[f"{pre}/layers_3/kernel"] + p[f"{pre}/layers_3/bias"]


def encoder_apply(p, cfg: NetCfg, obs, hstate, step_count, dones=None):
    """Encoder.__call__ / Encoder.recurrent (sable_network.py:121-156). hstate [B,nh,nb,hs,hs]."""
    on = _rec("enc/on", rmsnorm(obs, p["encoder/obs_encoder/layers_0/scale"]))
    x = gelu(_rec("enc/z0", on @ p["encoder/obs_encoder/layers_1/kernel"]))
    new_h = []
    for b in range(cfg.n_block):
        pre = f"encoder/encoder_block_{b}"
        xin = _rec("enc/xin", rmsnorm(x, p["encoder/ln/scale"]))
        ret, nh = msr(p, f"{pre}/retn", cfg, xin, xin, xin, hstate[:, :, b], step_count, masked=False, dones=dones)
        x1 = _rec("enc/x1", rmsnorm(xin + ret, p[f"{pre}/ln1/scale"]))
        x = _rec("enc/x", rmsnorm(x1 + swiglu(p, f"{pre}/ffn", x1), p[f"{pre}/ln2/scale"]))
        new_h.append(nh)
    value = _head(p, "encoder/head", x)
    return value, x, torch.stack(new_h, dim=2)


def decoder_apply(p, cfg: NetCfg, action_tok, obs_rep, hs_self, hs_cross, step_count, dones=None):
    """Decoder.__call__ / Decoder.recurrent (sable_network.py:296-343)."""
    x = _rec("dec/xD", rmsnorm(gelu(action_tok @ p["decoder/action_encoder/layers_0/kernel"]), p["decoder/ln/scale"]))
    n1, n2 = [], []
    for b in range(cfg.n_block):
        pre = f"decoder/decoder_block_{b}"
        ret, h1 = msr(p, f"{pre}/retn1", cfg, x, x, x, hs_self[:, :, b], step_count, masked=True, dones=dones)
        r = rmsnorm(x + ret, p[f"{pre}/ln1/scale"])
        ret2, h2 = msr(p, f"{pre}/retn2", cfg, r, obs_rep, r, hs_cross[:, :, b], step_count, masked=True, dones=dones)
        y = _rec("dec/y", rmsnorm(obs_rep + ret2, p[f"{pre}/ln2/scale"]))
        x = _rec("dec/xd", rmsnorm(y + swiglu(p, f"{pre}/ffn", y), p[f"{pre}/ln3/scale"]))
        n1.append(h1)
        n2.append(h2)
    logit = _head(p, "decoder/head", x)
    return logit, torch.stack(n1, dim=2), torch.stack(n2, dim=2)


def log_softmax(logits):
    return logits - torch.logsumexp(logits, dim=-1, keepdim=True)


def sable_get_actions(p, cfg: NetCfg, obs, action_mask, step_count, hstates, key, *, forced_actions=None, return_logits=False):
    """SableNetwork.get_actions (sable_network.py:443-482) + discrete_autoregressive_act (decode.py:111-153).

    obs float[B,A,d]; action_mask bool[B,A,a]; step_count int[B,A]; hstates = (enc, dec_self, dec_cross)
    each [B,nh,nb,hs,hs]; key uint32[2].  Returns (action int32[B,A], log_prob[B,A], value[B,A], new hstates).
    `forced_actions` (teacher forcing) is used only by the recurrent==chunkwise self-consistency test.
    """
    B, A, a = action_mask.shape
    dtype = obs.dtype
    kap = torch.tensor(cfg.kappas(), dtype=dtype)[None, :, None, None, None]
    enc_h, ds_h, dc_h = (h * kap for h in hstates)  # decay once per timestep (:457)
    value, obs_rep, enc_new = encoder_apply(p, cfg, obs, enc_h, step_count)
    shifted = torch.zeros(B, A, a + 1, dtype=dtype)
    shifted[:, 0, 0] = 1
    actions = np.zeros((B, A), np.int32)
    logps = torch.zeros(B, A, dtype=dtype)
    all_logits = []
    key = np.asarray(key, np.uint32)
    for i in range(A):
        logit, ds_h, dc_h = decoder_apply(p, cfg, shifted[:, i : i + 1], obs_rep[:, i : i + 1], ds_h, dc_h, step_count[:, i : i + 1])
        masked = torch.where(action_mask[:, i : i + 1], logit, torch.full((), F32_MIN, dtype=dtype))
        all_logits.append(masked[:, 0])
        ks = prng.split(key)
        key, sample_key = ks[0], ks[1]
        norm = log_softmax(masked)[:, 0]  # distrax stores normalised logits
        g = prng.gumbel(sample_key, (1, B, 1, a)).reshape(B, a)
        act = np.argmax(g + norm.detach().to(torch.float32).numpy(), axis=-1).astype(np.int32)
        if forced_actions is not None:
            act = np.asarray(forced_actions[:, i], np.int32)
        actions[:, i] = act
        act_t = torch.from_numpy(act.astype(np.int64))
        logps[:, i] = norm.gather(-1, act_t[:, None])[:, 0]
        if i + 1 < A:
            shifted[:, i + 1, 1:] = F.one_hot(act_t, a).to(dtype)
    out = (actions, logps, value[..., 0], (enc_new, ds_h, dc_h))
    if return_logits:
        return out + (torch.stack(all_logits, dim=1),)
    return out


def shifted_discrete_actions(action, a, n_agents, dtype):
    """get_shifted_discrete_actions (decode.py:86-108)."""
    B, S = action.shape
    sh = torch.zeros(B, S, a + 1, dtype=dtype)
    sh[:, :, 1:] = F.one_hot(action.to(torch.int64), a).to(dtype)
    sh = torch.roll(sh, shifts=1, dims=1)
    start = torch.zeros(a + 1, dtype=dtype)
    start[0] = 1
    sh[:, ::n_agents, :] = start
    return sh


def sable_apply(p, cfg: NetCfg, obs, action_mask, step_count, action, hstates, dones, T):
    """SableNetwork.__call__ (sable_network.py:412-441) with train_encoder_fn / discrete_train_decoder_fn.

    Sequence tensors are [N, C=T*A, ...]. Returns (value[N,C], log_prob[N,C], entropy[N,C], masked logits[N,C,a]).
    """
    N, C = action.shape
    A = cfg.n_agents
    chunk = (cfg.timestep_chunk_size * A) if cfg.timestep_chunk_size else T * A  # rec_magpo.py:552-557
    enc_h, ds_h, dc_h = hstates
    vals, reps = [], []
    for s in range(0, C, chunk):
        sl = slice(s, s + chunk)
        v, r, enc_h = encoder_apply(p, cfg, obs[:, sl], enc_h, step_count[:, sl], dones=dones[:, sl])
        vals.append(v)
        reps.append(r)
    value = torch.cat(vals, dim=1)[..., 0]
    obs_rep = torch.cat(reps, dim=1)
    a = action_mask.shape[-1]
    sh = shifted_discrete_actions(action, a, A, obs.dtype)
    logits = []
    for s in range(0, C, chunk):
        sl = slice(s, s + chunk)
        lg, ds_h, dc_h = decoder_apply(p, cfg, sh[:, sl], obs_rep[:, sl], ds_h, dc_h, step_count[:, sl], dones=dones[:, sl])
        logits.append(lg)
    logit = torch.cat(logits, dim=1)
    masked = torch.where(action_mask, logit, torch.full((), F32_MIN, dtype=obs.dtype))
    logp_all = log_softmax(masked)
    logp = logp_all.gather(-1, action.to(torch.int64)[..., None])[..., 0]
    pr = torch.exp(logp_all)
    ent = -(torch.where(pr == 0, torch.zeros_like(pr), logp_all) * pr).sum(-1)
    return value, logp, ent, masked


# ----------------------------------------------------------------------------- learner (GRU)
def actor_apply(p, cfg: NetCfg, h, obs, done, action_mask):
    """RecurrentActor.__call__ (base.py:161-184) + ScannedRNN (:124-142) + flax GRUCell (Appendix A8).

    h [E,A,H]; obs float[T,E,A,d]; done bool[T,E,A]; action_mask bool[T,E,A,a].
    Returns (h_T, masked logits [T,E,A,a]).
    """
    g = "ScannedRNN_0/GRUCell_0"
    e = torch.relu(obs @ p["pre_torso/Dense_0/kernel"] + p["pre_torso/Dense_0/bias"])
    ys = []
    for t in range(obs.shape[0]):
        h = torch.where(done[t][..., None], torch.zeros_like(h), h)
        x = e[t]
        r = torch.sigmoid(x @ p[f"{g}/ir/kernel"] + p[f"{g}/ir/bias"] + h @ p[f"{g}/hr/kernel"])
        z = torch.sigmoid(x @ p[f"{g}/iz/kernel"] + p[f"{g}/iz/bias"] + h @ p[f"{g}/hz/kernel"])
        n = torch.tanh(x @ p[f"{g}/in/kernel"] + p[f"{g}/in/bias"] + r * (h @ p[f"{g}/hn/kernel"] + p[f"{g}/hn/bias"]))
        h = (1.0 - z) * n + z * h
        ys.append(h)
    y = torch.stack(ys, dim=0)
    y = torch.relu(y @ p["post_torso/Dense_0/kernel"] + p["post_torso/Dense_0/bias"])
    logits = y @ p["action_head/Dense_0/kernel"] + p["action_head/Dense_0/bias"]
    masked = torch.where(action_mask, logits, torch.full((), F32_MIN, dtype=obs.dtype))
    return h, masked
