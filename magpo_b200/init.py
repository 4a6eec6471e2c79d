"""Parameter initialisation and key derivation of `learner_setup` (rec_magpo.py:533-685).

Initialisers follow the flax ones named in the reference (orthogonal(sqrt(2)) torsos / Sable encoders,
orthogonal(0.01) output layers, normal(1/embed_dim) retention weights, zeros SwiGLU, lecun_normal / orthogonal
GRU kernels — networks/torsos.py:40,89-95, sable_network.py:97-107,263-282, retention.py:50-64,237-246, flax
GRUCell). Two families: `init_guider / init_actor` draw from a NumPy generator (benchmarks and parity tests: parameters are passed
explicitly to both sides), `flax_init_guider / flax_init_actor` (bottom of the file, used by `learner_setup`) follow flax's own
derivation from the net keys: per-parameter keys folded from the module path, jax.random.normal / truncated_normal draws, QR.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib as L


def _orthogonal(rng, rows, cols, gain):
    a = rng.standard_normal((max(rows, cols), min(rows, cols)))
    q, r = np.linalg.qr(a)
    q = q * np.sign(np.diag(r))
    if rows < cols:
        q = q.T
    return (gain * q[:rows, :cols]).astype(np.float32)


def _normal(rng, rows, cols, std):
    return (rng.standard_normal((rows, cols)) * std).astype(np.float32)


def init_guider(n_agents: int, obs_dim: int, action_dim: int, seed: int = 0, D: int = 64, n_head: int = 1, n_block: int = 1) -> dict:
    rng = np.random.default_rng(seed)
    hs = D // n_head
    ones, zeros = (lambda n: np.ones(n, np.float32)), (lambda *s: np.zeros(s, np.float32))
    p = {"encoder/obs_encoder/layers_0/scale": ones(obs_dim),
         "encoder/obs_encoder/layers_1/kernel": _orthogonal(rng, obs_dim, D, math.sqrt(2)),
         "encoder/ln/scale": ones(D)}

    def retn(pre):
        p[f"{pre}/w_g"], p[f"{pre}/w_o"] = _normal(rng, D, D, 1 / D), _normal(rng, D, D, 1 / D)
        p[f"{pre}/group_norm/scale"], p[f"{pre}/group_norm/bias"] = ones(hs), zeros(hs)
        for h in range(n_head):
            for w in ("w_q", "w_k", "w_v"):
                p[f"{pre}/retention_heads_{h}/{w}"] = _normal(rng, D, hs, 1 / D)

    def ffn(pre):
        for w in ("W_linear", "W_gate", "W_output"):
            p[f"{pre}/{w}"] = zeros(D, D)

    def head(pre, nout):
        p[f"{pre}/layers_0/kernel"], p[f"{pre}/layers_0/bias"] = _orthogonal(rng, D, D, math.sqrt(2)), zeros(D)
        p[f"{pre}/layers_2/scale"] = ones(D)
        p[f"{pre}/layers_3/kernel"], p[f"{pre}/layers_3/bias"] = _orthogonal(rng, D, nout, 0.01), zeros(nout)

    for b in range(n_block):
        eb = f"encoder/encoder_block_{b}"
        p[f"{eb}/ln1/scale"], p[f"{eb}/ln2/scale"] = ones(D), ones(D)
        retn(f"{eb}/retn")
        ffn(f"{eb}/ffn")
    head("encoder/head", 1)
    p["decoder/action_encoder/layers_0/kernel"] = _orthogonal(rng, action_dim + 1, D, math.sqrt(2))
    p["decoder/ln/scale"] = ones(D)
    for b in range(n_block):
        db = f"decoder/decoder_block_{b}"
        for ln in ("ln1", "ln2", "ln3"):
            p[f"{db}/{ln}/scale"] = ones(D)
        retn(f"{db}/retn1")
        retn(f"{db}/retn2")
        ffn(f"{db}/ffn")
    head("decoder/head", action_dim)
    return p


def init_actor(obs_dim: int, action_dim: int, seed: int = 1, H: int = 128) -> dict:
    rng = np.random.default_rng(seed)
    zeros = lambda *s: np.zeros(s, np.float32)
    g = "ScannedRNN_0/GRUCell_0"
    p = {"pre_torso/Dense_0/kernel": _orthogonal(rng, obs_dim, H, math.sqrt(2)), "pre_torso/Dense_0/bias": zeros(H)}
    for n in ("ir", "iz", "in"):
        p[f"{g}/{n}/kernel"], p[f"{g}/{n}/bias"] = _normal(rng, H, H, 1 / math.sqrt(H)), zeros(H)
    for n in ("hr", "hz", "hn"):
        p[f"{g}/{n}/kernel"] = _orthogonal(rng, H, H, 1.0)
    p[f"{g}/hn/bias"] = zeros(H)
    p["post_torso/Dense_0/kernel"], p["post_torso/Dense_0/bias"] = _orthogonal(rng, H, H, math.sqrt(2)), zeros(H)
    p["action_head/Dense_0/kernel"], p["action_head/Dense_0/bias"] = _orthogonal(rng, H, action_dim, 0.01), zeros(action_dim)
    return p


def prng_key(seed: int) -> np.ndarray:
    """jax.random.PRNGKey(seed) as raw uint32[2]."""
    return np.array([(seed >> 32) & 0xFFFFFFFF, seed & 0xFFFFFFFF], dtype=np.uint32)


def split(key: np.ndarray, num: int = 2, device="cuda:0") -> np.ndarray:
    """jax.random.split through the library's threefry kernel (jax_threefry_partitionable scheme)."""
    k = torch.as_tensor(np.asarray(key, np.uint32).view(np.int32)).to(device)
    out = torch.zeros(num, 2, dtype=torch.int32, device=device)
    L.call("magpo_prng_split", L.stream_ptr(), L.ptr(k), num, L.ptr(out))
    return out.cpu().numpy().view(np.uint32)


def setup_keys(seed: int, n_devices: int, U: int, E: int, device="cuda:0"):
    """Key plumbing of run_experiment / learner_setup (rec_magpo.py:699-701, 642-673):
    returns (env reset keys [n_devices, U*E, 2], the step key shared by every device and slot, net keys)."""
    key, key_e, actor_net_key, net_key = split(prng_key(seed), 4, device)
    allk = split(key, n_devices * U * E + 1, device)
    key, env_keys = allk[0], allk[1:].reshape(n_devices, U * E, 2)
    step_key = split(key, 2, device)[1]
    return env_keys, step_key, (actor_net_key, net_key)


# ----------------------------------------------------------------------------- flax-shaped initialisation from the net keys
# `sable_network.init(net_key, ...)` / `actor_network.init(actor_net_key, ...)` (rec_magpo.py:596-606). flax gives every parameter its
# own key, derived on the host from the module path (flax.core.scope, 0.10.3, restated from memory — unverifiable here):
#     key(param) = jax.random.fold_in(root_key, uint32(sha1(name_1 + name_2 + ... + counter_bytes)[:4]))
# with the names of the enclosing scopes from the root down and `counter` = how many parameters that scope created before this one
# (big-endian bytes, empty for 0). The draws are jax.random.normal / truncated_normal from that key (library kernels over the same
# threefry bits), the orthogonal initialiser is flax's: QR of a normal matrix (LAPACK Householder, as jnp.linalg.qr on CPU), columns
# signed by diag(R), transposed when rows < cols. Same keys as the reference; the last bits can differ (erf_inv's log1p, the QR).
def _flax_param_key(root_key: np.ndarray, path: tuple, counter: int) -> np.ndarray:
    import hashlib

    m = hashlib.sha1()
    for name in path:
        m.update(name.encode("utf-8"))
    if counter:
        m.update(counter.to_bytes((counter.bit_length() + 7) // 8, byteorder="big"))
    data = int.from_bytes(m.digest()[:4], byteorder="big")
    key = (C.c_uint32 * 2)(*[int(x) for x in np.asarray(root_key, np.uint32)])
    out = (C.c_uint32 * 2)()
    L.check(L.lib().magpo_prng_fold_in_host(key, C.c_uint32(data), out), "magpo_prng_fold_in_host")
    return np.array([out[0], out[1]], np.uint32)


def _draw(key: np.ndarray, n: int, device, truncated: bool = False) -> np.ndarray:
    k = torch.as_tensor(np.asarray(key, np.uint32).view(np.int32)).to(device)
    out = torch.empty(n, dtype=torch.float32, device=device)
    if truncated:
        L.call("magpo_prng_truncated_normal", L.stream_ptr(), L.ptr(k), C.c_int64(n), C.c_float(-2.0), C.c_float(2.0), L.ptr(out))
    else:
        L.call("magpo_prng_normal", L.stream_ptr(), L.ptr(k), C.c_int64(n), L.ptr(out))
    return out.cpu().numpy()


def _flax_normal(key, shape, stddev, device):
    return (_draw(key, int(np.prod(shape)), device).reshape(shape) * np.float32(stddev)).astype(np.float32)


def _flax_orthogonal(key, shape, scale, device):
    """flax.linen.initializers.orthogonal(scale): rows = prod(shape[:-1]), cols = shape[-1]."""
    rows, cols = int(np.prod(shape[:-1])), int(shape[-1])
    mshape = (cols, rows) if rows < cols else (rows, cols)
    a = _draw(key, mshape[0] * mshape[1], device).reshape(mshape)
    q, r = np.linalg.qr(a)  # float32 LAPACK geqrf / orgqr
    d = np.diag(r)
    q = q * np.where(d >= 0, 1.0, -1.0).astype(np.float32)  # jnp: Q *= sign-like factor of diag(R) (expand_dims over rows)
    if rows < cols:
        q = q.T
    return (np.float32(scale) * q.reshape(shape)).astype(np.float32)


def _flax_lecun_normal(key, shape, device):
    """variance_scaling(1.0, "fan_in", "truncated_normal"): truncated_normal(-2, 2) * sqrt(1 / fan_in) / .87962566103423978."""
    std = np.float32(np.sqrt(1.0 / shape[0]) / 0.87962566103423978)
    return (_draw(key, int(np.prod(shape)), device, truncated=True).reshape(shape) * std).astype(np.float32)


def flax_init_guider(net_key, n_agents: int, obs_dim: int, action_dim: int, device="cuda:0", D: int = 64, n_head: int = 1,
                     n_block: int = 1) -> dict:
    """SableNetwork.init(net_key, ...) (rec_magpo.py:596-601): the parameter tree of networks/sable_network.py with flax's own
    per-parameter keys and initialisers (orthogonal(sqrt 2) encoders / head hidden layers, orthogonal(0.01) output layers, normal(1 / D)
    retention weights, zeros SwiGLU, ones norms)."""
    p = init_guider(n_agents, obs_dim, action_dim, 0, D, n_head, n_block)  # shapes + the constant (ones / zeros) tensors
    sq2 = np.sqrt(np.float32(2.0))
    hs = D // n_head

    def orth(path, shape, scale):  # a Dense kernel is its scope's first parameter
        return _flax_orthogonal(_flax_param_key(net_key, path, 0), shape, scale, device)

    p["encoder/obs_encoder/layers_1/kernel"] = orth(("encoder", "obs_encoder", "layers_1"), (obs_dim, D), sq2)
    p["decoder/action_encoder/layers_0/kernel"] = orth(("decoder", "action_encoder", "layers_0"), (action_dim + 1, D), sq2)
    for side, nout in (("encoder", 1), ("decoder", action_dim)):
        p[f"{side}/head/layers_0/kernel"] = orth((side, "head", "layers_0"), (D, D), sq2)
        p[f"{side}/head/layers_3/kernel"] = orth((side, "head", "layers_3"), (D, nout), 0.01)
    retns = [f"encoder/encoder_block_{b}/retn" for b in range(n_block)]
    retns += [f"decoder/decoder_block_{b}/{r}" for b in range(n_block) for r in ("retn1", "retn2")]
    for retn in retns:
        path = tuple(retn.split("/"))
        for i, w in enumerate(("w_g", "w_o")):  # MultiScaleRetention.setup: w_g, w_o, then the submodules (retention.py:237-246)
            p[f"{retn}/{w}"] = _flax_normal(_flax_param_key(net_key, path, i), (D, D), 1.0 / D, device)
        for h in range(n_head):
            for i, w in enumerate(("w_q", "w_k", "w_v")):  # SimpleRetention.setup (retention.py:47-64)
                p[f"{retn}/retention_heads_{h}/{w}"] = _flax_normal(_flax_param_key(net_key, path + (f"retention_heads_{h}",), i), (D, hs),
                                                                    1.0 / D, device)
    return p


def flax_init_actor(actor_net_key, obs_dim: int, action_dim: int, device="cuda:0", H: int = 128) -> dict:
    """RecurrentActor.init(actor_net_key, ...) (rec_magpo.py:602-606; networks/base.py:152-184, torsos.py:36-47, heads.py:32-46, flax
    GRUCell): orthogonal(sqrt 2) torsos, lecun_normal input kernels, orthogonal recurrent kernels, orthogonal(0.01) action head."""
    p = init_actor(obs_dim, action_dim, 0, H)
    sq2 = np.float32(np.sqrt(2.0))
    g = ("ScannedRNN_0", "GRUCell_0")
    p["pre_torso/Dense_0/kernel"] = _flax_orthogonal(_flax_param_key(actor_net_key, ("pre_torso", "Dense_0"), 0), (obs_dim, H), sq2, device)
    for n in ("ir", "iz", "in"):
        p[f"ScannedRNN_0/GRUCell_0/{n}/kernel"] = _flax_lecun_normal(_flax_param_key(actor_net_key, g + (n,), 0), (H, H), device)
    for n in ("hr", "hz", "hn"):
        p[f"ScannedRNN_0/GRUCell_0/{n}/kernel"] = _flax_orthogonal(_flax_param_key(actor_net_key, g + (n,), 0), (H, H), 1.0, device)
    p["post_torso/Dense_0/kernel"] = _flax_orthogonal(_flax_param_key(actor_net_key, ("post_torso", "Dense_0"), 0), (H, H), sq2, device)
    p["action_head/Dense_0/kernel"] = _flax_orthogonal(_flax_param_key(actor_net_key, ("action_head", "Dense_0"), 0), (H, action_dim), 0.01, device)
    return p


def flax_init_critic(critic_net_key, obs_dim: int, device="cuda:0", H: int = 128) -> dict:
    """RecurrentValueNet.init(critic_net_key, ...) (rec_ippo.py learner_setup; networks/base.py:187-226): the actor's torsos and GRU
    with flax_init_actor's initialisers, and a Dense(1) head with orthogonal(1.0) under the path the parameter table names."""
    p = flax_init_actor(critic_net_key, obs_dim, 1, device, H)
    del p["action_head/Dense_0/kernel"], p["action_head/Dense_0/bias"]
    p["Dense_0/kernel"] = _flax_orthogonal(_flax_param_key(critic_net_key, ("Dense_0",), 0), (H, 1), 1.0, device)
    p["Dense_0/bias"] = np.zeros(1, np.float32)
    return p
