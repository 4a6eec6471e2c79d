"""ctypes binding of libmagpo_b200.so (the C ABI declared in include/magpo_b200.h).

The product path has no CPU fallback: if the shared library is missing this module raises at
import of the first symbol.  torch is used by the callers only as the owner of device memory
and streams; every entry point takes raw device pointers.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmagpo_b200.so")

OK, ERR_ARG, ERR_UNSUPPORTED, ERR_CUDA, ERR_WORKSPACE = 0, -1, -2, -3, -4
_ERR = {ERR_ARG: "bad argument", ERR_UNSUPPORTED: "unsupported configuration", ERR_CUDA: "CUDA error",
        ERR_WORKSPACE: "workspace too small"}

ENV_COORDSUM, ENV_LBF, ENV_RWARE = 0, 1, 2

vp = C.c_void_p


class MagpoError(RuntimeError):
    pass


class NetCfg(C.Structure):
    _fields_ = [("n_agents", C.c_int32), ("obs_dim", C.c_int32), ("action_dim", C.c_int32),
                ("embed_dim", C.c_int32), ("n_head", C.c_int32), ("n_block", C.c_int32),
                ("hidden", C.c_int32), ("timestep_pe", C.c_int32), ("decay_scaling_factor", C.c_float),
                ("max_step_count", C.c_int32)]


class SysCfg(C.Structure):
    _fields_ = [("num_envs", C.c_int32), ("update_batch_size", C.c_int32), ("rollout_length", C.c_int32),
                ("ppo_epochs", C.c_int32), ("num_minibatches", C.c_int32)] + [
        (n, C.c_double) for n in ("gamma", "gae_lambda", "clip_eps", "ent_coef", "vf_coef", "max_grad_norm",
                                  "clip_gpo", "alpha", "lr")] + [("sable_only", C.c_int32)]


class TimeStep(C.Structure):
    _fields_ = [(n, vp) for n in ("step_type", "reward", "discount", "agents_view", "action_mask", "step_count",
                                  "next_agents_view", "next_step_count", "episode_return", "episode_length",
                                  "is_terminal_step")]


class CoordSumCfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("num_agents", "num_actions", "time_limit", "maxval")]


class CoordSumState(C.Structure):
    _fields_ = [(n, vp) for n in ("step_count", "target", "record", "key", "metrics_key", "running_return",
                                  "running_length", "episode_return", "episode_length")]


class LbfCfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("grid_size", "fov", "num_agents", "num_food", "max_agent_level", "force_coop",
                                         "time_limit", "agent_mask_rows")]


class LbfState(C.Structure):
    _fields_ = [(n, vp) for n in ("agent_pos", "agent_level", "agent_loading", "food_pos", "food_level", "food_eaten",
                                  "step_count", "key", "metrics_key", "running_return", "running_length", "episode_return",
                                  "episode_length")]


class RwareCfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("column_height", "shelf_rows", "shelf_columns", "num_agents", "sensor_range",
                                         "request_queue_size", "time_limit")]


class RwareState(C.Structure):
    _fields_ = [(n, vp) for n in ("grid", "agent_pos", "agent_dir", "agent_carry", "shelf_pos", "shelf_req", "request_queue",
                                  "step_count", "action_mask", "key", "metrics_key", "running_return", "running_length",
                                  "episode_return", "episode_length")]


class SableHState(C.Structure):
    _fields_ = [(n, vp) for n in ("encoder", "decoder_self", "decoder_cross")]


class Trajectory(C.Structure):
    _fields_ = [(n, vp) for n in ("done", "agents_view", "action_mask", "step_count", "action", "value", "reward",
                                  "log_prob", "policy_h0")] + [("sable_h0", SableHState)] + [
        (n, vp) for n in ("episode_return", "episode_length", "is_terminal_step", "last_value")]


class Minibatch(C.Structure):
    _fields_ = [("T", C.c_int32), ("N", C.c_int32)] + [
        (n, vp) for n in ("agents_view", "action_mask", "step_count", "done", "action", "value", "log_prob",
                          "advantages", "targets", "policy_h0")] + [("sable_h0", SableHState)]


_lib = None


def lib() -> C.CDLL:
    """The loaded library; raises (no fallback) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MagpoError(f"{LIB_PATH} not found: run `make` (or __graft_entry__.build()) first — there is no CPU fallback")
        _lib = C.CDLL(LIB_PATH)
        _lib.magpo_version.restype = C.c_char_p
        _lib.magpo_last_cuda_error.restype = C.c_char_p
        for name in ("magpo_param_count", "magpo_rollout_workspace_bytes", "magpo_update_workspace_bytes"):
            if hasattr(_lib, name):
                getattr(_lib, name).restype = C.c_int64
    return _lib


_contexts: dict = {}


def create_context(device=None) -> vp:
    """A new MagpoContext (include/magpo_b200.h) on `device` (torch device / ordinal; default: the current CUDA device). The caller
    owns it: `destroy_context` when done. Every MagpoLearner creates its own."""
    import torch

    idx = torch.cuda.current_device() if device is None else torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    out = vp()
    check(lib().magpo_context_create(int(idx), C.byref(out)), "magpo_context_create")
    return out


def destroy_context(ctx: vp) -> None:
    if ctx:
        lib().magpo_context_destroy(ctx)


def context(device=None) -> vp:
    """The shared per-device context of helper code that has no learner of its own (evaluator loops, tests, tools)."""
    import torch

    idx = torch.cuda.current_device() if device is None else (torch.device(device).index or 0)
    if idx not in _contexts:
        _contexts[idx] = create_context(idx)
    return _contexts[idx]


def ptr(t) -> vp:
    """Device (or host) pointer of a torch tensor / None."""
    if t is None:
        return vp(0)
    assert t.is_contiguous(), "C ABI needs contiguous buffers"
    return vp(t.data_ptr())


def struct_of(cls, **tensors):
    s = cls()
    for k, v in tensors.items():
        if isinstance(v, C.Structure):
            setattr(s, k, v)
        elif isinstance(v, int):
            setattr(s, k, v)
        else:
            setattr(s, k, ptr(v))
    s._keepalive = tensors  # the tensors must outlive the call
    return s


def check(rc: int, what: str = "") -> None:
    if rc != OK:
        msg = _ERR.get(rc, f"error {rc}")
        if rc == ERR_CUDA:
            msg += ": " + lib().magpo_last_cuda_error().decode()
        raise MagpoError(f"{what}: {msg}")


def call(name: str, *args) -> None:
    check(getattr(lib(), name)(*args), name)


def workspace_bytes(name: str, *args) -> int:
    """The workspace size of an entry point that answers the CUB-style query (the rec_ippo ones): `args` are every argument before
    `workspace`; called with workspace NULL it writes the size to its `size_t* workspace_bytes`."""
    n = C.c_size_t(0)
    check(getattr(lib(), name)(*args, None, C.byref(n)), name)
    return int(n.value)


def stream_ptr(stream=None) -> vp:
    import torch

    s = stream if stream is not None else torch.cuda.current_stream()
    return vp(s.cuda_stream)
