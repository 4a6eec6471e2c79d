"""The training-pass retention kernels against float64, at every chunk geometry and at the configs' rollout length.

retention_fwd / retention_bwd (csrc/retention.cu) run T = 1 as a register scan and T > 1 as the chunkwise tensor-core kernels of
csrc/retention_chunk.cu. A chunk holds Lc = 32 / A timesteps (the host-only query magpo_debug_retention_chunk_len calls the
function the launches call), so A = 3, 5, 6 and 7 leave padded token rows, and a sequence that is not a multiple of Lc ends in a
ragged chunk. Every A in 1..8 runs
at T = 1, 2, Lc, Lc + 1 and 3 Lc - 1, and the configs' training shapes run at T = 128 (A = 2 at the LBF benchmark's minibatch of
4096 envs), each as the encoder (non-causal) and the decoder (causal), at three decays.

Dones are placed on purpose: on the first and on the last timestep of every chunk, on two consecutive timesteps across each chunk
boundary, on every step, never (with a nonzero H0), at t = 0 only, and at random (p = 0.1) in every other env. q, k and v are packed
with row stride ld at column offsets 0, 64 and 128, and dq, dk and dv go into one buffer of row stride 256, as the training forward
and backward lay them out. Every output starts as NaN and sits between guard regions filled with a sentinel; columns 192..255 of the
gradient buffer (the gate gradients in the training backward) hold the sentinel too. A missed row stays NaN, a stray write changes a
sentinel.

The reference is the oracle's chunkwise form (oracle.nets.simple_retention_chunk: the D matrix / xi formulation) with autograd in
float64; the checkpoints (the state entering each chunk) come from a plain float64 recurrent scan. The same reference in float32 is
the control: each output's bound is max(fixed, 4 x |f32 - f64|) in the max-norm rel_err, over all sampled envs and per env.
"""
import ctypes as C
import zlib
from dataclasses import dataclass

import numpy as np
import pytest
import torch

from magpo_b200 import _lib as L
from oracle import nets as onets

from gpu_util import rel_err

RC_ROWS = 32
# A -> (Lc timesteps per chunk, real token rows of a full chunk)
CHUNKS = {1: (32, 32), 2: (16, 32), 3: (10, 30), 4: (8, 32), 5: (6, 30), 6: (5, 30), 7: (4, 28), 8: (4, 32)}
FIXED = {"ret": 2e-5, "Hout": 2e-5, "Hck": 2e-5, "dq": 5e-5, "dk": 5e-5, "dv": 5e-5}
SENTINEL = 0x7F7FDEAD  # the bits of a finite float no kernel computes here
PATTERNS = ("first", "last", "pair", "every", "never", "t0")


@dataclass(frozen=True)
class Case:
    A: int
    T: int
    N: int
    expect: tuple  # (chunks, timesteps in the last chunk, real token rows of a full chunk)
    ld: int = 256
    h0: bool = True

    @property
    def id(self):
        return f"A{self.A}-T{self.T}-N{self.N}" + (f"-ld{self.ld}" if self.ld != 256 else "") + ("" if self.h0 else "-H0null")


def _geometry_cases():
    out = []
    for A, (lc, rows) in CHUNKS.items():
        N = 8 if A % 2 else 7
        out += [Case(A, 1, N, (1, 1, rows)),                  # the register scan
                Case(A, 2, N, (1, 2, rows)),                  # the smallest chunked sequence
                Case(A, lc, N, (1, lc, rows)),                # one full chunk
                Case(A, lc + 1, N, (2, 1, rows)),             # a last chunk of one timestep
                Case(A, 3 * lc - 1, N, (3, lc - 1, rows))]    # three chunks, the last one short by a step
    return out


CASES = _geometry_cases() + [
    Case(3, 29, 5, (3, 9, 30), ld=196),        # q / k / v rows not 256 floats apart
    Case(2, 17, 3, (2, 1, 32), ld=196),
    Case(7, 11, 5, (3, 3, 28), h0=False),      # H0 = nullptr: a zero initial state
    Case(1, 1, 3, (1, 1, 32), h0=False),
    Case(2, 128, 4096, (8, 16, 32)),           # LBF, the benchmark: the minibatch of 4096 envs
    Case(3, 128, 300, (13, 8, 30)),            # CoordSum 3x10-30: a ragged last chunk of 8 timesteps
    Case(4, 128, 512, (16, 8, 32)),            # RWARE tiny-4ag
]


def chunk_len(A):
    return int(L.lib().magpo_debug_retention_chunk_len(C.c_int(A)))


def geometry(T, A):
    lc = chunk_len(A)
    nch = -(-T // lc)
    return nch, T - (nch - 1) * lc, lc * A


def kappas():
    """(name, kappa as the kernel receives it): the library's default, decay_scaling_factor 0.5, and the slowest head decay of the
    general network, under which a state that is never reset builds up over the whole rollout."""
    return [("default", float(onets.NetCfg(2, 4, 4).kappas()[0])),
            ("scale0.5", float(onets.NetCfg(2, 4, 4, decay_scaling_factor=0.5).kappas()[0])),
            ("1-1/512", float(np.float32(1 - 1 / 512)))]


def test_chunk_geometry_and_case_coverage():
    """No GPU: the chunk length per agent count, that every case still has the geometry it is listed under (if RC_ROWS or the chunk
    rule changes, this names the cases that no longer test what they were written for), and that the test hook refuses what the
    kernels do not run before it touches a device."""
    assert [chunk_len(A) for A in range(1, 9)] == [32, 16, 10, 8, 6, 5, 4, 4]
    assert {A: (chunk_len(A), chunk_len(A) * A) for A in CHUNKS} == CHUNKS
    stale = [(c.id, c.expect, geometry(c.T, c.A)) for c in CASES if geometry(c.T, c.A) != c.expect]
    assert not stale, f"cases no longer on their listed chunk geometry (case, listed, actual): {stale}"
    assert {c.A for c in CASES} == set(range(1, 9))
    assert {c.expect[2] for c in CASES} >= {28, 30, 32}
    lib, nul = L.lib(), None
    for bwd in (0, 1):
        for A, ld, ldd in ((0, 256, 256), (9, 256, 256), (2, 258, 256), (2, 194, 256)) + (((2, 256, 254),) if bwd else ()):
            rc = lib.magpo_test_retention(nul, bwd, 4, 3, A, C.c_float(0.5), 1, nul, nul, nul, ld, nul, nul, nul, nul, nul, nul, nul,
                                          nul, nul, ldd)
            assert rc == L.ERR_UNSUPPORTED, (bwd, A, ld, ldd, rc)


# ----------------------------------------------------------------------------- inputs
def pattern_envs(N):
    """The env each done pattern is placed in: envs 0.. for a small batch, spread over the grid (the last env never done) for a large
    one."""
    if N < 16:
        return dict(zip(PATTERNS, range(N)))
    return {"first": 1, "last": N // 5, "pair": 2 * N // 5, "every": N // 2, "t0": 3 * N // 5 + 1, "never": N - 1}


def make_done(T, N, lc, rng):
    done = rng.random((T, N)) < 0.1
    t = np.arange(T)
    bounds = list(range(lc, T, lc)) or [T // 2]
    cols = {"first": t % lc == 0,
            "last": (t % lc == lc - 1) | (t == T - 1),
            "pair": np.isin(t, [b - 1 for b in bounds] + bounds),
            "every": np.ones(T, bool),
            "never": np.zeros(T, bool),
            "t0": t == 0}
    envs = pattern_envs(N)
    for p, n in envs.items():
        done[:, n] = cols[p]
    return done, envs


def sample_envs(N, envs, rng):
    """Every env of a small batch; of a large one env 0, env N - 1, every patterned env and 16 random envs (one CTA owns one env)."""
    if N <= 32:
        return np.arange(N)
    s = {0, N - 1} | set(envs.values()) | set(rng.choice(N, 16, replace=False).tolist())
    return np.array(sorted(s))


def env_major(x):
    """[T, S, A, ...] -> the oracle's [S, T * A, ...]"""
    T, S, A = x.shape[:3]
    return np.ascontiguousarray(np.swapaxes(x, 0, 1).reshape(S, T * A, *x.shape[3:]))


class Guarded:
    """`n` floats between two guard regions of `guard` floats: pointer() is the start of the body."""

    def __init__(self, n, guard, dev):
        self.n, self.g = n, guard
        self.buf = torch.empty(guard + n + guard, device=dev)

    @property
    def body(self):
        return self.buf[self.g:self.g + self.n]

    def pointer(self, off=0):
        return C.c_void_p(self.body.data_ptr() + 4 * off)

    def reset(self):
        self.buf.view(torch.int32).fill_(SENTINEL)
        self.body.fill_(float("nan"))

    def guards_intact(self):
        bits = self.buf.view(torch.int32)
        return bool((bits[:self.g] == SENTINEL).all()) and bool((bits[self.g + self.n:] == SENTINEL).all())


# ----------------------------------------------------------------------------- reference
def reference(q, k, v, h0, done, dret, kappa, A, lc, causal, dtype):
    """q, k, v, dret [S, T * A, 64], h0 [S, 64, 64], done [S, T]. ret and Hout from the oracle's chunkwise form, the gradients of
    sum(ret * dret) by autograd, and the checkpoints (state entering each chunk; for T = 1 the state after timestep 0, what the
    register scan saves) from the recurrence H_t = lam_t H_{t-1} + sum_i k_ti^T v_ti with lam_t = 0 where done_t."""
    S, T = done.shape
    qt, kt, vt = (torch.tensor(x, dtype=dtype, requires_grad=True) for x in (q, k, v))
    H0 = torch.tensor(h0, dtype=dtype)
    eye = {f"h/{w}": torch.eye(64, dtype=dtype) for w in ("w_q", "w_k", "w_v")}
    dn = torch.tensor(done)
    ret, nh = onets.simple_retention_chunk(eye, "h", kt, qt, vt, H0, dn.repeat_interleave(A, dim=1), kappa, A, causal)
    dq, dk, dv = torch.autograd.grad((ret * torch.tensor(dret, dtype=dtype)).sum(), [qt, kt, vt])
    kv = torch.einsum("stai,staj->stij", kt.detach().reshape(S, T, A, 64), vt.detach().reshape(S, T, A, 64))
    H, after = H0, []
    for t in range(T):
        H = torch.where(dn[:, t, None, None], torch.zeros((), dtype=dtype), H * kappa) + kv[:, t]
        after.append(H)
    ck = [after[0]] if T == 1 else [H0] + [after[ch * lc - 1] for ch in range(1, -(-T // lc))]
    out = dict(ret=ret, Hout=nh, Hck=torch.stack(ck, 1), dq=dq, dk=dk, dv=dv)
    return {n: x.detach().numpy() for n, x in out.items()}


def locate(name, d, s, sample, envs, done, A, lc):
    """Where the largest |cuda - f64| of output `name` lies in sampled env s: timestep, chunk, chunk-local token row and whether a
    done fell in that chunk."""
    env = int(sample[s])
    tag = f"env {env}" + "".join(f" ({p})" for p, n in envs.items() if n == env)
    i = np.unravel_index(d[s].argmax(), d[s].shape)
    if name == "Hout":
        return f"{tag} H[{i[0]}, {i[1]}]"
    if name == "Hck":
        ch = int(i[0])
        prev = bool(done[(ch - 1) * lc:ch * lc, env].any()) if ch else False
        return f"{tag} checkpoint {ch} H[{i[1]}, {i[2]}] (done in chunk {ch - 1}: {prev})"
    c = int(i[0])
    t, a = c // A, c % A
    ch = t // lc
    return (f"{tag} t={t} agent {a} col {i[1]}: chunk {ch}, chunk row {(t % lc) * A + a}, "
            f"done in chunk: {bool(done[ch * lc:(ch + 1) * lc, env].any())}")


# ----------------------------------------------------------------------------- the test
@pytest.mark.gpu
@pytest.mark.parametrize("causal", [False, True], ids=["encoder", "decoder"])
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_retention_matches_float64(dev, case, causal):
    A, T, N, ld = case.A, case.T, case.N, case.ld
    lc = chunk_len(A)
    nch, last, rows = geometry(T, A)
    assert (nch, last, rows) == case.expect
    seed = zlib.crc32(f"{case.id}-{causal}".encode())
    rng = np.random.default_rng(seed)
    g = torch.Generator(device=dev).manual_seed(seed)
    done, envs = make_done(T, N, lc, rng)
    sample = sample_envs(N, envs, rng)
    X = torch.randn(T, N, A, ld, generator=g, device=dev) * 0.5  # q | k | v at columns 0, 64, 128 of each row
    H0 = torch.randn(N, 64, 64, generator=g, device=dev) * 0.3 if case.h0 else None
    dret = torch.randn(T, N, A, 64, generator=g, device=dev)
    done_d = torch.as_tensor(done.astype(np.uint8)).to(dev)

    R = T * N * A
    ret, hout = Guarded(R * 64, 4096, dev), Guarded(N * 4096, 4096, dev)
    hck = Guarded(nch * N * 4096, N * 4096, dev)  # a whole checkpoint of guard past the last one the kernel may write
    grads = Guarded(R * 256, 4096, dev)
    gview = grads.body.view(R, 256)

    idx = torch.as_tensor(sample, device=dev)
    xs = X.index_select(1, idx).cpu().numpy()
    q, k, v = (env_major(xs[..., o:o + 64]) for o in (0, 64, 128))
    h0 = H0.index_select(0, idx).cpu().numpy() if case.h0 else np.zeros((len(sample), 64, 64), np.float32)
    dr = env_major(dret.index_select(1, idx).cpu().numpy())
    dn = np.ascontiguousarray(done[:, sample].T)

    branch = "register scan" if T == 1 else f"chunkwise, Lc={lc}, {nch} chunks, last {last} steps, {rows} of {RC_ROWS} rows real"
    print(f"\nA={A} T={T} N={N} ld={ld} H0={'random' if case.h0 else 'null'} {'decoder' if causal else 'encoder'}: {branch}; "
          f"{len(sample)} envs vs float64")
    p, s = L.ptr, L.stream_ptr()
    xb = X.data_ptr()
    fails = []
    for kname, kappa in kappas():
        for b in (ret, hout, hck, grads):
            b.reset()
        gview[:, 192:].view(torch.int32).fill_(SENTINEL)
        L.call("magpo_test_retention", s, 0, T, N, A, C.c_float(kappa), int(causal), C.c_void_p(xb), C.c_void_p(xb + 256),
               C.c_void_p(xb + 512), ld, p(H0), p(done_d), ret.pointer(), hck.pointer(), hout.pointer(), None, None, None, None, 0)
        L.call("magpo_test_retention", s, 1, T, N, A, C.c_float(kappa), int(causal), C.c_void_p(xb), C.c_void_p(xb + 256),
               C.c_void_p(xb + 512), ld, p(H0), p(done_d), None, hck.pointer(), None, p(dret), grads.pointer(0), grads.pointer(64),
               grads.pointer(128), 256)
        torch.cuda.synchronize()
        tag = f"kappa {kname}"

        # every output written, nothing written outside it: over all N envs
        for name, b in (("ret", ret), ("Hout", hout), ("Hck", hck), ("dq/dk/dv", grads)):
            if not b.guards_intact():
                fails.append(f"{tag}: {name} written outside its buffer" + (f" (past checkpoint {nch - 1})" if name == "Hck" else ""))
        for name, x in (("ret", ret.body), ("Hout", hout.body), ("Hck", hck.body), ("dq/dk/dv", gview[:, :192])):
            if not bool(torch.isfinite(x).all()):
                fails.append(f"{tag}: {name} not finite (an output row was not written)")
        if not bool((gview[:, 192:].view(torch.int32) == SENTINEL).all()):
            fails.append(f"{tag}: gradient columns 192..255 overwritten")

        gs = grads.body.view(T, N, A, 256).index_select(1, idx).cpu().numpy()
        got = dict(ret=env_major(ret.body.view(T, N, A, 64).index_select(1, idx).cpu().numpy()),
                   Hout=hout.body.view(N, 64, 64).index_select(0, idx).cpu().numpy(),
                   Hck=np.ascontiguousarray(np.swapaxes(hck.body.view(nch, N, 64, 64).index_select(1, idx).cpu().numpy(), 0, 1)),
                   dq=env_major(gs[..., 0:64]), dk=env_major(gs[..., 64:128]), dv=env_major(gs[..., 128:192]))
        r64 = reference(q, k, v, h0, dn, dr, kappa, A, lc, causal, torch.float64)
        r32 = reference(q, k, v, h0, dn, dr, kappa, A, lc, causal, torch.float32)
        line = []
        for name, fixed in FIXED.items():
            e, o = rel_err(got[name], r64[name]), rel_err(r32[name], r64[name])
            bound = max(fixed, 4 * o)
            # per env: an env with small values (reset at every step) must not hide behind the others
            en = np.array([rel_err(got[name][j], r64[name][j]) for j in range(len(sample))])
            bn = np.array([max(fixed, 4 * rel_err(r32[name][j], r64[name][j])) for j in range(len(sample))])
            w = int(np.argmax(en / bn))
            line.append(f"{name} {e:.1e}/{bound:.0e} (env {sample[w]} {en[w]:.1e}/{bn[w]:.0e})")
            if not (e <= bound and (en <= bn).all()):
                d = np.abs(got[name].astype(np.float64) - r64[name])
                worst = int(np.argmax([dj.max() for dj in d])) if not e <= bound else w
                err, bd = (e, bound) if not e <= bound else (en[w], bn[w])
                fails.append(f"{tag}: {name} {err:.3e} > {bd:.1e} at {locate(name, d, worst, sample, envs, done, A, lc)}")
        print(f"  {tag:16s} cuda vs f64 / bound: " + "  ".join(line[:3]) + "\n" + " " * 39 + "  ".join(line[3:]))
    assert not fails, f"A={A} T={T} N={N} ld={ld} {'decoder' if causal else 'encoder'}: " + "; ".join(fails)
