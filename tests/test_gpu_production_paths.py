"""The launch shapes the benchmark actually runs, against float64 references.

Two hot-path kernels pick their launch shape from the problem size:
  * the persistent GRU scans (csrc/gru_scan.cu) own 32, 64 or 128 rows per CTA depending on Rs = envs x agents
    (gru_rows_per_tile): the LBF benchmark chunk (4096 envs x 2 agents) runs 128, the RWARE shard (1024 x 4) 64;
  * the fused Sable rollout step (csrc/sable_step.cu) runs 1 or 2 envs per warp (EPW) and 6..8 warps per CTA; the benchmark's
    rollout (B = 2 slots x 4096 envs) is EPW = 2 with the sampler's gumbel rows wrapping at E = 4096.
The other parity tests run small batches, which only reach the 32-row tile and EPW = 1. Here every case first asserts (through the
host-only queries magpo_debug_gru_rows_per_tile / magpo_debug_step_plan, which call the functions the launches call) which branch it
covers, then compares the kernel with a float64 reference. The tolerance is max(fixed bound, 4 x the float32 CPU reference's own
deviation from float64), in the max-norm rel_err of gpu_util.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from magpo_b200 import _lib as L
from oracle import nets as onets
from oracle import prng as oprng

H = 128
F32_MIN = float(np.finfo(np.float32).min)

# (T, N, A) -> rows per tile. Rs = 2048 is the last 32-row size (64 CTAs), 4096 the RWARE shard at its rollout length, 8192 the LBF
# benchmark chunk; 2049 / 4097 / 8193 leave a last tile of one row.
GRU_CASES = [((33, 32, 2), 32), ((33, 1024, 2), 32), ((33, 683, 3), 64), ((128, 1024, 4), 64), ((33, 4097, 1), 128),
             ((128, 4096, 2), 128), ((17, 2731, 3), 128)]
# (B, A, d, a, gumbel_rows) -> envs per warp
STEP_CASES = [((2048, 2, 14, 6, 2048), 1),   # the last EPW = 1 size
              ((2049, 2, 14, 6, 2049), 2),   # the first EPW = 2 size: the last warp has one live env
              ((8192, 2, 14, 6, 4096), 2),   # the LBF benchmark rollout: two slots, gumbel rows wrap at E
              ((4099, 4, 75, 5, 4099), 2),   # RWARE tiny-4ag observations: the d > 16 template
              ((3001, 3, 4, 10, 3001), 2),   # the d <= 4 template
              ((2500, 1, 8, 32, 2500), 2)]   # A = 1, a = 32: every lane owns an action


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


def rows_per_tile(Rs):
    lib = L.lib()
    lib.magpo_debug_gru_rows_per_tile.restype = C.c_int
    return int(lib.magpo_debug_gru_rows_per_tile(C.c_int64(Rs)))


def step_plan(B):
    epw, warps = C.c_int32(), C.c_int32()
    L.call("magpo_debug_step_plan", C.c_int32(B), C.byref(epw), C.byref(warps))
    return epw.value, warps.value


def test_dispatch_boundaries_and_case_coverage():
    """No GPU: the thresholds of both launch heuristics, and that every case below still covers the branch it is listed under. If a
    threshold moves, this names the cases that no longer test the benchmark's branch."""
    assert [rows_per_tile(rs) for rs in (2048, 2049, 4096, 4097)] == [32, 64, 64, 128]
    assert step_plan(2048)[0] == 1 and step_plan(2049)[0] == 2
    stale = [(c, rpt, rows_per_tile(c[1] * c[2])) for c, rpt in GRU_CASES if rows_per_tile(c[1] * c[2]) != rpt]
    assert not stale, f"GRU cases no longer on their rows-per-tile branch (case, listed, actual): {stale}"
    assert {rpt for _, rpt in GRU_CASES} == {32, 64, 128}
    stale = [(c, epw, step_plan(c[0])[0]) for c, epw in STEP_CASES if step_plan(c[0])[0] != epw]
    assert not stale, f"step cases no longer on their envs-per-warp branch (case, listed, actual): {stale}"
    assert {step_plan(c[0])[0] for c, _ in STEP_CASES} == {1, 2}
    assert len({step_plan(c[0])[1] for c, _ in STEP_CASES}) >= 2
    # the GRU test hook refuses what the scans do not run (T = 1 is the stepwise path) before touching the device
    nul = L.ptr(None)
    assert L.lib().magpo_test_gru_scan(nul, 0, 1, 4, 2, *([nul] * 15)) == L.ERR_UNSUPPORTED


# ----------------------------------------------------------------------------- GRU scan forward + BPTT
def gru_reference(gi, Wh, bhn, done, h0, dY, dtype):
    """flax GRUCell over T steps, as oracle/nets.py:actor_apply and gru_gate_fwd_kernel: the carry is zeroed where done[t] is set,
    gh = hu @ Wh, r, z = sigmoid(gi + gh), n = tanh(gi_n + r (gh_n + bhn)), h = (1 - z) n + z hu. Rows are independent.
    gi [T, S, 384], done bool [T, S] (per row), h0 [S, 128], dY [T, S, 128] = dL/dY. Returns the forward tensors of the kernel
    (Y, HU [T+1], rzn, ghn) and dL/dgi, dL/dgh (gh = hu @ Wh, bias excluded) and dL/dWh."""
    gi = torch.tensor(gi, dtype=dtype, requires_grad=True)
    Wh = torch.tensor(Wh, dtype=dtype, requires_grad=True)
    bhn = torch.tensor(bhn, dtype=dtype)
    done = torch.tensor(done)[..., None]
    h = torch.tensor(h0, dtype=dtype)
    HU, Y, rzn, ghn, gh_all = [], [], [], [], []
    for t in range(gi.shape[0]):
        hu = torch.where(done[t], torch.zeros((), dtype=dtype), h)
        gh = hu @ Wh
        gh.retain_grad()
        r = torch.sigmoid(gi[t, :, :H] + gh[:, :H])
        z = torch.sigmoid(gi[t, :, H:2 * H] + gh[:, H:2 * H])
        gn = gh[:, 2 * H:] + bhn
        n = torch.tanh(gi[t, :, 2 * H:] + r * gn)
        h = (1.0 - z) * n + z * hu
        HU.append(hu)
        Y.append(h)
        rzn.append(torch.cat([r, z, n], -1))
        ghn.append(gn)
        gh_all.append(gh)
    HU.append(h)
    Yt = torch.stack(Y)
    (Yt * torch.tensor(dY, dtype=dtype)).sum().backward()
    out = dict(Y=Yt, HU=torch.stack(HU), rzn=torch.stack(rzn), ghn=torch.stack(ghn), dgi=gi.grad,
               dgh=torch.stack([g.grad for g in gh_all]), dWh=Wh.grad)
    return {k: v.detach().numpy() for k, v in out.items()}


def gru_sample_rows(Rs, rpt, rng):
    """Rows the float64 reference checks: the first and last row of every tile, the sub-partition (32-row) and 16x256b fragment
    (8 / 16-row) edges inside the first, a middle and the last tile, every row of the last tile, and 128 random rows."""
    ntiles = -(-Rs // rpt)
    rows = set()
    for tile in range(ntiles):
        rows.update((tile * rpt, min(tile * rpt + rpt, Rs) - 1))
    for tile in {0, ntiles // 2, ntiles - 1}:
        rows.update(tile * rpt + r for r in (1, 7, 8, 15, 16, 31, 32, 33, 63, 64, 65, 95, 96, 127) if r < rpt and tile * rpt + r < Rs)
    rows.update(range((ntiles - 1) * rpt, Rs))
    rows.update(rng.choice(Rs, min(Rs, 128), replace=False).tolist())
    return np.array(sorted(rows))


def gru_done(T, N, rng):
    done = rng.random((T, N)) < 0.1
    done[0, ::5] = True           # initial states reset at t = 0
    done[:, N // 2] = True        # one env reset at every step
    done[T - 1, 1::3] = True      # resets at the last step
    done[:, N - 1] = False        # the last env (the ragged tile) never reset...
    done[T // 2, N - 1] = True    # ... but once, mid-sequence
    return done


@pytest.mark.gpu
@pytest.mark.parametrize("case,rpt", GRU_CASES, ids=[f"Rs{c[1] * c[2]}-T{c[0]}-A{c[2]}" for c, _ in GRU_CASES])
def test_gru_scan_matches_float64(dev, case, rpt):
    T, N, A = case
    Rs = N * A
    assert rows_per_tile(Rs) == rpt
    rng = np.random.default_rng(Rs + T)
    g = torch.Generator(device=dev).manual_seed(Rs + T)
    scale = torch.ones(Rs, device=dev)
    scale[::5] = 6.0  # every fifth row's pre-activations saturate its gates
    gi = torch.randn(T, Rs, 3 * H, generator=g, device=dev) * scale[None, :, None]
    Wh = torch.randn(H, 3 * H, generator=g, device=dev) * 0.09
    bhn = torch.randn(H, generator=g, device=dev) * 0.3
    h0 = torch.randn(Rs, H, generator=g, device=dev) * 0.5
    dY = torch.randn(T, Rs, H, generator=g, device=dev)
    done = gru_done(T, N, rng)
    done_d = torch.as_tensor(done.astype(np.uint8)).to(dev)
    nan = lambda *s: torch.full(s, float("nan"), device=dev)  # noqa: E731  (an output row the kernel misses stays NaN)
    rzn, ghn, Y, HU = nan(T, Rs, 3 * H), nan(T, Rs, H), nan(T, Rs, H), nan(T + 1, Rs, H)
    dgi, dgh = nan(T, Rs, 3 * H), nan(T, Rs, 3 * H)
    dbi, dbhn = torch.zeros(3 * H, device=dev), torch.zeros(H, device=dev)
    scratch = torch.zeros(3 * H * 3 * H, device=dev)
    p, nul, s = L.ptr, L.ptr(None), L.stream_ptr()
    L.call("magpo_test_gru_scan", s, 0, T, N, A, p(gi), p(Wh), p(bhn), p(done_d), p(h0), nul, p(scratch), p(rzn), p(ghn), p(Y), p(HU),
           nul, nul, nul, nul)
    L.call("magpo_test_gru_scan", s, 1, T, N, A, p(gi), p(Wh), p(bhn), p(done_d), p(h0), p(dY), p(scratch), p(rzn), p(ghn), p(Y), p(HU),
           p(dgi), p(dgh), p(dbi), p(dbhn))
    torch.cuda.synchronize()

    rows = gru_sample_rows(Rs, rpt, rng)
    ri = torch.as_tensor(rows, device=dev)
    pick = lambda x: x.index_select(1, ri).cpu().numpy()  # noqa: E731
    got = dict(Y=pick(Y), HU=pick(HU), rzn=pick(rzn), ghn=pick(ghn), dgi=pick(dgi), dgh=pick(dgh))
    args = (pick(gi), Wh.cpu().numpy(), bhn.cpu().numpy(), done[:, rows // A], h0[ri].cpu().numpy(), pick(dY))
    r64, r32 = gru_reference(*args, torch.float64), gru_reference(*args, torch.float32)
    # W_h gradient over the sampled rows from the kernel's own saved carries and dgh: HU[:T]^T dgh
    got["dWh"] = np.einsum("tsk,tsj->kj", got["HU"][:T].astype(np.float64), got["dgh"].astype(np.float64))
    print(f"\nRs={Rs} T={T} A={A}: {rpt} rows per tile, {-(-Rs // rpt)} CTAs, {len(rows)} rows vs float64")
    fails = []
    for name, fixed in (("Y", 2e-5), ("HU", 2e-5), ("rzn", 2e-5), ("ghn", 2e-5), ("dgi", 5e-5), ("dgh", 5e-5), ("dWh", 5e-5)):
        assert np.isfinite(got[name]).all(), f"{name}: non-finite (an output row was not written)"
        e, o = rel_err(got[name], r64[name]), rel_err(r32[name], r64[name])
        bound = max(fixed, 4 * o)
        print(f"  {name:4s} cuda vs f64 {e:.2e}   f32 vs f64 {o:.2e}   bound {bound:.1e}")
        if e > bound:
            d = np.abs(got[name].astype(np.float64) - r64[name])
            if d.ndim == 3:  # where: (timestep, tile-local row) of the worst element
                t, s_, _ = np.unravel_index(d.argmax(), d.shape)
                where = f"t={t} row={rows[s_]} (tile row {rows[s_] % rpt}, env done at t: {bool(done[t, rows[s_] // A])})"
            else:
                where = ""
            fails.append(f"{name}: {e:.3e} > {bound:.1e} {where}")
    # the bias gradients the backward sums in shared memory and across CTAs, against float64 column sums of its own full dgi / dgh_n:
    # a float32 sum of n terms stays far inside 1e-5 of the sum of their magnitudes, a missing group of rows does not
    col, mag = torch.zeros(4 * H, dtype=torch.float64, device=dev), torch.zeros(4 * H, dtype=torch.float64, device=dev)
    for t in range(T):
        x = torch.cat([dgi[t], dgh[t, :, 2 * H:]], 1).double()
        col += x.sum(0)
        mag += x.abs().sum(0)
    sums = torch.cat([dbi, dbhn]).double()
    ratio = float(((sums - col).abs() / mag.clamp_min(1e-30)).max())
    print(f"  dbi/dbhn |kernel - f64 column sum| / column sum of |x|: {ratio:.2e} (bound 1e-5)")
    if not ratio <= 1e-5:
        fails.append(f"bias sums {ratio:.3e}")
    assert not fails, fails


# ----------------------------------------------------------------------------- fused rollout step
def setup_guider(A, d, a, dev, seed):
    """The default network (64, 1, 1) with every guider tensor moved off its init value (as test_gpu_networks.setup_nets)."""
    from magpo_b200.learner import NetworkConfig, load_params, param_table

    cfg = onets.NetCfg(A, d, a)
    rng = np.random.default_rng(seed + 7)
    gp = {k: (v + 0.05 * rng.standard_normal(v.shape)).astype(np.float32) for k, v in onets.init_guider_params(cfg, seed, ffn_zero=False).items()}
    net = NetworkConfig(A, d, a, 100)
    table, n = param_table(net, 0)
    flat = torch.zeros(n, device=dev)
    load_params(flat, table, gp)
    return cfg, net, gp, flat


def sample_keys(key, A):
    """discrete_autoregressive_act (decode.py:135-140): key, sample_key = split(key) per agent."""
    out = np.zeros((A, 2), np.uint32)
    for i in range(A):
        key, out[i] = oprng.split(key)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("case,epw", STEP_CASES, ids=[f"B{c[0]}-A{c[1]}-d{c[2]}-a{c[3]}-E{c[4]}" for c, _ in STEP_CASES])
def test_fused_rollout_step_matches_float64(dev, case, epw):
    B, A, d, a, E = case
    plan = step_plan(B)
    assert plan[0] == epw
    cfg, net, gp, gflat = setup_guider(A, d, a, dev, seed=B)
    rng = np.random.default_rng(B + A)
    obs = rng.integers(-1, 8, (B, A, d)).astype(np.float32)  # the LBF range: coordinates and levels, -1 where nothing is seen
    mask = rng.random((B, A, a)) < 0.6
    mask[np.arange(B)[:, None], np.arange(A)[None], rng.integers(0, a, (B, A))] = True  # at least one legal action
    mask[::13] = False
    mask[::13, :, 0] = True  # rows with a single legal action
    step = np.repeat(rng.integers(0, net.max_step_count + 1, (B, 1)), A, 1).astype(np.int32)
    step[:2] = [[0], [net.max_step_count]]
    hs = [(rng.standard_normal((B, *net.state_shape)) * 0.2).astype(np.float32) for _ in range(3)]
    prev_done = rng.random(B) < 0.2
    key = oprng.prng_key(B)
    sk = sample_keys(key, A)

    lib = L.lib()
    lib.magpo_rollout_workspace_bytes.restype = C.c_size_t
    nbytes = int(lib.magpo_rollout_workspace_bytes(C.byref(net.c_struct()), B, 1))
    ws = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
    to = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(dev)  # noqa: E731
    obs_d, mask_d, step_d, done_d = to(obs), to(mask.astype(np.uint8)), to(step), to(prev_done.astype(np.uint8))
    sk_d = to(sk.view(np.int32))

    def get_actions(full):
        st = {k: to(h) for k, h in zip(("encoder", "decoder_self", "decoder_cross"), hs)}
        act, logp = torch.full((B, A), -1, dtype=torch.int32, device=dev), torch.full((B, A), float("nan"), device=dev)
        value, logits = torch.full((B, A), float("nan"), device=dev), torch.full((B, A, a), float("nan"), device=dev)
        p = L.ptr if full else (lambda _: L.ptr(None))
        L.call("magpo_sable_get_actions", L.context(), L.stream_ptr(), C.byref(net.c_struct()), B, E, L.ptr(gflat), L.ptr(obs_d),
               L.ptr(mask_d), L.ptr(step_d), L.ptr(done_d), L.ptr(sk_d), L.struct_of(L.SableHState, **st), p(act), p(logp), L.ptr(value),
               p(logits), L.ptr(ws), C.c_size_t(nbytes))
        torch.cuda.synchronize()
        return act.cpu().numpy(), logp.cpu().numpy(), value.cpu().numpy(), logits.cpu().numpy(), [st[k].cpu().numpy() for k in st]

    act, logp, value, logits, states = get_actions(True)
    _, _, dry_value, _, dry_states = get_actions(False)

    # the reference, per block of E envs with the same keys (noise row b % E, as the rollout calls it), teacher-forced with the kernel's
    # actions so that agent i + 1's decoder sees the same previous action; the kernel's decay of 0 after a reset is a zero input state
    hs_in = [np.where(prev_done[:, None, None, None, None], np.float32(0), h) for h in hs]
    ref = {}
    for dt_ in (torch.float64, torch.float32):
        p_ = onets.to_torch(gp, dt_)
        parts = []
        for b0 in range(0, B, E):
            sl = slice(b0, min(b0 + E, B))
            _, lp_, v_, st_, lg_ = onets.sable_get_actions(p_, cfg, torch.tensor(obs[sl], dtype=dt_), torch.tensor(mask[sl]),
                                                           torch.tensor(step[sl]), tuple(torch.tensor(h[sl], dtype=dt_) for h in hs_in),
                                                           key, forced_actions=act[sl], return_logits=True)
            parts.append([lp_.numpy(), v_.numpy(), lg_.numpy()] + [s_.numpy() for s_ in st_])
        ref[dt_] = [np.concatenate(x) for x in zip(*parts)]
    r64, r32 = ref[torch.float64], ref[torch.float32]

    print(f"\nB={B} A={A} d={d} a={a} gumbel_rows={E}: {plan[0]} envs per warp, {plan[1]} warps per CTA")
    fails = []
    legal = mask
    names = ("log_prob", "value", "logits", "encoder", "decoder_self", "decoder_cross", "value (dry)")
    for name, got, i in zip(names, [logp, value, logits[legal]] + states + [dry_value], (0, 1, 2, 3, 4, 5, 1)):
        r, o = r64[i], r32[i]
        if name == "logits":
            r, o = r[legal], o[legal]
        e, y = rel_err(got, r), rel_err(o, r)
        bound = max(1e-4, 4 * y)
        print(f"  {name:14s} cuda vs f64 {e:.2e}   f32 vs f64 {y:.2e}   bound {bound:.1e}")
        if not e <= bound:
            row = np.unravel_index(np.abs(got - r).argmax(), got.shape)[0] if name != "logits" else None
            fails.append(f"{name}: {e:.3e} > {bound:.1e}" + (f" worst env {row} (warp env {row % epw})" if row is not None else ""))
    if not (logits[~legal] == F32_MIN).all():
        fails.append("illegal logits are not finfo(float32).min")
    for name, before, after in zip(("encoder", "decoder_self", "decoder_cross"), hs, dry_states):
        if not np.array_equal(before, after):
            fails.append(f"dry run changed the {name} state")

    # sampling: argmax of gumbel + log-softmax with the noise of the same keys, row b reading noise row b % E
    norm = torch.log_softmax(torch.tensor(r64[2]), -1).numpy()
    exempt, same = 0, 0
    for i in range(A):
        g = oprng.gumbel(sk[i], (1, E, 1, a)).reshape(E, a).astype(np.float64)
        score = g[np.arange(B) % E] + norm[:, i]
        top2 = np.argsort(-score, axis=1, kind="stable")[:, :2]
        gap = score[np.arange(B), top2[:, 0]] - score[np.arange(B), top2[:, 1]]
        bad = act[:, i] != top2[:, 0]
        tie = bad & (gap < 1e-5) & (act[:, i] == top2[:, 1])
        exempt += int(tie.sum())
        same += int((~bad).sum())
        if (bad & ~tie).any():
            b = int(np.flatnonzero(bad & ~tie)[0])
            fails.append(f"agent {i}: {int((bad & ~tie).sum())} sampled actions differ, first env {b} (warp env {b % epw}, noise row {b % E}): "
                         f"kernel {act[b, i]} reference {top2[b, 0]} gap {gap[b]:.2e}")
    print(f"  sampled actions: {same} / {B * A} equal the float64 argmax, {exempt} near-ties (gap < 1e-5) exempted")
    if not exempt < 1e-3 * B * A:
        fails.append(f"{exempt} near-tie exemptions")
    assert not fails, fails
