"""CPU: the RobotWarehouse restatement (oracle/rware.py) against hand-computed cases and generator invariants.
These pin the restatement, not a Jumanji run (parity unpinned, see the oracle's header)."""
import json
import os

import numpy as np
import pytest

from oracle import prng, rware


def _env(spec, seed=0):
    b = rware.base_reset(spec, prng.split(prng.prng_key(seed), 1))
    return {k: v[0].copy() for k, v in b.items()}


def _place(spec, e, agent, pos, direction, carry=False):
    x, y = e["agent_pos"][agent]
    e["grid"][1, x, y] = 0
    e["agent_pos"][agent] = pos
    e["grid"][1, pos[0], pos[1]] = agent + 1
    e["agent_dir"][agent] = direction
    e["agent_carry"][agent] = carry
    e["action_mask"] = rware._action_mask(spec, e["grid"], e["agent_pos"], e["agent_dir"], e["agent_carry"])


def test_layouts_and_scenarios_match_the_reference_configs():
    # the reference's mava/configs/env/scenario/*.yaml, as stored by tests/golden/make_golden.py --reference
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_configs.json")) as f:
        ref = json.load(f)["scenario"]
    for name, kw in rware.SCENARIOS.items():
        assert ref[name]["task_config"] == kw, name
    tiny, small = rware.RwareSpec(**rware.SCENARIOS["tiny-4ag"]), rware.RwareSpec(**rware.SCENARIOS["small-4ag"])
    assert tiny.grid_size == (11, 10) and len(tiny.shelf_cells) == 32 and tiny.obs_dim == 75 and tiny.goals == [(10, 4), (10, 5)]
    assert small.grid_size == (20, 10) and len(small.shelf_cells) == 80
    hw = tiny.highways
    assert hw[:, 0].all() and hw[:, 3].all() and hw[0].all() and hw[9].all() and hw[10].all() and hw[1:, 4:6].all()
    assert not hw[1:9, 1:3].any() and not hw[1:9, 7:9].any()


@pytest.mark.parametrize("scenario", ["tiny-4ag", "small-4ag", "medium-6ag"])
def test_generator_invariants(scenario):
    spec = rware.RwareSpec(**rware.SCENARIOS[scenario])
    H, W = spec.grid_size
    b = rware.base_reset(spec, prng.split(prng.prng_key(1), 100))
    S = len(spec.shelf_cells)
    assert ((b["grid"][:, 0] > 0).sum((1, 2)) == S).all() and ((b["grid"][:, 1] > 0).sum((1, 2)) == spec.num_agents).all()
    for e in range(100):
        assert len({tuple(p) for p in b["agent_pos"][e]}) == spec.num_agents
        assert len(set(b["request_queue"][e])) == spec.request_queue_size
        assert b["shelf_req"][e].sum() == spec.request_queue_size and b["shelf_req"][e][b["request_queue"][e]].all()
        for i, (x, y) in enumerate(b["agent_pos"][e]):
            assert b["grid"][e, 1, x, y] == i + 1
    assert ((b["agent_dir"] >= 0) & (b["agent_dir"] < 4)).all() and set(np.unique(b["agent_dir"])) == {0, 1, 2, 3}
    assert not b["agent_carry"].any() and (b["step_count"] == 0).all()
    assert b["action_mask"][:, :, [0, 2, 3, 4]].all()


def test_movement_load_and_delivery():
    spec = rware.RwareSpec(**rware.SCENARIOS["tiny-2ag"])
    e = _env(spec)
    _place(spec, e, 1, (0, 9), 0)  # out of the way, facing the wall
    assert not e["action_mask"][1, rware.FORWARD]
    # agent 0 under shelf at (1,1): pick it up, carry it down the column is blocked by the shelf at (2,1)
    _place(spec, e, 0, (1, 1), 2)
    sid = e["grid"][0, 1, 1]
    assert sid > 0
    e, r, done = rware._step_one(spec, e, np.array([rware.TOGGLE_LOAD, rware.NOOP]))
    assert e["agent_carry"][0] and r == 0 and not done and e["step_count"] == 1
    assert not e["action_mask"][0, rware.FORWARD]  # carrying and the next cell holds a shelf
    # a masked FORWARD is a NOOP
    e2, _, _ = rware._step_one(spec, e, np.array([rware.FORWARD, rware.NOOP]))
    assert e2["agent_pos"][0].tolist() == [1, 1]
    # turn LEFT from DOWN(2) -> RIGHT(1)... LEFT is dir - 1
    e, _, _ = rware._step_one(spec, e, np.array([rware.LEFT, rware.NOOP]))
    assert e["agent_dir"][0] == 1
    e, _, _ = rware._step_one(spec, e, np.array([rware.RIGHT, rware.NOOP]))
    e, _, _ = rware._step_one(spec, e, np.array([rware.RIGHT, rware.NOOP]))
    assert e["agent_dir"][0] == 3  # LEFT: towards the highway column 0
    e, _, _ = rware._step_one(spec, e, np.array([rware.FORWARD, rware.NOOP]))
    assert e["agent_pos"][0].tolist() == [1, 0] and e["grid"][0, 1, 0] == sid and e["grid"][0, 1, 1] == 0
    assert e["shelf_pos"][sid - 1].tolist() == [1, 0]
    # on a highway the shelf cannot be put down
    e, _, _ = rware._step_one(spec, e, np.array([rware.TOGGLE_LOAD, rware.NOOP]))
    assert e["agent_carry"][0]
    # delivery: requested shelf carried onto a goal cell -> reward 1, request replaced by a shelf that was not requested
    e["shelf_req"][:] = False
    e["shelf_req"][sid - 1] = True
    e["request_queue"][:] = [sid - 1, (sid + 5) % 32]
    e["shelf_req"][(sid + 5) % 32] = True
    e["grid"][0, 1, 0] = 0
    e["grid"][0, 9, 4] = sid
    e["shelf_pos"][sid - 1] = (9, 4)
    _place(spec, e, 0, (9, 4), 2, carry=True)
    key_before = e["key"].copy()
    e, r, done = rware._step_one(spec, e, np.array([rware.FORWARD, rware.NOOP]))
    assert r == 1.0 and not done and e["grid"][0, 10, 4] == sid
    assert not e["shelf_req"][sid - 1] and e["shelf_req"].sum() == 2
    new = [q for q in e["request_queue"] if q != (sid + 5) % 32]
    assert len(new) == 1 and new[0] != sid - 1 and e["shelf_req"][new[0]]
    assert (e["key"] == prng.split(key_before)[0]).all()
    # an un-requested shelf on the goal gives nothing
    e, r, _ = rware._step_one(spec, e, np.array([rware.NOOP, rware.NOOP]))
    assert r == 0


def test_collision_terminates_and_observation_layout():
    spec = rware.RwareSpec(**rware.SCENARIOS["tiny-2ag"])
    e = _env(spec)
    _place(spec, e, 0, (0, 4), 1)  # facing RIGHT towards (0,5)... agent 1 at (0,6) facing LEFT towards (0,5)
    _place(spec, e, 1, (0, 6), 3)
    assert e["action_mask"][:, rware.FORWARD].all()
    obs, _ = rware.observe(spec, {k: v[None] for k, v in e.items()})
    o = obs[0, 0]
    assert o[:8].tolist() == [0, 4, 0, 0, 1, 0, 0, 1]  # x, y, carrying, one_hot(RIGHT), on highway
    cells = o[8:].reshape(9, 7)
    assert not cells[:3].any()  # the row above the grid is padding
    assert cells[4].tolist() == [1, 0, 1, 0, 0, 0, 0]  # own cell: agent present, facing RIGHT, no shelf
    assert not cells[5].any() and not cells[3].any()
    e2, r, done = rware._step_one(spec, e, np.array([rware.FORWARD, rware.FORWARD]))
    assert done and e2["agent_pos"].tolist() == [[0, 5], [0, 5]]
    # through the wrapper stack: termination -> discount 0, auto-reset from split(state.key)[0]
    st = dict(env_state={k: v[None] for k, v in e.items()}, key=np.array([[3, 4]], np.uint32),
              running_count_episode_return=np.zeros(1, np.float32), running_count_episode_length=np.array([5], np.int32),
              episode_return=np.zeros(1, np.float32), episode_length=np.zeros(1, np.int32))
    nst, ts = rware.step(spec, st, np.array([[rware.FORWARD, rware.FORWARD]], np.int32))
    assert ts["step_type"][0] == rware.STEP_LAST and (ts["discount"][0] == 0).all()
    assert ts["extras"]["episode_metrics"]["episode_length"][0] == 6
    rb = rware.base_reset(spec, prng.split(e["key"])[:1])
    assert (rb["agent_pos"] == nst["env_state"]["agent_pos"]).all() and (nst["env_state"]["step_count"] == 0).all()
    # a shelf cell seen from below: shelf present + requested flag
    e = _env(spec)
    _place(spec, e, 1, (10, 9), 0)
    _place(spec, e, 0, (9, 1), 0)
    sid = e["grid"][0, 8, 1]
    e["shelf_req"][sid - 1] = True
    obs, _ = rware.observe(spec, {k: v[None] for k, v in e.items()})
    assert obs[0, 0, 8 + 7 * 1 + 5] == 1 and obs[0, 0, 8 + 7 * 1 + 6] == 1
