"""GPU tier of the closed-loop rollouts (DummySimulator.rollout,
pp2d_sim_rollout_mdp*, DESIGN.md section 7): trajectories, statistics and
final beliefs bit for bit against the CPU oracle (tests/rollout_oracle.c), a
replay through the filter and plan entry points that needs no oracle, the
sampling law measured on the device, independence from the other episodes of
a call, both belief placements (shared memory and global memory), and the
argument and state rules."""
import ctypes

import numpy as np
import pytest

import cases
import rollout_oracle_py as ro
from path_planning_2d_b200 import DummySimulator, MdpBatchPathPlanning2d, MdpPathPlanning2d, _lib

pytestmark = pytest.mark.gpu
GAMMA = cases.GAMMA
MAPS = ["map_3x3", "map_10x10", "map_100x40", "sparse_map_100x40"]
KEYS = ["steps", "reached", "collisions", "final_cell"]
REC = KEYS + ["final_belief", "cells", "actions", "measurements"]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _same(got, want, keys=REC):
    for k in keys:
        g, w = np.asarray(got[k]), np.asarray(want[k])
        if g.dtype == np.float32:
            g, w = _bits(g), _bits(w)
        assert np.array_equal(g, w), k


def _goal(name):
    return (95, 34) if "100x40" in name else cases.BUNDLED[name][0]


def _free_starts(grid, n, seed):
    ys, xs = np.nonzero(grid == 0)
    pick = np.random.default_rng(seed).integers(len(xs), size=n)
    return np.stack([xs[pick], ys[pick]], axis=1).astype(np.uint32)


def _uniform_free(grid, n):
    free = (grid.reshape(-1) == 0).astype(np.float32)
    return np.broadcast_to(free / free.sum(dtype=np.float32), (n, grid.size)).copy()


def _max_steps(grid):
    return 120 if grid.size > 1000 else 30


@pytest.mark.parametrize("belief", ["point", "uniform"])
@pytest.mark.parametrize("name", MAPS)
def test_single_handle_equals_the_oracle(name, belief):
    grid = cases.load_bundled(name)
    goal = _goal(name)
    n = 24
    starts = _free_starts(grid, n, seed=len(name))
    beliefs = _uniform_free(grid, n) if belief == "uniform" else None
    steps = _max_steps(grid)
    with MdpPathPlanning2d(grid, goal, GAMMA) as mdp, DummySimulator(grid) as sim:
        mdp.valueIteration()
        _, act = mdp.download()
        got = sim.rollout(mdp, starts, steps, seed=11, beliefs=beliefs, first_episode=3,
                          record=True)
    want = ro.rollout(grid, act, goal, starts, steps, 11, first_episode=3, beliefs=beliefs)
    _same(got, want)
    if "100x40" in name:
        assert got["reached"].sum() > 0


@pytest.mark.parametrize("belief", ["point", "uniform"])
@pytest.mark.parametrize("name", MAPS)
def test_batch_one_goal_per_instance_equals_the_oracle(name, belief):
    grid = cases.load_bundled(name)
    K = 6
    goals = _free_starts(grid, K, seed=99)
    goals[0] = _goal(name)
    n = 18
    inst = np.arange(n, dtype=np.uint32) % K
    starts = _free_starts(grid, n, seed=7)
    beliefs = _uniform_free(grid, n) if belief == "uniform" else None
    steps = _max_steps(grid)
    with MdpBatchPathPlanning2d(grid, goals, GAMMA) as b, DummySimulator(grid) as sim:
        b.valueIteration()
        _, act = b.download()
        got = sim.rollout(b, starts, steps, seed=2**40 + 5, beliefs=beliefs, instances=inst,
                          record=True)
    want = ro.rollout(grid, act[inst], goals[inst], starts, steps, 2**40 + 5, beliefs=beliefs)
    _same(got, want)


def _replay(sim, plan, starts, res, hw, beliefs=None):
    """Recorded actions and measurements through updateBelief and the plan
    entry point: the same beliefs and the same actions."""
    n = len(starts)
    W = sim.map_width
    if beliefs is None:
        bel = np.zeros((n, hw), np.float32)
        bel[np.arange(n), starts[:, 1] * W + starts[:, 0]] = 1.0
    else:
        bel = beliefs.copy()
    for t in range(int(res["steps"].max())):
        live = np.nonzero(res["steps"] > t)[0]
        a = plan(live, bel[live])
        assert np.array_equal(a, res["actions"][live, t]), t
        m = res["measurements"][live, t]
        meas = ((m[:, None] >> np.arange(4, dtype=np.uint8)) & 1).astype(np.uint8)
        bel[live] = sim.updateBelief(bel[live], action=a, measurement=meas)
    assert np.array_equal(_bits(bel), _bits(res["final_belief"]))


def _staggered():
    """Four empty maps, whose instances stop early, and one with a wall, whose
    occupied cells keep its residual up (test_mdp_batch_gpu's staggered
    batch); the world is the walled map."""
    h, w = 30, 100
    world = np.zeros((h, w), np.uint8)
    world[5:25, 30] = 1
    maps = np.stack([np.zeros((h, w), np.uint8)] * 4 + [world])
    goals = np.array([(w // 2 + 3 * i, h // 2) for i in range(4)] + [(2, 2)], np.uint32)
    return world, maps, goals


def test_replay_through_filter_and_plan_matches_frozen_snapshots():
    world, maps, goals = _staggered()
    K = len(goals)
    n = 40
    inst = np.arange(n, dtype=np.uint32) % K
    starts = _free_starts(world, n, seed=3)
    with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b, DummySimulator(world) as sim:
        sweeps, _ = b.valueIteration()
        assert len(set(int(v) for v in sweeps)) >= 2, sweeps
        res = sim.rollout(b, starts, 80, seed=5, instances=inst, record=True)
        assert res["reached"].sum() > 0
        _replay(sim, lambda live, bel: b.plan_batch(inst[live], bel), starts, res, world.size)
        _, act = b.download()
    _same(res, ro.rollout(world, act[inst], goals[inst], starts, 80, 5))


def test_replay_single_handle_on_map_100x40():
    grid = cases.load_bundled("map_100x40")
    starts = _free_starts(grid, 64, seed=21)
    beliefs = _uniform_free(grid, 64)
    with MdpPathPlanning2d(grid, (95, 34), GAMMA) as mdp, DummySimulator(grid) as sim:
        mdp.valueIteration()
        res = sim.rollout(mdp, starts, 150, seed=9, beliefs=beliefs, record=True)
        _replay(sim, lambda live, bel: mdp.plan_batch(bel), starts, res, grid.size, beliefs)


def _one_step(grid, goal, n, seed):
    """One step of n episodes from random free starts (the goal excluded)."""
    h, w = grid.shape
    ys, xs = np.nonzero((grid == 0) & ~((np.arange(w)[None, :] == goal[0]) &
                                        (np.arange(h)[:, None] == goal[1])))
    pick = np.random.default_rng(seed).integers(len(xs), size=n)
    starts = np.stack([xs[pick], ys[pick]], axis=1).astype(np.uint32)
    with MdpPathPlanning2d(grid, goal, GAMMA) as mdp, DummySimulator(grid) as sim:
        mdp.valueIteration()
        res = sim.rollout(mdp, starts, 1, seed=seed, record=True)
    assert np.all(res["steps"] == 1)
    return starts[:, 0].astype(int), starts[:, 1].astype(int), res


def test_sampling_law_on_an_open_map():
    """One step of 2^18 episodes on an open map, starts off the border so that
    nothing blocks: the device's move gives the slot, whose frequencies per
    action are within 5 sigma of 0.7 / 0.1; the sensor readings differ from
    the truth at the new cell at a rate within 5 sigma of 0.02."""
    h = w = 64
    grid = np.zeros((h, w), np.uint8)
    n = 1 << 18
    goal = (32, 32)
    ys, xs = np.mgrid[1:h - 1, 1:w - 1]
    sx0, sy0 = xs.reshape(-1), ys.reshape(-1)
    keep = ~((sx0 == goal[0]) & (sy0 == goal[1]))
    sx0, sy0 = sx0[keep], sy0[keep]
    pick = np.random.default_rng(1).integers(len(sx0), size=n)
    starts = np.stack([sx0[pick], sy0[pick]], axis=1).astype(np.uint32)
    with MdpPathPlanning2d(grid, goal, GAMMA) as mdp, DummySimulator(grid) as sim:
        mdp.valueIteration()
        res = sim.rollout(mdp, starts, 1, seed=2024, record=True)
    sx, sy = starts[:, 0].astype(int), starts[:, 1].astype(int)
    assert np.all(res["collisions"] == 0)
    fx, fy = res["cells"][:, 1] % w, res["cells"][:, 1] // w
    slot = (fy.astype(int) - sy + 1) * 3 + (fx.astype(int) - sx + 1)
    acts = res["actions"][:, 0]
    seen = 0
    for u in range(9):
        sel = acts == u
        m = int(sel.sum())
        if m < 2000:
            continue
        seen += 1
        freq = np.bincount(slot[sel], minlength=9) / m
        for i in range(9):
            p = float(ro.NAIVE[u, i])
            assert abs(freq[i] - p) <= 5 * np.sqrt(p * (1 - p) / m) + 1e-12, (u, i, freq[i])
    assert seen >= 4
    truth = np.zeros(n, np.uint8)
    for j, (ox, oy) in enumerate([(0, -1), (-1, 0), (1, 0), (0, 1)]):
        mx, my = fx.astype(int) + ox, fy.astype(int) + oy
        out = (mx < 0) | (mx >= w) | (my < 0) | (my >= h)
        truth |= out.astype(np.uint8) << j
    flips = np.unpackbits((res["measurements"][:, 0] ^ truth)[:, None], axis=1).sum()
    rate = flips / (4 * n)
    assert abs(rate - 0.02) <= 5 * np.sqrt(0.02 * 0.98 / (4 * n)), rate


def test_collisions_exactly_where_the_target_is_blocked():
    """Slots drawn by the numpy Philox and sampler from the recorded action:
    a collision exactly when the target is outside or occupied, and the robot
    stays there and moves by the slot elsewhere."""
    grid, goal = cases.synthetic_map(48, 48, 0.3, seed=17, goal=(24, 24))
    h, w = grid.shape
    n = 1 << 16
    sx, sy, res = _one_step(grid, goal, n, seed=606)
    r = ro.step_uniforms_np(606, np.arange(n, dtype=np.uint64), 0)
    slot = ro.motion_slots_np(res["actions"][:, 0], r[:, 0])
    tx, ty = sx + slot % 3 - 1, sy + slot // 3 - 1
    out = (tx < 0) | (tx >= w) | (ty < 0) | (ty >= h)
    occ = grid[np.clip(ty, 0, h - 1), np.clip(tx, 0, w - 1)] > 0
    blocked = (slot != 4) & (out | occ)
    assert blocked.sum() > 1000
    assert np.array_equal(res["collisions"], blocked.astype(np.uint32))
    fx, fy = np.where(blocked, sx, tx), np.where(blocked, sy, ty)
    assert np.array_equal(res["final_cell"], (fy * w + fx).astype(np.uint32))


def test_episodes_do_not_depend_on_the_rest_of_the_call():
    grid = cases.load_bundled("sparse_map_100x40")
    N = 64
    starts = _free_starts(grid, N, seed=4)
    with MdpPathPlanning2d(grid, (95, 34), GAMMA) as mdp, DummySimulator(grid) as sim:
        mdp.valueIteration()
        whole = sim.rollout(mdp, starts, 100, seed=77, record=True)
        a = sim.rollout(mdp, starts[:N // 2], 100, seed=77, record=True)
        b = sim.rollout(mdp, starts[N // 2:], 100, seed=77, first_episode=N // 2, record=True)
        for k in REC:
            assert np.array_equal(np.concatenate([a[k], b[k]]).view(np.uint8),
                                  np.asarray(whole[k]).view(np.uint8)), k
        pick = np.random.default_rng(0).permutation(N)[:20]
        # one call per episode id: first_episode carries the id
        for i in pick[:5]:
            one = sim.rollout(mdp, starts[i:i + 1], 100, seed=77, first_episode=int(i),
                              record=True)
            for k in REC:
                assert np.array_equal(np.asarray(one[k])[:1].view(np.uint8),
                                      np.asarray(whole[k])[i:i + 1].view(np.uint8)), k
        # a shuffled subset through a batch whose instance 0 is the same planner
        with MdpBatchPathPlanning2d(grid, [(95, 34)], GAMMA) as bt:
            bt.valueIteration()
            _, act_b = bt.download()
            _, act_s = mdp.download()
            assert np.array_equal(act_b[0], act_s)
            # ids travel with the episodes: each call below is one episode,
            # so shuffle by calling in permuted order with matching ids
            res = [sim.rollout(bt, starts[i:i + 1], 100, seed=77, instances=[0],
                               first_episode=int(i)) for i in pick]
            for j, i in enumerate(pick):
                for k in KEYS:
                    assert np.array_equal(res[j][k][0], whole[k][i]), k


def test_world_map_differs_from_the_planner_map():
    plan_map = cases.load_bundled("map_100x40")
    world = plan_map.copy()
    rng = np.random.default_rng(8)
    ys, xs = np.nonzero(world == 0)
    pick = rng.choice(len(xs), 150, replace=False)
    world[ys[pick], xs[pick]] = 1
    world[34, 95] = 0
    starts = _free_starts(world, 20, seed=6)
    with MdpPathPlanning2d(plan_map, (95, 34), GAMMA) as mdp, DummySimulator(world) as sim:
        mdp.valueIteration()
        _, act = mdp.download()
        got = sim.rollout(mdp, starts, 120, seed=3, record=True)
    _same(got, ro.rollout(world, act, (95, 34), starts, 120, 3))
    assert got["collisions"].sum() > 0


@pytest.mark.parametrize("belief", ["point", "uniform"])
def test_map_beyond_shared_memory_equals_the_oracle(belief):
    """200 x 200 = 40000 cells: two planes need 320 KB, more than a CTA's
    shared memory, so the belief lives in global memory."""
    grid, goal = cases.synthetic_map(200, 200, 0.15, seed=31, goal=(150, 120))
    n = 4
    starts = _free_starts(grid, n, seed=2)
    near = np.argwhere(grid[118:123, 146:150] == 0)[0]      # a free cell next to the goal
    starts[0] = (146 + near[1], 118 + near[0])
    beliefs = _uniform_free(grid, n) if belief == "uniform" else None
    with MdpPathPlanning2d(grid, goal, GAMMA) as mdp, DummySimulator(grid) as sim:
        mdp.sweeps(300)
        _, act = mdp.download()
        got = sim.rollout(mdp, starts, 12, seed=19, beliefs=beliefs, record=True)
    _same(got, ro.rollout(grid, act, goal, starts, 12, 19, beliefs=beliefs))


def test_edges():
    grid = cases.load_bundled("map_10x10")
    goal = cases.BUNDLED["map_10x10"][0]
    with MdpPathPlanning2d(grid, goal, GAMMA) as mdp, DummySimulator(grid) as sim:
        mdp.valueIteration()
        r = sim.rollout(mdp, [goal], 10, seed=1, record=True)
        assert r["steps"][0] == 0 and r["reached"][0] == 1
        assert r["final_cell"][0] == goal[1] * 10 + goal[0]
        assert r["cells"][0, 0] == goal[1] * 10 + goal[0]
        start = cases.BUNDLED["map_10x10"][1]
        r = sim.rollout(mdp, [start], 0, seed=1, record=True)
        assert r["steps"][0] == 0 and r["reached"][0] == 0
        assert r["final_belief"][0, start[1] * 10 + start[0]] == 1.0
        r = sim.rollout(mdp, np.zeros((0, 2), np.uint32), 10, seed=1, record=True)
        assert r["steps"].size == 0


def _rc(fn, *args):
    out = _lib.Rollout()
    return fn(*args, ctypes.byref(out))


def test_argument_and_state_errors():
    lib = _lib.load()
    grid = cases.load_bundled("map_10x10")
    goal = cases.BUNDLED["map_10x10"][0]
    free = np.argwhere(grid == 0)[0][::-1].astype(np.uint32)
    occ = np.argwhere(grid > 0)[0][::-1].astype(np.uint32)
    starts = np.stack([free, free, occ]).astype(np.uint32)
    with MdpPathPlanning2d(grid, goal, GAMMA) as mdp, DummySimulator(grid) as sim, \
            DummySimulator(np.zeros((5, 10), np.uint8)) as small, \
            MdpBatchPathPlanning2d(grid, [goal, goal], GAMMA) as bt, \
            MdpPathPlanning2d(grid, goal, GAMMA, rows=(0, 5)) as shard:
        f, fb = lib.pp2d_sim_rollout_mdp, lib.pp2d_sim_rollout_mdp_batch
        assert _rc(f, sim._h, mdp._h, 3, starts.ctypes.data, None, 5, 1, 0) == \
            _lib.PP2D_ERR_INVALID
        assert b"episode 2" in lib.pp2d_last_error()
        outside = np.array([[10, 0]], np.uint32)
        assert _rc(f, sim._h, mdp._h, 1, outside.ctypes.data, None, 5, 1, 0) == \
            _lib.PP2D_ERR_INVALID
        assert b"episode 0" in lib.pp2d_last_error()
        assert _rc(f, sim._h, mdp._h, 1, None, None, 5, 1, 0) == _lib.PP2D_ERR_INVALID
        assert _rc(f, None, mdp._h, 1, starts.ctypes.data, None, 5, 1, 0) == \
            _lib.PP2D_ERR_INVALID
        assert _rc(f, small._h, mdp._h, 1, starts.ctypes.data, None, 5, 1, 0) == \
            _lib.PP2D_ERR_INVALID
        assert _rc(f, sim._h, shard._h, 1, starts.ctypes.data, None, 5, 1, 0) == \
            _lib.PP2D_ERR_STATE
        inst = np.array([0, 2], np.uint32)
        assert _rc(fb, sim._h, bt._h, inst.ctypes.data, 2, starts.ctypes.data, None, 5, 1, 0) \
            == _lib.PP2D_ERR_INVALID
        assert b"episode 1" in lib.pp2d_last_error()
        assert _rc(fb, sim._h, bt._h, None, 1, starts.ctypes.data, None, 5, 1, 0) == \
            _lib.PP2D_ERR_INVALID
        assert _rc(f, sim._h, mdp._h, 0, None, None, 5, 1, 0) == _lib.PP2D_OK
        with pytest.raises(ValueError):
            sim.rollout(bt, [free], 5, seed=1)
    try:
        multi = MdpPathPlanning2d(grid, goal, GAMMA, devices=1)
    except _lib.Pp2dError:
        return
    with multi, DummySimulator(grid) as sim:
        assert _rc(lib.pp2d_sim_rollout_mdp, sim._h, multi._h, 1, starts.ctypes.data, None, 5,
                   1, 0) == _lib.PP2D_ERR_STATE
