"""GPU tier of the closed-loop episodes of the QV-tree planner
(DummySimulator.rollout with a PomdpPathPlanning2d, pp2d_sim_rollout_pomdp,
DESIGN.md section 7d): trajectories, actions, measurements, statistics and
final beliefs bit for bit against a CPU loop of the oracle's tree and the
rollouts' Philox and motion helpers, the same episodes through a host loop of
SearchTree handles, independence from how the episodes are split into calls,
a replay of the recorded world steps through the numpy Philox helpers, the
reference's own SearchTree fed one episode's (a, z) sequence, and the argument
rules."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import cases
import pomdp_fixtures as pf
import pomdp_oracle_py as po
import rollout_oracle_py as ro
from path_planning_2d_b200 import DummySimulator, PomdpPathPlanning2d, SearchTree, _lib

pytestmark = pytest.mark.gpu
GAMMA = cases.GAMMA
REC = ["steps", "reached", "collisions", "final_cell", "cells", "actions", "measurements"]
REF_SO = os.path.join(cases.ROOT, "oracle", "_ref", "libpp2d_ref_pomdp_full.so")
# name -> goal, PBVI vectors, episodes, steps, depth cap, expansions per step
CASES = {"map_10x10": ((8, 7), 20, 8, 30, 50, 4),
         "sparse_map_100x40": ((95, 34), 40, 4, 20, 50, 3)}


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same(got, want, keys):
    for k in keys:
        g, w = np.asarray(got[k]), np.asarray(want[k])
        if g.dtype == np.float32:
            g, w = bits(g), bits(w)
        assert np.array_equal(g, w), k


def world_step(world, cell, u, seed, e, t):
    """DESIGN.md section 7c's motion and sensors from the oracle's Philox and
    motion-slot helpers."""
    h, w = world.shape
    r = ro.step_uniforms(seed, e, t)
    slot = ro.motion_slot(u, r[0])
    x, y = cell % w, cell // w
    coll = 0
    if slot != 4:
        tx, ty = x + slot % 3 - 1, y + slot // 3 - 1
        if tx < 0 or tx >= w or ty < 0 or ty >= h or world[ty, tx] > 0:
            coll = 1
        else:
            x, y = tx, ty
    m = 0
    for j, (dx, dy) in enumerate(((0, -1), (-1, 0), (1, 0), (0, 1))):
        mx, my = x + dx, y + dy
        v = 1 if (mx < 0 or mx >= w or my < 0 or my >= h) else int(world[my, mx] > 0)
        if r[1 + j] < np.float32(0.02):
            v ^= 1
        m |= v << j
    return int(y * w + x), m, coll


def loop(make_tree, world, goal, starts, b0, max_steps, d, it, seed, first=0, model=None):
    """The episodes on the host: make_tree(belief) -> object with plan(d, it)
    -> (a, ...) and update(a, z); the root belief follows the Bayes updates of
    `model` (the oracle's) when given."""
    h, w = world.shape
    n = len(starts)
    out = {"steps": np.zeros(n, np.uint32), "reached": np.zeros(n, np.uint8),
           "collisions": np.zeros(n, np.uint32), "final_cell": np.zeros(n, np.uint32),
           "cells": np.zeros((n, max_steps + 1), np.uint32),
           "actions": np.zeros((n, max_steps), np.uint8),
           "measurements": np.zeros((n, max_steps), np.uint8),
           "final_belief": np.array(b0, np.float32, copy=True)}
    g = goal[1] * w + goal[0]
    for i in range(n):
        cell = int(starts[i, 1]) * w + int(starts[i, 0])
        out["cells"][i, 0] = cell
        tree = make_tree(b0[i])
        bel = out["final_belief"][i]
        t = 0
        while cell != g and t < max_steps:
            a = int(tree.plan(d, it)[0])
            cell, z, c = world_step(world, cell, a, seed, first + i, t)
            assert tree.update(a, z) in (0, None)
            if model is not None:
                bel, _ = model.bayes(bel, a, z, normalize=True)
            out["collisions"][i] += c
            out["cells"][i, t + 1] = cell
            out["actions"][i, t] = a
            out["measurements"][i, t] = z
            t += 1
        out["final_belief"][i] = bel
        out["steps"][i] = t
        out["reached"][i] = cell == g
        out["final_cell"][i] = cell
        if hasattr(tree, "close"):
            tree.close()
    return out


def setup(name):
    goal, n_pbvi, n, steps, d, it = CASES[name]
    grid = cases.load_bundled(name)
    m, fib, pbvi, fa, pa = pf.alphas(name, goal, n_pbvi=n_pbvi)
    free = np.argwhere(grid == 0)
    free = free[(free[:, 0] != goal[1]) | (free[:, 1] != goal[0])]
    pick = np.random.default_rng(len(name)).choice(len(free), size=n + 3, replace=False)
    starts = free[pick[:n]][:, ::-1].astype(np.uint32)
    # the world: the planner's map with three more obstacles
    world = grid.copy()
    for y, x in free[pick[n:]]:
        world[y, x] = 1
    return grid, world, goal, (m, fib, pbvi, fa, pa), starts, steps, d, it


@pytest.mark.parametrize("belief", ["point", "given"])
@pytest.mark.parametrize("name", list(CASES))
def test_episodes_equal_the_oracle_loop_and_single_trees(name, belief):
    grid, world, goal, (m, fib, pbvi, fa, pa), starts, steps, d, it = setup(name)
    n = len(starts)
    if belief == "point":
        b0 = np.zeros((n, grid.size), np.float32)
        b0[np.arange(n), starts[:, 1] * grid.shape[1] + starts[:, 0]] = 1
        given = None
    else:
        b0 = given = pf.gaussian_beliefs(grid, n, sigma=1.5, seed=5)
    seed = 2**33 + 9
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p, DummySimulator(world) as sim:
        p.set_alphas(fib, pbvi, fa, pa)
        got = sim.rollout(p, starts, steps, seed, beliefs=given, first_episode=5, record=True,
                          max_depth=d, max_iter=it)
        # one call per episode, and two calls split unevenly: the same episodes
        for i in range(n):
            one = sim.rollout(p, starts[i:i + 1], steps, seed, beliefs=None if given is None
                              else given[i:i + 1], first_episode=5 + i, record=True,
                              max_depth=d, max_iter=it)
            same({k: v[i:i + 1] for k, v in got.items()}, one, REC + ["final_belief"])
        k = n // 3 + 1
        parts = [sim.rollout(p, starts[s], steps, seed,
                             beliefs=None if given is None else given[s],
                             first_episode=5 + s.start, record=True, max_depth=d, max_iter=it)
                 for s in (slice(0, k), slice(k, n))]
        same({key: np.concatenate([q[key] for q in parts]) for key in got}, got,
             REC + ["final_belief"])
        host = loop(lambda b: SearchTree(p, b), world, goal, starts, b0, steps, d, it, seed, 5)
    same(got, host, REC)
    oracle = loop(lambda b: po.Tree(m, GAMMA, fib, pbvi, pf.uniforms(), b, fa, pa), world, goal,
                  starts, b0, steps, d, it, seed, 5, model=m)
    same(got, oracle, REC + ["final_belief"])
    assert got["steps"].sum() > n                 # the episodes move
    # the recorded world steps through the numpy Philox helpers
    W = grid.shape[1]
    for t in range(int(got["steps"].max())):
        live = np.nonzero(got["steps"] > t)[0]
        r = ro.step_uniforms_np(seed, 5 + live, t)
        slot = ro.motion_slots_np(got["actions"][live, t], r[:, 0])
        c = got["cells"][live, t].astype(np.int64)
        tx, ty = c % W + slot % 3 - 1, c // W + slot // 3 - 1
        inside = (tx >= 0) & (tx < W) & (ty >= 0) & (ty < grid.shape[0])
        ok = (slot != 4) & inside
        ok[ok] = world[ty[ok], tx[ok]] == 0
        nxt = np.where(ok, ty * W + tx, c)
        assert np.array_equal(nxt, got["cells"][live, t + 1]), t
        x, y = nxt % W, nxt // W
        m_ = np.zeros(len(live), np.uint8)
        for j, (dx, dy) in enumerate(((0, -1), (-1, 0), (1, 0), (0, 1))):
            mx, my = x + dx, y + dy
            out = (mx < 0) | (mx >= W) | (my < 0) | (my >= grid.shape[0])
            v = np.where(out, 1, world[np.clip(my, 0, grid.shape[0] - 1),
                                       np.clip(mx, 0, W - 1)]).astype(np.uint8)
            v ^= (r[:, 1 + j] < np.float32(0.02)).astype(np.uint8)
            m_ |= v << j
        assert np.array_equal(m_, got["measurements"][live, t]), t


_REF_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import pomdp_oracle_py as po
d = np.load(sys.argv[2])
ref = po.RefFull(d["grid"], tuple(int(v) for v in d["goal"]), float(d["gamma"]),
                 int(d["pbvi"].shape[0]))
ref.set_alphas(d["fib"], d["pbvi"], d["fa"], d["pa"])
ref.create(d["b0"], seed=1)
acts = []
for a, z in d["az"]:
    acts.append(int(ref.plan(int(d["depth"]), int(d["iters"]))[0]))
    assert ref.update(int(a), int(z)) == 0
print(json.dumps(acts))
ref.R.ref_full_tree_destroy()
ref.close()
"""


def test_one_episode_replays_through_the_reference_search_tree():
    if not os.path.exists(REF_SO):
        pytest.skip("oracle/_ref/libpp2d_ref_pomdp_full.so not built")
    name = "sparse_map_100x40"
    grid, world, goal, (m, fib, pbvi, fa, pa), starts, steps, d, it = setup(name)
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p, DummySimulator(grid) as sim:
        p.set_alphas(fib, pbvi, fa, pa)
        got = sim.rollout(p, starts[:1], steps, 77, record=True, max_depth=d, max_iter=it)
    t = int(got["steps"][0])
    assert t > 0
    b0 = np.zeros(grid.size, np.float32)
    b0[starts[0, 1] * grid.shape[1] + starts[0, 0]] = 1
    az = np.stack([got["actions"][0, :t], got["measurements"][0, :t]], axis=1)
    with tempfile.TemporaryDirectory() as tmp:
        f = os.path.join(tmp, "in.npz")
        np.savez(f, grid=grid, goal=np.array(goal), gamma=np.float32(GAMMA), fib=fib, pbvi=pbvi,
                 fa=fa, pa=pa, b0=b0, az=az, depth=d, iters=it)
        res = subprocess.run([sys.executable, "-c", _REF_SCRIPT, os.path.dirname(__file__), f],
                             capture_output=True, text=True, timeout=900, check=True)
    assert json.loads(res.stdout.strip().splitlines()[-1]) == got["actions"][0, :t].tolist()


def test_argument_and_state_rules():
    grid, world, goal, (m, fib, pbvi, fa, pa), starts, steps, d, it = setup("map_10x10")
    INV, ST = _lib.PP2D_ERR_INVALID, _lib.PP2D_ERR_STATE
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p, DummySimulator(world) as sim:
        with pytest.raises(_lib.Pp2dError) as e:
            sim.rollout(p, starts, 5, 1)
        assert e.value.code == ST                 # no alpha vectors yet
        p.set_alphas(fib, pbvi, fa, pa)
        for kw in ({"max_depth": 0}, {"max_iter": 0}):
            with pytest.raises(_lib.Pp2dError) as e:
                sim.rollout(p, starts, 5, 1, **kw)
            assert e.value.code == INV
        occupied = np.argwhere(world == 1)[0][::-1].astype(np.uint32)
        with pytest.raises(_lib.Pp2dError) as e:
            sim.rollout(p, np.stack([starts[0], occupied]), 5, 1)
        assert e.value.code == INV and "episode 1" in str(e.value)
        with pytest.raises(ValueError):
            sim.rollout(p, starts, 5, 1, instances=[0] * len(starts))
        res = sim.rollout(p, starts[:0], 5, 1)
        assert res["steps"].size == 0
    with PomdpPathPlanning2d(np.zeros((4, 4), np.uint8), (1, 1), GAMMA) as p2, \
            DummySimulator(grid) as sim:
        with pytest.raises(_lib.Pp2dError) as e:
            sim.rollout(p2, starts, 5, 1)
        assert e.value.code == INV                # size mismatch
