"""Closed-loop episodes of the QV-tree planner: persistent tree batches against
fresh trees, and the rollout against a host loop of single trees.

Bundled sparse_map_100x40, goal (95, 34), gamma 0.95, the bench's alpha
vectors (FIB solver + 500 PBVI vectors from the uniform initial belief),
depth cap 50, 15 expansions per step, K episodes in {256, 1250} from seeded
free starts with point-mass beliefs, 100 steps.
  steps:    the loop driven from here through SearchTreeBatch: per step, the
            plan of the live trees (timed, executed belief x row products from
            pp2d_pomdp_work_counters) against plan_batch of fresh trees on the
            same root beliefs (tracked with pp2d_pomdp_bayes_update), then the
            world step (numpy Philox helpers of tests/rollout_oracle_py.py) and
            the update.
  rollout:  DummySimulator.rollout with the planner, once with the roots
            planned in mode order (PP2D_POMDP_SORT=1) and once in creation
            order (=0): wall time and executed products of each.
  host:     the same episodes through single SearchTree handles, for the first
            --host episodes (time per episode-step).
The tool fails unless every loop gives the same actions, measurements, cells
and steps.  Host wall clock around calls that end in a device synchronise.
First line: the card and its power limit, read in the same run.

  python tools/pomdp_rollout_steps.py [--ks 256,1250] [--steps 100] [--host 8] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from batch_steps import card  # noqa: E402

GAMMA = 0.95
GOAL = (95, 34)
SEED = 0x70D
DIRS = ((0, -1), (-1, 0), (1, 0), (0, 1))


def world_steps(world, cells, acts, seed, episodes, t):
    """Motion and sensors of DESIGN.md section 7c for many episodes at once."""
    import rollout_oracle_py as ro
    h, w = world.shape
    r = ro.step_uniforms_np(seed, episodes, t)
    slot = ro.motion_slots_np(acts, r[:, 0])
    c = cells.astype(np.int64)
    tx, ty = c % w + slot % 3 - 1, c // w + slot // 3 - 1
    ok = (slot != 4) & (tx >= 0) & (tx < w) & (ty >= 0) & (ty < h)
    ok[ok] = world[ty[ok], tx[ok]] == 0
    nxt = np.where(ok, ty * w + tx, c)
    x, y = nxt % w, nxt // w
    z = np.zeros(len(c), np.uint8)
    for j, (dx, dy) in enumerate(DIRS):
        mx, my = x + dx, y + dy
        out = (mx < 0) | (mx >= w) | (my < 0) | (my >= h)
        v = np.where(out, 1, world[np.clip(my, 0, h - 1), np.clip(mx, 0, w - 1)]).astype(np.uint8)
        v ^= (r[:, 1 + j] < np.float32(0.02)).astype(np.uint8)
        z |= v << j
    return nxt.astype(np.uint32), z


def planner(grid, alphas):
    from path_planning_2d_b200 import PomdpPathPlanning2d
    p = PomdpPathPlanning2d(grid, GOAL, GAMMA)
    p.set_alphas(*alphas)
    return p


def steps_loop(grid, alphas, starts, max_steps):
    """The loop through SearchTreeBatch, with plan_batch of fresh trees on the
    same root beliefs beside every plan."""
    from path_planning_2d_b200 import SearchTreeBatch
    k, hw, w = len(starts), grid.size, grid.shape[1]
    goal = GOAL[1] * w + GOAL[0]
    cells = (starts[:, 1] * w + starts[:, 0]).astype(np.uint32)
    bel = np.zeros((k, hw), np.float32)
    bel[np.arange(k), cells] = 1
    rec = {"actions": np.zeros((k, max_steps), np.uint8),
           "measurements": np.zeros((k, max_steps), np.uint8),
           "cells": np.zeros((k, max_steps + 1), np.uint32), "steps": np.zeros(k, np.uint32)}
    rec["cells"][:, 0] = cells
    per = []
    p = planner(grid, alphas)
    b = SearchTreeBatch(p, bel)
    for t in range(max_steps):
        live = np.nonzero(cells != goal)[0].astype(np.uint32)
        if live.size == 0:
            break
        w0 = p.work_counters()[2]
        t0 = time.perf_counter()
        acts, _ = b.plan(live)
        t1 = time.perf_counter()
        w1 = p.work_counters()[2]
        fa, _ = p.plan_batch(bel[live])
        t2 = time.perf_counter()
        w2 = p.work_counters()[2]
        # fresh trees pick the same action only where the kept tree adds nothing;
        # the comparison is of cost, not of actions
        cells[live], z = world_steps(grid, cells[live], acts, SEED, live, t)
        b.update(live, acts, z)
        bel[live] = p.bayes_update(bel[live], acts, z, normalize=True)[0]
        rec["actions"][live, t], rec["measurements"][live, t] = acts, z
        rec["cells"][live, t + 1] = cells[live]
        rec["steps"][live] = t + 1
        per.append({"t": t, "live": int(live.size), "batch_s": t1 - t0, "fresh_s": t2 - t1,
                    "batch_products": w1 - w0, "fresh_products": w2 - w1,
                    "fresh_same_action": int((fa == acts).sum())})
    b.close()
    p.close()
    return rec, per


def rollout(grid, alphas, starts, max_steps, sort):
    from path_planning_2d_b200 import DummySimulator
    os.environ["PP2D_POMDP_SORT"] = sort         # read when the handle is created
    p = planner(grid, alphas)
    del os.environ["PP2D_POMDP_SORT"]
    with DummySimulator(grid) as sim:
        sim.rollout(p, starts[:8], 3, SEED)     # warm-up
        w0 = p.work_counters()[2]
        t0 = time.perf_counter()
        res = sim.rollout(p, starts, max_steps, SEED, record=True)
        dt = time.perf_counter() - t0
        w1 = p.work_counters()[2]
    p.close()
    return res, dt, w1 - w0


def host_loop(grid, alphas, starts, max_steps):
    from path_planning_2d_b200 import SearchTree
    w = grid.shape[1]
    goal = GOAL[1] * w + GOAL[0]
    p = planner(grid, alphas)
    acts = np.zeros((len(starts), max_steps), np.uint8)
    n_steps = 0
    t0 = time.perf_counter()
    for i, (x, y) in enumerate(starts):
        cell = np.array([y * w + x], np.uint32)
        b = np.zeros(grid.size, np.float32)
        b[cell[0]] = 1
        tree = SearchTree(p, b)
        for t in range(max_steps):
            if cell[0] == goal:
                break
            a, _ = tree.plan(50, 15)
            cell, z = world_steps(grid, cell, np.array([a], np.uint8), SEED, [i], t)
            tree.update(a, int(z[0]))
            acts[i, t] = a
            n_steps += 1
        tree.close()
    dt = time.perf_counter() - t0
    p.close()
    return acts, dt, n_steps


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--ks", default="256,1250")
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--host", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import cases
    from path_planning_2d_b200 import PomdpPathPlanning2d
    grid = cases.load_bundled("sparse_map_100x40")
    with PomdpPathPlanning2d(grid, GOAL, GAMMA) as p:
        fib, fa, _ = p.fastInformedBound()
        _, pbvi, pa = p.pointBasedValueIteration(p.initial_belief, 500, rand_seed=1)
    alphas = (fib, pbvi, fa, pa)
    lines = [{"card": card()}]
    free = np.argwhere(grid == 0)
    for k in [int(v) for v in args.ks.split(",")]:
        pick = np.random.default_rng(k).choice(len(free), size=k, replace=False)
        starts = free[pick][:, ::-1].astype(np.uint32)
        rec, per = steps_loop(grid, alphas, starts, args.steps)
        sorted_res, t_sorted, w_sorted = rollout(grid, alphas, starts, args.steps, "1")
        plain_res, t_plain, w_plain = rollout(grid, alphas, starts, args.steps, "0")
        for key in ("actions", "measurements", "cells", "steps"):
            assert np.array_equal(sorted_res[key], rec[key]), key
            assert np.array_equal(plain_res[key], rec[key]), key
        assert np.array_equal(sorted_res["final_belief"].view(np.uint32),
                              plain_res["final_belief"].view(np.uint32))
        h = min(args.host, k)
        hacts, t_host, host_steps = host_loop(grid, alphas, starts[:h], args.steps)
        assert np.array_equal(hacts, rec["actions"][:h])
        ep_steps = int(rec["steps"].sum())
        lines.append({
            "episodes": k, "max_steps": args.steps, "episode_steps": ep_steps,
            "reached": int(sorted_res["reached"].sum()),
            "plan_s": {"batch": sum(q["batch_s"] for q in per),
                       "fresh_plan_batch": sum(q["fresh_s"] for q in per)},
            "products": {"batch": int(sum(q["batch_products"] for q in per)),
                         "fresh_plan_batch": int(sum(q["fresh_products"] for q in per))},
            "rollout": {"mode_order": {"s": t_sorted, "products": int(w_sorted)},
                        "creation_order": {"s": t_plain, "products": int(w_plain)}},
            "host_single_trees": {"episodes": h, "episode_steps": host_steps, "s": t_host,
                                  "s_per_episode_step": t_host / max(host_steps, 1)},
            "rollout_s_per_episode_step": t_sorted / max(ep_steps, 1),
            "per_step": per,
        })
    text = "\n".join(json.dumps(x) for x in lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
