"""Closed-loop episodes of a POMDP fleet whose robots go to different goals:
one planner handle holding G goals against G single-goal handles.

Bundled sparse_map_100x40, gamma 0.95, goal 0 = (95, 34) and seeded free
cells as goals 1..15; per goal the FIB solver and 500 PBVI vectors from the
uniform initial belief, both on the GPU from a handle created with that goal.
1 250 robots from seeded free starts with point-mass beliefs, spread evenly
over G in {1, 4, 16} goals (robot i goes to goal i * G // 1250), depth cap 50,
15 expansions per step, 100 steps.
  goals:   DummySimulator.rollout on one handle with the G goals (goals=...).
  single:  the G single-goal handles one after the other, each rolling out its
           own robots with their episode ids.
The tool fails unless both give the same steps, reached, collisions, cells,
actions, measurements and final beliefs.  Per G and variant: wall time (host
clock around calls that end in a device synchronise, after a warm-up call on
every handle), microseconds per episode-step and the executed belief x
inner-row products of the bound evaluations (pp2d_pomdp_work_counters), with
the share spent on padded entries (pp2d_pomdp_padding_counters).  First line:
the card and its power limit, read in the same run.

  python tools/pomdp_goals_steps.py [--gs 1,4,16] [--robots 1250] [--steps 100] [--out FILE]
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
GOAL0 = (95, 34)
SEED = 0x60A1


def goal_cells(grid, n):
    free = np.argwhere(grid == 0)
    pick = np.random.default_rng(16).choice(len(free), size=n - 1, replace=False)
    return [GOAL0] + [(int(free[i][1]), int(free[i][0])) for i in pick]


def solve(grid, goal):
    from path_planning_2d_b200 import PomdpPathPlanning2d
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
        fib, fa, _ = p.fastInformedBound()
        _, pbvi, pa = p.pointBasedValueIteration(p.initial_belief, 500, rand_seed=1)
    return fib, pbvi, fa, pa


def counters(p):
    return p.work_counters()[2], p.padding_counters()[1]


def timed_rollout(sim, p, starts, steps, first, goals=None):
    w0 = counters(p)
    t0 = time.perf_counter()
    res = sim.rollout(p, starts, steps, SEED, first_episode=first, record=True, goals=goals)
    dt = time.perf_counter() - t0
    w1 = counters(p)
    return res, dt, w1[0] - w0[0], w1[1] - w0[1]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--gs", default="1,4,16")
    ap.add_argument("--robots", type=int, default=1250)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import cases
    from path_planning_2d_b200 import DummySimulator, PomdpPathPlanning2d
    grid = cases.load_bundled("sparse_map_100x40")
    gs = [int(v) for v in args.gs.split(",")]
    cells = goal_cells(grid, max(gs))
    t0 = time.perf_counter()
    alphas = [solve(grid, c) for c in cells]
    lines = [{"card": card(), "goals": cells, "solve_s": time.perf_counter() - t0}]
    free = np.argwhere(grid == 0)
    n = args.robots
    starts = free[np.random.default_rng(n).choice(len(free), size=n, replace=False)][:, ::-1]
    starts = np.ascontiguousarray(starts, np.uint32)
    with DummySimulator(grid) as sim:
        for G in gs:
            goal_of = (np.arange(n) * G // n).astype(np.uint32)    # contiguous per goal
            # (a) one handle with G goals
            p = PomdpPathPlanning2d(grid, cells[0], GAMMA)
            p.set_alphas(*alphas[0])
            p.set_goals(cells[1:G])
            for g in range(1, G):
                p.set_goal_alphas(g, *alphas[g])
            sim.rollout(p, starts[:8], 3, SEED, goals=goal_of[:8])     # warm-up
            ra, ta, wa, pa = timed_rollout(sim, p, starts, args.steps, 0, goal_of)
            p.close()
            # (b) G single-goal handles, one after the other
            singles = []
            for g in range(G):
                q = PomdpPathPlanning2d(grid, cells[g], GAMMA)
                q.set_alphas(*alphas[g])
                sim.rollout(q, starts[:8], 3, SEED)                    # warm-up
                singles.append(q)
            tb, wb, rb = 0.0, 0, {}
            for g, q in enumerate(singles):
                idx = np.flatnonzero(goal_of == g)
                r, dt, w, _ = timed_rollout(sim, q, starts[idx], args.steps, int(idx[0]))
                tb += dt
                wb += w
                for key, v in r.items():
                    rb.setdefault(key, []).append(v)
                q.close()
            rb = {k: np.concatenate(v) for k, v in rb.items()}
            for key in ra:
                assert np.array_equal(ra[key].view(np.uint8), rb[key].view(np.uint8)), (G, key)
            ep_steps = int(ra["steps"].sum())
            lines.append({
                "goals": G, "robots": n, "max_steps": args.steps, "episode_steps": ep_steps,
                "reached": int(ra["reached"].sum()),
                "one_handle": {"s": ta, "us_per_episode_step": 1e6 * ta / max(ep_steps, 1),
                               "products": int(wa), "padded_products": int(pa),
                               "padded_share": pa / max(wa, 1)},
                "single_handles": {"s": tb, "us_per_episode_step": 1e6 * tb / max(ep_steps, 1),
                                   "products": int(wb)},
                "speedup": tb / ta,
            })
            print(json.dumps(lines[-1]), flush=True)
    text = "\n".join(json.dumps(x) for x in lines)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
