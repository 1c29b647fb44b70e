"""Re-planning inside a batch: pp2d_mdp_batch_update + solve against the only
way a batch could re-plan before it, reset + solve of all K instances.

K seeded free goals on the bundled map_100x40 (one shared map, gamma 0.95),
K in {16, 256, 4096}, one robot per goal.  Both sides start from a batch
solved on the original map; only the re-plan is timed.
  (i)  shared edit: one costmap edit (a 6x6 block added, 40 occupied cells
       freed; goals it covers move to a free cell) for the whole fleet:
       update all K instances with the one map, then solve;
  (ii) goal move: one robot's goal moves: update instance K/2, then solve.
The baseline resets the batch to the new map and goals and solves all K.
Replan and baseline alternate, --reps times; host wall clock around calls that
end in a device synchronise (every library call does).  Per line: medians, the
sweeps the solve ran (max over the updated instances; the baseline's), the
fused units run / launched by the re-plan, and a bit-equality check of the
updated instances (all of them up to K = 256, a seeded sample of 64 above)
against single handles doing solve, update_map, solve, plus the check that
the instances not updated kept their download.

  python tools/batch_replan_steps.py [--ks 16,256,4096] [--reps 5] [--out FILE]
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

from batch_steps import card, workload  # noqa: E402

GAMMA = 0.95


def shared_edit(grid, goals, seed=7):
    """(new map, new goals) of workload (i)."""
    rng = np.random.default_rng(seed)
    g = grid.copy()
    h, w = g.shape
    y, x = int(rng.integers(0, h - 6)), int(rng.integers(0, w - 6))
    g[y:y + 6, x:x + 6] = 1
    occ = np.argwhere(grid == 1)
    for yy, xx in occ[rng.choice(len(occ), size=min(40, len(occ)), replace=False)]:
        g[yy, xx] = 0
    free = np.argwhere(g == 0)
    out = []
    for gx, gy in goals:
        if g[gy, gx] != 0:
            d = np.abs(free[:, 0] - gy) + np.abs(free[:, 1] - gx)
            fy, fx = free[int(np.argmin(d))]
            gx, gy = int(fx), int(fy)
        out.append((gx, gy))
    return g, out


def goal_move(grid, goals, k, seed=11):
    """(instances, new goals) of workload (ii): instance k gets a new free goal."""
    rng = np.random.default_rng(seed)
    free = np.argwhere(grid == 0)
    y, x = free[rng.integers(len(free))]
    return [k], [(int(x), int(y))]


def replan(batch, grid, goals, listed, map2, goals2_listed):
    batch.reset(grid, goals)
    batch.valueIteration()
    before = batch.download()
    w0 = batch.work_counters()
    t0 = time.perf_counter()
    batch.update_map(listed, map2, goals2_listed)
    n, res = batch.valueIteration()
    t1 = time.perf_counter()
    w1 = batch.work_counters()
    return t1 - t0, n, res, before, (w1[0] - w0[0], w1[1] - w0[1])


def baseline(batch, grid, goals, map2, goals2):
    batch.reset(grid, goals)
    batch.valueIteration()
    t0 = time.perf_counter()
    batch.reset(map2, goals2)
    n, _ = batch.valueIteration()
    return time.perf_counter() - t0, n


def check_against_single(batch, grid, goals, listed, map2, goals2_listed, n, res, before, sample):
    """Updated instances (a sample of them) equal single handles bit for bit;
    the others kept their download."""
    from path_planning_2d_b200 import MdpPathPlanning2d
    cost, action = batch.download()
    rng = np.random.default_rng(5)
    pick = range(len(listed)) if len(listed) <= sample else \
        sorted(rng.choice(len(listed), size=sample, replace=False))
    same = True
    with MdpPathPlanning2d(grid, goals[0], GAMMA) as m:
        for i in pick:
            k = listed[i]
            m.reset(grid, goals[k])
            m.valueIteration()
            m.update_map(map2, goals2_listed[i])
            sn, sres = m.valueIteration()
            c, a = m.download()
            same &= bool(n[k] == sn and np.array_equal(res[k].view(np.uint64), sres.view(np.uint64))
                         and np.array_equal(c.view(np.uint32), cost[k].view(np.uint32))
                         and np.array_equal(a, action[k]))
    others = np.setdiff1d(np.arange(len(goals)), listed)
    kept = bool(np.array_equal(before[0][others].view(np.uint32), cost[others].view(np.uint32))
                and np.array_equal(before[1][others], action[others]))
    return same, len(pick), kept


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="16,256,4096")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("batch_replan_steps.py measures on a GPU; none found")
    from path_planning_2d_b200 import MdpBatchPathPlanning2d
    lines = [dict(kind="card", **card())]
    print(json.dumps(lines[0]), flush=True)
    for k in [int(v) for v in args.ks.split(",")]:
        grid, goals = workload("goals", k)
        map2_i, goals2_i = shared_edit(grid, goals)
        listed_ii, goals2_ii = goal_move(grid, goals, k // 2)
        all_goals_ii = list(goals)
        all_goals_ii[k // 2] = goals2_ii[0]
        cases = {
            "shared_edit": (list(range(k)), map2_i, goals2_i, map2_i, goals2_i),
            "goal_move": (listed_ii, grid, goals2_ii, grid, all_goals_ii),
        }
        with MdpBatchPathPlanning2d(grid, goals, GAMMA) as a, \
                MdpBatchPathPlanning2d(grid, goals, GAMMA) as b:
            for name, (listed, map2, g2_listed, base_map, base_goals) in cases.items():
                # warm-up of both paths
                replan(a, grid, goals, listed, map2, g2_listed)
                baseline(b, grid, goals, base_map, base_goals)
                t_re, t_base = [], []
                for rep in range(args.reps):
                    order = ("replan", "baseline") if rep % 2 == 0 else ("baseline", "replan")
                    for which in order:
                        if which == "replan":
                            t, n_re, res_re, before, work = replan(a, grid, goals, listed, map2,
                                                                  g2_listed)
                            t_re.append(t)
                        else:
                            t, n_base = baseline(b, grid, goals, base_map, base_goals)
                            t_base.append(t)
                same, checked, kept = check_against_single(
                    a, grid, goals, listed, map2, g2_listed, n_re, res_re, before, 64)
                tr, tb = float(np.median(t_re)), float(np.median(t_base))
                line = dict(
                    kind=name, K=k, updated=len(listed), reps=args.reps,
                    replan_s=tr, reset_solve_s=tb, replan_all_s=t_re, reset_solve_all_s=t_base,
                    speedup=tb / tr,
                    replan_sweeps_max=int(max(n_re[i] for i in listed)),
                    reset_solve_sweeps_max=int(n_base.max()),
                    units_run=work[0], units_launched=work[1],
                    run_share=work[0] / max(work[1], 1),
                    bitwise_equal_to_single=same, instances_checked=checked,
                    others_unchanged=kept)
                lines.append(line)
                print(json.dumps(line), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
