"""Many small problems: one batch (pp2d_mdp_batch_*) against one handle per
problem solved back to back.

Workloads on the reference's launch-file map size, 100x40 (gamma 0.95):
  goals: K seeded free goals on the bundled map_100x40 (one shared map);
  maps:  K seeded random 100x40 maps (densities 0.05 .. 0.25), one goal each.
For K in {1, 16, 256, 1024, 4096}, in alternating order, repeated --reps times:
  (a) single: one MdpPathPlanning2d handle; per instance reset + solve
      (pp2d_mdp_solve) + download, what a user does today;
  (b) batch:  one MdpBatchPathPlanning2d created beforehand; reset + solve +
      download of all instances.
Host wall clock around calls that end in a device synchronise (every call of
the library does).  Per line: medians of both, instances/s, useful
cell-updates/s (sum over instances of sweeps * 4000 cells / time), the unit
launches run / launched by the batch's fused sweeps, the sweep-count spread,
and a check that the batch's results equal the single handle's bit for bit.
idle_lane_share_geometric is computed from the strip geometry (1 - W / (60 *
strips)), not measured: the share of the lanes of a fused launch that hold no
map column at W = 100.

  python tools/batch_steps.py [--ks 1,16,256,1024,4096] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

STRIP = 60          # columns of a fused launch's strip


def card():
    import torch
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        out["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


def workload(kind, k, seed=2024):
    import cases
    rng = np.random.default_rng(seed + k)
    if kind == "goals":
        grid = cases.load_bundled("map_100x40")
        free = np.argwhere(grid == 0)
        pick = free[rng.choice(len(free), size=k, replace=len(free) < k)]
        return grid, [(int(x), int(y)) for y, x in pick]
    maps = np.empty((k, 40, 100), np.uint8)
    goals = []
    for i in range(k):
        p = 0.05 + 0.2 * rng.random()
        maps[i] = rng.random((40, 100)) < p
        g = (int(rng.integers(100)), int(rng.integers(40)))
        maps[i, g[1], g[0]] = 0
        goals.append(g)
    return maps, goals


def run_single(mdp, grid_maps, goals):
    t0 = time.perf_counter()
    sweeps, cost, action = [], [], []
    for i, g in enumerate(goals):
        mdp.reset(grid_maps if grid_maps.ndim == 2 else grid_maps[i], g)
        n, _ = mdp.valueIteration()
        c, a = mdp.download()
        sweeps.append(n)
        cost.append(c.copy())
        action.append(a.copy())
    return time.perf_counter() - t0, np.array(sweeps), np.stack(cost), np.stack(action)


def run_batch(batch, grid_maps, goals):
    w0 = batch.work_counters()
    t0 = time.perf_counter()
    batch.reset(grid_maps, goals)
    n, _ = batch.valueIteration()
    t1 = time.perf_counter()
    cost, action = batch.download()
    t2 = time.perf_counter()
    w1 = batch.work_counters()
    return t2 - t0, t1 - t0, n, cost, action, (w1[0] - w0[0], w1[1] - w0[1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="1,16,256,1024,4096")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kinds", default="goals,maps")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("batch_steps.py measures on a GPU; none found")
    from path_planning_2d_b200 import MdpBatchPathPlanning2d, MdpPathPlanning2d
    gamma = 0.95
    lines = [dict(kind="card", **card())]
    print(json.dumps(lines[0]), flush=True)
    for kind in args.kinds.split(","):
        for k in [int(v) for v in args.ks.split(",")]:
            grid_maps, goals = workload(kind, k)
            first = grid_maps if grid_maps.ndim == 2 else grid_maps[0]
            with MdpPathPlanning2d(first, goals[0], gamma) as mdp, \
                    MdpBatchPathPlanning2d(grid_maps, goals, gamma) as batch:
                # warm-up of both paths (module load, launch geometry)
                run_single(mdp, grid_maps, goals[:min(k, 4)])
                run_batch(batch, grid_maps, goals)
                t_single, t_batch, t_solve, work = [], [], [], None
                same = True
                for rep in range(args.reps):
                    order = ("single", "batch") if rep % 2 == 0 else ("batch", "single")
                    for which in order:
                        if which == "single":
                            t, n_s, c_s, a_s = run_single(mdp, grid_maps, goals)
                            t_single.append(t)
                        else:
                            t, ts, n_b, c_b, a_b, work = run_batch(batch, grid_maps, goals)
                            t_batch.append(t)
                            t_solve.append(ts)
                    same &= bool(np.array_equal(n_s, n_b)
                                 and np.array_equal(c_s.view(np.uint32), c_b.view(np.uint32))
                                 and np.array_equal(a_s, a_b))
            cells = 40 * 100
            useful = float(np.sum(n_b)) * cells
            ts_med, tb_med = float(np.median(t_single)), float(np.median(t_batch))
            vals, counts = np.unique(n_b, return_counts=True)
            line = dict(
                kind=kind, K=k, reps=args.reps,
                single_s=ts_med, batch_s=tb_med, batch_solve_s=float(np.median(t_solve)),
                single_all_s=t_single, batch_all_s=t_batch,
                speedup=ts_med / tb_med,
                single_instances_per_s=k / ts_med, batch_instances_per_s=k / tb_med,
                single_cell_updates_per_s=useful / ts_med,
                batch_cell_updates_per_s=useful / tb_med,
                units_run=work[0], units_launched=work[1],
                run_share=work[0] / max(work[1], 1),
                sweeps_min=int(n_b.min()), sweeps_max=int(n_b.max()),
                sweeps_hist={str(int(v)): int(c) for v, c in zip(vals, counts)},
                idle_lane_share_geometric=1.0 - 100 / (-(-100 // STRIP) * STRIP),
                bitwise_equal_to_single=same)
            lines.append(line)
            print(json.dumps(line), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
