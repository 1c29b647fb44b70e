"""Closed-loop episodes on the device against the same loop driven from the host.

K episodes on the bundled map_100x40 (gamma 0.95), K in {256, 4096, 16384},
one batch planner with one seeded free goal per episode (solved once, not
timed), seeded free starts, 200 max steps, point-mass and uniform-over-free
start beliefs.
  device: DummySimulator.rollout (pp2d_sim_rollout_mdp_batch), one call;
  host:   the loop through the per-step API: per step, plan_batch on the live
          episodes' beliefs, the numpy Philox and sampler of
          tests/rollout_oracle_py.py for motion and sensors, and
          DummySimulator.updateBelief (beliefs up and down every step).
Both loops must give identical steps, reached, collisions, final cells and
final-belief bits; the tool fails otherwise.  Host wall clock around work
that ends in a device synchronise (every library call does); the device loop
is warmed up with a small call first and timed --reps times (median).  First
line: the card and its power limit, read in the same run.

  python tools/rollout_steps.py [--ks 256,4096,16384] [--reps 3] [--out FILE]
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
MAX_STEPS = 200
SEED = 0x5EED


def host_loop(sim, batch, goals, grid, inst, starts, beliefs, max_steps, seed):
    import rollout_oracle_py as ro
    h, w = grid.shape
    n = len(starts)
    goals = np.asarray(goals, np.int64)[inst]
    x, y = starts[:, 0].astype(np.int64), starts[:, 1].astype(np.int64)
    bel = beliefs.copy()
    steps = np.zeros(n, np.uint32)
    coll = np.zeros(n, np.uint32)
    live = np.nonzero((x != goals[:, 0]) | (y != goals[:, 1]))[0]
    t = 0
    pad = np.ones((h + 2, w + 2), np.uint8)
    pad[1:-1, 1:-1] = grid > 0
    while live.size and t < max_steps:
        u = batch.plan_batch(inst[live], bel[live])
        r = ro.step_uniforms_np(seed, live.astype(np.uint64), t)
        slot = ro.motion_slots_np(u, r[:, 0])
        tx, ty = x[live] + slot % 3 - 1, y[live] + slot // 3 - 1
        blocked = (slot != 4) & (pad[ty + 1, tx + 1] > 0)
        coll[live] += blocked
        x[live] = np.where(blocked, x[live], tx)
        y[live] = np.where(blocked, y[live], ty)
        meas = np.empty((live.size, 4), np.uint8)
        for j, (ox, oy) in enumerate([(0, -1), (-1, 0), (1, 0), (0, 1)]):
            meas[:, j] = pad[y[live] + oy + 1, x[live] + ox + 1] ^ (r[:, 1 + j] < np.float32(0.02))
        bel[live] = sim.updateBelief(bel[live], action=u, measurement=meas)
        steps[live] += 1
        t += 1
        at_goal = (x[live] == goals[live, 0]) & (y[live] == goals[live, 1])
        live = live[~at_goal]
    reached = ((x == goals[:, 0]) & (y == goals[:, 1])).astype(np.uint8)
    return {"steps": steps, "reached": reached, "collisions": coll,
            "final_cell": (y * w + x).astype(np.uint32), "final_belief": bel}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="256,4096,16384")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_rollout_steps.jsonl"))
    a = ap.parse_args()
    import cases
    from path_planning_2d_b200 import DummySimulator, MdpBatchPathPlanning2d

    lines = [dict(kind="card", **card())]
    print(json.dumps(lines[0]), flush=True)
    grid = cases.load_bundled("map_100x40")
    hw = grid.size
    free = np.argwhere(grid == 0)
    uniform = (grid.reshape(-1) == 0).astype(np.float32)
    uniform /= uniform.sum(dtype=np.float32)
    with DummySimulator(grid) as sim:
        for k in [int(v) for v in a.ks.split(",")]:
            rng = np.random.default_rng(k)
            g = free[rng.choice(len(free), size=k, replace=len(free) < k)]
            batch_goals = [(int(xx), int(yy)) for yy, xx in g]
            s = free[rng.choice(len(free), size=k, replace=len(free) < k)]
            starts = np.stack([s[:, 1], s[:, 0]], axis=1).astype(np.uint32)
            inst = np.arange(k, dtype=np.uint32)
            with MdpBatchPathPlanning2d(grid, batch_goals, GAMMA) as b:
                b.valueIteration()
                for belief in ("point", "uniform"):
                    if belief == "point":
                        b0 = np.zeros((k, hw), np.float32)
                        b0[np.arange(k), starts[:, 1] * grid.shape[1] + starts[:, 0]] = 1.0
                        arg = None
                    else:
                        b0 = np.broadcast_to(uniform, (k, hw)).copy()
                        arg = b0
                    sim.rollout(b, starts[:8], MAX_STEPS, SEED, beliefs=None, instances=inst[:8])
                    dev_t = []
                    for _ in range(a.reps):
                        t0 = time.perf_counter()
                        dev = sim.rollout(b, starts, MAX_STEPS, SEED, beliefs=arg, instances=inst,
                                          record=True)
                        dev_t.append(time.perf_counter() - t0)
                    t0 = time.perf_counter()
                    host = host_loop(sim, b, batch_goals, grid, inst, starts, b0, MAX_STEPS, SEED)
                    host_s = time.perf_counter() - t0
                    same = all(np.array_equal(np.asarray(dev[key]), np.asarray(host[key]))
                               for key in ("steps", "reached", "collisions", "final_cell"))
                    same_bel = np.array_equal(dev["final_belief"].view(np.uint32),
                                              host["final_belief"].view(np.uint32))
                    ep_steps = int(dev["steps"].sum())
                    dev_s = float(np.median(dev_t))
                    line = dict(kind="rollout", K=k, belief=belief, max_steps=MAX_STEPS,
                                reps=a.reps, device_s=dev_s, device_all_s=dev_t, host_s=host_s,
                                speedup=host_s / dev_s, episode_steps=ep_steps,
                                reached=int(dev["reached"].sum()),
                                collisions=int(dev["collisions"].sum()),
                                device_episodes_per_s=k / dev_s,
                                device_episode_steps_per_s=ep_steps / dev_s,
                                host_episodes_per_s=k / host_s,
                                host_episode_steps_per_s=ep_steps / host_s,
                                stats_identical=bool(same), final_beliefs_identical=bool(same_bel))
                    lines.append(line)
                    print(json.dumps(line), flush=True)
                    if not (same and same_bel):
                        raise SystemExit("device and host loops differ")
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
