"""Re-planning on a stream of local map edits: cold re-solve against warm
start (pp2d_mdp_update_map).

The 4096^2 grid of bench.py (seed 12345, goal at the centre) is solved cold to
the reference's stopping rule.  Then a seeded stream of edits is applied:
32x32 blocks appearing at random free spots away from the goal or disappearing
again, and one goal move.  For each edit two handles run, in alternating
order:
  (a) reset + solve        (J = 0, the reference's stopping rule)
  (b) update_map + solve   (from the previous solution, the same stopping rule)
Per edit: sweeps to the stopping rule, device time of the two calls (CUDA
events on the stream the library runs on), the executed unit share of the
fused launches (pp2d_mdp_work_counters), and, for information, max |J_b - J_a|
and the share of equal actions (different start, same stopping rule: not
expected to be bit-equal).

Two regimes: (b) starts right after the cold solve (300 sweeps, most units
still changing in their last bits), or after 1000 sweeps (the fp32 fixed point).
Writes one JSON line for the card, one per edit and one summary per regime.

  python tools/replan_steps.py [--edits 20] [--out FILE]
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

N = 4096
BLOCK = 32


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


def edit_stream(grid, goal, n_edits, seed):
    """[(map, goal, description)]: every map is the previous one plus one edit."""
    rng = np.random.default_rng(seed)
    cur, g = grid.copy(), goal
    placed, out = [], []
    for i in range(n_edits):
        desc = {}
        if i == n_edits // 2:
            free = np.argwhere(cur[g[1] - 300:g[1] + 300, g[0] - 300:g[0] + 300] == 0)
            y, x = free[rng.integers(len(free))]
            g = (int(g[0] - 300 + x), int(g[1] - 300 + y))
            desc = {"kind": "goal_move", "goal": list(g)}
        elif placed and rng.random() < 0.35:
            y, x, saved = placed.pop(int(rng.integers(len(placed))))
            cur[y:y + BLOCK, x:x + BLOCK] = saved
            desc = {"kind": "block_removed", "y": y, "x": x}
        else:
            while True:
                y, x = int(rng.integers(0, N - BLOCK)), int(rng.integers(0, N - BLOCK))
                far = abs(y + BLOCK // 2 - g[1]) > 2 * BLOCK or abs(x + BLOCK // 2 - g[0]) > 2 * BLOCK
                if far and cur[y:y + BLOCK, x:x + BLOCK].mean() < 0.5:
                    break
            placed.append((y, x, cur[y:y + BLOCK, x:x + BLOCK].copy()))
            cur[y:y + BLOCK, x:x + BLOCK] = 1
            desc = {"kind": "block_added", "y": y, "x": x}
        cur[g[1], g[0]] = 0
        out.append((cur.copy(), g, desc))
    return out


def timed(fn):
    """fn() on the library's stream (the legacy default stream), CUDA events
    around it; the library's calls synchronise before they return."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    res = fn()
    e1.record()
    torch.cuda.synchronize()
    return res, e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3


def regime(name, grid, goal, stream, warm_sweeps):
    import cases
    from path_planning_2d_b200 import MdpPathPlanning2d
    a = MdpPathPlanning2d(grid, goal, cases.GAMMA)
    b = MdpPathPlanning2d(grid, goal, cases.GAMMA)
    (sa, _), ms_cold, _ = timed(a.valueIteration)
    (sb, _), _, _ = timed(b.valueIteration)
    if warm_sweeps > sb:
        b.sweeps(warm_sweeps - sb)
    lines = [{"regime": name, "record": "start", "cold_solve_sweeps": sa,
              "cold_solve_ms": ms_cold, "b_sweep_count": b.sweep_count}]
    for i, (m, g, desc) in enumerate(stream):
        rec = {"regime": name, "record": "edit", "edit": i, **desc}

        def run_a():
            a.reset(m, g)
            return a.valueIteration()

        def run_b():
            b.update_map(m, g)
            return b.valueIteration()

        order = [("a", a, run_a), ("b", b, run_b)]
        if i % 2:
            order.reverse()
        for tag, h, fn in order:
            w0 = h.work_counters()
            (sweeps, res), ms, host_ms = timed(fn)
            w1 = h.work_counters()
            rec[f"sweeps_{tag}"] = sweeps
            rec[f"device_ms_{tag}"] = ms
            rec[f"host_ms_{tag}"] = host_ms
            rec[f"executed_share_{tag}"] = (w1[0] - w0[0]) / max(1, w1[1] - w0[1])
            rec[f"last_residual_{tag}"] = float(res[-1])
        ja, aa = (x.copy() for x in a.download())
        jb, ab = b.download()
        rec["max_abs_jb_minus_ja"] = float(np.abs(jb.astype(np.float64) - ja).max())
        rec["equal_action_share"] = float((aa == ab).mean())
        rec["b_sweep_count"] = b.sweep_count
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    edits = [r for r in lines if r["record"] == "edit"]
    summary = {"regime": name, "record": "summary", "edits": len(edits)}
    for tag in ("a", "b"):
        summary[f"median_device_ms_{tag}"] = float(np.median([r[f"device_ms_{tag}"] for r in edits]))
        summary[f"total_device_ms_{tag}"] = float(sum(r[f"device_ms_{tag}"] for r in edits))
        summary[f"median_sweeps_{tag}"] = float(np.median([r[f"sweeps_{tag}"] for r in edits]))
        summary[f"mean_executed_share_{tag}"] = float(np.mean([r[f"executed_share_{tag}"]
                                                               for r in edits]))
    lines.append(summary)
    print(json.dumps(summary), flush=True)
    a.close()
    b.close()
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--edits", type=int, default=20)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import cases
    from path_planning_2d_b200 import MdpPathPlanning2d
    if not torch.cuda.is_available():
        sys.exit("replan_steps.py measures on the GPU; no CUDA device found")
    head = {"record": "card", **card(), "grid": [N, N], "seed": 12345, "edit_seed": args.seed,
            "block": BLOCK, "edits": args.edits}
    print(json.dumps(head), flush=True)
    grid, goal = cases.synthetic_map(N, N, 0.20, seed=12345, goal=(N // 2, N // 2))
    stream = edit_stream(grid, goal, args.edits, args.seed)
    # warm-up: module load and every kernel the timed calls launch
    g, gl = cases.synthetic_map(512, 512, 0.2, seed=1)
    with MdpPathPlanning2d(g, gl, cases.GAMMA) as w:
        w.valueIteration()
        w.update_map(g, gl)
        w.valueIteration()
        w.reset(g, gl)
        w.download()
    lines = [head]
    lines += regime("after_cold_solve", grid, goal, stream, 0)
    lines += regime("from_fixed_point_1000", grid, goal, stream, 1000)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(l) for l in lines) + "\n")


if __name__ == "__main__":
    main()
