"""Per-step timing of the benchmark's headline solve with unit skipping off and
on (PP2D_MDP_SKIP, DESIGN.md section 4): the 4096^2 grid of bench.py, reset to
J = 0, then K check periods of 100 sweeps + the residual, each timed with CUDA
events.  Prints one JSON line per setting: per-step ms, the fused value-only
launch time (98 sweeps / 49 launches) per step, and the executed unit fraction
per step (pp2d_mdp_work_counters; the arg-min launch always runs every unit).

  python tools/skip_steps.py [--steps K] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def run(skip, steps):
    import torch
    import cases
    from path_planning_2d_b200.distributed import ShardedValueIteration
    os.environ["PP2D_MDP_SKIP"] = str(skip)
    n = 4096
    grid, goal = cases.synthetic_map(n, n, 0.20, seed=12345, goal=(n // 2, n // 2))
    vi = ShardedValueIteration(grid, goal, cases.GAMMA, rank=0, world_size=1)
    mdp = vi.shard.mdp

    def step(evs):
        evs[0].record()
        vi.sweeps(98, want_action=False)
        evs[1].record()
        vi.sweeps(2, want_action=True)
        r = vi.shard.residual_tensor()
        evs[2].record()
        return r

    ev = lambda: [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    for _ in range(3):
        step(ev())
    vi.reset(grid, goal)
    torch.cuda.synchronize()
    out = {"skip": skip, "step_ms": [], "fused_launch_us": [], "executed_fraction": []}
    residual = None
    for _ in range(steps):
        w0 = mdp.work_counters()
        e = ev()
        r = step(e)
        torch.cuda.synchronize()
        w1 = mdp.work_counters()
        out["step_ms"].append(e[0].elapsed_time(e[2]))
        out["fused_launch_us"].append(e[0].elapsed_time(e[1]) / 49 * 1e3)
        out["executed_fraction"].append((w1[0] - w0[0]) / max(1, w1[1] - w0[1]))
        residual = float(r.item())
    out["total_ms"] = sum(out["step_ms"])
    out["residual_after_last_step"] = residual
    out["cell_updates_per_sec"] = n * n * 100 * steps / (out["total_ms"] * 1e-3)
    vi.shard.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--skip", type=int, choices=(0, 1), default=None,
                    help="one setting only (default: off, then on)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []
    for skip in ([args.skip] if args.skip is not None else [0, 1]):
        lines.append(json.dumps(run(skip, args.steps)))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
