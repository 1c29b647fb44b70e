"""Expected share of units the fused sweep launches run with unit skipping
(PP2D_MDP_SKIP, DESIGN.md section 4), simulated on the CPU oracle
(oracle/mdp_oracle.c, bit-identical to the device J).  No GPU needed.

Geometry of the fused row-block launch: strips of 60 useful columns, the row
blocks that fill the warp slots of one wave (mdp.cu launch_sweep).  The slots
are SMs x resident CTAs per SM x 8 warps: 148 x 2 x 8 on a B200, where the
library reads the CTA count from cudaOccupancyMaxActiveBlocksPerMultiprocessor.
A build or a setting that changes it (other register counts,
PP2D_MDP_ROWS_PER_UNIT) launches another geometry: pass --sms /
--ctas-per-sm / --rows-per-unit to match it, or the prediction is off.

changed[k][u]: launch k (sweeps 2k+1, 2k+2) wrote a J that differs from the J it read on some cell of unit u.  Launch k+1 runs
unit u iff u or one of its 8 neighbours changed in launch k; the first launch
after the reset and the arg-min launch (the last of every 100-sweep step) run
every unit.

  python tools/stationarity_sim.py [--height 4096] [--width 4096] [--seed 12345]
                                   [--occupied 0.2] [--steps 10] [--threads 8]
                                   [--sms 148] [--ctas-per-sm 2] [--rows-per-unit R]

The benchmark grid (4096^2, seed 12345, goal at the centre) takes about 5
minutes on 8 cores for 10 steps.
"""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
import oracle_py  # noqa: E402

STRIP = 60            # useful columns of a warp (T = 2, CW = 2: 30 lanes x 2)
WARPS_PER_CTA = 8


def geometry(h, w, slots, rows_per_unit=0):
    n_strips = -(-w // STRIP)
    if rows_per_unit <= 0:
        blocks = max(1, slots // n_strips)
        rows_per_unit = max(8, -(-h // blocks))
    return n_strips, -(-h // rows_per_unit), rows_per_unit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--height", type=int, default=4096)
    ap.add_argument("--width", type=int, default=4096)
    ap.add_argument("--seed", type=int, default=12345)
    ap.add_argument("--occupied", type=float, default=0.20)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--threads", type=int, default=8)
    ap.add_argument("--sms", type=int, default=148)
    ap.add_argument("--ctas-per-sm", type=int, default=2)
    ap.add_argument("--rows-per-unit", type=int, default=0,
                    help="fixed row-block height (PP2D_MDP_ROWS_PER_UNIT); 0: one wave")
    args = ap.parse_args()
    h, w = args.height, args.width
    grid, goal = cases.synthetic_map(h, w, args.occupied, seed=args.seed, goal=(w // 2, h // 2))
    ns, nb, rpu = geometry(h, w, args.sms * args.ctas_per_sm * WARPS_PER_CTA,
                           args.rows_per_unit)
    print(f"{h}x{w}: {ns} strips x {nb} row blocks of {rpu} rows", flush=True)
    oracle_py.set_threads(args.threads)
    o = oracle_py.OracleMdp(grid, goal, cases.GAMMA)

    def unit_any(mask):
        m = np.zeros((nb * rpu, ns * STRIP), bool)
        m[:h, :w] = mask
        return m.reshape(nb, rpu, ns, STRIP).any(axis=(1, 3))

    def dilate(u):
        p = np.pad(u, 1)
        out = np.zeros_like(u)
        for dy in range(3):
            for dx in range(3):
                out |= p[dy:dy + u.shape[0], dx:dx + u.shape[1]]
        return out

    prev = o.cost.copy()
    changed = np.ones((nb, ns), bool)       # after a reset: everything runs
    total = run = 0
    per_launch = []
    t0 = time.time()
    for k in range(args.steps * 50):
        need = np.ones_like(changed) if k % 50 == 49 else dilate(changed)
        total += need.size
        run += int(need.sum())
        per_launch.append(need.mean())
        o.sweeps(2)
        cur = o.cost
        changed = unit_any(cur != prev)
        prev = cur.copy()
        if k % 50 == 49:
            print(f"step {k // 50 + 1:3d}: units run {np.mean(per_launch[-50:]):.3f} "
                  f"(cumulative {run / total:.3f})  t={time.time() - t0:.0f}s", flush=True)
    print(f"executed fraction of unit-launches over {args.steps} steps: {run / total:.4f}")


if __name__ == "__main__":
    main()
