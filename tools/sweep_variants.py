"""Time the fused sweep kernel for the tuning knobs (GPU box).
usage: python tools/sweep_variants.py [size] -> table on stdout"""
import itertools
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
from path_planning_2d_b200 import MdpPathPlanning2d  # noqa: E402

size = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
grid, goal = cases.synthetic_map(size, size, 0.20, seed=12345)
rows = []
quick = len(sys.argv) > 2
combos = [(2, 0), (2, 64), (2, 128)]
for cw2, rpu in combos:
    os.environ["PP2D_MDP_CW2"] = str(cw2)
    os.environ["PP2D_MDP_ROWS_PER_UNIT"] = str(rpu)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as m:
        m.set_stream(torch.cuda.current_stream().cuda_stream, asynchronous=True)
        m.sweeps(20, want_action=False)
        torch.cuda.synchronize()
        best = 1e9
        for rep in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            m.sweeps(100, want_action=False)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        rate = size * size * 100 / (best * 1e-3)
        rows.append((cw2, rpu, best / 50, rate))
        print(f"T=2 cw={cw2} rows_per_unit={rpu:4d}  {best/50*1e3:8.1f} us/launch  "
              f"{rate/1e9:8.1f} Gcell/s  {rate*10/6537.6e9:.3f} of HBM roofline", flush=True)
for cw1 in ([] if quick else [1, 2, 4]):
    os.environ["PP2D_MDP_CW1"] = str(cw1)
    os.environ["PP2D_MDP_ROWS_PER_UNIT"] = "0"
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as m:
        m.set_stream(torch.cuda.current_stream().cuda_stream, asynchronous=True)
        for label, wa in (("plain ", False), ("policy", True)):
            for _ in range(5):
                m.sweeps(1, want_action=wa)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                m.sweeps(1, want_action=wa)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 20
            print(f"T=1 {label} cw={cw1}  {ms*1e3:8.1f} us/launch  "
                  f"{size*size/(ms*1e-3)/1e9:8.1f} Gcell/s", flush=True)
