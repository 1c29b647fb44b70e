"""GPU box: time the fused 2-sweep kernel of the library in PP2D_LIB (4096^2 syn grid)
and print a checksum of J after 100 sweeps.  usage: PP2D_LIB=... python tools/time_fused.py [size]
The timed sweeps (100-600) are where unit skipping starts: run with
PP2D_MDP_SKIP=0 to time the dense kernel."""
import os
import sys
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
from path_planning_2d_b200 import MdpPathPlanning2d  # noqa: E402

size = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
grid, goal = cases.synthetic_map(size, size, 0.20, seed=12345)
with MdpPathPlanning2d(grid, goal, cases.GAMMA) as m:
    m.set_stream(torch.cuda.current_stream().cuda_stream, asynchronous=True)
    m.sweeps(100, want_action=False)
    torch.cuda.synchronize()
    cost, _ = m.download()
    crc = zlib.crc32(cost.tobytes())
    best = 1e9
    for rep in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        m.sweeps(100, want_action=False)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
rate = size * size * 100 / (best * 1e-3)
print(f"{os.path.basename(os.environ.get('PP2D_LIB', 'libpp2d.so')):28s} {best/50*1e3:7.2f} us/launch "
      f"{rate/1e9:7.1f} Gcell/s  frac {rate*10/6537.6e9:.3f}  crc {crc:08x}", flush=True)
