"""GPU tier: skipping unchanged units (PP2D_MDP_SKIP, DESIGN.md section 4)
changes no bit.  Every case builds two handles in one process, one with
PP2D_MDP_SKIP=0 and one with skipping on, drives both through the same calls
and compares J, the action grid and the residual bit for bit after every
period."""
import os

import numpy as np
import pytest
import torch

import cases
from path_planning_2d_b200 import MdpPathPlanning2d

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _handle(skip, grid, goal, **kw):
    old = os.environ.get("PP2D_MDP_SKIP")
    os.environ["PP2D_MDP_SKIP"] = "1" if skip else "0"
    try:
        return MdpPathPlanning2d(grid, goal, cases.GAMMA, **kw)
    finally:
        if old is None:
            del os.environ["PP2D_MDP_SKIP"]
        else:
            os.environ["PP2D_MDP_SKIP"] = old


class Pair:
    """The same calls on a handle without and one with skipping."""

    def __init__(self, grid, goal, **kw):
        self.off = _handle(False, grid, goal, **kw)
        self.on = _handle(True, grid, goal, **kw)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.off.close()
        self.on.close()

    def call(self, name, *args, **kw):
        a = getattr(self.off, name)(*args, **kw)
        b = getattr(self.on, name)(*args, **kw)
        return a, b

    def check(self, what, residual=True):
        if residual:
            r0, r1 = self.call("residual")
            assert np.float32(r0).view(np.uint32) == np.float32(r1).view(np.uint32), \
                f"residual differs {what}: {r0} vs {r1}"
        (c0, a0), (c1, a1) = self.call("download")
        assert np.array_equal(_bits(c0), _bits(c1)), f"J differs {what}"
        assert np.array_equal(a0, a1), f"action differs {what}"


def _blocky_map(h, w, seed):
    grid, goal = cases.synthetic_map(h, w, 0.20, seed=seed)
    rng = np.random.default_rng(seed)
    for _ in range(6):      # large all-occupied blocks, away from the goal
        y, x = int(rng.integers(0, h - 150)), int(rng.integers(0, w - 200))
        if not (y <= goal[1] < y + 150 and x <= goal[0] < x + 200):
            grid[y:y + 150, x:x + 200] = 1
    return grid, goal


def test_bench_grid_1000_sweeps_and_executed_fraction():
    n = 4096
    grid, goal = cases.synthetic_map(n, n, 0.20, seed=12345, goal=(n // 2, n // 2))
    with Pair(grid, goal) as p:
        for period in range(10):
            p.call("sweeps", 100)
            p.check(f"after {100 * (period + 1)} sweeps")
        run_off, total_off = p.off.work_counters()
        run, total = p.on.work_counters()
    assert run_off == total_off == total
    assert run < 0.6 * total, f"{run} of {total} unit-launches executed"


def test_bench_path_shard_handle_two_sweeps_per_call():
    """The benchmark's call pattern: a row-shard handle covering the whole grid
    on torch's stream, 2 sweeps per call, the residual on the device."""
    grid, goal = cases.synthetic_map(1536, 1024, 0.20, seed=7)
    with Pair(grid, goal, rows=(0, 1536)) as p:
        s = torch.cuda.current_stream().cuda_stream
        p.call("set_stream", s, asynchronous=True)
        for period in range(8):
            for _ in range(48):
                p.call("sweeps", 2, want_action=False)
            p.call("sweeps", 2, want_action=True)
            torch.cuda.synchronize()
            p.check(f"period {period}")
        run, total = p.on.work_counters()
        assert run < total


def test_large_occupied_blocks():
    grid, goal = _blocky_map(900, 1300, seed=3)
    with Pair(grid, goal) as p:
        for period in range(6):
            p.call("sweeps", 100)
            p.check(f"period {period}")
        run, total = p.on.work_counters()
        assert run < total


@pytest.mark.parametrize("shape", [(517, 1001), (130, 61), (1000, 59), (9, 700), (2, 2)])
def test_ragged_shapes(shape):
    h, w = shape
    grid, goal = cases.synthetic_map(h, w, 0.20, seed=h * 7 + w)
    with Pair(grid, goal) as p:
        for period in range(6):
            p.call("sweeps", 100)
            p.check(f"{shape} period {period}")


def test_reset_and_stage_map_halfway():
    grid, goal = cases.synthetic_map(700, 1000, 0.20, seed=11)
    other, _ = _blocky_map(700, 1000, seed=12)
    other[goal[1], goal[0]] = 0
    third, _ = cases.synthetic_map(700, 1000, 0.30, seed=13)
    third[goal[1], goal[0]] = 0
    with Pair(grid, goal) as p:
        for period in range(5):
            p.call("sweeps", 100)
        p.check("before the reset")
        p.call("reset", other, goal)
        for period in range(5):
            p.call("sweeps", 100)
            p.check(f"after reset, period {period}")
        p.call("stage_map", third)
        p.call("sweeps", 100)
        p.call("reset", third, (goal[0] + 1, goal[1]) if not third[goal[1], goal[0] + 1]
               else goal)
        for period in range(5):
            p.call("sweeps", 100)
            p.check(f"after the staged reset, period {period}")


def test_odd_sweep_counts_mix_single_sweeps():
    grid, goal = _blocky_map(600, 800, seed=21)
    with Pair(grid, goal) as p:
        for n, wa in [(300, True), (7, True), (13, False), (1, True), (2, False), (1, False),
                      (98, False), (2, True), (51, True), (200, False), (3, True)]:
            p.call("sweeps", n, want_action=wa)
            p.check(f"after {n} sweeps (want_action={wa})")


def test_solve_with_the_reference_stopping_rule():
    grid, goal = _blocky_map(800, 1200, seed=31)
    with Pair(grid, goal) as p:
        (n0, r0), (n1, r1) = p.call("valueIteration")
        assert n0 == n1
        assert np.array_equal(r0, r1)
        p.check("after the solve", residual=False)
        # past the solve: periods the unit masks can skip in
        for period in range(6):
            p.call("sweeps", 100)
            p.check(f"period {period} past the solve")


def test_multi_shard_handle_without_peer_rows():
    """Two row shards on one device exchange ghost rows between launches: the
    row blocks next to them always run.  1025 rows: the upper shard has 513 rows,
    8-row blocks and a last block of 1 row, so the 2-row cone of the block
    before it reaches the ghost rows too."""
    grid, goal = _blocky_map(1025, 700, seed=41)
    with Pair(grid, goal, devices=[0, 0]) as p:
        assert not p.on.peer_to_peer
        for period in range(8):
            p.call("sweeps", 100)
            p.check(f"period {period}")
        run, total = p.on.work_counters()
        assert run < total


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_multi_gpu_handle():
    grid, goal = cases.synthetic_map(2048, 1536, 0.20, seed=51)
    with Pair(grid, goal, devices=2) as p:
        for period in range(8):
            p.call("sweeps", 100)
            p.check(f"period {period}")
