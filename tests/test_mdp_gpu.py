"""GPU tier: the sm_100a path through the C ABI against the oracle.

Bar: bit-exact J (float bit patterns), byte-exact greedy action, identical
sweep count and residuals, identical way-point indices."""
import ctypes
import os

import numpy as np
import pytest

import cases
import oracle_py
from path_planning_2d_b200 import MdpPathPlanning2d, _lib

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _assert_same(mdp, ora, what=""):
    cost, action = mdp.download()
    assert np.array_equal(_bits(cost), _bits(ora.cost)), f"J differs {what}"
    assert np.array_equal(action, ora.act), f"action differs {what}"


@pytest.mark.parametrize("name", list(cases.BUNDLED))
def test_bundled_maps_converge_like_the_reference(name):
    """BASELINE.json configs[1]: value iteration to convergence on every
    bundled map; policy bit-exact, V bit-exact (bar: 1e-5 relative)."""
    goal, start = cases.BUNDLED[name]
    grid = cases.load_bundled(name)
    J, A, n, res = oracle_py.value_iteration(grid, goal, cases.GAMMA)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as mdp:
        sweeps, residuals = mdp.initialize()
        assert sweeps == n == 300
        assert np.array_equal(residuals, res)
        assert np.array_equal(_bits(mdp.optimal_cost), _bits(J))
        assert np.array_equal(mdp.optimal_action, A)
        rel = np.abs(mdp.optimal_cost - J) / np.maximum(np.abs(J), 1e-30)
        assert rel.max() <= 1e-5
        assert np.array_equal(mdp.waypoints(start), oracle_py.waypoints(A, start))


@pytest.mark.parametrize("path", sorted(
    __import__("glob").glob(os.path.join(cases.GOLDEN, "ref_*.npz"))) or [None])
def test_against_reference_golden_vectors(path):
    if path is None:
        pytest.skip("tests/golden/ref_*.npz not generated yet")
    g = np.load(path)
    grid, goal = g["grid"], tuple(int(v) for v in g["goal"])
    with MdpPathPlanning2d(grid, goal, float(g["gamma"])) as mdp:
        for _ in range(int(g["sweeps"]) // 100):
            mdp.sweeps(100)
        cost, action = mdp.download()
    assert np.array_equal(_bits(cost), _bits(g["J"]))
    assert np.array_equal(action, g["action"])


SHAPES = [(1, 1), (1, 40), (40, 1), (2, 2), (3, 3), (7, 5), (16, 28), (17, 29),
          (33, 61), (64, 120), (65, 121), (100, 257), (300, 333), (513, 1030)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("p_occ", [0.0, 0.2, 0.6])
def test_ragged_shapes_step_by_step(shape, p_occ):
    """Every strip/row-block remainder, every sweep-count parity (1 = arg-min
    kernel only, 2 = plain + arg-min, 3 = fused pair + arg-min, ...)."""
    h, w = shape
    grid, goal = cases.synthetic_map(h, w, p_occ, seed=h * 1000 + w)
    ora = oracle_py.OracleMdp(grid, goal, cases.GAMMA)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as mdp:
        for k in (1, 2, 3, 4, 7):
            mdp.sweeps(k)
            ora.sweeps(k)
            _assert_same(mdp, ora, f"after {ora.n} sweeps on {shape} p={p_occ}")
        assert mdp.sweep_count == ora.n


@pytest.mark.parametrize("cw2,cw1,rpu,lin", [(1, 1, 16, -1), (2, 2, 5, -1), (4, 4, 64, -1),
                                             (2, 4, 0, 0), (4, 1, 7, -1), (2, 4, 0, 1),
                                             (4, 2, 0, 1), (1, 1, 0, 1)])
def test_every_kernel_variant(monkeypatch, cw2, cw1, rpu, lin):
    """Column widths per lane (1/2/4), rows per unit and the unit scheme (whole
    row blocks per strip / equal runs of the strip-major row sequence) are
    tuning knobs; all variants must give the same bits."""
    monkeypatch.setenv("PP2D_MDP_CW2", str(cw2))
    monkeypatch.setenv("PP2D_MDP_CW1", str(cw1))
    monkeypatch.setenv("PP2D_MDP_ROWS_PER_UNIT", str(rpu))
    monkeypatch.setenv("PP2D_MDP_LINEAR_UNITS", str(lin))
    grid, goal = cases.synthetic_map(211, 387, 0.25, seed=7)
    ora = oracle_py.OracleMdp(grid, goal, 0.9)
    with MdpPathPlanning2d(grid, goal, 0.9) as mdp:
        for k in (6, 1, 9):
            mdp.sweeps(k)
            ora.sweeps(k)
            _assert_same(mdp, ora, f"variant cw2={cw2} cw1={cw1} rpu={rpu} lin={lin}")


@pytest.mark.parametrize("gamma", [0.5, 0.9, 0.99, 0.999])
def test_discount_factors(gamma):
    grid, goal = cases.synthetic_map(90, 150, 0.3, seed=3)
    ora = oracle_py.OracleMdp(grid, goal, gamma)
    with MdpPathPlanning2d(grid, goal, gamma) as mdp:
        mdp.sweeps(25)
        ora.sweeps(25)
        _assert_same(mdp, ora, f"gamma={gamma}")


def test_residual_matches_host_inf_norm():
    grid, goal = cases.synthetic_map(120, 200, 0.2, seed=11)
    ora = oracle_py.OracleMdp(grid, goal, cases.GAMMA)
    prev = ora.cost.copy()
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as mdp:
        for k in (10, 100, 3):
            mdp.sweeps(k)
            ora.sweeps(k)
            want = float(np.abs(ora.cost - prev).max())
            prev = ora.cost.copy()
            assert mdp.residual() == np.float32(want)


def test_no_occupied_cells_and_all_but_goal_occupied():
    grid = np.zeros((20, 30), np.uint8)
    ora = oracle_py.OracleMdp(grid, (3, 4), cases.GAMMA)
    with MdpPathPlanning2d(grid, (3, 4), cases.GAMMA) as mdp:
        mdp.sweeps(50)
        ora.sweeps(50)
        _assert_same(mdp, ora)
        assert mdp.residual() == np.float32(np.abs(ora.cost).max())
    grid = np.ones((9, 9), np.uint8)
    grid[4, 4] = 0
    ora = oracle_py.OracleMdp(grid, (4, 4), cases.GAMMA)
    with MdpPathPlanning2d(grid, (4, 4), cases.GAMMA) as mdp:
        mdp.sweeps(13)
        ora.sweeps(13)
        _assert_same(mdp, ora)


def test_goal_occupied_is_rejected():
    grid = np.zeros((8, 8), np.uint8)
    grid[2, 3] = 1
    with pytest.raises(_lib.Pp2dError) as e:
        MdpPathPlanning2d(grid, (3, 2), cases.GAMMA)
    assert e.value.code == _lib.PP2D_ERR_GOAL_OCCUPIED


def test_belief_callback_and_batch():
    name = "sparse_map_100x40"
    goal, start = cases.BUNDLED[name]
    grid = cases.load_bundled(name)
    rng = np.random.default_rng(0)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as mdp:
        mdp.initialize()
        A = mdp.optimal_action
        beliefs = rng.random((64, grid.size), dtype=np.float32)
        beliefs[0] = 0.0                      # all zero -> index 0
        beliefs[1, [100, 2000]] = 2.0         # tie -> first
        beliefs[2, -1] = 3.0
        got = mdp.plan_batch(beliefs)
        want = [oracle_py.plan(b, A) for b in beliefs]
        assert got.tolist() == want
        assert mdp.beliefCallback(beliefs[5]) == want[5]


def test_sharded_handles_reproduce_the_unsharded_solve():
    """Row shards on ONE GPU with host-mediated ghost-row copies: the
    partition must not change a single bit (SURVEY.md section 8e)."""
    import torch
    grid, goal = cases.synthetic_map(150, 170, 0.2, seed=5)
    ora = oracle_py.OracleMdp(grid, goal, cases.GAMMA)
    bounds = [0, 37, 39, 100, 150]
    shards = [MdpPathPlanning2d(grid, goal, cases.GAMMA, rows=(a, b))
              for a, b in zip(bounds[:-1], bounds[1:])]

    def exchange():
        from path_planning_2d_b200.distributed import device_tensor
        halos = [s.halo() for s in shards]
        for i in range(len(shards) - 1):
            up, dn = halos[i], halos[i + 1]
            assert up.bytes == dn.bytes
            t = lambda p: device_tensor(p, up.bytes)
            # lower rows of shard i -> ghost rows above shard i+1, and back
            t(dn.recv_top).copy_(t(up.send_bottom))
            t(up.recv_bottom).copy_(t(dn.send_top))
        torch.cuda.synchronize()
    try:
        total = 0
        for k, want_action in [(2, False), (2, False), (1, False), (2, True),
                               (1, True), (2, False), (1, True)]:
            for s in shards:
                s.sweeps(k, want_action)
            exchange()
            ora.sweeps(k)
            total += k
        cost = np.concatenate([s.download()[0] for s in shards])
        action = np.concatenate([s.download()[1] for s in shards])
        assert np.array_equal(_bits(cost), _bits(ora.cost))
        assert np.array_equal(action, ora.act)
        res = max(s.residual() for s in shards)
        assert res == np.float32(np.abs(ora.cost).max())
    finally:
        for s in shards:
            s.close()


@pytest.mark.parametrize("devices", [[0], [0, 0], [0, 0, 0, 0, 0]])
def test_single_process_multi_shard_handle(devices):
    """pp2d_mdp_create_multi through every entry point a planner uses; here all
    shards on device 0 (ghost rows copied between event-ordered streams), so the
    test also runs on a 1-GPU box.  tests/test_distributed_gpu.py repeats it on
    distinct devices (peer-to-peer ghost rows)."""
    grid, goal = cases.synthetic_map(157, 203, 0.2, seed=31)
    ora = oracle_py.OracleMdp(grid, goal, cases.GAMMA)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA, devices=devices) as mdp:
        assert mdp.device_count == len(devices) and not mdp.peer_to_peer
        for k, wa in [(1, True), (2, False), (5, True), (4, False), (3, True), (100, True)]:
            mdp.sweeps(k, wa)
            ora.sweeps(k)
            if wa:
                _assert_same(mdp, ora, f"{len(devices)} shards after {ora.n} sweeps")
        assert mdp.sweep_count == ora.n
        assert mdp.residual() == np.float32(np.abs(ora.cost).max())
        rng = np.random.default_rng(1)
        beliefs = rng.random((9, grid.size), dtype=np.float32)
        beliefs[0] = 0
        assert mdp.plan_batch(beliefs).tolist() == [oracle_py.plan(b, ora.act) for b in beliefs]
        start = tuple(int(v) for v in np.argwhere(grid == 0)[5][::-1])
        assert np.array_equal(mdp.waypoints(start), oracle_py.waypoints(ora.act, start))
        # a new map on the same handle, then the reference's stopping rule
        grid2, goal2 = cases.synthetic_map(157, 203, 0.3, seed=32, goal=(7, 100))
        mdp.reset(grid2, goal2)
        J, A, n, res = oracle_py.value_iteration(grid2, goal2, cases.GAMMA)
        sweeps, residuals = mdp.initialize()
        assert sweeps == n and np.array_equal(residuals, res)
        assert np.array_equal(_bits(mdp.optimal_cost), _bits(J))
        assert np.array_equal(mdp.optimal_action, A)
    with pytest.raises(_lib.Pp2dError):
        MdpPathPlanning2d(grid, goal, cases.GAMMA, devices=[0, 99])
    with pytest.raises(_lib.Pp2dError):
        MdpPathPlanning2d(grid[:3], (0, 0), cases.GAMMA, devices=[0, 0])


def test_full_size_properties_4096():
    """BASELINE.json configs[2] size: the oracle is too slow here, so check
    size-independent properties: (a) sweeps(6)+sweeps(5) == sweeps(11) bit for
    bit (fused pairs vs arg-min tail), (b) the single-sweep kernel path equals
    the fused path, (c) goal stays 0 / stay only at the goal, (d) a 256-row
    band cut out of the middle agrees with the oracle run on that band with
    exact ghost rows is covered by the sharded test; here the first 3 sweeps
    of the top-left 256x256 corner are compared with the oracle on the corner
    (information travels one cell per sweep, so cells >= 3 away from the cut
    are exact)."""
    h = w = 4096
    grid, goal = cases.synthetic_map(h, w, 0.20, seed=12345)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as a, \
            MdpPathPlanning2d(grid, goal, cases.GAMMA) as b:
        a.sweeps(6)
        a.sweeps(5)
        for _ in range(11):
            b.sweeps(1)
        ca, aa = a.download()
        cb, ab = b.download()
        assert np.array_equal(_bits(ca), _bits(cb))
        assert np.array_equal(aa, ab)
        assert ca[goal[1], goal[0]] == 0.0
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as c:
        c.sweeps(3)
        cc, ac = c.download()
    corner = grid[:256, :256].copy()
    cgoal = (0, 0) if corner[0, 0] == 0 else tuple(np.argwhere(corner == 0)[0][::-1])
    ora = oracle_py.OracleMdp(corner, (int(cgoal[0]), int(cgoal[1])), cases.GAMMA)
    ora.sweeps(3)
    # exclude the oracle's goal neighbourhood and the cut edges
    sel = np.zeros((256, 256), bool)
    sel[8:250, 8:250] = True
    assert np.array_equal(_bits(cc[:256, :256])[sel], _bits(ora.cost)[sel])
    assert np.array_equal(ac[:256, :256][sel], ora.act[sel])


@pytest.mark.parametrize("shape,goal", [((4096, 4096), (2048, 2048)),
                                        ((1536, 16384), (8192, 700))])
def test_benchmarked_sizes_to_convergence_vs_the_reference_kernels(shape, goal):
    """BASELINE.json configs[2] (the bench grid: 4096 x 4096, seed 12345, goal
    at the centre) and one shard-shaped grid of configs[3], 16384 wide -- 1536
    rows rather than the 2048 of an 8-GPU shard, because the reference kernels
    index their tables with 32-bit ints (81 * idx, path_planning_2d_cuda.cu:
    222-235) and fail beyond 2^31 / 81 = 26.5 M cells --, solved
    to the reference's stopping rule by pp2d_mdp_solve and by the UNMODIFIED
    reference kernels in the reference's own loop (oracle/_ref,
    src/mdp/path_planning_2d.cu:223-263): same number of sweeps, same
    residuals, J bit for bit, action byte for byte."""
    import sys
    so = os.path.join(cases.ROOT, "oracle", "_ref", "libpp2d_ref_mdp.so")
    if not os.path.exists(so):
        pytest.skip("oracle/_ref not built")
    sys.path.insert(0, os.path.join(cases.ROOT, "tests", "golden"))
    import make_golden
    h, w = shape
    grid, goal = cases.synthetic_map(h, w, 0.20, seed=12345, goal=goal)
    J, A, n, res = make_golden.ref_solve(make_golden.ref_lib(), grid, goal, cases.GAMMA)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as mdp:
        sweeps, residuals = mdp.initialize()
        assert sweeps == n
        assert np.array_equal(residuals, res)
        assert np.array_equal(_bits(mdp.optimal_cost), _bits(J))
        assert np.array_equal(mdp.optimal_action, A)
    assert n >= 300 and res[-1] <= 5.0 / (1.0 - np.float32(cases.GAMMA)) * 1e-3 < res[-2]


@pytest.mark.parametrize("shape,goal", [((4096, 4096), (2048, 2048)),
                                        ((1536, 16384), (8192, 700))])
def test_benchmarked_sizes_to_convergence_vs_the_reference_record(shape, goal):
    """The comparison above against its stored record (tests/golden/
    bench_ref_<h>x<w>.npz): same number of sweeps, same residuals, and the
    CRC-32 of every J row (bits) and action row."""
    import sys
    sys.path.insert(0, cases.GOLDEN)
    import make_golden
    h, w = shape
    g = np.load(os.path.join(cases.GOLDEN, f"bench_ref_{h}x{w}.npz"))
    grid, goal = cases.synthetic_map(h, w, 0.20, seed=12345, goal=goal)
    assert tuple(int(v) for v in g["goal"]) == goal
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as mdp:
        sweeps, residuals = mdp.initialize()
        assert sweeps == int(g["sweeps"])
        assert np.array_equal(residuals, g["residuals"])
        assert np.array_equal(make_golden.crc_rows(_bits(mdp.optimal_cost)), g["J_crc"])
        assert np.array_equal(make_golden.crc_rows(mdp.optimal_action), g["action_crc"])


def test_full_size_16384_row_shards_equal_the_unsharded_grid():
    """BASELINE.json configs[3] size (16384 x 16384, 2.7e8 cells) on one GPU:
    8 row shards of 2048 rows with ghost-row exchange after every launch must
    reproduce the unsharded solve bit for bit (Jacobi is partition invariant;
    the oracle is too slow at this size).  Fused pairs, a single sweep and the
    arg-min sweep are all exercised."""
    import torch
    from path_planning_2d_b200.distributed import device_tensor
    n = 16384
    grid, goal = cases.synthetic_map(n, n, 0.20, seed=12345, goal=(n // 2, 2048))
    plan = [(2, False), (2, False), (1, False), (2, True)]
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as whole:
        for k, wa in plan:
            whole.sweeps(k, wa)
        cost, action = whole.download()
        res = whole.residual()
    bounds = list(range(0, n + 1, 2048))
    shards = [MdpPathPlanning2d(grid, goal, cases.GAMMA, rows=(a, b))
              for a, b in zip(bounds[:-1], bounds[1:])]
    try:
        for k, wa in plan:
            for s in shards:
                s.sweeps(k, wa)
            halos = [s.halo() for s in shards]
            for i in range(len(shards) - 1):
                up, dn = halos[i], halos[i + 1]
                t = lambda p: device_tensor(p, up.bytes)
                t(dn.recv_top).copy_(t(up.send_bottom))
                t(up.recv_bottom).copy_(t(dn.send_top))
            torch.cuda.synchronize()
        for s, a, b in zip(shards, bounds[:-1], bounds[1:]):
            c, act = s.download()
            assert np.array_equal(_bits(c), _bits(cost[a:b])), (a, b)
            assert np.array_equal(act, action[a:b]), (a, b)
        assert max(s.residual() for s in shards) == res
    finally:
        for s in shards:
            s.close()
    assert cost[goal[1], goal[0]] == 0.0
    assert np.all(action[grid == 1] == 0)


def test_asynchronous_download_overlaps_the_next_solve():
    """pp2d_mdp_download_begin snapshots the solution; the handle is reset and
    swept on another map right away; _wait then delivers the FIRST solution.
    Also on a multi-shard handle."""
    import torch
    grid, goal = cases.synthetic_map(301, 257, 0.2, seed=41)
    grid2, goal2 = cases.synthetic_map(301, 257, 0.35, seed=42, goal=(9, 200))
    ora = oracle_py.OracleMdp(grid, goal, cases.GAMMA)
    ora.sweeps(37)
    ora2 = oracle_py.OracleMdp(grid2, goal2, cases.GAMMA)
    ora2.sweeps(12)
    for devices in (None, [0, 0, 0]):
        cost = torch.empty(grid.size, dtype=torch.float32).pin_memory()
        act = torch.empty(grid.size, dtype=torch.uint8).pin_memory()
        cost2 = torch.empty(grid.size, dtype=torch.float32).pin_memory()
        with MdpPathPlanning2d(grid, goal, cases.GAMMA, devices=devices) as mdp:
            mdp.sweeps(37)
            mdp.download_begin(cost.data_ptr(), act.data_ptr())
            mdp.reset(grid2, goal2)
            mdp.sweeps(12)
            mdp.download_begin(cost2.data_ptr(), None)      # second one queues behind the first
            mdp.download_wait()
            assert np.array_equal(_bits(cost.numpy().reshape(grid.shape)), _bits(ora.cost))
            assert np.array_equal(act.numpy().reshape(grid.shape), ora.act)
            assert np.array_equal(_bits(cost2.numpy().reshape(grid.shape)), _bits(ora2.cost))
            _assert_same(mdp, ora2, "after the overlapped downloads")


def test_staged_map_upload_overlaps_the_running_solve():
    """pp2d_mdp_stage_map uploads the NEXT map while sweeps of the current one
    are queued; reset() with the same pointer uses the staged rows, with
    another pointer it drops them.  Three maps in a row (both staging buffers
    are reused), also on a multi-shard handle."""
    import torch
    maps = [cases.synthetic_map(301, 257, d, seed=s, goal=g)
            for d, s, g in ((0.2, 51, None), (0.35, 52, (9, 200)), (0.1, 53, (250, 7)),
                            (0.3, 54, (128, 150)))]
    pinned = [torch.from_numpy(m.copy()).pin_memory().numpy() for m, _ in maps]
    for devices in (None, [0, 0, 0]):
        with MdpPathPlanning2d(pinned[0], maps[0][1], cases.GAMMA, devices=devices) as mdp:
            for k in range(1, 4):
                mdp.sweeps(8)                     # queued work of map k-1
                mdp.stage_map(pinned[k])          # travels meanwhile
                ora_prev = oracle_py.OracleMdp(maps[k - 1][0], maps[k - 1][1], cases.GAMMA)
                ora_prev.sweeps(8)
                _assert_same(mdp, ora_prev, f"map {k - 1} while map {k} is staged")
                mdp.reset(pinned[k], maps[k][1])
                assert mdp.sweep_count == 0
            ora = oracle_py.OracleMdp(maps[3][0], maps[3][1], cases.GAMMA)
            mdp.sweeps(11)
            ora.sweeps(11)
            _assert_same(mdp, ora, "after three staged resets")
            # a staged map that is NOT the one reset() gets is dropped
            mdp.stage_map(pinned[1])
            mdp.reset(pinned[2], maps[2][1])
            ora = oracle_py.OracleMdp(maps[2][0], maps[2][1], cases.GAMMA)
            mdp.sweeps(6)
            ora.sweeps(6)
            _assert_same(mdp, ora, "staged map dropped")
            # ... and the next staged upload still works
            mdp.stage_map(pinned[0])
            mdp.reset(pinned[0], maps[0][1])
            ora = oracle_py.OracleMdp(maps[0][0], maps[0][1], cases.GAMMA)
            mdp.sweeps(5)
            ora.sweeps(5)
            _assert_same(mdp, ora, "staged after a dropped one")
        with pytest.raises(ValueError):
            with MdpPathPlanning2d(pinned[0], maps[0][1], cases.GAMMA) as mdp:
                mdp.stage_map(pinned[0][:100])


def test_reset_reuses_the_handle():
    grid, goal = cases.synthetic_map(97, 143, 0.25, seed=21)
    grid2, goal2 = cases.synthetic_map(97, 143, 0.1, seed=22, goal=(5, 90))
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as mdp:
        mdp.sweeps(9)
        mdp.residual()
        mdp.reset(grid2, goal2)
        assert mdp.sweep_count == 0
        ora = oracle_py.OracleMdp(grid2, goal2, cases.GAMMA)
        mdp.sweeps(12)
        ora.sweeps(12)
        _assert_same(mdp, ora, "after reset")
        assert mdp.residual() == np.float32(np.abs(ora.cost).max())
        grid2[goal2[1], goal2[0]] = 1
        with pytest.raises(_lib.Pp2dError):
            mdp.reset(grid2, goal2)
