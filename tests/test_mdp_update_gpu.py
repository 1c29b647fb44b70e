"""GPU tier: pp2d_mdp_update_map, re-planning on a changed map from the
current solution.

After the update J' is the previous download with the occupied cells of the
new map at trapped(n) and the new goal at 0; the sweep count carries on.  From
there the library must compute exactly what the oracle computes on the new
map started from J' (bit for bit), on every handle kind, with and without
unit skipping."""
import os
import subprocess

import numpy as np
import pytest
import torch

import cases
import oracle_py
from path_planning_2d_b200 import MdpPathPlanning2d, _lib
from test_host_mirror import fnv
from test_mdp_skip_gpu import Pair

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAMMA32 = float(np.float32(cases.GAMMA))


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


_TRAPPED = {}


def _trapped(n):
    """J of an occupied cell after n sweeps, from the oracle (a 1x2 map whose
    left cell is occupied)."""
    if n not in _TRAPPED:
        ora = oracle_py.OracleMdp(np.array([[1, 0]], np.uint8), (1, 0), cases.GAMMA)
        ora.sweeps(n)
        _TRAPPED[n] = np.float32(ora.cost[0, 0])
    return _TRAPPED[n]


def _jprime(j_prev, grid, goal, n):
    j = np.array(j_prev, dtype=np.float32, copy=True)
    j[grid == 1] = _trapped(n)
    j[goal[1], goal[0]] = 0.0
    return j


def _oracle_from(grid, goal, j, n):
    ora = oracle_py.OracleMdp(grid, goal, cases.GAMMA)
    ora.J[ora.cur][:] = np.asarray(j, np.float32).ravel()
    ora.n = n
    return ora


def _oracle_solve(ora):
    """The reference's valueIteration loop from the oracle's current J."""
    prev = ora.cost.copy()
    total, res = 0, []
    while True:
        ora.sweeps(100)
        total += 100
        r = float(np.abs(ora.cost - prev).max())
        prev = ora.cost.copy()
        res.append(r)
        if not r > 5.0 / (1.0 - GAMMA32) * 1e-3:
            return total, np.array(res)


def _assert_same(mdp, ora, what):
    cost, action = mdp.download()
    assert np.array_equal(_bits(cost), _bits(ora.cost)), f"J differs {what}"
    assert np.array_equal(action, ora.act), f"action differs {what}"


def _free_block(grid, goal, size, rng, avoid=3, holds=0):
    """Top-left corner of a size x size block away from the goal that holds a
    cell of value `holds` (so that writing 1 - holds there changes the map)."""
    h, w = grid.shape
    while True:
        y, x = int(rng.integers(0, max(1, h - size + 1))), int(rng.integers(0, max(1, w - size + 1)))
        if (not (y - avoid <= goal[1] < y + size + avoid and x - avoid <= goal[0] < x + size + avoid)
                and (grid[y:y + size, x:x + size] == holds).any()):
            return y, x


def _edit(grid, goal, kind, seed):
    """(new map, new goal) for one kind of edit."""
    rng = np.random.default_rng(seed)
    g = grid.copy()
    h, w = g.shape
    gx, gy = goal
    s = max(1, min(6, h // 4, w // 4))
    avoid = 3 if min(h, w) > 20 else 0
    if kind == "add":
        y, x = _free_block(g, goal, s, rng, avoid)
        g[y:y + s, x:x + s] = 1
    elif kind == "remove":
        occ = np.argwhere(g == 1)
        assert len(occ) > 0
        for y, x in occ[rng.choice(len(occ), size=min(len(occ), 40), replace=False)]:
            g[y, x] = 0
    elif kind == "both":
        y, x = _free_block(g, goal, s, rng, avoid)
        g[y:y + s, x:x + s] = 1
        y, x = _free_block(g, goal, s, rng, avoid, holds=1)
        g[y:y + s, x:x + s] = 0
    elif kind == "border":
        g[0:s, 0:s] = 1 - g[0:s, 0:s]
        g[h - s:h, w - s:w] = 1
        g[h - 1, :] = 1 - g[h - 1, :]
    elif kind == "near_goal":
        g[max(0, gy - 1):gy + 2, max(0, gx - 1):gx + 2] = 1
    elif kind == "goal_move":
        free = np.argwhere(g == 0)
        y, x = free[rng.integers(len(free))]
        goal = (int(x), int(y))
    elif kind == "goal_to_freed":
        occ = np.argwhere(g == 1)
        y, x = occ[rng.integers(len(occ))]
        g[y, x] = 0
        goal = (int(x), int(y))
    elif kind != "noop":
        raise ValueError(kind)
    g[goal[1], goal[0]] = 0
    return g, goal


def _tiny(h, w, seed):
    grid, goal = cases.synthetic_map(h, w, 0.3, seed=seed, goal=(0, 0))
    grid[0, 0] = 0
    return grid, goal


KINDS = ["add", "remove", "both", "border", "near_goal", "goal_move", "goal_to_freed", "noop"]
MAPS = {
    "map_100x40": lambda: (cases.load_bundled("map_100x40"), cases.BUNDLED["map_100x40"][0]),
    "sparse_map_100x40": lambda: (cases.load_bundled("sparse_map_100x40"),
                                  cases.BUNDLED["sparse_map_100x40"][0]),
    "syn_512x384": lambda: cases.synthetic_map(384, 512, 0.2, seed=384512),
    "syn_1x17": lambda: _tiny(1, 17, 17),
    "syn_2x2": lambda: _tiny(2, 2, 22),
}
PARITY = [(m, k) for m in ("map_100x40", "sparse_map_100x40") for k in KINDS] + \
         [("syn_512x384", k) for k in ("both", "border", "goal_move", "noop")] + \
         [(m, k) for m in ("syn_1x17", "syn_2x2") for k in ("add", "remove", "goal_move", "noop")]


@pytest.mark.parametrize("name,kind", PARITY)
def test_update_matches_the_oracle_from_jprime(name, kind):
    grid, goal = MAPS[name]()
    grid2, goal2 = _edit(grid, goal, kind, seed=len(name) * 31 + KINDS.index(kind))
    if kind not in ("noop", "goal_move"):
        assert not np.array_equal(grid, grid2)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as mdp:
        mdp.valueIteration()
        n = mdp.sweep_count
        j_prev, a_prev = (x.copy() for x in mdp.download())
        mdp.update_map(grid2, goal2)
        assert mdp.sweep_count == n
        want = _jprime(j_prev, grid2, goal2, n)
        j1, a1 = mdp.download()
        assert np.array_equal(_bits(j1), _bits(want)), "J' differs from the rule"
        assert np.array_equal(a1, a_prev), "the action grid must be left as it was"
        if kind == "noop":
            assert np.array_equal(_bits(j1), _bits(j_prev))
        ora = _oracle_from(grid2, goal2, want, n)
        for k in (1, 2, 3, 100):
            mdp.sweeps(k)
            ora.sweeps(k)
            _assert_same(mdp, ora, f"{k} sweeps after the update ({name}, {kind})")
        assert mdp.sweep_count == ora.n
        # back to the first map, then the reference's stopping rule from J''
        j_prev = mdp.download()[0].copy()
        mdp.update_map(grid, goal)
        want = _jprime(j_prev, grid, goal, ora.n)
        ora = _oracle_from(grid, goal, want, ora.n)
        sweeps, residuals = mdp.valueIteration()
        n_ora, res_ora = _oracle_solve(ora)
        assert sweeps == n_ora
        assert np.array_equal(residuals, res_ora)
        _assert_same(mdp, ora, f"after the solve from J'' ({name}, {kind})")


def test_update_right_after_create_and_residual_semantics():
    """An update before any sweep (sweep count 0) and the first residual
    after an update: it measures the change since the update."""
    grid, goal = cases.synthetic_map(120, 200, 0.2, seed=11)
    grid2, goal2 = _edit(grid, goal, "both", seed=5)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as mdp:
        mdp.update_map(grid2, goal2)
        ora = oracle_py.OracleMdp(grid2, goal2, cases.GAMMA)
        for k in (10, 100, 3):
            prev = ora.cost.copy()
            mdp.sweeps(k)
            ora.sweeps(k)
            assert mdp.residual() == np.float32(np.abs(ora.cost - prev).max())
        prev_j = mdp.download()[0].copy()
        grid3, goal3 = _edit(grid2, goal2, "add", seed=6)
        mdp.update_map(grid3, goal3)
        want = _jprime(prev_j, grid3, goal3, ora.n)
        ora = _oracle_from(grid3, goal3, want, ora.n)
        mdp.sweeps(7)
        ora.sweeps(7)
        assert mdp.residual() == np.float32(np.abs(ora.cost - want).max())
        _assert_same(mdp, ora, "after update, 7 sweeps")


def _bench_grid():
    n = 4096
    return cases.synthetic_map(n, n, 0.20, seed=12345, goal=(n // 2, n // 2))


def _two_edits(grid, goal, seed):
    g = grid.copy()
    rng = np.random.default_rng(seed)
    for i in range(2):
        y, x = _free_block(g, goal, 32, rng, avoid=200, holds=i)
        g[y:y + 32, x:x + 32] = 1 if i == 0 else 0
    return g


def test_skipping_stays_exact_after_local_edits_on_the_bench_grid():
    grid, goal = _bench_grid()
    grid2 = _two_edits(grid, goal, seed=1)
    with Pair(grid, goal) as p:
        for _ in range(10):
            p.call("sweeps", 100)
        p.check("after 1000 sweeps")
        p.call("update_map", grid2, goal)
        p.check("right after the update")
        for period in range(3):
            before = p.on.work_counters()
            p.call("sweeps", 100)
            run, total = (a - b for a, b in zip(p.on.work_counters(), before))
            p.check(f"period {period} after the update")
            if period == 0:
                assert run < 0.10 * total, f"{run} of {total} unit-launches executed"
        run_off, total_off = p.off.work_counters()
        assert run_off == total_off


def test_noop_update_leaves_the_next_launches_alone():
    grid, goal = cases.synthetic_map(1024, 1536, 0.20, seed=77)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as a, \
            MdpPathPlanning2d(grid, goal, cases.GAMMA) as b:
        for _ in range(8):
            a.sweeps(100)
            b.sweeps(100)
        ca, cb = a.work_counters(), b.work_counters()
        assert ca == cb
        b.update_map(grid.copy(), goal)
        for _ in range(2):
            a.sweeps(100, want_action=False)
            b.sweeps(100, want_action=False)
        assert np.array_equal(_bits(a.download()[0]), _bits(b.download()[0]))
        da = [x - y for x, y in zip(a.work_counters(), ca)]
        db = [x - y for x, y in zip(b.work_counters(), cb)]
        assert da == db


def test_staged_map_equals_the_copied_map():
    grid, goal = cases.synthetic_map(700, 1000, 0.20, seed=11)
    grid2, goal2 = _edit(grid, goal, "both", seed=3)
    pinned = torch.from_numpy(grid2.copy()).pin_memory().numpy()
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as a, \
            MdpPathPlanning2d(grid, goal, cases.GAMMA) as b:
        for m in (a, b):
            m.sweeps(300)
        a.stage_map(pinned)
        a.sweeps(100)
        b.sweeps(100)
        a.update_map(pinned, goal2)
        b.update_map(grid2, goal2)
        for what in ("right after the update", "100 sweeps later"):
            ja, aa = a.download()
            jb, ab = b.download()
            assert np.array_equal(_bits(ja), _bits(jb)), f"J differs {what}"
            assert np.array_equal(aa, ab), f"action differs {what}"
            assert a.residual() == b.residual()
            a.sweeps(100)
            b.sweeps(100)


def _crossing_edit(grid, goal, rows):
    """An edit over every shard boundary in `rows`, plus a goal move."""
    g = grid.copy()
    w = g.shape[1]
    for i, r in enumerate(rows):
        x = (97 * (i + 1)) % (w - 40)
        g[r - 12:r + 12, x:x + 30] = 1 if i % 2 == 0 else 0
        g[r - 3:r + 3, x + 34:x + 40] = 1 - g[r - 3:r + 3, x + 34:x + 40]
    goal2 = (goal[0] + 3, goal[1] + 2)
    g[goal2[1], goal2[0]] = 0
    return g, goal2


def _drive(handles, steps, exchange=None):
    for k, wa in steps:
        for m in handles:
            m.sweeps(k, wa)
        if exchange:
            exchange()


@pytest.mark.parametrize("devices,shape", [([0, 0, 0], (1539, 700)), ([0, 0], (1025, 700))])
def test_multi_shard_handle_equals_the_single_handle(devices, shape):
    """Shards of 513 rows: 8-row blocks and a last block of 1 row."""
    h, w = shape
    grid, goal = cases.synthetic_map(h, w, 0.2, seed=h + w)
    bounds = [h * i // len(devices) for i in range(1, len(devices))]
    grid2, goal2 = _crossing_edit(grid, goal, bounds)
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as one, \
            MdpPathPlanning2d(grid, goal, cases.GAMMA, devices=devices) as multi:
        assert not multi.peer_to_peer
        for m in (one, multi):
            m.valueIteration()
            m.sweeps(300)
            m.update_map(grid2, goal2)
        for k, wa in [(1, True), (2, False), (3, True), (100, True)]:
            for m in (one, multi):
                m.sweeps(k, wa)
            if wa:
                j1, a1 = one.download()
                j2, a2 = multi.download()
                assert np.array_equal(_bits(j1), _bits(j2)) and np.array_equal(a1, a2)
        assert one.residual() == multi.residual()
        for m in (one, multi):
            m.update_map(grid, goal)
        (n1, r1), (n2, r2) = one.valueIteration(), multi.valueIteration()
        assert n1 == n2 and np.array_equal(r1, r2)
        j1, a1 = one.download()
        j2, a2 = multi.download()
        assert np.array_equal(_bits(j1), _bits(j2)) and np.array_equal(a1, a2)
        run, total = multi.work_counters()
        assert run < total


def test_host_exchanged_shards_equal_the_single_handle():
    from path_planning_2d_b200.distributed import device_tensor
    grid, goal = cases.synthetic_map(150, 170, 0.2, seed=5)
    bounds = [0, 37, 39, 100, 150]
    grid2, goal2 = _crossing_edit(grid, goal, [38, 100])
    one = MdpPathPlanning2d(grid, goal, cases.GAMMA)
    shards = [MdpPathPlanning2d(grid, goal, cases.GAMMA, rows=(a, b))
              for a, b in zip(bounds[:-1], bounds[1:])]

    def exchange():
        halos = [s.halo() for s in shards]
        for i in range(len(shards) - 1):
            up, dn = halos[i], halos[i + 1]
            t = lambda p: device_tensor(p, up.bytes)
            t(dn.recv_top).copy_(t(up.send_bottom))
            t(up.recv_bottom).copy_(t(dn.send_top))
        torch.cuda.synchronize()

    steps = [(2, False)] * 60 + [(1, True), (2, True)]
    try:
        _drive(shards, steps, exchange)
        _drive([one], steps)
        for m in shards + [one]:
            m.update_map(grid2, goal2)
        _drive(shards, steps, exchange)
        _drive([one], steps)
        j1, a1 = one.download()
        assert np.array_equal(_bits(j1), _bits(np.concatenate([s.download()[0] for s in shards])))
        assert np.array_equal(a1, np.concatenate([s.download()[1] for s in shards]))
        assert one.residual() == max(s.residual() for s in shards)
    finally:
        one.close()
        for s in shards:
            s.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_peer_to_peer_multi_gpu_handle():
    grid, goal = cases.synthetic_map(2048, 1536, 0.20, seed=51)
    grid2, goal2 = _crossing_edit(grid, goal, [1024])
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as one, \
            MdpPathPlanning2d(grid, goal, cases.GAMMA, devices=2) as multi:
        for m in (one, multi):
            m.valueIteration()
            m.update_map(grid2, goal2)
        (n1, r1), (n2, r2) = one.valueIteration(), multi.valueIteration()
        assert n1 == n2 and np.array_equal(r1, r2)
        j1, a1 = one.download()
        j2, a2 = multi.download()
        assert np.array_equal(_bits(j1), _bits(j2)) and np.array_equal(a1, a2)


def test_errors_leave_the_handle_unchanged():
    grid, goal = cases.synthetic_map(90, 150, 0.3, seed=3)
    bad = grid.copy()
    other = (goal[0] + 5, goal[1])
    bad[other[1], other[0]] = 1
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as a, \
            MdpPathPlanning2d(grid, goal, cases.GAMMA) as b:
        a.sweeps(120)
        b.sweeps(120)
        with pytest.raises(_lib.Pp2dError) as e:
            a.update_map(bad, other)
        assert e.value.code == _lib.PP2D_ERR_GOAL_OCCUPIED
        with pytest.raises(_lib.Pp2dError) as e:
            a.update_map(grid, (150, 0))
        assert e.value.code == _lib.PP2D_ERR_INVALID
        assert a.goal == b.goal and a.sweep_count == b.sweep_count
        for m in (a, b):
            m.sweeps(3)
        ja, aa = a.download()
        jb, ab = b.download()
        assert np.array_equal(_bits(ja), _bits(jb)) and np.array_equal(aa, ab)
        assert a.residual() == b.residual()
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as c:
        c.policyIteration(max_rounds=1)
        with pytest.raises(_lib.Pp2dError) as e:
            c.update_map(grid, goal)
        assert e.value.code == _lib.PP2D_ERR_STATE


def test_cpp_update_map_matches_the_python_path(tmp_path):
    import cv2
    name = "sparse_map_100x40"
    goal, _ = cases.BUNDLED[name]
    png = os.path.join(cases.GOLDEN, "maps", name + "_rgb.png")
    img = cv2.imread(png, cv2.IMREAD_GRAYSCALE)
    _, grid = cv2.threshold(img, 250.0, 1.0, cv2.THRESH_BINARY_INV)
    grid = np.ascontiguousarray(grid, np.uint8)
    if grid[goal[1], goal[0]]:
        pytest.skip("noise fixture blocked the goal")
    grid2, goal2 = _edit(grid, goal, "both", seed=9)
    (tmp_path / "next.bin").write_bytes(grid2.tobytes())
    exe = str(tmp_path / "update_map")
    libdir = os.path.join(ROOT, "path_planning_2d_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-o", exe,
                    os.path.join(ROOT, "tests", "cpp", "update_map_main.cpp"), "-L", libdir,
                    "-lpp2d", "-lz", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([exe, png, str(goal[0]), str(goal[1]), "0.95", str(tmp_path / "next.bin"),
                          str(goal2[0]), str(goal2[1])], capture_output=True, text=True)
    line = [l for l in out.stdout.splitlines() if l.startswith("RESULT")]
    assert line, out.stdout + out.stderr
    kv = dict(t.split("=") for t in line[0].split()[1:])
    with MdpPathPlanning2d(grid, goal, cases.GAMMA) as mdp:
        n0, _ = mdp.valueIteration()
        mdp.update_map(grid2, goal2)
        n1, _ = mdp.valueIteration()
        cost, action = mdp.download()
    assert int(kv["sweeps0"]) == n0 and int(kv["sweeps"]) == n0 + n1
    assert kv["cost"] == fnv(np.ascontiguousarray(cost, np.float32).tobytes())
    assert kv["action"] == fnv(action.tobytes())
    bad = subprocess.run([exe, png, str(goal[0]), str(goal[1]), "0.95",
                          str(tmp_path / "next.bin"), "0", "0"] if grid2[0, 0] else
                         [exe, png, str(goal[0]), str(goal[1]), "0.95",
                          str(tmp_path / "next.bin"), "100", "0"],
                         capture_output=True, text=True)
    assert "UPDATE_FAILED" in bad.stdout
