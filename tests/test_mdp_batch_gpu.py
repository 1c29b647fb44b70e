"""GPU tier: MDP batches (pp2d_mdp_batch_*), many goals or maps of one size
solved together in one tall grid with occupied separator rows.

Every instance must compute bit for bit what a single handle computes on its
map and goal: J, actions, sweep counts and residuals, after any number of
sweeps and after the per-instance stopping rule; stopped instances are frozen
and stop costing work."""
import os
import subprocess

import numpy as np
import pytest

import cases
import oracle_py
from path_planning_2d_b200 import MdpBatchPathPlanning2d, MdpPathPlanning2d, _lib
from test_host_mirror import fnv

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAMMA = cases.GAMMA
STRIP = 60          # columns of a fused launch's strip (StripGeom<2, 2>::S)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _free_goals(grid):
    ys, xs = np.nonzero(grid == 0)
    return [(int(x), int(y)) for y, x in zip(ys, xs)]


def _seeded_goals(grid, n, seed):
    free = _free_goals(grid)
    rng = np.random.default_rng(seed)
    return [free[i] for i in rng.choice(len(free), size=n, replace=len(free) < n)]


def _random_map(h, w, p, seed):
    rng = np.random.default_rng(seed)
    return (rng.random((h, w)) < p).astype(np.uint8)


def _maze(h, w):
    """Serpentine corridor: walls on every other row with the gap alternating
    between the ends, so the cost-to-go field converges slowly."""
    grid = np.zeros((h, w), np.uint8)
    for i, y in enumerate(range(1, h - 1, 2)):
        grid[y, :] = 1
        grid[y, w - 1 if i % 2 == 0 else 0] = 0
    return grid


class Single:
    """What a user does today: one handle, reset per problem."""

    def __init__(self, shape):
        self.shape = shape
        self.mdp = None

    def _handle(self, grid, goal):
        if self.mdp is None:
            self.mdp = MdpPathPlanning2d(grid, goal, GAMMA)
        else:
            self.mdp.reset(grid, goal)
        return self.mdp

    def solve(self, grid, goal):
        mdp = self._handle(grid, goal)
        n, res = mdp.valueIteration()
        cost, action = mdp.download()
        return n, res, cost.copy(), action.copy()

    def close(self):
        if self.mdp is not None:
            self.mdp.close()


def _check_solve_against_single(maps, goals, batch_n, batch_res, cost, action, oracle=False):
    """Instance k of a solved batch equals a single handle's solve (and the
    CPU oracle's value_iteration when `oracle`)."""
    cache = {}
    single = Single(maps[0].shape)
    try:
        for k, goal in enumerate(goals):
            key = (id(maps[k]), goal)
            if key not in cache:
                cache[key] = single.solve(maps[k], goal)
            n, res, c, a = cache[key]
            assert batch_n[k] == n, f"instance {k} (goal {goal}): sweeps"
            assert np.array_equal(batch_res[k].view(np.uint64), res.view(np.uint64)), \
                f"instance {k}: residuals"
            assert np.array_equal(_bits(cost[k]), _bits(c)), f"instance {k}: J"
            assert np.array_equal(action[k], a), f"instance {k}: actions"
            if oracle:
                J, A, on, ores = oracle_py.value_iteration(maps[k], goal, GAMMA)
                assert on == n and np.array_equal(_bits(J), _bits(cost[k]))
                assert np.array_equal(A, action[k])
                assert np.array_equal(ores.view(np.uint64), res.view(np.uint64))
    finally:
        single.close()


def _solve(grid_maps, goals):
    with MdpBatchPathPlanning2d(grid_maps, goals, GAMMA) as b:
        n, res = b.valueIteration()
        assert np.array_equal(b.sweep_counts(), n)
        cost, action = b.download()
        work = b.work_counters()
    return n, res, cost, action, work


# -- 1. multi-goal on each bundled map ----------------------------------------
@pytest.mark.parametrize("name", ["map_3x3", "map_5x5", "map_10x10", "map_100x40",
                                  "sparse_map_100x40"])
def test_multi_goal_on_bundled_maps(name):
    grid = cases.load_bundled(name)
    small = grid.size <= 100
    goals = _free_goals(grid) if small else _seeded_goals(grid, 64, seed=7)
    n, res, cost, action, _ = _solve(grid, goals)
    _check_solve_against_single([grid] * len(goals), goals, n, res, cost, action, oracle=small)


# -- 2. different maps per instance ---------------------------------------------
def _mixed_maps(h=24, w=70):
    """Random maps of several densities and a corridor.  Maps with an
    occupied cell stop at the sweep count where the occupied cells' closed form
    settles; the empty maps (densities 0) stop earlier."""
    maps, goals = [], []
    for i, p in enumerate([0.0, 0.08, 0.15, 0.25, 0.3, 0.0, 0.05, 0.2]):
        g = _random_map(h, w, p, seed=100 + i)
        goal = (int(3 + 7 * i) % w, int(2 + 3 * i) % h)
        g[goal[1], goal[0]] = 0
        maps.append(g)
        goals.append(goal)
    maze = _maze(h, w)
    maps.append(maze)
    goals.append((0, 0))
    return np.stack(maps), goals


def test_different_maps_per_instance():
    maps, goals = _mixed_maps()
    n, res, cost, action, _ = _solve(maps, goals)
    assert len(set(int(v) for v in n)) >= 2, f"one sweep count for all: {n}"
    _check_solve_against_single(list(maps), goals, n, res, cost, action)


# -- 3. step semantics ------------------------------------------------------------
@pytest.mark.parametrize("steps", [[1], [2], [3], [100], [1, 2, 100]])
def test_sweeps_and_residual_equal_the_oracle_and_the_single_handle(steps):
    maps, goals = _mixed_maps(h=12, w=20)
    K = len(goals)
    oracles = [oracle_py.OracleMdp(maps[k], goals[k], GAMMA) for k in range(K)]
    singles = [MdpPathPlanning2d(maps[k], goals[k], GAMMA) for k in range(K)]
    try:
        with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
            done = 0
            for s in steps:
                b.sweeps(s)
                done += s
                cost, action = b.download()
                assert np.array_equal(b.sweep_counts(), [done] * K)
                r = b.residual()
                for k in range(K):
                    oracles[k].sweeps(s)
                    singles[k].sweeps(s)
                    assert np.array_equal(_bits(cost[k]), _bits(oracles[k].cost)), (k, done)
                    assert np.array_equal(action[k], oracles[k].act), (k, done)
                    assert _bits(r[k]) == _bits(singles[k].residual()), (k, done)
    finally:
        for s in singles:
            s.close()


# -- 4. edge shapes -------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(1, 17), (23, 1), (2, 2)])
def test_edge_shapes(shape):
    h, w = shape
    grid = _random_map(h, w, 0.2, seed=h * 100 + w)
    if grid.min() == 1:
        grid[0, 0] = 0
    goals = _free_goals(grid)
    n, res, cost, action, _ = _solve(grid, goals)
    _check_solve_against_single([grid] * len(goals), goals, n, res, cost, action, oracle=True)
    # and after a few single steps
    with MdpBatchPathPlanning2d(grid, goals, GAMMA) as b:
        b.sweeps(3)
        cost, action = b.download()
    for k, goal in enumerate(goals):
        ora = oracle_py.OracleMdp(grid, goal, GAMMA)
        ora.sweeps(3)
        assert np.array_equal(_bits(cost[k]), _bits(ora.cost))
        assert np.array_equal(action[k], ora.act)


def test_one_instance_equals_the_single_handle():
    name = "sparse_map_100x40"
    grid = cases.load_bundled(name)
    goal, _ = cases.BUNDLED[name]
    n, res, cost, action, _ = _solve(grid[None], [goal])
    _check_solve_against_single([grid], [goal], n, res, cost, action)


def test_4096_goals_on_10x10():
    grid = cases.load_bundled("map_10x10")
    goals = _seeded_goals(grid, 4096, seed=3)
    n, res, cost, action, work = _solve(grid, goals)
    assert work[1] > 0
    _check_solve_against_single([grid] * len(goals), goals, n, res, cost, action)


# -- 5. freezing ----------------------------------------------------------------------
def _with_env(env, fn):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return fn()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _staggered_batch():
    """Six empty maps, which stop early, and one corridor, which runs on
    alone (its occupied cells keep its residual up)."""
    h, w = 30, 100
    maps = [np.zeros((h, w), np.uint8) for _ in range(6)]
    goals = [(w // 2 + 3 * i, h // 2) for i in range(6)]
    maps.append(_maze(h, w))
    goals.append((0, 0))
    return np.stack(maps), goals


def test_freezing_cuts_the_work_and_stays_exact():
    maps, goals = _staggered_batch()
    K, H, W = maps.shape
    rpu = 8
    n, res, cost, action, (run, launched) = _with_env(
        {"PP2D_MDP_ROWS_PER_UNIT": str(rpu)}, lambda: _solve(maps, goals))
    assert len(set(int(v) for v in n)) >= 2, n
    rows = K * (H + 1) - 1
    n_rb = -(-rows // rpu)
    n_strips = -(-W // STRIP)
    n_units = n_rb * n_strips
    assert launched % n_units == 0
    batches = int(max(n)) // 100
    assert launched == batches * 50 * n_units
    # Bound per fused launch of batch b: the row blocks that hold a row of an
    # instance still running, and one block on each side of them.  The first
    # launch of the solve and the arg-min launch that ends each batch run
    # every unit.
    bound_total = 0
    tight = 0
    for bt in range(batches):
        blocks = set()
        for k in range(K):
            if n[k] > 100 * bt:
                r0, r1 = k * (H + 1), k * (H + 1) + H
                for rb in range(r0 // rpu - 1, (r1 - 1) // rpu + 2):
                    if 0 <= rb < n_rb:
                        blocks.add(rb)
        bound = len(blocks) * n_strips
        launches_bounded = 48 if bt == 0 else 49
        bound_total += launches_bounded * bound + (50 - launches_bounded) * n_units
        if sum(1 for k in range(K) if n[k] > 100 * bt) == 1:
            tight += 1
            assert bound < n_units // 2
    assert tight >= 1, "no batch with a single running instance"
    assert run <= bound_total, (run, bound_total, launched)
    # the same batch without unit skipping computes the same bits
    n0, res0, cost0, action0, (run0, launched0) = _with_env(
        {"PP2D_MDP_ROWS_PER_UNIT": str(rpu), "PP2D_MDP_SKIP": "0"},
        lambda: _solve(maps, goals))
    assert run0 == launched0 == launched
    assert np.array_equal(n0, n)
    for k in range(K):
        assert np.array_equal(res0[k].view(np.uint64), res[k].view(np.uint64))
    assert np.array_equal(_bits(cost0), _bits(cost))
    assert np.array_equal(action0, action)
    _check_solve_against_single(list(maps), goals, n, res, cost, action)


# -- 6. plan and waypoints ------------------------------------------------------------
def test_plan_and_waypoints_equal_the_oracle_on_the_instance_grid():
    maps, goals = _mixed_maps(h=16, w=30)
    K, H, W = maps.shape
    rng = np.random.default_rng(5)
    with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
        for phase in ("live", "frozen"):
            if phase == "live":
                b.sweeps(7)
            else:
                b.valueIteration()
            _, action = b.download()
            idx = rng.integers(0, K, size=40)
            beliefs = rng.random((40, H * W), dtype=np.float32)
            beliefs[::5] = 0.0                    # all-zero beliefs: index 0
            got = b.plan_batch(idx, beliefs)
            assert b.plan_batch([], np.empty((0, H * W), np.float32)).shape == (0,)
            for i in range(40):
                assert got[i] == oracle_py.plan(beliefs[i], action[idx[i]]), (phase, i)
            for k in range(K):
                free = np.argwhere(maps[k] == 0)
                y, x = free[rng.integers(len(free))]
                start = (int(x), int(y))
                assert np.array_equal(b.waypoints(k, start),
                                      oracle_py.waypoints(action[k], start)), (phase, k)
                assert np.array_equal(b.waypoints(k, start, max_len=3),
                                      oracle_py.waypoints(action[k], start, 3))


# -- 7. reset ----------------------------------------------------------------------------
def test_reset_equals_a_fresh_batch():
    maps, goals = _mixed_maps(h=16, w=30)
    maps2 = maps[::-1].copy()
    goals2 = goals[::-1]
    with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
        b.valueIteration()
        b.reset(maps2, goals2)
        assert np.array_equal(b.sweep_counts(), np.zeros(len(goals)))
        n, res = b.valueIteration()
        cost, action = b.download()
        # shared-map reset on the same handle
        b.reset(maps2[0], [goals2[0]] * len(goals))
        b.sweeps(5)
        c5, a5 = b.download()
    n_f, res_f, cost_f, action_f, _ = _solve(maps2, goals2)
    assert np.array_equal(n, n_f)
    for k in range(len(goals)):
        assert np.array_equal(res[k].view(np.uint64), res_f[k].view(np.uint64))
    assert np.array_equal(_bits(cost), _bits(cost_f))
    assert np.array_equal(action, action_f)
    ora = oracle_py.OracleMdp(maps2[0], goals2[0], GAMMA)
    ora.sweeps(5)
    for k in range(len(goals)):
        assert np.array_equal(_bits(c5[k]), _bits(ora.cost))
        assert np.array_equal(a5[k], ora.act)


def test_reset_from_a_shared_map_to_one_map_per_instance():
    """A batch created on one shared map keeps room for one map per instance:
    a reset with per-instance maps equals a fresh batch on them, and so does
    a reset back to a shared map."""
    maps, goals = _mixed_maps(h=16, w=30)
    K = len(goals)
    shared = maps[1]
    shared_goals = [g for g in _free_goals(shared)[:K]]
    with MdpBatchPathPlanning2d(shared, shared_goals, GAMMA) as b:
        b.sweeps(3)
        b.reset(maps, goals)
        n, res = b.valueIteration()
        cost, action = b.download()
        b.reset(shared, shared_goals)
        n2, _ = b.valueIteration()
        cost2, action2 = b.download()
    n_f, res_f, cost_f, action_f, _ = _solve(maps, goals)
    assert np.array_equal(n, n_f)
    for k in range(K):
        assert np.array_equal(res[k].view(np.uint64), res_f[k].view(np.uint64))
    assert np.array_equal(_bits(cost), _bits(cost_f))
    assert np.array_equal(action, action_f)
    n_s, _, cost_s, action_s, _ = _solve(shared, shared_goals)
    assert np.array_equal(n2, n_s)
    assert np.array_equal(_bits(cost2), _bits(cost_s))
    assert np.array_equal(action2, action_s)


# -- 8. state and errors ------------------------------------------------------------------
def test_state_and_errors():
    maps, goals = _mixed_maps(h=12, w=20)
    K, H, W = maps.shape
    lib = _lib.load()
    with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
        b.sweeps(4)
        with pytest.raises(_lib.Pp2dError) as e:
            b.download(range(K - 1, K + 1))
        assert e.value.code == _lib.PP2D_ERR_INVALID
        with pytest.raises(_lib.Pp2dError) as e:
            b.download(K)
        assert e.value.code == _lib.PP2D_ERR_INVALID
        with pytest.raises(_lib.Pp2dError) as e:
            b.plan_batch([0, K], np.ones((2, H * W), np.float32))
        assert e.value.code == _lib.PP2D_ERR_INVALID
        with pytest.raises(_lib.Pp2dError) as e:
            b.waypoints(K, (0, 0))
        assert e.value.code == _lib.PP2D_ERR_INVALID
        with pytest.raises(_lib.Pp2dError) as e:
            b.waypoints(0, (W, 0))
        assert e.value.code == _lib.PP2D_ERR_INVALID
        n, _ = b.valueIteration()
        before = b.download()
        for call in (lambda: b.sweeps(1), lambda: b.valueIteration(), lambda: b.residual()):
            with pytest.raises(_lib.Pp2dError) as e:
                call()
            assert e.value.code == _lib.PP2D_ERR_STATE
        # a failed reset (occupied goal of instance 2) changes nothing
        bad = maps.copy()
        bad_goals = list(goals)
        bad[2, 1, 1] = 1
        bad_goals[2] = (1, 1)
        with pytest.raises(_lib.Pp2dError) as e:
            b.reset(bad, bad_goals)
        assert e.value.code == _lib.PP2D_ERR_GOAL_OCCUPIED
        assert "instance 2" in str(e.value)
        assert lib.pp2d_mdp_batch_reset(b._h, maps.ctypes.data, 0, None) == \
            _lib.PP2D_ERR_INVALID
        after = b.download()
        assert np.array_equal(b.sweep_counts(), n + 4)     # the 4 sweeps before the solve count
        assert np.array_equal(_bits(before[0]), _bits(after[0]))
        assert np.array_equal(before[1], after[1])
        with pytest.raises(_lib.Pp2dError) as e:
            b.sweeps(1)
        assert e.value.code == _lib.PP2D_ERR_STATE


# -- 9. C++ class --------------------------------------------------------------------------
def test_cpp_batch_matches_the_python_path(tmp_path):
    maps, goals = _mixed_maps(h=16, w=30)
    K, H, W = maps.shape
    (tmp_path / "maps.bin").write_bytes(maps.tobytes())
    (tmp_path / "goals.bin").write_bytes(np.asarray(goals, np.uint32).tobytes())
    exe = str(tmp_path / "batch_main")
    libdir = os.path.join(ROOT, "path_planning_2d_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-o", exe,
                    os.path.join(ROOT, "tests", "cpp", "batch_main.cpp"), "-L", libdir,
                    "-lpp2d", "-lz", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([exe, str(tmp_path / "maps.bin"), str(H), str(W),
                          str(tmp_path / "goals.bin"), "0.95"], capture_output=True, text=True)
    lines = [l for l in out.stdout.splitlines() if l.startswith("RESULT")]
    assert len(lines) == K, out.stdout + out.stderr
    n, res, cost, action, _ = _solve(maps, goals)
    for k, line in enumerate(lines):
        kv = dict(t.split("=") for t in line.split()[1:])
        assert int(kv["k"]) == k
        assert int(kv["sweeps"]) == n[k] and int(kv["batches"]) == len(res[k])
        assert kv["cost"] == fnv(np.ascontiguousarray(cost[k], np.float32).tobytes())
        assert kv["action"] == fnv(action[k].tobytes())
