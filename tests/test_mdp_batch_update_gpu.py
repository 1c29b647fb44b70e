"""GPU tier: pp2d_mdp_batch_update, re-planning chosen instances of a batch
on a changed map or goal from their previous solutions.

Every listed instance must compute bit for bit what a single handle computes
when it solves, calls update_map and solves again: sweeps, residuals, J,
actions and sweep counts.  Unlisted instances stay bit for bit as they were,
and instances that a solve froze are re-activated from their results."""
import os
import subprocess

import numpy as np
import pytest

import cases
from path_planning_2d_b200 import MdpBatchPathPlanning2d, MdpPathPlanning2d, _lib
from test_host_mirror import fnv
from test_mdp_batch_gpu import Single, _mixed_maps, _staggered_batch
from test_mdp_update_gpu import KINDS, _edit, _jprime, _oracle_from

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAMMA = cases.GAMMA
STRIP = 60          # columns of a fused launch's strip (StripGeom<2, 2>::S)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _free_goals(grid, n, seed):
    free = np.argwhere(grid == 0)
    rng = np.random.default_rng(seed)
    pick = rng.choice(len(free), size=n, replace=len(free) < n)
    return [(int(free[i][1]), int(free[i][0])) for i in pick]


def _update_args(grids, goals, listed, kind, shared, seed):
    """(maps2, goals2) for the listed instances: one edit of `kind` for all
    of them (shared: an (H, W) map; a listed goal that the edit occupies, or
    any goal for kind goal_move, moves to a free cell) or one edit each
    ((n, H, W))."""
    if not shared:
        pairs = [_edit(grids[k], goals[k], kind, seed + 7 * k) for k in listed]
        return np.stack([m for m, _ in pairs]), [g for _, g in pairs]
    g2, first = _edit(grids[listed[0]], goals[listed[0]], kind, seed)
    free = np.argwhere(g2 == 0)
    rng = np.random.default_rng(seed)
    goals2 = [first]
    for k in listed[1:]:
        gx, gy = goals[k]
        if kind == "goal_move" or g2[gy, gx] != 0:
            y, x = free[rng.integers(len(free))]
            gx, gy = int(x), int(y)
        goals2.append((gx, gy))
    return g2, goals2


def _map_of(maps2, i):
    return maps2 if maps2.ndim == 2 else maps2[i]


class Replanned:
    """One single handle per instance: solve, then update_map and solve for
    each round the instance is listed in."""

    def __init__(self, grids, goals):
        self.h = [MdpPathPlanning2d(grids[k], goals[k], GAMMA) for k in range(len(goals))]
        for m in self.h:
            m.valueIteration()

    def update(self, k, grid, goal):
        m = self.h[k]
        m.update_map(grid, goal)
        n, res = m.valueIteration()
        cost, action = m.download()
        return n, res, cost.copy(), action.copy(), m.sweep_count

    def close(self):
        for m in self.h:
            m.close()


def _observe(b, rng_seed=0):
    """Everything a user can read from each instance: download, sweep
    counts, a plan and a way-point list per instance."""
    cost, action = b.download()
    K, H, W = cost.shape
    rng = np.random.default_rng(rng_seed)
    beliefs = rng.random((K, H * W), dtype=np.float32)
    plans = b.plan_batch(np.arange(K), beliefs)
    paths = [b.waypoints(k, (int(rng.integers(W)), int(rng.integers(H)))) for k in range(K)]
    return _bits(cost).copy(), action.copy(), b.sweep_counts().copy(), plans, paths


def _assert_unchanged(before, after, ks, what=""):
    for k in ks:
        assert np.array_equal(before[0][k], after[0][k]), f"instance {k}: J {what}"
        assert np.array_equal(before[1][k], after[1][k]), f"instance {k}: actions {what}"
        assert before[2][k] == after[2][k], f"instance {k}: sweep count {what}"
        assert before[3][k] == after[3][k], f"instance {k}: plan {what}"
        assert np.array_equal(before[4][k], after[4][k]), f"instance {k}: way-points {what}"


def _check_round(b, singles, listed, maps2, goals2, n, res, cost, action):
    """Listed instance k equals its single handle after update_map + solve;
    the others did not run in this solve."""
    counts = b.sweep_counts()
    for i, k in enumerate(listed):
        sn, sres, sc, sa, scount = singles.update(k, _map_of(maps2, i), goals2[i])
        assert n[k] == sn, f"instance {k}: sweeps"
        assert np.array_equal(res[k].view(np.uint64), np.asarray(sres).view(np.uint64)), \
            f"instance {k}: residuals"
        assert np.array_equal(_bits(cost[k]), _bits(sc)), f"instance {k}: J"
        assert np.array_equal(action[k], sa), f"instance {k}: actions"
        assert counts[k] == scount, f"instance {k}: sweep count"
    for k in set(range(len(n))) - set(listed):
        assert n[k] == 0 and len(res[k]) == 0, f"unlisted instance {k} ran"


# -- 1. parity with single handles ----------------------------------------------
def _bundled(name):
    return cases.load_bundled(name)


def _tiny(h, w, seed):
    grid, _ = cases.synthetic_map(h, w, 0.3, seed=seed, goal=(0, 0))
    return grid


BASE = {
    "map_100x40": lambda: _bundled("map_100x40"),
    "sparse_map_100x40": lambda: _bundled("sparse_map_100x40"),
    "syn_1x17": lambda: _tiny(1, 17, 17),
    "syn_2x2": lambda: _tiny(2, 2, 22),
}
PARITY = [(m, k, s) for m in ("map_100x40", "sparse_map_100x40") for k in KINDS
          for s in ("shared", "per_instance")] + \
         [(m, k, s) for m in ("syn_1x17", "syn_2x2") for k in ("add", "remove", "goal_move", "noop")
          for s in ("shared", "per_instance")]


@pytest.mark.parametrize("name,kind,mode", PARITY)
def test_update_matches_single_handles(name, kind, mode):
    grid = BASE[name]()
    K = 8 if grid.size > 100 else 4
    goals = _free_goals(grid, K, seed=len(name) + K)
    listed = [K - 3, 1, K - 1, K // 2] if K > 4 else [3, 0]
    shared = mode == "shared"
    grids = [grid] * K
    seed = 31 * len(name) + KINDS.index(kind)
    maps2, goals2 = _update_args(grids, goals, listed, kind, shared, seed)
    singles = Replanned(grids, goals)
    try:
        create_maps = grid if shared else np.stack(grids)
        with MdpBatchPathPlanning2d(create_maps, goals, GAMMA) as b:
            b.valueIteration()
            before = _observe(b)
            b.update_map(listed, maps2, goals2)
            # the J' rule, and the action grid left as it was
            after = _observe(b)
            for i, k in enumerate(listed):
                want = _jprime(before[0][k].view(np.float32), _map_of(maps2, i), goals2[i],
                               int(before[2][k]))
                assert np.array_equal(after[0][k], _bits(want)), f"instance {k}: J'"
            for k in range(K):
                assert np.array_equal(before[1][k], after[1][k])
                assert before[2][k] == after[2][k]
                assert before[3][k] == after[3][k]
                assert np.array_equal(before[4][k], after[4][k])
            unlisted = [k for k in range(K) if k not in listed]
            _assert_unchanged(before, after, unlisted, "after the update")
            n, res = b.valueIteration()
            cost, action = b.download()
            _check_round(b, singles, listed, maps2, goals2, n, res, cost, action)
            _assert_unchanged(before, _observe(b), unlisted, "after the solve")
    finally:
        singles.close()


# -- 2. different stop counts ----------------------------------------------------
def test_early_and_late_stopped_instances_in_one_call():
    maps, goals = _staggered_batch()
    K = len(goals)
    singles = Replanned(list(maps), goals)
    try:
        with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
            n0, _ = b.valueIteration()
            listed = [K - 1, 0, 3]
            assert len({int(n0[k]) for k in listed}) >= 2, n0
            pairs = [_edit(maps[K - 1], goals[K - 1], "goal_move", 3),
                     _edit(maps[0], goals[0], "add", 4),
                     _edit(maps[3], goals[3], "noop", 5)]
            maps2 = np.stack([m for m, _ in pairs])
            goals2 = [g for _, g in pairs]
            b.update_map(listed, maps2, goals2)
            n, res = b.valueIteration()
            cost, action = b.download()
            _check_round(b, singles, listed, maps2, goals2, n, res, cost, action)
    finally:
        singles.close()


# -- 3. the J' rule on instances frozen at different counts ----------------------
def test_jprime_rule_and_unchanged_actions():
    maps, goals = _mixed_maps(h=16, w=30)
    K, H, W = maps.shape
    with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
        n0, _ = b.valueIteration()
        assert len(set(int(v) for v in n0)) >= 2
        before = _observe(b, 9)
        listed = list(range(K))[::-1]
        pairs = [_edit(maps[k], goals[k], "both" if (maps[k] == 1).any() else "add", 40 + k)
                 for k in listed]
        maps2 = np.stack([m for m, _ in pairs])
        goals2 = [g for _, g in pairs]
        b.update_map(listed, maps2, goals2)
        after = _observe(b, 9)
        for i, k in enumerate(listed):
            want = _jprime(before[0][k].view(np.float32), maps2[i], goals2[i], int(n0[k]))
            assert np.array_equal(after[0][k], _bits(want)), f"instance {k}: J'"
            assert np.array_equal(after[1][k], before[1][k])
            assert after[3][k] == before[3][k]
            assert np.array_equal(after[4][k], before[4][k])
        assert np.array_equal(after[2], n0)
        # every instance is active again: sweeps work, each from its own count
        b.sweeps(3)
        assert np.array_equal(b.sweep_counts(), n0 + 3)
        cost, action = b.download()
        for i, k in enumerate(listed):
            want = _jprime(before[0][k].view(np.float32), maps2[i], goals2[i], int(n0[k]))
            ora = _oracle_from(maps2[i], goals2[i], want, int(n0[k]))
            ora.sweeps(3)
            assert np.array_equal(_bits(cost[k]), _bits(ora.cost)), k
            assert np.array_equal(action[k], ora.act), k


# -- 4. update before any solve ------------------------------------------------------
def test_update_on_a_live_batch_then_steps():
    maps, goals = _mixed_maps(h=12, w=20)
    K = len(goals)
    listed = [6, 2, 8]
    pairs = [_edit(maps[k], goals[k], kind, 60 + k)
             for k, kind in zip(listed, ("goal_move", "add", "near_goal"))]
    maps2 = np.stack([m for m, _ in pairs])
    goals2 = [g for _, g in pairs]
    singles = [MdpPathPlanning2d(maps[k], goals[k], GAMMA) for k in range(K)]
    try:
        with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
            b.sweeps(5)
            r = b.residual()
            prev = b.download()[0].copy()
            b.update_map(listed, maps2, goals2)
            oras = {}
            for k in range(K):
                singles[k].sweeps(5)
                assert _bits(singles[k].residual()) == _bits(r[k])
                if k in listed:
                    i = listed.index(k)
                    singles[k].update_map(maps2[i], goals2[i])
                    oras[k] = _oracle_from(maps2[i], goals2[i],
                                           _jprime(prev[k], maps2[i], goals2[i], 5), 5)
                else:
                    oras[k] = _oracle_from(maps[k], goals[k], prev[k], 5)
            done = 5
            for s in (1, 2, 3, 100):
                b.sweeps(s)
                done += s
                cost, action = b.download()
                assert np.array_equal(b.sweep_counts(), [done] * K)
                r = b.residual()
                for k in range(K):
                    oras[k].sweeps(s)
                    singles[k].sweeps(s)
                    assert np.array_equal(_bits(cost[k]), _bits(oras[k].cost)), (k, done)
                    assert np.array_equal(action[k], oras[k].act), (k, done)
                    assert _bits(r[k]) == _bits(singles[k].residual()), (k, done)
    finally:
        for s in singles:
            s.close()


# -- 5. work ---------------------------------------------------------------------------
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


def _one_instance_replan(maps, goals, k, map2, goal2):
    with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
        b.valueIteration()
        w0 = b.work_counters()
        b.update_map([k], map2[None], [goal2])
        n, res = b.valueIteration()
        w1 = b.work_counters()
        cost, action = b.download()
    return n, res, cost, action, (w1[0] - w0[0], w1[1] - w0[1])


def test_one_instance_update_runs_only_its_units():
    maps, goals = _staggered_batch()
    K, H, W = maps.shape
    k = 2
    map2, goal2 = _edit(maps[k], goals[k], "add", 8)
    rpu = 8
    n, res, cost, action, (run, launched) = _with_env(
        {"PP2D_MDP_ROWS_PER_UNIT": str(rpu)},
        lambda: _one_instance_replan(maps, goals, k, map2, goal2))
    rows = K * (H + 1) - 1
    n_rb = -(-rows // rpu)
    n_strips = -(-W // STRIP)
    n_units = n_rb * n_strips
    batches = int(n[k]) // 100
    assert batches >= 1 and launched == batches * 50 * n_units
    # value-only launches: the row blocks of instance k and one on each side;
    # the arg-min launch that ends each batch of 100 runs every unit
    r0, r1 = k * (H + 1), k * (H + 1) + H
    blocks = [rb for rb in range(r0 // rpu - 1, (r1 - 1) // rpu + 2) if 0 <= rb < n_rb]
    bound = len(blocks) * n_strips
    assert bound < n_units // 2
    assert run <= batches * (49 * bound + n_units), (run, bound, n_units, launched)
    # the same without unit skipping
    n0, res0, cost0, action0, (run0, launched0) = _with_env(
        {"PP2D_MDP_ROWS_PER_UNIT": str(rpu), "PP2D_MDP_SKIP": "0"},
        lambda: _one_instance_replan(maps, goals, k, map2, goal2))
    assert run0 == launched0 == launched
    assert np.array_equal(n0, n)
    assert np.array_equal(res0[k].view(np.uint64), res[k].view(np.uint64))
    assert np.array_equal(_bits(cost0), _bits(cost))
    assert np.array_equal(action0, action)
    # and the single handle
    with MdpPathPlanning2d(maps[k], goals[k], GAMMA) as m:
        m.valueIteration()
        m.update_map(map2, goal2)
        sn, sres = m.valueIteration()
        sc, sa = m.download()
    assert n[k] == sn and np.array_equal(res[k].view(np.uint64), sres.view(np.uint64))
    assert np.array_equal(_bits(cost[k]), _bits(sc)) and np.array_equal(action[k], sa)


# -- 6. several rounds, then a reset ------------------------------------------------------
def test_several_rounds_then_reset():
    maps, goals = _mixed_maps(h=16, w=30)
    K = len(goals)
    grids = list(maps)
    cur_maps, cur_goals = list(maps), list(goals)
    singles = Replanned(grids, goals)
    try:
        with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
            b.valueIteration()
            rounds = [([1, 3], "both", False), ([3, 5, 8], "goal_move", False),
                      (list(range(K)), "add", True), ([0], "noop", False)]
            for r, (listed, kind, shared) in enumerate(rounds):
                if shared:
                    # one costmap edit for the whole fleet (instance 0's map)
                    m2, g0 = _edit(cur_maps[0], cur_goals[0], kind, 90 + r)
                    maps2 = m2
                    goals2 = [g if m2[g[1], g[0]] == 0 else g0 for g in cur_goals]
                    goals2[0] = g0
                else:
                    maps2, goals2 = _update_args(cur_maps, cur_goals, listed, kind, False, 90 + r)
                before = _observe(b, r)
                b.update_map(listed, maps2, goals2)
                n, res = b.valueIteration()
                cost, action = b.download()
                _check_round(b, singles, listed, maps2, goals2, n, res, cost, action)
                _assert_unchanged(before, _observe(b, r),
                                  [k for k in range(K) if k not in listed], f"round {r}")
                for i, k in enumerate(listed):
                    cur_maps[k] = _map_of(maps2, i)
                    cur_goals[k] = goals2[i]
            # a reset afterwards equals a fresh batch
            b.reset(maps, goals)
            assert np.array_equal(b.sweep_counts(), np.zeros(K))
            n, res = b.valueIteration()
            cost, action = b.download()
        with MdpBatchPathPlanning2d(maps, goals, GAMMA) as f:
            n_f, res_f = f.valueIteration()
            cost_f, action_f = f.download()
        assert np.array_equal(n, n_f)
        for k in range(K):
            assert np.array_equal(res[k].view(np.uint64), res_f[k].view(np.uint64))
        assert np.array_equal(_bits(cost), _bits(cost_f))
        assert np.array_equal(action, action_f)
    finally:
        singles.close()


# -- 7. errors and state --------------------------------------------------------------------
def test_errors_leave_the_handle_unchanged_and_state_rules():
    maps, goals = _mixed_maps(h=12, w=20)
    K, H, W = maps.shape
    lib = _lib.load()
    with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
        b.valueIteration()
        before = _observe(b)
        g = np.asarray(goals, np.uint32)

        def refused(code, instances, m, gl, words=()):
            with pytest.raises(_lib.Pp2dError) as e:
                b.update_map(instances, m, gl)
            assert e.value.code == code, str(e.value)
            for w in words:
                assert w in str(e.value), str(e.value)

        refused(_lib.PP2D_ERR_INVALID, [K], maps[0], [goals[0]])
        refused(_lib.PP2D_ERR_INVALID, [2, 5, 2], maps[0], [goals[0]] * 3, ["instance 2"])
        out = [(W, 0)]
        refused(_lib.PP2D_ERR_INVALID, [4], maps[4], out, ["instance 4", "outside"])
        occ = maps[6].copy()
        occ[goals[6][1], goals[6][0]] = 1
        refused(_lib.PP2D_ERR_GOAL_OCCUPIED, [1, 6], np.stack([maps[1], occ]),
                [goals[1], goals[6]], ["instance 6", "occupied"])
        # a shared map: the goal of the second listed instance is occupied there
        shared = maps[0].copy()
        shared[goals[3][1], goals[3][0]] = 1
        shared[goals[0][1], goals[0][0]] = 0
        refused(_lib.PP2D_ERR_GOAL_OCCUPIED, [0, 3], shared, [goals[0], goals[3]], ["instance 3"])
        idx = np.array([0, 1], np.uint32)
        two = np.ascontiguousarray(maps[:2])
        for args in ((None, idx.ctypes.data, 2, two.ctypes.data, H * W, g.ctypes.data),
                     (b._h, None, 2, two.ctypes.data, H * W, g.ctypes.data),
                     (b._h, idx.ctypes.data, 2, None, H * W, g.ctypes.data),
                     (b._h, idx.ctypes.data, 2, two.ctypes.data, H * W, None),
                     (b._h, idx.ctypes.data, 2, two.ctypes.data, H * W - 1, g.ctypes.data)):
            assert lib.pp2d_mdp_batch_update(*args) == _lib.PP2D_ERR_INVALID
        assert lib.pp2d_mdp_batch_update(b._h, idx.ctypes.data, 0, two.ctypes.data, 0,
                                         g.ctypes.data) == _lib.PP2D_OK
        _assert_unchanged(before, _observe(b), range(K), "after a refused update")
        # every instance frozen: nothing to solve, no sweeps, no residual
        for call in (lambda: b.valueIteration(), lambda: b.sweeps(1), lambda: b.residual()):
            with pytest.raises(_lib.Pp2dError) as e:
                call()
            assert e.value.code == _lib.PP2D_ERR_STATE
        # one instance active again: solve runs it; sweeps and residual still
        # refuse while the others are frozen
        b.update_map([5], maps[5], [goals[5]])
        for call in (lambda: b.sweeps(1), lambda: b.residual()):
            with pytest.raises(_lib.Pp2dError) as e:
                call()
            assert e.value.code == _lib.PP2D_ERR_STATE
        n, res = b.valueIteration()
        assert n[5] > 0 and all(n[k] == 0 for k in range(K) if k != 5)
        with pytest.raises(_lib.Pp2dError) as e:
            b.valueIteration()
        assert e.value.code == _lib.PP2D_ERR_STATE


# -- 8. C++ ------------------------------------------------------------------------------------
def test_cpp_update_map_matches_the_python_path(tmp_path):
    maps, goals = _mixed_maps(h=16, w=30)
    K, H, W = maps.shape
    listed = [7, 0, 4]
    maps2, goals2 = _update_args(list(maps), goals, listed, "both", False, 77)
    files = {"maps": maps, "goals": np.asarray(goals, np.uint32),
             "instances": np.asarray(listed, np.uint32), "maps2": maps2,
             "goals2": np.asarray(goals2, np.uint32)}
    for name, arr in files.items():
        (tmp_path / f"{name}.bin").write_bytes(np.ascontiguousarray(arr).tobytes())
    exe = str(tmp_path / "batch_update_main")
    libdir = os.path.join(ROOT, "path_planning_2d_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-o", exe,
                    os.path.join(ROOT, "tests", "cpp", "batch_update_main.cpp"), "-L", libdir,
                    "-lpp2d", "-lz", f"-Wl,-rpath,{libdir}"], check=True)
    f = {name: str(tmp_path / f"{name}.bin") for name in files}
    out = subprocess.run([exe, f["maps"], str(H), str(W), f["goals"], "0.95", f["instances"],
                          f["maps2"], f["goals2"]], capture_output=True, text=True)
    lines = [l for l in out.stdout.splitlines() if l.startswith("RESULT")]
    assert len(lines) == K, out.stdout + out.stderr
    with MdpBatchPathPlanning2d(maps, goals, GAMMA) as b:
        b.valueIteration()
        b.update_map(listed, maps2, goals2)
        n, res = b.valueIteration()
        cost, action = b.download()
    for k, line in enumerate(lines):
        kv = dict(t.split("=") for t in line.split()[1:])
        assert int(kv["k"]) == k
        assert int(kv["sweeps"]) == n[k] and int(kv["batches"]) == len(res[k])
        assert kv["cost"] == fnv(np.ascontiguousarray(cost[k], np.float32).tobytes())
        assert kv["action"] == fnv(action[k].tobytes())


# -- 9. size --------------------------------------------------------------------------------------
def test_4096_instances_one_shared_edit():
    grid = cases.load_bundled("map_10x10")
    K = 4096
    goals = _free_goals(grid, K, seed=3)
    grid2, _ = _edit(grid, goals[0], "both", 12)
    free = np.argwhere(grid2 == 0)
    goals2 = [g if grid2[g[1], g[0]] == 0 else (int(free[0][1]), int(free[0][0])) for g in goals]
    with MdpBatchPathPlanning2d(grid, goals, GAMMA) as b:
        b.valueIteration()
        b.update_map(np.arange(K), grid2, goals2)
        n, res = b.valueIteration()
        cost, action = b.download()
        counts = b.sweep_counts()
    single = Single(grid.shape)
    cache = {}
    try:
        for k in range(K):
            key = (goals[k], goals2[k])
            if key not in cache:
                m = single._handle(grid, goals[k])
                m.valueIteration()
                m.update_map(grid2, goals2[k])
                sn, sres = m.valueIteration()
                sc, sa = m.download()
                cache[key] = (sn, sres, sc.copy(), sa.copy(), m.sweep_count)
            sn, sres, sc, sa, scount = cache[key]
            assert n[k] == sn and counts[k] == scount, k
            assert np.array_equal(res[k].view(np.uint64), sres.view(np.uint64)), k
            assert np.array_equal(_bits(cost[k]), _bits(sc)), k
            assert np.array_equal(action[k], sa), k
    finally:
        single.close()
