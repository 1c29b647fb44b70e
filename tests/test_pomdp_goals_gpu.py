"""GPU tier of goal sets (pp2d_pomdp_set_goals, pp2d_pomdp_set_goal_alphas,
pp2d_tree_batch_create_goals, pp2d_sim_rollout_pomdp_goals; DESIGN.md
section 7e).  The reference is one single-goal handle per goal, created with
that goal, with the same tables and that goal's alpha vectors: every tree of a
mixed-goal batch gives the bits of a SearchTree on its goal's handle fed the
same calls (actions, values, stats, full dumps), a sample also those of the
CPU oracle's tree, and every episode of a mixed-goal rollout the bits of the
same episode on its goal's handle.  Goals holding a single tree make the
padding of goal segments run in every round."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import cases
import pomdp_fixtures as pf
import pomdp_oracle_py as po
from path_planning_2d_b200 import (DummySimulator, PomdpPathPlanning2d, SearchTree,
                                   SearchTreeBatch, _lib)
from test_tree_batch_gpu import bits, observation, same_dump

pytestmark = pytest.mark.gpu
GAMMA = cases.GAMMA
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# goal 0 (the launch goal) and the PBVI count per map
MAPS = {"map_3x3": ((1, 1), 12), "map_10x10": ((8, 7), 20), "sparse_map_100x40": ((95, 34), 6)}


def goal_cells(name, G):
    """Goal 0 and G - 1 more free cells (seeded; a cell may repeat on small maps)."""
    grid = cases.load_bundled(name)
    free = np.argwhere(grid == 0)
    rng = np.random.default_rng(7)
    pick = rng.choice(len(free), size=17, replace=len(free) < 17)
    cells = [MAPS[name][0]] + [(int(free[i][1]), int(free[i][0])) for i in pick]
    return cells[:G]


def alphas(name, goal):
    return pf.alphas(name, goal, n_pbvi=MAPS[name][1])


class Fleet:
    """A handle with goal set `cells`, and one single-goal handle per goal."""

    def __init__(self, name, cells, nan_goal=None):
        self.grid = cases.load_bundled(name)
        self.cells = cells
        self.al = []
        for g, c in enumerate(cells):
            m, fib, pbvi, fa, pa = alphas(name, c)
            if g == nan_goal:
                fib = fib.copy()
                fib[np.flatnonzero(self.grid.reshape(-1) == 0)[3], 2] = np.nan
            self.al.append((m, fib, pbvi, fa, pa))
        self.p = PomdpPathPlanning2d(self.grid, cells[0], GAMMA)
        self.p.set_alphas(*self.al[0][1:])
        self.p.set_goals(np.array(cells[1:], np.int64).reshape(-1, 2))
        for g in range(1, len(cells)):
            self.p.set_goal_alphas(g, *self.al[g][1:])
        self.ref = []
        for g, c in enumerate(cells):
            r = PomdpPathPlanning2d(self.grid, c, GAMMA)
            r.set_alphas(*self.al[g][1:])
            self.ref.append(r)

    def close(self):
        for r in self.ref:
            r.close()
        self.p.close()


def tree_goals(n, G, seed):
    """Goal 0 holds most trees, goal 1 one tree, goal G - 1 none (G >= 3),
    the others a few; shuffled so that the plan order is not the creation order."""
    if G == 1:
        return np.zeros(n, np.uint32)
    g = np.zeros(n, np.uint32)
    g[1] = 1
    rest = list(range(2, G - 1)) if G >= 3 else []
    for j, goal in enumerate(rest):
        if 2 + 2 * j + 1 < n // 2:
            g[2 + 2 * j: 4 + 2 * j] = goal
    return np.random.default_rng(seed).permutation(g).astype(np.uint32)


def start_beliefs(grid, n, seed, dense=()):
    b = pf.gaussian_beliefs(grid, n, seed=seed)
    occ = np.flatnonzero(grid.reshape(-1) == 1)
    for k in dense:                                # mass on occupied cells: dense products
        b[k, occ[: 2]] = np.float32(1e-3)
        b[k] /= b[k].sum(dtype=np.float32)
    return b


class Lockstep:
    """A mixed-goal batch and, for the trees in `watch`, SearchTrees on their
    goals' single-goal handles, fed the same calls."""

    def __init__(self, fleet, beliefs, goals, watch):
        self.f = fleet
        self.goals = goals
        self.batch = SearchTreeBatch(fleet.p, beliefs, goals)
        self.single = {k: SearchTree(fleet.ref[int(goals[k])], beliefs[k]) for k in watch}
        self.log = {k: [] for k in watch}
        self.best = {}

    def close(self):
        for t in self.single.values():
            t.close()
        self.batch.close()

    def plan(self, idx, d, it):
        idx = np.asarray(idx, np.uint32)
        acts, vals, stats = self.batch.plan(idx, d, it, with_stats=True)
        for j, k in enumerate(idx.tolist()):
            self.best[k] = int(acts[j])
            if k not in self.single:
                continue
            a, v = self.single[k].plan(d, it)
            self.log[k].append(("plan", d, it, a, np.float32(v)))
            assert (acts[j], bits(vals[j])) == (a, bits(np.float32(v))), k
            assert stats[j, 2] == self.single[k].getDepth(), k
            assert same_dump(self.batch.dump(k), self.single[k].dump()), k
        return acts, bits(vals), stats

    def update(self, idx, salt=0):
        idx = [int(k) for k in idx]
        acts = np.array([self.best[k] for k in idx], np.uint8)
        obs = np.array([observation(self.batch.dump(k), self.best[k], k + salt) for k in idx],
                       np.uint8)
        self.batch.update(idx, acts, obs)
        for k, a, z in zip(idx, acts.tolist(), obs.tolist()):
            if k in self.single:
                self.single[k].update(a, z)
                self.log[k].append(("update", a, z))
                assert same_dump(self.batch.dump(k), self.single[k].dump()), k


def replay_on_oracle(fleet, ls, k, belief):
    m, fib, pbvi, fa, pa = fleet.al[int(ls.goals[k])]
    ot = po.Tree(m, GAMMA, fib, pbvi, pf.uniforms(), belief, fa, pa)
    try:
        for op in ls.log[k]:
            if op[0] == "plan":
                oa, orr, _, rc = ot.plan(op[1], op[2])
                assert rc == 0 and (oa, bits(np.float32(orr))) == (op[3], bits(op[4])), k
            else:
                assert ot.update(op[1], op[2]) == 0
        assert same_dump(ot.dump(), ls.batch.dump(k)), k
    finally:
        ot.close()


# -- reward tables --------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(MAPS))
def test_goal_reward_tables(name):
    grid = cases.load_bundled(name)
    cells = goal_cells(name, 5)
    p = PomdpPathPlanning2d(grid, cells[0], GAMMA)
    sr0 = p.model_tables()[2]
    p.set_goals(cells[1:])
    assert np.array_equal(p.goals(), np.array(cells, np.uint32))
    for g, c in enumerate(cells):
        with PomdpPathPlanning2d(grid, c, GAMMA) as r:
            assert np.array_equal(bits(p.goal_reward(g)), bits(r.model_tables()[2])), g
    assert np.array_equal(bits(p.model_tables()[2]), bits(sr0))      # goal 0 unchanged
    # given tables come back as given (checkpoint text rounds the rewards)
    given = pf.text_round(np.stack([p.goal_reward(g) for g in range(1, 5)]))
    given[0, 0, 0] = np.float32(-1.3)
    p.set_goals(cells[1:], stage_rewards=given)
    for g in range(1, 5):
        assert np.array_equal(bits(p.goal_reward(g)), bits(given[g - 1])), g
    # set_model_tables changes goal 0's reward only
    tp, mp, sr = p.model_tables()
    p.set_model_tables(stage_reward=pf.text_round(sr))
    assert np.array_equal(bits(p.goal_reward(0)), bits(pf.text_round(sr)))
    assert np.array_equal(bits(p.goal_reward(1)), bits(given[0]))
    p.set_goals(np.zeros((0, 2), np.uint32))
    assert p.goals().shape == (1, 2)
    p.close()


# -- tree batches against single trees --------------------------------------------------------
@pytest.mark.parametrize("G", [1, 2, 5, 17])
@pytest.mark.parametrize("name", list(MAPS))
def test_batch_equals_single_goal_trees_and_the_oracle(name, G):
    n = {"map_3x3": 12, "map_10x10": 24, "sparse_map_100x40": 40}[name]
    f = Fleet(name, goal_cells(name, G))
    goals = tree_goals(n, G, seed=G)
    beliefs = start_beliefs(f.grid, n, seed=G, dense=(0,) if f.grid.size > 9 else ())
    ls = Lockstep(f, beliefs, goals, range(n))
    pads0 = f.p.padding_counters()
    try:
        for r, (d, it) in enumerate([(50, 3), (50, 4), (50, 2), (50, 5)]):
            ls.plan(range(n), d, it)
            ls.update(range(n), salt=r)
        ls.plan(range(n), 50, 3)
        # the trees of goal 1 and a tree of goal 0, on the CPU oracle
        for k in [int(np.flatnonzero(goals == goals.max())[0]), int(np.flatnonzero(goals == 0)[0])]:
            replay_on_oracle(f, ls, k, beliefs[k])
    finally:
        ls.close()
    pads = f.p.padding_counters()
    if G > 1:                                      # goal segments were padded
        assert pads[0] > pads0[0] and pads[1] > pads0[1]
    else:
        assert pads == pads0 == (0, 0)
    f.close()


def _switch_run(monkeypatch, env, n, f_args, beliefs, goals, watch):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    f = Fleet(*f_args)
    ls = Lockstep(f, beliefs[:n], goals, watch)
    out = []
    try:
        out.append(ls.plan(range(n), 50, 5))
        ls.update(range(n))
        out.append(ls.plan(range(n), 50, 4))
        ls.update(range(n), salt=1)
        sub = np.arange(0, n, 2)
        out.append(ls.plan(sub, 50, 3))
        out.append([ls.batch.dump(k).tobytes() for k in range(n)])
    finally:
        ls.close()
        f.close()
        for k in env:
            monkeypatch.delenv(k)
    return out


@pytest.mark.parametrize("n", [64, 128, 256, 384])
def test_sizes_and_switches_do_not_change_a_bit(monkeypatch, n):
    """Across the 64 / 128 / 256 / 384 thresholds, with mode order, group count,
    per-tile rows and dense products switched; dense and sparse start beliefs
    mixed.  Watched: every tree of the small goals and a few of goal 0."""
    name, G = "sparse_map_100x40", 5
    cells = goal_cells(name, G)
    grid = cases.load_bundled(name)
    goals = tree_goals(n, G, seed=n)
    beliefs = start_beliefs(grid, n, seed=n, dense=(3, n // 2))
    watch = sorted(set(np.flatnonzero(goals != 0).tolist()) | {3, n // 2, n - 1})
    runs = []
    for env in ({}, {"PP2D_POMDP_SORT": "0"}, {"PP2D_POMDP_GROUPS": "1"},
                {"PP2D_POMDP_GROUPS": "3"}, {"PP2D_POMDP_TILE_SUPPORT": "0"},
                {"PP2D_POMDP_DENSE": "1"}):
        runs.append(_switch_run(monkeypatch, env, n, (name, cells), beliefs, goals,
                                watch if not env else watch[:3]))
    for r in runs[1:]:
        for got, want in zip(r[:-1], runs[0][:-1]):
            for g, w in zip(got, want):
                assert np.array_equal(g, w)
        assert r[-1] == runs[0][-1]


def test_a_goal_with_a_nan_alpha():
    """One goal's FIB alphas hold a NaN: nothing is skipped for any goal, and
    every goal still gives its single handle's bits."""
    name = "map_10x10"
    f = Fleet(name, goal_cells(name, 5), nan_goal=2)
    n = 20
    goals = tree_goals(n, 5, seed=3)
    goals[:3] = 2
    beliefs = start_beliefs(f.grid, n, seed=3)
    ls = Lockstep(f, beliefs, goals, range(n))
    try:
        ls.plan(range(n), 50, 4)
        ls.update(range(n))
        ls.plan(range(n), 50, 4)
    finally:
        ls.close()
        f.close()


def test_all_zero_goals_equal_the_plain_batch():
    name = "map_10x10"
    f = Fleet(name, goal_cells(name, 3))
    n = 30
    beliefs = start_beliefs(f.grid, n, seed=11)
    a = SearchTreeBatch(f.p, beliefs, np.zeros(n, np.uint32))
    b = SearchTreeBatch(f.p, beliefs)
    try:
        for it in (3, 5):
            ra, rb = a.plan(None, 50, it, with_stats=True), b.plan(None, 50, it, with_stats=True)
            assert np.array_equal(ra[0], rb[0]) and np.array_equal(bits(ra[1]), bits(rb[1]))
            assert np.array_equal(ra[2], rb[2])
            obs = [observation(a.dump(k), int(ra[0][k]), k) for k in range(n)]
            a.update(None, ra[0], obs)
            b.update(None, rb[0], obs)
        assert all(same_dump(a.dump(k), b.dump(k)) for k in range(n))
    finally:
        a.close()
        b.close()
        f.close()


# -- rollouts -----------------------------------------------------------------------------------
def test_rollout_goals_equal_single_goal_rollouts():
    name = "map_10x10"
    cells = goal_cells(name, 4)
    f = Fleet(name, cells)
    grid = f.grid
    n, steps, seed, first = 24, 30, 99, 5
    rng = np.random.default_rng(1)
    free = np.argwhere(grid == 0)
    starts = np.array([(x, y) for y, x in free[rng.choice(len(free), n)]], np.uint32)
    goals = (np.arange(n) % 4).astype(np.uint32)
    rng.shuffle(goals)
    beliefs = np.zeros((n, grid.size), np.float32)
    beliefs[np.arange(n), starts[:, 1] * grid.shape[1] + starts[:, 0]] = 1.0
    beliefs[1] = pf.gaussian_beliefs(grid, 1, seed=2)[0]
    with DummySimulator(grid) as sim:
        got = sim.rollout(f.p, starts, steps, seed, beliefs=beliefs, first_episode=first,
                          record=True, max_depth=50, max_iter=6, goals=goals)
        for i in range(n):
            want = sim.rollout(f.ref[int(goals[i])], starts[i:i + 1], steps, seed,
                               beliefs=beliefs[i:i + 1], first_episode=first + i, record=True,
                               max_depth=50, max_iter=6)
            for key, v in want.items():
                assert np.array_equal(np.atleast_1d(got[key][i]).view(np.uint8),
                                      np.atleast_1d(v[0]).view(np.uint8)), (i, key)
    goal_cell = np.array([c[1] * grid.shape[1] + c[0] for c in cells])
    own = got["reached"].astype(bool) & (goals != 0)
    assert own.any(), "no episode reached a goal other than goal 0"
    assert np.array_equal(got["final_cell"][own], goal_cell[goals[own]])
    assert (goal_cell[goals[own]] != goal_cell[0]).any()
    f.close()


# -- error paths --------------------------------------------------------------------------------
def test_refusals_change_nothing():
    name = "map_10x10"
    cells = goal_cells(name, 3)
    f = Fleet(name, cells)
    p, lib = f.p, f.p._lib
    INV, ST, OCC = _lib.PP2D_ERR_INVALID, _lib.PP2D_ERR_STATE, _lib.PP2D_ERR_GOAL_OCCUPIED
    grid = f.grid
    occ = np.argwhere(grid == 1)[0]
    beliefs = start_beliefs(grid, 4, seed=1)
    b = SearchTreeBatch(p, beliefs, [0, 1, 2, 1])   # (a refusal below: nothing changes)
    b.plan(None, 50, 3)
    before = [b.dump(k) for k in range(4)]
    sr = [p.goal_reward(g) for g in range(3)]

    def refused(code, fn, *args, **kw):
        with pytest.raises(_lib.Pp2dError) as e:
            fn(*args, **kw)
        assert e.value.code == code
        assert all(same_dump(b.dump(k), before[k]) for k in range(4))
        assert np.array_equal(p.goals(), np.array(cells, np.uint32))
        assert all(np.array_equal(bits(p.goal_reward(g)), bits(sr[g])) for g in range(3))
        return str(e.value)

    # resident beliefs: the goal set is fixed
    assert "resident" in refused(ST, p.set_goals, cells[1:])
    b.close()
    b = None
    before = []

    def refused_nb(code, fn, *args, **kw):
        with pytest.raises(_lib.Pp2dError) as e:
            fn(*args, **kw)
        assert e.value.code == code
        assert np.array_equal(p.goals(), np.array(cells, np.uint32))
        return str(e.value)

    assert "goal 2" in refused_nb(INV, p.set_goals, [cells[1], (10, 0)])
    assert "goal 2" in refused_nb(INV, p.set_goals, [cells[1], (0, 10)])
    assert "goal 1" in refused_nb(OCC, p.set_goals, [(int(occ[1]), int(occ[0]))])
    m, fib, pbvi, fa, pa = f.al[1]
    assert "goal 3" in refused_nb(INV, p.set_goal_alphas, 3, fib, pbvi, fa, pa)
    # one PBVI count for the whole handle
    assert "goal 0" in refused_nb(INV, p.set_goal_alphas, 1, fib, pbvi[:5], fa, pa[:5])
    assert "goal 1" in refused_nb(INV, p.set_alphas, fib, pbvi[:5], fa, pa[:5])
    assert lib.pp2d_pomdp_goal_reward(p._h, 3, np.zeros(grid.size * 9, np.float32).ctypes.data) \
        == INV
    # tree batches: an index above the set, a goal without alpha vectors
    out = ctypes.c_void_p()
    g = np.array([0, 3], np.uint32)
    assert lib.pp2d_tree_batch_create_goals(p._h, beliefs.ctypes.data, g.ctypes.data, 2,
                                            ctypes.byref(out)) == INV
    assert "tree 1" in lib.pp2d_last_error().decode()
    p.set_goals(cells[1:] + [cells[2]])            # goal 3 without alpha vectors
    assert p.goals().shape == (4, 2)
    with pytest.raises(_lib.Pp2dError) as e:
        SearchTreeBatch(p, beliefs[:2], [0, 3])
    assert e.value.code == ST and "tree 1" in str(e.value)
    with DummySimulator(grid) as sim:
        st = np.array([cells[1]], np.uint32)
        for goals, code in (([3], ST), ([4], INV)):
            with pytest.raises(_lib.Pp2dError) as e:
                sim.rollout(p, st, 5, 1, goals=goals, max_depth=50, max_iter=2)
            assert e.value.code == code and "episode 0" in str(e.value)
        r = _lib.Rollout()
        assert lib.pp2d_sim_rollout_pomdp_goals(sim._h, p._h, None, 1, st.ctypes.data, None, 5,
                                                50, 2, 1, 0, ctypes.byref(r)) == INV
    # goal sets with another count once no goal holds alpha vectors but goal 0
    p.set_goals([])
    p.set_alphas(fib, pbvi[:5], fa, pa[:5])
    p.set_goals(cells[1:])
    p.set_goal_alphas(1, fib, pbvi[:5], fa, pa[:5])
    f.close()


# -- C++ mirror ---------------------------------------------------------------------------------
def test_cpp_goal_sets_give_the_python_results(tmp_path):
    import cv2
    name = "map_10x10"
    png = os.path.join(cases.GOLDEN, "maps", name + "_gray.png")
    img = cv2.imread(png, cv2.IMREAD_GRAYSCALE)
    _, grid = cv2.threshold(img, 250.0, 1.0, cv2.THRESH_BINARY_INV)
    grid = np.ascontiguousarray(grid, np.uint8)
    free = np.argwhere(grid == 0)
    cells = [(int(x), int(y)) for y, x in free[np.random.default_rng(3).choice(len(free), 4,
                                                                            replace=False)]]
    n_pbvi, iters = 10, 5
    hw = grid.size
    rounded = []
    for g, c in enumerate(cells):                   # save_data of a planner with goal c
        d = tmp_path / f"goal{g}"
        d.mkdir()
        m, fib, pbvi, fa, pa = pf.alphas(grid, c, n_pbvi=n_pbvi)
        tables = (("model_data_trans_prob", m.tp.reshape(hw * 9, 9)),
                  ("model_data_meas_prob", m.mp.reshape(hw, 16)),
                  ("model_data_stage_reward", m.sr.reshape(hw, 9)))
        for fname, arr in tables + (("fib_alphas", fib), ("pbvi_alphas", pbvi)):
            pf.write_text_rows(d / fname, arr)
        pf.write_actions(d / "fib_actions", fa)
        pf.write_actions(d / "pbvi_actions", pa)
        rounded.append((pf.text_round(m.tp), pf.text_round(m.mp), pf.text_round(m.sr),
                        pf.text_round(fib), pf.text_round(pbvi), fa, pa))
    n = 20
    beliefs = pf.gaussian_beliefs(grid, n, seed=6)
    goals = tree_goals(n, 4, seed=6)
    (tmp_path / "goals.bin").write_bytes(np.array(cells[1:], np.uint32).tobytes())
    (tmp_path / "beliefs.bin").write_bytes(beliefs.tobytes())
    (tmp_path / "tree_goals.bin").write_bytes(goals.tobytes())
    exe = str(tmp_path / "pomdp_goals_main")
    libdir = os.path.join(ROOT, "path_planning_2d_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-o", exe,
                    os.path.join(ROOT, "tests", "cpp", "pomdp_goals_main.cpp"), "-L", libdir,
                    "-lpp2d", "-lz", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([exe, png, str(cells[0][0]), str(cells[0][1]), "0.95",
                          str(tmp_path / "goal0"), str(n_pbvi), str(iters),
                          str(tmp_path / "goals.bin"), str(tmp_path / "beliefs.bin"),
                          str(tmp_path / "tree_goals.bin")] +
                         [str(tmp_path / f"goal{g}") for g in range(1, 4)],
                         capture_output=True, text=True)
    lines = [l for l in out.stdout.splitlines() if l.startswith("RESULT")]
    assert len(lines) == n, out.stdout + out.stderr
    # the same start-up in Python: rounded tables and alpha vectors per goal
    tp, mp, sr, fib, pbvi, fa, pa = rounded[0]
    with PomdpPathPlanning2d(grid, cells[0], GAMMA) as p:
        p.set_model_tables(tp, mp, sr)
        p.set_alphas(fib, pbvi, fa, pa)
        p.set_goals(cells[1:], stage_rewards=np.stack([r[2] for r in rounded[1:]]))
        for g in range(1, 4):
            p.set_goal_alphas(g, *rounded[g][3:])
        with SearchTreeBatch(p, beliefs, goals) as b:
            a0, v0 = b.plan(None, 50, iters)
            b.update(None, a0, 0)
            a1, v1 = b.plan(None, 50, iters)
    for k, line in enumerate(lines):
        kv = dict(t.split("=") for t in line.split()[1:])
        assert int(kv["k"]) == k and int(kv["a0"]) == a0[k] and int(kv["a1"]) == a1[k]
        assert kv["r0"] == "%08x" % int(bits(v0[k])[0])
        assert kv["r1"] == "%08x" % int(bits(v1[k])[0])
