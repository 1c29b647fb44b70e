"""GPU tier, QV-tree half (SURVEY.md rows B1-B10) through the C ABI.

Bar: bit-exact everywhere.  The device-side arithmetic of the reference
(FFMA / flush-to-zero) and its host-side arithmetic (sequential float mul+add,
IEEE division) are both reproduced exactly, so tables, beliefs, bounds, chosen
actions and tree sizes must be identical to the oracle's."""
import os

import numpy as np
import pytest

import cases
import pomdp_fixtures as pf
import pomdp_oracle_py as po
from path_planning_2d_b200 import PomdpPathPlanning2d, SearchTree, _lib

pytestmark = pytest.mark.gpu
bits = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)


def same(a, b):
    """Bit-equal, except that any NaN equals any NaN (0/0 has a different sign
    and payload on x86 and on the GPU)."""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    return bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


@pytest.mark.parametrize("name,goal", [("map_3x3", (1, 1)), ("map_10x10", (8, 7)),
                                       ("sparse_map_100x40", (95, 34))])
def test_model_tables_bit_exact(name, goal):
    grid = cases.load_bundled(name)
    m = po.Model(grid, goal)
    with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
        tp, mp, sr = p.model_tables()
    hw = grid.size
    assert np.array_equal(bits(tp), bits(m.tp.reshape(hw, 9, 9)))
    assert np.array_equal(bits(mp), bits(m.mp.reshape(hw, 16)))
    assert np.array_equal(bits(sr), bits(m.sr.reshape(hw, 9)))


def test_goal_occupied_is_rejected():
    grid = np.zeros((6, 6), np.uint8)
    grid[2, 2] = 1
    with pytest.raises(_lib.Pp2dError) as e:
        PomdpPathPlanning2d(grid, (2, 2), cases.GAMMA)
    assert e.value.code == _lib.PP2D_ERR_GOAL_OCCUPIED


def test_sampling_uniforms_match_the_fixture():
    grid = cases.load_bundled("map_3x3")
    with PomdpPathPlanning2d(grid, (1, 1), cases.GAMMA) as p:
        un = p.sampling_uniforms()
    assert np.array_equal(bits(un), bits(pf.uniforms()))
    assert np.all(un > 0) and np.all(un <= 1)


@pytest.mark.parametrize("shape", [(1, 1), (1, 9), (9, 1), (7, 5), (40, 100), (33, 65)])
def test_bayes_update_batch_bit_exact(shape):
    h, w = shape
    grid, goal = cases.synthetic_map(h, w, 0.25, seed=h * 131 + w)
    m = po.Model(grid, goal)
    rng = np.random.default_rng(1)
    n = 37
    beliefs = rng.random((n, h * w), dtype=np.float32)
    beliefs[::3] = (beliefs[::3] ** 20 * 1e-32).astype(np.float32)   # subnormals
    beliefs[1::5, ::2] = 0
    acts = rng.integers(9, size=n).astype(np.uint8)
    obs = rng.integers(16, size=n).astype(np.uint8)
    with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
        out = p.bayes_update(beliefs, acts, obs)
        outn, sums = p.bayes_update(beliefs, acts, obs, normalize=True)
    for i in range(n):
        want, _ = m.bayes(beliefs[i], int(acts[i]), int(obs[i]))
        assert np.array_equal(bits(out[i]), bits(want)), i
        wantn, s = m.bayes(beliefs[i], int(acts[i]), int(obs[i]), normalize=True)
        assert bits(np.float32(sums[i])) == bits(np.float32(s)), i
        assert same(outn[i], wantn), i


def test_evaluate_bounds_bit_exact():
    name, goal = "map_10x10", (8, 7)
    grid = cases.load_bundled(name)
    m, fib, pbvi, fa, pa = pf.alphas(name, goal, n_pbvi=70)
    beliefs = np.concatenate([pf.gaussian_beliefs(grid, 90, seed=2),
                              np.random.default_rng(3).random((45, grid.size), dtype=np.float32)])
    with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
        p.set_alphas(fib, pbvi, fa, pa)
        up, ua, lo, la = p.evaluate(beliefs)
    for i, b in enumerate(beliefs):
        wu, wua, wl, wla = po.evaluate(b, fib, pbvi, fa, pa)
        assert bits(np.float32(up[i])) == bits(np.float32(wu)), i
        assert bits(np.float32(lo[i])) == bits(np.float32(wl)), i
        assert (ua[i], la[i]) == (wua, wla), i


def _tree_pair(name, goal, n_pbvi, seed):
    grid = cases.load_bundled(name)
    m, fib, pbvi, fa, pa = pf.alphas(name, goal, n_pbvi=n_pbvi)
    b = pf.gaussian_beliefs(grid, 1, seed=seed)[0]
    p = PomdpPathPlanning2d(grid, goal, cases.GAMMA)
    p.set_alphas(fib, pbvi, fa, pa)
    ot = po.Tree(m, cases.GAMMA, fib, pbvi, pf.uniforms(), b, fa, pa)
    return p, ot, b


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_search_tree_expand_step_by_step(seed):
    p, ot, b = _tree_pair("map_10x10", (8, 7), 20, seed)
    try:
        st = SearchTree(p, b)
        assert tuple(bits(np.float32(v)) for v in st.rootBounds()) == \
            tuple(bits(np.float32(v)) for v in ot.root_bounds())
        for step in range(6):
            st.expand()
            assert ot.expand() == 0
            assert st.getDepth() == ot.depth
            a, r = st.getOptimalAction()
            oa, orr = ot.best()
            assert a == oa and bits(np.float32(r)) == bits(np.float32(orr)), step
            assert tuple(bits(np.float32(v)) for v in st.rootBounds()) == \
                tuple(bits(np.float32(v)) for v in ot.root_bounds())
        # re-root on the chosen action and an observation, three times
        for z in (0, 5, 15):
            a, _ = st.getOptimalAction()
            st.update(a, z)
            assert ot.update(a, z) == 0
            assert st.getDepth() == ot.depth
            assert tuple(bits(np.float32(v)) for v in st.rootBounds()) == \
                tuple(bits(np.float32(v)) for v in ot.root_bounds())
            st.expand()
            ot.expand()
            assert st.getOptimalAction()[0] == ot.best()[0]
            assert bits(np.float32(st.getOptimalAction()[1])) == bits(np.float32(ot.best()[1]))
        st.close()
    finally:
        ot.close()
        p.close()


def test_belief_callback_on_the_launch_file_map():
    """BASELINE.json configs[0/1] for the POMDP planner: bundled sparse map,
    goal (95,34), depth 50, 15 online iterations."""
    p, ot, b = _tree_pair("sparse_map_100x40", (95, 34), 16, 7)
    try:
        a = p.beliefCallback(b)
        oa, orr, stats, rc = ot.plan(50, 15)
        assert rc == 0 and a == oa
        assert p.search_tree.getDepth() == stats[4]
        assert bits(np.float32(p.search_tree.getOptimalAction()[1])) == bits(np.float32(orr))
    finally:
        ot.close()
        p.close()


def test_plan_batch_equals_independent_oracle_plans():
    name, goal = "map_10x10", (8, 7)
    grid = cases.load_bundled(name)
    m, fib, pbvi, fa, pa = pf.alphas(name, goal, n_pbvi=20)
    beliefs = pf.gaussian_beliefs(grid, 24, seed=11)
    with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
        p.set_alphas(fib, pbvi, fa, pa)
        acts, vals, stats = p.plan_batch(beliefs, max_depth=50, max_iter=5, with_stats=True)
    for i, b in enumerate(beliefs):
        ot = po.Tree(m, cases.GAMMA, fib, pbvi, pf.uniforms(), b, fa, pa)
        oa, orr, ostats, rc = ot.plan(50, 5)
        ot.close()
        assert acts[i] == oa, i
        assert bits(np.float32(vals[i])) == bits(np.float32(orr)), i
        assert stats[i, 0] == ostats[0] and stats[i, 1] == ostats[1], i
        assert stats[i, 2] == ostats[4], i


def test_plan_batch_at_bench_scale_equals_single_query_trees(monkeypatch):
    """BASELINE.json configs[4] as the bench runs it: 640 Gaussian start
    beliefs on sparse_map_100x40, the REAL 9 FIB + 500 PBVI alpha vectors of
    the GPU offline solvers, depth cap 50, 15 expansions.  Large enough for
    the two staggered halves (>= 256 queries) and the OpenMP host loops (>= 64),
    and the pool starts so small (64 slots per query for trees of ~470 V nodes)
    that it grows in place several times mid-batch.  Every query must give the
    action, value and depth of its own pp2d_tree_plan on a fresh SearchTree,
    and -- for the first 32 -- of the CPU oracle, tree sizes included."""
    monkeypatch.setenv("PP2D_POMDP_SLOTS_PER_QUERY", "64")
    name, goal = "sparse_map_100x40", (95, 34)
    grid = cases.load_bundled(name)
    n = 640
    beliefs = pf.gaussian_beliefs(grid, n, sigma=2.0, seed=0)
    with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
        fib, fa, _ = p.fastInformedBound()
        _, pbvi, pa = p.pointBasedValueIteration(p.initial_belief, 500, rand_seed=1)
        p.set_alphas(fib, pbvi, fa, pa)
        acts, vals, stats = p.plan_batch(beliefs, max_depth=50, max_iter=15, with_stats=True)
        # a second batch on the grown pool (slots recycled) gives the same
        acts2, vals2, stats2 = p.plan_batch(beliefs[::-1], max_depth=50, max_iter=15,
                                            with_stats=True)
        assert np.array_equal(acts2[::-1], acts) and np.array_equal(bits(vals2[::-1]), bits(vals))
        assert np.array_equal(stats2[::-1], stats)
        assert stats[:, 0].mean() > 200 and np.all(stats[:, 3] <= 15)
        for i in range(n):
            st = SearchTree(p, beliefs[i])
            a, r = st.plan(50, 15)
            d = st.getDepth()
            st.close()
            assert (a, bits(np.float32(r)), d) == (acts[i], bits(vals[i]), stats[i, 2]), i
    m = po.Model(grid, goal)
    for i in range(32):
        ot = po.Tree(m, cases.GAMMA, fib, pbvi, pf.uniforms(), beliefs[i], fa, pa)
        oa, orr, ostats, rc = ot.plan(50, 15)
        ot.close()
        assert rc == 0 and acts[i] == oa, i
        assert bits(np.float32(vals[i])) == bits(np.float32(orr)), i
        assert stats[i, 0] == ostats[0] and stats[i, 1] == ostats[1], i
        assert stats[i, 2] == ostats[4], i


def test_per_tile_inner_rows_and_query_order_do_not_change_a_bit(monkeypatch):
    """The values launches of a batch walk, per tile of 128 children, only the
    inner rows on which some belief of the tile is non-zero, and the queries
    are planned in the order of their start beliefs' modes so that those lists
    are short.  Both are exact: with either or both switched off
    (PP2D_POMDP_TILE_SUPPORT=0, PP2D_POMDP_SORT=0) every action, value bit and
    tree statistic is the same -- and equals the oracle's for a sample."""
    name, goal = "sparse_map_100x40", (95, 34)
    grid = cases.load_bundled(name)
    fib, pbvi, fa, pa = pf.bundled_alphas(60)
    n = 300
    beliefs = pf.gaussian_beliefs(grid, n, sigma=2.0, seed=3)
    # a start belief that is zero nowhere on the free cells, and one point mass
    free = np.flatnonzero(grid.reshape(-1) == 0)
    beliefs[5] = 0
    beliefs[5, free] = np.float32(1.0 / len(free))
    beliefs[6] = 0
    beliefs[6, free[1234]] = 1
    results = []
    for tile, sort in (("1", "1"), ("0", "1"), ("1", "0"), ("0", "0")):
        monkeypatch.setenv("PP2D_POMDP_TILE_SUPPORT", tile)
        monkeypatch.setenv("PP2D_POMDP_SORT", sort)
        with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
            p.set_alphas(fib, pbvi, fa, pa)
            results.append(p.plan_batch(beliefs, max_depth=50, max_iter=6, with_stats=True))
    acts, vals, stats = results[0]
    for a, v, s in results[1:]:
        assert np.array_equal(a, acts) and np.array_equal(bits(v), bits(vals))
        assert np.array_equal(s, stats)
    m = po.Model(grid, goal)
    for i in (0, 5, 6, 150, 299):
        ot = po.Tree(m, cases.GAMMA, fib, pbvi, pf.uniforms(), beliefs[i], fa, pa)
        oa, orr, ostats, rc = ot.plan(50, 6)
        ot.close()
        assert rc == 0 and acts[i] == oa, i
        assert bits(np.float32(vals[i])) == bits(np.float32(orr)), i
        assert stats[i, 0] == ostats[0] and stats[i, 1] == ostats[1], i


@pytest.mark.parametrize("dense_env", ["0", "1"])
def test_beliefs_with_mass_on_dead_cells_take_the_dense_products(monkeypatch, dense_env):
    """The sequential inner products skip the cells no probability mass can
    enter (exact while the belief is +0 there).  A start belief that is NOT
    zero on occupied cells -- or is -0 there -- must switch its whole tree to
    the dense products; mixed with conforming queries in one batch, every
    query still equals the oracle bit for bit.  PP2D_POMDP_DENSE=1 (skipping
    off) gives the same bits."""
    monkeypatch.setenv("PP2D_POMDP_DENSE", dense_env)
    name, goal = "map_10x10", (8, 7)
    grid = cases.load_bundled(name)
    m, fib, pbvi, fa, pa = pf.alphas(name, goal, n_pbvi=20)
    beliefs = pf.gaussian_beliefs(grid, 70, seed=21)
    occ = np.flatnonzero(grid.reshape(-1) == 1)
    rng = np.random.default_rng(5)
    beliefs[3] = rng.random(grid.size, dtype=np.float32)
    beliefs[3] /= beliefs[3].sum(dtype=np.float32)
    beliefs[17, occ[:4]] = np.float32(1e-3)
    beliefs[40, occ[1]] = np.float32(-0.0)
    with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
        p.set_alphas(fib, pbvi, fa, pa)
        acts, vals, stats = p.plan_batch(beliefs, max_depth=50, max_iter=4, with_stats=True)
        st = SearchTree(p, beliefs[17])
        a17, r17 = st.plan(50, 4)
        st.close()
    assert (a17, bits(np.float32(r17))) == (acts[17], bits(vals[17]))
    for i in (0, 3, 17, 40, 69):
        ot = po.Tree(m, cases.GAMMA, fib, pbvi, pf.uniforms(), beliefs[i], fa, pa)
        oa, orr, ostats, rc = ot.plan(50, 4)
        ot.close()
        assert acts[i] == oa and same(np.float32(vals[i]), np.float32(orr)), i
        assert stats[i, 0] == ostats[0] and stats[i, 1] == ostats[1], i


def test_c_abi_rejects_out_of_range_actions_and_observations():
    """pp2d_pomdp_bayes_update / pp2d_tree_update index the tables with the
    action and observation: out-of-range values are refused before anything
    is touched (the reference has no such check; it would read out of bounds)."""
    name, goal = "map_10x10", (8, 7)
    grid = cases.load_bundled(name)
    m, fib, pbvi, fa, pa = pf.alphas(name, goal, n_pbvi=20)
    b = pf.gaussian_beliefs(grid, 1, seed=0)[0]
    with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
        p.set_alphas(fib, pbvi, fa, pa)
        for a, z in ((9, 0), (0, 16), (255, 255)):
            with pytest.raises(_lib.Pp2dError) as e:
                p.bayes_update(b[None], a, z)
            assert e.value.code == _lib.PP2D_ERR_INVALID
        st = SearchTree(p, b)
        st.expand()
        before = st.dump()
        for a, z in ((9, 0), (0, 16)):
            with pytest.raises(_lib.Pp2dError):
                st.update(a, z)
        assert np.array_equal(bits(st.dump()), bits(before))     # tree untouched
        st.expand()
        # many re-roots: the node arrays are rebuilt, not grown without bound
        for _ in range(12):
            a, _r = st.getOptimalAction()
            st.update(a, 3)
            st.plan(50, 2)
        assert st.dump().shape[0] < 2000
        st.close()


def test_reference_pomdp_kernels_vs_restatement():
    """Live pin of oracle/pomdp_oracle.c against the reference kernels."""
    so = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                      "oracle", "_ref", "libpp2d_ref_pomdp.so")
    if not os.path.exists(so):
        pytest.skip("oracle/_ref not built")
    R = po.ref()
    grid, goal = cases.synthetic_map(23, 31, 0.3, seed=4)
    h, w = grid.shape
    hw = h * w
    m = po.Model(grid, goal)
    tp = np.zeros(hw * 81, np.float32); mp = np.zeros(hw * 16, np.float32)
    sr = np.zeros(hw * 9, np.float32)
    R.ref_pomdp_model(h, w, grid.ctypes.data, goal[0], goal[1], tp.ctypes.data,
                      mp.ctypes.data, sr.ctypes.data)
    assert np.array_equal(bits(tp), bits(m.tp)) and np.array_equal(bits(mp), bits(m.mp))
    assert np.array_equal(bits(sr), bits(m.sr))
    b = (np.random.default_rng(0).random(hw, dtype=np.float32) ** 18 * 1e-30).astype(np.float32)
    us = np.arange(9, dtype=np.uint8); zs = (np.arange(9) * 7 % 16).astype(np.uint8)
    out = np.zeros((9, hw), np.float32)
    R.ref_pomdp_bayes(h, w, grid.ctypes.data, goal[0], goal[1], b.ctypes.data, 9,
                      us.ctypes.data, zs.ctypes.data, out.ctypes.data)
    for i in range(9):
        want, _ = m.bayes(b, int(us[i]), int(zs[i]))
        assert np.array_equal(bits(out[i]), bits(want)), i
    fib = np.zeros(hw * 9, np.float32)
    n = R.ref_pomdp_fib(h, w, grid.ctypes.data, goal[0], goal[1], cases.GAMMA,
                        fib.ctypes.data, 30)
    ofib, on = m.fib(cases.GAMMA, 30)
    assert n == on and np.array_equal(bits(fib), bits(ofib.reshape(-1)))


def test_pomdp_kernels_equal_the_reference_record():
    """The case of the live pin above, against its stored record
    (tests/golden/kernels_ref_syn_23x31.npz): the product's model tables,
    unnormalised Bayes updates and capped FIB solve, bit for bit."""
    import sys
    sys.path.insert(0, cases.GOLDEN)
    import make_golden
    g = np.load(os.path.join(cases.GOLDEN, "kernels_ref_syn_23x31.npz"))
    grid, goal, b, us, zs, cap = make_golden.pomdp_live_case()
    with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
        tp, mp, sr = p.model_tables()
        assert np.array_equal(bits(tp).reshape(-1), bits(g["trans_prob"]))
        assert np.array_equal(bits(mp).reshape(-1), bits(g["meas_prob"]))
        assert np.array_equal(bits(sr).reshape(-1), bits(g["stage_reward"]))
        out = p.bayes_update(np.stack([b] * len(us)), us, zs)
        assert np.array_equal(bits(out), bits(g["bayes"]))
        fib, _, n = p.fastInformedBound(cap)
    assert n == int(g["fib_sweeps"])
    assert np.array_equal(bits(fib).reshape(-1), bits(g["fib"]))


@pytest.mark.parametrize("name,goal", [("map_10x10", (8, 7)), ("sparse_map_100x40", (95, 34))])
def test_fib_solver_bit_exact(name, goal):
    """"next" row 1: the FIB offline solver, same sweeps and bits as the
    oracle (itself pinned to the reference kernel by the golden vectors)."""
    grid = cases.load_bundled(name)
    m = po.Model(grid, goal)
    want, n = m.fib(cases.GAMMA)
    with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
        got, acts, sweeps = p.fastInformedBound()
    assert sweeps == n
    assert acts.tolist() == list(range(9))
    assert np.array_equal(bits(got), bits(want))
