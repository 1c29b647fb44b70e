"""GPU tier of the persistent tree batches (SearchTreeBatch, pp2d_tree_batch_*):
every tree of a batch, fed plan and update calls together with others, gives
the bits of a single SearchTree fed the same calls (actions, values, depths,
full dumps, so root bounds too), and a sample those of the CPU oracle's tree.
Batch sizes across the group and sort thresholds, the order and group
switches, subsets, pool growth mid-plan, interleaving with plan_batch and
single trees on one handle, and the argument rules (a refused call changes
nothing)."""
import ctypes

import numpy as np
import pytest

import cases
import pomdp_fixtures as pf
import pomdp_oracle_py as po
import tree_scenario as ts
from path_planning_2d_b200 import PomdpPathPlanning2d, SearchTree, SearchTreeBatch, _lib

pytestmark = pytest.mark.gpu
GAMMA = cases.GAMMA
CASES = {"map_3x3": ((1, 1), 12, 4), "map_10x10": ((8, 7), 20, 10),
         "sparse_map_100x40": ((95, 34), 40, 6)}


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_dump(a, b):
    return a.shape == b.shape and np.array_equal(bits(a), bits(b))


def observation(dump, a, k):
    """An observation under the root's Q node for `a` that has a V child when
    k is even (the kept subtree is re-rooted), one without when k is odd (a
    Bayes update makes the new root)."""
    obs = ts._root_q_children(dump, a)
    missing = [z for z in range(16) if z not in obs]
    if obs and (k % 2 == 0 or not missing):
        return obs[len(obs) // 2]
    return missing[k % len(missing)]


class Lockstep:
    """A batch and single SearchTrees of the trees in `watch`, fed the same
    calls; every call compares the watched trees."""

    def __init__(self, p, beliefs, watch=None):
        self.p = p
        self.n = len(beliefs)
        self.watch = list(range(self.n)) if watch is None else list(watch)
        self.batch = SearchTreeBatch(p, beliefs)
        self.single = {k: SearchTree(p, beliefs[k]) for k in self.watch}
        self.log = {k: [] for k in self.watch}
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
        return acts, vals, stats

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
        return acts, obs

    def dumps(self):
        return [self.batch.dump(k) for k in range(self.n)]


def planner(name, alphas=None):
    goal, n_pbvi, _ = CASES[name]
    grid = cases.load_bundled(name)
    m, fib, pbvi, fa, pa = pf.alphas(name, goal, n_pbvi=n_pbvi) if alphas is None else alphas
    p = PomdpPathPlanning2d(grid, goal, GAMMA)
    p.set_alphas(fib, pbvi, fa, pa)
    return grid, p, (m, fib, pbvi, fa, pa)


def start_beliefs(grid, n, seed):
    b = pf.gaussian_beliefs(grid, n, seed=seed)
    if grid.size <= 9:                            # a flat belief on the 3x3 map
        free = (grid.reshape(-1) == 0).astype(np.float32)
        b[0] = free / free.sum(dtype=np.float32)
    return b


@pytest.mark.parametrize("name", list(CASES))
def test_batch_equals_single_trees_and_the_oracle(name):
    grid, p, (m, fib, pbvi, fa, pa) = planner(name)
    n = CASES[name][2]
    beliefs = start_beliefs(grid, n, seed=4)
    ls = Lockstep(p, beliefs)
    try:
        for r, (d, it) in enumerate([(50, 3), (50, 4), (50, 2), (50, 5), (50, 3)]):
            ls.plan(range(n), d, it)
            ls.update(range(n), salt=r)
        ls.plan(range(n), 50, 4)
        # a sample replayed on the CPU oracle's tree
        for k in (0, 1):
            ot = po.Tree(m, GAMMA, fib, pbvi, pf.uniforms(), beliefs[k], fa, pa)
            for op in ls.log[k]:
                if op[0] == "plan":
                    oa, orr, _, rc = ot.plan(op[1], op[2])
                    assert rc == 0 and (oa, bits(np.float32(orr))) == (op[3], bits(op[4])), k
                else:
                    assert ot.update(op[1], op[2]) == 0
            assert same_dump(ot.dump(), ls.batch.dump(k)), k
            ot.close()
    finally:
        ls.close()
        p.close()


def _sizes_run(monkeypatch, n, sort, groups, beliefs, alphas, watch):
    monkeypatch.setenv("PP2D_POMDP_SORT", sort)
    monkeypatch.setenv("PP2D_POMDP_GROUPS", groups)
    grid, p, _ = planner("sparse_map_100x40", alphas)
    ls = Lockstep(p, beliefs[:n], watch)
    out = []
    try:
        # fresh trees: what plan_batch gives for the same beliefs
        acts, vals, stats = ls.plan(range(n), 50, 6)
        fa, fv, fs = p.plan_batch(beliefs[:n], max_depth=50, max_iter=6, with_stats=True)
        assert np.array_equal(acts, fa) and np.array_equal(bits(vals), bits(fv))
        assert np.array_equal(stats, fs)
        out.append((acts, bits(vals), stats))
        ls.update(range(n))                       # kept subtrees and new roots
        # depth cap 1: kept roots that are already expanded stay as they are
        before = ls.dumps()
        acts, vals, stats = ls.plan(range(n), 1, 8)
        for k in range(n):
            if before[k][0, 6] >= 1:
                assert same_dump(ls.batch.dump(k), before[k]), k
        out.append((acts, bits(vals), stats))
        # max_iter = 0 changes nothing
        before = ls.dumps()
        acts, vals, stats = ls.plan(range(n), 50, 0)
        assert all(same_dump(ls.batch.dump(k), before[k]) for k in range(n))
        out.append((acts, bits(vals), stats))
        ls.update(range(n), salt=1)
        out.append(ls.plan(range(n), 50, 5))
        out[-1] = (out[-1][0], bits(out[-1][1]), out[-1][2])
        out.append([d.tobytes() for d in ls.dumps()])
    finally:
        ls.close()
        p.close()
    return out


@pytest.mark.parametrize("n", [64, 256, 384])
def test_sizes_order_and_groups_do_not_change_a_bit(monkeypatch, n):
    """Across the 64 (host threads), 128 (mode order), 256 and 384 (two and
    three groups) thresholds, with the mode order and the group count varied;
    start beliefs with mass on dead cells (dense products) mixed with sparse
    ones; kept roots already at the depth cap; max_iter = 0."""
    grid = cases.load_bundled("sparse_map_100x40")
    alphas = (None,) + pf.bundled_alphas(60)
    beliefs = pf.gaussian_beliefs(grid, 384, sigma=2.0, seed=8)
    occ = np.flatnonzero(grid.reshape(-1) == 1)
    beliefs[2, occ[:3]] = np.float32(1e-3)        # mass on occupied cells
    beliefs[2] /= beliefs[2].sum(dtype=np.float32)
    beliefs[7, occ[5]] = np.float32(-0.0)
    watch = [0, 2, 7, n // 2, n - 1]
    runs = []
    for sort, groups in (("1", "0"), ("0", "0"), ("1", "1"), ("1", "3")):
        runs.append(_sizes_run(monkeypatch, n, sort, groups, beliefs, alphas, watch))
    for r in runs[1:]:
        for got, want in zip(r[:-1], runs[0][:-1]):
            for g, w in zip(got, want):
                assert np.array_equal(g, w)
        assert r[-1] == runs[0][-1]


def test_subsets_order_growth_and_sharing_the_handle(monkeypatch):
    """Planning or updating a subset leaves the other trees' dumps as they
    were; a tree's results do not depend on which trees share its calls or in
    which order they are listed; a pool grown in place mid-plan
    (PP2D_POMDP_SLOTS_PER_QUERY=1) and plan_batch / single-tree calls on the
    same handle between batch calls give the same bits."""
    name = "map_10x10"
    grid = cases.load_bundled(name)
    n = 40
    beliefs = pf.gaussian_beliefs(grid, n, seed=13)
    other = pf.gaussian_beliefs(grid, 70, seed=14)

    def script(p, interleave):
        b = SearchTreeBatch(p, beliefs)
        res = []
        try:
            res.append(b.plan(None, 50, 4, with_stats=True))
            acts = res[-1][0]
            obs = [observation(b.dump(k), int(acts[k]), k) for k in range(n)]
            b.update(None, acts, obs)
            if interleave:
                p.plan_batch(other, max_depth=50, max_iter=3)
                t = SearchTree(p, other[0])
                t.plan(50, 3)
                t.close()
            # two calls in another order and split
            order = np.arange(n)[::-1]
            a1 = b.plan(order[:17], 50, 5, with_stats=True)
            if interleave:
                p.plan_batch(other[:30], max_depth=50, max_iter=2)
            a2 = b.plan(order[17:], 50, 5, with_stats=True)
            res.append(tuple(np.concatenate([x, y])[np.argsort(order)] for x, y in zip(a1, a2)))
            dumps = [b.dump(k).tobytes() for k in range(n)]
        finally:
            b.close()
        return [(a, bits(v), s) for a, v, s in res], dumps

    _, p, _ = planner(name)
    want, want_dumps = script(p, False)
    # subsets: the unlisted trees stay as they were
    b = SearchTreeBatch(p, beliefs)
    b.plan(None, 50, 4)
    before = [b.dump(k) for k in range(n)]
    sub = np.arange(0, n, 3)
    a, _ = b.plan(sub, 50, 3)
    rest = [k for k in range(n) if k not in set(sub.tolist())]
    assert all(same_dump(b.dump(k), before[k]) for k in rest)
    b.update(sub, a, [observation(b.dump(int(k)), int(a[j]), int(k)) for j, k in enumerate(sub)])
    assert all(same_dump(b.dump(k), before[k]) for k in rest)
    b.close()
    got, got_dumps = script(p, True)
    p.close()
    monkeypatch.setenv("PP2D_POMDP_SLOTS_PER_QUERY", "1")
    _, p, _ = planner(name)
    grown, grown_dumps = script(p, False)
    p.close()
    for g in (got, grown):
        for x, y in zip(g, want):
            for u, v in zip(x, y):
                assert np.array_equal(u, v)
    assert got_dumps == want_dumps and grown_dumps == want_dumps


def test_refused_calls_change_nothing_and_beliefs_stay_resident():
    grid, p, _ = planner("map_10x10")
    lib = p._lib
    beliefs = pf.gaussian_beliefs(grid, 6, seed=2)
    b = SearchTreeBatch(p, beliefs)
    acts, _ = b.plan([0, 1, 2, 3, 4], 50, 3)      # tree 5 stays unexpanded
    # a re-rooted tree gives the dropped subtrees' beliefs back (checked below)
    b.update([0], acts[:1], [observation(b.dump(0), int(acts[0]), 0)])
    b.plan([0], 50, 2)
    before = [b.dump(k) for k in range(6)]

    def refused(code, fn, *args):
        with pytest.raises(_lib.Pp2dError) as e:
            fn(*args)
        assert e.value.code == code
        assert all(same_dump(b.dump(k), before[k]) for k in range(6))
        return str(e.value)

    INV, ST = _lib.PP2D_ERR_INVALID, _lib.PP2D_ERR_STATE
    assert "tree 6" in refused(INV, b.update, [0, 6], [0, 0], [0, 0])
    assert "tree 1" in refused(INV, b.update, [1, 2, 1], [0, 0, 0], [0, 0, 0])
    assert "tree 3" in refused(INV, b.update, [0, 3], [0, 9], [0, 0])
    assert "tree 4" in refused(INV, b.update, [0, 4], [0, 0], [0, 16])
    assert "tree 5" in refused(ST, b.update, [0, 5], [0, 0], [0, 0])
    refused(INV, b.plan, [0, 7], 50, 3)
    refused(INV, b.plan, [2, 2], 50, 3)
    idx = np.zeros(1, np.uint32)
    z = np.zeros(1, np.uint8)
    assert lib.pp2d_tree_batch_update(b._b, None, 1, z.ctypes.data, z.ctypes.data) == INV
    assert lib.pp2d_tree_batch_update(b._b, idx.ctypes.data, 1, None, z.ctypes.data) == INV
    assert lib.pp2d_tree_batch_update(b._b, idx.ctypes.data, 1, z.ctypes.data, None) == INV
    assert lib.pp2d_tree_batch_plan(b._b, idx.ctypes.data, 1, 50, 3, None, None, None) == INV
    assert lib.pp2d_tree_batch_dump(b._b, 6, None, 0) < 0
    assert all(same_dump(b.dump(k), before[k]) for k in range(6))
    # the trees' beliefs stay in the pool: the model tables are fixed meanwhile
    tp, mp, sr = p.model_tables()
    refused(ST, p.set_model_tables, tp, mp, sr)
    b.close()
    p.set_model_tables(tp, mp, sr)                # destroy gave every slot back
    out = ctypes.c_void_p()
    assert lib.pp2d_tree_batch_create(p._h, None, 1, ctypes.byref(out)) == INV
    p.close()
