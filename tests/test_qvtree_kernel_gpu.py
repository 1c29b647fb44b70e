"""GPU tier, QV-tree half: bound evaluation, batched planning and the FIB
solver against the CPU oracle (oracle/pomdp_oracle.c) where kernels go wrong.

Every comparison is bit for bit (any NaN equals any NaN, see `same`); indices,
actions and tree statistics are exactly equal.  The cases sit at the edges of
the kernels' tiles and loops:
  * pomdp_values_kernel: 64 beliefs x 256 columns per CTA, K chunks of 16
    inner rows -- column counts 9 + n_pbvi at and across each column tile,
    belief counts across the 64-belief tile, maps whose live-cell count leaves
    a ragged last chunk of 0, 1 or 15 rows, or no live cell at all;
  * pomdp_bounds_kernel: 32 lanes, strided lane loop, xor butterfly -- the
    winning vector placed at lane / stride / column-tile edges, exact
    duplicates 16, 32 and 256 columns apart, NaN and +-inf values;
  * the batch: 1 x 9 to 96 x 97 maps (more than 8 192 live cells: the second
    pass of pomdp_support_list_kernel), query counts across the staging (64)
    and sorting (128) thresholds and the group counts, un-normalised starts
    (the sampling clamp) and point masses (plateaus in the prefix sums, a
    prefix sum equal to a draw);
  * the FIB solver on small and odd maps, at several discounts and caps, and
    the discounts its stopping rule cannot reach.
Each arg-max case asserts that the winners are not all in the first tile, so
that passing means something."""
import numpy as np
import pytest

import cases
import pomdp_fixtures as pf
import pomdp_oracle_py as po
from path_planning_2d_b200 import PomdpPathPlanning2d, SearchTree, _lib

pytestmark = pytest.mark.gpu
GAMMA = cases.GAMMA
bits = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)
NAN, INF = np.float32(np.nan), np.float32(np.inf)


@pytest.fixture(autouse=True)
def default_paths(monkeypatch):
    for k in ("PP2D_POMDP_DENSE", "PP2D_POMDP_TILE_SUPPORT", "PP2D_POMDP_SORT",
              "PP2D_POMDP_GROUPS", "PP2D_POMDP_SLOTS_PER_QUERY"):
        monkeypatch.delenv(k, raising=False)


def same(a, b):
    """Bit-equal, except that any NaN equals any NaN."""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    return bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


def live_mask(m):
    """numpy mirror of pomdp_dead_cells_kernel on the oracle's tables: a cell
    is live when some in-map neighbour s != itself has P(s, u, cell) != 0."""
    h, w = m.h, m.w
    tp = m.tp.reshape(h, w, 9, 9)
    ys, xs = np.mgrid[0:h, 0:w]
    live = np.zeros((h, w), bool)
    for s in range(9):
        if s == 4:
            continue
        sy, sx = ys + s // 3 - 1, xs + s % 3 - 1
        ok = (sy >= 0) & (sy < h) & (sx >= 0) & (sx < w)
        nz = (tp[:, :, :, 8 - s] != 0).any(-1)
        live[ok] |= nz[sy[ok], sx[ok]]
    return live.reshape(-1)


def walled_in():
    grid = np.ones((5, 5), np.uint8)
    grid[2, 2] = 0
    return grid, (2, 2)


MAPS = {
    "1x1": (np.zeros((1, 1), np.uint8), (0, 0)),
    "1x9": (np.zeros((1, 9), np.uint8), (4, 0)),
    "9x1": (np.zeros((9, 1), np.uint8), (0, 4)),
    "2x2": (np.zeros((2, 2), np.uint8), (1, 1)),
    "3x3": (cases.load_bundled("map_3x3"), (1, 1)),
    "7x5": cases.synthetic_map(7, 5, 0.2, seed=2),
    "33x65": cases.synthetic_map(33, 65, 0.25, seed=3),
    # live-cell count (checked below) 112 = 0, 113 = 1, 111 = 15 mod 16
    "11x13_K_mod16_0": cases.synthetic_map(11, 13, 0.25, seed=6),
    "11x13_K_mod16_1": cases.synthetic_map(11, 13, 0.25, seed=0),
    "11x13_K_mod16_15": cases.synthetic_map(11, 13, 0.25, seed=7),
    "walled_in": walled_in(),
    # 8 796 live cells: more than 8 192, the 256 mask words of one list pass
    "96x97": cases.synthetic_map(96, 97, 0.05, seed=0),
}
RESIDUE = {"11x13_K_mod16_0": 0, "11x13_K_mod16_1": 1, "11x13_K_mod16_15": 15}

_models = {}


def model(name):
    if name not in _models:
        grid, goal = MAPS[name]
        m = po.Model(grid, goal)
        _models[name] = (grid, goal, m, live_mask(m))
    return _models[name]


def check_live(p, name):
    grid, goal, m, live = model(name)
    K, mask = p.live_cells(mask=True)
    assert np.array_equal(mask.reshape(-1).astype(bool), live)
    if name in RESIDUE:
        assert K > 16 and K % 16 == RESIDUE[name], K
    if name == "walled_in":
        assert K == 0
    if name == "96x97":
        assert K > 8192
    return K


# ---------------------------------------------------------------- inputs ----
def beliefs_for(name, n, seed):
    """Gaussian bumps, uniform over the free cells, point masses and rows with
    subnormal entries, cycled to n rows; all +0 on the dead cells."""
    grid, goal, m, live = model(name)
    rng = np.random.default_rng(seed)
    hw = grid.size
    cells = np.flatnonzero(live)
    out = np.zeros((n, hw), np.float32)
    free = grid.reshape(-1) == 0
    if cells.size == 0:
        # no live cell: +0 rows, and rows with mass on the free (dead) cells,
        # which make the launch dense
        out[1::2, free] = np.float32(1.0 / free.sum())
        return out
    gauss = pf.gaussian_beliefs(grid, n, sigma=1.5, seed=seed)
    for i in range(n):
        k = i % 4
        if k == 0:
            out[i] = gauss[i] * live
            s = out[i].sum(dtype=np.float32)
            if s == 0:
                out[i, cells[0]] = 1
            else:
                out[i] /= s
        elif k == 1:
            out[i, cells] = np.float32(1.0 / cells.size)
        elif k == 2:
            out[i, rng.choice(cells)] = 1
        else:
            out[i, cells] = (rng.random(cells.size, dtype=np.float32) * np.float32(2.0 ** -140))
            out[i, rng.choice(cells)] = np.float32(3e-41)
    return out


PLACES = (0, 31, 32, 247, 248, 300)


def alpha_set(name, n_pbvi, seed, dup=False):
    """Random FIB and PBVI vectors with regional strong vectors: the maximiser
    of a belief depends on where its mass is.  The strong PBVI vectors sit at
    PLACES (lane, stride and column-tile edges); with dup, the strong vectors
    at 3 and 40 are copied exactly to +16, +32 and +256 (ties across lanes,
    strides and tiles: the smaller index must win)."""
    grid = MAPS[name][0]
    hw = grid.size
    rng = np.random.default_rng(seed)
    region = rng.integers(0, 6, size=hw)
    fib = rng.standard_normal((hw, 9)).astype(np.float32)
    for a in range(9):
        fib[region == a % 6, a] += np.float32(3 + a % 3)
    fib[:, 6] = fib[:, 2]                    # an exact FIB tie
    pbvi = rng.standard_normal((n_pbvi, hw)).astype(np.float32)
    strong = [j for j in ((3, 40) if dup else PLACES) if j < n_pbvi]
    for k, j in enumerate(strong):
        pbvi[j, region == k % 6] += np.float32(4)
    if dup:
        for j in strong:
            for d in (16, 32, 256):
                if j + d < n_pbvi:
                    pbvi[j + d] = pbvi[j]
    idx = np.arange(n_pbvi)
    # actions that tell j, j + 16, j + 32 and j + 256 apart
    pa = ((idx * 7 + 3) % 251).astype(np.uint8)
    return fib, pbvi, np.arange(9, dtype=np.uint8)[::-1].copy(), pa


def oracle_eval(beliefs, fib, pbvi):
    """Per belief: (upper, fib index, lower, pbvi index) of the oracle."""
    n_pbvi = pbvi.shape[0]
    idx = np.arange(max(n_pbvi, 1))
    lo8, hi8 = (idx & 255).astype(np.uint8), (idx >> 8).astype(np.uint8)
    out = []
    for b in beliefs:
        up, ua, lo, la = po.evaluate(b, fib, pbvi, None, lo8 if n_pbvi else None)
        lh = po.evaluate(b, fib, pbvi, None, hi8 if n_pbvi else None)[3] if n_pbvi else 0
        out.append((up, ua, lo, la | (lh << 8)))
    return out


def assert_evaluate(p, beliefs, fib, pbvi, fa, pa):
    up, ua, lo, la = p.evaluate(beliefs)
    want = oracle_eval(beliefs, fib, pbvi)
    for i, (wu, wi, wl, wj) in enumerate(want):
        assert same(up[i], wu) and ua[i] == fa[wi], i
        assert same(lo[i], wl), i
        assert la[i] == (pa[wj] if pbvi.shape[0] else 0), i
    return np.array([w[1] for w in want]), np.array([w[3] for w in want])


# ------------------------------------------------------- bound evaluation ---
@pytest.mark.parametrize("n_pbvi", [0, 1, 23, 31, 32, 33, 247, 248, 503, 504])
def test_evaluate_column_tiles_and_belief_counts(n_pbvi):
    """ncol = 9 + n_pbvi = 9 ... 513 (at and across the 256-column tiles),
    1 ... 257 beliefs (across the 64-belief tile), on a map whose 111 live
    cells leave a last K chunk of 15 rows."""
    name = "11x13_K_mod16_15"
    grid, goal, m, live = model(name)
    fib_winners, winners = [], []
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
        check_live(p, name)
        for dup in (False, True):
            fib, pbvi, fa, pa = alpha_set(name, n_pbvi, seed=n_pbvi, dup=dup)
            p.set_alphas(fib, pbvi, fa, pa)
            for n in (1, 63, 64, 65, 129, 257):
                B = beliefs_for(name, n, seed=n)
                wi, wj = assert_evaluate(p, B, fib, pbvi, fa, pa)
                fib_winners.append(wi)
                winners.append(wj)
    wj = np.concatenate(winners)
    assert np.unique(np.concatenate(fib_winners)).size >= 3
    if n_pbvi >= 248:
        assert (wj + 9 >= 256).any() and (wj + 9 < 256).any(), "winners in one column tile"
    if n_pbvi > 32:
        assert np.unique(wj).size >= 3 and (wj >= 32).any()


@pytest.mark.parametrize("name", [k for k in MAPS if k not in ("96x97",)])
def test_evaluate_maps(name):
    """Maps from 1 x 1 up, ragged last K chunks, the walled-in map (no live
    cell: the inner dimension falls back to one row)."""
    grid, goal, m, live = model(name)
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
        check_live(p, name)
        for n_pbvi in (0, 33, 248):
            fib, pbvi, fa, pa = alpha_set(name, n_pbvi, seed=7 + n_pbvi, dup=n_pbvi == 248)
            p.set_alphas(fib, pbvi, fa, pa)
            for n in (1, 65, 129):
                assert_evaluate(p, beliefs_for(name, n, seed=n + n_pbvi), fib, pbvi, fa, pa)


@pytest.mark.parametrize("variant", ["neg_zero_on_dead_cell", "mass_on_occupied_cell",
                                     "PP2D_POMDP_DENSE"])
def test_evaluate_dense_inner_dimension(variant, monkeypatch):
    name = "11x13_K_mod16_15"
    grid, goal, m, live = model(name)
    if variant == "PP2D_POMDP_DENSE":
        monkeypatch.setenv("PP2D_POMDP_DENSE", "1")
    B = beliefs_for(name, 129, seed=3)
    dead = np.flatnonzero(~live)
    if variant == "neg_zero_on_dead_cell":
        B[70, dead[0]] = np.float32(-0.0)
    elif variant == "mass_on_occupied_cell":
        B[70, dead[:3]] = np.float32(0.125)
    fib, pbvi, fa, pa = alpha_set(name, 300, seed=5, dup=True)
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
        p.set_alphas(fib, pbvi, fa, pa)
        assert_evaluate(p, B, fib, pbvi, fa, pa)


# ---------------------------------------------------- non-finite bounds -----
def nonfinite_alphas(name, n_pbvi=40):
    """Alpha sets with +inf, -inf and NaN in some FIB and some PBVI columns:
    a belief that is +0 where a column holds +-inf gets NaN there, one with
    mass gets +-inf, so rows mix NaN, infinities and finite values.  FIB: +inf
    at column 0 and 1, -inf at 5, the finite maximum at 7.  PBVI: NaN alpha in
    column 2, +inf in 1, the maxima at 17 and 34.  Column 0 of both holds -inf
    on one cell: rows with mass there have -inf at index 0, all others NaN
    (index 0 wins).  Returns the alphas and the six cells c."""
    grid, goal, m, live = model(name)
    hw = grid.size
    fib, pbvi, fa, pa = alpha_set(name, n_pbvi, seed=11)
    rng = np.random.default_rng(12)
    c = rng.choice(np.flatnonzero(live), size=6, replace=False)
    fib[:, 7] += np.float32(8)
    fib[c[0], 1] = INF
    fib[c[1], 5] = -INF
    fib[c[2], 0] = -INF
    pbvi[17] += np.float32(6)
    pbvi[34] += np.float32(7) * (np.arange(hw) % 2)
    pbvi[2, c[3]] = NAN
    pbvi[1, c[4]] = INF
    pbvi[0, c[5]] = -INF
    return (fib, pbvi, fa, pa), c


def nonfinite_rows(name, n, c, seed):
    """Beliefs with mass on c[2] and c[5] (-inf, not NaN, at both columns 0)
    and on a third live cell, none on c[0] and c[4]: NaN in FIB column 1 and
    PBVI columns 1 and 2 next to finite maxima (FIB 7; PBVI 17 or 34)."""
    grid, goal, m, live = model(name)
    rng = np.random.default_rng(seed)
    other = np.setdiff1d(np.flatnonzero(live), c)
    B = np.zeros((n, grid.size), np.float32)
    for i in range(n):
        w = rng.dirichlet(np.ones(3)).astype(np.float32)
        B[i, [c[2], c[5], rng.choice(other)]] = w
    return B


def test_evaluate_nonfinite_alphas():
    name = "33x65"
    grid, goal, m, live = model(name)
    (fib, pbvi, fa, pa), c = nonfinite_alphas(name)
    B = np.concatenate([beliefs_for(name, 100, seed=4), nonfinite_rows(name, 100, c, 5)])
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
        p.set_alphas(fib, pbvi, fa, pa)
        up, ua, lo, la = p.evaluate(B)
        wi, wj = assert_evaluate(p, B, fib, pbvi, fa, pa)
    # NaN values next to finite maxima, in both bounds, do occur
    assert np.isnan(up).any() and (wi == 7).any() and (wi == 0).any()
    assert (wj == 0).any() and ((wj == 17) | (wj == 34)).any()


def test_evaluate_nonfinite_beliefs_under_finite_alphas():
    """NaN and +inf entries on live cells (the inner products keep them)."""
    name = "33x65"
    grid, goal, m, live = model(name)
    fib, pbvi, fa, pa = alpha_set(name, 300, seed=9, dup=True)
    B = beliefs_for(name, 130, seed=6)
    cells = np.flatnonzero(live)
    B[::5, cells[100]] = NAN
    B[1::5, cells[-1]] = INF
    B[2::7, cells[7]] = NAN
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
        p.set_alphas(fib, pbvi, fa, pa)
        assert_evaluate(p, B, fib, pbvi, fa, pa)


def plan_all_ways(p, m, gamma, fib, pbvi, fa, pa, B, max_iter, oracle_rows, max_depth=50):
    """plan_batch against a fresh SearchTree.plan for every query and the
    oracle Tree for oracle_rows; returns the oracle stats of those rows."""
    acts, vals, stats = p.plan_batch(B, max_depth=max_depth, max_iter=max_iter,
                                     with_stats=True)
    for i in range(B.shape[0]):
        st = SearchTree(p, B[i])
        a, r = st.plan(max_depth, max_iter)
        d = st.getDepth()
        st.close()
        assert a == acts[i] and same(r, vals[i]) and d == stats[i, 2], i
    ostats = []
    for i in oracle_rows:
        ot = po.Tree(m, gamma, fib, pbvi, pf.uniforms(), B[i], fa, pa)
        oa, orr, os_, rc = ot.plan(max_depth, max_iter)
        ot.close()
        assert acts[i] == oa and same(vals[i], orr), i
        assert (stats[i, 0], stats[i, 1], stats[i, 2]) == (os_[0], os_[1], os_[4]), i
        ostats.append(os_)
    return acts, vals, stats, np.array(ostats)


@pytest.mark.parametrize("kind", ["alphas", "beliefs"])
def test_plan_with_nonfinite_bounds(kind):
    """SearchTree.plan and plan_batch against the oracle Tree with non-finite
    alpha sets, and with start beliefs holding NaN / +inf on live cells (their
    children are NaN: the per-tile row lists must keep NaN rows)."""
    name = "11x13_K_mod16_1"
    grid, goal, m, live = model(name)
    B = beliefs_for(name, 130, seed=8)
    if kind == "alphas":
        (fib, pbvi, fa, pa), c = nonfinite_alphas(name)
        B[1::2] = nonfinite_rows(name, 65, c, 9)
    else:
        _, fib, pbvi, fa, pa = pf.alphas(grid, goal, n_pbvi=40, fib_sweeps=30)
        cells = np.flatnonzero(live)
        B[0::6, cells[50]] = NAN
        B[1::6, cells[20]] = INF
        B[2::6] *= np.float32(0.5)
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
        p.set_alphas(fib, pbvi, fa, pa)
        plan_all_ways(p, m, GAMMA, fib, pbvi, fa, pa, B, 4, oracle_rows=range(0, 130, 3))
        # the root bounds, NaN for a start with a NaN entry, are the oracle's
        st = SearchTree(p, B[0])
        got = st.rootBounds()
        st.close()
    ot = po.Tree(m, GAMMA, fib, pbvi, pf.uniforms(), B[0], fa, pa)
    want = ot.root_bounds()
    ot.close()
    assert same(got, want)
    assert np.isnan(want).all() if kind == "beliefs" else np.isinf(want).all()


# ---------------------------------------------- batched planning, ragged ----
def starts(name, n, seed):
    """Gaussian starts, point masses (plateaus in the prefix sums), starts
    scaled by 0.5 (draws past the last prefix sum: the sampling clamp), and
    two-cell starts whose first prefix sum equals the tree's first draw."""
    grid, goal, m, live = model(name)
    B = beliefs_for(name, n, seed)
    cells = np.flatnonzero(live)
    rng = np.random.default_rng(seed)
    r0 = np.float32(po.glibc_rand(1, 1)[0]) / np.float32(2.0 ** 31)
    for i in range(n):
        if i % 5 == 3:
            B[i] *= np.float32(0.5)
        elif i % 5 == 4 and cells.size > 1:
            c1, c2 = np.sort(rng.choice(cells, 2, replace=False))
            B[i] = 0
            B[i, c1] = r0
            B[i, c2] = np.float32(1) - r0
    return B


@pytest.mark.parametrize("name", ["1x9", "9x1", "3x3", "7x5"])
def test_plan_batch_small_maps(name):
    grid, goal, m, live = model(name)
    _, fib, pbvi, fa, pa = pf.alphas(grid, goal, n_pbvi=40, fib_sweeps=30)
    B = starts(name, 70, seed=1)
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
        check_live(p, name)
        p.set_alphas(fib, pbvi, fa, pa)
        acts, vals, stats, ostats = plan_all_ways(p, m, GAMMA, fib, pbvi, fa, pa, B, 6,
                                                  oracle_rows=range(70))
    assert (ostats[3::5, 3] > 0).all(), "the sampling clamp did not run"
    assert stats[:, 0].max() > 20


@pytest.mark.parametrize("n", [1, 63, 64, 65, 127, 128, 129, 255, 256, 384])
def test_plan_batch_query_counts(n, monkeypatch):
    """Across the page-locked staging (64 queries), the mode sort (128) and
    the 1 / 2 / 3 pipelined groups (256, 384); 384 also with 4 groups."""
    name = "33x65"
    grid, goal, m, live = model(name)
    _, fib, pbvi, fa, pa = pf.alphas(grid, goal, n_pbvi=40, fib_sweeps=30)
    B = starts(name, n, seed=n)
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
        p.set_alphas(fib, pbvi, fa, pa)
        rows = sorted({0, n // 2, n - 1, 3 % n, 4 % n})
        acts, vals, stats, ostats = plan_all_ways(p, m, GAMMA, fib, pbvi, fa, pa, B, 3, rows)
        if n == 384:
            monkeypatch.setenv("PP2D_POMDP_GROUPS", "4")
            a4, v4, s4 = p.plan_batch(B, max_depth=50, max_iter=3, with_stats=True)
            assert np.array_equal(a4, acts) and same(v4, vals) and np.array_equal(s4, stats)
    if 3 in rows:
        assert ostats[rows.index(3), 3] > 0, "the sampling clamp did not run"


def test_plan_batch_more_than_8192_live_cells(monkeypatch):
    """96 x 97 map with 8 796 live cells: the row lists of the values launch
    need the second 256-word pass.  Per-tile rows off and mode sort off give
    the same bits; a sample equals the oracle."""
    name = "96x97"
    grid, goal, m, live = model(name)
    _, fib, pbvi, fa, pa = pf.alphas(grid, goal, n_pbvi=40, fib_sweeps=10)
    B = starts(name, 130, seed=2)
    # starts near the end of the live list, so that the rows past 8 192 matter
    cells = np.flatnonzero(live)
    for i in range(0, 130, 4):
        B[i] = 0
        B[i, cells[-1 - 7 * i]] = 1
    results = []
    with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
        check_live(p, name)
        p.set_alphas(fib, pbvi, fa, pa)
        results.append(p.plan_batch(B, max_depth=50, max_iter=2, with_stats=True))
    for tile, sort in (("0", "1"), ("1", "0")):
        monkeypatch.setenv("PP2D_POMDP_TILE_SUPPORT", tile)
        monkeypatch.setenv("PP2D_POMDP_SORT", sort)
        with PomdpPathPlanning2d(grid, goal, GAMMA) as p:
            p.set_alphas(fib, pbvi, fa, pa)
            results.append(p.plan_batch(B, max_depth=50, max_iter=2, with_stats=True))
    acts, vals, stats = results[0]
    for a, v, s in results[1:]:
        assert np.array_equal(a, acts) and same(v, vals) and np.array_equal(s, stats)
    for i in (0, 3, 8, 64, 129):
        ot = po.Tree(m, GAMMA, fib, pbvi, pf.uniforms(), B[i], fa, pa)
        oa, orr, os_, rc = ot.plan(50, 2)
        ot.close()
        assert acts[i] == oa and same(vals[i], orr), i
        assert (stats[i, 0], stats[i, 1], stats[i, 2]) == (os_[0], os_[1], os_[4]), i


# ------------------------------------------------------------ FIB solver ----
FIB_MAPS = ["1x1", "1x9", "9x1", "2x2", "7x5", "33x65"]


@pytest.mark.parametrize("gamma", [0.0, 0.5, 0.95, 0.99])
@pytest.mark.parametrize("name", FIB_MAPS)
def test_fib_solver(name, gamma):
    """Caps 1, 10 and 11 (a cap is rounded up to whole 10-sweep checks), and
    the uncapped stopping rule where the oracle runs it within a second."""
    grid, goal, m, live = model(name)
    caps = [1, 10, 11] + ([0] if grid.size < 100 or gamma <= 0.5 else [])
    with PomdpPathPlanning2d(grid, goal, gamma) as p:
        for cap in caps:
            want, n = m.fib(gamma, cap)
            got, acts, sweeps = p.fastInformedBound(cap)
            assert sweeps == n, cap
            assert acts.tolist() == list(range(9))
            assert np.array_equal(bits(got), bits(want)), cap
            if cap:
                assert sweeps == (cap + 9) // 10 * 10


@pytest.mark.parametrize("gamma", [1.0, 1.5, -1.0, float("nan")])
def test_fib_solver_without_cap_needs_a_contraction(gamma):
    """With |gamma| >= 1 or a NaN gamma the stopping rule is not reached in
    useful time: max_sweeps = 0 is refused, an explicit cap still runs.  (With
    a NaN gamma the first check already passes: NaN differences are dropped.)"""
    grid, goal, m, live = model("7x5")
    with PomdpPathPlanning2d(grid, goal, gamma) as p:
        with pytest.raises(_lib.Pp2dError) as e:
            p.fastInformedBound()
        assert e.value.code == _lib.PP2D_ERR_INVALID
        got, _, sweeps = p.fastInformedBound(20)
    want, n = m.fib(gamma, 20)
    assert sweeps == n == (10 if np.isnan(gamma) else 20)
    assert same(got, want)
