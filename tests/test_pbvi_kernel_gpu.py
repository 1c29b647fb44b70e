"""GPU tier: the offline PBVI solver's product path (PP2D_PBVI_CUBLAS=0, the
hand-written pbvi_sgemm_tn_kernel) against the CPU oracle of its defined
arithmetic (tests/pbvi_oracle.c), bit for bit: alpha vectors (as uint32),
actions and belief sets.

Unlike the comparison with the reference (tests/test_pbvi_gpu.py), which is
cuBLAS-ordered and therefore exact only where no arg-max is near-tied, this
comparison holds on every input, so the cases go where kernels go wrong:
set sizes at the edges of the 128 x 128 contraction tile, the 20-vector
Gamma_ao chunk and the 32-lane arg-max stride; maps whose live-cell count
leaves a ragged last K chunk of 16 (or fits in one); exact ties (duplicate
beliefs, point masses); subnormal belief entries (the contraction and the
rewards keep them, Gamma_ao flushes); the dense inner dimension; the
reference's iteration count; and the belief-set expansion at the sizes where
the heap sort and the mid-round break start.  Every backup case also checks
with the oracle's arg-max indices that its last iteration discriminated
between Gamma_ao vectors, so that equality is not vacuous."""
import os

import numpy as np
import pytest

import cases
import pbvi_oracle_py as pbo
from path_planning_2d_b200 import PomdpPathPlanning2d, _lib

pytestmark = pytest.mark.gpu
bits = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)
SMALL = ["pbvi_ref_map_3x3_g0.5_n12", "pbvi_ref_map_10x10_g0.8_n40",
         "pbvi_ref_map_10x10_g0.95_n60", "pbvi_ref_map_5x5_g0.7_n25"]


@pytest.fixture(autouse=True)
def product_kernel(monkeypatch):
    monkeypatch.setenv("PP2D_PBVI_CUBLAS", "0")
    monkeypatch.delenv("PP2D_POMDP_DENSE", raising=False)


def free_map(h, w):
    return np.zeros((h, w), np.uint8), (w // 2, h // 2)


def random_set(rng, live, n, support=0.6):
    """n beliefs with random support on the live cells, +0 elsewhere, each
    scaled to sum 1 in float32."""
    cells = np.flatnonzero(live.reshape(-1))
    B = np.zeros((n, live.size), np.float32)
    for b in range(n):
        pick = cells[rng.random(cells.size) < support]
        if pick.size == 0:
            pick = cells[rng.integers(cells.size, size=1)]
        B[b, pick] = rng.random(pick.size, dtype=np.float32) + np.float32(0.01)
        B[b] /= B[b].sum(dtype=np.float32)
    return B


def assert_backup_equals_oracle(grid, goal, gamma, B, iterations, min_distinct=3):
    with PomdpPathPlanning2d(grid, goal, gamma) as p:
        al, ac = p.backupAlphaVectors(B, iterations=iterations)
    want_al, want_ac, argmax, _ = pbo.Pbvi(grid, goal, gamma).backup(B, iterations)
    assert np.unique(argmax).size >= min(min_distinct, B.shape[0]), "case does not discriminate"
    assert np.array_equal(ac, want_ac)
    assert np.array_equal(bits(al), bits(want_al))


@pytest.mark.parametrize("name", SMALL)
def test_fixture_solve_equals_oracle(name):
    """The full pointBasedValueIteration; the 60- and 25-belief fixtures are
    the ones the reference pins only up to near-tied arg-max decisions."""
    g = np.load(os.path.join(cases.GOLDEN, name + ".npz"))
    n = g["belief_set"].shape[0]
    with PomdpPathPlanning2d(g["grid"], tuple(int(v) for v in g["goal"]), float(g["gamma"])) as p:
        bs, al, ac = p.pointBasedValueIteration(g["b0"], n, rand_seed=1)
    o = pbo.Pbvi(g["grid"], g["goal"], g["gamma"])
    want_bs = o.expand(g["b0"], n, rand_seed=1)
    want_al, want_ac, argmax, _ = o.backup(want_bs)
    assert np.array_equal(bits(bs), bits(want_bs))
    assert np.unique(argmax).size >= 3
    assert np.array_equal(ac, want_ac)
    assert np.array_equal(bits(al), bits(want_al))


@pytest.mark.parametrize("n", [1, 2, 19, 20, 21, 63, 64, 65, 127, 128, 129, 257])
def test_backup_set_size_at_tile_edges(n):
    """128 x 128 contraction tiles, 20-vector Gamma_ao chunks, 32-lane arg-max
    stride.  Iteration 1 contracts all-zero Gamma_ao, iteration 2 is full of
    exact ties."""
    grid = cases.load_bundled("map_10x10")
    goal = (8, 1)
    with PomdpPathPlanning2d(grid, goal, 0.9) as p:
        _, live = p.live_cells(mask=True)
    B = random_set(np.random.default_rng(n), live, n)
    assert_backup_equals_oracle(grid, goal, 0.9, B, iterations=3 + n % 4)


MAPS = {
    "free_1x9": (free_map(1, 9), None),
    "free_9x1": (free_map(9, 1), None),
    "syn_7x5": (cases.synthetic_map(7, 5, 0.2, seed=2), None),
    "map_10x10": ((cases.load_bundled("map_10x10"), (8, 1)), None),
    "syn_3x5_K_below_16": (cases.synthetic_map(3, 5, 0.25, seed=3), "below"),
    "syn_5x9_K_mod16_1": (cases.synthetic_map(5, 9, 0.25, seed=3), 1),
    "syn_6x11_K_mod16_0": (cases.synthetic_map(6, 11, 0.25, seed=3), 0),
    "syn_6x11_K_mod16_15": (cases.synthetic_map(6, 11, 0.25, seed=5), 15),
}


@pytest.mark.parametrize("name", list(MAPS))
def test_backup_maps(name):
    (grid, goal), residue = MAPS[name]
    with PomdpPathPlanning2d(grid, goal, 0.85) as p:
        K, live = p.live_cells(mask=True)
    if residue == "below":
        assert K < 16
    elif residue is not None:
        assert K > 16 and K % 16 == residue, K
    B = random_set(np.random.default_rng(K), live, 30)
    assert_backup_equals_oracle(grid, goal, 0.85, B, iterations=5)


def test_backup_duplicates_and_point_masses():
    """Exact ties: duplicate beliefs give duplicate alpha vectors (ties in R,
    first index wins) and duplicate rewards; point masses tie actions."""
    grid, goal = cases.load_bundled("map_10x10"), (8, 1)
    with PomdpPathPlanning2d(grid, goal, 0.9) as p:
        _, live = p.live_cells(mask=True)
    rng = np.random.default_rng(11)
    cells = np.flatnonzero(live.reshape(-1))
    point = np.zeros((12, grid.size), np.float32)
    point[np.arange(12), rng.choice(cells, 12, replace=False)] = 1.0
    base = np.concatenate([random_set(rng, live, 10), point])
    B = base[rng.integers(base.shape[0], size=70)]
    assert_backup_equals_oracle(grid, goal, 0.9, B, iterations=6)


def test_backup_subnormal_entries():
    """Beliefs with subnormal entries on live cells and whole rows in the
    subnormal range: the contraction and the rewards keep them (FTZ would make
    every product +0 and every decision a tie)."""
    grid, goal = cases.load_bundled("map_10x10"), (8, 1)
    with PomdpPathPlanning2d(grid, goal, 0.9) as p:
        _, live = p.live_cells(mask=True)
    rng = np.random.default_rng(12)
    B = random_set(rng, live, 40)
    B[:12] *= np.float32(2.0 ** -140)
    cells = np.flatnonzero(live.reshape(-1))
    for b in range(12, 24):
        B[b, rng.choice(cells, 5, replace=False)] = np.float32(3e-41)
    assert np.count_nonzero((B != 0) & (np.abs(B) < np.finfo(np.float32).tiny)) > 100
    assert_backup_equals_oracle(grid, goal, 0.9, B, iterations=5)


@pytest.mark.parametrize("variant", ["neg_zero_on_dead_cell", "mass_on_occupied_cell",
                                     "PP2D_POMDP_DENSE"])
def test_backup_dense_inner_dimension(variant, monkeypatch):
    """Each variant makes the kernel contract over all cells instead of the
    live ones; the oracle is always dense, so the bits must not change."""
    grid, goal = cases.load_bundled("map_10x10"), (8, 1)
    with PomdpPathPlanning2d(grid, goal, 0.9) as p:
        _, live = p.live_cells(mask=True)
    B = random_set(np.random.default_rng(13), live, 33)
    occ = np.flatnonzero(grid.reshape(-1) == 1)
    assert not live.reshape(-1)[occ].any()
    if variant == "neg_zero_on_dead_cell":
        B[5, occ[0]] = np.float32(-0.0)
    elif variant == "mass_on_occupied_cell":
        B[5, occ[:3]] = np.float32(0.125)
    else:
        monkeypatch.setenv("PP2D_POMDP_DENSE", "1")
    assert_backup_equals_oracle(grid, goal, 0.9, B, iterations=5)


@pytest.mark.parametrize("gamma", [0.5, 0.8])
def test_backup_reference_iteration_count(gamma):
    grid, goal = cases.synthetic_map(7, 5, 0.2, seed=2)
    with PomdpPathPlanning2d(grid, goal, gamma) as p:
        _, live = p.live_cells(mask=True)
    B = random_set(np.random.default_rng(14), live, 24)
    assert_backup_equals_oracle(grid, goal, gamma, B, iterations=0)


@pytest.mark.parametrize("gamma", [0.0, 1.0, 1.5, float("nan")])
def test_reference_iteration_count_needs_gamma_in_unit_interval(gamma):
    """The reference's count ceil(log(2e-4) / log(gamma)) is undefined outside
    0 < gamma < 1: both entry points refuse iterations = 0 there, and an
    explicit count still runs."""
    grid, goal = cases.synthetic_map(7, 5, 0.2, seed=2)
    with PomdpPathPlanning2d(grid, goal, gamma) as p:
        _, live = p.live_cells(mask=True)
        B = random_set(np.random.default_rng(15), live, 8)
        with pytest.raises(_lib.Pp2dError) as e:
            p.backupAlphaVectors(B)
        assert e.value.code == _lib.PP2D_ERR_INVALID
        with pytest.raises(_lib.Pp2dError) as e:
            p.pointBasedValueIteration(B[0], 8)
        assert e.value.code == _lib.PP2D_ERR_INVALID
        al, ac = p.backupAlphaVectors(B, iterations=2)
    want_al, want_ac, _, _ = pbo.Pbvi(grid, goal, gamma).backup(B, 2)
    assert np.array_equal(ac, want_ac)
    # a NaN's payload is the hardware's, not the arithmetic's: compare NaN positions
    nan = np.isnan(want_al)
    assert np.array_equal(np.isnan(al), nan)
    assert np.array_equal(bits(al)[~nan], bits(want_al)[~nan])


EXPAND_MAPS = {"map_10x10": (cases.load_bundled("map_10x10"), (8, 1)),
               "syn_9x13": cases.synthetic_map(9, 13, 0.2, seed=5)}


@pytest.mark.parametrize("seed", [1, 7])
@pytest.mark.parametrize("start", ["uniform", "point_mass"])
@pytest.mark.parametrize("name", list(EXPAND_MAPS))
def test_expansion_equals_oracle(name, start, seed):
    """generateBeliefSet below, at and above the 100 beliefs from which a round
    heap-sorts its candidates, and across the mid-round break; pool slots are
    recycled between calls on one handle, so a repeated call must give the
    same bits."""
    grid, goal = EXPAND_MAPS[name]
    free = (grid.reshape(-1) == 0).astype(np.float32)
    if start == "uniform":
        b0 = free / free.sum(dtype=np.float32)
    else:
        b0 = np.zeros(grid.size, np.float32)
        b0[np.flatnonzero(free)[3]] = 1.0
    o = pbo.Pbvi(grid, goal, 0.9)
    with PomdpPathPlanning2d(grid, goal, 0.9) as p:
        first = None
        for size in (2, 10, 99, 100, 101, 230):
            got = p.generateBeliefSet(b0, size, rand_seed=seed)
            assert np.array_equal(bits(got), bits(o.expand(b0, size, rand_seed=seed))), size
            first = got if first is None else first
        assert np.array_equal(bits(p.generateBeliefSet(b0, 2, rand_seed=seed)), bits(first))
