"""GPU tier: the offline PBVI solver (pp2d_pomdp_generate_belief_set /
backup_alphas / solve_pbvi, SURVEY.md section 8f "next" #2) against what the
reference's OWN solver produced.

Parity contract (DESIGN.md section 7a).  Belief-set expansion, Gamma_ao, the
gather/adds and the selection are order-defined in the reference and must be
bit-exact.  The one dense contraction R = Gamma_ao^T B (cublasSgemm in the
reference) only feeds an arg-max; cuBLAS's summation order is unspecified, so
the reference's alpha vectors are defined only up to arg-max decisions between
entries of R that agree to the last bits -- and PBVI amplifies a flipped
decision over its 167 iterations.  Therefore:
  * with PP2D_PBVI_CUBLAS=1 (the library call as a CHECKER) every fixture,
    including the 500-belief bundled-map case, must be reproduced bit for bit:
    this pins every other step of the solver;
  * the product path (hand-written pbvi_sgemm_tn_kernel, defined summation
    order) must be bit-exact wherever no near-tie occurs (the small fixtures,
    and any case for the first iterations) and otherwise produce a valid
    lower-bound set of the same quality: every alpha vector below the FIB
    upper bound, lower bound at the belief points within 1e-3 (500 beliefs) /
    5e-2 (60 beliefs) relative of the reference's.

tests/golden/pbvi_ref_*.npz are outputs of generateBeliefSet /
backupAlphaVectors / fastInformedBound of the unmodified reference
translation units (oracle/_ref/libpp2d_ref_pomdp_full.so) run on a B200 by
tools/ref_offline.py, rand() seeded like a fresh process; map_5x5 (the case of
the live test below) is its record in the same layout, `make_golden.py
live_cases`.  The bundled-map
case (500 beliefs x 4000 cells, 167 backups; 165 s + 228 s in the reference)
is stored as one CRC-32 per belief / alpha vector.  Bar: bit-exact."""
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import cases
from path_planning_2d_b200 import PomdpPathPlanning2d

pytestmark = pytest.mark.gpu
bits = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)
SMALL = ["pbvi_ref_map_3x3_g0.5_n12", "pbvi_ref_map_10x10_g0.8_n40",
         "pbvi_ref_map_10x10_g0.95_n60", "pbvi_ref_map_5x5_g0.7_n25"]


def crc_rows(rows):
    return np.array([zlib.crc32(np.ascontiguousarray(r).tobytes()) for r in rows], np.uint32)


@pytest.fixture(params=["kernel", "cublas"])
def gemm(request, monkeypatch):
    """Product contraction kernel / the reference's library call as a checker."""
    monkeypatch.setenv("PP2D_PBVI_CUBLAS", "1" if request.param == "cublas" else "0")
    return request.param


# fixtures on which the product kernel meets no near-tied arg-max
TIE_FREE = {"pbvi_ref_map_3x3_g0.5_n12", "pbvi_ref_map_10x10_g0.8_n40"}


def lower_bound(bs, al):
    return (bs.astype(np.float64) @ al.astype(np.float64).T).max(axis=1)


@pytest.mark.parametrize("name", SMALL)
def test_pbvi_equals_reference_solver(name, gemm):
    g = np.load(os.path.join(cases.GOLDEN, name + ".npz"))
    goal = tuple(int(v) for v in g["goal"])
    n = g["belief_set"].shape[0]
    with PomdpPathPlanning2d(g["grid"], goal, float(g["gamma"])) as p:
        fib, fa, _ = p.fastInformedBound()
        assert np.array_equal(bits(fib), bits(g["fib"]))
        assert np.array_equal(fa, g["fib_actions"])
        bs = p.generateBeliefSet(g["b0"], n, rand_seed=1)
        assert np.array_equal(bits(bs), bits(g["belief_set"]))
        al, ac = p.backupAlphaVectors(g["belief_set"])
        if gemm == "cublas" or name in TIE_FREE:
            assert np.array_equal(bits(al), bits(g["pbvi"]))
            assert np.array_equal(ac, g["pbvi_actions"])
        else:
            ref, got = lower_bound(bs, g["pbvi"]), lower_bound(bs, al)
            assert np.abs(got - ref).max() <= 5e-2 * np.abs(ref).max()
        # the fused entry point gives the same three arrays
        bs2, al2, ac2 = p.pointBasedValueIteration(g["b0"], n, rand_seed=1)
        assert np.array_equal(bits(bs2), bits(bs))
        assert np.array_equal(bits(al2), bits(al)) and np.array_equal(ac2, ac)
        # every alpha vector is a lower bound: below the FIB upper bound
        p.set_alphas(fib, al, fa, ac)
        up, _, lo, _ = p.evaluate(bs)
        assert np.all(lo <= up + 1e-3 * np.abs(up))


def test_pbvi_bundled_map_500_beliefs_equals_reference_solver(monkeypatch):
    g = np.load(os.path.join(cases.GOLDEN, "pbvi_ref_sparse_map_100x40_g0.95_n500_crc.npz"))
    grid = cases.load_bundled("sparse_map_100x40")
    goal = tuple(int(v) for v in g["goal"])
    out = {}
    for variant in ("cublas", "kernel"):
        monkeypatch.setenv("PP2D_PBVI_CUBLAS", "1" if variant == "cublas" else "0")
        with PomdpPathPlanning2d(grid, goal, float(g["gamma"])) as p:
            fib, fa, _ = p.fastInformedBound()
            assert zlib.crc32(fib.tobytes()) == int(g["fib_crc"])
            bs, al, ac = p.pointBasedValueIteration(g["b0"], 500, rand_seed=1)
            p.set_alphas(fib, al, fa, ac)
            up, _, lo, _ = p.evaluate(bs)
        out[variant] = (bs, al, ac)
        assert np.array_equal(bits(bs[:4]), bits(g["belief_set_head"]))
        assert np.array_equal(crc_rows(bs), g["belief_set_crc"])
        assert np.all(lo <= up + 1e-3 * np.abs(up))          # a lower bound everywhere
    # the checker reproduces the reference's solve bit for bit ...
    bs, al, ac = out["cublas"]
    assert np.array_equal(bits(al[:4]), bits(g["pbvi_head"]))
    assert np.array_equal(crc_rows(al), g["pbvi_crc"])
    assert np.array_equal(ac, g["pbvi_actions"])
    # ... and the product kernel gives a lower-bound set of the same quality
    ref, got = lower_bound(bs, al), lower_bound(bs, out["kernel"][1])
    assert np.abs(got - ref).max() <= 1e-3 * np.abs(ref).max()


@pytest.mark.parametrize("name", ["pbvi_ref_map_10x10_g0.95_n60"])
def test_handwritten_gemm_picks_the_same_vectors_as_the_library_call(monkeypatch, name):
    """pbvi_sgemm_tn_kernel (the product) vs the reference's cublasSgemm call
    (PP2D_PBVI_CUBLAS=1, checker only): the contraction only feeds an arg-max,
    so both must end with bit-identical alpha vectors and actions; a belief
    with mass on an occupied cell switches the kernel to the dense inner
    dimension and must still agree."""
    g = np.load(os.path.join(cases.GOLDEN, name + ".npz"))
    goal = tuple(int(v) for v in g["goal"])
    bs = g["belief_set"].copy()
    res = {}
    for variant in ("kernel", "cublas", "kernel_dense"):
        monkeypatch.setenv("PP2D_PBVI_CUBLAS", "1" if variant == "cublas" else "0")
        with PomdpPathPlanning2d(g["grid"], goal, float(g["gamma"])) as p:
            if variant == "kernel_dense":
                b2 = bs.copy()
                occ = np.flatnonzero(g["grid"].reshape(-1) == 1)[0]
                b2[3, occ] = np.float32(0.0)          # still zero: same problem ...
                b2[3, occ] = np.float32(-0.0)         # ... but -0 forces the dense path
                res[variant] = p.backupAlphaVectors(b2, iterations=12)
            else:
                res[variant] = p.backupAlphaVectors(bs, iterations=12)
    for variant in ("cublas", "kernel_dense"):
        assert np.array_equal(bits(res[variant][0]), bits(res["kernel"][0])), variant
        assert np.array_equal(res[variant][1], res["kernel"][1]), variant


def test_pbvi_single_belief_and_other_seed():
    grid, goal = cases.synthetic_map(7, 9, 0.2, seed=4)
    free = (grid.reshape(-1) == 0).astype(np.float32)
    b0 = free / free.sum(dtype=np.float32)
    with PomdpPathPlanning2d(grid, goal, 0.6) as p:
        bs = p.generateBeliefSet(b0, 1)
        assert np.array_equal(bits(bs[0]), bits(b0))
        al, ac = p.backupAlphaVectors(bs, iterations=3)
        assert al.shape == (1, grid.size) and np.all(np.isfinite(al))
        a = p.generateBeliefSet(b0, 30, rand_seed=1)
        b = p.generateBeliefSet(b0, 30, rand_seed=7)
        assert np.array_equal(bits(a), bits(p.generateBeliefSet(b0, 30, rand_seed=1)))
        assert not np.array_equal(bits(a), bits(b))
        s = a.sum(axis=1)
        assert np.allclose(s, 1.0, atol=1e-4)


def test_pbvi_equals_live_reference(tmp_path, monkeypatch):
    """The same comparison against the reference stack run now, in its own
    process (it keeps its state in globals), on a case that is not committed."""
    so = os.path.join(cases.ROOT, "oracle", "_ref", "libpp2d_ref_pomdp_full.so")
    if not os.path.exists(so):
        pytest.skip("oracle/_ref/libpp2d_ref_pomdp_full.so not built")
    out = str(tmp_path / "ref.npz")
    subprocess.run([sys.executable, os.path.join(cases.ROOT, "tools", "ref_offline.py"),
                    "map_5x5", "3", "2", "0.7", "25", out], check=True, timeout=600,
                   stdout=subprocess.DEVNULL)
    g = np.load(out)
    monkeypatch.setenv("PP2D_PBVI_CUBLAS", "1")          # the checker: bit-exact by contract
    with PomdpPathPlanning2d(g["grid"], (3, 2), 0.7) as p:
        bs, al, ac = p.pointBasedValueIteration(g["b0"], 25, rand_seed=1)
    assert np.array_equal(bits(bs), bits(g["belief_set"]))
    assert np.array_equal(bits(al), bits(g["pbvi"]))
    assert np.array_equal(ac, g["pbvi_actions"])
