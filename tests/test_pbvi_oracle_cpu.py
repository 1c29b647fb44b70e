"""CPU tier of the PBVI oracle (tests/pbvi_oracle.c): the solver of csrc/pbvi.cu
restated in its defined arithmetic, pinned to the reference's own outputs
(tests/golden/pbvi_ref_*.npz, see tests/test_pbvi_gpu.py).

* Expansion is order-defined in the reference: the oracle reproduces every
  committed belief set bit for bit, including the 500-belief bundled-map case,
  whose rounds of 128, 228, 328 and 428 beliefs take the heap-sort branch.
* The backup's contraction is cuBLAS-ordered in the reference and one
  ascending FMA chain per entry in the product (and in the oracle).  Where no
  arg-max is decided by the last bits (the two tie-free fixtures) the oracle
  reproduces the reference bit for bit; elsewhere it meets the lower-bound
  tolerance the GPU tier applies to the product kernel.
* The contraction on its own against float64, so that a transposed or
  mis-strided oracle cannot pass the comparisons of the GPU tier."""
import os
import zlib

import numpy as np
import pytest

import cases
import pbvi_oracle_py as pbo

bits = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)
SMALL = ["pbvi_ref_map_3x3_g0.5_n12", "pbvi_ref_map_10x10_g0.8_n40",
         "pbvi_ref_map_10x10_g0.95_n60", "pbvi_ref_map_5x5_g0.7_n25"]
TIE_FREE = {"pbvi_ref_map_3x3_g0.5_n12", "pbvi_ref_map_10x10_g0.8_n40"}


def lower_bound(bs, al):
    return (bs.astype(np.float64) @ al.astype(np.float64).T).max(axis=1)


@pytest.mark.parametrize("name", SMALL)
def test_expansion_reproduces_reference_belief_set(name):
    g = np.load(os.path.join(cases.GOLDEN, name + ".npz"))
    p = pbo.Pbvi(g["grid"], g["goal"], g["gamma"])
    bs = p.expand(g["b0"], g["belief_set"].shape[0], rand_seed=1)
    assert np.array_equal(bits(bs), bits(g["belief_set"]))


def test_expansion_reproduces_bundled_map_500_beliefs():
    g = np.load(os.path.join(cases.GOLDEN, "pbvi_ref_sparse_map_100x40_g0.95_n500_crc.npz"))
    p = pbo.Pbvi(cases.load_bundled("sparse_map_100x40"), g["goal"], g["gamma"])
    bs = p.expand(g["b0"], 500, rand_seed=1)
    assert np.array_equal(bits(bs[:4]), bits(g["belief_set_head"]))
    crc = np.array([zlib.crc32(np.ascontiguousarray(r).tobytes()) for r in bs], np.uint32)
    assert np.array_equal(crc, g["belief_set_crc"])


@pytest.mark.parametrize("name", SMALL)
def test_backup_against_reference_solver(name):
    g = np.load(os.path.join(cases.GOLDEN, name + ".npz"))
    p = pbo.Pbvi(g["grid"], g["goal"], g["gamma"])
    al, ac, _, it = p.backup(g["belief_set"])
    assert it == pbo.reference_iterations(g["gamma"])
    if name in TIE_FREE:
        assert np.array_equal(bits(al), bits(g["pbvi"]))
        assert np.array_equal(ac, g["pbvi_actions"])
    else:
        ref, got = lower_bound(g["belief_set"], g["pbvi"]), lower_bound(g["belief_set"], al)
        assert np.abs(got - ref).max() <= 5e-2 * np.abs(ref).max()


@pytest.mark.parametrize("gamma,count", [(0.5, 13), (0.8, 39), (0.95, 167), (0.7, 24)])
def test_reference_iteration_count(gamma, count):
    assert pbo.reference_iterations(gamma) == count


@pytest.mark.parametrize("n,hw", [(1, 1), (3, 17), (20, 100), (37, 131), (129, 45)])
def test_contraction_within_fp32_chain_bound_of_float64(n, hw):
    """R[o][b][i] = sum_s G[o][i][s] B[b][s]: a chain of hw FMAs from +0 is
    within hw * 2^-24 * sum |G||B| of the exact value (1 % slack).  G and B are
    not symmetric, so a transposed or mis-strided result fails."""
    rng = np.random.default_rng(n * 1000 + hw)
    G = rng.standard_normal((2, n, hw)).astype(np.float32)
    B = rng.random((n, hw), dtype=np.float32)
    B[:, rng.random(hw) < 0.2] = 0.0
    R = pbo.contract(G, B)
    assert R.shape == (2, n, n)
    G64, B64 = G.astype(np.float64), B.astype(np.float64)
    R64 = np.einsum("ois,bs->obi", G64, B64)
    mag = np.einsum("ois,bs->obi", np.abs(G64), np.abs(B64))
    assert np.all(np.abs(R - R64) <= 1.01 * hw * 2.0**-24 * mag)
    # the same contraction one observation at a time
    assert np.array_equal(bits(pbo.contract(G[1], B)), bits(R[1]))
