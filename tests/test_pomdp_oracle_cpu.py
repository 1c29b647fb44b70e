"""CPU tier, QV-tree half: the oracle restatement against known answers, libc
and the golden outputs of the reference kernels (tests/golden/pomdp_*.npz,
generated on a B200 by `make_golden.py pomdp` through oracle/_ref)."""
import ctypes
import glob
import os

import numpy as np
import pytest

import cases
import pomdp_oracle_py as po


def test_glibc_rand_replica_matches_libc():
    libc = ctypes.CDLL("libc.so.6")
    for seed in (1, 2, 12345):
        libc.srand(seed)
        want = [libc.rand() for _ in range(2000)]
        assert po.glibc_rand(seed, 2000).tolist() == want


def test_model_known_answers():
    grid = np.zeros((5, 5), np.uint8)
    grid[1, 3] = 1
    m = po.Model(grid, (4, 4))
    tp = m.tp.reshape(25, 9, 9); mp = m.mp.reshape(25, 16); sr = m.sr.reshape(25, 9)
    c = 2 * 5 + 2                                   # (2,2): up-right (3,1) occupied
    assert np.allclose(tp.sum(2), 1.0, atol=1e-6)
    assert tp[c, 2, 2] == 0.0 and tp[c, 2, 4] == np.float32(np.float32(0.1) + np.float32(0.7))
    assert np.allclose(mp.sum(1), 1.0, atol=1e-6)   # sensor rows sum to 1
    assert mp[c, 0] == np.float32(np.float32(np.float32(np.float32(0.98) * np.float32(0.98))
                                             * np.float32(0.98)) * np.float32(0.98))
    assert sr[c, 4] == -2.0 and sr[4 * 5 + 4, 4] == 0.0
    assert np.isclose(sr[c, 2], -(0.1 + 2 * 0.7 + 0.1 + 0.1))
    occ = 1 * 5 + 3                                 # trapped AFTER the naive copy
    assert tp[occ, 0, 4] == 1.0 and np.count_nonzero(tp[occ, 0]) == 1
    assert np.isclose(sr[occ, 0], -(0.7 + 0.1 + 0.1 + 2 * 0.1))


def test_bayes_update_moves_mass_like_the_model():
    grid = np.zeros((7, 7), np.uint8)
    m = po.Model(grid, (6, 6))
    b = np.zeros(49, np.float32)
    b[3 * 7 + 3] = 1.0
    out, _ = m.bayes(b, 5, 0)                       # action 5 = move right
    L = m.mp.reshape(49, 16)[:, 0]
    want = np.zeros(49, np.float32)
    for k, p in ((5, 0.7), (2, 0.1), (8, 0.1), (4, 0.1)):
        idx = (3 + k // 3 - 1) * 7 + (3 + k % 3 - 1)
        want[idx] = np.float32(p) * L[idx]
    assert np.array_equal(out, want)
    out2, s = m.bayes(b, 5, 0, normalize=True)
    assert np.isclose(out2.sum(), 1.0, atol=1e-6) and np.isclose(s, want.sum(), rtol=1e-6)


def _golden():
    return sorted(glob.glob(os.path.join(cases.GOLDEN, "pomdp_*.npz")))


@pytest.mark.parametrize("path", _golden() or [None])
def test_oracle_matches_reference_kernels(path):
    """Bit-exact: B1 tables, B2 updates (incl. subnormal inputs), FIB sweeps
    and the device half of forward sampling."""
    if path is None:
        pytest.skip("tests/golden/pomdp_*.npz not generated yet")
    g = np.load(path)
    grid, goal = g["grid"], tuple(int(v) for v in g["goal"])
    m = po.Model(grid, goal)
    hw = grid.size
    bits = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)
    assert np.array_equal(bits(m.mp.reshape(hw, 16)), bits(g["meas_prob"]))
    assert np.array_equal(bits(m.sr.reshape(hw, 9)), bits(g["stage_reward"]))
    if "trans_prob" in g:
        assert np.array_equal(bits(m.tp.reshape(hw, 9, 9)), bits(g["trans_prob"]))
    for tag in ("uniform", "tiny"):
        b = g["b_" + tag]
        for i, (u, z) in enumerate(zip(g["us"], g["zs"])):
            out, _ = m.bayes(b, int(u), int(z))
            assert np.array_equal(bits(out), bits(g["bayes_" + tag][i])), (tag, i)
    fib, n = m.fib(cases.GAMMA, int(g["fib_sweeps"]))
    assert n == int(g["fib_sweeps"])
    assert np.array_equal(bits(fib), bits(g["fib"]))
    # device half of forward sampling: feed the recorded state samples
    un = np.load(os.path.join(cases.GOLDEN, "curand_xorwow_1234.npy"))
    tp = m.tp.reshape(hw, 9, 9); mp = m.mp.reshape(hw, 16)
    for a in range(9):
        for k, s1 in enumerate(g["samples"]):
            cum = np.float32(0); s2 = 0; found = False
            for j in range(9):
                cum = tp[s1, a, j] if j == 0 else np.float32(tp[s1, a, j] + cum)
                if not found and un[2 * k] <= cum:
                    s2, found = j, True
            nxt = int(s1) + (s2 // 3 - 1) * grid.shape[1] + (s2 % 3 - 1)
            cum = np.float32(0); z = 0; found = False
            for j in range(16):
                cum = mp[nxt, j] if j == 0 else np.float32(mp[nxt, j] + cum)
                if not found and un[2 * k + 1] <= cum:
                    z, found = j, True
            assert z == g["obs"][a, k], (a, k)


def test_oracle_matches_reference_record_of_the_live_kernel_case():
    """tests/golden/kernels_ref_syn_23x31.npz: the case of test_pomdp_gpu's
    live pin against the reference kernels -- tables, Bayes updates, FIB."""
    import sys
    sys.path.insert(0, cases.GOLDEN)
    import make_golden
    g = np.load(os.path.join(cases.GOLDEN, "kernels_ref_syn_23x31.npz"))
    grid, goal, b, us, zs, cap = make_golden.pomdp_live_case()
    m = po.Model(grid, goal)
    bits = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32).reshape(-1)
    assert np.array_equal(bits(m.tp), bits(g["trans_prob"]))
    assert np.array_equal(bits(m.mp), bits(g["meas_prob"]))
    assert np.array_equal(bits(m.sr), bits(g["stage_reward"]))
    for i, (u, z) in enumerate(zip(us, zs)):
        assert np.array_equal(bits(m.bayes(b, int(u), int(z))[0]), bits(g["bayes"][i])), i
    fib, n = m.fib(cases.GAMMA, cap)
    assert n == int(g["fib_sweeps"]) and np.array_equal(bits(fib), bits(g["fib"]))


def test_tree_runs_and_is_deterministic():
    import pomdp_fixtures as pf
    grid = cases.load_bundled("map_10x10")
    goal = (8, 7)
    m, fib, pbvi, fa, pa = pf.alphas("map_10x10", goal, n_pbvi=12)
    if not os.path.exists(os.path.join(cases.GOLDEN, "curand_xorwow_1234.npy")):
        pytest.skip("uniforms fixture missing")
    un = pf.uniforms()
    b = pf.gaussian_beliefs(grid, 1, seed=3)[0]
    res = []
    for _ in range(2):
        t = po.Tree(m, cases.GAMMA, fib, pbvi, un, b, fa, pa)
        a, r, stats, rc = t.plan(50, 6)
        res.append((a, r, stats.tolist(), rc))
        up, lo = t.root_bounds()
        assert lo <= up + 1e-4
        t.close()
    assert res[0] == res[1]
    assert res[0][2][0] > 9 and res[0][2][4] >= 2
