"""CPU tier: the arg-max rule of pomdp_bounds_kernel, restated lane by lane.

The kernel gives one warp to a belief's row of values: FIB columns 0..8 on
lanes 0..8, PBVI column j on lane j % 32 (strided lane loop), then an xor
butterfly over (value, index) pairs.  `bounds_warp` below is that reduction
step for step; it is compared here with the oracle's choice
(`oracle_pomdp_evaluate_fib/pbvi`, i.e. std::max_element: index 0 if its value
is NaN, else the first maximum of the other values) on vectors full of NaN,
+-0, +-inf and exact ties.  The GPU tests hold the kernel itself to the oracle;
this file pins the rule on a machine without a GPU."""
import numpy as np
import pytest

import pomdp_oracle_py as po

NAN, INF = np.float32(np.nan), np.float32(np.inf)


def _take(b, i, ob, oi):
    """Butterfly step: does lane (b, i) take its partner's (ob, oi)?"""
    return oi >= 0 and (i < 0 or b < ob or (b == ob and oi < i) or ob != ob)


def bounds_warp(vals, n_pbvi):
    """(fib index, pbvi index) pomdp_bounds_kernel returns for one row
    [9 FIB values | n_pbvi PBVI values] (pbvi index 0 when n_pbvi = 0)."""
    v = np.asarray(vals, np.float32)
    bu, iu = [np.float32(0)] * 32, [-1] * 32
    bl, il = [np.float32(0)] * 32, [-1] * 32
    for lane in range(32):
        if lane < 9:
            bu[lane] = v[lane]
            if lane == 0 or bu[lane] == bu[lane]:
                iu[lane] = lane
        for j in range(lane, n_pbvi, 32):
            x = v[9 + j]
            if ((j == 0 or x == x) if il[lane] < 0 else bl[lane] < x):
                bl[lane], il[lane] = x, j
    off = 16
    while off:
        nu, niu, nl, nil = list(bu), list(iu), list(bl), list(il)
        for lane in range(32):
            o = lane ^ off
            if _take(bu[lane], iu[lane], bu[o], iu[o]):
                nu[lane], niu[lane] = bu[o], iu[o]
            if _take(bl[lane], il[lane], bl[o], il[o]):
                nl[lane], nil[lane] = bl[o], il[o]
        bu, iu, bl, il = nu, niu, nl, nil
        off >>= 1
    return iu[0], max(il[0], 0)


def max_element(v):
    best = 0
    for a in range(1, len(v)):
        if v[best] < v[a]:
            best = a
    return best


def oracle_choice(vals, n_pbvi):
    """The oracle's (fib index, pbvi index) for the row: on a one-cell map
    with belief [1] every inner product is +0 + 1 * alpha = alpha (a -0 alpha
    gives +0, which compares as -0 does).  The PBVI index comes back through
    two action tables (low and high byte)."""
    v = np.asarray(vals, np.float32)
    b = np.ones(1, np.float32)
    fib = v[None, :9]
    pbvi = np.ascontiguousarray(v[9:, None]) if n_pbvi else np.zeros((0, 1), np.float32)
    idx = np.arange(max(n_pbvi, 1))
    lo8, hi8 = (idx & 255).astype(np.uint8), (idx >> 8).astype(np.uint8)
    fa = np.arange(9, dtype=np.uint8)
    up, ua, lo, la = po.evaluate(b, fib, pbvi, fa, lo8 if n_pbvi else None)
    _, _, _, lh = po.evaluate(b, fib, pbvi, fa, hi8 if n_pbvi else None)
    return ua, la | (lh << 8), up, lo


def check(vals, n_pbvi):
    got = bounds_warp(vals, n_pbvi)
    ua, la, up, lo = oracle_choice(vals, n_pbvi)
    assert got == (ua, la), (got, (ua, la))
    v = np.asarray(vals, np.float32)
    assert got[0] == max_element(v[:9])
    if n_pbvi:
        assert got[1] == max_element(v[9:9 + n_pbvi])
    # the value the kernel reports is the chosen element (the oracle's is the
    # same up to the sign of a zero)
    for val, want in ((v[got[0]], up), (v[9 + got[1]] if n_pbvi else np.float32(0), lo)):
        assert (np.isnan(val) and np.isnan(want)) or val == want


@pytest.mark.parametrize("vals,n_pbvi,want", [
    # FIB: a NaN in lane 1 must not swallow the maximum in lane 7
    ([1, NAN, 0.5, 0, 0, 0, 0, 3, 0], 0, (7, 0)),
    # FIB: NaN at index 0 wins
    ([NAN, 1, 2, 3, 4, 5, 6, 7, 8], 0, (0, 0)),
    # PBVI, same lane: NaN at column 2, maximum at column 34
    ([0] * 9 + [0, 0, NAN] + [0] * 31 + [5] + [0] * 5, 40, (0, 34)),
    # PBVI, across the butterfly: NaN at column 1, maximum at column 17
    ([0] * 9 + [1, NAN] + [0] * 14 + [2, 3] + [0] * 22, 40, (0, 17)),
    # PBVI: NaN at column 0 beats +inf elsewhere
    ([0] * 9 + [NAN] + [INF] * 40, 40, (0, 0)),
    # every value NaN: index 0
    ([NAN] * 9 + [NAN] * 70, 70, (0, 0)),
    # +0 and -0 are a tie: the first one wins, wherever the lanes put it
    ([-0.0, 0.0, -1, -1, -1, -1, -1, -1, -1] + [-1] * 33 + [-0.0] + [-1] * 20 + [0.0], 55, (0, 33)),
])
def test_known_rows(vals, n_pbvi, want):
    assert bounds_warp(vals, n_pbvi) == want
    check(vals, n_pbvi)


@pytest.mark.parametrize("seed", range(4))
def test_random_rows_with_nan_zeros_infinities_and_ties(seed):
    """2 000 rows of 0..600 PBVI columns over a few distinct values (so that
    ties cross lanes, strides and column tiles), with NaN, +-0 and +-inf."""
    rng = np.random.default_rng(seed)
    pool = np.array([NAN, 0.0, -0.0, INF, -INF, 1.0, -1.0, 2.5, 2.5, -3.0], np.float32)
    for _ in range(500):
        n_pbvi = int(rng.choice([0, 1, 31, 32, 33, 64, 65, int(rng.integers(1, 601))]))
        v = rng.standard_normal(9 + n_pbvi).astype(np.float32)
        k = int(rng.integers(0, 9 + n_pbvi))
        pos = rng.integers(0, 9 + n_pbvi, size=k)
        v[pos] = pool[rng.integers(0, pool.size, size=k)]
        if rng.random() < 0.3:                        # exact duplicates of the maximum
            top = 9 + int(np.nanargmax(np.where(np.isnan(v[9:]), -np.inf, v[9:]))) if n_pbvi else 0
            for d in (16, 32, 256):
                if top + d < v.size:
                    v[top + d] = v[top]
        if rng.random() < 0.2:
            v[int(rng.choice([0, 9])) if n_pbvi else 0] = NAN
        check(v, n_pbvi)
