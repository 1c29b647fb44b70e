"""CPU tier of the closed-loop rollouts (pp2d_sim_rollout_mdp*): the shared
Philox4x32-10 against the Random123 known answers, the numpy mirror of the
generator and of the motion sampler against the oracle, the sampler's law, and
the argument checks that need no device."""
import ctypes

import numpy as np
import pytest

import rollout_oracle_py as ro
from path_planning_2d_b200 import _lib

KAT = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
       ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
       ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
        (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]


@pytest.mark.parametrize("counter,key,want", KAT)
def test_philox_known_answers(counter, key, want):
    assert tuple(int(v) for v in ro.philox(counter, key)) == want
    got = ro.philox_np(*[np.uint32(c) for c in counter], key[0], key[1])
    assert tuple(int(v) for v in got) == want


def test_numpy_uniforms_equal_the_oracle():
    seed = 0x0123456789abcdef
    episodes = np.array([0, 1, 7, 2**32 - 1, 2**32, 2**40 + 5], np.uint64)
    for t in (0, 1, 199, 2**31):
        got = ro.step_uniforms_np(seed, episodes, t)
        for i, e in enumerate(episodes):
            want = ro.step_uniforms(seed, int(e), t)
            assert np.array_equal(got[i].view(np.uint32), want.view(np.uint32))
    u = ro.step_uniforms_np(seed, np.arange(4096, dtype=np.uint64), 3)
    assert u.min() >= 0.0 and u.max() < 1.0


def test_sampler_law_equals_naive_prob():
    """Exact: a 24-bit uniform lands on slot i for ceil(cum_i 2^24) -
    ceil(cum_{i-1} 2^24) of the 2^24 values, which is naive_prob within 2^-22.
    The oracle agrees with the numpy sampler on both sides of every threshold
    and on a sample of Philox draws, whose frequencies are within 5 sigma."""
    full = 1 << 24
    for u in range(9):
        below = [min(int(np.ceil(np.float64(c) * full)), full) for c in ro.CUM[u]]
        counts = np.diff([0] + below)
        last = max(k for k in range(9) if ro.NAIVE[u, k] != 0)
        counts[last] += full - below[-1]      # r past the rounded total
        assert counts.sum() == full
        assert np.all(np.abs(counts / full - ro.NAIVE[u]) <= 2.0 ** -22), (u, counts)
        for c in ro.CUM[u]:
            for r in (np.nextafter(c, np.float32(0)), c):
                if 0 <= r < 1:
                    assert ro.motion_slot(u, r) == ro.motion_slots_np([u], [r])[0]
    r = ro.step_uniforms_np(7, np.arange(1 << 14, dtype=np.uint64), 0)[:, 0]
    n = r.size
    for u in range(9):
        slots = ro.motion_slots_np(np.full(n, u), r)
        sample = slots[:512]
        assert [ro.motion_slot(u, v) for v in r[:512]] == list(sample)
        freq = np.bincount(slots, minlength=9) / n
        for i in range(9):
            p = float(ro.NAIVE[u, i])
            assert abs(freq[i] - p) <= 5 * np.sqrt(max(p * (1 - p), 1e-12) / n) + 1e-12, (u, i)


def test_invalid_handles_without_a_device():
    lib = _lib.load()
    out = _lib.Rollout()
    starts = (ctypes.c_uint32 * 2)(0, 0)
    inst = (ctypes.c_uint32 * 1)(0)
    assert lib.pp2d_sim_rollout_mdp(None, None, 1, starts, None, 5, 1, 0,
                                    ctypes.byref(out)) == _lib.PP2D_ERR_INVALID
    assert lib.pp2d_sim_rollout_mdp_batch(None, None, inst, 1, starts, None, 5, 1, 0,
                                          ctypes.byref(out)) == _lib.PP2D_ERR_INVALID
    assert b"NULL" in lib.pp2d_last_error()
