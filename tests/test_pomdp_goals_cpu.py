"""CPU tier of goal sets: NULL handles and arguments of the new entry points
are refused before any device is touched, and the Python mirrors check their
arguments before calling the library."""
import ctypes

import numpy as np
import pytest

from path_planning_2d_b200 import DummySimulator, PomdpPathPlanning2d, SearchTreeBatch, _lib


def test_null_handles_and_arguments_are_refused_without_a_device():
    lib = _lib.load()
    INV = _lib.PP2D_ERR_INVALID
    xy = np.zeros(2, np.uint32)
    f = np.zeros(16, np.float32)
    u8 = np.zeros(9, np.uint8)
    out = ctypes.c_void_p()
    assert lib.pp2d_pomdp_set_goals(None, xy.ctypes.data, 1, None) == INV
    assert lib.pp2d_pomdp_goals(None, None, None) == INV
    assert lib.pp2d_pomdp_goal_reward(None, 0, f.ctypes.data) == INV
    assert lib.pp2d_pomdp_set_goal_alphas(None, 0, f.ctypes.data, u8.ctypes.data, None, None,
                                          0) == INV
    assert lib.pp2d_pomdp_padding_counters(None, np.zeros(2, np.uint64).ctypes.data) == INV
    assert lib.pp2d_tree_batch_create_goals(None, f.ctypes.data, xy.ctypes.data, 1,
                                            ctypes.byref(out)) == INV
    assert out.value is None
    assert b"NULL" in lib.pp2d_last_error()
    starts = np.zeros(2, np.uint32)
    g = np.zeros(1, np.uint32)
    for sim, planner, goals in ((None, None, g), (ctypes.c_void_p(1), None, g),
                                (ctypes.c_void_p(1), ctypes.c_void_p(1), None)):
        assert lib.pp2d_sim_rollout_pomdp_goals(
            sim, planner, goals.ctypes.data if goals is not None else None, 1,
            starts.ctypes.data, None, 10, 50, 15, 0, 0, None) == INV


def _fake_planner(h=3, w=4):
    """A PomdpPathPlanning2d without a device handle: only the Python-side
    argument checks can run on it."""
    p = object.__new__(PomdpPathPlanning2d)
    p.map_height, p.map_width = h, w
    p._lib = _lib.load()
    p._h = ctypes.c_void_p()
    p.search_tree = None
    p.max_search_tree_depth, p.max_online_iteration = 50, 15
    return p


def test_python_argument_checks():
    p = _fake_planner()
    hw = 12
    with pytest.raises(ValueError):
        p.set_goals([1, 2, 3])                            # not [n][2]
    with pytest.raises(ValueError):
        p.set_goals([(1, -1)])                            # negative coordinate
    with pytest.raises(ValueError):
        p.set_goals([(1.5, 1)])                           # not an integer
    with pytest.raises(ValueError):
        p.set_goals([(1, 1)], stage_rewards=np.zeros((2, hw, 9), np.float32))
    fib, pbvi = np.zeros((hw, 9), np.float32), np.zeros((3, hw), np.float32)
    with pytest.raises(ValueError):
        p.set_goal_alphas(-1, fib, pbvi)
    with pytest.raises(ValueError):
        p.set_goal_alphas(1.0, fib, pbvi)
    with pytest.raises(ValueError):
        p.set_goal_alphas(1, fib[:5], pbvi)
    beliefs = np.zeros((2, hw), np.float32)
    for goals in ([0], [0, 1, 2], [0, -1], [0.0, 1.0], [[0, 1]]):
        with pytest.raises(ValueError):
            SearchTreeBatch(p, beliefs, goals)
    sim = object.__new__(DummySimulator)
    sim.map_height, sim.map_width = 3, 4
    sim._lib, sim._h = _lib.load(), ctypes.c_void_p()
    starts = np.zeros((2, 2), np.uint32)
    with pytest.raises(ValueError):
        sim.rollout(p, starts, 5, 1, goals=[0])           # one goal per episode
    with pytest.raises(ValueError):
        sim.rollout(p, starts, 5, 1, goals=[0, -2])
    with pytest.raises(ValueError):
        sim.rollout(object(), starts, 5, 1, goals=[0, 0])  # goals are for the QV-tree planner
