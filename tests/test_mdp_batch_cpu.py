"""CPU tier: pp2d_mdp_batch_create / _reset refuse bad arguments before any
CUDA call, and every batch entry point is bound."""
import ctypes

import numpy as np

from path_planning_2d_b200 import MdpBatchPathPlanning2d, _lib

BATCH_SYMBOLS = [
    "pp2d_mdp_batch_create", "pp2d_mdp_batch_reset", "pp2d_mdp_batch_destroy",
    "pp2d_mdp_batch_set_stream", "pp2d_mdp_batch_sweeps", "pp2d_mdp_batch_residual",
    "pp2d_mdp_batch_solve", "pp2d_mdp_batch_download", "pp2d_mdp_batch_plan",
    "pp2d_mdp_batch_waypoints", "pp2d_mdp_batch_sweep_counts",
    "pp2d_mdp_batch_work_counters",
]


def _create(h, w, count, maps, stride, goals):
    lib = _lib.load()
    out = ctypes.c_void_p()
    rc = lib.pp2d_mdp_batch_create(h, w, count, maps, stride, goals, 0.95,
                                   ctypes.byref(out))
    assert out.value is None
    return rc, lib.pp2d_last_error().decode()


def test_null_pointers_are_refused():
    lib = _lib.load()
    grid = np.zeros((4, 4), np.uint8)
    goals = np.zeros((1, 2), np.uint32)
    assert _create(4, 4, 1, None, 0, goals.ctypes.data)[0] == _lib.PP2D_ERR_INVALID
    assert _create(4, 4, 1, grid.ctypes.data, 0, None)[0] == _lib.PP2D_ERR_INVALID
    assert lib.pp2d_mdp_batch_create(4, 4, 1, grid.ctypes.data, 0, goals.ctypes.data, 0.95,
                                     None) == _lib.PP2D_ERR_INVALID
    assert lib.pp2d_mdp_batch_reset(None, grid.ctypes.data, 0,
                                    goals.ctypes.data) == _lib.PP2D_ERR_INVALID
    for name in ("pp2d_mdp_batch_sweeps",):
        assert getattr(lib, name)(None, 1) == _lib.PP2D_ERR_INVALID
    assert lib.pp2d_mdp_batch_residual(None, None) == _lib.PP2D_ERR_INVALID
    assert lib.pp2d_mdp_batch_solve(None, None, None, 0) == _lib.PP2D_ERR_INVALID
    assert lib.pp2d_mdp_batch_download(None, 0, 1, None, None) == _lib.PP2D_ERR_INVALID
    assert lib.pp2d_mdp_batch_plan(None, None, None, 0, None) == _lib.PP2D_ERR_INVALID
    n = ctypes.c_uint32()
    assert lib.pp2d_mdp_batch_waypoints(None, 0, 0, 0, None, 0,
                                        ctypes.byref(n)) == _lib.PP2D_ERR_INVALID
    assert lib.pp2d_mdp_batch_sweep_counts(None, None) == _lib.PP2D_ERR_INVALID
    assert lib.pp2d_mdp_batch_work_counters(None, None) == _lib.PP2D_ERR_INVALID
    assert lib.pp2d_mdp_batch_set_stream(None, None) == _lib.PP2D_ERR_INVALID
    lib.pp2d_mdp_batch_destroy(None)


def test_empty_batch_and_bad_stride_are_refused():
    grid = np.zeros((4, 4), np.uint8)
    goals = np.zeros((2, 2), np.uint32)
    rc, msg = _create(4, 4, 0, grid.ctypes.data, 0, goals.ctypes.data)
    assert rc == _lib.PP2D_ERR_INVALID and "instance" in msg
    rc, _ = _create(0, 4, 2, grid.ctypes.data, 0, goals.ctypes.data)
    assert rc == _lib.PP2D_ERR_INVALID
    rc, msg = _create(4, 4, 2, grid.ctypes.data, 15, goals.ctypes.data)
    assert rc == _lib.PP2D_ERR_INVALID and "map_stride" in msg


def test_goal_outside_the_map_names_the_instance():
    maps = np.zeros((3, 4, 5), np.uint8)
    goals = np.array([[0, 0], [4, 3], [5, 0]], np.uint32)
    rc, msg = _create(4, 5, 3, maps.ctypes.data, 20, goals.ctypes.data)
    assert rc == _lib.PP2D_ERR_INVALID
    assert "instance 2" in msg and "outside" in msg


def test_occupied_goal_names_the_instance():
    maps = np.zeros((3, 4, 4), np.uint8)
    maps[1, 2, 3] = 1
    goals = np.array([[3, 2], [3, 2], [0, 0]], np.uint32)
    rc, msg = _create(4, 4, 3, maps.ctypes.data, 16, goals.ctypes.data)
    assert rc == _lib.PP2D_ERR_GOAL_OCCUPIED
    assert "instance 1" in msg and "occupied" in msg
    # the shared map (stride 0): every instance reads the same map
    rc, msg = _create(4, 4, 3, maps[1].ctypes.data, 0, goals.ctypes.data)
    assert rc == _lib.PP2D_ERR_GOAL_OCCUPIED and "instance 0" in msg


def test_stacked_grid_too_large_is_refused_before_reading_the_goals():
    grid = np.zeros((1, 1), np.uint8)
    goals = np.zeros((1, 2), np.uint32)     # far fewer than `count`: never read
    # 2^31 instances of 1x1: 2^32 - 1 rows
    rc, msg = _create(1, 1, 1 << 31, grid.ctypes.data, 0, goals.ctypes.data)
    assert rc == _lib.PP2D_ERR_INVALID and "too large" in msg
    # few rows, but too many elements in one plane
    rc, msg = _create(1, 1 << 28, 16, grid.ctypes.data, 0, goals.ctypes.data)
    assert rc == _lib.PP2D_ERR_INVALID and "too large" in msg


def test_batch_symbols_are_bound():
    lib = _lib.load()
    for name in BATCH_SYMBOLS:
        assert name in _lib.SIGNATURES, name
        assert hasattr(lib, name), name
    assert _lib.SIGNATURES["pp2d_mdp_batch_create"][1][4] is ctypes.c_size_t
    for m in ("valueIteration", "sweeps", "residual", "reset", "sweep_counts",
              "work_counters", "download", "plan_batch", "waypoints", "close", "__enter__"):
        assert callable(getattr(MdpBatchPathPlanning2d, m)), m


def test_python_class_checks_shapes_before_the_library():
    import pytest
    with pytest.raises(ValueError):
        MdpBatchPathPlanning2d(np.zeros((2, 4, 4), np.uint8), [(0, 0)] * 3, 0.95)
    with pytest.raises(ValueError):
        MdpBatchPathPlanning2d(np.zeros(4, np.uint8), [(0, 0)], 0.95)
