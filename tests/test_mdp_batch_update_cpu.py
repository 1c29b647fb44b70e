"""CPU tier: pp2d_mdp_batch_update refuses a NULL handle and NULL arguments
before any CUDA call, and is bound in Python with the header's signature."""
import ctypes

import numpy as np
import pytest

from path_planning_2d_b200 import MdpBatchPathPlanning2d, _lib


def test_null_handle_and_arguments_are_refused():
    lib = _lib.load()
    idx = np.zeros(1, np.uint32)
    grid = np.zeros((4, 4), np.uint8)
    goals = np.zeros((1, 2), np.uint32)
    args = [None, idx.ctypes.data, 1, grid.ctypes.data, 0, goals.ctypes.data]
    assert lib.pp2d_mdp_batch_update(*args) == _lib.PP2D_ERR_INVALID
    assert b"NULL" in lib.pp2d_last_error()
    # a non-NULL handle with a NULL argument is refused before the handle is read
    fake = ctypes.c_void_p(1)
    for i in (1, 3, 5):
        bad = [fake] + args[1:]
        bad[i] = None
        assert lib.pp2d_mdp_batch_update(*bad) == _lib.PP2D_ERR_INVALID
        assert b"NULL" in lib.pp2d_last_error()


def test_update_is_bound_with_the_header_signature():
    assert "pp2d_mdp_batch_update" in _lib.SIGNATURES
    res, argtypes = _lib.SIGNATURES["pp2d_mdp_batch_update"]
    assert res is ctypes.c_int
    assert argtypes == [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p,
                        ctypes.c_size_t, ctypes.c_void_p]
    assert hasattr(_lib.load(), "pp2d_mdp_batch_update")
    assert callable(MdpBatchPathPlanning2d.update_map)


def test_python_update_map_checks_shapes_before_the_library():
    b = MdpBatchPathPlanning2d.__new__(MdpBatchPathPlanning2d)
    b.map_height, b.map_width, b.count = 4, 5, 3
    b._h = ctypes.c_void_p()
    with pytest.raises(ValueError):       # wrong map size
        b.update_map([0], np.zeros((4, 4), np.uint8), [(0, 0)])
    with pytest.raises(ValueError):       # one goal for two instances
        b.update_map([0, 1], np.zeros((4, 5), np.uint8), [(0, 0)])
    with pytest.raises(ValueError):       # three maps for two instances
        b.update_map([0, 1], np.zeros((3, 4, 5), np.uint8), [(0, 0), (1, 1)])
