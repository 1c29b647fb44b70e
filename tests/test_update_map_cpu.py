"""CPU tier: pp2d_mdp_update_map refuses NULL arguments before any CUDA
call, with the error codes of pp2d_mdp_reset."""
import ctypes

import numpy as np

from path_planning_2d_b200 import MdpPathPlanning2d, _lib


def test_update_map_null_arguments():
    lib = _lib.load()
    grid = np.zeros((4, 4), np.uint8)
    assert lib.pp2d_mdp_update_map(None, grid.ctypes.data, 0, 0) == _lib.PP2D_ERR_INVALID
    assert b"NULL" in lib.pp2d_last_error()
    assert lib.pp2d_mdp_update_map(None, None, 0, 0) == _lib.PP2D_ERR_INVALID
    # a non-NULL handle with a NULL map is refused before the handle is read
    fake = ctypes.c_void_p(1)
    assert lib.pp2d_mdp_update_map(fake, None, 0, 0) == _lib.PP2D_ERR_INVALID


def test_python_update_map_is_bound():
    assert callable(MdpPathPlanning2d.update_map)
    assert _lib.SIGNATURES["pp2d_mdp_update_map"][1][0] is ctypes.c_void_p
