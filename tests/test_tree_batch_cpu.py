"""CPU tier of the persistent tree batches and the QV-tree rollouts: NULL
handles and arguments are refused before any device is touched."""
import ctypes

import numpy as np

from path_planning_2d_b200 import _lib


def test_null_handles_are_refused_without_a_device():
    lib = _lib.load()
    INV = _lib.PP2D_ERR_INVALID
    b = np.zeros(4, np.float32)
    idx = np.zeros(1, np.uint32)
    u8 = np.zeros(1, np.uint8)
    out = ctypes.c_void_p()
    assert lib.pp2d_tree_batch_create(None, b.ctypes.data, 1, ctypes.byref(out)) == INV
    assert out.value is None
    assert lib.pp2d_tree_batch_update(None, idx.ctypes.data, 1, u8.ctypes.data,
                                      u8.ctypes.data) == INV
    assert lib.pp2d_tree_batch_plan(None, idx.ctypes.data, 1, 50, 15, u8.ctypes.data, None,
                                    None) == INV
    assert lib.pp2d_tree_batch_dump(None, 0, None, 0) < 0
    assert b"NULL" in lib.pp2d_last_error()
    lib.pp2d_tree_batch_destroy(None)
    starts = np.zeros(2, np.uint32)
    for sim, planner in ((None, None), (ctypes.c_void_p(1), None)):
        assert lib.pp2d_sim_rollout_pomdp(sim, planner, 1, starts.ctypes.data, None, 10, 50, 15,
                                          0, 0, None) == INV
