"""ctypes binding of libpp2d.so (the C ABI in include/pp2d.h).

Loading fails loudly: there is no Python or CPU fallback for any entry point.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PP2D_LIB: alternate build of the same ABI (tuning experiments only).
LIB_PATH = os.environ.get("PP2D_LIB") or os.path.join(_HERE, "libpp2d.so")

PP2D_OK = 0
PP2D_ERR_INVALID = -1
PP2D_ERR_GOAL_OCCUPIED = -2
PP2D_ERR_CUDA = -3
PP2D_ERR_STATE = -4
IPC_DESC_BYTES = 256

_vp = ctypes.c_void_p
_u32 = ctypes.c_uint32
_i = ctypes.c_int


class Halo(ctypes.Structure):
    _fields_ = [("send_top", _vp), ("send_bottom", _vp), ("recv_top", _vp),
                ("recv_bottom", _vp), ("bytes", ctypes.c_size_t)]


class Rollout(ctypes.Structure):
    """pp2d_rollout: output arrays of pp2d_sim_rollout_*, each may be NULL."""
    _fields_ = [("steps", _vp), ("reached", _vp), ("collisions", _vp), ("final_cell", _vp),
                ("final_belief", _vp), ("cells", _vp), ("actions", _vp),
                ("measurements", _vp)]


# name -> (restype, argtypes); every symbol declared in include/pp2d.h.
SIGNATURES = {
    "pp2d_last_error": (ctypes.c_char_p, []),
    "pp2d_abi_version": (_i, []),
    "pp2d_kernel_launches": (ctypes.c_uint64, []),
    "pp2d_mdp_create": (_i, [_u32, _u32, _vp, _u32, _u32, ctypes.c_float,
                             ctypes.POINTER(_vp)]),
    "pp2d_mdp_create_shard": (_i, [_u32, _u32, _vp, _u32, _u32, ctypes.c_float,
                                   _u32, _u32, ctypes.POINTER(_vp)]),
    "pp2d_mdp_create_multi": (_i, [_u32, _u32, _vp, _u32, _u32, ctypes.c_float, _u32, _vp,
                                   ctypes.POINTER(_vp)]),
    "pp2d_mdp_device_count": (_i, [_vp, ctypes.POINTER(_i)]),
    "pp2d_mdp_reset": (_i, [_vp, _vp, _u32, _u32]),
    "pp2d_mdp_stage_map": (_i, [_vp, _vp]),
    "pp2d_mdp_update_map": (_i, [_vp, _vp, _u32, _u32]),
    "pp2d_mdp_destroy": (None, [_vp]),
    "pp2d_mdp_set_stream": (_i, [_vp, _vp]),
    "pp2d_mdp_set_async": (_i, [_vp, _i]),
    "pp2d_mdp_sweeps": (_i, [_vp, _u32]),
    "pp2d_mdp_sweeps_ex": (_i, [_vp, _u32, _i]),
    "pp2d_mdp_residual": (_i, [_vp, ctypes.POINTER(ctypes.c_float)]),
    "pp2d_mdp_residual_device": (_i, [_vp, ctypes.POINTER(_vp)]),
    "pp2d_mdp_solve": (_i, [_vp, ctypes.POINTER(_u32), _vp, _u32]),
    "pp2d_mdp_policy_iteration": (_i, [_vp, _vp, _vp, _vp, _u32, _u32]),
    "pp2d_mdp_download": (_i, [_vp, _vp, _vp]),
    "pp2d_mdp_download_begin": (_i, [_vp, _vp, _vp]),
    "pp2d_mdp_download_wait": (_i, [_vp]),
    "pp2d_mdp_plan": (_i, [_vp, _vp, _vp]),
    "pp2d_mdp_plan_batch": (_i, [_vp, _vp, _u32, _vp]),
    "pp2d_mdp_waypoints": (_i, [_vp, _u32, _u32, _vp, _u32,
                                ctypes.POINTER(_u32)]),
    "pp2d_mdp_sweep_count": (_u32, [_vp]),
    "pp2d_mdp_work_counters": (_i, [_vp, _vp]),
    "pp2d_mdp_halo": (_i, [_vp, ctypes.POINTER(Halo)]),
    "pp2d_mdp_ipc_export": (_i, [_vp, _vp]),
    "pp2d_mdp_ipc_connect": (_i, [_vp, _vp, _vp]),
    "pp2d_mdp_p2p_status": (_i, [_vp, ctypes.POINTER(_i)]),
    "pp2d_mdp_batch_create": (_i, [_u32, _u32, _u32, _vp, ctypes.c_size_t, _vp,
                                   ctypes.c_float, ctypes.POINTER(_vp)]),
    "pp2d_mdp_batch_reset": (_i, [_vp, _vp, ctypes.c_size_t, _vp]),
    "pp2d_mdp_batch_destroy": (None, [_vp]),
    "pp2d_mdp_batch_set_stream": (_i, [_vp, _vp]),
    "pp2d_mdp_batch_sweeps": (_i, [_vp, _u32]),
    "pp2d_mdp_batch_residual": (_i, [_vp, _vp]),
    "pp2d_mdp_batch_solve": (_i, [_vp, _vp, _vp, _u32]),
    "pp2d_mdp_batch_update": (_i, [_vp, _vp, _u32, _vp, ctypes.c_size_t, _vp]),
    "pp2d_mdp_batch_download": (_i, [_vp, _u32, _u32, _vp, _vp]),
    "pp2d_mdp_batch_plan": (_i, [_vp, _vp, _vp, _u32, _vp]),
    "pp2d_mdp_batch_waypoints": (_i, [_vp, _u32, _u32, _u32, _vp, _u32,
                                      ctypes.POINTER(_u32)]),
    "pp2d_mdp_batch_sweep_counts": (_i, [_vp, _vp]),
    "pp2d_mdp_batch_work_counters": (_i, [_vp, _vp]),
    "pp2d_pomdp_create": (_i, [_u32, _u32, _vp, _u32, _u32, ctypes.c_float,
                               ctypes.POINTER(_vp)]),
    "pp2d_pomdp_destroy": (None, [_vp]),
    "pp2d_pomdp_model_tables": (_i, [_vp, _vp, _vp, _vp]),
    "pp2d_pomdp_set_model_tables": (_i, [_vp, _vp, _vp, _vp]),
    "pp2d_pomdp_sampling_uniforms": (_i, [_vp, _vp]),
    "pp2d_pomdp_set_alphas": (_i, [_vp, _vp, _vp, _vp, _vp, _u32]),
    "pp2d_pomdp_solve_fib": (_i, [_vp, _vp, _vp, ctypes.POINTER(_u32), _u32]),
    "pp2d_pomdp_reserve": (_i, [_vp, _u32]),
    "pp2d_pomdp_live_cells": (_i, [_vp, _vp, ctypes.POINTER(_u32)]),
    "pp2d_pomdp_work_counters": (_i, [_vp, _vp]),
    "pp2d_pomdp_bayes_update": (_i, [_vp, _vp, _u32, _vp, _vp, _i, _vp, _vp]),
    "pp2d_pomdp_evaluate": (_i, [_vp, _vp, _u32, _vp, _vp, _vp, _vp]),
    "pp2d_pomdp_plan_batch": (_i, [_vp, _vp, _u32, _u32, _u32, _vp, _vp, _vp]),
    "pp2d_pomdp_generate_belief_set": (_i, [_vp, _vp, _u32, _u32, _vp]),
    "pp2d_pomdp_backup_alphas": (_i, [_vp, _vp, _u32, _u32, _vp, _vp]),
    "pp2d_pomdp_solve_pbvi": (_i, [_vp, _vp, _u32, _u32, _u32, _vp, _vp, _vp]),
    "pp2d_set_host_threads": (None, [_i]),
    "pp2d_sim_create": (_i, [_u32, _u32, _vp, ctypes.POINTER(_vp)]),
    "pp2d_sim_destroy": (None, [_vp]),
    "pp2d_sim_update_belief_action": (_i, [_vp, _vp, _u32, _vp]),
    "pp2d_sim_update_belief_measurement": (_i, [_vp, _vp, _u32, _vp]),
    "pp2d_sim_step": (_i, [_vp, _vp, _u32, _vp, _vp]),
    "pp2d_sim_rollout_mdp": (_i, [_vp, _vp, _u32, _vp, _vp, _u32, ctypes.c_uint64,
                                  ctypes.c_uint64, ctypes.POINTER(Rollout)]),
    "pp2d_sim_rollout_mdp_batch": (_i, [_vp, _vp, _vp, _u32, _vp, _vp, _u32, ctypes.c_uint64,
                                        ctypes.c_uint64, ctypes.POINTER(Rollout)]),
    "pp2d_tree_create": (_i, [_vp, _vp, ctypes.POINTER(_vp)]),
    "pp2d_tree_destroy": (None, [_vp]),
    "pp2d_tree_expand": (_i, [_vp]),
    "pp2d_tree_depth": (_u32, [_vp]),
    "pp2d_tree_best_action": (_i, [_vp, _vp, _vp]),
    "pp2d_tree_update": (_i, [_vp, ctypes.c_uint8, ctypes.c_uint8]),
    "pp2d_tree_root_bounds": (_i, [_vp, _vp, _vp]),
    "pp2d_tree_plan": (_i, [_vp, _u32, _u32, _vp, _vp]),
    "pp2d_tree_dump": (ctypes.c_int64, [_vp, _vp, ctypes.c_uint64]),
    "pp2d_tree_batch_create": (_i, [_vp, _vp, _u32, ctypes.POINTER(_vp)]),
    "pp2d_tree_batch_destroy": (None, [_vp]),
    "pp2d_tree_batch_update": (_i, [_vp, _vp, _u32, _vp, _vp]),
    "pp2d_tree_batch_plan": (_i, [_vp, _vp, _u32, _u32, _u32, _vp, _vp, _vp]),
    "pp2d_tree_batch_dump": (ctypes.c_int64, [_vp, _u32, _vp, ctypes.c_uint64]),
    "pp2d_sim_rollout_pomdp": (_i, [_vp, _vp, _u32, _vp, _vp, _u32, _u32, _u32, ctypes.c_uint64,
                                    ctypes.c_uint64, ctypes.POINTER(Rollout)]),
    "pp2d_pomdp_set_goals": (_i, [_vp, _vp, _u32, _vp]),
    "pp2d_pomdp_goals": (_i, [_vp, ctypes.POINTER(_u32), _vp]),
    "pp2d_pomdp_goal_reward": (_i, [_vp, _u32, _vp]),
    "pp2d_pomdp_set_goal_alphas": (_i, [_vp, _u32, _vp, _vp, _vp, _vp, _u32]),
    "pp2d_pomdp_padding_counters": (_i, [_vp, _vp]),
    "pp2d_tree_batch_create_goals": (_i, [_vp, _vp, _vp, _u32, ctypes.POINTER(_vp)]),
    "pp2d_sim_rollout_pomdp_goals": (_i, [_vp, _vp, _vp, _u32, _vp, _vp, _u32, _u32, _u32,
                                          ctypes.c_uint64, ctypes.c_uint64,
                                          ctypes.POINTER(Rollout)]),
}

_lib = None


class Pp2dError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"pp2d error {code}: {message}")
        self.code = code


def load():
    """Return the loaded library; raise if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g;"
            " g.build()'` (nvcc, sm_100a).  There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if a symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != PP2D_OK:
        raise Pp2dError(rc, load().pp2d_last_error().decode())
