"""ctypes access to the TEST-ONLY closed-loop rollout oracle (tests/rollout_oracle.c,
compiled on first use into a temporary directory) and a vectorised numpy
Philox4x32-10 with the rollouts' step uniforms (DESIGN.md section 7,
"Closed-loop rollouts")."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "rollout_oracle.c"),
           os.path.join(ROOT, "oracle", "sim_oracle.c"),
           os.path.join(ROOT, "path_planning_2d_b200", "csrc", "philox.h")]
_lib = None
_vp, _u32, _u64, _i32, _u8 = (ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int32,
                              ctypes.c_uint8)


def _load():
    global _lib
    if _lib is not None:
        return _lib
    digest = hashlib.sha1(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), f"pp2d_rollout_oracle_{os.getuid()}_{digest}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}"
        subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", tmp,
                        SOURCES[0], "-lm"], check=True)
        os.replace(tmp, so)
    L = ctypes.CDLL(so)
    L.oracle_philox.argtypes = [_vp, _u32, _u32]
    L.oracle_step_uniforms.argtypes = [_u64, _u64, _u32, _vp]
    L.oracle_motion_slot.argtypes = [_u8, ctypes.c_float]
    L.oracle_motion_slot.restype = _i32
    L.oracle_rollout_episode.argtypes = [_i32, _i32, _vp, _vp, _u32, _u32, _u32, _u32, _vp, _u32,
                                         _u64, _u64, _vp, _vp, _vp, _vp]
    _lib = L
    return L


def philox(counter, key):
    """Philox4x32-10 of one counter (4 words) and key (2 words), through the oracle."""
    c = np.array(counter, np.uint32)
    _load().oracle_philox(c.ctypes.data, int(key[0]), int(key[1]))
    return c


def step_uniforms(seed, episode, t):
    r = np.zeros(5, np.float32)
    _load().oracle_step_uniforms(seed, episode, t, r.ctypes.data)
    return r


def motion_slot(u, r):
    return _load().oracle_motion_slot(int(u), float(np.float32(r)))


def rollout(grid, act, goal, starts, max_steps, seed, first_episode=0, beliefs=None):
    """Episodes first_episode + i from starts[i] = (x, y); act: [n][H][W] or
    [H][W] action grids, goal: (x, y) or [n][2].  Returns a dict like
    DummySimulator.rollout(record=True)."""
    grid = np.ascontiguousarray(grid, np.uint8)
    h, w = grid.shape
    starts = np.asarray(starts, np.uint32).reshape(-1, 2)
    n = starts.shape[0]
    act = np.broadcast_to(np.asarray(act, np.uint8).reshape(-1, h * w), (n, h * w))
    goal = np.broadcast_to(np.asarray(goal, np.uint32).reshape(-1, 2), (n, 2))
    if beliefs is None:
        bel = np.zeros((n, h * w), np.float32)
        bel[np.arange(n), starts[:, 1] * w + starts[:, 0]] = 1.0
    else:
        bel = np.array(beliefs, np.float32, copy=True).reshape(n, h * w)
    stats = np.zeros((n, 4), np.uint32)
    cells = np.zeros((n, max_steps + 1), np.uint32)
    actions = np.zeros((n, max_steps), np.uint8)
    meas = np.zeros((n, max_steps), np.uint8)
    L = _load()
    for i in range(n):
        a = np.ascontiguousarray(act[i])
        b = np.ascontiguousarray(bel[i])
        L.oracle_rollout_episode(h, w, grid.ctypes.data, a.ctypes.data, int(goal[i, 0]),
                                 int(goal[i, 1]), int(starts[i, 0]), int(starts[i, 1]),
                                 b.ctypes.data, max_steps, seed, first_episode + i,
                                 stats[i].ctypes.data, cells[i].ctypes.data,
                                 actions[i].ctypes.data, meas[i].ctypes.data)
        bel[i] = b
    return {"steps": stats[:, 0].copy(), "reached": stats[:, 1].astype(np.uint8),
            "collisions": stats[:, 2].copy(), "final_cell": stats[:, 3].copy(),
            "final_belief": bel, "cells": cells, "actions": actions, "measurements": meas}


# ---- vectorised numpy Philox4x32-10 ---------------------------------------------------------
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
_LO = np.uint64(0xFFFFFFFF)
_SH = np.uint64(32)


def philox_np(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of arrays of counter words (broadcast) under one key."""
    c0, c1, c2, c3 = (np.asarray(v, np.uint32) for v in np.broadcast_arrays(c0, c1, c2, c3))
    k0, k1 = np.uint32(k0), np.uint32(k1)
    with np.errstate(over="ignore"):
        for r in range(10):
            if r:
                k0 = np.uint32(k0 + _W0)
                k1 = np.uint32(k1 + _W1)
            p0 = _M0 * c0.astype(np.uint64)
            p1 = _M1 * c2.astype(np.uint64)
            c0, c1, c2, c3 = (((p1 >> _SH).astype(np.uint32) ^ c1 ^ k0),
                              (p1 & _LO).astype(np.uint32),
                              ((p0 >> _SH).astype(np.uint32) ^ c3 ^ k1),
                              (p0 & _LO).astype(np.uint32))
    return c0, c1, c2, c3


def step_uniforms_np(seed, episodes, t):
    """[len(episodes)][5] float32 uniforms of step t: motion, then sensors up,
    left, right, down."""
    e = np.asarray(episodes, np.uint64)
    lo = (e & _LO).astype(np.uint32)
    hi = (e >> _SH).astype(np.uint32)
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    a = philox_np(np.uint32(t), lo, hi, np.uint32(0), k0, k1)
    b = philox_np(np.uint32(t), lo, hi, np.uint32(1), k0, k1)
    words = np.stack([a[0], a[1], a[2], a[3], b[0]], axis=1)
    return (words >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)


# naive probabilities (sim.cu:naive_prob) and their ascending float32 running sums
NAIVE = np.zeros((9, 9), np.float32)
for _u, _row in enumerate([(0, 1, 3), (1, 0, 2), (2, 1, 5), (3, 0, 6), None, (5, 2, 8),
                           (6, 3, 7), (7, 6, 8), (8, 5, 7)]):
    if _row is None:
        NAIVE[_u, 4] = 1.0
    else:
        NAIVE[_u, _row[0]] = 0.7
        NAIVE[_u, _row[1]] = NAIVE[_u, _row[2]] = NAIVE[_u, 4] = 0.1
CUM = np.zeros((9, 9), np.float32)
for _u in range(9):
    _acc = np.float32(0)
    for _i in range(9):
        _acc = np.float32(_acc + NAIVE[_u, _i])
        CUM[_u, _i] = _acc


def motion_slots_np(u, r):
    """Vectorised oracle_motion_slot."""
    u = np.asarray(u, np.intp)
    cum = CUM[u]
    hit = np.asarray(r, np.float32)[:, None] < cum
    last = np.array([max(i for i in range(9) if NAIVE[k, i] != 0) for k in range(9)])[u]
    return np.where(hit.any(axis=1), hit.argmax(axis=1), last)
