"""ctypes access to the TEST-ONLY PBVI oracle (tests/pbvi_oracle.c, compiled on
first use into a temporary directory): the offline solver of csrc/pbvi.cu in
its own defined arithmetic (DESIGN.md section 7a), on the model tables of
oracle/pomdp_oracle.c."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "pbvi_oracle.c"),
           os.path.join(ROOT, "oracle", "pomdp_oracle.c")]
_lib = None
_vp, _u32, _i32, _i64, _f = (ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int32, ctypes.c_int64,
                             ctypes.c_float)


def _load():
    global _lib
    if _lib is not None:
        return _lib
    digest = hashlib.sha1(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), f"pp2d_pbvi_oracle_{os.getuid()}_{digest}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}"
        subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared",
                        "-o", tmp, SOURCES[0], "-lm"], check=True)
        os.replace(tmp, so)
    L = ctypes.CDLL(so)
    L.oracle_pomdp_generate_model.argtypes = [_u32, _u32, _i32, _i32, _vp, _vp, _vp, _vp]
    L.pbvi_oracle_reference_iterations.argtypes = [_f]
    L.pbvi_oracle_reference_iterations.restype = _u32
    L.pbvi_oracle_contract.argtypes = [_i32, _i32, _i64, _vp, _vp, _vp]
    L.pbvi_oracle_backup.argtypes = [_i32, _i32, _f, _vp, _vp, _vp, _i32, _vp, _u32, _vp, _vp,
                                     _vp]
    L.pbvi_oracle_backup.restype = _u32
    L.pbvi_oracle_expand.argtypes = [_i32, _i32, _vp, _vp, _vp, _u32, _u32, _vp]
    _lib = L
    return L


def reference_iterations(gamma):
    """The reference's backup count for gamma (float arithmetic as written)."""
    return _load().pbvi_oracle_reference_iterations(float(np.float32(gamma)))


def contract(G, B):
    """R[o][b][i] = one ascending FMA chain from +0 over all cells of
    G[o][i][s] * B[b][s]; G [n_o][n][HW] (or [n][HW]), B [n][HW]."""
    G = np.ascontiguousarray(G, np.float32)
    B = np.ascontiguousarray(B, np.float32)
    G3 = G.reshape(-1, *B.shape)
    R = np.empty((G3.shape[0], B.shape[0], B.shape[0]), np.float32)
    _load().pbvi_oracle_contract(G3.shape[0], B.shape[0], B.shape[1], G3.ctypes.data,
                                 B.ctypes.data, R.ctypes.data)
    return R.reshape(G.shape[:-2] + (B.shape[0], B.shape[0]))


class Pbvi:
    """Model tables of one map (oracle/pomdp_oracle.c) and the PBVI solver on them."""

    def __init__(self, grid, goal, gamma):
        self.grid = np.ascontiguousarray(grid, np.uint8)
        self.h, self.w = self.grid.shape
        self.hw = self.h * self.w
        self.gamma = np.float32(gamma)
        self.tp = np.zeros(self.hw * 81, np.float32)
        self.mp = np.zeros(self.hw * 16, np.float32)
        self.sr = np.zeros(self.hw * 9, np.float32)
        _load().oracle_pomdp_generate_model(self.h, self.w, int(goal[0]), int(goal[1]),
                                            self.grid.ctypes.data, self.tp.ctypes.data,
                                            self.mp.ctypes.data, self.sr.ctypes.data)

    def backup(self, belief_set, iterations=0):
        """backupAlphaVectors from zero vectors -> (alphas [n][HW], actions [n],
        argmax [9][16][n] of the last iteration, iterations run)."""
        B = np.ascontiguousarray(belief_set, np.float32)
        n = B.shape[0]
        al = np.empty((n, self.hw), np.float32)
        ac = np.empty(n, np.uint8)
        am = np.zeros((9, 16, n), np.int32)
        it = _load().pbvi_oracle_backup(self.h, self.w, float(self.gamma), self.tp.ctypes.data,
                                        self.mp.ctypes.data, self.sr.ctypes.data, n,
                                        B.ctypes.data, iterations, al.ctypes.data,
                                        ac.ctypes.data, am.ctypes.data)
        return al, ac, am, it

    def expand(self, b0, max_size, rand_seed=1):
        """generateBeliefSet -> [max_size][HW]."""
        b0 = np.ascontiguousarray(b0, np.float32).reshape(-1)
        out = np.empty((max_size, self.hw), np.float32)
        _load().pbvi_oracle_expand(self.h, self.w, self.tp.ctypes.data, self.mp.ctypes.data,
                                   b0.ctypes.data, max_size, rand_seed, out.ctypes.data)
        return out
