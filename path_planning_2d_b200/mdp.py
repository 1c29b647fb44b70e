"""Host-side mirror of the reference's MdpPathPlanning2d over the C ABI.

Reference: /root/reference/path_planning_2d/src/mdp/path_planning_2d.cu
(class MdpPathPlanning2d).  Method names follow the reference
(initialize / valueIteration / beliefCallback); ROS parameter loading and
publishing are outside the hot path and are replaced by plain arguments.
All numerical work happens in libpp2d.so on the GPU.
"""
import ctypes

import numpy as np

from . import _lib


def load_map_png(path):
    """loadMapFromFile (path_planning_2d.cu:191-205): grayscale read, then
    threshold(250, 1, THRESH_BINARY_INV): gray > 250 -> 0 (free), else 1."""
    import cv2
    img = cv2.imread(path, cv2.IMREAD_GRAYSCALE)
    if img is None:
        raise FileNotFoundError(path)
    _, grid = cv2.threshold(img, 250.0, 1.0, cv2.THRESH_BINARY_INV)
    return np.ascontiguousarray(grid, dtype=np.uint8)


class MdpPathPlanning2d:
    """Value-iteration planner on one GPU (or one row shard of the grid)."""

    def __init__(self, grid_map, goal, discount_factor, rows=None, devices=None):
        grid_map = np.ascontiguousarray(grid_map, dtype=np.uint8)
        if grid_map.ndim != 2:
            raise ValueError("grid_map must be 2-D (height, width)")
        self.map_height, self.map_width = grid_map.shape
        self.goal = (int(goal[0]), int(goal[1]))
        self.discount_factor = np.float32(discount_factor)
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        self._map = grid_map
        if devices is not None:
            # one process, several GPUs: devices = number of GPUs (devices
            # 0..n-1) or an explicit list of CUDA device ordinals, one per shard
            if rows is not None:
                raise ValueError("rows= and devices= are exclusive")
            self.row_begin, self.row_end = 0, self.map_height
            if isinstance(devices, int):
                n, arr = devices, None
            else:
                arr = (ctypes.c_int * len(devices))(*[int(d) for d in devices])
                n = len(devices)
            rc = self._lib.pp2d_mdp_create_multi(
                self.map_height, self.map_width, grid_map.ctypes.data,
                self.goal[0], self.goal[1], float(self.discount_factor), n, arr,
                ctypes.byref(self._h))
        elif rows is None:
            self.row_begin, self.row_end = 0, self.map_height
            rc = self._lib.pp2d_mdp_create(
                self.map_height, self.map_width, grid_map.ctypes.data,
                self.goal[0], self.goal[1], float(self.discount_factor),
                ctypes.byref(self._h))
        else:
            self.row_begin, self.row_end = int(rows[0]), int(rows[1])
            rc = self._lib.pp2d_mdp_create_shard(
                self.map_height, self.map_width, grid_map.ctypes.data,
                self.goal[0], self.goal[1], float(self.discount_factor),
                self.row_begin, self.row_end, ctypes.byref(self._h))
        _lib.check(rc)
        self.rows = self.row_end - self.row_begin
        self.optimal_cost = None
        self.optimal_action = None

    # -- lifetime ---------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.pp2d_mdp_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def reset(self, grid_map=None, goal=None):
        """New map (same shape) and/or goal on the same device buffers."""
        if grid_map is not None:
            grid_map = np.ascontiguousarray(grid_map, dtype=np.uint8)
            if grid_map.shape != (self.map_height, self.map_width):
                raise ValueError("reset() needs a map of the same shape")
            self._map = grid_map
        if goal is not None:
            self.goal = (int(goal[0]), int(goal[1]))
        _lib.check(self._lib.pp2d_mdp_reset(self._h, self._map.ctypes.data,
                                            self.goal[0], self.goal[1]))

    def update_map(self, grid_map=None, goal=None):
        """New map (same shape) and/or goal, keeping the current solution as
        the start of the next sweeps (pp2d_mdp_update_map): occupied cells of
        the new map take the trapped cost of the current sweep count, the new
        goal 0, every other cell keeps its J; the sweep count carries on and
        the next residual measures the change since this call.  Pass an array
        given to stage_map() to use the staged rows."""
        new_map, new_goal = self._map, self.goal
        if grid_map is not None:
            new_map = grid_map
            if not (isinstance(grid_map, np.ndarray) and grid_map.dtype == np.uint8
                    and grid_map.flags.c_contiguous):
                new_map = np.ascontiguousarray(grid_map, dtype=np.uint8)
            if new_map.shape != (self.map_height, self.map_width):
                raise ValueError("update_map() needs a map of the same shape")
        if goal is not None:
            new_goal = (int(goal[0]), int(goal[1]))
        _lib.check(self._lib.pp2d_mdp_update_map(self._h, new_map.ctypes.data,
                                                 new_goal[0], new_goal[1]))
        self._map, self.goal = new_map, new_goal

    def stage_map(self, grid_map):
        """Start uploading the map of the next reset() while the current solve
        runs (pp2d_mdp_stage_map); pass the SAME array to reset() afterwards.
        The array must be C-contiguous uint8 (page-locked for a real overlap)
        and stay unchanged until that reset()."""
        if (not isinstance(grid_map, np.ndarray) or grid_map.dtype != np.uint8
                or not grid_map.flags.c_contiguous
                or grid_map.shape != (self.map_height, self.map_width)):
            raise ValueError("stage_map() needs a C-contiguous uint8 map of the handle's shape")
        self._staged = grid_map          # keep it alive
        _lib.check(self._lib.pp2d_mdp_stage_map(self._h, grid_map.ctypes.data))

    # -- solver -----------------------------------------------------------
    def set_stream(self, cuda_stream_ptr, asynchronous=False):
        _lib.check(self._lib.pp2d_mdp_set_stream(self._h, cuda_stream_ptr))
        _lib.check(self._lib.pp2d_mdp_set_async(self._h, int(asynchronous)))

    def sweeps(self, n, want_action=True):
        """n launches of cudaOneStepValueIteration."""
        _lib.check(self._lib.pp2d_mdp_sweeps_ex(self._h, n, int(want_action)))

    def residual(self):
        r = ctypes.c_float()
        _lib.check(self._lib.pp2d_mdp_residual(self._h, ctypes.byref(r)))
        return r.value

    def residual_device(self):
        p = ctypes.c_void_p()
        _lib.check(self._lib.pp2d_mdp_residual_device(self._h, ctypes.byref(p)))
        return p.value

    def valueIteration(self, max_batches=64):
        """The reference's stopping rule; returns (sweeps, [inf-norm per batch])."""
        n = ctypes.c_uint32()
        res = np.zeros(max_batches, dtype=np.float64)
        _lib.check(self._lib.pp2d_mdp_solve(self._h, ctypes.byref(n),
                                            res.ctypes.data, max_batches))
        return n.value, res[:min(max_batches, n.value // 100)].copy()

    def policyIteration(self, max_rounds=0):
        """src/mdp/path_planning_2d.cu:271-357 on a fresh / reset handle; returns
        (evaluation sweeps, [inf-norm per round], [changed actions per round])."""
        n = ctypes.c_uint32()
        cap = max_rounds if max_rounds else 4096
        res = np.zeros(cap, dtype=np.float64)
        chg = np.zeros(cap, dtype=np.uint32)
        _lib.check(self._lib.pp2d_mdp_policy_iteration(
            self._h, ctypes.byref(n), res.ctypes.data, chg.ctypes.data, cap, max_rounds))
        rounds = min(n.value // 50, cap)
        return n.value, res[:rounds].copy(), chg[:rounds].copy()

    def download(self, cost=True, action=True):
        n = self.rows * self.map_width
        c = np.empty(n, dtype=np.float32) if cost else None
        a = np.empty(n, dtype=np.uint8) if action else None
        _lib.check(self._lib.pp2d_mdp_download(
            self._h, c.ctypes.data if cost else None,
            a.ctypes.data if action else None))
        if cost:
            self.optimal_cost = c.reshape(self.rows, self.map_width)
        if action:
            self.optimal_action = a.reshape(self.rows, self.map_width)
        return self.optimal_cost, self.optimal_action

    def download_begin(self, cost_ptr, action_ptr):
        """Asynchronous download into caller-owned (page-locked) host memory given
        by raw addresses (either may be None); pair with download_wait()."""
        _lib.check(self._lib.pp2d_mdp_download_begin(self._h, cost_ptr, action_ptr))

    def download_wait(self):
        _lib.check(self._lib.pp2d_mdp_download_wait(self._h))

    def initialize(self):
        """initialize() minus ROS: solve and download (path_planning_2d.cu:72-140)."""
        sweeps, residuals = self.valueIteration()
        self.download()
        return sweeps, residuals

    @property
    def device_count(self):
        return self._lib.pp2d_mdp_device_count(self._h, None)

    @property
    def peer_to_peer(self):
        p = ctypes.c_int()
        self._lib.pp2d_mdp_device_count(self._h, ctypes.byref(p))
        return bool(p.value)

    @property
    def sweep_count(self):
        return self._lib.pp2d_mdp_sweep_count(self._h)

    def work_counters(self):
        """(units run, units launched) of the fused two-sweep launches so far
        (pp2d_mdp_work_counters)."""
        out = np.zeros(2, dtype=np.uint64)
        _lib.check(self._lib.pp2d_mdp_work_counters(self._h, out.ctypes.data))
        return int(out[0]), int(out[1])

    # -- online -----------------------------------------------------------
    def beliefCallback(self, belief):
        """Action at the belief mode (path_planning_2d.cu:168-189)."""
        b = np.ascontiguousarray(belief, dtype=np.float32).reshape(-1)
        if b.size != self.map_height * self.map_width:
            raise ValueError("belief size != height*width")
        out = ctypes.c_uint8()
        _lib.check(self._lib.pp2d_mdp_plan(self._h, b.ctypes.data,
                                           ctypes.addressof(out)))
        return out.value

    def plan_batch(self, beliefs):
        b = np.ascontiguousarray(beliefs, dtype=np.float32)
        n = b.shape[0]
        out = np.empty(n, dtype=np.uint8)
        _lib.check(self._lib.pp2d_mdp_plan_batch(self._h, b.ctypes.data, n,
                                                 out.ctypes.data))
        return out

    def waypoints(self, start, max_len=None):
        max_len = max_len or self.map_height * self.map_width
        cells = np.empty(max_len, dtype=np.uint32)
        n = ctypes.c_uint32()
        _lib.check(self._lib.pp2d_mdp_waypoints(
            self._h, int(start[0]), int(start[1]), cells.ctypes.data, max_len,
            ctypes.byref(n)))
        return cells[:n.value].copy()

    def ipc_export(self):
        buf = ctypes.create_string_buffer(_lib.IPC_DESC_BYTES)
        _lib.check(self._lib.pp2d_mdp_ipc_export(self._h, buf))
        return buf.raw

    def ipc_connect(self, up_desc, down_desc):
        _lib.check(self._lib.pp2d_mdp_ipc_connect(self._h, up_desc, down_desc))

    def p2p_timed_out(self):
        e = ctypes.c_int()
        _lib.check(self._lib.pp2d_mdp_p2p_status(self._h, ctypes.byref(e)))
        return bool(e.value)

    def halo(self):
        h = _lib.Halo()
        _lib.check(self._lib.pp2d_mdp_halo(self._h, ctypes.byref(h)))
        return h


class MdpBatchPathPlanning2d:
    """Many value-iteration instances of one size solved together on one GPU
    (pp2d_mdp_batch_*): one goal per robot on a shared map, or one map per
    instance.  Every instance computes bit for bit what MdpPathPlanning2d
    computes on its map and goal.

    grid_maps: (H, W) shared by all instances, or (K, H, W); goals: K (x, y)
    pairs."""

    def __init__(self, grid_maps, goals, discount_factor):
        self.discount_factor = np.float32(discount_factor)
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        maps, stride, goals = self._arguments(grid_maps, goals)
        self.count = goals.shape[0]
        self.map_height, self.map_width = maps.shape[-2:]
        _lib.check(self._lib.pp2d_mdp_batch_create(
            self.map_height, self.map_width, self.count, maps.ctypes.data, stride,
            goals.ctypes.data, float(self.discount_factor), ctypes.byref(self._h)))

    def _arguments(self, grid_maps, goals, shape=None):
        maps = np.ascontiguousarray(grid_maps, dtype=np.uint8)
        goals = np.ascontiguousarray(goals, dtype=np.uint32).reshape(-1, 2)
        if maps.ndim not in (2, 3):
            raise ValueError("grid_maps must be (H, W) or (K, H, W)")
        if maps.ndim == 3 and maps.shape[0] != goals.shape[0]:
            raise ValueError("one map per goal, or one shared (H, W) map")
        if shape is not None and (maps.shape[-2:] != shape or goals.shape[0] != self.count):
            raise ValueError("reset() needs maps of the same shape and the same count")
        stride = 0 if maps.ndim == 2 else maps.shape[1] * maps.shape[2]
        return maps, stride, goals

    # -- lifetime ---------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.pp2d_mdp_batch_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def reset(self, grid_maps, goals):
        """New maps and goals (same shape and count) on the same buffers."""
        maps, stride, goals = self._arguments(grid_maps, goals,
                                              (self.map_height, self.map_width))
        _lib.check(self._lib.pp2d_mdp_batch_reset(self._h, maps.ctypes.data, stride,
                                                  goals.ctypes.data))

    # -- solver -----------------------------------------------------------
    def set_stream(self, cuda_stream_ptr):
        _lib.check(self._lib.pp2d_mdp_batch_set_stream(self._h, cuda_stream_ptr))

    def sweeps(self, n):
        """n sweeps of every instance."""
        _lib.check(self._lib.pp2d_mdp_batch_sweeps(self._h, n))

    def residual(self):
        """Per-instance inf-norm of the change since the previous call."""
        out = np.zeros(self.count, dtype=np.float32)
        _lib.check(self._lib.pp2d_mdp_batch_residual(self._h, out.ctypes.data))
        return out

    def valueIteration(self, max_batches=64):
        """The reference's stopping rule per instance; returns (sweeps[K],
        [inf-norm per batch] for each instance)."""
        n = np.zeros(self.count, dtype=np.uint32)
        res = np.zeros((self.count, max_batches), dtype=np.float64)
        _lib.check(self._lib.pp2d_mdp_batch_solve(self._h, n.ctypes.data, res.ctypes.data,
                                                  max_batches))
        return n, [res[k, :min(max_batches, int(n[k]) // 100)].copy()
                   for k in range(self.count)]

    def update_map(self, instances, grid_maps, goals):
        """New maps and goals for the listed instances, each continuing from
        its current solution as MdpPathPlanning2d.update_map does; an instance
        that valueIteration() stopped becomes active again.  grid_maps: (H, W)
        shared by the listed instances, or (n, H, W); goals: n (x, y) pairs."""
        idx = np.ascontiguousarray(instances, dtype=np.uint32).reshape(-1)
        maps = np.ascontiguousarray(grid_maps, dtype=np.uint8)
        goals = np.ascontiguousarray(goals, dtype=np.uint32).reshape(-1, 2)
        if maps.ndim not in (2, 3) or maps.shape[-2:] != (self.map_height, self.map_width):
            raise ValueError("grid_maps must be (H, W) or (n, H, W) of the batch's map size")
        if goals.shape[0] != idx.size or (maps.ndim == 3 and maps.shape[0] != idx.size):
            raise ValueError("one goal per listed instance, and one map each or one shared map")
        stride = 0 if maps.ndim == 2 else self.map_height * self.map_width
        _lib.check(self._lib.pp2d_mdp_batch_update(self._h, idx.ctypes.data, idx.size,
                                                   maps.ctypes.data, stride, goals.ctypes.data))

    def sweep_counts(self):
        out = np.zeros(self.count, dtype=np.uint32)
        _lib.check(self._lib.pp2d_mdp_batch_sweep_counts(self._h, out.ctypes.data))
        return out

    def work_counters(self):
        """(units run, units launched) of the fused two-sweep launches so far."""
        out = np.zeros(2, dtype=np.uint64)
        _lib.check(self._lib.pp2d_mdp_batch_work_counters(self._h, out.ctypes.data))
        return int(out[0]), int(out[1])

    def download(self, instances=None):
        """(cost[K, H, W], action[K, H, W]) of the instances range(first, stop)
        given as a range or slice (default: all)."""
        if instances is None:
            first, stop = 0, self.count
        elif isinstance(instances, (range, slice)):
            first, stop, step = instances.start or 0, instances.stop, instances.step or 1
            if stop is None:
                stop = self.count
            if step != 1:
                raise ValueError("download() takes a contiguous range of instances")
        else:
            first = int(instances)
            stop = first + 1
        n = max(stop - first, 0)
        c = np.empty((n, self.map_height, self.map_width), dtype=np.float32)
        a = np.empty((n, self.map_height, self.map_width), dtype=np.uint8)
        _lib.check(self._lib.pp2d_mdp_batch_download(self._h, first, n, c.ctypes.data,
                                                     a.ctypes.data))
        return c, a

    # -- online -----------------------------------------------------------
    def plan_batch(self, instances, beliefs):
        """Action at the mode of beliefs[i] on the action grid of instances[i]."""
        idx = np.ascontiguousarray(instances, dtype=np.uint32).reshape(-1)
        b = np.ascontiguousarray(beliefs, dtype=np.float32).reshape(
            idx.size, self.map_height * self.map_width) if idx.size else None
        if idx.size == 0:
            return np.empty(0, dtype=np.uint8)
        if b.shape[1] != self.map_height * self.map_width:
            raise ValueError("belief size != height*width")
        out = np.empty(idx.size, dtype=np.uint8)
        _lib.check(self._lib.pp2d_mdp_batch_plan(self._h, idx.ctypes.data, b.ctypes.data,
                                                 idx.size, out.ctypes.data))
        return out

    def waypoints(self, k, start, max_len=None):
        max_len = max_len or self.map_height * self.map_width
        cells = np.empty(max_len, dtype=np.uint32)
        n = ctypes.c_uint32()
        _lib.check(self._lib.pp2d_mdp_batch_waypoints(
            self._h, int(k), int(start[0]), int(start[1]), cells.ctypes.data, max_len,
            ctypes.byref(n)))
        return cells[:n.value].copy()
