"""Host-side mirror of the reference's PomdpPathPlanning2d / SearchTree over
the C ABI (reference: /root/reference/path_planning_2d/src/pomdp/
path_planning_2d.cu, search_tree_cuda.cu, include/.../search_tree.h).

Names follow the reference (initialize-time model generation, beliefCallback,
SearchTree.expand/update/getOptimalAction/getDepth).  The alpha vectors are
inputs (set_alphas), exactly like the reference's read_data_from_file=true
path; all belief arithmetic runs in libpp2d.so on the GPU.
"""
import ctypes

import numpy as np

from . import _lib


class SearchTree:
    """search_tree.h:130-165 on the GPU belief pool of a PomdpPathPlanning2d."""

    def __init__(self, planner, belief):
        self._lib = planner._lib
        self._planner = planner
        b = np.ascontiguousarray(belief, dtype=np.float32).reshape(-1)
        if b.size != planner.map_height * planner.map_width:
            raise ValueError("belief size != height*width")
        self._t = ctypes.c_void_p()
        _lib.check(self._lib.pp2d_tree_create(planner._h, b.ctypes.data,
                                              ctypes.byref(self._t)))

    def close(self):
        if getattr(self, "_t", None) is not None and self._t.value:
            self._lib.pp2d_tree_destroy(self._t)
            self._t = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def expand(self):
        _lib.check(self._lib.pp2d_tree_expand(self._t))

    def update(self, action, observation):
        _lib.check(self._lib.pp2d_tree_update(self._t, action, observation))

    def getDepth(self):
        return self._lib.pp2d_tree_depth(self._t)

    def getOptimalAction(self):
        a, r = ctypes.c_uint8(), ctypes.c_float()
        _lib.check(self._lib.pp2d_tree_best_action(self._t, ctypes.addressof(a),
                                                   ctypes.addressof(r)))
        return a.value, r.value

    def rootBounds(self):
        u, l = ctypes.c_float(), ctypes.c_float()
        _lib.check(self._lib.pp2d_tree_root_bounds(self._t, ctypes.addressof(u),
                                                   ctypes.addressof(l)))
        return u.value, l.value

    def plan(self, max_depth, max_iter):
        a, r = ctypes.c_uint8(), ctypes.c_float()
        _lib.check(self._lib.pp2d_tree_plan(self._t, max_depth, max_iter,
                                            ctypes.addressof(a), ctypes.addressof(r)))
        return a.value, r.value

    def dump(self):
        """print() of search_tree_cuda.cu:628-633 as an array [nodes][9], see
        pp2d_tree_dump in include/pp2d.h."""
        n = self._lib.pp2d_tree_dump(self._t, None, 0)
        if n < 0:
            raise _lib.Pp2dError(_lib.PP2D_ERR_INVALID, "pp2d_tree_dump failed")
        out = np.zeros((n, 9), np.float32)
        self._lib.pp2d_tree_dump(self._t, out.ctypes.data, n)
        return out


def _goal_indices(goals, n, what):
    """Goal indices as uint32 [n]; negative or non-integer entries are refused
    here (the library checks the upper end)."""
    g = np.asarray(goals)
    if g.ndim != 1 or g.size != n:
        raise ValueError(f"one goal index per {what} ({n}), got shape {g.shape}")
    if g.size and (not np.issubdtype(g.dtype, np.integer) or g.min() < 0):
        raise ValueError("goal indices must be integers >= 0")
    return np.ascontiguousarray(g, dtype=np.uint32)


class SearchTreeBatch:
    """Many SearchTrees on the GPU belief pool of one PomdpPathPlanning2d that
    live across belief callbacks (one per robot of a fleet), updated and
    planned together (pp2d_tree_batch_* in include/pp2d.h).  Tree k behaves
    bit for bit like SearchTree(planner, beliefs[k]) fed the same calls.
    goals (optional, one per tree): tree k plans to goal goals[k] of the
    planner's goal set (set_goals), bit for bit like a SearchTree on a planner
    created with that goal."""

    def __init__(self, planner, beliefs, goals=None):
        self._lib = planner._lib
        self._planner = planner
        hw = planner.map_height * planner.map_width
        b = np.ascontiguousarray(beliefs, dtype=np.float32)
        if b.size % hw:
            raise ValueError("beliefs must be [n][height*width]")
        b = b.reshape(-1, hw)
        self.count = b.shape[0]
        self._b = ctypes.c_void_p()
        if goals is None:
            _lib.check(self._lib.pp2d_tree_batch_create(planner._h, b.ctypes.data, self.count,
                                                        ctypes.byref(self._b)))
            return
        g = _goal_indices(goals, self.count, "tree")
        _lib.check(self._lib.pp2d_tree_batch_create_goals(planner._h, b.ctypes.data, g.ctypes.data,
                                                          self.count, ctypes.byref(self._b)))

    def close(self):
        if getattr(self, "_b", None) is not None and self._b.value:
            self._lib.pp2d_tree_batch_destroy(self._b)
            self._b = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _trees(self, trees):
        if trees is None:
            return np.arange(self.count, dtype=np.uint32)
        return np.ascontiguousarray(trees, dtype=np.uint32).reshape(-1)

    def update(self, trees, actions, observations):
        """SearchTree.update(actions[i], observations[i]) on tree trees[i]
        (None: every tree); nothing changes if any entry is refused."""
        idx = self._trees(trees)
        n = idx.size
        a = np.ascontiguousarray(np.broadcast_to(actions, (n,)), dtype=np.uint8)
        z = np.ascontiguousarray(np.broadcast_to(observations, (n,)), dtype=np.uint8)
        _lib.check(self._lib.pp2d_tree_batch_update(self._b, idx.ctypes.data, n, a.ctypes.data,
                                                    z.ctypes.data))

    def plan(self, trees=None, max_depth=None, max_iter=None, with_stats=False):
        """SearchTree.plan on the listed trees (None: every tree), defaults
        from the planner (depth 50, 15 iterations).  Returns (actions, values)
        and with with_stats the [n][4] {V nodes, Q nodes, depth, expansions}."""
        idx = self._trees(trees)
        n = idx.size
        acts = np.zeros(n, np.uint8)
        vals = np.zeros(n, np.float32)
        stats = np.zeros((n, 4), np.uint32)
        _lib.check(self._lib.pp2d_tree_batch_plan(
            self._b, idx.ctypes.data, n,
            self._planner.max_search_tree_depth if max_depth is None else max_depth,
            self._planner.max_online_iteration if max_iter is None else max_iter,
            acts.ctypes.data, vals.ctypes.data, stats.ctypes.data))
        return (acts, vals, stats) if with_stats else (acts, vals)

    def dump(self, k):
        """SearchTree.dump() of tree k."""
        n = self._lib.pp2d_tree_batch_dump(self._b, k, None, 0)
        if n < 0:
            raise _lib.Pp2dError(_lib.PP2D_ERR_INVALID, self._lib.pp2d_last_error().decode())
        out = np.zeros((n, 9), np.float32)
        self._lib.pp2d_tree_batch_dump(self._b, k, out.ctypes.data, n)
        return out


class PomdpPathPlanning2d:
    def __init__(self, grid_map, goal, discount_factor, max_search_tree_depth=50,
                 max_online_iteration=15):
        grid_map = np.ascontiguousarray(grid_map, dtype=np.uint8)
        self.map_height, self.map_width = grid_map.shape
        self.goal = (int(goal[0]), int(goal[1]))
        self.discount_factor = np.float32(discount_factor)
        # launch/pomdp_path_planning_2d.launch: depth 50, 15 online iterations
        self.max_search_tree_depth = max_search_tree_depth
        self.max_online_iteration = max_online_iteration
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        _lib.check(self._lib.pp2d_pomdp_create(
            self.map_height, self.map_width, grid_map.ctypes.data, self.goal[0],
            self.goal[1], float(self.discount_factor), ctypes.byref(self._h)))
        self.search_tree = None
        # path_planning_2d.cu:99-107: uniform over the free cells
        s = np.float32(0)
        for v in (1.0 - grid_map.astype(np.float32)).reshape(-1):
            s = np.float32(s + v)
        self.initial_belief = ((1.0 - grid_map.astype(np.float32)) / s).astype(np.float32)

    def close(self):
        if self.search_tree is not None:
            self.search_tree.close()
            self.search_tree = None
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.pp2d_pomdp_destroy(self._h)
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

    # -- model / alphas -----------------------------------------------------
    def model_tables(self):
        n = self.map_height * self.map_width
        tp = np.empty(n * 81, np.float32)
        mp = np.empty(n * 16, np.float32)
        sr = np.empty(n * 9, np.float32)
        _lib.check(self._lib.pp2d_pomdp_model_tables(self._h, tp.ctypes.data,
                                                     mp.ctypes.data, sr.ctypes.data))
        return tp.reshape(n, 9, 9), mp.reshape(n, 16), sr.reshape(n, 9)

    def set_model_tables(self, trans_prob=None, meas_prob=None, stage_reward=None):
        """Upload half of loadModelDataFromFile (model_generation_cuda.cu:150-156)."""
        n = self.map_height * self.map_width
        arrs = []
        for a, k in ((trans_prob, 81), (meas_prob, 16), (stage_reward, 9)):
            if a is None:
                arrs.append(None)
                continue
            a = np.ascontiguousarray(a, dtype=np.float32).reshape(-1)
            if a.size != n * k:
                raise ValueError(f"table must have {n}*{k} entries")
            arrs.append(a)
        _lib.check(self._lib.pp2d_pomdp_set_model_tables(
            self._h, *[a.ctypes.data if a is not None else None for a in arrs]))

    def live_cells(self, mask=False):
        """Number of cells probability mass can enter (and the mask, if asked)."""
        n = ctypes.c_uint32()
        m = np.zeros(self.map_height * self.map_width, np.uint8) if mask else None
        _lib.check(self._lib.pp2d_pomdp_live_cells(
            self._h, m.ctypes.data if mask else None, ctypes.byref(n)))
        return (n.value, m.reshape(self.map_height, self.map_width)) if mask else n.value

    def work_counters(self):
        """(V nodes created, Bayes updates, belief x inner-row products of the
        bound evaluations) on this handle so far."""
        out = np.zeros(3, np.uint64)
        _lib.check(self._lib.pp2d_pomdp_work_counters(self._h, out.ctypes.data))
        return int(out[0]), int(out[1]), int(out[2])

    def sampling_uniforms(self):
        out = np.empty(100, np.float32)
        _lib.check(self._lib.pp2d_pomdp_sampling_uniforms(self._h, out.ctypes.data))
        return out

    def fastInformedBound(self, max_sweeps=0):
        """fast_informed_bound_cuda.cu:206-276 on the GPU; returns
        (alphas [HW][9], actions [9], sweeps)."""
        n = self.map_height * self.map_width
        al = np.empty((n, 9), np.float32)
        ac = np.empty(9, np.uint8)
        sw = ctypes.c_uint32()
        _lib.check(self._lib.pp2d_pomdp_solve_fib(self._h, al.ctypes.data, ac.ctypes.data,
                                                  ctypes.byref(sw), max_sweeps))
        return al, ac, sw.value

    def generateBeliefSet(self, initial_belief, max_size=500, rand_seed=1):
        """point_based_value_iteration_cuda.cu:165-293 on the GPU -> [max_size][HW]."""
        n = self.map_height * self.map_width
        b0 = np.ascontiguousarray(initial_belief, dtype=np.float32).reshape(-1)
        if b0.size != n:
            raise ValueError("belief size != height*width")
        out = np.empty((max_size, n), np.float32)
        _lib.check(self._lib.pp2d_pomdp_generate_belief_set(
            self._h, b0.ctypes.data, max_size, rand_seed, out.ctypes.data))
        return out

    def backupAlphaVectors(self, belief_set, iterations=0):
        """point_based_value_iteration_cuda.cu:344-641 -> (alphas [N][HW], actions [N])."""
        n = self.map_height * self.map_width
        bs = np.ascontiguousarray(belief_set, dtype=np.float32)
        if bs.ndim != 2 or bs.shape[1] != n:
            raise ValueError("belief_set must be [N][HW]")
        al = np.empty_like(bs)
        ac = np.empty(bs.shape[0], np.uint8)
        _lib.check(self._lib.pp2d_pomdp_backup_alphas(
            self._h, bs.ctypes.data, bs.shape[0], iterations, al.ctypes.data, ac.ctypes.data))
        return al, ac

    def pointBasedValueIteration(self, initial_belief, belief_set_size=500, rand_seed=1,
                                 iterations=0):
        """point_based_value_iteration_cuda.cu:643-676 -> (belief_set, alphas, actions)."""
        n = self.map_height * self.map_width
        b0 = np.ascontiguousarray(initial_belief, dtype=np.float32).reshape(-1)
        if b0.size != n:
            raise ValueError("belief size != height*width")
        bs = np.empty((belief_set_size, n), np.float32)
        al = np.empty((belief_set_size, n), np.float32)
        ac = np.empty(belief_set_size, np.uint8)
        _lib.check(self._lib.pp2d_pomdp_solve_pbvi(
            self._h, b0.ctypes.data, belief_set_size, rand_seed, iterations,
            bs.ctypes.data, al.ctypes.data, ac.ctypes.data))
        return bs, al, ac

    def set_alphas(self, fib_alphas, pbvi_alphas, fib_actions=None, pbvi_actions=None):
        fa = np.ascontiguousarray(fib_alphas, dtype=np.float32)
        pa = np.ascontiguousarray(pbvi_alphas, dtype=np.float32)
        n = self.map_height * self.map_width
        if fa.shape != (n, 9) or pa.ndim != 2 or pa.shape[1] != n:
            raise ValueError("fib_alphas must be [HW][9], pbvi_alphas [N][HW]")
        fac = np.ascontiguousarray(fib_actions, np.uint8) if fib_actions is not None else None
        pac = np.ascontiguousarray(pbvi_actions, np.uint8) if pbvi_actions is not None else None
        _lib.check(self._lib.pp2d_pomdp_set_alphas(
            self._h, fa.ctypes.data, fac.ctypes.data if fac is not None else None,
            pa.ctypes.data, pac.ctypes.data if pac is not None else None, pa.shape[0]))

    # -- goal sets (include/pp2d.h, DESIGN.md section 7e) -----------------------
    def set_goals(self, goals, stage_rewards=None):
        """Goals 1..n of this handle's goal set = goals [n][2] (x, y); goal 0
        stays the goal it was created with.  stage_rewards [n][HW][9]: the
        goals' reward tables as given (e.g. read back from checkpoint files);
        None: generated by the model rule."""
        n = self.map_height * self.map_width
        g = np.asarray(goals)
        if g.size == 0:
            g = np.zeros((0, 2), np.int64)
        if g.ndim != 2 or g.shape[1] != 2:
            raise ValueError("goals must be [n][2] = (x, y)")
        if not np.issubdtype(g.dtype, np.integer) or (g.size and g.min() < 0):
            raise ValueError("goal coordinates must be integers >= 0")
        g = np.ascontiguousarray(g, dtype=np.uint32)
        sr = None
        if stage_rewards is not None:
            sr = np.ascontiguousarray(stage_rewards, dtype=np.float32)
            if sr.size != g.shape[0] * n * 9:
                raise ValueError(f"stage_rewards must be [{g.shape[0]}][{n}][9]")
        _lib.check(self._lib.pp2d_pomdp_set_goals(self._h, g.ctypes.data if g.size else None,
                                                  g.shape[0],
                                                  sr.ctypes.data if sr is not None else None))

    def goals(self):
        """The goal set as [count][2] (x, y), goal 0 first."""
        c = ctypes.c_uint32()
        _lib.check(self._lib.pp2d_pomdp_goals(self._h, ctypes.byref(c), None))
        out = np.zeros((c.value, 2), np.uint32)
        _lib.check(self._lib.pp2d_pomdp_goals(self._h, ctypes.byref(c), out.ctypes.data))
        return out

    def goal_reward(self, g):
        """Goal g's stage reward table [HW][9]."""
        out = np.empty((self.map_height * self.map_width, 9), np.float32)
        _lib.check(self._lib.pp2d_pomdp_goal_reward(self._h, g, out.ctypes.data))
        return out

    def set_goal_alphas(self, g, fib_alphas, pbvi_alphas, fib_actions=None, pbvi_actions=None):
        """set_alphas for goal g of the goal set (g = 0: set_alphas)."""
        if not isinstance(g, (int, np.integer)) or g < 0:
            raise ValueError("goal index must be an integer >= 0")
        fa = np.ascontiguousarray(fib_alphas, dtype=np.float32)
        pa = np.ascontiguousarray(pbvi_alphas, dtype=np.float32)
        n = self.map_height * self.map_width
        if fa.shape != (n, 9) or pa.ndim != 2 or pa.shape[1] != n:
            raise ValueError("fib_alphas must be [HW][9], pbvi_alphas [N][HW]")
        fac = np.ascontiguousarray(fib_actions, np.uint8) if fib_actions is not None else None
        pac = np.ascontiguousarray(pbvi_actions, np.uint8) if pbvi_actions is not None else None
        _lib.check(self._lib.pp2d_pomdp_set_goal_alphas(
            self._h, int(g), fa.ctypes.data, fac.ctypes.data if fac is not None else None,
            pa.ctypes.data, pac.ctypes.data if pac is not None else None, pa.shape[0]))

    def padding_counters(self):
        """(padded entries, their belief x inner-row products): the part of
        work_counters()[2] spent on padding goal segments to whole tiles."""
        out = np.zeros(2, np.uint64)
        _lib.check(self._lib.pp2d_pomdp_padding_counters(self._h, out.ctypes.data))
        return int(out[0]), int(out[1])

    # -- batched primitives ---------------------------------------------------
    def bayes_update(self, beliefs, actions, observations, normalize=False):
        b = np.ascontiguousarray(beliefs, dtype=np.float32)
        b = b.reshape(-1, self.map_height * self.map_width)
        n = b.shape[0]
        a = np.ascontiguousarray(np.broadcast_to(actions, (n,)), dtype=np.uint8)
        z = np.ascontiguousarray(np.broadcast_to(observations, (n,)), dtype=np.uint8)
        out = np.empty_like(b)
        sums = np.empty(n, np.float32)
        _lib.check(self._lib.pp2d_pomdp_bayes_update(
            self._h, b.ctypes.data, n, a.ctypes.data, z.ctypes.data, int(normalize),
            out.ctypes.data, sums.ctypes.data))
        return (out, sums) if normalize else out

    def evaluate(self, beliefs):
        b = np.ascontiguousarray(beliefs, dtype=np.float32)
        b = b.reshape(-1, self.map_height * self.map_width)
        n = b.shape[0]
        up, lo = np.empty(n, np.float32), np.empty(n, np.float32)
        ua, la = np.empty(n, np.uint8), np.empty(n, np.uint8)
        _lib.check(self._lib.pp2d_pomdp_evaluate(self._h, b.ctypes.data, n, up.ctypes.data,
                                                 ua.ctypes.data, lo.ctypes.data,
                                                 la.ctypes.data))
        return up, ua, lo, la

    def plan_batch(self, beliefs, max_depth=None, max_iter=None, with_stats=False):
        b = np.ascontiguousarray(beliefs, dtype=np.float32)
        b = b.reshape(-1, self.map_height * self.map_width)
        n = b.shape[0]
        acts = np.empty(n, np.uint8)
        vals = np.empty(n, np.float32)
        stats = np.zeros((n, 4), np.uint32)
        _lib.check(self._lib.pp2d_pomdp_plan_batch(
            self._h, b.ctypes.data, n,
            self.max_search_tree_depth if max_depth is None else max_depth,
            self.max_online_iteration if max_iter is None else max_iter,
            acts.ctypes.data, vals.ctypes.data, stats.ctypes.data))
        return (acts, vals, stats) if with_stats else (acts, vals)

    # -- online (path_planning_2d.cu:199-241) ---------------------------------
    def beliefCallback(self, belief, action=0, measurement=(0, 0, 0, 0)):
        observation = ((measurement[3] << 3) + (measurement[2] << 2) +
                       (measurement[1] << 1) + measurement[0])
        if self.search_tree is None:
            self.search_tree = SearchTree(self, belief)
        else:
            self.search_tree.update(action, observation)
        new_action, _ = self.search_tree.plan(self.max_search_tree_depth,
                                              self.max_online_iteration)
        return new_action

    def resetSearchTree(self):
        if self.search_tree is not None:
            self.search_tree.close()
            self.search_tree = None
