"""Host-side mirror of the belief filter of the reference's DummySimulator
(/root/reference/dummy_simulator/src/dummy_simulator.cpp:671-773) over the C
ABI.  The reference keeps ONE belief and updates it on the CPU once per
control message; here any number of independent beliefs (many simulated
robots) are filtered in one call on the GPU, each with its own action /
measurement, with the reference's bits.

rollout() runs the whole closed loop of the reference's planner + simulator
pair on the GPU for many episodes at once (Monte-Carlo runs of an MDP
planner): plan at the belief mode, move, sense, filter, until the goal or a
step limit, with motion and sensor noise drawn from a counter-based Philox
generator so that every episode is reproducible on its own (DESIGN.md
section 7, "Closed-loop rollouts")."""
import ctypes

import numpy as np

from . import _lib
from .mdp import MdpBatchPathPlanning2d, MdpPathPlanning2d
from .pomdp import PomdpPathPlanning2d, _goal_indices


class DummySimulator:
    def __init__(self, grid_map):
        grid_map = np.ascontiguousarray(grid_map, dtype=np.uint8)
        self.map_height, self.map_width = grid_map.shape
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        _lib.check(self._lib.pp2d_sim_create(self.map_height, self.map_width,
                                             grid_map.ctypes.data, ctypes.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.pp2d_sim_destroy(self._h)
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

    def _beliefs(self, beliefs):
        b = np.array(beliefs, dtype=np.float32, order="C", copy=True)
        return b.reshape(-1, self.map_height * self.map_width)

    def updateBelief(self, beliefs, action=None, measurement=None):
        """updateBelief(u) when `action` is given (one value or one per belief),
        updateBelief(meas) when `measurement` is given ([4] or [n][4]); both:
        controlCallback's order, action first.  Returns the new beliefs."""
        b = self._beliefs(beliefs)
        n = b.shape[0]
        a = m = None
        if action is not None:
            a = np.ascontiguousarray(np.broadcast_to(action, (n,)), dtype=np.uint8)
        if measurement is not None:
            m = np.ascontiguousarray(np.broadcast_to(measurement, (n, 4)), dtype=np.uint8)
        if a is not None and m is not None:
            rc = self._lib.pp2d_sim_step(self._h, b.ctypes.data, n, a.ctypes.data, m.ctypes.data)
        elif a is not None:
            rc = self._lib.pp2d_sim_update_belief_action(self._h, b.ctypes.data, n, a.ctypes.data)
        elif m is not None:
            rc = self._lib.pp2d_sim_update_belief_measurement(self._h, b.ctypes.data, n,
                                                              m.ctypes.data)
        else:
            raise ValueError("give an action, a measurement, or both")
        _lib.check(rc)
        return b

    def rollout(self, planner, starts, max_steps, seed, beliefs=None, instances=None,
                first_episode=0, record=False, max_depth=None, max_iter=None, goals=None):
        """Closed-loop episodes of `planner` (MdpPathPlanning2d, or
        MdpBatchPathPlanning2d with `instances`: the instance each episode
        follows, or PomdpPathPlanning2d: one search tree per episode, planned
        with max_depth / max_iter, default the planner's 50 / 15, and updated
        with each action and measurement; final_belief is then the tree's
        root belief; with `goals`, episode i plans to goal goals[i] of the
        planner's goal set and stops on that goal's cell) in this simulator's map, from starts [n][2] = (x, y), with
        beliefs [n][H*W] (default: a point mass at each start).  Episode i
        draws its noise as episode first_episode + i of `seed`.  Returns a dict
        of steps, reached, collisions and final_cell (y*W+x) per episode; with
        record=True also final_belief [n][H*W], cells [n][max_steps+1] (the
        start first), actions and measurements [n][max_steps] (bit j = sensor
        j of up, left, right, down).  Entries past an episode's last step are
        0."""
        st = np.ascontiguousarray(starts, dtype=np.uint32).reshape(-1, 2)
        n = st.shape[0]
        hw = self.map_height * self.map_width
        b = None
        if beliefs is not None:
            b = np.ascontiguousarray(beliefs, dtype=np.float32).reshape(n, hw)
        res = {"steps": np.zeros(n, np.uint32), "reached": np.zeros(n, np.uint8),
               "collisions": np.zeros(n, np.uint32), "final_cell": np.zeros(n, np.uint32)}
        if record:
            res["final_belief"] = np.zeros((n, hw), np.float32)
            res["cells"] = np.zeros((n, max_steps + 1), np.uint32)
            res["actions"] = np.zeros((n, max_steps), np.uint8)
            res["measurements"] = np.zeros((n, max_steps), np.uint8)
        out = _lib.Rollout(**{k: v.ctypes.data for k, v in res.items()})
        bp = b.ctypes.data if b is not None else None
        if not isinstance(planner, PomdpPathPlanning2d) and (max_depth, max_iter) != (None, None):
            raise ValueError("max_depth / max_iter are for a PomdpPathPlanning2d")
        if not isinstance(planner, PomdpPathPlanning2d) and goals is not None:
            raise ValueError("`goals` is for a PomdpPathPlanning2d")
        if isinstance(planner, PomdpPathPlanning2d):
            if instances is not None:
                raise ValueError("`instances` is for a batch planner")
            depth = planner.max_search_tree_depth if max_depth is None else max_depth
            it = planner.max_online_iteration if max_iter is None else max_iter
            if goals is None:
                rc = self._lib.pp2d_sim_rollout_pomdp(self._h, planner._h, n, st.ctypes.data, bp,
                                                      max_steps, depth, it, seed, first_episode,
                                                      ctypes.byref(out))
            else:
                g = _goal_indices(goals, n, "episode")
                rc = self._lib.pp2d_sim_rollout_pomdp_goals(
                    self._h, planner._h, g.ctypes.data, n, st.ctypes.data, bp, max_steps, depth,
                    it, seed, first_episode, ctypes.byref(out))
        elif isinstance(planner, MdpBatchPathPlanning2d):
            if instances is None:
                raise ValueError("a batch planner needs `instances`, one per episode")
            idx = np.ascontiguousarray(instances, dtype=np.uint32).reshape(-1)
            if idx.size != n:
                raise ValueError("one instance per episode")
            rc = self._lib.pp2d_sim_rollout_mdp_batch(self._h, planner._h, idx.ctypes.data, n,
                                                      st.ctypes.data, bp, max_steps, seed,
                                                      first_episode, ctypes.byref(out))
        elif isinstance(planner, MdpPathPlanning2d):
            if instances is not None:
                raise ValueError("`instances` is for a batch planner")
            rc = self._lib.pp2d_sim_rollout_mdp(self._h, planner._h, n, st.ctypes.data, bp,
                                                max_steps, seed, first_episode,
                                                ctypes.byref(out))
        else:
            raise TypeError("planner must be an MdpPathPlanning2d, MdpBatchPathPlanning2d or "
                            "PomdpPathPlanning2d")
        _lib.check(rc)
        return res
