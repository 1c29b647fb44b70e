"""B200-native hot path of path_planning_2d (MDP value iteration and QV-tree
node expansion) behind the C ABI of include/pp2d.h."""
from . import _lib  # noqa: F401
from .mdp import MdpBatchPathPlanning2d, MdpPathPlanning2d, load_map_png  # noqa: F401
from .pomdp import PomdpPathPlanning2d, SearchTree, SearchTreeBatch  # noqa: F401
from .simulator import DummySimulator  # noqa: F401
from .distributed import ShardedValueIteration, partition_rows  # noqa: F401

__all__ = ["MdpPathPlanning2d", "MdpBatchPathPlanning2d", "PomdpPathPlanning2d", "SearchTree",
           "SearchTreeBatch", "DummySimulator", "ShardedValueIteration", "load_map_png", "partition_rows"]
