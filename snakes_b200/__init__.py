"""snakes_b200 -- B200-native batched multi-snake environment.

Host-side mirror of the reference's Gym / VecEnv interface over libsnk.so (include/snk.h).
Importing this package loads the CUDA library and fails if it has not been built.
"""
from . import _lib
from ._lib import CELL_EMPTY, CELL_FRUIT, CELL_WALL, SnkError, cell_body, cell_head  # noqa: F401

_lib.lib()  # no CPU fallback: a missing extension is an import error

from .vec_env import EnvStates, Infos, MonitorCSV, SnakeVecEnv, StepGraph, expand_views, split_state  # noqa: E402,F401
from .grid_conv import grid_conv84_in, grid_conv_in  # noqa: E402,F401
from .sharding import all_reduce_stats, make_sharded_env, shard_range  # noqa: E402,F401
from .rollout import gae  # noqa: E402,F401
from . import arena, search  # noqa: E402,F401
from .search import RolloutSearch  # noqa: E402,F401
from .registration import ENV_IDS, SnakeGymEnv, make, make_basic_env, register  # noqa: E402,F401

__version__ = "0.3.5"
