"""hironaka_b200 — B200-native batched Hironaka game engine (env-step path of honglu2875/hironaka).

Layers (bottom up):
  csrc/            hand-written sm_100a kernels + the extern "C" boundary (include/hironaka_b200.h)
  _lib, ops        ctypes loader and tensor-level launch wrappers (no fallback path)
  src              drop-in for hironaka.src torch ops (shift_torch, get_newton_polytope_torch, ...)
  TensorPoints     drop-in for hironaka.core.TensorPoints (the `point_cls=` seam)
  FusedGame        drop-in for hironaka.trainer.fused_game.FusedGame (one launch per move)
  functional       drop-in for hironaka/jax/util.py (take_actions, get_dones, reward_fn, feature_fn, ...)
  GameBatch        resident int32 batches, fused T-step rollouts, sharding + rollout all-gather
  HostSession      NumPy host-buffer sessions over hk_session_*
  VecHironaka*Env  batched forms of the gym environments (hironaka/gym_env)
  search_depth     game-tree search of a fixed host against every agent reply (hironaka/util/search.py)
  search_value     game value: the shortest game the best host can force against every agent reply
  search_*_line    the same searches with a line of play per root; play_line replays lines into states
  search_value_labels  every state the value search solved: exact value, optimal host moves, path and rows
"""
from . import constants
from .constants import *  # noqa: F401,F403
from ._lib import HironakaB200Error, LIB_PATH

__version__ = "0.1.0"


def __getattr__(name):  # lazy: importing the package must not require torch or a built library
    if name in ("TensorPoints", "CudaTensorPoints"):
        from .tensor_points import TensorPoints
        return TensorPoints
    if name == "PointsBase":
        from .points_base import PointsBase
        return PointsBase
    if name in ("GameBatch", "shard_range", "gather_rollout", "compute_rho"):
        from . import engine
        return getattr(engine, name)
    if name == "HostSession":
        from .session import HostSession
        return HostSession
    if name == "ReplayBuffer":
        from .replay_buffer import ReplayBuffer
        return ReplayBuffer
    if name == "FusedGame":
        from .fused_game import FusedGame
        return FusedGame
    if name in ("VecHironakaAgentEnv", "VecHironakaHostEnv"):
        from . import vec_env
        return getattr(vec_env, name)
    if name in ("search_depth", "SearchResult", "STATUS_RESOLVED", "STATUS_MAX_DEPTH", "STATUS_MAX_NODES",
                "STATUS_CAPACITY", "STATUS_INT32_BOUND", "search_value", "ValueResult", "STATUS_HISTORY",
                "search_depth_line", "DepthLine", "search_value_line", "ValueLine", "play_line", "search_value_labels",
                "ValueLabels"):
        from . import search
        return getattr(search, name)
    if name == "HostActionEncoder":
        from .host_action import HostActionEncoder
        return HostActionEncoder
    if name in ("ops", "src", "functional", "engine", "session", "host_action", "build", "fused_game", "players", "replay_buffer", "vec_env",
                "search"):
        import importlib
        return importlib.import_module(f".{name}", __name__)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
