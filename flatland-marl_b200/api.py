"""Public names of the package."""
from . import _lib
from ._lib import FlatlandB200Error
from .batch import BatchedRailEnv, EnvSnapshot
from .rail_env import AgentView, RailEnv, TrainState, TreeObsForRailEnv
from .evaluator import FlatlandRemoteClient
from .persistence import RailEnvPersister, load_env_dict, load_level, world_from_env_dict
from .reset_pipeline import GeneratorPool, PackSource, ResetPipeline, WorldSource
from .learner import PolicyLearner
from .rollout import Rollout
from .shard import final_metric, max_over_ranks, reduce_episode_stats, shard_range, weak_offset
from .worlds import (draw_schedule, draw_schedule_fast, load_worlds_npz, save_worlds_npz, unique_target_slots,
                     world_from_reference_env)

__all__ = ["BatchedRailEnv", "EnvSnapshot", "RailEnv", "TreeObsForRailEnv", "TrainState", "AgentView", "FlatlandB200Error",
           "world_from_reference_env", "draw_schedule", "draw_schedule_fast", "load_worlds_npz", "save_worlds_npz",
           "unique_target_slots", "shard_range", "weak_offset", "reduce_episode_stats", "max_over_ranks",
           "final_metric", "load_level", "load_env_dict", "world_from_env_dict", "ResetPipeline", "PackSource", "GeneratorPool",
           "WorldSource", "Rollout", "PolicyLearner", "FlatlandRemoteClient", "RailEnvPersister", "_lib"]
