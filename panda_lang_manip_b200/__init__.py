"""panda_lang_manip_b200 -- B200-native batched Panda manipulation environments behind the panda_gym API.

Hot path: ``PandaVecEnv`` (batched step in one CUDA kernel launch) and ``compute_reward`` / ``is_success`` (HER relabelling).
Drop-in layer: ``panda_lang_manip_b200.panda_gym`` mirrors the reference package (env classes, ids, Task / robot plug-ins).
"""
from ._lib import PandaB200Error, build, kernel_launches, load  # noqa: F401
from .bare_world import PandaBareWorld  # noqa: F401
from .vec_env import MAX_EPISODE_STEPS, PandaVecEnv, compute_reward, future_goal_indices, her_relabel, her_sample_indices, is_success  # noqa: F401
from .motion import CartesianMotion  # noqa: F401

__all__ = ["PandaVecEnv", "PandaBareWorld", "CartesianMotion", "compute_reward", "is_success", "her_relabel", "future_goal_indices", "her_sample_indices", "build", "load", "kernel_launches", "PandaB200Error", "MAX_EPISODE_STEPS"]
