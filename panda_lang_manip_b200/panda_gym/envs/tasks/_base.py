"""Shared implementation of the six task plug-ins (reference panda_gym/envs/tasks/*.py)."""
from typing import Any, Dict

import numpy as np

from ..core import Task
from ...sampling import default_ranges, sample_reset

_G = {"stack": 6, "flip": 4}


class BuiltinTask(Task):
    name = ""
    default_threshold = 0.05

    def __init__(self, sim, reward_type: str = "sparse", distance_threshold: float = None, goal_range: float = None, goal_xy_range: float = None,
                 goal_z_range: float = None, goal_x_offset: float = None, obj_xy_range: float = None) -> None:
        """Keyword arguments as in the reference constructors (reach.py:15-23, push.py:12-25, slide.py:12-27, pick_and_place.py:13-29,
        stack.py:11-25, flip.py:13-24); they become parameters of the step / reset kernels (pg_set_task_params)."""
        super().__init__(sim)
        self.reward_type = reward_type
        self.distance_threshold = self.default_threshold if distance_threshold is None else float(distance_threshold)
        self.goal_range_low, self.goal_range_high, self.obj_range_low, self.obj_range_high = default_ranges(
            self.name, goal_range=goal_range, goal_xy_range=goal_xy_range, goal_z_range=goal_z_range, goal_x_offset=goal_x_offset, obj_xy_range=obj_xy_range)
        if self.distance_threshold != self.default_threshold or any(v is not None for v in (goal_range, goal_xy_range, goal_z_range, goal_x_offset, obj_xy_range)):
            self.sim._require().set_task_params(self.distance_threshold, self.goal_range_low, self.goal_range_high, self.obj_range_low[:2], self.obj_range_high[:2])
        self.np_random = np.random.default_rng()
        self._object_positions = []
        with self.sim.no_rendering():
            self._create_scene()

    def _create_scene(self) -> None:
        self.sim.create_plane(z_offset=-0.4)
        self.sim.create_table(length=1.4 if self.name == "slide" else 1.1, width=0.7, height=0.4, x_offset=-0.1 if self.name == "slide" else -0.3)

    def reset(self) -> None:
        self.goal, self._object_positions = sample_reset(self.name, self.np_random, (self.goal_range_low, self.goal_range_high, self.obj_range_low, self.obj_range_high))

    def get_obs(self) -> np.ndarray:
        o = (self.sim._last_obs[0] if self.sim._last_obs is not None else self.sim._reset_obs)["observation"]
        return np.asarray(o[6 if self.name in ("reach", "push", "slide") else 7:], dtype=np.float64)

    def get_achieved_goal(self) -> np.ndarray:
        return np.asarray((self.sim._last_obs[0] if self.sim._last_obs is not None else self.sim._reset_obs)["achieved_goal"], dtype=np.float64)

    # HER entry points: numpy in, numpy out, evaluated by the CUDA kernels through the host-buffer C-ABI calls
    def _goals(self, achieved_goal, desired_goal):
        a, d = np.asarray(achieved_goal), np.asarray(desired_goal)
        assert a.shape == d.shape
        dt = np.float64 if a.dtype == np.float64 or d.dtype == np.float64 else np.float32
        return np.ascontiguousarray(a, dtype=dt), np.ascontiguousarray(d, dtype=dt), a.shape[:-1], (1 if dt == np.float64 else 0)

    def is_success(self, achieved_goal: np.ndarray, desired_goal: np.ndarray, info: Dict[str, Any] = {}) -> np.ndarray:
        from .... import _lib
        a, d, lead, code = self._goals(achieved_goal, desired_goal)
        out = np.empty(lead, dtype=np.uint8)
        m = int(np.prod(lead)) if lead else 1
        _lib.check(_lib.load().pg_is_success_host(_lib.TASKS[self.name], float(self.distance_threshold), a.ctypes.data, d.ctypes.data, out.ctypes.data, m, code,
                                                  self.sim._require().device_index))
        return np.array(out.astype(np.bool_))

    def compute_reward(self, achieved_goal: np.ndarray, desired_goal: np.ndarray, info: Dict[str, Any] = {}) -> np.ndarray:
        from .... import _lib
        a, d, lead, code = self._goals(achieved_goal, desired_goal)
        out = np.empty(lead, dtype=np.float32)
        m = int(np.prod(lead)) if lead else 1
        _lib.check(_lib.load().pg_compute_reward_host(_lib.TASKS[self.name], _lib.REWARD[self.reward_type], float(self.distance_threshold), a.ctypes.data, d.ctypes.data,
                                                      out.ctypes.data, m, code, self.sim._require().device_index))
        return out
