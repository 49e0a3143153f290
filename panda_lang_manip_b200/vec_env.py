"""Batched Panda environments on one B200: the vectorised counterpart of the reference's ``RobotTaskEnv``.

``PandaVecEnv(task, num_envs)`` advances ``num_envs`` independent copies of one panda_gym task in lock-step with one
kernel launch per ``step`` (reference hot path: panda_gym/envs/core.py:280-289).  Observations follow the reference's
Dict layout (core.py:229-238) with a leading batch axis, as torch CUDA tensors.
"""
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib

DEFAULT_THRESHOLD = {"reach": 0.05, "push": 0.05, "slide": 0.05, "pick_and_place": 0.05, "stack": 0.1, "flip": 0.2}   # tasks/*.py distance_threshold defaults
MAX_EPISODE_STEPS = {"reach": 50, "push": 50, "slide": 50, "pick_and_place": 50, "stack": 100, "flip": 50}  # panda_gym/__init__.py


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


class _Handle:
    """What task envs and bare worlds do alike with their pg_env handle: raw state, link state, snapshots, rendering and closing.
    Subclasses set ``lib`` (the loaded library), ``_h`` (the handle), ``num_envs``, ``device`` and ``state_dim``."""

    def close(self) -> None:
        if getattr(self, "_h", None) is not None:
            self.lib.pg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    # -- snapshots / raw state ---------------------------------------------------------------------------------------
    def save_state(self) -> int:
        """Stream-ordered snapshot (one device-to-device copy on the current stream, no synchronisation)."""
        import ctypes
        sid = ctypes.c_int()
        _lib.check(self.lib.pg_save_state(self._h, ctypes.byref(sid), self._stream()))
        return sid.value

    def restore_state(self, state_id: int) -> None:
        _lib.check(self.lib.pg_restore_state(self._h, int(state_id), self._stream()))

    def remove_state(self, state_id: int) -> None:
        _lib.check(self.lib.pg_remove_state(self._h, int(state_id)))

    def get_state(self) -> torch.Tensor:
        """[N, state_dim] float64: q(9) qd(9) | per object pos3 quat4 lin3 ang3 | goal (task envs only) | episode step."""
        s = torch.empty((self.num_envs, self.state_dim), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.pg_get_state(self._h, _ptr(s), self._stream()))
        return s

    def set_state(self, state: torch.Tensor, mask: Optional[torch.Tensor] = None) -> None:
        s = state.to(device=self.device, dtype=torch.float64).contiguous()
        m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self.lib.pg_set_state(self._h, _ptr(s), _ptr(m), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def link_state(self, link: int) -> torch.Tensor:
        """[N,13] float64 = getLinkState(link, computeLinkVelocity=1): CoM-frame position, quaternion (x,y,z,w), linear and angular
        velocity of link 0..11, with pybullet's one-sub-step-stale link-transform cache (SURVEY App. B.5)."""
        out = torch.empty((self.num_envs, 13), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.pg_get_link_state(self._h, int(link), _ptr(out), self._stream()))
        return out

    def render(self, width: int = 480, height: int = 480, target_position=(0.0, 0.0, 0.0), distance: float = 1.4, yaw: float = 45, pitch: float = -30, roll: float = 0,
               crop: bool = True, rgb: bool = True, points: bool = True, segmentation: bool = False) -> Dict[str, torch.Tensor]:
        """PyBullet.render (the fork's camera path, pybullet.py:149-264) for every env: analytic ray casting of the primitive scene.
        Returns a dict of device tensors: ``depth`` [N,H,W] (OpenGL depth-buffer values), ``rgb`` [N,H,W,3] uint8, ``points`` [N,H,W,3]
        (the reference's deprojection; NaN where filtered) with ``valid`` [N,H,W] bool (depth < 0.99 and, with ``crop``, the
        reference's workspace box), ``segmentation`` [N,H,W] uint8."""
        n, dev = self.num_envs, self.device
        cam = np.ascontiguousarray([*[float(x) for x in target_position], float(distance), float(yaw), float(pitch), float(roll)], dtype=np.float64)
        out = {"depth": torch.empty((n, height, width), dtype=torch.float32, device=dev)}
        rgba = torch.empty((n, height, width, 4), dtype=torch.uint8, device=dev) if rgb else None
        pts = torch.empty((n, height, width, 3), dtype=torch.float32, device=dev) if points else None
        val = torch.empty((n, height, width), dtype=torch.uint8, device=dev) if points else None
        seg = torch.empty((n, height, width), dtype=torch.uint8, device=dev) if segmentation else None
        _lib.check(self.lib.pg_render(self._h, int(width), int(height), cam.ctypes.data, int(bool(crop)), _ptr(out["depth"]), _ptr(rgba), _ptr(seg), _ptr(pts), _ptr(val), self._stream()))
        if rgb:
            out["rgb"] = rgba[..., :3]
        if points:
            out["points"], out["valid"] = pts, val.bool()
        if segmentation:
            out["segmentation"] = seg
        return out


class PandaVecEnv(_Handle):
    """num_envs lock-stepped panda_gym environments resident in HBM.

    Args mirror the reference constructors (panda_gym/envs/panda_tasks.py): ``reward_type`` "sparse"|"dense",
    ``control_type`` "ee"|"joints".  ``env_id_offset`` is the global index of env 0 (sharded runs), ``precision`` "f32"
    (product path) or "f64" (parity debugging).  ``n_substeps`` is PyBullet(n_substeps) (pybullet.py:26); ``distance_threshold`` and the
    ``*_range_low/high`` noise boxes are the task constructors' keyword arguments (tasks/*.py __init__), see ``set_task_params``.
    ``contact_report``: every ``step`` also reports the contacts of its last sub-step (pybullet getContactPoints), see ``contacts``.
    """

    def __init__(self, task: str, num_envs: int, reward_type: str = "sparse", control_type: str = "ee", device: int = 0,
                 seed: int = 0, env_id_offset: int = 0, precision: str = "f32", auto_reset: bool = True, n_substeps: int = 20,
                 distance_threshold: Optional[float] = None, goal_range_low=None, goal_range_high=None, obj_range_low=None, obj_range_high=None,
                 contact_report: bool = False) -> None:
        import ctypes
        if not torch.cuda.is_available():
            raise _lib.PandaB200Error("PandaVecEnv needs a CUDA device: the B200 kernels are the only implementation")
        self.lib = _lib.load()
        self.task, self.reward_type, self.control_type = task, reward_type, control_type
        self.num_envs, self.device_index, self.auto_reset = int(num_envs), int(device), bool(auto_reset)
        self.device = torch.device("cuda", self.device_index)
        h = ctypes.c_void_p()
        _lib.check(self.lib.pg_create(_lib.TASKS[task], _lib.CONTROL[control_type], _lib.REWARD[reward_type], self.num_envs, self.device_index,
                                      int(seed) & (2**64 - 1), int(env_id_offset), _lib.PRECISION[precision], ctypes.byref(h)))
        self._h = h
        self._pinned = {}
        self.distance_threshold = DEFAULT_THRESHOLD[task]
        self.n_substeps = 20
        if int(n_substeps) != 20:
            self.set_substeps(n_substeps)
        if any(v is not None for v in (distance_threshold, goal_range_low, goal_range_high, obj_range_low, obj_range_high)):
            self.set_task_params(distance_threshold, goal_range_low, goal_range_high, obj_range_low, obj_range_high)
        d = [ctypes.c_int() for _ in range(5)]
        _lib.check(self.lib.pg_dims(h, *[ctypes.byref(x) for x in d]))
        self.obs_dim, self.goal_dim, self.action_dim, self.max_episode_steps, self.state_dim = [x.value for x in d]
        n, f32 = self.num_envs, torch.float32
        self.obs = torch.empty((n, self.obs_dim), dtype=f32, device=self.device)
        self.achieved_goal = torch.empty((n, self.goal_dim), dtype=f32, device=self.device)
        self.desired_goal = torch.empty((n, self.goal_dim), dtype=f32, device=self.device)
        self.reward = torch.empty((n,), dtype=f32, device=self.device)
        self.terminated = torch.empty((n,), dtype=torch.uint8, device=self.device)
        self.truncated = torch.empty((n,), dtype=torch.uint8, device=self.device)
        self._contacts = self._contact_count = None
        if contact_report:
            c = ctypes.c_int()
            _lib.check(self.lib.pg_max_contacts(h, ctypes.byref(c)))
            self.max_contacts = c.value
            self._contacts = torch.zeros((n, self.max_contacts, 16), dtype=f32, device=self.device)
            self._contact_count = torch.zeros((n,), dtype=torch.uint8, device=self.device)
        self.reset()

    # -- lifecycle ---------------------------------------------------------------------------------------------------
    def pin_host(self, array: np.ndarray) -> np.ndarray:
        """Page-lock a caller-owned numpy array (e.g. a reusable action buffer) so that ``step_host`` copies from / to it directly;
        it is unpinned when the env is closed (or with ``unpin_host``).  Keep the array alive until then."""
        a = np.ascontiguousarray(array)
        if a.ctypes.data not in self._pinned:
            _lib.check(self.lib.pg_host_pin(a.ctypes.data, a.nbytes))
            self._pinned[a.ctypes.data] = a
        return a

    def unpin_host(self, array: np.ndarray) -> None:
        if self._pinned.pop(array.ctypes.data, None) is not None:
            _lib.check(self.lib.pg_host_unpin(array.ctypes.data))

    def close(self) -> None:
        for ptr in list(getattr(self, "_pinned", {})):
            self.lib.pg_host_unpin(ptr)
            self._pinned.pop(ptr, None)
        super().close()

    def _obs_dict(self) -> Dict[str, torch.Tensor]:
        return {"observation": self.obs, "achieved_goal": self.achieved_goal, "desired_goal": self.desired_goal}

    # -- RobotTaskEnv API, batched -----------------------------------------------------------------------------------
    def reset(self, mask: Optional[torch.Tensor] = None, goals=None, object_positions=None, seeds=None) -> Dict[str, torch.Tensor]:
        """Reset all envs (or those with mask != 0).  ``goals`` [N,G] / ``object_positions`` [N,3*n_obj] override the device sampler;
        ``seeds`` [N] (ints) is the batched ``reset(seed=k)``: each env's draws are keyed by its own seed only."""
        def f64(x):
            return None if x is None else torch.as_tensor(np.asarray(x, dtype=np.float64) if not torch.is_tensor(x) else x, dtype=torch.float64, device=self.device).contiguous()
        g, o = f64(goals), f64(object_positions)
        m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
        sd = None
        if seeds is not None:       # uint64 bit patterns travel as int64
            sd = torch.as_tensor(np.asarray(seeds.cpu() if torch.is_tensor(seeds) else seeds).astype(np.uint64).view(np.int64), device=self.device).reshape(self.num_envs).contiguous()
        _lib.check(self.lib.pg_reset(self._h, _ptr(m), _ptr(sd), _ptr(g), _ptr(o), _ptr(self.obs), _ptr(self.achieved_goal), _ptr(self.desired_goal), self._stream()))
        if sd is not None:
            torch.cuda.current_stream(self.device).synchronize()
        return self._obs_dict()

    def set_task_params(self, distance_threshold: Optional[float] = None, goal_range_low=None, goal_range_high=None, obj_range_low=None, obj_range_high=None) -> None:
        """The reference task constructors' keyword arguments as kernel parameters: success / sparse-reward threshold, goal noise box
        (3-vectors; what reach.py:21-23 / push.py:20-21 / slide.py:22-23 / pick_and_place.py:24-25 build from goal_range, goal_xy_range,
        goal_z_range, goal_x_offset) and object xy noise box (2-vectors; obj_xy_range).  None keeps a value."""
        def arr(x, k):
            return None if x is None else np.ascontiguousarray(np.asarray(x, dtype=np.float64).reshape(-1)[:k])
        thr = self.distance_threshold if distance_threshold is None else float(distance_threshold)
        gl, gh, ol, oh = arr(goal_range_low, 3), arr(goal_range_high, 3), arr(obj_range_low, 2), arr(obj_range_high, 2)
        _lib.check(self.lib.pg_set_task_params(self._h, thr, *[None if a is None else a.ctypes.data for a in (gl, gh, ol, oh)]))
        self.distance_threshold = thr

    def set_substeps(self, n_substeps: int) -> None:
        """PyBullet(n_substeps) (pybullet.py:26): stepSimulation calls per env step."""
        _lib.check(self.lib.pg_set_substeps(self._h, int(n_substeps)))
        self.n_substeps = int(n_substeps)

    def set_action_scale(self, ee_scale: float = 0.05, finger_scale: float = 0.2) -> None:
        """Action scaling of Panda.set_action (panda.py:65,81); the fork's panda_cartesian robot uses (1.0, 1.0)."""
        _lib.check(self.lib.pg_set_action_scale(self._h, float(ee_scale), float(finger_scale)))

    def step(self, actions: torch.Tensor, target_orientation: Optional[torch.Tensor] = None):
        """One env step.  ``target_orientation`` [N,4] (x,y,z,w): EE orientation target of the fork's panda_ori robot (ee control)."""
        a = actions.to(device=self.device, dtype=torch.float32).contiguous()
        if a.shape != (self.num_envs, self.action_dim):
            raise ValueError(f"actions must be [{self.num_envs}, {self.action_dim}], got {tuple(a.shape)}")
        tq = None if target_orientation is None else target_orientation.to(device=self.device, dtype=torch.float32).reshape(self.num_envs, 4).contiguous()
        _lib.check(self.lib.pg_step(self._h, _ptr(a), _ptr(tq), _ptr(self.obs), _ptr(self.achieved_goal), _ptr(self.desired_goal), _ptr(self.reward),
                                    _ptr(self.terminated), _ptr(self.truncated), int(self.auto_reset), _ptr(self._contacts), _ptr(self._contact_count),
                                    self._stream()))
        return self._obs_dict(), self.reward, self.terminated, self.truncated, {"is_success": self.terminated}

    def contacts(self) -> Dict[str, torch.Tensor]:
        """pybullet getContactPoints after the last ``step``, for every env (env built with ``contact_report=True``): the contacts of the
        step's last sub-step, padded to ``max_contacts`` per env (10, or 22 for Stack); entries at and beyond ``count[i]`` are unspecified.
        The float entries are views of the env's report buffer, overwritten by the next step: ``position`` [N,C,3] (world), ``normal`` [N,C,3] (on B, from B to
        A), ``normal_force`` [N,C] (N), ``lateral_friction1`` / ``lateral_friction2`` [N,C] (N) with ``lateral_friction_dir1`` /
        ``lateral_friction_dir2`` [N,C,3], ``body_a`` / ``body_b`` [N,C] int32 segmentation ids (1 plane, 2 table, 3 / 4 objects, 14 hand,
        15 / 16 fingers) and ``count`` [N] int32 are decoded copies.  With auto-reset the report describes the finished step, like ``reward``."""
        if self._contacts is None:
            raise _lib.PandaB200Error("contacts(): this env was built without contact_report=True")
        r = self._contacts
        ids = r[..., 15].to(torch.int32)
        return {"position": r[..., 0:3], "normal": r[..., 3:6], "normal_force": r[..., 6], "lateral_friction1": r[..., 7], "lateral_friction_dir1": r[..., 8:11],
                "lateral_friction2": r[..., 11], "lateral_friction_dir2": r[..., 12:15], "body_a": ids % 32, "body_b": ids // 32,
                "count": self._contact_count.to(torch.int32)}

    def step_host(self, actions: np.ndarray):
        """End-to-end step with host buffers (numpy in, numpy out): H2D copy, kernel, D2H copy inside the call."""
        a = np.ascontiguousarray(actions, dtype=np.float32)
        n = self.num_envs
        if not hasattr(self, "_host"):
            self._host = dict(obs=np.empty((n, self.obs_dim), np.float32), ag=np.empty((n, self.goal_dim), np.float32), dg=np.empty((n, self.goal_dim), np.float32),
                              rew=np.empty(n, np.float32), term=np.empty(n, np.uint8), trunc=np.empty(n, np.uint8))
            for v in self._host.values():           # the env owns its output arrays: page-lock them, the D2H copies land in them directly
                self.pin_host(v)
        hb = self._host
        _lib.check(self.lib.pg_step_host(self._h, a.ctypes.data, hb["obs"].ctypes.data, hb["ag"].ctypes.data, hb["dg"].ctypes.data, hb["rew"].ctypes.data,
                                         hb["term"].ctypes.data, hb["trunc"].ctypes.data, int(self.auto_reset)))
        return {"observation": hb["obs"], "achieved_goal": hb["ag"], "desired_goal": hb["dg"]}, hb["rew"], hb["term"], hb["trunc"], {"is_success": hb["term"]}

    def compute_reward(self, achieved_goal: torch.Tensor, desired_goal: torch.Tensor, info=None) -> torch.Tensor:
        return compute_reward(self.task, self.reward_type, achieved_goal, desired_goal, threshold=self.distance_threshold)

    def is_success(self, achieved_goal: torch.Tensor, desired_goal: torch.Tensor) -> torch.Tensor:
        return is_success(self.task, achieved_goal, desired_goal, threshold=self.distance_threshold)

    # -- snapshots / raw state ---------------------------------------------------------------------------------------
    def lookahead(self, candidate_actions: torch.Tensor, commit: bool = True):
        """Batched greedy look-ahead search (reference docs/usage/save_restore_state.rst:8-41: save_state, try K sampled actions
        from the same state, keep the one with the best reward): ``candidate_actions`` is [K, N, A]; every env evaluates its K
        candidates from the current state (one snapshot, K restored steps without auto-reset) and, with ``commit``, is then stepped
        with its own best action.  Returns (best_action [N, A], best_reward [N], step result or None).  Ties keep the first candidate."""
        c = candidate_actions.to(device=self.device, dtype=torch.float32)
        if c.dim() != 3 or c.shape[1:] != (self.num_envs, self.action_dim):
            raise ValueError(f"candidate_actions must be [K, {self.num_envs}, {self.action_dim}], got {tuple(c.shape)}")
        sid = self.save_state()
        keep = self.auto_reset
        self.auto_reset = False                      # a candidate that ends the episode must not restart it
        best_r = torch.full((self.num_envs,), -float("inf"), dtype=torch.float32, device=self.device)
        best_k = torch.zeros((self.num_envs,), dtype=torch.long, device=self.device)
        try:
            for k in range(c.shape[0]):
                if k > 0:
                    self.restore_state(sid)
                _, r, _, _, _ = self.step(c[k])
                better = r > best_r
                best_r = torch.where(better, r, best_r)
                best_k = torch.where(better, torch.full_like(best_k, k), best_k)
        finally:
            self.auto_reset = keep
            self.restore_state(sid)
            self.remove_state(sid)
        best_a = c.gather(0, best_k.view(1, -1, 1).expand(1, self.num_envs, self.action_dim))[0].contiguous()
        out = self.step(best_a) if commit else None
        return best_a, best_r, out

    def inverse_kinematics(self, position, orientation, link: Optional[int] = None) -> torch.Tensor:
        """calculateInverseKinematics from the current joint state.  ``link=None``: the env path's link-11 solve, [N,7] arm angles;
        ``link=k``: PyBullet.inverse_kinematics(body, k, ...) for any link 0..11, all nine joint values [N,9]."""
        p = torch.as_tensor(position, dtype=torch.float64, device=self.device).reshape(self.num_envs, 3).contiguous()
        o = torch.as_tensor(orientation, dtype=torch.float64, device=self.device).reshape(self.num_envs, 4).contiguous()
        if link is None:
            out = torch.empty((self.num_envs, 7), dtype=torch.float64, device=self.device)
            _lib.check(self.lib.pg_inverse_kinematics(self._h, _ptr(p), _ptr(o), _ptr(out), self._stream()))
        else:
            out = torch.empty((self.num_envs, 9), dtype=torch.float64, device=self.device)
            _lib.check(self.lib.pg_inverse_kinematics_link(self._h, int(link), _ptr(p), _ptr(o), _ptr(out), self._stream()))
        return out

    def ee_pose(self) -> torch.Tensor:
        """[N,7] float64: end-effector position and quaternion (x,y,z,w) from the current joint state."""
        out = torch.empty((self.num_envs, 7), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.pg_get_ee_pose(self._h, _ptr(out), self._stream()))
        return out

    def diverged(self) -> int:
        """Env-steps that ended in a non-finite state since creation (0 in a healthy run)."""
        import ctypes
        torch.cuda.current_stream(self.device).synchronize()
        c = ctypes.c_longlong()
        _lib.check(self.lib.pg_diverged(self._h, ctypes.byref(c)))
        return int(c.value)

    def contact_overflows(self) -> int:
        """Contact candidates dropped at the per-sub-step cap of the on-chip contact store since creation (10 / 22 for Stack)."""
        import ctypes
        torch.cuda.current_stream(self.device).synchronize()
        c = ctypes.c_longlong()
        _lib.check(self.lib.pg_contact_overflows(self._h, ctypes.byref(c)))
        return int(c.value)

    def stats(self) -> np.ndarray:
        """{episodes, successes, return_sum, length_sum} accumulated by auto-reset on this device."""
        import ctypes
        torch.cuda.current_stream(self.device).synchronize()
        out = (ctypes.c_double * 4)()
        _lib.check(self.lib.pg_stats(self._h, out))
        return np.array(out[:], dtype=np.float64)


def _goal_args(task: str, achieved_goal: torch.Tensor, desired_goal: torch.Tensor):
    if not (torch.is_tensor(achieved_goal) and achieved_goal.is_cuda):
        raise _lib.PandaB200Error("compute_reward/is_success on the B200 path take CUDA tensors (use the panda_gym facade for numpy inputs)")
    g = {"stack": 6, "flip": 4}.get(task, 3)
    if achieved_goal.shape != desired_goal.shape or achieved_goal.shape[-1] != g:
        raise ValueError(f"goals must have matching shapes [..., {g}]")
    dt = torch.float64 if achieved_goal.dtype == torch.float64 else torch.float32
    a = achieved_goal.to(dt).contiguous()
    d = desired_goal.to(device=a.device, dtype=dt).contiguous()
    return a, d, (1 if dt == torch.float64 else 0), a.shape[:-1], a.numel() // g


def compute_reward(task: str, reward_type: str, achieved_goal: torch.Tensor, desired_goal: torch.Tensor, threshold: Optional[float] = None) -> torch.Tensor:
    """Vectorised Task.compute_reward (tasks/<task>.py, utils.py:4-30) for HER relabelling: float32 rewards, bit-exact vs numpy.
    ``threshold``: the task's distance_threshold (default: the reference's 0.05 / 0.1 Stack / 0.2 Flip)."""
    a, d, code, lead, m = _goal_args(task, achieved_goal, desired_goal)
    out = torch.empty(lead, dtype=torch.float32, device=a.device)
    thr = DEFAULT_THRESHOLD[task] if threshold is None else float(threshold)
    with torch.cuda.device(a.device):
        _lib.check(_lib.load().pg_compute_reward(_lib.TASKS[task], _lib.REWARD[reward_type], thr, _ptr(a), _ptr(d), _ptr(out), m, code, torch.cuda.current_stream(a.device).cuda_stream))
    return out


def is_success(task: str, achieved_goal: torch.Tensor, desired_goal: torch.Tensor, threshold: Optional[float] = None) -> torch.Tensor:
    a, d, code, lead, m = _goal_args(task, achieved_goal, desired_goal)
    out = torch.empty(lead, dtype=torch.uint8, device=a.device)
    thr = DEFAULT_THRESHOLD[task] if threshold is None else float(threshold)
    with torch.cuda.device(a.device):
        _lib.check(_lib.load().pg_is_success(_lib.TASKS[task], thr, _ptr(a), _ptr(d), _ptr(out), m, code, torch.cuda.current_stream(a.device).cuda_stream))
    return out.bool()


def her_relabel(task: str, reward_type: str, next_achieved_goal: torch.Tensor, desired_goal: torch.Tensor, src: torch.Tensor, goal_src: torch.Tensor,
                return_achieved: bool = False, threshold: Optional[float] = None):
    """HER relabelling fused with compute_reward, on the device (the learner-side caller of the step path: the reference's
    examples/train_push.py:1-12 sets up stable-baselines3's HerReplayBuffer, which does this with a numpy gather and
    ``env.compute_reward``).  ``next_achieved_goal`` / ``desired_goal`` are the replay buffer's goal arrays flattened to [R, G];
    ``src`` [M] indexes the sampled transitions and ``goal_src`` [M] the transitions whose next achieved goal becomes the new goal
    (negative: keep the stored goal).  Returns (new_desired_goal [M, G], reward [M] float32[, next_achieved_goal[src] [M, G]]).
    Goal arrays passed as ``padded[:, :G]`` views of a buffer with 32-byte rows (``torch.zeros(R, 8)`` for fp32) are gathered in place,
    one DRAM sector per row."""
    if not (torch.is_tensor(next_achieved_goal) and next_achieved_goal.is_cuda):
        raise _lib.PandaB200Error("her_relabel takes CUDA tensors: the replay buffer lives in HBM")
    g = {"stack": 6, "flip": 4}.get(task, 3)
    dt = torch.float64 if next_achieved_goal.dtype == torch.float64 else torch.float32

    def rows(t):
        """[R, G] view and its row pitch in elements: a 2-D tensor whose rows are unit-stride slices of a wider (padded) buffer is used
        in place (the pitch argument of pg_her_relabel); anything else is flattened to dense rows."""
        t = t.to(device=next_achieved_goal.device, dtype=dt)
        if t.dim() == 2 and t.shape[1] == g and t.stride(1) == 1 and t.stride(0) >= g:
            return t, t.stride(0)
        t = t.reshape(-1, g).contiguous()
        return t, g
    a, pa = rows(next_achieved_goal)
    d, pd = rows(desired_goal)
    if pa != pd:                                        # one pitch for both arrays
        a, d, pa = a.contiguous(), d.contiguous(), g
    if a.shape != d.shape:
        raise ValueError("next_achieved_goal and desired_goal must have the same [R, G] shape")
    s_ = src.to(device=a.device, dtype=torch.long).contiguous()
    gs = goal_src.to(device=a.device, dtype=torch.long).contiguous()
    if s_.shape != gs.shape or s_.dim() != 1:
        raise ValueError("src and goal_src must be 1-D and of equal length")
    m = s_.numel()
    new_dg = torch.empty((m, g), dtype=dt, device=a.device)
    ag_out = torch.empty((m, g), dtype=dt, device=a.device) if return_achieved else None
    rew = torch.empty((m,), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(_lib.load().pg_her_relabel(_lib.TASKS[task], _lib.REWARD[reward_type], DEFAULT_THRESHOLD[task] if threshold is None else float(threshold),
                                              _ptr(a), _ptr(d), pa, _ptr(s_), _ptr(gs), _ptr(new_dg), _ptr(ag_out), _ptr(rew),
                                              m, 1 if dt == torch.float64 else 0, torch.cuda.current_stream(a.device).cuda_stream))
    return (new_dg, rew, ag_out) if return_achieved else (new_dg, rew)


def future_goal_indices(episode_start: torch.Tensor, episode_length: torch.Tensor, src: torch.Tensor, her_ratio: float = 0.8,
                        generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """The "future" goal-selection strategy of HER for ``her_relabel``: transition ``src[j]`` belongs to an episode stored in the
    flat rows [episode_start[j], episode_start[j] + episode_length[j]); with probability ``her_ratio`` pick a row uniformly from
    the transition's own row to the episode's last row, else -1 (keep the stored goal)."""
    off = src - episode_start
    span = (episode_length - off).clamp_min(1)
    u = torch.rand(src.shape, device=src.device, generator=generator)
    fut = src + (u * span).long().clamp_max(span - 1)
    keep = torch.rand(src.shape, device=src.device, generator=generator) >= her_ratio
    return torch.where(keep, torch.full_like(fut, -1), fut)


def her_sample_indices(num_rows: int, batch: int, episode_length: int, her_ratio: float = 0.8, device=None,
                       generator: Optional[torch.Generator] = None, sort: bool = True):
    """Sampled transitions and their "future" goal rows for ``her_relabel`` on a replay buffer whose episodes are stored back to back
    (``episode_length`` rows each, as stable-baselines3's HerReplayBuffer lays them out per env): returns ``(src, goal_src)``.
    With ``sort=True`` (default) ``src`` is ascending: a batch is a set, so its order is free, and an index-sorted batch turns the two
    random row gathers into near-sequential ones -- the sampled rows are ~num_rows / batch apart and a transition's future goal lies at
    most ``episode_length`` rows behind it, so consecutive threads read neighbouring DRAM pages (and sectors of the same cache lines)
    instead of one random 32-byte sector each.  The same ``src`` then serves the observation / action gathers of the batch."""
    device = torch.device("cuda") if device is None else device
    src = torch.randint(0, num_rows, (batch,), device=device, generator=generator)
    if sort:
        src = torch.sort(src).values
    start = (src // episode_length) * episode_length
    length = torch.minimum(torch.full_like(src, episode_length), num_rows - start)
    return src, future_goal_indices(start, length, src, her_ratio, generator)

