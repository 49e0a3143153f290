"""The fork's scripted motion primitives for every env of a ``PandaVecEnv``: the batched counterpart of ``move`` / ``grasp`` / ``release``
in robots/panda_cartesian.py (the facade ``panda_gym.envs.robots.panda_cartesian.Panda``, one env at a time).

Each env runs its own primitive with its own step count, and envs may be in different primitives at once.  A primitive step is one
small per-env kernel (actions and EE target orientations from the current joint state) plus the env step, enqueued on the current
stream with no host synchronisation.  Steps taken here never auto-reset; reset explicitly with ``env.reset(mask=...)``.
"""
import ctypes
from typing import Dict, Optional, Tuple

import torch

from . import _lib
from .vec_env import PandaVecEnv, _ptr

GRIPPER_STEPS = 30          # panda_cartesian.py:60-68


def quat_from_euler_xyz_deg(euler: torch.Tensor) -> torch.Tensor:
    """[..., 3] xyz extrinsic Euler angles in degrees -> [..., 4] quaternions (x, y, z, w), float64 (panda_ori.quat_from_euler_xyz_deg)."""
    r, p, y = (torch.deg2rad(euler.to(torch.float64)) / 2).unbind(-1)
    cr, sr, cp, sp, cy, sy = torch.cos(r), torch.sin(r), torch.cos(p), torch.sin(p), torch.cos(y), torch.sin(y)
    return torch.stack([sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy, cr * cp * sy - sr * sp * cy, cr * cp * cy + sr * sp * sy], dim=-1)


class CartesianMotion:
    """move / grasp / release for every env of ``env`` (an ee-controlled ``PandaVecEnv``).  Sets the env's action scale to the fork's
    unscaled (1.0, 1.0).  ``mask`` ([N] bool or uint8, default all) selects the envs a primitive begins on; a primitive begun on an env
    replaces the one it was running.  An env with no primitive left is stepped in place (zero displacement, fingers held)."""

    def __init__(self, env: PandaVecEnv) -> None:
        if env.control_type != "ee":
            raise _lib.PandaB200Error("CartesianMotion needs an ee-controlled PandaVecEnv")
        self.env, self.lib = env, env.lib
        env.set_action_scale(1.0, 1.0)
        h = ctypes.c_void_p()
        _lib.check(self.lib.pg_motion_create(env.num_envs, env.device_index, ctypes.byref(h)))
        self._h = h
        self.remaining = torch.zeros((env.num_envs,), dtype=torch.int32, device=env.device)

    def _rows(self, x, width: int) -> torch.Tensor:
        return torch.as_tensor(x, dtype=torch.float64, device=self.env.device).expand(self.env.num_envs, width).contiguous()

    def _mask(self, mask) -> Optional[torch.Tensor]:
        return None if mask is None else torch.as_tensor(mask, device=self.env.device).to(torch.uint8).reshape(self.env.num_envs).contiguous()

    def move(self, goal_pos, goal_euler=None, goal_quat=None, mask=None) -> None:
        """Move the EE to ``goal_pos`` ([N,3] or [3], m) in 1.5 cm way-points while turning it to ``goal_euler`` (xyz Euler angles in
        degrees, as the facade takes them) or ``goal_quat`` ((x, y, z, w)); exactly one of the two."""
        if (goal_euler is None) == (goal_quat is None):
            raise ValueError("move: give exactly one of goal_euler and goal_quat")
        q = self._rows(goal_quat, 4) if goal_euler is None else quat_from_euler_xyz_deg(self._rows(goal_euler, 3)).contiguous()
        p, m = self._rows(goal_pos, 3), self._mask(mask)
        _lib.check(self.lib.pg_motion_move(self._h, self.env._h, _ptr(p), _ptr(q), _ptr(m), self.env._stream()))

    def _gripper(self, finger_action: float, mask) -> None:
        m = self._mask(mask)
        _lib.check(self.lib.pg_motion_gripper(self._h, self.env._h, float(finger_action), GRIPPER_STEPS, _ptr(m), self.env._stream()))

    def grasp(self, mask=None) -> None:
        """Close the fingers: 30 steps of finger action -1 with the EE held in place."""
        self._gripper(-1.0, mask)

    def release(self, width: float = 1.0, mask=None) -> None:
        """Open the fingers: 30 steps of finger action ``width`` with the EE held in place."""
        self._gripper(width, mask)

    def step(self) -> Tuple[Dict[str, torch.Tensor], torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
        """One env step of every env's primitive: (obs dict, reward, terminated, truncated, remaining), device tensors.  The obs buffers
        are the env's own; ``remaining`` [N] int32 counts the steps of each env's primitive still to take."""
        e = self.env
        _lib.check(self.lib.pg_motion_step(self._h, e._h, _ptr(e.obs), _ptr(e.achieved_goal), _ptr(e.desired_goal), _ptr(e.reward), _ptr(e.terminated),
                                           _ptr(e.truncated), _ptr(self.remaining), e._stream()))
        return e._obs_dict(), e.reward, e.terminated, e.truncated, self.remaining

    def run(self):
        """Step until every env's primitive is done: one step, one read of ``remaining.max()``, then that many steps.  Returns the last
        ``step`` result."""
        out = self.step()
        for _ in range(int(self.remaining.max())):
            out = self.step()
        return out

    def close(self) -> None:
        if getattr(self, "_h", None) is not None:
            self.lib.pg_motion_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
