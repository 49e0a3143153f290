"""The reference's sim facade used without a task, batched: ``PandaBareWorld`` is what ``PyBullet()`` + ``loadURDF`` + ``create_box`` +
``control_joints`` + ``step`` give in the reference (panda_gym/pybullet.py:16-68, 462-477, 510-771), for ``num_envs`` identical worlds
on one B200.  It exists so that the reference's own known-answer tests (test/pybullet_test.py) run against the CUDA kernels, and as the
backend of the unbound ``panda_gym.pybullet.PyBullet`` facade."""
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .vec_env import _Handle, _ptr

JOINT_TO_DOF = {0: 0, 1: 1, 2: 2, 3: 3, 4: 4, 5: 5, 6: 6, 9: 7, 10: 8}


class PandaBareWorld(_Handle):
    """num_envs worlds: Panda at ``robot_base`` (None: no robot), up to two free bodies, optional table top (z = 0) and ground plane.

    ``bodies``: sequence of dicts ``{"shape": "box"|"cylinder", "half_extents": (hx,hy,hz) | "radius"/"height", "mass", "position",
    "orientation" (x,y,z,w), "lateral_friction"}`` (reference create_box / create_cylinder arguments, pybullet.py:531-640).
    """

    def __init__(self, num_envs: int = 1, robot_base: Optional[Sequence[float]] = (0.0, 0.0, 0.0), bodies: Sequence[dict] = (), table_rect: Optional[Sequence[float]] = None,
                 ground_z: Optional[float] = None, device: int = 0, precision: str = "f32") -> None:
        import ctypes
        if not torch.cuda.is_available():
            raise _lib.PandaB200Error("PandaBareWorld needs a CUDA device: the B200 kernels are the only implementation")
        self.lib = _lib.load()
        self.num_envs, self.device = int(num_envs), torch.device("cuda", int(device))
        rows = []
        for b in bodies:
            if b.get("shape", "box") == "box":
                h = [float(x) for x in b["half_extents"]]; shape = 0.0
            else:
                h = [float(b["radius"]), float(b["radius"]), float(b["height"]) / 2]; shape = 1.0
            rows.append([shape, *h, float(b.get("mass", 1.0)), float(b.get("lateral_friction", 0.5)), *[float(x) for x in b.get("position", (0, 0, 0))],
                         *[float(x) for x in b.get("orientation", (0, 0, 0, 1))]])
        self.n_bodies = len(rows)
        body_arr = np.ascontiguousarray(np.array(rows, dtype=np.float64).reshape(-1, 13))
        base = None if robot_base is None else np.ascontiguousarray(robot_base, dtype=np.float64)
        rect = None if table_rect is None else np.ascontiguousarray(table_rect, dtype=np.float64)
        gz = None if ground_z is None else np.array([ground_z], dtype=np.float64)
        self.has_robot = robot_base is not None
        h = ctypes.c_void_p()
        _lib.check(self.lib.pg_create_bare(self.num_envs, int(device), _lib.PRECISION[precision], None if base is None else base.ctypes.data, self.n_bodies,
                                           body_arr.ctypes.data if self.n_bodies else None, None if rect is None else rect.ctypes.data, None if gz is None else gz.ctypes.data, ctypes.byref(h)))
        self._h = h
        self.state_dim = 18 + 13 * self.n_bodies + 1

    # ---- PyBullet.step / control_joints ---------------------------------------------------------------------------------------------
    def step(self, n_substeps: int = 20) -> None:
        """pybullet.py:52-55: n_substeps x stepSimulation (1/500 s each)."""
        _lib.check(self.lib.pg_sim_step(self._h, int(n_substeps), self._stream()))

    def get_motors(self) -> torch.Tensor:
        """[N,9,5]: position gain, velocity gain, target angle, target velocity, max force of joints 0-6, 9, 10."""
        out = torch.empty((self.num_envs, 9, 5), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.pg_get_motors(self._h, _ptr(out), self._stream()))
        return out

    def set_motors(self, motors: torch.Tensor, mask: Optional[torch.Tensor] = None) -> None:
        m = motors.to(device=self.device, dtype=torch.float64).reshape(self.num_envs, 9, 5).contiguous()
        k = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self.lib.pg_set_motors(self._h, _ptr(m), _ptr(k), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()       # m / k may be temporaries

    def control_joints(self, joints: Sequence[int], target_angles: Sequence[float], forces: Sequence[float]) -> None:
        """pybullet.py:462-477: POSITION_CONTROL (gains 0.1 / 1.0, target velocity 0) on the listed joints of every world."""
        m = self.get_motors()
        for j, a, f in zip(joints, target_angles, forces):
            d = JOINT_TO_DOF[int(j)]
            m[:, d, 0], m[:, d, 1], m[:, d, 2], m[:, d, 3], m[:, d, 4] = 0.1, 1.0, float(a), 0.0, float(f)
        self.set_motors(m)

    def inverse_kinematics(self, link: int, position, orientation) -> torch.Tensor:
        p = torch.as_tensor(np.asarray(position, dtype=np.float64), device=self.device).expand(self.num_envs, 3).contiguous()
        o = torch.as_tensor(np.asarray(orientation, dtype=np.float64), device=self.device).expand(self.num_envs, 4).contiguous()
        out = torch.empty((self.num_envs, 9), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.pg_inverse_kinematics_link(self._h, int(link), _ptr(p), _ptr(o), _ptr(out), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()
        return out
