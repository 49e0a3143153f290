"""The motion primitives without a GPU.

1. Their per-env math (csrc/panda_motion.cuh, compiled for the host by tests/hostcheck/motion.cpp) against the facade's own static
   helpers ``Panda.get_waypoint`` / ``Panda.get_ori`` (robots/panda_cartesian.py): way-point counts equal, way-point positions
   bit-identical, Slerp orientations equal to scipy's as rotations.
2. The argument errors of the motion entry points of the C ABI, which are rejected before any CUDA call."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial.transform import Rotation as R

from panda_lang_manip_b200 import _lib
from panda_lang_manip_b200.panda_gym.envs.robots.panda_cartesian import Panda

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DP = ctypes.POINTER(ctypes.c_double)


@pytest.fixture(scope="module")
def hc():
    """TEST-ONLY host build of panda_motion.cuh (tests/hostcheck/motion.cpp), unfused as numpy computes."""
    d = os.path.join(ROOT, "tests", "hostcheck")
    so = os.path.join(d, "libhostcheck_motion.so")
    srcs = [os.path.join(d, "motion.cpp")] + [os.path.join(ROOT, "panda_lang_manip_b200", "csrc", f) for f in ("panda_motion.cuh", "panda_dyn.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, srcs[0]], check=True)
    lib = ctypes.CDLL(so)
    lib.hc_waypoint_count.argtypes = [DP, DP]
    lib.hc_waypoints.argtypes = [DP, DP, DP]
    lib.hc_slerp.argtypes = [DP, DP, ctypes.c_int, ctypes.c_int, DP]
    return lib


def _p(a):
    return np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(DP)


def _facade(start, goal):
    """Panda.move's way-point generator and count (panda_cartesian.py:50-53)."""
    if np.linalg.norm(goal - start) < 0.03:
        return Panda.get_waypoint(start, goal, 0.015, num_steps=20)
    return Panda.get_waypoint(start, goal, 0.015)


def _kernel_count(hc, start, goal):
    s, g = np.ascontiguousarray(start, dtype=np.float64), np.ascontiguousarray(goal, dtype=np.float64)
    return hc.hc_waypoint_count(_p(s), _p(g))


def test_waypoint_count_random_distances(hc):
    rng = np.random.default_rng(0)
    start = rng.uniform([-0.3, -0.3, 0.0], [0.3, 0.3, 0.3], (10000, 3))
    goal = start + rng.normal(size=(10000, 3)) * rng.uniform(0.0, 0.4, (10000, 1))
    for s, g in zip(start, goal):
        assert _kernel_count(hc, s, g) == _facade(s, g)[1], (s, g)


def _edge_distances():
    """Distances on the count's decision boundaries: exact multiples of 0.015, 0.015 k + 1e-3 and 0.03, each +- 1 ulp."""
    out = []
    for k in range(1, 41):
        for x in (0.015 * k, 0.015 * k + 1e-3):
            out += [np.nextafter(x, 0.0), x, np.nextafter(x, 1.0)]
    out += [np.nextafter(0.03, 0.0), 0.03, np.nextafter(0.03, 1.0), 0.0]
    return out


def test_waypoint_count_edges(hc):
    """Along one axis the norm is the distance exactly, so the edge values reach the count as written."""
    start = np.array([0.1, -0.2, 0.05])
    counts = set()
    for x in _edge_distances():
        for axis in range(3):
            g = np.zeros(3); g[axis] = x
            s0 = np.zeros(3)
            want = _facade(s0, g)[1]
            assert _kernel_count(hc, s0, g) == want, (x, axis)
            counts.add(want)
        assert _kernel_count(hc, start, start + np.array([x, 0.0, 0.0])) == _facade(start, start + np.array([x, 0.0, 0.0]))[1], x
    assert 20 in counts and len(counts) >= 40


def test_waypoint_positions_bit_identical(hc):
    rng = np.random.default_rng(1)
    for t in range(500):
        s = rng.uniform([-0.3, -0.3, 0.0], [0.3, 0.3, 0.3])
        g = s + rng.normal(size=3) * rng.uniform(0.0, 0.3) if t % 5 else s + np.array([0.015 * (t % 23), 0.0, 0.0])
        fn, n = _facade(s, g)
        out = np.zeros((n, 3))
        hc.hc_waypoints(_p(s), _p(g), out.ctypes.data_as(DP))
        want = np.array([fn(i) for i in range(1, n + 1)])
        assert out.tobytes() == want.tobytes(), (t, s, g)


def _angle(qa, qb):
    return float((R.from_quat(qa).inv() * R.from_quat(qb)).magnitude())


def _slerp_cases():
    rng = np.random.default_rng(2)
    cases = [(R.random(random_state=rng).as_quat(), R.random(random_state=rng).as_quat()) for _ in range(300)]
    for _ in range(200):                                        # near-antipodal: q1 = q0 turned by pi - eps
        q0 = R.random(random_state=rng)
        axis = rng.normal(size=3); axis /= np.linalg.norm(axis)
        eps = 10.0 ** rng.uniform(-9, -3)
        cases.append((q0.as_quat(), (q0 * R.from_rotvec(axis * (np.pi - eps))).as_quat()))
    for _ in range(50):                                         # nearly equal: the small-angle series
        q0 = R.random(random_state=rng)
        cases.append((q0.as_quat(), (q0 * R.from_rotvec(rng.normal(size=3) * 1e-5)).as_quat()))
    return cases, rng


def test_slerp_matches_scipy(hc):
    """The kernel's orientation targets against scipy's Slerp([1, K], [q0, q1]) as the facade builds it, 1e-12 rad as rotations.  The
    facade's get_ori returns Euler angles, so the same Slerp is also evaluated before that conversion."""
    from scipy.spatial.transform import Slerp
    cases, rng = _slerp_cases()
    worst, worst_ori = 0.0, 0.0
    for j, (q0, q1) in enumerate(cases):
        n = int(rng.integers(1, 60))
        e0, e1 = R.from_quat(q0).as_euler("xyz", degrees=True), R.from_quat(q1).as_euler("xyz", degrees=True)
        ori = Panda.get_ori(e0, e1, n)
        K = max(n, 2)
        sl = Slerp([1, K], R.from_quat([q0, q1]))
        for i in sorted({0, 1, 2, n // 2, n, n + 1, int(rng.integers(1, n + 1))}):
            out = np.zeros(4)
            hc.hc_slerp(_p(q0), _p(q1), n, i, out.ctypes.data_as(DP))
            worst = max(worst, _angle(out, sl(min(max(i, 1), K)).as_quat()))
            worst_ori = max(worst_ori, _angle(out, R.from_euler("xyz", ori(i), degrees=True).as_quat()))
    print(f"slerp: worst {worst:.2e} rad against scipy's Slerp, {worst_ori:.2e} rad against Panda.get_ori (Euler round trip included)")
    assert worst < 1e-12
    assert worst_ori < 1e-9


# ---- argument errors of the C ABI (no device needed)
PG_OK, PG_ERR_ARG = 0, -1
_BUF = (ctypes.c_double * 16)()
P = ctypes.addressof(_BUF)             # dummy non-NULL pointer: never dereferenced on the rejected paths


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def _rejected(lib, rc, text):
    assert (rc, lib.pg_last_error().decode()) == (PG_ERR_ARG, text)


def test_motion_create_and_destroy_arguments(lib):
    h = ctypes.c_void_p()
    _rejected(lib, lib.pg_motion_create(4, 0, None), "pg_motion_create: out is NULL")
    for n in (0, -3):
        _rejected(lib, lib.pg_motion_create(n, 0, ctypes.byref(h)), "pg_motion_create: num_envs must be > 0")
        assert h.value is None
    assert lib.pg_motion_destroy(None) == PG_OK


@pytest.mark.parametrize("plan,env", [(None, None), (None, P), (P, None)], ids=["None-None", "None-ptr", "ptr-None"])   # P is an address: not an id
def test_motion_null_plan_or_env(lib, plan, env):
    _rejected(lib, lib.pg_motion_move(plan, env, P, P, None, None), "pg_motion_move: NULL plan or env")
    _rejected(lib, lib.pg_motion_gripper(plan, env, -1.0, 30, None, None), "pg_motion_gripper: NULL plan or env")
    _rejected(lib, lib.pg_motion_step(plan, env, P, P, P, P, P, P, P, None), "pg_motion_step: NULL plan or env")


def test_motion_gripper_negative_steps(lib):
    for plan, env in ((None, None), (P, P)):
        _rejected(lib, lib.pg_motion_gripper(plan, env, 1.0, -1, None, None), "pg_motion_gripper: steps must be >= 0")
