"""Argument validation of the C ABI: the error code and pg_last_error() text of every rejected call.

Each call here is rejected before the library makes any CUDA call, so this runs without a device.  Only NULL or small dummy host
pointers are passed, and never a handle other than NULL."""
import ctypes
import os
import re

import pytest

from panda_lang_manip_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PG_OK, PG_ERR_ARG = 0, -1
_BUF = (ctypes.c_double * 64)()         # dummy host storage: never read on the rejected paths
P = ctypes.addressof(_BUF)


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def _rejected(lib, rc, text):
    assert (rc, lib.pg_last_error().decode()) == (PG_ERR_ARG, text)


def _int():
    return ctypes.byref(ctypes.c_int())


def _ll():
    return ctypes.byref(ctypes.c_longlong())


# entry point -> (arguments after the NULL handle, error text)
NULL_HANDLE = {
    "pg_dims": (lambda: [_int() for _ in range(5)], "pg_dims: NULL handle"),
    "pg_reset": (lambda: [P] * 7 + [None], "pg_reset: NULL handle"),
    "pg_set_task_params": (lambda: [0.05] + [P] * 4, "pg_set_task_params: needs a task handle"),
    "pg_set_substeps": (lambda: [20], "pg_set_substeps: needs a task handle (bare worlds pass the count to pg_sim_step)"),
    "pg_step": (lambda: [P] * 8 + [1, P, P, None], "pg_step: NULL handle or actions"),
    "pg_max_contacts": (lambda: [_int()], "pg_max_contacts: NULL argument"),
    "pg_set_action_scale": (lambda: [0.05, 0.2], "pg_set_action_scale: bad argument"),
    "pg_step_host": (lambda: [P] * 7 + [1], "pg_step_host: NULL handle or actions"),
    "pg_save_state": (lambda: [_int(), None], "pg_save_state: NULL argument"),
    "pg_restore_state": (lambda: [0, None], "pg_restore_state: NULL handle"),
    "pg_remove_state": (lambda: [0], "pg_remove_state: NULL handle"),
    "pg_get_state": (lambda: [P, None], "pg_get_state: NULL argument"),
    "pg_set_state": (lambda: [P, P, None], "pg_set_state: NULL argument"),
    "pg_inverse_kinematics": (lambda: [P, P, P, None], "pg_inverse_kinematics: NULL argument"),
    "pg_inverse_kinematics_link": (lambda: [6, P, P, P, None], "pg_inverse_kinematics_link: NULL argument"),
    "pg_get_link_state": (lambda: [6, P, None], "pg_get_link_state: NULL argument"),
    "pg_set_motors": (lambda: [P, P, None], "pg_set_motors: NULL argument"),
    "pg_get_motors": (lambda: [P, None], "pg_get_motors: NULL argument"),
    "pg_sim_step": (lambda: [1, None], "pg_sim_step: bad argument"),
    "pg_render": (lambda: [8, 8, P, 1, P, P, P, P, P, None], "pg_render: bad argument"),
    "pg_get_ee_pose": (lambda: [P, None], "pg_get_ee_pose: NULL argument"),
    "pg_debug_schedule": (lambda: [P, P], "pg_debug_schedule: NULL argument"),
    "pg_debug_timing": (lambda: [P], "pg_debug_timing: NULL argument"),
    "pg_diverged": (lambda: [_ll()], "pg_diverged: NULL argument"),
    "pg_contact_overflows": (lambda: [_ll()], "pg_contact_overflows: NULL argument"),
    "pg_stats": (lambda: [_BUF], "pg_stats: NULL argument"),
}


def test_every_handle_entry_point_is_covered():
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "panda_b200.h")).read(), flags=re.S)
    takes_handle = set(re.findall(r"\b(pg_[a-z_0-9]+)\s*\(\s*(?:const\s+)?pg_env\s*\*\s*\w", text))
    assert takes_handle == set(NULL_HANDLE) | {"pg_destroy"}


@pytest.mark.parametrize("name", sorted(NULL_HANDLE))
def test_null_handle(lib, name):
    args, text = NULL_HANDLE[name]
    _rejected(lib, getattr(lib, name)(None, *args()), text)


def test_destroy_null_handle(lib):
    assert lib.pg_destroy(None) == PG_OK


# pg_create(task, control_type, reward_type, num_envs, device, seed, env_id_offset, precision, out)
CREATE_OK = dict(task=0, control_type=0, reward_type=0, num_envs=4, device=0, seed=0, env_id_offset=0, precision=0)


def test_create_out_null(lib):
    _rejected(lib, lib.pg_create(*CREATE_OK.values(), None), "pg_create: out is NULL")


@pytest.mark.parametrize("field,value", [("task", -1), ("task", 6), ("control_type", -1), ("control_type", 2), ("reward_type", -1),
                                         ("reward_type", 2), ("num_envs", 0), ("num_envs", -4), ("precision", -1), ("precision", 2)])
def test_create_bad_argument(lib, field, value):
    h = ctypes.c_void_p()
    _rejected(lib, lib.pg_create(*dict(CREATE_OK, **{field: value}).values(), ctypes.byref(h)),
              "pg_create: bad task / control_type / reward_type / num_envs / precision")
    assert h.value is None


BODY = [0.0, 0.02, 0.02, 0.02, 1.0, 0.5, 0.0, 0.0, 0.42, 0.0, 0.0, 0.0, 1.0]      # shape hx hy hz mass mu pos3 quat4
BARE_BAD = "pg_create_bare: bad num_envs / precision / n_bodies (at most 2 free bodies)"
BODY_BAD = "pg_create_bare: body rows are [shape(0 box,1 z-cylinder) hx hy hz mass(>0) mu pos3 quat4]"


def _create_bare(lib, rows, n_bodies=None, num_envs=4, precision=0, out=True):
    a = (ctypes.c_double * max(13 * len(rows), 1))(*[x for r in rows for x in r])
    h = ctypes.c_void_p()
    rc = lib.pg_create_bare(num_envs, 0, precision, None, len(rows) if n_bodies is None else n_bodies, a if rows else None, None, None,
                            ctypes.byref(h) if out else None)
    assert h.value is None
    return rc


def test_create_bare_out_null(lib):
    _rejected(lib, _create_bare(lib, [BODY], out=False), "pg_create_bare: out is NULL")


@pytest.mark.parametrize("kw", [dict(rows=[BODY] * 3), dict(rows=[BODY], n_bodies=-1), dict(rows=[], n_bodies=1), dict(rows=[BODY], num_envs=0),
                                dict(rows=[BODY], precision=2)])
def test_create_bare_bad_argument(lib, kw):
    _rejected(lib, _create_bare(lib, **kw), BARE_BAD)


@pytest.mark.parametrize("col,value", [(0, 2.0), (1, 0.0), (2, -0.02), (3, float("nan")), (4, 0.0), (5, -0.1)])
def test_create_bare_bad_body_row(lib, col, value):
    bad = list(BODY)
    bad[col] = value
    _rejected(lib, _create_bare(lib, [BODY, bad]), BODY_BAD)


def test_create_bare_zero_quaternion(lib):
    _rejected(lib, _create_bare(lib, [BODY, BODY[:9] + [0.0] * 4]), "pg_create_bare: zero quaternion")


# goal-array entry points (all take a threshold, pg_her_relabel also a row pitch): name -> (takes reward_type, error text)
REWARD = {
    "pg_compute_reward": (True, "pg_compute_reward: bad argument"),
    "pg_is_success": (False, "pg_is_success: bad argument"),
    "pg_compute_reward_host": (True, "pg_compute_reward_host: bad argument"),
    "pg_is_success_host": (False, "pg_is_success_host: bad argument"),
    "pg_her_relabel": (True, "pg_her_relabel: bad argument"),
}


def _arrays(name):
    """The arrays that must not be NULL: ag, dg, out -- or next_ag, dg, src, goal_src, dg_out, reward for HER."""
    return 6 if name.startswith("pg_her") else 3


def _goal_call(lib, name, task=0, reward_type=0, threshold=0.05, arrays=None, m=4, pitch=3):
    takes_rt, _ = REWARD[name]
    a = [P] * _arrays(name) if arrays is None else arrays
    args = [task] + ([reward_type] if takes_rt else []) + [threshold]
    if name.startswith("pg_her"):
        args += a[:2] + [pitch] + a[2:5] + [None, a[5]]      # achieved_goal_out may be NULL
    else:
        args += a
    return getattr(lib, name)(*args, m, 0, 0 if "_host" in name else None)


@pytest.mark.parametrize("name", sorted(REWARD))
def test_goal_entry_points(lib, name):
    takes_rt, text = REWARD[name]
    for task in (-1, 6):
        _rejected(lib, _goal_call(lib, name, task=task), text)
    if takes_rt:
        for rt in (-1, 2):
            _rejected(lib, _goal_call(lib, name, reward_type=rt), text)
    for k in range(_arrays(name)):
        a = [P] * _arrays(name)
        a[k] = None
        _rejected(lib, _goal_call(lib, name, arrays=a), text)
    for thr in (-0.05, float("nan")):
        _rejected(lib, _goal_call(lib, name, threshold=thr), text)
    _rejected(lib, _goal_call(lib, name, m=-1), text)
    if name == "pg_her_relabel":
        for task, pitch in ((0, 2), (4, 5), (5, 3)):
            _rejected(lib, _goal_call(lib, name, task=task, pitch=pitch),
                      "pg_her_relabel: the row pitch is smaller than the goal dimension")
    assert _goal_call(lib, name, arrays=[None] * _arrays(name), m=0) == PG_OK
