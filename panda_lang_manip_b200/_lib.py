"""ctypes binding of libpanda_b200.so (C ABI: include/panda_b200.h).

The library is the product path; there is no CPU fallback.  Loading fails loudly if the shared object has not been
built (``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C panda_lang_manip_b200/csrc``).
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("PANDA_B200_LIB", os.path.join(CSRC, "libpanda_b200.so"))   # override: A/B builds of the same ABI

TASKS = {"reach": 0, "push": 1, "slide": 2, "pick_and_place": 3, "stack": 4, "flip": 5}
TASK_BARE = 6
CONTROL = {"ee": 0, "joints": 1}
REWARD = {"sparse": 0, "dense": 1}
PRECISION = {"f32": 0, "f64": 1}

SYMBOLS = [
    "pg_create", "pg_destroy", "pg_dims", "pg_reset", "pg_step", "pg_max_contacts", "pg_set_action_scale", "pg_step_host", "pg_host_pin", "pg_host_unpin", "pg_compute_reward", "pg_is_success",
    "pg_compute_reward_host", "pg_is_success_host", "pg_her_relabel", "pg_save_state", "pg_restore_state", "pg_remove_state", "pg_get_state", "pg_set_state",
    "pg_inverse_kinematics", "pg_get_ee_pose", "pg_create_bare", "pg_set_motors", "pg_get_motors", "pg_sim_step", "pg_inverse_kinematics_link", "pg_get_link_state",
    "pg_host_stage_allocations", "pg_set_task_params", "pg_set_substeps",
    "pg_render", "pg_debug_schedule", "pg_debug_timing", "pg_diverged", "pg_contact_overflows", "pg_stats", "pg_kernel_launches", "pg_last_error",
    "pg_motion_create", "pg_motion_destroy", "pg_motion_move", "pg_motion_gripper", "pg_motion_step",
]

_lib = None


class PandaB200Error(RuntimeError):
    pass


def build(jobs: int = 8) -> str:
    """Compile the CUDA extension in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    subprocess.run(["make", "-C", CSRC, f"-j{jobs}"], check=True, stdout=subprocess.DEVNULL)
    return LIB_PATH


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PandaB200Error(f"{LIB_PATH} is missing: build the CUDA extension first (make -C {CSRC}); there is no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    c_int, c_ll, c_ull, vp, cd = ctypes.c_int, ctypes.c_longlong, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_double
    pi = ctypes.POINTER(c_int)
    lib.pg_create.argtypes = [c_int, c_int, c_int, c_int, c_int, c_ull, c_ll, c_int, ctypes.POINTER(vp)]
    lib.pg_destroy.argtypes = [vp]
    lib.pg_dims.argtypes = [vp, pi, pi, pi, pi, pi]
    lib.pg_reset.argtypes = [vp] * 9
    lib.pg_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, c_int, vp, vp, vp]
    lib.pg_max_contacts.argtypes = [vp, pi]
    lib.pg_set_action_scale.argtypes = [vp, ctypes.c_double, ctypes.c_double]
    lib.pg_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, c_int]
    lib.pg_host_pin.argtypes = [vp, ctypes.c_size_t]
    lib.pg_host_unpin.argtypes = [vp]
    lib.pg_compute_reward.argtypes = [c_int, c_int, cd, vp, vp, vp, c_ll, c_int, vp]
    lib.pg_is_success.argtypes = [c_int, cd, vp, vp, vp, c_ll, c_int, vp]
    lib.pg_compute_reward_host.argtypes = [c_int, c_int, cd, vp, vp, vp, c_ll, c_int, c_int]
    lib.pg_is_success_host.argtypes = [c_int, cd, vp, vp, vp, c_ll, c_int, c_int]
    lib.pg_her_relabel.argtypes = [c_int, c_int, cd, vp, vp, c_ll, vp, vp, vp, vp, vp, c_ll, c_int, vp]
    lib.pg_save_state.argtypes = [vp, pi, vp]
    lib.pg_restore_state.argtypes = [vp, c_int, vp]
    lib.pg_remove_state.argtypes = [vp, c_int]
    lib.pg_get_state.argtypes = [vp, vp, vp]
    lib.pg_set_state.argtypes = [vp, vp, vp, vp]
    lib.pg_inverse_kinematics.argtypes = [vp, vp, vp, vp, vp]
    lib.pg_get_ee_pose.argtypes = [vp, vp, vp]
    lib.pg_create_bare.argtypes = [c_int, c_int, c_int, vp, c_int, vp, vp, vp, ctypes.POINTER(vp)]
    lib.pg_set_motors.argtypes = [vp, vp, vp, vp]
    lib.pg_get_motors.argtypes = [vp, vp, vp]
    lib.pg_sim_step.argtypes = [vp, c_int, vp]
    lib.pg_inverse_kinematics_link.argtypes = [vp, c_int, vp, vp, vp, vp]
    lib.pg_get_link_state.argtypes = [vp, c_int, vp, vp]
    lib.pg_host_stage_allocations.restype = c_ll
    lib.pg_set_task_params.argtypes = [vp, cd, vp, vp, vp, vp]
    lib.pg_set_substeps.argtypes = [vp, c_int]
    lib.pg_render.argtypes = [vp, c_int, c_int, vp, c_int, vp, vp, vp, vp, vp, vp]
    lib.pg_debug_schedule.argtypes = [vp, vp, vp]
    lib.pg_debug_timing.argtypes = [vp, vp]
    lib.pg_diverged.argtypes = [vp, ctypes.POINTER(ctypes.c_longlong)]
    lib.pg_contact_overflows.argtypes = [vp, ctypes.POINTER(ctypes.c_longlong)]
    lib.pg_stats.argtypes = [vp, ctypes.POINTER(ctypes.c_double)]
    lib.pg_motion_create.argtypes = [c_int, c_int, ctypes.POINTER(vp)]
    lib.pg_motion_destroy.argtypes = [vp]
    lib.pg_motion_move.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.pg_motion_gripper.argtypes = [vp, vp, cd, c_int, vp, vp]
    lib.pg_motion_step.argtypes = [vp] * 10
    lib.pg_kernel_launches.restype = c_ll
    lib.pg_last_error.restype = ctypes.c_char_p
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise PandaB200Error(f"libpanda_b200 error {rc}: {load().pg_last_error().decode()}")


def kernel_launches() -> int:
    return int(load().pg_kernel_launches())
