"""The contact report (pybullet getContactPoints after a step, pg_step's contacts): row layout, the oracle's rows, and physical invariants
that any backend's report must satisfy on the scenes of tests/contact_kats.py."""
import ctypes

import numpy as np

from tests.contact_kats import DT, G, state_row
from tests.oracle_util import NOBJ, P, load_oracle

WORDS = 16
PLANE, TABLE, OBJ0, OBJ1, HAND, FINGER1, FINGER2 = 1, 2, 3, 4, 14, 15, 16
ROBOT = (HAND, FINGER1, FINGER2)
MAX_CONTACTS = {"reach": 10, "push": 10, "slide": 10, "pick_and_place": 10, "flip": 10, "stack": 22}


TABLE_RECT = {"slide": (-0.8, 0.6, -0.35, 0.35)}         # x0, x1, y0, y1 of the table top (z = 0) per task; the others use DEFAULT_TABLE
DEFAULT_TABLE = (-0.85, 0.25, -0.35, 0.35)
GROUND_Z = -0.4


def _plane_space(n):
    """btPlaneSpace1, as the oracle and the kernel compute the friction directions"""
    if abs(n[2]) > 0.7071067811865475244:
        a = n[1] * n[1] + n[2] * n[2]; k = 1.0 / np.sqrt(a)
        p = np.array([0.0, -n[2] * k, n[1] * k])
        return p, np.array([a * k, -n[0] * p[2], n[0] * p[1]])
    a = n[0] * n[0] + n[1] * n[1]; k = 1.0 / np.sqrt(a)
    p = np.array([-n[1] * k, n[0] * k, 0.0])
    return p, np.array([-n[2] * p[1], n[2] * p[0], a * k])


def oracle_rows(oe):
    """[n, 16] float64 report rows of the oracle env's last sub-step, in the layout, ids and collection order of the kernel's report.

    Built from the oracle's contact accessor po_get_contact: P(3) n(3) dist, robot link of A (>= 0) or -link - 100 of B, object of A
    (>= 0) or -object - 100 of B, and the three accumulated impulses (normal, friction along btPlaneSpace1(n)).  The accessor keeps one
    object per contact; the other end follows from the contact model: with no robot link and object a on side A, B is static (the table
    or the ground plane, by collect_contacts' rule) or, in a two-object scene, the other object.  A static contact is recognisable exactly:
    its normal is +z and its distance is the vertex height over the plane that rule picks."""
    lib = load_oracle()
    lib.po_get_contact.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    x0, x1, y0, y1 = TABLE_RECT.get(oe.task, DEFAULT_TABLE)
    two_objects = NOBJ[oe.task] == 2
    n = lib.po_last_num_contacts(oe.sim)
    rows = np.zeros((n, WORDS))
    g = np.zeros(12)
    for c in range(n):
        assert lib.po_get_contact(oe.sim, c, P(g)) == 0
        pos, nrm, dist, la, ob = g[0:3], g[3:6], g[6], int(g[7]), int(g[8])
        plane = 0.0 if (x0 <= pos[0] <= x1 and y0 <= pos[1] <= y1 and pos[2] > -0.05) else GROUND_Z
        static_id = TABLE if plane == 0.0 else PLANE
        if la >= 0:                                   # robot link on side A: against the table, or against object -ob - 100
            ia, ib = la + 6, TABLE if ob == -1 else 3 + (-ob - 100)
        elif la <= -100:                              # object ob on side A, robot link on side B
            ia, ib = 3 + ob, -la - 100 + 6
        elif two_objects and not (nrm[0] == 0.0 and nrm[1] == 0.0 and nrm[2] == 1.0 and dist == pos[2] - plane):
            ia, ib = 3 + ob, 3 + (1 - ob)             # object against object
        else:
            ia, ib = 3 + ob, static_id
        t1, t2 = _plane_space(nrm)
        rows[c, 0:6] = g[0:6]
        rows[c, 6], rows[c, 7], rows[c, 11] = g[9] / DT, g[10] / DT, g[11] / DT
        rows[c, 8:11], rows[c, 12:15] = t1, t2
        rows[c, 15] = ia + 32 * ib
    return rows


def ids(rows):
    code = np.asarray(rows)[:, 15].astype(np.int64)
    return code % 32, code // 32


def force_on_a(rows):
    """[n, 3] total contact force on body A of each row: normal + both lateral friction forces."""
    r = np.asarray(rows, np.float64)
    return r[:, 3:6] * r[:, 6:7] + r[:, 8:11] * r[:, 7:8] + r[:, 12:15] * r[:, 11:12]


def pair(rows, x, y):
    """rows between bodies x and y (either order) and the sign that turns the force on A into the force on x."""
    a, b = ids(rows)
    m = ((a == x) & (b == y)) | ((a == y) & (b == x))
    return np.asarray(rows)[m], np.where(a[m] == x, 1.0, -1.0)


def invariants(make_runner):
    """make_runner(task) -> object with .set(state_row), .step(action) -> report rows [n, 16] of that step, .close().
    Returns {name: (got, want, tol)} as tests/contact_kats.check takes it."""
    out = {}
    zero7, zero8 = np.zeros(7, np.float32), np.zeros(8, np.float32)
    r = make_runner("push")
    # a 1 kg cube resting on the table: the table carries m g, nothing pulls sideways
    r.set(state_row("push", [([0.1, 0.05, 0.02], [0, 0, 0])], [0, 0, 0.02]))
    for _ in range(25):
        rows = r.step(zero7)
    on_table, _ = pair(rows, OBJ0, TABLE)
    out["resting_cube_table_contacts"] = (len(on_table), 4, 0)
    out["resting_cube_normal_force_sum"] = (on_table[:, 6].sum(), 1.0 * G, 0.01 * G)
    out["resting_cube_max_friction"] = (float(np.abs(on_table[:, [7, 11]]).max()), 0.0, 0.01)
    # free fall (the cube 5 cm up, the gripper 20 cm above the table): nothing touches anything
    r.set(state_row("push", [([0.1, 0.05, 0.07], [0, 0, 0])], [0, 0, 0.02]))
    out["free_fall_contacts"] = (len(r.step(zero7)), 0, 0)
    # a cube sliding at 0.5 m/s along +x (mu = 0.5 x 0.5): every contact is on the friction cone, the force points against the motion
    r.set(state_row("push", [([-0.1, 0.0, 0.02], [0.5, 0, 0])], [0, 0, 0.02]))
    rows = r.step(zero7)
    sliding, sg = pair(rows, OBJ0, TABLE)
    fric = np.hypot(sliding[:, 7], sliding[:, 11])
    f_obj = (sliding[:, 8:11] * sliding[:, 7:8] + sliding[:, 12:15] * sliding[:, 11:12]) * sg[:, None]
    out["sliding_cube_table_contacts"] = (len(sliding), 4, 0)
    out["sliding_cube_friction_on_the_cone"] = (float(np.abs(fric / (0.25 * sliding[:, 6]) - 1).max()), 0.0, 1e-6)
    out["sliding_cube_friction_against_the_motion"] = (float((-f_obj[:, 0] / np.linalg.norm(f_obj, axis=1)).min()), 1.0, 1e-6)
    r.close()
    # Stack, the 1 kg cube resting on the 2 kg one, aligned and turned: the lower cube carries 1 kg, the table 3 kg
    r = make_runner("stack")
    for name, ang, off in (("aligned", 0.0, 0.0), ("turned_20_deg", np.radians(20.0), 0.0005), ("turned_45_deg", np.pi / 4, 0.002)):
        quat = [0, 0, np.sin(ang / 2), np.cos(ang / 2)]
        r.set(state_row("stack", [([0.1, 0.05, 0.02], [0, 0, 0]), ([0.1 + off, 0.05 + off / 2, 0.06], [0, 0, 0], quat)], [0.1, 0.05, 0.02, 0.1, 0.05, 0.06]))
        for _ in range(25):
            rows = r.step(zero8)
        between, _ = pair(rows, OBJ1, OBJ0)
        lower, _ = pair(rows, OBJ0, TABLE)
        out[f"stack_{name}_upper_on_lower_normal_force_sum"] = (between[:, 6].sum(), 1.0 * G, 0.01 * G)
        out[f"stack_{name}_lower_on_table_normal_force_sum"] = (lower[:, 6].sum(), 3.0 * G, 0.03 * G)
        out[f"stack_{name}_upper_on_table_contacts"] = (len(pair(rows, OBJ1, TABLE)[0]), 0, 0)
    r.close()
    # PickAndPlace: the cube held between the closing fingers 18 cm above the table: the robot holds m g, the table holds nothing
    r = make_runner("pick_and_place")
    row = state_row("pick_and_place", [([0.0384, 0.0, 0.1974], [0, 0, 0])], [0, 0, 0.1])
    row[7] = row[8] = 0.0205
    r.set(row)
    act = zero8.copy(); act[7] = -1.0
    for _ in range(30):
        rows = r.step(act)
    a, b = ids(rows)
    held = np.isin(a, ROBOT) & (b == OBJ0) | (a == OBJ0) & np.isin(b, ROBOT)
    fz = (force_on_a(rows)[:, 2] * np.where(a == OBJ0, 1.0, -1.0))[held].sum()
    out["grasped_cube_finger_contacts"] = (int(held.sum()) > 0, True, 0)
    out["grasped_cube_vertical_robot_force"] = (fz, 1.0 * G, 0.05 * G)
    out["grasped_cube_table_contacts"] = (len(pair(rows, OBJ0, TABLE)[0]), 0, 0)
    r.close()
    return out
