"""The step kernel's contact-report decode (contact_report_row in csrc/panda_contact.cuh, compiled for the host by tests/hostcheck/contact_report.cpp) against
the oracle's report, fp64, without a GPU: the gripper is driven down onto the objects and the table, then three teacher-forced steps
(the kernel math continues from the oracle's state) compare every row.  Counts and body ids must be identical, forces agree to 1e-4 N
(the two fp64 formulations agree to ~1e-12 until a sweep-count exit falls differently)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests.contact_report_util import MAX_CONTACTS, WORDS, ids, oracle_rows
from tests.oracle_util import GOAL_DIM, NOBJ, OracleEnv, P
from tests.test_hostcheck import BASE, TASK_ID

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hc_report():
    """TEST-ONLY host build of the kernel math with the report decode (tests/hostcheck/contact_report.cpp)."""
    d = os.path.join(ROOT, "tests", "hostcheck")
    so = os.path.join(d, "libhostcheck_contact_report.so")
    srcs = [os.path.join(d, "contact_report.cpp")] + [os.path.join(ROOT, "panda_lang_manip_b200", "csrc", f) for f in
                                                      ("panda_dyn.cuh", "panda_contact.cuh", "panda_env.cuh", "panda_model.h", "panda_scene.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, srcs[0]], check=True)
    lib = ctypes.CDLL(so)
    lib.hc_env_step_contacts.argtypes = [ctypes.c_int] * 3 + [ctypes.c_void_p] * 5
    return lib


def _hc_step(hc, task, oe, a):
    nobj, G = NOBJ[task], GOAL_DIM[task]
    fs = oe.full_state()
    st = np.zeros(50); st[:18 + 13 * nobj] = fs[:18 + 13 * nobj]; st[44:44 + G] = fs[18 + 13 * nobj:]
    rows, n = np.zeros((MAX_CONTACTS[task], WORDS)), np.zeros(1, np.int32)
    hc.hc_env_step_contacts(1, TASK_ID[task], 0, P(BASE), P(st), P(a), P(rows), P(n))
    return rows[:n[0]]


@pytest.mark.parametrize("task", ["push", "pick_and_place", "stack"])
def test_kernel_contact_report_matches_the_oracle_fp64(hc_report, task):
    worst, seen_ids = 0.0, set()
    for seed in range(4):
        rng = np.random.default_rng(seed)
        goal = np.zeros(6); goal[:3] = rng.uniform([-0.15, -0.15, 0.0], [0.15, 0.15, 0.2])
        objpos = np.array([0.04 + 0.01 * seed, 0.005 * seed, 0.02, 0.04 + 0.01 * seed, 0.0, 0.06])      # under the gripper
        oe = OracleEnv(task, "ee")
        oe.reset(goal, objpos)

        def act(t):
            a = np.zeros(oe.action_dim, np.float32); a[2] = -1.0; a[0] = 0.3 * np.sin(0.7 * t + seed)
            if oe.action_dim > 3:
                a[3] = -1.0 if t > 4 else 1.0
            return a
        for t in range(4 + seed):                 # free-running approach
            oe.step(act(t))
        for t in range(4 + seed, 7 + seed):       # three teacher-forced steps
            got = _hc_step(hc_report, task, oe, act(t))
            oe.step(act(t))
            want = oracle_rows(oe)
            assert len(got) == len(want), (seed, t, len(got), len(want))
            assert np.array_equal(got[:, 15], want[:, 15]), (seed, t, got[:, 15], want[:, 15])
            if len(got):
                worst = max(worst, float(np.abs(got[:, [6, 7, 11]] - want[:, [6, 7, 11]]).max()))
                assert np.abs(got[:, :6] - want[:, :6]).max() < 1e-9 and np.abs(got[:, [8, 9, 10, 12, 13, 14]] - want[:, [8, 9, 10, 12, 13, 14]]).max() < 1e-9
                a, b = ids(got)
                seen_ids |= set(zip(a.tolist(), b.tolist()))
        oe.close()
    print(task, "worst force difference", worst, "N; body pairs", sorted(seen_ids))
    assert worst < 1e-4, worst
    assert any(a in (14, 15, 16) or b in (14, 15, 16) for a, b in seen_ids), seen_ids      # the gripper did touch something
