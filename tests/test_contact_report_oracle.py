"""Physical invariants of the contact report on the CPU oracle (tests/contact_report_util.py): normal forces that carry the bodies' weight,
friction on the cone while sliding, no contact in free fall.  The CUDA path is held to the same answers in tests/test_gpu_contact_report.py."""
import numpy as np

from tests.contact_kats import check
from tests.contact_report_util import invariants, oracle_rows
from tests.oracle_util import OracleEnv


class OracleRunner:
    def __init__(self, task):
        self.env = OracleEnv(task, "joints")

    def set(self, row):
        self.env.set_full_state(row)

    def step(self, action):
        self.env.step(np.asarray(action, np.float32))
        return oracle_rows(self.env)

    def close(self):
        self.env.close()


def test_contact_report_invariants_on_the_oracle():
    res = invariants(OracleRunner)
    for k, v in res.items():
        print(f"{k}: got {float(v[0]):.9g} want {float(v[1]):.9g} tol {v[2]:.2e}")
    check(res)
