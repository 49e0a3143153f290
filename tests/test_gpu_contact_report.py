"""The contact report (PandaVecEnv(contact_report=True).contacts(), pg_step's contacts) on the GPU: the physical invariants of
tests/contact_report_util.py, per-step parity with the oracle's report, no effect on any other output, invisibility of the scheduling,
and the auto-reset rule (the report describes the finished step)."""
import numpy as np
import pytest

from tests.contact_kats import check
from tests.contact_report_util import MAX_CONTACTS, ROBOT, WORDS, force_on_a, ids, invariants, oracle_rows
from tests.oracle_util import GOAL_DIM, NOBJ, OracleEnv

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _rows(env, i):
    c = env.contacts()
    return env._contacts[i, :int(c["count"][i])].double().cpu().numpy()


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_contact_report_invariants_on_the_gpu(precision):
    import panda_lang_manip_b200 as p

    class GpuRunner:
        def __init__(self, task):
            self.env = p.PandaVecEnv(task, 1, control_type="joints", precision=precision, auto_reset=False, contact_report=True)

        def set(self, row):
            st = self.env.get_state().cpu().numpy()
            st[0, :-1] = row
            self.env.set_state(torch.from_numpy(st))

        def step(self, action):
            self.env.step(torch.from_numpy(np.asarray(action, np.float32)[None]).cuda())
            return _rows(self.env, 0)

        def close(self):
            self.env.close()

    res = invariants(GpuRunner)
    for k, v in res.items():
        print(f"{precision} {k}: got {float(v[0]):.9g} want {float(v[1]):.9g} tol {v[2]:.2e}")
    check(res)


def _pair_forces(rows):
    """{(low id, high id): summed contact force on the low-id body}"""
    a, b = ids(rows)
    f = force_on_a(rows)
    out = {}
    for k in range(len(rows)):
        lo, hi, s = (a[k], b[k], 1.0) if a[k] < b[k] else (b[k], a[k], -1.0)
        out[(lo, hi)] = out.get((lo, hi), 0.0) + s * f[k]
    return out


def _net_forces(rows):
    """{object id: total contact force on the object}"""
    a, b = ids(rows)
    f = force_on_a(rows)
    return {o: f[a == o].sum(axis=0) - f[b == o].sum(axis=0) for o in (3, 4) if ((a == o) | (b == o)).any()}


@pytest.mark.parametrize("task", ["push", "pick_and_place", "stack"])
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_contact_report_per_step_parity(task, precision):
    """Teacher-forced, 8 envs x 25 steps, the grippers driven down on to objects placed under them: f64 reports match the oracle's in
    every env-step (counts, ids; forces to 1e-3 N); f32 reports have the oracle's counts and ids in >= 99 % of env-steps.  f32 forces are
    printed, not asserted: while the fingers squeeze a cube, or a cube presses on the other, the split between opposing contacts is what a
    50-sweep PGS determines least, and f32 solves of the same state differ from the fp64 oracle by more than 1 % + 0.05 N there (B200:
    per body pair up to 7.3 x that bar on PickAndPlace, net force on the two Stack cubes 2.4 x; Push within it)."""
    import panda_lang_manip_b200 as p
    n, steps, G, nobj = 8, 25, GOAL_DIM[task], NOBJ[task]
    rng = np.random.default_rng(11)
    goals = np.zeros((n, 6)); goals[:, :3] = rng.uniform([-0.15, -0.15, 0.02], [0.15, 0.15, 0.2], (n, 3))
    objs = np.zeros((n, 6))
    objs[:, :2] = np.array([0.04, 0.0]) + rng.uniform(-0.03, 0.03, (n, 2)); objs[:, 2] = 0.02
    objs[:, 3:5] = objs[:, :2] + rng.uniform(-0.01, 0.01, (n, 2)); objs[:, 5] = 0.06
    env = p.PandaVecEnv(task, n, control_type="ee", precision=precision, auto_reset=False, contact_report=True)
    env.reset(goals=goals[:, :G], object_positions=objs[:, :3 * nobj])
    oracles = [OracleEnv(task, "ee") for _ in range(n)]
    for i, oe in enumerate(oracles):
        oe.reset(goals[i], objs[i])
    A = env.action_dim
    same = total = robot_steps = 0
    worst_f64, worst_rel, worst_obj, worst_net = 0.0, 0.0, 0.0, 0.0
    for t in range(steps):
        a = rng.uniform(-0.3, 0.3, (n, A)).astype(np.float32); a[:, 2] = -1.0
        if A > 3:
            a[:, 3] = np.where(t > 6, -1.0, 1.0)
        env.step(torch.from_numpy(a).cuda())
        assert int(env.contacts()["count"].max()) <= MAX_CONTACTS[task]
        st = env.get_state().cpu().numpy()
        for i, oe in enumerate(oracles):
            oe.step(a[i])
            got, want = _rows(env, i), oracle_rows(oe)
            total += 1
            ok = len(got) == len(want) and np.array_equal(got[:, 15], want[:, 15])
            robot_steps += int(np.isin(ids(want)[0], ROBOT).any() or np.isin(ids(want)[1], ROBOT).any())
            if precision == "f64":
                assert ok, (t, i, got[:, 15], want[:, 15])
                if len(got):
                    worst_f64 = max(worst_f64, float(np.abs(got[:, [6, 7, 11]] - want[:, [6, 7, 11]]).max()))
            elif ok:
                same += 1
                fg, fw = _pair_forces(got), _pair_forces(want)
                for k in fw:
                    err = float(np.linalg.norm(fg[k] - fw[k]))
                    worst_rel = max(worst_rel, err / (0.01 * np.linalg.norm(fw[k]) + 0.05))
                ng, nw = _net_forces(got), _net_forces(want)
                for k in nw:
                    worst_obj = max(worst_obj, float(np.linalg.norm(ng[k] - nw[k])) / (0.01 * np.linalg.norm(nw[k]) + 0.05))
                tg, tw = sum(ng.values(), np.zeros(3)), sum(nw.values(), np.zeros(3))
                worst_net = max(worst_net, float(np.linalg.norm(tg - tw)) / (0.01 * np.linalg.norm(tw) + 0.05))
            # teacher forcing: continue from the oracle's state
            q, qd = oe.joints()
            st[i, :9], st[i, 9:18] = q, qd
            for o in range(nobj):
                st[i, 18 + 13 * o:18 + 13 * o + 13] = oe.object_state(o)
        env.set_state(torch.from_numpy(st))
    for oe in oracles:
        oe.close()
    env.close()
    print(f"{task} {precision}: env-steps {total}, with robot contacts {robot_steps}; worst f64 force difference {worst_f64:.3e} N; "
          f"f32 same counts and ids {same}/{total}, worst error / (1 % + 0.05 N): net force on the objects {worst_net:.3f}, per object {worst_obj:.3f}, body-pair sum {worst_rel:.3f}")
    assert robot_steps > 0
    if precision == "f64":
        assert worst_f64 < 1e-3, worst_f64
    else:
        assert same >= 0.99 * total, (same, total)


@pytest.mark.parametrize("task,n", [("push", 300), ("stack", 5000), ("pick_and_place", 5000)])
def test_report_changes_no_other_output(task, n):
    """A twin env without the report: observations, rewards, flags and the raw state are bit-identical (small batches: the tiled
    one-launch path; >= 4096 envs: sorted, segmented launches), with auto-reset on."""
    import panda_lang_manip_b200 as p
    on = p.PandaVecEnv(task, n, seed=5, contact_report=True)
    off = p.PandaVecEnv(task, n, seed=5)
    g = torch.Generator(device="cuda").manual_seed(2)
    for t in range(60):
        a = torch.rand((n, on.action_dim), device="cuda", generator=g) * 2 - 1
        a[:, 2] = -a[:, 2].abs()
        o1, r1, te1, tr1, _ = on.step(a)
        o2, r2, te2, tr2, _ = off.step(a)
        for k in o1:
            assert torch.equal(o1[k], o2[k]), (t, k)
        assert torch.equal(r1, r2) and torch.equal(te1, te2) and torch.equal(tr1, tr2)
    assert torch.equal(on.get_state(), off.get_state())
    assert int(on.contacts()["count"].sum()) > 0
    on.close(); off.close()


@pytest.mark.parametrize("task,ctrl", [("push", "ee"), ("stack", "joints")])
def test_report_scheduling_is_invisible(task, ctrl):
    """The report of a 512-env window of a 16,684-env batch (re-sorted, segmented launches in env groups) equals, bit for bit, that of
    the same envs stepped as a 512-env batch (identity map, one launch)."""
    import panda_lang_manip_b200 as p
    n, k0, k = 16384 + 300, 9000, 512
    big = p.PandaVecEnv(task, n, control_type=ctrl, seed=3, contact_report=True)
    small = p.PandaVecEnv(task, k, control_type=ctrl, seed=3, env_id_offset=k0, contact_report=True)
    g = torch.Generator(device="cuda").manual_seed(1)
    C = MAX_CONTACTS[task]
    touched = 0
    for t in range(12):
        a = torch.rand((n, big.action_dim), device="cuda", generator=g) * 2 - 1
        a[:, 2] = -a[:, 2].abs()
        big.step(a)
        small.step(a[k0:k0 + k].contiguous())
        cb, cs = big.contacts()["count"][k0:k0 + k], small.contacts()["count"]
        assert torch.equal(cb, cs) and int(cb.max()) <= C
        valid = (torch.arange(C, device="cuda")[None, :] < cs[:, None].long())[..., None].expand(k, C, WORDS)
        assert torch.equal(big._contacts[k0:k0 + k][valid], small._contacts[valid])
        touched += int((cs > 0).sum())
    assert touched > 0
    big.close(); small.close()


def test_report_of_a_terminating_step_describes_that_step():
    """Goals placed on the cubes: every env succeeds in its first step and, with auto-reset, restarts in the same call.  The report is
    the finished step's (bit-identical to a twin without auto-reset), not the reset scene's."""
    import panda_lang_manip_b200 as p
    n = 256
    rng = np.random.default_rng(3)
    objs = np.column_stack([rng.uniform(-0.15, 0.15, (n, 2)), np.full(n, 0.02)])
    envs = [p.PandaVecEnv("push", n, seed=9, auto_reset=ar, contact_report=True) for ar in (True, False)]
    for e in envs:
        e.reset(goals=objs, object_positions=objs)
    a = torch.zeros((n, 3), device="cuda")
    out = [e.step(a) for e in envs]
    assert bool(out[0][2].all()) and bool(out[1][2].all())                       # terminated (success) everywhere
    assert not torch.equal(envs[0].get_state()[:, 18:21], envs[1].get_state()[:, 18:21])   # the auto-reset env restarted
    c0, c1 = envs[0].contacts(), envs[1].contacts()
    assert torch.equal(c0["count"], c1["count"]) and bool((c0["count"] == 4).all())   # the cube's four bottom corners on the table
    assert torch.equal(envs[0]._contacts[:, :4], envs[1]._contacts[:, :4])
    pos = c0["position"][:, :4].mean(dim=1).cpu().numpy()
    assert np.abs(pos[:, :2] - objs[:, :2]).max() < 1e-3                           # where the cube was, not where it was reset to
    for e in envs:
        e.close()


def test_contacts_needs_the_flag():
    import panda_lang_manip_b200 as p
    env = p.PandaVecEnv("push", 4)
    with pytest.raises(p.PandaB200Error):
        env.contacts()
    env.close()
