"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on identical goals and actions.

Tolerances (BASELINE.json north_star): joint state 1e-4 rad and end-effector position 1e-4 m at every step of a 50-step
episode; rewards / success bit-exact.  Velocities are compared at 2e-2 (the PGS early-exit makes them the most sensitive
quantity).  Contact tasks: object pose over short horizons, tolerance stated per test.
"""
import numpy as np
import pytest

from tests.oracle_util import GOAL_DIM, NOBJ, OBS_DIM, OracleEnv, reward_np

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _sample(task, rng):
    goal = np.zeros(6)
    goal[:3] = rng.uniform([-0.15, -0.15, 0.0], [0.15, 0.15, 0.2])
    if task in ("push", "slide", "stack"):
        goal[2] = 0.03 if task == "slide" else 0.02
    if task == "stack":
        goal[3:] = goal[:3] + [0, 0, 0.04]
    if task == "flip":
        q = rng.normal(size=4); goal[:4] = q / np.linalg.norm(q)
    obj = np.zeros(6)
    obj[:3] = [rng.uniform(-0.15, 0.15), rng.uniform(-0.15, 0.15), 0.03 if task == "slide" else 0.02]
    obj[3:] = [rng.uniform(-0.15, 0.15), rng.uniform(-0.15, 0.15), 0.06]
    return goal, obj


def _rollout(task, control, n_envs, steps, precision="f32", seed=0, action_scale=1.0, teacher=False):
    import panda_lang_manip_b200 as p
    rng = np.random.default_rng(seed)
    G, nobj = GOAL_DIM[task], NOBJ[task]
    goals, objs = zip(*[_sample(task, rng) for _ in range(n_envs)])
    goals, objs = np.array(goals), np.array(objs)
    env = p.PandaVecEnv(task, n_envs, control_type=control, precision=precision, auto_reset=False)
    o0 = env.reset(goals=goals[:, :G], object_positions=objs[:, :3 * nobj] if nobj else None)
    oracles = [OracleEnv(task, control) for _ in range(n_envs)]
    ref0 = [oe.reset(goals[i], objs[i]) for i, oe in enumerate(oracles)]
    assert np.allclose(o0["observation"].cpu().numpy(), np.array([r[0] for r in ref0]), atol=1e-6)
    errs = dict(q=0.0, qd=0.0, ee=0.0, obs=0.0, obj=0.0, rew=0, succ=0, rew_oracle=0, compared=0, q_env=np.zeros(n_envs), ee_env=np.zeros(n_envs), obj_env=np.zeros(n_envs))
    A = env.action_dim
    thr = {"stack": 0.1, "flip": 0.2}.get(task, 0.05)
    for t in range(steps):
        a = (rng.uniform(-1, 1, (n_envs, A)) * action_scale).astype(np.float32)
        obs, rew, term, trunc, _ = env.step(torch.from_numpy(a).cuda())
        st = env.get_state().cpu().numpy()
        obs_g, ag_g, dg_g = obs["observation"].cpu().numpy(), obs["achieved_goal"].cpu().numpy(), obs["desired_goal"].cpu().numpy()
        rew_g, term_g = rew.cpu().numpy(), term.cpu().numpy()
        for i, oe in enumerate(oracles):
            ob, ag, dg, r, s = oe.step(a[i])
            q, qd = oe.joints()
            errs["q"] = max(errs["q"], np.abs(st[i, :9] - q).max()); errs["qd"] = max(errs["qd"], np.abs(st[i, 9:18] - qd).max())
            errs["ee"] = max(errs["ee"], np.abs(obs_g[i, :3] - ob[:3]).max()); errs["obs"] = max(errs["obs"], np.abs(obs_g[i] - ob).max())
            errs["q_env"][i] = max(errs["q_env"][i], np.abs(st[i, :9] - q).max()); errs["ee_env"][i] = max(errs["ee_env"][i], np.abs(obs_g[i, :3] - ob[:3]).max())
            for o in range(nobj):
                eo = np.abs(st[i, 18 + 13 * o:18 + 13 * o + 7] - oe.object_state(o)[:7]).max()
                errs["obj"] = max(errs["obj"], eo); errs["obj_env"][i] = max(errs["obj_env"][i], eo)
            # reward / success of EVERY env at EVERY step, teacher-forced or free-running: bit-exact against the reference's arithmetic
            # (numpy) on the inputs RobotTaskEnv.step passes (core.py:285-288): the float32 achieved goal the kernel itself emitted and
            # the task's FLOAT64 goal (numpy promotes the distance to float64) ...
            g0 = 18 + 13 * nobj
            r_np, s_np = reward_np(task, "sparse", ag_g[i], st[i, g0:g0 + GOAL_DIM[task]])
            errs["rew"] += int(np.float32(rew_g[i]).tobytes() != np.float32(r_np).tobytes()); errs["succ"] += int(bool(term_g[i]) != bool(s_np))
            errs["compared"] += 1
            # ... and against the oracle's own decision, unless the oracle's distance sits within 1 mm of the threshold (an fp32 state
            # 1e-4 away from the fp64 one may legitimately fall on the other side there)
            d_or = float(1 - np.dot(ag.astype(np.float64), dg.astype(np.float64)) ** 2) if task == "flip" else float(np.linalg.norm(ag.astype(np.float64) - dg.astype(np.float64)))
            if abs(d_or - thr) > 1e-3:
                errs["rew_oracle"] += int(bool(term_g[i]) != bool(s)) + int(float(rew_g[i]) != float(r))
            if teacher:     # per-step comparison: continue from the oracle's state
                st[i, :9], st[i, 9:18] = q, qd
                for o in range(nobj):
                    st[i, 18 + 13 * o:18 + 13 * o + 13] = oe.object_state(o)
        if teacher:
            env.set_state(torch.from_numpy(st))
    for oe in oracles:
        oe.close()
    env.close()
    return errs


@pytest.mark.parametrize("control", ["joints", "ee"])
def test_reach_per_step_parity_f32(control):
    """north_star: joint state within 1e-4 rad and end-effector within 1e-4 m PER STEP over 50-step episodes: every step starts from
    the oracle's state (fp32 kernels vs fp64 oracle), all envs, all steps."""
    e = _rollout("reach", control, n_envs=16, steps=50, precision="f32", seed=1, teacher=True)
    assert e["q"] < 1e-4 and e["ee"] < 1e-4, e
    assert e["compared"] == 16 * 50 and e["rew"] == 0 and e["succ"] == 0 and e["rew_oracle"] == 0, e


@pytest.mark.parametrize("control", ["joints", "ee"])
def test_reach_free_running_parity_f32(control):
    """Free-running 50-step episodes (errors accumulate; the solver's iteration-count early exit and contact on/off events are
    discontinuities that an fp32 trajectory crosses at slightly different times than the fp64 oracle): the typical env must stay
    well inside 1e-4, and at least 80% of the envs inside 1e-4 over the whole episode; nothing may exceed 5e-3."""
    e = _rollout("reach", control, n_envs=32, steps=50, precision="f32", seed=1)
    assert np.median(e["q_env"]) < 2e-5 and np.median(e["ee_env"]) < 2e-5, e
    assert (e["q_env"] < 1e-4).mean() >= 0.8 and (e["ee_env"] < 1e-4).mean() >= 0.8, e
    assert e["q"] < 5e-3 and e["compared"] == 32 * 50 and e["rew"] == 0 and e["succ"] == 0 and e["rew_oracle"] == 0, e


@pytest.mark.parametrize("control", ["joints", "ee"])
def test_reach_episode_parity_f64(control):
    """fp64 kernels vs the fp64 oracle, free-running: two independent formulations (CRBA+Cholesky+operational-space contacts vs
    ABA+impulse responses+generalized rows) agree to 1e-4 over whole episodes."""
    e = _rollout("reach", control, n_envs=8, steps=50, precision="f64", seed=2)
    assert e["q"] < 1e-4 and e["ee"] < 1e-4 and e["compared"] == 8 * 50 and e["rew"] == 0 and e["succ"] == 0 and e["rew_oracle"] == 0, e
    assert np.median(e["q_env"]) < 2e-5, e


@pytest.mark.parametrize("task", ["push", "slide", "pick_and_place", "stack", "flip"])
def test_contact_tasks_short_horizon(task):
    """Random actions, 25 steps free-running, fp32: typical env 2e-5 rad / 3e-4 m object pose, worst env 1e-3 rad / 2e-2 m (a tumbling object amplifies fp32 noise)."""
    e = _rollout(task, "ee", n_envs=8, steps=25, precision="f32", seed=3)
    assert np.median(e["q_env"]) < 2e-5 and e["q"] < 1e-3 and np.median(e["obj_env"]) < 3e-4 and e["obj"] < 2e-2, e
    assert e["compared"] == 8 * 25 and e["rew"] == 0 and e["succ"] == 0, e


@pytest.mark.parametrize("task", ["reach", "push", "slide", "pick_and_place", "stack", "flip"])
def test_f64_parity_mode_every_task(task):
    """precision="f64" on every task (two-object scenes run 32-env blocks there: 416 slots x 8 B x 128 envs would not fit a block's shared
    memory): three teacher-forced steps against the fp64 oracle -- two fp64 formulations of the same model agree to 1e-6 (measured 2e-7 at worst: the
    sweep loop's exit test is a discontinuity that two formulations cross at slightly different residuals)."""
    e = _rollout(task, "ee", n_envs=4, steps=3, precision="f64", seed=6, teacher=True)
    assert e["q"] < 1e-6 and e["ee"] < 1e-6 and e["obj"] < 1e-6 and e["compared"] == 4 * 3 and e["rew"] == 0 and e["succ"] == 0, e


@pytest.mark.parametrize("task", ["push", "pick_and_place", "stack"])
def test_contact_tasks_per_step(task):
    """Per-step (teacher-forced) agreement on contact tasks: robot 1e-4, object pose (position, quaternion) 5e-4."""
    e = _rollout(task, "ee", n_envs=8, steps=25, precision="f32", seed=4, teacher=True)
    assert e["q"] < 1e-4 and e["ee"] < 1e-4 and e["obj"] < 5e-4 and np.median(e["obj_env"]) < 1e-4, e
    assert e["compared"] == 8 * 25 and e["rew"] == 0 and e["succ"] == 0 and e["rew_oracle"] == 0, e


@pytest.mark.parametrize("task,G", [("reach", 3), ("stack", 6)])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_compute_reward_bit_exact(task, G, dtype):
    import panda_lang_manip_b200 as p
    rng = np.random.default_rng(5)
    m = 100003
    thr = {"stack": 0.1, "flip": 0.2}.get(task, 0.05)
    dg = rng.uniform(-0.3, 0.3, (m, G)).astype(dtype)
    ag = (dg + rng.normal(0, thr / np.sqrt(G), (m, G))).astype(dtype)
    if task == "flip":
        ag /= np.linalg.norm(ag, axis=-1, keepdims=True); dg /= np.linalg.norm(dg, axis=-1, keepdims=True)
    ag[:7] = dg[:7]                                  # d == 0
    ag[7, 0] = dg[7, 0] + np.asarray(thr, dtype)     # sits on / next to the threshold
    for rt in ("sparse", "dense"):
        got = p.compute_reward(task, rt, torch.from_numpy(ag).cuda(), torch.from_numpy(dg).cuda()).cpu().numpy()
        want, succ = reward_np(task, rt, ag, dg)
        assert got.dtype == np.float32 and got.tobytes() == want.tobytes(), (task, rt, dtype, np.abs(got - want).max())
    got_s = p.is_success(task, torch.from_numpy(ag).cuda(), torch.from_numpy(dg).cuda()).cpu().numpy()
    assert np.array_equal(got_s, succ)


@pytest.mark.parametrize("task", ["reach", "push", "slide", "pick_and_place", "stack", "flip"])
@pytest.mark.parametrize("rt", ["sparse", "dense"])
@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_compute_reward_reference_golden(task, rt, dt):
    """Against vectors produced by the reference's own compute_reward / is_success (tests/golden/make_golden.py).
    Bit-exact, except Flip: its np.inner goes through a BLAS dot whose summation order is CPU-kernel dependent, so Flip is
    checked to 1 ulp-level tolerance (2e-7 f32 / 1e-15 f64) and its threshold decisions away from the boundary."""
    import os
    import panda_lang_manip_b200 as p
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_rewards.npz"))
    k = f"{task}_{rt}_{dt}"
    ag, dg, want, succ = gold[k + "_ag"], gold[k + "_dg"], gold[k + "_reward"], gold[k + "_success"]
    got = p.compute_reward(task, rt, torch.from_numpy(ag).cuda(), torch.from_numpy(dg).cuda()).cpu().numpy()
    got_s = p.is_success(task, torch.from_numpy(ag).cuda(), torch.from_numpy(dg).cuda()).cpu().numpy()
    if task != "flip":
        assert got.tobytes() == want.tobytes() and np.array_equal(got_s, succ)
    else:
        d = 1 - np.einsum("ij,ij->i", ag.astype(np.float64), dg.astype(np.float64)) ** 2
        safe = np.abs(d - 0.2) > 1e-5
        assert np.allclose(got[safe], want[safe], atol=2e-7 if dt == "float32" else 1e-15) and np.array_equal(got_s[safe], succ[safe])


def test_seed_determinism_and_snapshot():
    """reference test/seed_test.py (same seed -> same trajectory) and test/save_and_restore_test.py:9-27 (bit-identical)."""
    import panda_lang_manip_b200 as p
    n = 256
    a = torch.rand((6, n, 4), device="cuda") * 2 - 1
    outs = []
    for rep in range(2):
        env = p.PandaVecEnv("pick_and_place", n, seed=11)
        for t in range(6):
            obs, *_ = env.step(a[t])
        outs.append(torch.cat([obs["observation"], obs["achieved_goal"], obs["desired_goal"]], 1).clone())
        env.close()
    assert torch.equal(outs[0], outs[1])
    env = p.PandaVecEnv("pick_and_place", n, seed=11)
    sid = env.save_state()
    o1 = {k: v.clone() for k, v in env.step(a[0])[0].items()}
    env.reset()
    env.restore_state(sid)
    o2 = env.step(a[0])[0]
    assert all(torch.equal(o1[k], o2[k]) for k in o1)
    env.remove_state(sid)
    with pytest.raises(p.PandaB200Error):
        env.restore_state(sid)
    env.close()


def test_auto_reset_truncation_and_stats():
    import panda_lang_manip_b200 as p
    n = 512
    for precision in ("f32", "f64"):
        env = p.PandaVecEnv("reach", n, control_type="joints", seed=3, precision=precision)
        zero = torch.zeros((n, 7), device="cuda")
        term_seen = torch.zeros(n, dtype=torch.uint8, device="cuda")
        for t in range(50):
            _, _, term, trunc, _ = env.step(zero)
            term_seen |= term
            if t < 49:
                assert int(trunc.sum()) == 0
        assert bool(((trunc == 1) | (term_seen == 1)).all())      # at step 50 every env has either succeeded earlier (and restarted) or is truncated now
        st = env.stats()
        assert st[0] >= int(trunc.sum()) and st[3] > 0
        assert env.diverged() == 0
        bad = env.get_state(); bad[:7, 0] = float("nan")          # poison 7 envs: they are counted, truncated and restarted
        env.set_state(bad)
        _, _, term, trunc, _ = env.step(zero)
        assert env.diverged() == 7 and int(trunc[:7].sum()) == 7 and bool(torch.isfinite(env.get_state()).all())
        env.close()


def test_large_batch_properties():
    """Full bench size (65,536 envs): size-independent properties -- finite outputs, joint limits respected to 1e-2 rad,
    reward consistent with the goals the kernel itself wrote, EE inside the arm's reach."""
    import panda_lang_manip_b200 as p
    n = 65536
    env = p.PandaVecEnv("reach", n, control_type="joints", reward_type="dense", seed=1, auto_reset=False)
    g = torch.Generator(device="cuda").manual_seed(0)
    for t in range(10):
        obs, rew, term, trunc, _ = env.step(torch.rand((n, 7), device="cuda", generator=g) * 2 - 1)
    o = obs["observation"]
    assert torch.isfinite(o).all() and torch.isfinite(rew).all()
    d = torch.linalg.norm(obs["achieved_goal"] - obs["desired_goal"], dim=-1)
    assert torch.allclose(-d, rew, atol=1e-6)
    st = env.get_state()
    lo = torch.tensor([-2.9671, -1.8326, -2.9671, -3.1416, -2.9671, -0.0873, -2.9671, 0.0, 0.0], device="cuda", dtype=torch.float64)
    hi = torch.tensor([2.9671, 1.8326, 2.9671, 0.0, 2.9671, 3.8223, 2.9671, 0.04, 0.04], device="cuda", dtype=torch.float64)
    assert (st[:, :9] > lo - 1e-2).all() and (st[:, :9] < hi + 1e-2).all()
    assert (torch.linalg.norm(o[:, :3] - torch.tensor([-0.6, 0.0, 0.333], device="cuda"), dim=-1) < 1.2).all()
    env.close()


def test_oriented_ee_control_parity():
    """SURVEY section 8f rank 1 (the fork's robots/panda_ori.py:52-99 and panda_cartesian.py:67,157): a per-env EE target orientation
    fed to the IK, with the fork's unscaled actions; per-step parity against the oracle at the Reach tolerances."""
    import panda_lang_manip_b200 as p
    from panda_lang_manip_b200.panda_gym.envs.robots.panda_ori import quat_from_euler_xyz_deg
    from scipy.spatial.transform import Rotation as R
    n, steps = 8, 30
    rng = np.random.default_rng(9)
    goals = rng.uniform([-0.15, -0.15, 0.05], [0.15, 0.15, 0.3], (n, 3))
    env = p.PandaVecEnv("pick_and_place", n, control_type="ee", auto_reset=False)
    env.set_action_scale(1.0, 1.0)
    objs = np.stack([rng.uniform(-0.15, 0.15, n), rng.uniform(-0.15, 0.15, n), np.full(n, 0.02)], -1)
    env.reset(goals=goals, object_positions=objs)
    oracles = [OracleEnv("pick_and_place", "ee") for _ in range(n)]
    for i, oe in enumerate(oracles):
        oe.reset(goals[i], objs[i])
    worst_q = worst_ee = 0.0
    for t in range(steps):
        eul = np.stack([180 + rng.uniform(-25, 25, n), rng.uniform(-25, 25, n), rng.uniform(-40, 40, n)], -1)
        quats = np.array([quat_from_euler_xyz_deg(e) for e in eul])
        assert np.allclose(np.abs((quats * R.from_euler("xyz", eul, degrees=True).as_quat()).sum(-1)), 1.0, atol=1e-12)
        a = np.concatenate([rng.uniform(-0.03, 0.03, (n, 3)), rng.uniform(-0.02, 0.02, (n, 1))], -1).astype(np.float32)
        obs, *_ = env.step(torch.from_numpy(a).cuda(), target_orientation=torch.from_numpy(quats.astype(np.float32)).cuda())
        st = env.get_state().cpu().numpy()
        og = obs["observation"].cpu().numpy()
        for i, oe in enumerate(oracles):
            ob, *_ = oe.step_oriented(a[i], quats[i].astype(np.float32).astype(np.float64), 1.0, 1.0)
            q, qd = oe.joints()
            worst_q = max(worst_q, np.abs(st[i, :9] - q).max()); worst_ee = max(worst_ee, np.abs(og[i, :3] - ob[:3]).max())
            st[i, :9], st[i, 9:18] = q, qd
            st[i, 18:31] = oe.object_state(0)
        env.set_state(torch.from_numpy(st))
    for oe in oracles:
        oe.close()
    env.close()
    assert worst_q < 1e-4 and worst_ee < 1e-4, (worst_q, worst_ee)


def test_target_orientation_needs_ee_control():
    import panda_lang_manip_b200 as p
    env = p.PandaVecEnv("reach", 4, control_type="joints", auto_reset=False)
    q = torch.tensor([[1.0, 0.0, 0.0, 0.0]] * 4, device="cuda")
    with pytest.raises(p.PandaB200Error) as err:
        env.step(torch.zeros((4, 7), device="cuda"), target_orientation=q)
    assert str(err.value).endswith("pg_step: a target orientation needs ee control")
    env.close()


def test_edge_cases_ragged_unaligned_empty():
    """Ragged env counts (not a multiple of the 128-thread block, sorted and identity thread->env maps), unaligned goal views
    (scalar path of the reward kernel), empty batches, host-buffer stepping, every task's kernels."""
    import panda_lang_manip_b200 as p
    for task, ctrl in (("reach", "joints"), ("reach", "ee"), ("pick_and_place", "ee"), ("stack", "joints"), ("slide", "ee"), ("flip", "ee")):
        for n in (1, 130, 4096 + 37):
            env = p.PandaVecEnv(task, n, control_type=ctrl, seed=1)
            g = torch.Generator(device="cuda").manual_seed(0)
            for t in range(2):
                obs, rew, term, trunc, _ = env.step(torch.rand((n, env.action_dim), device="cuda", generator=g) * 2 - 1)
            assert torch.isfinite(obs["observation"]).all() and obs["observation"].shape == (n, env.obs_dim)
            ho, hr, ht, htr, _ = env.step_host(np.zeros((n, env.action_dim), np.float32))
            assert np.isfinite(ho["observation"]).all() and hr.shape == (n,)
            env.close()
    ag = torch.rand((100003, 3), device="cuda"); dg = torch.rand((100003, 3), device="cuda")
    full = p.compute_reward("reach", "dense", ag, dg)
    view = p.compute_reward("reach", "dense", ag[1:], dg[1:])           # 12-byte offset: not 16-byte aligned
    assert torch.equal(full[1:], view)
    assert p.compute_reward("reach", "sparse", ag[:0], dg[:0]).shape == (0,)
    assert p.is_success("stack", torch.rand((5, 6), device="cuda"), torch.rand((5, 6), device="cuda")).shape == (5,)
    with pytest.raises(ValueError):
        p.compute_reward("reach", "sparse", ag, dg[:, :2])


@pytest.mark.gpu
@pytest.mark.parametrize("task,ctrl", [("pick_and_place", "ee"), ("reach", "joints"), ("stack", "ee")])
def test_scheduling_is_invisible(task, ctrl):
    """The contact-aware scheduling of large batches (per-launch re-sort, a step cut into sub-step launches, env groups on their
    own streams) only decides which thread runs which env: a window of a 16,684-env batch must evolve bit-identically to the same
    envs stepped as a small batch (identity map, one launch per step)."""
    import panda_lang_manip_b200 as p
    n, k0, k = 16384 + 300, 9000, 512
    big = p.PandaVecEnv(task, n, control_type=ctrl, seed=3)
    small = p.PandaVecEnv(task, k, control_type=ctrl, seed=3, env_id_offset=k0)
    assert torch.equal(big.get_state()[k0:k0 + k], small.get_state())            # same reset stream (keyed by global env id)
    g = torch.Generator(device="cuda").manual_seed(1)
    for t in range(12):
        a = torch.rand((n, big.action_dim), device="cuda", generator=g) * 2 - 1
        if task != "reach":
            a[:, 2] = -a[:, 2].abs()                                             # drive the grippers into the table / objects
        ob, rb, tb, ub, _ = big.step(a)
        os_, rs, ts, us, _ = small.step(a[k0:k0 + k].contiguous())
        assert torch.equal(ob["observation"][k0:k0 + k], os_["observation"]) and torch.equal(rb[k0:k0 + k], rs)
        assert torch.equal(tb[k0:k0 + k], ts) and torch.equal(ub[k0:k0 + k], us)
    assert torch.equal(big.get_state()[k0:k0 + k], small.get_state())
    big.close(); small.close()


@pytest.mark.gpu
def test_host_path_pinned_and_pageable_buffers_agree():
    """pg_step_host copies directly from / to page-locked buffers (pg_host_pin) and through its staging slabs otherwise: same results."""
    import panda_lang_manip_b200 as p
    n = 300
    for precision in ("f32", "f64"):
        a_env = p.PandaVecEnv("push", n, seed=4, auto_reset=False, precision=precision)
        b_env = p.PandaVecEnv("push", n, seed=4, auto_reset=False, precision=precision)
        rng = np.random.default_rng(0)
        pinned = a_env.pin_host(np.zeros((n, 3), np.float32))
        for t in range(3):
            act = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
            pinned[:] = act
            oa, ra, ta, ua, _ = a_env.step_host(pinned)
            ob, rb, tb, ub, _ = b_env.step(torch.from_numpy(act).cuda())
            assert np.array_equal(oa["observation"], ob["observation"].cpu().numpy()) and np.array_equal(oa["desired_goal"], ob["desired_goal"].cpu().numpy())
            assert np.array_equal(ra, rb.cpu().numpy()) and np.array_equal(ta, tb.cpu().numpy())
        # the raw entry point with pageable outputs (staging slabs) on a third twin
        c_env = p.PandaVecEnv("push", n, seed=4, auto_reset=False, precision=precision)
        rng = np.random.default_rng(0)
        o2, g2, d2, r2, t2, u2 = np.empty((n, 18), np.float32), np.empty((n, 3), np.float32), np.empty((n, 3), np.float32), np.empty(n, np.float32), np.empty(n, np.uint8), np.empty(n, np.uint8)
        for t in range(3):
            act = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
            rc = c_env.lib.pg_step_host(c_env._h, act.ctypes.data, o2.ctypes.data, g2.ctypes.data, d2.ctypes.data, r2.ctypes.data, t2.ctypes.data, u2.ctypes.data, 0)
            assert rc == 0
        assert np.array_equal(o2, oa["observation"]) and np.array_equal(r2, ra) and np.array_equal(t2, ta)
        a_env.unpin_host(pinned)
        a_env.close(); b_env.close(); c_env.close()
