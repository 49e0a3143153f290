"""CartesianMotion on the GPU: the batched move / grasp / release against the facade (robots/panda_cartesian.py, one env at a time),
per-env independence in a large sorted batch, the pick-up success rate, and the argument errors that need a device."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from tests.motion_util import DOWN, GRASP, MOVE, RELEASE, pick_and_lift, run_program  # noqa: E402

PG_ERR_ARG, PG_ERR_STATE = -1, -3


def _env(task, n, precision="f32", control_type="ee"):
    import panda_lang_manip_b200 as p
    return p.PandaVecEnv(task, n, control_type=control_type, precision=precision, auto_reset=False)


# ---------------------------------------------------------------------------------------------- facade agreement
N_FACADE = 8


def _facade_setup(precision):
    """8 PickAndPlace envs, cubes at distinct places.  Programs: release -> move above the cube -> move down -> grasp -> move to a
    lifted goal, each env with its own yaw.  Env 0's first move is under 3 cm (20 way-points); env 1 starts with a move of exactly
    4.5 cm along x from its reset pose (3 way-points, the distance an exact multiple of 1.5 cm) and releases after it."""
    import panda_lang_manip_b200 as p
    env = _env("pick_and_place", N_FACADE, precision)
    dev = env.device
    cubes = np.array([[0.0, 0.0, 0.02], [0.06, -0.04, 0.02], [-0.08, 0.05, 0.02], [0.1, 0.1, 0.02], [-0.12, -0.09, 0.02], [0.03, 0.12, 0.02],
                      [0.14, -0.12, 0.02], [-0.05, -0.14, 0.02]])
    goals = np.array([[0.1, 0.0, 0.15], [-0.1, 0.05, 0.2], [0.0, 0.1, 0.1], [0.05, -0.1, 0.25], [0.12, 0.08, 0.12], [-0.1, -0.1, 0.18],
                      [0.0, 0.0, 0.3], [0.08, 0.0, 0.05]])
    env.reset(goals=goals, object_positions=cubes)
    ee = env.ee_pose()[:, :3].cpu().numpy()
    kinds = np.tile([RELEASE, MOVE, MOVE, GRASP, MOVE], (N_FACADE, 1))
    tgt = np.stack([cubes, cubes + np.array([0.0, 0.0, 0.10]), cubes, cubes, goals], axis=1)
    tgt[0, 1] = ee[0] + np.array([0.01, -0.008, -0.012])            # |d| < 3 cm (the release before it holds the EE in place)
    x = ee[1, 0] + 0.045
    for _ in range(64):                                             # the goal whose x distance from the EE is 0.045 exactly
        if x - ee[1, 0] == 0.045:
            break
        x = np.nextafter(x, np.inf if x - ee[1, 0] < 0.045 else -np.inf)
    assert x - ee[1, 0] == 0.045
    kinds[1, :2] = [MOVE, RELEASE]
    tgt[1, 0] = [x, ee[1, 1], ee[1, 2]]
    yaw = np.array([0.0, 20.0, -35.0, 45.0, 10.0, -60.0, 90.0, -15.0])
    eul = np.zeros((N_FACADE, 5, 3)); eul[:] = DOWN; eul[:, 4, 2] = yaw; eul[:, 1, 2] = yaw / 2
    t = lambda a: torch.as_tensor(a, device=dev)
    return env, p, t(kinds), t(tgt), t(eul), kinds, tgt, eul


def _facade_run(precision, state_row, kinds, tgt, eul):
    """The same program through the facade (one env): joint angles after every step, and the step at which each primitive ended."""
    import panda_lang_manip_b200.panda_gym as pg
    from panda_lang_manip_b200.panda_gym.envs.robots.panda_cartesian import Panda as PandaCartesian
    fe = pg.make("PandaPickAndPlace-v3", precision=precision)
    fe.robot.__class__ = PandaCartesian
    fe.reset()
    sim, robot = fe.sim, fe.robot
    sim._vec.set_state(torch.as_tensor(state_row[None, :]))
    qs, ends = [], []
    step = sim.step

    def recorded():
        step()
        qs.append(sim._vec.get_state()[0, :9].cpu().numpy())
    sim.step = recorded
    for j, kind in enumerate(kinds):
        if kind == MOVE:
            robot.move(tgt[j], eul[j])
        elif kind == GRASP:
            robot.grasp()
        else:
            robot.release()
        ends.append(len(qs))
    fe.close()
    return np.array(qs), ends


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_batched_primitives_match_the_facade(precision):
    env, p, kinds, goals, eulers, kinds_np, tgt, eul = _facade_setup(precision)
    state0 = env.get_state().cpu().numpy()
    motion = p.CartesianMotion(env)
    qs, phases = [], []

    def rec(t, phase):
        qs.append(env.get_state()[:, :9].cpu().numpy())
        phases.append(phase.cpu().numpy())
    run_program(motion, kinds, goals, eulers, on_step=rec)
    qs, phases = np.array(qs), np.array(phases)
    worst = 0.0
    counts = []
    for k in range(N_FACADE):
        fq, fends = _facade_run(precision, state0[k], kinds_np[k], tgt[k], eul[k])
        # batched: primitive j of env k ended at the step after which its phase became j + 1
        bends = [int(np.argmax(phases[:, k] >= j + 1)) + 1 for j in range(5)]
        assert bends == fends, (k, bends, fends)
        counts.append(np.diff([0] + fends).tolist())
        worst = max(worst, float(np.abs(qs[:len(fq), k] - fq).max()))
    motion.close(); env.close()
    print(f"{precision}: primitive step counts per env {counts}; worst joint difference against the facade {worst:.3e} rad")
    assert counts[0][1] == 20 and counts[1][0] == 3
    # f64: the same arithmetic up to the Euler round trip the facade makes.  f32: one-ulp differences of the joint angles appear in free
    # motion (the facade's quaternion can carry the opposite sign, and the IK's wrap of the angle to (-pi, pi] rounds differently in
    # float) and grow while the fingers squeeze the cube; measured on a B200: 7.7e-5 rad at worst, 3e-6 rad outside the grasps.
    assert worst < (1e-12 if precision == "f64" else 2e-4), worst


# ---------------------------------------------------------------------------------------------- independence
def _random_programs(cubes, seed):
    """Per env, a random program of 6 primitives: pick-ups, moves to random places and gripper calls in random order."""
    g = torch.Generator(device=cubes.device).manual_seed(seed)
    n = cubes.shape[0]
    kinds = torch.randint(0, 3, (n, 6), generator=g, device=cubes.device)
    kinds[:, 0] = torch.randint(0, 3, (n,), generator=g, device=cubes.device)
    lo = torch.tensor([-0.15, -0.15, 0.0], dtype=torch.float64, device=cubes.device)
    goals = lo + torch.rand((n, 6, 3), generator=g, device=cubes.device, dtype=torch.float64) * torch.tensor([0.3, 0.3, 0.25], dtype=torch.float64, device=cubes.device)
    goals[:, 2] = cubes                                             # some envs descend onto their cube
    eulers = torch.tensor(DOWN, dtype=torch.float64, device=cubes.device).expand(n, 6, 3).clone()
    eulers[..., 2] = (torch.rand((n, 6), generator=g, device=cubes.device, dtype=torch.float64) - 0.5) * 120.0
    return kinds, goals, eulers


def test_every_env_is_independent_of_the_batch():
    """4096 + 37 envs (the contact-sorted schedule, with a partial last chunk) with out-of-phase random programs: the state rows of the
    envs run alone in a batch of one, over the same number of steps, are bit-identical."""
    import panda_lang_manip_b200 as p
    n = 4096 + 37
    env = _env("pick_and_place", n)
    state0 = env.get_state()
    cubes = state0[:, 18:21].contiguous()
    kinds, goals, eulers = _random_programs(cubes, 7)
    motion = p.CartesianMotion(env)
    steps, phase = run_program(motion, kinds, goals, eulers)
    big = env.get_state()
    assert bool((phase >= kinds.shape[1]).all())
    motion.close(); env.close()
    picks = [0, 1, 127, 128, 2047, 2048, 4095, 4096, 4100, n - 1]
    for k in picks:
        one = _env("pick_and_place", 1)
        one.set_state(state0[k:k + 1])
        m1 = p.CartesianMotion(one)
        run_program(m1, kinds[k:k + 1], goals[k:k + 1], eulers[k:k + 1], steps=steps)
        row = one.get_state()
        m1.close(); one.close()
        assert torch.equal(row[0], big[k]), (k, (row[0] - big[k]).abs().max().item())
    print(f"{n} envs, {steps} steps: envs {picks} bit-identical to their batch-of-one runs")


# ---------------------------------------------------------------------------------------------- outcome
def test_pick_and_lift_success_rate():
    """1024 cubes at the sampler's random places: release, above, down, grasp, lift 15 cm.  Each cube's height is read at the step its
    env's program ends (as the facade's program ends there; the fingers' hold at finger action 0 is not meant to last indefinitely)."""
    import panda_lang_manip_b200 as p
    n = 1024
    env = _env("pick_and_place", n)
    cube0 = env.get_state()[:, 18:21].clone()
    kinds, goals, eulers = pick_and_lift(cube0)
    end_z = torch.full((n,), float("nan"), dtype=torch.float64, device=env.device)
    motion = p.CartesianMotion(env)

    def rec(t, phase):
        just = (phase >= kinds.shape[1]) & torch.isnan(end_z)
        end_z[just] = env.get_state()[just, 20]
    steps, _ = run_program(motion, kinds, goals, eulers, on_step=rec)
    rate = float(((end_z - cube0[:, 2]) > 0.10).double().mean())
    motion.close(); env.close()
    print(f"pick and lift: {rate * 100:.2f} % of {n} cubes more than 10 cm above their start when their program ends ({steps} steps)")
    assert rate >= 0.99, rate


# ---------------------------------------------------------------------------------------------- errors that need a device
def _err(lib, rc):
    return rc, lib.pg_last_error().decode()


def test_motion_errors_with_a_device():
    import panda_lang_manip_b200 as p
    lib = p.load()
    plan = ctypes.c_void_p()
    assert lib.pg_motion_create(4, 0, ctypes.byref(plan)) == 0
    q = torch.zeros((4, 4), dtype=torch.float64, device="cuda"); q[:, 3] = 1
    x = torch.zeros((4, 3), dtype=torch.float64, device="cuda")
    joints = _env("pick_and_place", 4, control_type="joints")
    assert _err(lib, lib.pg_motion_move(plan, joints._h, x.data_ptr(), q.data_ptr(), None, None)) == \
        (PG_ERR_STATE, "pg_motion_move: the motion primitives need an ee-controlled handle")
    with pytest.raises(p.PandaB200Error):
        p.CartesianMotion(joints)
    bare = p.PandaBareWorld(4)
    assert _err(lib, lib.pg_motion_step(plan, bare._h, *[None] * 7, None)) == (PG_ERR_STATE, "pg_motion_step: a bare world has no ee action to drive")
    five = _env("pick_and_place", 5)
    assert _err(lib, lib.pg_motion_gripper(plan, five._h, -1.0, 30, None, None)) == \
        (PG_ERR_ARG, "pg_motion_gripper: the plan was created for another batch size or device")
    reach = _env("reach", 4)
    assert _err(lib, lib.pg_motion_gripper(plan, reach._h, -1.0, 30, None, None)) == \
        (PG_ERR_STATE, "pg_motion_gripper: this task blocks the gripper (Reach, Push, Slide have no finger action)")
    m = p.CartesianMotion(reach)
    with pytest.raises(p.PandaB200Error):
        m.grasp()
    m.move(torch.tensor([0.05, 0.0, 0.1]), goal_quat=torch.tensor([1.0, 0.0, 0.0, 0.0]))      # Reach moves: 3-D actions
    m.run()
    assert float((reach.ee_pose()[:, :3].cpu() - torch.tensor([0.05, 0.0, 0.1], dtype=torch.float64)).norm(dim=1).max()) < 0.01
    m.close()
    assert lib.pg_motion_destroy(plan) == 0
    for e in (joints, bare, five, reach):
        e.close()
