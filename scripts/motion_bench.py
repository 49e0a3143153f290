"""Cost of the batched motion primitives (CartesianMotion / pg_motion_step) on one GPU.

1. Device time per env step, pg_motion_step against pg_step with the same actions and orientations: PickAndPlace at 32,768 envs (a release:
   finger action 1, zero displacement, the current EE orientation) and Reach ee at 65,536 envs (idle: zero displacement, the current
   EE orientation).  Both legs start from the same snapshot; the pg_step leg reads each step's orientation with pg_get_ee_pose
   outside its timed window, so both legs step the same trajectory.  Blocks of the two legs alternate.  CUDA events around every step;
   the state fits in L2 and is not flushed (the step kernel is compute-bound).  A move's motion step is timed as well.
2. The per-step kernel's own device time (motion_step_kernel), from torch.profiler in a run of its own.
3. End-to-end env-steps/s of the pick-and-lift program (release, above, down, grasp, lift 15 cm) on 1024 PickAndPlace envs chained by
   the torch phase machine of tests/motion_util.py, against the facade (robots/panda_cartesian.py) running the same program on one env.

Prints one JSON document (also written to --out) with the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import panda_lang_manip_b200 as p  # noqa: E402
from tests.motion_util import pick_and_lift, run_program  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return out.strip().splitlines()[0] if out.strip() else "unknown"


def timed(fn, before=None):
    """Device time (ms) of fn() between two events; before() runs outside the window."""
    if before is not None:
        before()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); fn(); b.record()
    b.synchronize()
    return a.elapsed_time(b)


def step_legs(task, n, steps, blocks):
    env = p.PandaVecEnv(task, n, control_type="ee", auto_reset=False)
    motion = p.CartesianMotion(env)
    gripper = task != "reach"
    act = torch.zeros((n, env.action_dim), dtype=torch.float32, device=env.device)
    if gripper:
        act[:, -1] = 1.0
    quat = {}
    sid = env.save_state()

    def begin():
        if gripper:
            motion.release()              # 30 steps of finger action 1 (the steps below stay inside it)
    # warm-up of both legs
    for _ in range(3):
        begin(); motion.step()
        env.step(act, env.ee_pose()[:, 3:].float())
    torch.cuda.synchronize()
    res = {"motion_step_ms": [], "step_oriented_ms": []}
    for _ in range(blocks):
        env.restore_state(sid); begin()
        res["motion_step_ms"] += [timed(motion.step) for _ in range(steps)]
        env.restore_state(sid)
        res["step_oriented_ms"] += [timed(lambda: env.step(act, quat["q"]), before=lambda: quat.update(q=env.ee_pose()[:, 3:].float())) for _ in range(steps)]
    # a move of every env (long enough to outlast the timed steps)
    env.restore_state(sid)
    goal = env.ee_pose()[:, :3] + torch.tensor([0.0, 0.0, -0.12], dtype=torch.float64, device=env.device)
    motion.move(goal, goal_euler=[180.0, 0.0, 30.0])
    res["motion_step_move_ms"] = [timed(motion.step) for _ in range(steps)]
    motion.close(); env.remove_state(sid); env.close()
    m, o = statistics.median(res["motion_step_ms"]), statistics.median(res["step_oriented_ms"])
    return {"task": task, "envs": n, "timed_steps_per_leg": steps * blocks, "motion_step_ms_median": m, "step_oriented_ms_median": o,
            "motion_minus_oriented_ms": m - o, "overhead_pct": 100.0 * (m - o) / o, "motion_step_during_move_ms_median": statistics.median(res["motion_step_move_ms"])}


def kernel_time(task, n, steps):
    from torch.profiler import ProfilerActivity, profile
    env = p.PandaVecEnv(task, n, control_type="ee", auto_reset=False)
    motion = p.CartesianMotion(env)
    goal = env.ee_pose()[:, :3] + torch.tensor([0.0, 0.0, -0.12], dtype=torch.float64, device=env.device)
    motion.move(goal, goal_euler=[180.0, 0.0, 30.0])
    motion.step(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            motion.step()
        torch.cuda.synchronize()
    ks = {}
    for ev in prof.events():
        if str(ev.device_type).endswith("CUDA"):
            ks.setdefault(ev.name, []).append(ev.time_range.elapsed_us())
    motion.close(); env.close()
    mk = [v for k, v in ks.items() if "motion_step_kernel" in k]
    step_total = sum(sum(v) for v in ks.values()) / steps
    mean_us = float(np.mean(mk[0])) if mk else float("nan")
    return {"task": task, "envs": n, "motion_step_kernel_us_mean": mean_us, "all_kernels_us_per_step": step_total,
            "motion_kernel_share_pct": 100.0 * mean_us / step_total if mk else float("nan")}


def program_rates():
    n = 1024
    env = p.PandaVecEnv("pick_and_place", n, control_type="ee", auto_reset=False)
    cube = env.get_state()[:, 18:21].clone()
    sid = env.save_state()
    motion = p.CartesianMotion(env)
    run_program(motion, *pick_and_lift(cube))                  # warm-up
    env.restore_state(sid); torch.cuda.synchronize()
    t0 = time.perf_counter()
    steps, _ = run_program(motion, *pick_and_lift(cube))
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    motion.close(); env.close()
    import panda_lang_manip_b200.panda_gym as pg
    from panda_lang_manip_b200.panda_gym.envs.robots.panda_cartesian import Panda as PandaCartesian
    fe = pg.make("PandaPickAndPlace-v3")
    fe.robot.__class__ = PandaCartesian
    fe.reset(seed=0)
    robot, sim = fe.robot, fe.sim
    calls = {"n": 0}
    step = sim.step

    def counted():
        step(); calls["n"] += 1
    sim.step = counted

    def program():
        c = sim.get_base_position("object")
        robot.release(); robot.move(c + np.array([0.0, 0.0, 0.10]), [180.0, 0.0, 0.0]); robot.move(c, [180.0, 0.0, 0.0])
        robot.grasp(); robot.move(c + np.array([0.0, 0.0, 0.15]), [180.0, 0.0, 0.0])
    fsid = fe.save_state()
    program()                                                   # warm-up
    fe.restore_state(fsid); calls["n"] = 0
    t0 = time.perf_counter()
    program()
    fdt = time.perf_counter() - t0
    fe.close()
    return {"batched_envs": n, "batched_steps": steps, "batched_seconds": dt, "batched_env_steps_per_s": steps * n / dt,
            "facade_steps": calls["n"], "facade_seconds": fdt, "facade_env_steps_per_s": calls["n"] / fdt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed steps per block and leg")
    ap.add_argument("--blocks", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("motion_bench.py measures on the GPU; no CUDA device here")
    res = {"gpu": gpu_info(),
           "step_legs": [step_legs("pick_and_place", 32768, args.steps, args.blocks), step_legs("reach", 65536, args.steps, args.blocks)],
           "kernel": [kernel_time("pick_and_place", 32768, 10), kernel_time("reach", 65536, 10)],
           "program": program_rates()}
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(s + "\n")


if __name__ == "__main__":
    main()
