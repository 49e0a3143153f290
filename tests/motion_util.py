"""Scripted programs for CartesianMotion: a torch phase machine that chains each env's primitives on the device.

A program is, per env, a list of P primitives: ``kinds`` [N, P] (MOVE, GRASP, RELEASE), ``goals`` [N, P, 3] and ``eulers`` [N, P, 3]
(xyz, degrees; used by MOVE).  Every env begins its next primitive right after the step at which its previous one ended
(``remaining == 0``), so envs run out of phase; an env whose program is over is stepped in place."""
import torch

MOVE, GRASP, RELEASE = 0, 1, 2
DOWN = (180.0, 0.0, 0.0)          # gripper pointing down, as the facade's pick-up test commands it


def begin(motion, kinds, goals, eulers, phase, mask):
    """Begin primitive ``phase[i]`` on the envs of ``mask`` (envs past the end of their program are skipped)."""
    n, p = kinds.shape
    pc = phase.clamp(max=p - 1)
    ar = torch.arange(n, device=kinds.device)
    kind = kinds[ar, pc]
    live = mask & (phase < p)
    motion.move(goals[ar, pc], goal_euler=eulers[ar, pc], mask=live & (kind == MOVE))
    motion.grasp(mask=live & (kind == GRASP))
    motion.release(mask=live & (kind == RELEASE))


def run_program(motion, kinds, goals, eulers, steps=None, on_step=None):
    """Run the program from its first primitive.  ``steps=None``: until every env has finished (checked every 16 steps, the only
    synchronisation) and return the step count; otherwise exactly ``steps`` steps.  ``on_step(t, phase)`` is called after every step
    with the phase each env is in for the next one.  Returns (steps taken, phase)."""
    n, p = kinds.shape
    phase = torch.zeros(n, dtype=torch.long, device=kinds.device)
    begin(motion, kinds, goals, eulers, phase, torch.ones(n, dtype=torch.bool, device=kinds.device))
    t = 0
    while (steps is None and (t % 16 or not bool((phase >= p).all()))) or (steps is not None and t < steps):
        _, _, _, _, remaining = motion.step()
        t += 1
        done = remaining == 0
        phase = phase + done.long()
        begin(motion, kinds, goals, eulers, phase, done)
        if on_step is not None:
            on_step(t, phase)
    return t, phase


def pick_and_lift(cube: torch.Tensor, lift: float = 0.15):
    """release -> above the cube -> down to it -> grasp -> lift, for cube positions [N, 3] (float64)."""
    n, dev = cube.shape[0], cube.device
    up = lambda dz: cube + torch.tensor([0.0, 0.0, dz], dtype=torch.float64, device=dev)
    kinds = torch.tensor([RELEASE, MOVE, MOVE, GRASP, MOVE], device=dev).expand(n, 5).contiguous()
    goals = torch.stack([cube, up(0.10), up(0.0), cube, up(lift)], dim=1)
    eulers = torch.tensor(DOWN, dtype=torch.float64, device=dev).expand(n, 5, 3).contiguous()
    return kinds, goals, eulers
