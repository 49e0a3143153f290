"""SURVEY section 8 row f4: the analytic depth / point-cloud renderer (pg_render) against the numpy oracle (oracle/render_oracle.py),
scene by scene: depth buffer, segmentation, the reference's deprojection and its filters, and the facade's PyBullet.render tuple."""
import numpy as np
import pytest

from oracle import render_oracle as ro

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

LINK_BOX = [([0, -0.04, -0.05], [0.11, 0.13, 0.25]), ([0, -0.04, 0.06], [0.11, 0.25, 0.13]), ([0.01, 0.01, -0.05], [0.19, 0.15, 0.18]), ([-0.03, 0.03, 0.02], [0.19, 0.18, 0.15]),
            ([0, 0.04, -0.12], [0.11, 0.19, 0.32]), ([0.04, 0, 0], [0.20265085784266038, 0.13, 0.12]), ([0, 0, 0.08], [0.11, 0.11, 0.10])]
RB = {8: ([0, 0, 0.021], [0.032, 0.102, 0.045]), 9: ([0, 0.0105, 0.027], [0.0105, 0.0105, 0.027]), 10: ([0, -0.0105, 0.027], [0.0105, 0.0105, 0.027])}


def _quat_R(q):
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)], [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)], [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def _scene_prims(env, i, task):
    """The primitive list the kernel builds, rebuilt independently from the state (free bodies) and from getLinkState-style link poses
    with computeForwardKinematics (pg_get_ee_pose-equivalent: the oracle's FK on the fresh joint state), and that FK's EE (link 11) pose."""
    from tests.oracle_util import OracleSim
    st = env.get_state()[i].cpu().numpy()
    slide = task == "slide"
    prims = [("box", 1, [0, 0, -0.41], np.eye(3), [3, 3, 0.01]),
             ("box", 2, [(-0.1 if slide else -0.3), 0, -0.2], np.eye(3), [0.7 if slide else 0.55, 0.35, 0.2])]
    nobj = {"reach": 0, "stack": 2}.get(task, 1)
    for o in range(nobj):
        b = st[18 + 13 * o:18 + 13 * o + 7]
        prims.append(("cyl" if slide else "box", 3 + o, b[:3], _quat_R(b[3:7]), [0.03, 0.03, 0.015] if slide else [0.02, 0.02, 0.02]))
    base = np.array([-0.6, 0.0, 0.0])
    prims.append(("box", 5, base + [-0.04, 0, 0.07], np.eye(3), [0.11, 0.1, 0.07]))
    s = OracleSim(base=tuple(base))
    for d, l in enumerate([0, 1, 2, 3, 4, 5, 6, 9, 10]):
        s.reset_joint(l, st[d])                                      # resetJointState refreshes the link cache: fresh FK
    for l in list(range(7)) + [8, 9, 10]:
        p, q, _, _ = s.link_state(l)                                 # CoM frame pose
        R = _quat_R(q)
        c, box = (LINK_BOX[l][0], [0.5 * x for x in LINK_BOX[l][1]]) if l < 7 else RB[l]
        com = np.array(LINK_BOX[l][0]) if l < 7 else np.array({8: [0, 0, 0.04], 9: [0, 0.01, 0.02], 10: [0, -0.01, 0.02]}[l])
        origin = p - R @ com                                         # link frame origin
        prims.append(("box", 6 + l, origin + R @ np.array(c), R, box))
    ee_p, ee_q, _, _ = s.link_state(11)
    s.close()
    return prims, np.concatenate([ee_p, ee_q])


RENDER_TASKS = ["reach", "push", "slide", "stack"]


@pytest.mark.parametrize("task,precision", [pytest.param(t, "f32", id=t) for t in RENDER_TASKS] + [pytest.param(t, "f64", id=f"{t}-f64") for t in RENDER_TASKS])
def test_render_matches_the_oracle(task, precision):
    import panda_lang_manip_b200 as p
    n, W, H = 3, 160, 120
    env = p.PandaVecEnv(task, n, control_type="joints", seed=4, auto_reset=False, precision=precision)
    g = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(6):
        env.step(torch.rand((n, env.action_dim), device="cuda", generator=g) * 2 - 1)
    cam = dict(target_position=(-0.1, 0.0, 0.05), distance=1.1, yaw=35.0, pitch=-32.0, roll=0.0)
    out = env.render(W, H, crop=True, segmentation=True, **cam)
    assert out["depth"].shape == (n, H, W) and out["rgb"].shape == (n, H, W, 3) and out["points"].shape == (n, H, W, 3)
    ee = env.ee_pose().cpu().numpy()
    for i in range(n):
        prims, ee_ref = _scene_prims(env, i, task)
        assert np.abs(ee[i, :3] - ee_ref[:3]).max() < 1e-5, (ee[i], ee_ref)
        assert min(np.abs(ee[i, 3:] - ee_ref[3:]).max(), np.abs(ee[i, 3:] + ee_ref[3:]).max()) < 1e-5, (ee[i], ee_ref)    # q and -q: one rotation
        d, seg, pts, valid = ro.render(prims, W, H, target=cam["target_position"], distance=cam["distance"], yaw=cam["yaw"], pitch=cam["pitch"], roll=cam["roll"], crop=True)
        gd, gs, gp, gv = out["depth"][i].cpu().numpy(), out["segmentation"][i].cpu().numpy(), out["points"][i].cpu().numpy(), out["valid"][i].cpu().numpy()
        same = gs == seg
        assert same.mean() > 0.995, (task, i, same.mean())            # silhouette pixels may fall on either side in float32
        assert np.abs(gd - d)[same].max() < 2e-5, np.abs(gd - d)[same].max()
        both = same & gv & valid
        assert (gv == valid)[same].mean() > 0.998 and both.sum() > 1000
        assert np.abs(gp[both] - pts[both]).max() < 5e-4
        assert np.isnan(gp[~gv]).all()
        for body in (2, 5) + ((3,) if task != "reach" else ()):      # table, robot base and the object are in the picture
            assert (gs == body).sum() > 5, (task, body)
    env.close()


def test_facade_render_returns_the_reference_tuple():
    """reference pybullet.py:149-264: (rgb, depth, points, colors, pixels_2d, waypoints_proj) with the reference's defaults."""
    from panda_lang_manip_b200.panda_gym.envs import PandaPickAndPlaceEnv
    env = PandaPickAndPlaceEnv()
    env.reset(seed=1)
    rgb, depth, points, colors, pixels_2d, wps = env.sim.render(width=240, height=240, waypoints=[[0.0, 0.0, 0.0]])
    assert rgb.shape == (240, 240, 3) and rgb.dtype == np.uint8 and depth.shape == (240, 240)
    assert len(points) == len(colors) == len(pixels_2d) > 1000 and points.shape[1] == 3
    assert (points[:, 2] > 0).all() and (points[:, 2] < 0.67).all() and (points[:, 0] > -0.5).all() and (points[:, 0] < 0.2).all()
    assert abs(wps[0][0] - 120) <= 1 and abs(wps[0][1] - 120) <= 1                  # the camera target projects to the image centre
    # deproject() of the kept pixels reproduces the point list (the reference's own consistency between render and deproject)
    _, _, T = env.sim.get_cam2world_transforms(240, 240)
    px = pixels_2d.astype(int)
    again = env.sim.deproject(depth, px, T, 240, 240)
    assert np.allclose(again, points, atol=2e-3)
    obj = env.sim.get_base_position("object")
    assert np.linalg.norm(points - obj, axis=1).min() < 0.04                         # the cube is in the cloud
    env.close()
