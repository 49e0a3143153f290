"""The callers on the learner side of the step path (SURVEY §8f ranks 2-3), on the GPU:
HER relabelling fused with compute_reward against the reference's arithmetic (numpy gather + utils.distance + compute_reward, the
code path stable-baselines3's HerReplayBuffer drives in examples/train_push.py), the batched look-ahead search of
docs/usage/save_restore_state.rst against the same loop written out by hand, and the Gymnasium / SB3 vector-env adapters."""
import numpy as np
import pytest

from tests.oracle_util import reward_np

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("task,g", [("reach", 3), ("push", 3), ("stack", 6), ("flip", 4)])
@pytest.mark.parametrize("reward_type", ["sparse", "dense"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_her_relabel_matches_reference_arithmetic(task, g, reward_type, dtype):
    import panda_lang_manip_b200 as p
    rng = np.random.default_rng(5)
    R, M = 5000, 20011
    dg = rng.uniform(-0.2, 0.2, (R, g)).astype(dtype)
    nag = (dg + rng.normal(0, {"stack": 0.05, "flip": 0.3}.get(task, 0.03), (R, g))).astype(dtype)
    if task == "flip":
        dg /= np.linalg.norm(dg, axis=-1, keepdims=True); nag /= np.linalg.norm(nag, axis=-1, keepdims=True)
    src = rng.integers(0, R, M)
    gsrc = np.where(rng.uniform(size=M) < 0.8, rng.integers(0, R, M), -1)
    gsrc[:7] = src[:7]                                            # goal == own next achieved goal: d = 0 -> reward -0.0 / success
    new_dg, rew, ag = p.her_relabel(task, reward_type, torch.from_numpy(nag).cuda(), torch.from_numpy(dg).cuda(), torch.from_numpy(src).cuda(),
                                    torch.from_numpy(gsrc).cuda(), return_achieved=True)
    want_dg = np.where((gsrc >= 0)[:, None], nag[np.maximum(gsrc, 0)], dg[src])
    assert new_dg.cpu().numpy().tobytes() == want_dg.tobytes() and ag.cpu().numpy().tobytes() == nag[src].tobytes()
    want_r, _ = reward_np(task, reward_type, nag[src], want_dg)
    got = rew.cpu().numpy()
    if task == "flip":      # np.inner's BLAS summation order is not reproducible bit-for-bit (DESIGN §6): 1 ulp
        assert np.allclose(got, want_r, rtol=0, atol=2e-7 if dtype == np.float32 else 1e-7)
    else:
        assert got.tobytes() == want_r.tobytes()
    # the same gather from goal arrays stored with padded (32-byte for fp32) rows, and from a misaligned dense view (scalar-load path)
    pad = 8 if dtype == np.float32 else 6 + (g % 2)
    nag_p = torch.zeros((R, pad), dtype=torch.from_numpy(nag).dtype, device="cuda"); dg_p = torch.zeros_like(nag_p)
    nag_p[:, :g] = torch.from_numpy(nag).cuda(); dg_p[:, :g] = torch.from_numpy(dg).cuda()
    p_dg, p_rew, p_ag = p.her_relabel(task, reward_type, nag_p[:, :g], dg_p[:, :g], torch.from_numpy(src).cuda(), torch.from_numpy(gsrc).cuda(), return_achieved=True)
    assert torch.equal(p_dg, new_dg) and torch.equal(p_ag, ag) and p_rew.cpu().numpy().tobytes() == got.tobytes()
    flat = torch.zeros(R * g + 1, dtype=nag_p.dtype, device="cuda"); flat2 = torch.zeros_like(flat)
    flat[1:] = torch.from_numpy(nag).cuda().reshape(-1); flat2[1:] = torch.from_numpy(dg).cuda().reshape(-1)
    u_dg, u_rew = p.her_relabel(task, reward_type, flat[1:].view(R, g), flat2[1:].view(R, g), torch.from_numpy(src).cuda(), torch.from_numpy(gsrc).cuda())
    assert torch.equal(u_dg, new_dg) and u_rew.cpu().numpy().tobytes() == got.tobytes()
    # empty batch
    e_dg, e_r = p.her_relabel(task, reward_type, torch.from_numpy(nag).cuda(), torch.from_numpy(dg).cuda(), torch.zeros(0, dtype=torch.long, device="cuda"),
                              torch.zeros(0, dtype=torch.long, device="cuda"))
    assert e_dg.shape == (0, g) and e_r.shape == (0,)


def test_future_goal_indices_stay_inside_the_episode():
    import panda_lang_manip_b200 as p
    gen = torch.Generator(device="cuda").manual_seed(0)
    n_ep, T, M = 200, 50, 100000
    src = torch.randint(0, n_ep * T, (M,), device="cuda", generator=gen)
    start = (src // T) * T
    length = torch.full_like(src, T)
    gi = p.future_goal_indices(start, length, src, her_ratio=0.8, generator=gen)
    rel = gi >= 0
    assert abs(rel.float().mean().item() - 0.8) < 0.01
    assert bool(((gi >= src) & (gi < start + T))[rel].all())
    last = src == start + T - 1
    assert bool((gi[last & rel] == src[last & rel]).all())          # the last step of an episode can only pick itself


def test_lookahead_equals_the_documented_loop():
    """docs/usage/save_restore_state.rst:8-41, batched: the best of K sampled actions per env, then one committed step."""
    import panda_lang_manip_b200 as p
    n, K = 96, 5
    env = p.PandaVecEnv("reach", n, reward_type="dense", control_type="ee", seed=2, auto_reset=False)
    ref = p.PandaVecEnv("reach", n, reward_type="dense", control_type="ee", seed=2, auto_reset=False)
    gen = torch.Generator(device="cuda").manual_seed(3)
    for it in range(3):
        cand = torch.rand((K, n, 3), device="cuda", generator=gen) * 2 - 1
        # by hand on the twin env
        sid = ref.save_state()
        rewards = []
        for k in range(K):
            ref.restore_state(sid)
            rewards.append(ref.step(cand[k])[1].clone())
        rewards = torch.stack(rewards)
        best_k = rewards.argmax(0)
        ref.restore_state(sid); ref.remove_state(sid)
        best_a = cand[best_k, torch.arange(n, device="cuda")]
        ref_out = ref.step(best_a)
        a, r, out = env.lookahead(cand)
        assert torch.equal(a, best_a) and torch.equal(r, rewards.max(0).values)
        assert torch.equal(out[0]["observation"], ref_out[0]["observation"]) and torch.equal(out[1], ref_out[1])
        assert torch.equal(env.get_state(), ref.get_state())
    # commit=False leaves the state untouched
    before = env.get_state()
    env.lookahead(torch.rand((2, n, 3), device="cuda", generator=gen), commit=False)
    assert torch.equal(env.get_state(), before)
    with pytest.raises(ValueError):
        env.lookahead(torch.zeros((2, n + 1, 3), device="cuda"))
    env.close(); ref.close()


def test_gymnasium_vector_env_interface():
    from panda_lang_manip_b200.adapters import PandaGymVectorEnv
    n = 40
    venv = PandaGymVectorEnv("push", n, seed=1)
    obs, info = venv.reset(seed=7)
    assert obs["observation"].shape == (n, 18) and obs["observation"].dtype == np.float32 and info == {}
    assert venv.single_action_space.shape == (3,) and venv.action_space.shape == (n, 3) and venv.observation_space["desired_goal"].shape == (n, 3)
    first_goal = obs["desired_goal"].copy()
    rng = np.random.default_rng(0)
    age, n_trunc = np.zeros(n, int), 0
    for t in range(1, 51):
        obs, rew, term, trunc, infos = venv.step(rng.uniform(-1, 1, (n, 3)).astype(np.float32))
        assert rew.shape == (n,) and term.dtype == np.bool_ and trunc.dtype == np.bool_
        done = term | trunc
        age += 1
        assert np.array_equal(trunc, age == 50)                     # TimeLimit of 50 steps per episode (__init__.py:18)
        age[done] = 0; n_trunc += int(trunc.sum())
        if done.any():
            assert np.array_equal(infos["_final_observation"], done)
            i = int(np.flatnonzero(done)[0])
            fo = infos["final_observation"][i]
            assert set(fo) == {"observation", "achieved_goal", "desired_goal"}
            if (~done).any():
                assert infos["final_observation"][np.flatnonzero(~done)[0]] is None
            # same-step auto-reset: the returned observation is the new episode's first one (robot back at its neutral pose, a new goal)
            assert np.allclose(obs["observation"][i, :3], [0.0384, 0.0, 0.1974], atol=2e-3) and np.abs(obs["observation"][i, 3:6]).max() < 1e-6
    assert n_trunc > n // 2
    assert not np.array_equal(obs["desired_goal"], first_goal)
    # seeded determinism of the device sampler (test/seed_test.py, batched)
    o1, _ = venv.reset(seed=11); o2, _ = venv.reset(seed=11)
    assert all(np.array_equal(o1[k], o2[k]) for k in o1)
    r = venv.call("compute_reward", obs["achieved_goal"], obs["desired_goal"], {})
    assert r.tobytes() == reward_np("push", "sparse", obs["achieved_goal"], obs["desired_goal"])[0].tobytes()
    venv.close()
    tv = PandaGymVectorEnv("reach", 8, output="torch")
    o, _ = tv.reset()
    o, rew, term, trunc, infos = tv.step(torch.zeros((8, 3), device="cuda"))
    assert o["observation"].is_cuda and rew.is_cuda and term.dtype == torch.bool
    tv.close()


def test_sb3_vec_env_interface():
    from panda_lang_manip_b200.adapters import PandaSB3VecEnv
    n = 24
    venv = PandaSB3VecEnv("pick_and_place", n, reward_type="dense", seed=0)
    obs = venv.reset()
    assert obs["observation"].shape == (n, 19) and venv.action_space.shape == (4,) and venv.num_envs == n
    rng = np.random.default_rng(1)
    for t in range(1, 51):
        venv.step_async(rng.uniform(-1, 1, (n, 4)).astype(np.float32))
        obs, rew, dones, infos = venv.step_wait()
        assert len(infos) == n and rew.dtype == np.float32 and dones.dtype == np.bool_
        for i in np.flatnonzero(dones):
            assert "terminal_observation" in infos[i] and infos[i]["terminal_observation"]["observation"].shape == (19,)
            assert infos[i]["TimeLimit.truncated"] == (not infos[i]["is_success"])
    assert dones.sum() > n // 2
    # HerReplayBuffer's call: env_method("compute_reward", next_achieved_goal, new_goals, infos, indices=[0])[0]
    ag = rng.uniform(-0.2, 0.2, (1000, 3)).astype(np.float32); dg = rng.uniform(-0.2, 0.2, (1000, 3)).astype(np.float32)
    r = venv.env_method("compute_reward", ag, dg, [{}] * 1000, indices=[0])[0]
    assert r.tobytes() == reward_np("pick_and_place", "dense", ag, dg)[0].tobytes()
    assert venv.get_attr("reward_type") == ["dense"] * n and venv.env_is_wrapped(object) == [False] * n
    assert venv.seed(5)[:2] == [5, 6]
    venv.close()


def test_host_reward_staging_grows_only():
    """pg_compute_reward_host / pg_is_success_host stage through per-device buffers that only grow: once a size has been served,
    calls of that size allocate nothing (pg_host_stage_allocations is unchanged) and a larger call grows them.  Page-locked and
    pageable host arrays give the same results."""
    from panda_lang_manip_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(4)

    def call(m, pinned):
        ag, dg = rng.uniform(-0.2, 0.2, (2, m, 3))
        rew, ok = np.empty(m, np.float32), np.empty(m, np.uint8)
        if pinned:
            ag, dg, rew, ok = (torch.from_numpy(x).pin_memory().numpy() for x in (ag, dg, rew, ok))
        _lib.check(lib.pg_compute_reward_host(0, 1, 0.05, ag.ctypes.data, dg.ctypes.data, rew.ctypes.data, m, 1, 0))
        _lib.check(lib.pg_is_success_host(0, 0.05, ag.ctypes.data, dg.ctypes.data, ok.ctypes.data, m, 1, 0))
        want_r, want_s = reward_np("reach", "dense", ag, dg)
        assert rew.tobytes() == want_r.tobytes() and np.array_equal(ok, want_s)

    call(10_000, False)
    before = lib.pg_host_stage_allocations()
    for pinned in (False, True, False, True):
        call(10_000, pinned)
    assert lib.pg_host_stage_allocations() == before
    call(1 << 21, False)                # larger than any other host reward call of the suite
    assert lib.pg_host_stage_allocations() > before


@pytest.mark.gpu
def test_index_sorted_her_batch_is_the_same_set_of_transitions():
    """her_sample_indices(sort=True): ascending src, goals inside the transition's own episode, and the relabelled batch is what the unsorted
    one is, row for row, after undoing the order."""
    import torch
    import panda_lang_manip_b200 as p
    R, M, L = 50_000, 20_000, 50
    gen = torch.Generator(device="cuda").manual_seed(5)
    src, gs = p.her_sample_indices(R, M, L, 0.8, generator=gen, sort=True)
    assert bool((src[1:] >= src[:-1]).all())
    fut = gs >= 0
    assert bool(((gs[fut] >= src[fut]) & (gs[fut] // L == src[fut] // L)).all())
    assert 0.75 < fut.float().mean().item() < 0.85
    nag = torch.rand((R, 3), device="cuda"); dg = torch.rand((R, 3), device="cuda")
    d1, r1 = p.her_relabel("push", "sparse", nag, dg, src, gs)
    perm = torch.randperm(M, device="cuda")
    d2, r2 = p.her_relabel("push", "sparse", nag, dg, src[perm], gs[perm])
    assert torch.equal(d1[perm], d2) and torch.equal(r1[perm], r2)

