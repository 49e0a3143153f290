#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched Panda step on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--task reach] [--control joints] [--envs 65536]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
  python bench.py --impl reference ...      # the CPU arm: the oracle port of the reference's PyBullet path on the host cores
  python bench.py --dump-outputs DIR ...    # also write the last timed step's outputs as DIR/<name>.npy (compare two builds)

A step = one RobotTaskEnv.step of every environment (20 physics sub-steps + controller + observation + reward, auto-reset
on success / TimeLimit), one kernel launch.  Default workload = BASELINE.json configs[1]: PandaReachJoints-v3, 65,536 envs
per GPU, sparse reward, random actions resident in HBM.  `value` is device-timed (CUDA events on the launching stream, L2
flushed between timed steps); `e2e` goes through the C-ABI call with HOST buffers (pg_step_host: H2D actions, kernel, D2H
observations/rewards inside the timed region).
"""
import argparse
import ctypes
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree, which may be read-only

METRIC = "env-steps/sec"
# `roofline.traffic` / `launches_per_step` come from profiles/kernel_traffic.json, which scripts/ncu_traffic.py writes from an
# `ncu --set full` capture of this very command (dram__bytes_read.sum + dram__bytes_write.sum of the step kernel, per launch; ncu
# flushes the caches before every replay pass, so these are cold-cache figures) -- null where no capture exists for the configuration.
PREROLL = 60          # untimed steps before any timed region: every env is past its first episode, contact states are mixed (steady state)


def kernel_traffic(task, control, envs):
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
        return d.get(f"{task}/{control}/{envs}")
    except Exception:
        return None


ENV_IDS = {"reach": "PandaReach", "push": "PandaPush", "slide": "PandaSlide", "pick_and_place": "PandaPickAndPlace", "stack": "PandaStack", "flip": "PandaFlip"}
TASK_ID = {"reach": 0, "push": 1, "slide": 2, "pick_and_place": 3, "stack": 4, "flip": 5}
# algorithmic bytes per env-step, fp32 SoA (SURVEY.md section 8d): read state+goal+action, write state+obs+ag+dg+reward+2 flags
OBS = {"reach": 6, "push": 18, "slide": 18, "pick_and_place": 19, "stack": 31, "flip": 20}
GOAL = {"reach": 3, "push": 3, "slide": 3, "pick_and_place": 3, "stack": 6, "flip": 4}
NOBJ = {"reach": 0, "push": 1, "slide": 1, "pick_and_place": 1, "stack": 2, "flip": 1}


def action_dim(task, control):
    return (3 if control == "ee" else 7) + (0 if task in ("reach", "push", "slide") else 1)


def bytes_per_step(task, control):
    state = 72 + 52 * NOBJ[task]
    g, a, o = 4 * GOAL[task], 4 * action_dim(task, control), 4 * OBS[task]
    return (state + g + a) + (state + o + g + g + 4 + 2)


def workload_name(task, control, reward, envs):
    return f"{ENV_IDS[task]}{'Joints' if control == 'joints' else ''}{'Dense' if reward == 'dense' else ''}-v3, {envs} envs/GPU, random actions, auto-reset"


# ------------------------------------------------------------------------------------------------ CPU arm (oracle port)
def oracle_lib():
    """The CPU oracle as build() left it in oracle/; when that library is missing or older than its sources, a private copy is
    compiled in a temporary directory, so that the tree stays untouched."""
    src = os.path.join(ROOT, "oracle")
    so = os.path.join(src, "libpanda_oracle.so")
    if os.path.exists(so) and all(os.path.getmtime(os.path.join(src, f)) <= os.path.getmtime(so) for f in ("panda_oracle.c", "panda_oracle.h")):
        return ctypes.CDLL(so)
    tmp = tempfile.mkdtemp(prefix="panda_oracle_")
    try:
        for f in ("Makefile", "panda_oracle.c", "panda_oracle.h"):
            shutil.copy(os.path.join(src, f), tmp)
        subprocess.run(["make", "-C", tmp], check=True, stdout=subprocess.DEVNULL)
        return ctypes.CDLL(os.path.join(tmp, "libpanda_oracle.so"))      # stays mapped after the directory is removed
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


# what PandaVecEnv.step returns (info["is_success"] is `terminated` again), written by --dump-outputs
OUTPUT_NAMES = ("observation", "achieved_goal", "desired_goal", "reward", "terminated", "truncated")
DUMP_BYTES = 63 * 10**6         # under 64 MB in all with the .npy headers


def dump_outputs(out_dir, step_out):
    """Writes one step's outputs as out_dir/<name>.npy in float32 (flags as 0 / 1), one row per env, plus env_index.npy (float64)
    with the index of each row's env.  Above DUMP_BYTES in all, the rows are a fixed sample of envs (seed 0, sorted)."""
    import numpy as np
    import torch
    obs, rew, term, trunc, _ = step_out
    arrays = dict(zip(OUTPUT_NAMES, (obs["observation"], obs["achieved_goal"], obs["desired_goal"], rew, term, trunc)))
    n = rew.shape[0]
    row_bytes = 8 + 4 * sum(a[0].numel() for a in arrays.values())
    rows = min(n, DUMP_BYTES // row_bytes)
    idx = np.arange(n) if rows == n else np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
    sel = torch.from_numpy(idx).to(rew.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.index_select(0, sel).float().cpu().numpy())
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))


class CpuPool:
    """`threads` persistent OS threads (ctypes releases the GIL), each owning one persistent oracle env for the whole run."""

    def __init__(self, lib, task, control, threads):
        from concurrent.futures import ThreadPoolExecutor
        self.lib, self.threads = lib, threads
        lib.po_bench_open.restype = ctypes.c_void_p
        lib.po_bench_open.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong]
        lib.po_bench_steps.restype = ctypes.c_double
        lib.po_bench_steps.argtypes = [ctypes.c_void_p, ctypes.c_int]
        lib.po_bench_close.argtypes = [ctypes.c_void_p]
        self.handles = [lib.po_bench_open(TASK_ID[task], 0 if control == "ee" else 1, 1 + i) for i in range(threads)]
        self.pool = ThreadPoolExecutor(max_workers=threads)
        self.run(60)                                    # the same pre-roll as the GPU arm: envs past their first episode

    def run(self, steps_per_thread):
        """Every thread advances its env by steps_per_thread env-steps; returns (env-steps/s, seconds)."""
        t0 = time.perf_counter()
        list(self.pool.map(lambda h: self.lib.po_bench_steps(h, steps_per_thread), self.handles))
        dt = time.perf_counter() - t0
        return self.threads * steps_per_thread / dt, dt

    def close(self):
        self.pool.shutdown()
        for h in self.handles:
            self.lib.po_bench_close(h)


def run_reference(args):
    """The reference's own CPU implementation of the path.  pybullet is not installable here (SURVEY.md section 8c), so this arm
    times the oracle port (fp64 C restatement of the PyBullet path, -O3) on all host cores: kind = "port"."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    lib = oracle_lib()
    pool = CpuPool(lib, args.task, args.control, cores)
    rate, _ = pool.run(50)                                                               # calibration
    total = args.steps + args.warmup
    per_thread = max(1, min(256, int(120.0 * rate / max(1, total) / cores)))            # bounded sample: whole run <= ~2 min
    for _ in range(args.warmup):
        pool.run(per_thread)
    t0 = time.perf_counter()
    for k in range(args.steps):
        pool.run(per_thread)
    dt = time.perf_counter() - t0
    pool.close()
    sample = cores * per_thread
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.task, args.control, args.reward, args.envs), "sample": f"{sample} env-steps per bench step"},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port",
                         "sample": f"{cores} persistent threads x {per_thread} env-steps per bench step, oracle/panda_oracle.c -O3 (PyBullet unavailable on this box)"},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        out = self.proc.communicate()[0]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except Exception:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def run_gpu(args):
    import numpy as np
    import torch
    import panda_lang_manip_b200 as p

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    ncyc = 8
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)                   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_leg(task, control, n, steps, warmup):
        """PREROLL + warmup untimed steps, then `steps` device-timed steps (CUDA events around each step on the launching stream, L2
        flushed between them).  Returns (env, actions, device seconds on this rank, launches, what the last timed step returned)."""
        A = action_dim(task, control)
        env = p.PandaVecEnv(task, n, reward_type=args.reward, control_type=control, device=local, seed=args.seed, env_id_offset=rank * n, auto_reset=True)
        actions = torch.rand((ncyc, n, A), device=dev, generator=gen) * 2 - 1      # synthetic actions, resident in HBM
        # steady state: spread the episode phases (all envs are created at step 0 and would otherwise walk through their episodes in
        # lock-step: contact-free early steps, TimeLimit resets in bursts) by giving every env a random age, then pre-roll
        st = env.get_state()
        st[:, -1] = torch.randint(0, env.max_episode_steps, (n,), device=dev, generator=gen).to(st.dtype)
        env.set_state(st); del st
        for w in range(PREROLL + warmup):
            env.step(actions[w % ncyc])
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        l0 = p.kernel_launches()
        for k, (a, b) in enumerate(ev):
            flush.zero_()                              # L2 flush between timed iterations (outside the event pair)
            a.record(); last = env.step(actions[(k + warmup) % ncyc]); b.record()
        barrier()
        return env, actions, sum(a.elapsed_time(b) for a, b in ev) / 1e3, p.kernel_launches() - l0, last

    n, A = args.envs, action_dim(args.task, args.control)
    sampler = ClockSampler(local) if rank == 0 else None
    t_wall0 = time.perf_counter()
    env, actions, dev_s_local, launches, last = timed_leg(args.task, args.control, n, args.steps, args.warmup)
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)                                   # rank 0's envs
    dev_s = allmax(dev_s_local)                                                     # max over ranks
    stats = torch.tensor(env.stats(), dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)   # the only data-path-adjacent collective: episode statistics (4 doubles, NCCL)
    value = world * n * args.steps / dev_s

    # end to end through the C ABI with host buffers (per env group: H2D actions, kernels, D2H observations / rewards, pipelined)
    e2e_steps = max(3, min(args.steps, 50))
    host_actions = [env.pin_host(np.ascontiguousarray(actions[i].cpu().numpy())) for i in range(ncyc)]     # pinned host inputs (the e2e contract)
    env.step_host(host_actions[0]); env.step_host(host_actions[1])
    barrier()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        env.step_host(host_actions[k % ncyc])
    torch.cuda.synchronize(dev)
    e2e_local = time.perf_counter() - t0
    e2e_s = allmax(e2e_local)
    per_rank = torch.zeros(world, dtype=torch.float64, device=dev); per_rank[rank] = e2e_local
    if world > 1:
        dist.all_reduce(per_rank, op=dist.ReduceOp.SUM)
    e2e_value = world * n * e2e_steps / e2e_s
    h2d = n * A * 4
    d2h = n * (OBS[args.task] + 2 * GOAL[args.task] + 1) * 4 + 2 * n
    diverged = env.diverged(); overflows = env.contact_overflows()
    env.close(); del actions

    # BASELINE.json's metric and configs name more workloads than the headline one: the default run also reports them, each at its
    # BASELINE batch size per GPU and timed the same way (PREROLL, device events, L2 flush).  Informational: the headline `value`
    # is the workload named in `config`.
    also = None
    if args.task == "reach" and args.control == "joints" and not args.no_her:
        also = []
        for task2, ctrl2, n2, k2 in (("reach", "ee", 65536, 30), ("pick_and_place", "ee", 32768, 30), ("push", "ee", 65536, 20), ("slide", "ee", 65536, 20), ("stack", "ee", 65536, 15)):
            sec2, err2 = -1.0, None
            try:                          # rank-local work only inside the try: a failure on one rank must not leave the others in a collective
                env2, act2, sec2, _, _ = timed_leg(task2, ctrl2, n2, k2, 3)
                env2.close(); del act2
            except Exception as exc:
                err2 = repr(exc)
            t2 = torch.tensor([sec2, 1.0 if err2 is None else 0.0], dtype=torch.float64, device=dev)
            if world > 1:
                tmax = t2.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)       # slowest rank
                tmin = t2.clone(); dist.all_reduce(tmin, op=dist.ReduceOp.MIN)       # did every rank succeed?
                t2 = torch.stack([tmax[0], tmin[1]])
            if float(t2[1].item()) == 1.0 and float(t2[0].item()) > 0:
                bps2 = bytes_per_step(task2, ctrl2)
                also.append({"workload": workload_name(task2, ctrl2, args.reward, n2), "value": world * n2 * k2 / float(t2[0].item()), "unit": "env-steps/s",
                             "ms_per_step": 1e3 * float(t2[0].item()) / k2, "steps": k2, "preroll": PREROLL, "envs_per_gpu": n2,
                             "hbm_frac": bps2 * n2 * k2 / float(t2[0].item()) / 1e9 / 6541.8})
            else:
                also.append({"workload": workload_name(task2, ctrl2, args.reward, n2), "error": err2 or "failed on another rank"})

    # HER relabelling kernel (the one genuinely HBM-bound kernel of the path): compute_reward on M transitions
    her = None
    if rank == 0 and not args.no_her:
        her = {}
        for name, task, G, M in (("stack_1M_rows_6d (BASELINE configs[4], L2-resident)", "stack", 6, 1 << 20), ("reach_32M_rows_3d (HBM-resident)", "reach", 3, 1 << 25)):
            ag = torch.rand((M, G), device=dev); dg = torch.rand((M, G), device=dev)
            for _ in range(3):
                p.compute_reward(task, "sparse", ag, dg)
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
            for a, b in evs:
                if M < (1 << 24):
                    flush.zero_()
                a.record(); p.compute_reward(task, "sparse", ag, dg); b.record()
            torch.cuda.synchronize(dev)
            ms = sorted(a.elapsed_time(b) for a, b in evs)[len(evs) // 2]
            nbytes = M * (2 * G * 4 + 4)
            her[name] = {"transitions_per_s": M / (ms / 1e3), "ms": ms, "achieved_gbs": nbytes / (ms / 1e3) / 1e9, "bytes_per_transition": 2 * G * 4 + 4}
            del ag, dg
        # fused relabel (gather + compute_reward): 1 M transitions sampled from a 16 M-row replay buffer of 6-D goals (HBM-resident), once with
        # dense 24-byte rows (768 MB of goals: a row straddles two 32-byte sectors half the time) and once with rows padded to 32 bytes
        # (1 GB: every gathered row is exactly one sector)
        R, M, G = 1 << 24, 1 << 20, 6
        src = torch.randint(0, R, (M,), device=dev); gs = torch.where(torch.rand(M, device=dev) < 0.8, torch.randint(0, R, (M,), device=dev), torch.full((M,), -1, device=dev))
        for label, pitch, sectors in (("dense_24B_rows", G, 1.5), ("padded_32B_rows", 8, 1.0)):
            nag = torch.rand((R, pitch), device=dev); dgb = torch.rand((R, pitch), device=dev)
            for _ in range(3):
                p.her_relabel("stack", "sparse", nag[:, :G], dgb[:, :G], src, gs)
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
            for a, b in evs:
                flush.zero_()
                a.record(); p.her_relabel("stack", "sparse", nag[:, :G], dgb[:, :G], src, gs); b.record()
            torch.cuda.synchronize(dev)
            ms = sorted(a.elapsed_time(b) for a, b in evs)[len(evs) // 2]
            nbytes = M * (16 + 3 * G * 4 + 4)
            sector_bytes = M * (16 + 2 * 32 * sectors + G * 4 + 4)      # what DRAM moves: index pair, two gathered rows in 32-byte sectors, goal + reward out
            her[f"her_relabel_1M_of_16M_rows_6d_{label} (gather + reward, includes the two output allocations)"] = {
                "transitions_per_s": M / (ms / 1e3), "ms": ms, "achieved_gbs": nbytes / (ms / 1e3) / 1e9, "bytes_per_transition": 16 + 3 * G * 4 + 4,
                "achieved_gbs_in_sector_terms": sector_bytes / (ms / 1e3) / 1e9, "sector_bytes_per_transition": 16 + 2 * 32 * sectors + G * 4 + 4,
                "note": "random row gather: DRAM moves 32-byte sectors, so the sector figure is the one to hold against the HBM peak"}
            if label == "dense_24B_rows":
                # the same relabelling with indices as a replay buffer produces them (a future goal lies in the transition's own episode, at
                # most 100 rows behind it) and an index-sorted batch (her_sample_indices): near-sequential gathers instead of random sectors
                gen2 = torch.Generator(device=dev).manual_seed(99)
                for lab2, srt in (("episode_local_goals_unsorted_batch", False), ("episode_local_goals_index_sorted_batch", True)):
                    s2, g2 = p.her_sample_indices(R, M, 100, 0.8, device=dev, generator=gen2, sort=srt)
                    for _ in range(3):
                        p.her_relabel("stack", "sparse", nag[:, :G], dgb[:, :G], s2, g2)
                    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
                    for a, b in evs:
                        flush.zero_()
                        a.record(); p.her_relabel("stack", "sparse", nag[:, :G], dgb[:, :G], s2, g2); b.record()
                    torch.cuda.synchronize(dev)
                    ms2 = sorted(a.elapsed_time(b) for a, b in evs)[len(evs) // 2]
                    t0s = time.perf_counter(); torch.sort(s2); torch.cuda.synchronize(dev); sort_ms = (time.perf_counter() - t0s) * 1e3
                    her[f"her_relabel_1M_of_16M_rows_6d_dense_24B_rows_{lab2}"] = {
                        "transitions_per_s": M / (ms2 / 1e3), "ms": ms2, "achieved_gbs": nbytes / (ms2 / 1e3) / 1e9, "bytes_per_transition": 16 + 3 * G * 4 + 4,
                        "note": "algorithmic bytes; torch.sort of the 1 M sampled indices (outside the timed region) took %.3f ms wall" % sort_ms}
            del nag, dgb
        del src, gs
    # analytic depth / point-cloud renderer (SURVEY 8f rank 4): 256 PickAndPlace envs x the reference's 480 x 480 camera (pybullet.py:149-160),
    # depth + colour + deprojected points + validity = 21 B written per pixel
    render = None
    if rank == 0 and not args.no_her:
        try:
            renv = p.PandaVecEnv("pick_and_place", 256, control_type="ee", device=local)
            for _ in range(2):
                out = renv.render(width=480, height=480)
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
            for a, b in evs:
                flush.zero_()
                a.record(); out = renv.render(width=480, height=480); b.record()
            torch.cuda.synchronize(dev)
            ms = sorted(a.elapsed_time(b) for a, b in evs)[len(evs) // 2]
            npix = 256 * 480 * 480
            render = {"workload": "256 envs x 480 x 480, depth + rgba + points + valid", "ms": ms, "pixels_per_s": npix / (ms / 1e3), "bytes_per_pixel": 21,
                      "achieved_gbs": npix * 21 / (ms / 1e3) / 1e9, "valid_fraction": float(out["valid"].float().mean().item()),
                      "note": "includes the output allocations of PandaVecEnv.render and the per-env primitive set-up launch"}
            renv.close(); del out
        except Exception as exc:
            render = {"error": repr(exc)}
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        bps = bytes_per_step(args.task, args.control)
        kernel_s = dev_s / args.steps
        achieved = bps * n / kernel_s / 1e9
        kt = kernel_traffic(args.task, args.control, n) or {}
        line = {
            "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.task, args.control, args.reward, n), "envs_per_gpu": n, "sub_steps_per_step": 20,
                       "preroll_steps": PREROLL, "l2": "flushed between timed steps (256 MiB memset outside the event pair)", "parallelism": f"env-sharded x{world}, no data-path collective"},
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps, "api": "pg_step_host (C ABI, host buffers)",
                    "per_rank_s": [float(x) for x in per_rank.tolist()], "device_s_for_the_same_steps": dev_s * e2e_steps / args.steps},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (kt.get("dram_bytes_per_launch") * kt.get("step_kernel_launches_per_step")) if kt else None,
                         "kernel": "step_kernel", "launches_per_step": kt.get("launches_per_step") if kt else None, "traffic_source": kt.get("source") if kt else None,
                         "ncu": {k: kt.get(k) for k in ("fma_pipe_pct", "issue_active_pct", "threads_per_instruction", "warps_active_pct", "kernel_us_under_ncu")} if kt else None,
                         "bytes_per_env_step": bps, "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s",
                         "note": "latency/issue-bound kernel (~1 MFLOP of serial dynamics per env-step): the HBM fraction is structurally tiny, see DESIGN.md"},
            "also": also,
            "her_compute_reward": her,
            "render": render,
            "clocks": clocks,
            "wall_s_timed_leg": t_wall,
            "episode_stats": {"diverged_env_steps": diverged, "contact_candidates_dropped_at_cap": overflows, "episodes": stats[0].item(), "success_rate": (stats[1] / stats[0]).item() if stats[0].item() > 0 else None,
                              "mean_return": (stats[2] / stats[0]).item() if stats[0].item() > 0 else None},
        }
        if render and "achieved_gbs" in render:
            render["frac_of_measured_hbm"] = render["achieved_gbs"] / peak
        if her:
            for v in her.values():
                v["frac_of_measured_hbm"] = v["achieved_gbs"] / peak
                if "achieved_gbs_in_sector_terms" in v:
                    v["frac_of_measured_hbm_in_sector_terms"] = v["achieved_gbs_in_sector_terms"] / peak
            # what DRAM really moved for these kernels (ncu dram__bytes, profiles/her_kernel_traffic.json written by scripts/her_traffic.py): a random
            # 24-byte row gather costs one or two 64-byte DRAM accesses, so the gather kernel is HBM-bound at a small algorithmic fraction
            try:
                traffic = json.load(open(os.path.join(ROOT, "profiles", "her_kernel_traffic.json")))
                match = {"stack_1M_rows_6d": "stack_1M_rows_6d", "reach_32M_rows_3d": "reach_32M_rows_3d", "dense_24B_rows (": "her_relabel_random_indices",
                         "unsorted_batch": "her_relabel_episode_local_goals_unsorted_batch", "index_sorted_batch": "her_relabel_episode_local_goals_index_sorted_batch"}
                for name, v in her.items():
                    for frag, key in match.items():
                        if frag in name and key in traffic:
                            t = traffic[key]
                            v["traffic"] = t["dram_bytes_read"] + t["dram_bytes_write"]
                            v["frac_of_measured_hbm_by_dram_traffic"] = v["traffic"] / (v["ms"] / 1e3) / 1e9 / peak
                            v["traffic_source"] = t["source"]
            except Exception:
                pass
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            lib = oracle_lib()
            pool = CpuPool(lib, args.task, args.control, cores)
            rate, _ = pool.run(25)
            per_thread = max(25, int(12.0 * rate / cores))                      # ~12 s of CPU work
            cpu_value, cpu_dt = pool.run(per_thread)
            pool.close()
            line["cpu_baseline"] = {"value": cpu_value, "unit": "env-steps/s", "cores": cores, "kind": "port",
                                    "sample": f"{cores} persistent threads x {per_thread} env-steps of the same workload ({cpu_dt:.1f} s), oracle/panda_oracle.c -O3 (PyBullet unavailable)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--task", default="reach", choices=list(TASK_ID))
    ap.add_argument("--control", default="joints", choices=["ee", "joints"])
    ap.add_argument("--reward", default="sparse", choices=["sparse", "dense"])
    ap.add_argument("--envs", type=int, default=65536, help="environments per GPU")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-her", action="store_true", help="skip the HER compute_reward measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (rank 0's envs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
