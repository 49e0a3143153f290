"""Cost of the contact report: device time of PandaVecEnv.step with contact_report off and on, same seed, same actions.

Each configuration builds the two envs, gives every env a random episode age and runs bench.py's pre-roll on both, then alternates
blocks of BLOCK timed steps (off, on, off, on, ...) so that both arms see the same machine state; CUDA events around each step on the
launching stream, L2 flushed (256 MiB memset) between steps outside the event pair, as bench.py does.  Prints one JSON line per
configuration and, with --out, writes them all to a JSON file together with the GPU's name and power limit read in the same run.

    python scripts/contact_report_bench.py --rounds 6 --out profiles/contact_report_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import panda_lang_manip_b200 as p  # noqa: E402
from bench import PREROLL  # noqa: E402

CONFIGS = [("reach", "joints", 65536), ("pick_and_place", "joints", 32768), ("stack", "joints", 65536)]
BLOCK = 20


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:          # the measurement stands without it, but says so
        info["power_limit_w"] = f"unavailable ({e})"
    return info


def measure(task, control, n, rounds):
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(1234)
    A = p.PandaVecEnv(task, 1, control_type=control).action_dim
    actions = torch.rand((8, n, A), device=dev, generator=gen) * 2 - 1
    envs = {"off": p.PandaVecEnv(task, n, control_type=control, seed=0), "on": p.PandaVecEnv(task, n, control_type=control, seed=0, contact_report=True)}
    age = torch.randint(0, envs["off"].max_episode_steps, (n,), device=dev, generator=gen)
    for e in envs.values():
        st = e.get_state(); st[:, -1] = age.to(st.dtype); e.set_state(st)
        for w in range(PREROLL):
            e.step(actions[w % 8])
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ms = {"off": [], "on": []}
    k = {"off": PREROLL, "on": PREROLL}
    for r in range(rounds):
        for arm in ("off", "on"):
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(BLOCK)]
            for a, b in ev:
                flush.zero_()
                a.record(); envs[arm].step(actions[k[arm] % 8]); b.record()
                k[arm] += 1
            torch.cuda.synchronize(dev)
            ms[arm].append(sum(a.elapsed_time(b) for a, b in ev) / BLOCK)
    rep = envs["on"].contacts()
    cnt = rep["count"].float()
    assert torch.equal(envs["on"].obs, envs["off"].obs)          # the report changes nothing else
    for e in envs.values():
        e.close()
    off, on = np.array(ms["off"]), np.array(ms["on"])
    return {"task": task, "control": control, "envs": n, "timed_steps_per_arm": rounds * BLOCK, "block": BLOCK, "preroll": PREROLL,
            "ms_per_step_off": float(np.median(off)), "ms_per_step_on": float(np.median(on)),
            "overhead_pct": float(100 * (np.median(on) / np.median(off) - 1)),
            "block_ms_off": [round(float(x), 4) for x in off], "block_ms_on": [round(float(x), 4) for x in on],
            "spread_pct_off": float(100 * (off.max() - off.min()) / np.median(off)), "spread_pct_on": float(100 * (on.max() - on.min()) / np.median(on)),
            "mean_contacts_per_env": float(cnt.mean()), "report_bytes_written_per_step": int(cnt.sum().item()) * 64 + n}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=6, help="off / on blocks of %d steps per arm" % BLOCK)
    ap.add_argument("--out", help="JSON file for all configurations")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("contact_report_bench.py needs a CUDA device")
    res = {"gpu": gpu_info(), "configs": []}
    for task, control, n in CONFIGS:
        line = measure(task, control, n, args.rounds)
        res["configs"].append(line)
        print(json.dumps(line), flush=True)
    print(json.dumps(res["gpu"]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
