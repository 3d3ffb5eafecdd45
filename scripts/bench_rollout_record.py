"""Cost of recording a rollout (BatchedCAVEnv.rollout(..., record=every field)) against the plain rollout, on one GPU.

    python scripts/bench_rollout_record.py [--reps 10] [--steps 20] [--envs 1048576] [--out FILE]

Workloads: pedestrians (2 bodies) and bus stop (5 bodies) with their on-device agents, 1,048,576 envs, 20-step windows,
fp64 and fp32, 200 steps into their episodes.  The plain and the recorded launch alternate on one engine, each timed call
after a 512 MB write, so neither the engine's state nor the slabs (3.9 GB for pedestrians in fp64) are read from the 126 MB
L2; times are CUDA-event medians and include the allocation of the record's tensors (caching allocator).  A record of every
field is T x N x (M x (4 + 2 + 4 + 1) x real + 10) bytes: observation, action, state, reward, then done, winner, tangent and
timestep.  "record_GBps" is those bytes over the recorded launch's time; "copy_GBps" is torch copy_ of a buffer of the same
size (bytes read + written over time), the copy rate this card reaches.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
from cavgym_b200 import BatchedCAVEnv  # noqa: E402

FIELDS = ("observation", "action", "state", "reward", "done", "winner", "tangent", "timestep")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def timed(fn, flush):
    flush.zero_()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop)


def workload(label, scenario, n, dtype, steps, reps, flush):
    from helpers import compile_from_meta, load_golden
    env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=compile_from_meta(load_golden(scenario)[0], mode="device"),
                        device="cuda:0", seed=1)
    env.rollout(200, auto_reset=True)
    m, real = env.num_bodies, env.dtype.itemsize
    recorded = steps * n * (m * (4 + 2 + 4 + 1) * real + 10)
    calls = {"plain": lambda: env.rollout(steps, auto_reset=True),
             "record": lambda: env.rollout(steps, auto_reset=True, record=FIELDS)}
    a = torch.empty(recorded // 2, dtype=torch.uint8, device=env.device)
    b = torch.empty_like(a)
    calls["copy_"] = lambda: b.copy_(a)
    for fn in calls.values():   # warm-up: modules, the allocator's blocks for the slabs
        fn()
        fn()
    torch.cuda.synchronize()
    times = {key: [] for key in calls}
    for _ in range(reps):       # alternate
        for key, fn in calls.items():
            times[key].append(timed(fn, flush))
    ms = {key: float(np.median(v)) for key, v in times.items()}
    out = {"workload": label, "dtype": dtype, "envs": n, "bodies": m, "steps_per_launch": steps, "ms_per_launch": ms,
           "spread_ms": {key: [float(min(v)), float(max(v))] for key, v in times.items()},
           "slowdown": ms["record"] / ms["plain"], "recorded_bytes": recorded,
           "record_GBps": recorded / ms["record"] / 1e6, "copy_GBps": 2 * a.numel() / ms["copy_"] / 1e6,
           "env_steps_per_s": {"plain": n * steps / ms["plain"] * 1e3, "record": n * steps / ms["record"] * 1e3}}
    out["record_over_copy"] = out["record_GBps"] / out["copy_GBps"]
    env.close()
    del env, a, b
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--out", default=None, help="also write the results here as JSON")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_rollout_record.py measures on a CUDA device; there is none")
    name, limit = card()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:0")
    results = []
    for dtype in ("float64", "float32"):
        for label, scenario in (("pedestrians", "pedestrians_rc_seed0"), ("bus stop", "busstop_random_all_seed8")):
            row = workload(label, scenario, args.envs, dtype, args.steps, args.reps, flush)
            row.update({"card": name, "power_limit": limit})
            print(json.dumps(row), flush=True)
            results.append(row)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"card": name, "power_limit": limit, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
