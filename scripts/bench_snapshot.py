"""Save, load and fork of environments (kernels_snapshot.cuh) against torch.Tensor.copy_ of the same bytes, on one GPU.

    python scripts/bench_snapshot.py [--reps 20] [--out FILE]

Workloads: C2 pedestrians (2 bodies) at 65,536 and 4,194,304 envs, bus stop (5 bodies) at 1,048,576 envs, the 320-body
dense scenario at 100,000 envs; fp64 and fp32; on-device agents, 200 steps into their episodes.  Per workload:
  save / load of all envs (BatchedCAVEnv.save_envs / load_envs) next to copy_ of a blob of the same size,
  a broadcast fork (env 0 into every slot) and a random resample (sources drawn with repeats, targets = all),
  both through BatchedCAVEnv.fork (index checks included) and through cavgym_fork_envs alone (the two kernel pairs);
  for bus stop, a 100-step rollout of the same engine, the yardstick of the resample.
Every timed call is preceded by a write of 512 MB, so no input is read from the 126 MB L2; times are CUDA-event medians.
GB/s counts the bytes a call must move: save / load / copy_ read and write the blob's size once, a fork twice (gather into
the engine's staging snapshot, scatter out of it).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from cavgym_b200 import BatchedCAVEnv  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def compiled(name):
    from helpers import compile_from_meta, load_golden
    if name == "dense320":
        from bench_dense import scenario
        return scenario(64, 256, 0.01)   # the 320-body scenario of smoke() and of tests/test_gpu_snapshot.py
    return compile_from_meta(load_golden(name)[0], mode="device")


def timed(fn, reps, flush):
    """Median milliseconds of fn() over reps calls, each after an L2-evicting write."""
    times = []
    for _ in range(reps):
        flush.zero_()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        fn()
        stop.record()
        torch.cuda.synchronize()
        times.append(start.elapsed_time(stop))
    return float(np.median(times))


def workload(label, scenario, n, dtype, reps, flush, rollout_steps=0):
    env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=compiled(scenario), device="cuda:0", seed=1)
    env.reset()
    env.rollout(200, auto_reset=True)
    snap = env.save_envs()
    nbytes = int(snap.layout.total_bytes)
    a, b = torch.empty(nbytes, dtype=torch.uint8, device=env.device), torch.empty(nbytes, dtype=torch.uint8, device=env.device)
    a.copy_(snap.data)
    gen = torch.Generator(device=env.device).manual_seed(0)
    resample_src = torch.randint(0, n, (n,), device=env.device, generator=gen)
    every = torch.arange(n, device=env.device)
    broadcast_src = torch.zeros(n, dtype=torch.int64, device=env.device)
    lib, h = env._lib, env._handle

    def raw_fork(src):
        return lambda: lib.cavgym_fork_envs(h, ctypes.c_void_p(src.data_ptr()), ctypes.c_void_p(every.data_ptr()), n, env._stream())

    calls = {"copy_": lambda: b.copy_(a), "save_all": lambda: env.save_envs(), "load_all": lambda: env.load_envs(snap),
             "fork_broadcast": lambda: env.fork(0, every), "fork_resample": lambda: env.fork(resample_src, every),
             "fork_broadcast_kernels": raw_fork(broadcast_src), "fork_resample_kernels": raw_fork(resample_src)}
    if rollout_steps:
        calls["rollout_%d" % rollout_steps] = lambda: env.rollout(rollout_steps, auto_reset=True)
    for fn in calls.values():   # warm-up: modules, the staging snapshot, the allocator
        fn()
        fn()
    torch.cuda.synchronize()
    ms = {}
    for _ in range(2):          # alternate the calls twice, keep the better median of each
        for key, fn in calls.items():
            t = timed(fn, reps, flush)
            ms[key] = min(ms.get(key, t), t)
    moved = {"copy_": 2 * nbytes, "save_all": 2 * nbytes, "load_all": 2 * nbytes}
    for key in ms:
        if key.startswith("fork"):
            moved[key] = 4 * nbytes
    out = {"workload": label, "dtype": dtype, "envs": n, "bodies": env.num_bodies, "snapshot_bytes": nbytes,
           "bytes_per_env": nbytes / n, "ms": ms, "GBps": {k: moved[k] / ms[k] / 1e6 for k in moved},
           "save_over_copy": ms["save_all"] / ms["copy_"], "load_over_copy": ms["load_all"] / ms["copy_"]}
    if rollout_steps:
        out["resample_over_rollout"] = ms["fork_resample"] / ms["rollout_%d" % rollout_steps]
    env.close()
    del env, snap, a, b
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the results here as JSON")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_snapshot.py measures on a CUDA device; there is none")
    name, limit = card()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:0")
    plan = [("C2 pedestrians", "pedestrians_rc_seed0", 65536, 0), ("bus stop", "busstop_random_all_seed8", 1 << 20, 100),
            ("C2 pedestrians", "pedestrians_rc_seed0", 1 << 22, 0), ("dense 64 cars + 256 pedestrians", "dense320", 100000, 0)]
    results = []
    for dtype in ("float64", "float32"):
        for label, scenario, n, rollout in plan:
            row = workload(label, scenario, n, dtype, args.reps, flush, rollout)
            row.update({"card": name, "power_limit": limit})
            print(json.dumps(row), flush=True)
            results.append(row)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"card": name, "power_limit": limit, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
