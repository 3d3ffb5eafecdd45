"""Cost of regenerating logged episodes (BatchedCAVEnv.regenerate_episodes / regenerate) on one GPU.

    python scripts/bench_regenerate.py [--reps 7] [--steps 100] [--envs 1048576] [--episodes 10000000] [--out FILE]

1. Kernel: regenerate_episodes of `--envs` keys (env ids 0..N-1, episode 1) for `--steps` steps recording every field,
   against rollout(steps, record=every field) of an engine of the same size, 200 steps into its episodes.  The two alternate,
   each timed call after a 512 MB write, so neither the engine's state nor the slabs are read from the 126 MB L2; CUDA-event
   medians, the record's allocation included (caching allocator).
2. End to end, C5-shaped: a run of `--envs` envs with auto-reset (BatchedSimulation, 100 steps per launch) until
   `--episodes` episodes have finished, keeping the start step of the first `--interesting` interesting episodes (default:
   all), then regenerate() of them to host episodes (wall clock, synchronised), against recording the same number of steps in 100-step windows
   (rollout(100, record=every field), device time only: extracting the episodes from the windows is not included, so that
   arm is a lower bound).
Workloads: pedestrians (2 bodies) and bus stop (5 bodies) with their stock on-device agents, fp64 and fp32.
"""
import argparse
import dataclasses
import json
import os
import subprocess
import sys
import timeit

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


def kernel(label, scenario, n, dtype, steps, reps, flush):
    from helpers import compile_from_meta, load_golden
    comp = compile_from_meta(load_golden(scenario)[0], mode="device")
    env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=comp, device="cuda:0", seed=1)
    env.rollout(200, auto_reset=True)
    ids, eps = np.arange(n, dtype=np.int64), np.ones(n, dtype=np.int64)
    calls = {"rollout_record": lambda: env.rollout(steps, auto_reset=True, record=FIELDS),
             "regenerate": lambda: env.regenerate_episodes(ids, eps, steps, record=FIELDS)}
    for fn in calls.values():
        fn()
        fn()
    torch.cuda.synchronize()
    times = {key: [] for key in calls}
    for _ in range(reps):
        for key, fn in calls.items():
            times[key].append(timed(fn, flush))
    ms = {key: float(np.median(v)) for key, v in times.items()}
    env.close()
    torch.cuda.empty_cache()
    return {"workload": label, "dtype": dtype, "keys": n, "steps": steps, "ms": ms,
            "spread_ms": {key: [float(min(v)), float(max(v))] for key, v in times.items()},
            "regenerate_over_rollout_record": ms["regenerate"] / ms["rollout_record"]}


def end_to_end(label, scenario, n, dtype, episodes, keep, flush):
    from helpers import load_golden
    from cavgym_b200.config import make_config
    from cavgym_b200.simulation import BatchedSimulation
    config = dataclasses.replace(make_config(load_golden(scenario)[0]["config"]), episode_log=None, run_log=None)
    sim = BatchedSimulation(config, n, dtype=dtype)
    sim.console.disabled = True
    sim.save_interesting = keep
    start = timeit.default_timer()
    summary = sim.run(episodes=episodes, reduce=False)
    torch.cuda.synchronize()
    run_and_regenerate = timeit.default_timer() - start
    hits = len(sim.interesting)
    assert all(ep["reproduced"] for ep in sim.interesting)
    steps = sim.steps_run
    sim.env.close()
    # the same steps recorded in 100-step windows, device time
    env = config.batched(n, dtype=dtype)
    env.reset()
    recorded_ms = 0.0
    for _ in range(steps // 100):
        recorded_ms += timed(lambda: env.rollout(100, auto_reset=True, record=FIELDS), flush)
    env.close()
    torch.cuda.empty_cache()
    return {"workload": label, "dtype": dtype, "envs": n, "episodes": int(summary.episodes), "steps_per_env": steps, "kept": keep,
            "interesting": hits, "run_and_regenerate_s": run_and_regenerate, "recorded_windows_device_s": recorded_ms / 1e3,
            "speedup_over_recording": recorded_ms / 1e3 / run_and_regenerate}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--episodes", type=int, default=10_000_000)
    ap.add_argument("--interesting", type=int, default=1 << 62, help="regenerate the first K interesting episodes (default: all)")
    ap.add_argument("--skip-kernel", action="store_true", help="end-to-end part only")
    ap.add_argument("--out", default=None, help="also write the results here as JSON")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_regenerate.py measures on a CUDA device; there is none")
    name, limit = card()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:0")
    results = {"card": name, "power_limit": limit, "kernel": [], "end_to_end": []}
    for dtype in ("float64", "float32") if not args.skip_kernel else ():
        for label, scenario in (("pedestrians", "pedestrians_rc_seed0"), ("bus stop", "busstop_random_all_seed8")):
            row = kernel(label, scenario, args.envs, dtype, args.steps, args.reps, flush)
            print(json.dumps(row), flush=True)
            results["kernel"].append(row)
    for dtype in ("float64", "float32"):
        for label, scenario in (("pedestrians", "pedestrians_rc_seed0"), ("bus stop", "busstop_random_all_seed8")):
            row = end_to_end(label, scenario, args.envs, dtype, args.episodes, args.interesting, flush)
            print(json.dumps(row), flush=True)
            results["end_to_end"].append(row)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
