"""Cost and gain of per-env tester parameters (BatchedCAVEnv.set_agent_params, cavgym_b200.sweep) on one GPU.

    python scripts/bench_sweep.py [--reps 10] [--rounds 4] [--out FILE]

(a) Cost: rollout(100) at 1,048,576 envs on the parameter kernels with every slot set to the scenario's own values, against
    the plain kernels, for the two-body pedestrians scenario (homogeneous) and the five-body bus stop (generic), fp64 and
    fp32.  Two engines start from the same saved state (loaded before each timed call, outside the timing), the calls
    alternate, and a 512 MB write evicts the 126 MB L2 before each timed call.  CUDA-event medians; the end states of the
    first pair are compared bitwise.
(b) Gain: config C5's pair of RandomConstrained epsilons, 0.5 and 0.01, as one batch of 2 x 524,288 envs (cavgym_b200.sweep)
    against two engines of 524,288 envs (global ids 0.. and 524,288..) run one after the other.  Both run the same number of
    whole-episode rounds (reset + rollout(max_timesteps, auto_reset=False)); device time by CUDA events around each round.
    The per-point counters of the batch must equal the two engines' stats().
The GPU's name and power limit are read in the same run and recorded.
"""
import argparse
import copy
import dataclasses
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from cavgym_b200 import BatchedCAVEnv, sweep  # noqa: E402

COST = {"pedestrians (2 bodies, homogeneous)": "pedestrians_rc_seed0", "bus stop (5 bodies, generic)": "busstop_random_all_seed8"}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def golden_config(golden):
    from helpers import load_golden
    return copy.deepcopy(load_golden(golden)[0])


def own_values(env):
    eps_rows, thr_rows = env.agent_rows()
    m, n = env.num_bodies, env.num_envs
    eps = torch.full((m, n), float("nan"), dtype=torch.float64, device=env.device)
    thr = torch.full((m, n), float("nan"), dtype=torch.float64, device=env.device)
    for b in eps_rows:
        eps[b] = env.compiled.struct.bodies[b].agent_epsilon
    for b in thr_rows:
        thr[b] = env.compiled.struct.bodies[b].agent_threshold
    return eps, thr


def timed(fn, flush):
    flush.zero_()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop)


def cost(golden, n, dtype, steps, reps, flush):
    from helpers import compile_from_meta
    engines = {}
    for key in ("plain", "parameters"):
        engines[key] = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=compile_from_meta(golden_config(golden), mode="device"),
                                     device="cuda:0", seed=1)
    engines["parameters"].set_agent_params(*own_values(engines["parameters"]))
    engines["plain"].reset()
    start = engines["plain"].save_envs()
    for env in engines.values():   # warm-up
        env.load_envs(start)
        env.rollout(steps)
    times = {key: [] for key in engines}
    bitwise = None
    for rep in range(reps):
        for key, env in engines.items():
            env.load_envs(start)
            torch.cuda.synchronize()
            times[key].append(timed(lambda: env.rollout(steps), flush))
        if rep == 0:
            a, b = engines["plain"].save_envs(), engines["parameters"].save_envs()
            bitwise = bool(torch.equal(a.data, b.data))
    for env in engines.values():
        env.close()
    med = {key: statistics.median(v) for key, v in times.items()}
    return {"envs": n, "steps": steps, "ms_median": med, "ms_all": times, "parameters_over_plain": med["parameters"] / med["plain"],
            "end_state_bitwise_equal": bitwise}


def rounds_timed(env, rounds):
    ms = 0.0
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        start.record()
        env.reset()
        env.rollout(env.max_timesteps, auto_reset=False)
        stop.record()
        stop.synchronize()
        ms += start.elapsed_time(stop)
    return ms


def gain(n_p, rounds, dtype):
    from cavgym_b200.config import make_config
    config = make_config(golden_config("pedestrians_rc_seed0")["config"])
    values = (0.5, 0.01)
    batch = config.batched(len(values) * n_p, device="cuda:0", dtype=dtype, seed=0)
    batch.set_agent_params(epsilon=sweep.parameter_grid(batch, "epsilon", values, n_p))
    batch.reset()
    batch.rollout(10, auto_reset=False)     # warm-up of the parameter kernels
    results, _ = sweep.run(batch, "epsilon", values, n_p, episodes=rounds * n_p)
    batch.close()
    separate, identical = [], True
    for p, value in enumerate(values):
        single = dataclasses.replace(config, tester_config=dataclasses.replace(config.tester_config, epsilon=value))
        env = single.batched(n_p, device="cuda:0", dtype=dtype, seed=0, env_offset=p * n_p)
        env.reset()
        env.rollout(10, auto_reset=False)   # warm-up, as the batch's: every env then starts its rounds at the same episode number
        base = env.stats()
        ms = rounds_timed(env, rounds)
        stats = {k: v - base[k] for k, v in env.stats().items()}
        got = results[p]
        # (env_steps of a point counts the steps of its episodes: stats' sum_t; its env_steps also holds the warm-up's 10 steps
        #  per env, abandoned by the first round's reset)
        same = (got.episodes, got.interesting, got.env_steps) == (stats["episodes"], stats["interesting"], stats["sum_t"])
        same = same and (got.confidence_timesteps.value, got.confidence_score.value) == (
            stats["sum_t_interesting"] / stats["interesting"], stats["sum_score"] / stats["interesting"])
        identical = identical and same
        separate.append({"epsilon": value, "device_ms": ms, "stats": stats})
        env.close()
    batch_ms = results[0].device_seconds * 1000.0
    return {"envs_per_point": n_p, "rounds": rounds, "dtype": dtype, "batch_device_ms": batch_ms,
            "separate_device_ms": sum(s["device_ms"] for s in separate), "separate": separate,
            "separate_over_batch": sum(s["device_ms"] for s in separate) / batch_ms,
            "points": [r.to_data() for r in results], "per_point_counters_identical": identical}


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--reps", type=int, default=10)
    parser.add_argument("--rounds", type=int, default=4)
    parser.add_argument("--envs", type=int, default=1 << 20)
    parser.add_argument("--out", default=None)
    args = parser.parse_args()
    name, limit = card()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:0")
    out = {"gpu": name, "power_limit": limit, "cost": {}, "gain": {}}
    for label, golden in COST.items():
        for dtype in ("float64", "float32"):
            out["cost"][f"{label}, {dtype}"] = cost(golden, args.envs, dtype, 100, args.reps, flush)
            print(label, dtype, json.dumps(out["cost"][f"{label}, {dtype}"]["ms_median"]), flush=True)
    for dtype in ("float64", "float32"):
        out["gain"][dtype] = gain(args.envs // 2, args.rounds, dtype)
        print("gain", dtype, out["gain"][dtype]["batch_device_ms"], out["gain"][dtype]["separate_device_ms"], flush=True)
    text = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as handle:
            handle.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
