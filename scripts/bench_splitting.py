"""Cost and gain of multilevel splitting (cavgym_b200.splitting) on one GPU.

    python scripts/bench_splitting.py [--reps 10] [--out FILE]

(a) Cost of scoring and parking: rollout_until(100, +inf) against rollout(100, auto_reset=False) at 1,048,576 envs, for the
    two-body pedestrians and the crossroads scenario (heterogeneous: three bodies, one pedestrian), fp64 and fp32.  Both
    start from the same saved state (loaded before each timed call, outside the timing), they alternate, and a 512 MB write
    evicts the 126 MB L2 before each timed call.  CUDA-event medians.
(b) Gain: on the configurations of RARE, crude Monte Carlo (rounds of reset + rollout(max_timesteps, auto_reset=False)
    over N envs, each env one whole episode per round, until at least E episodes; p = interesting / episodes from stats()) against splitting.estimate (N envs per stage, R repetitions, the
    levels given).  Work-normalised relative variance = (variance of the estimate / p^2) x device seconds spent on it:
    smaller is better, and the ratio crude / splitting is the speed-up at equal precision.  Crude's variance is p(1 - p) / E
    with its own p, or with splitting's p when crude found no hit (marked).  "auto_reset_stopped_at_a_step" is the win rate
    that an auto-reset rollout stopped once E episodes have finished reports, beside the whole-episode count (DESIGN §3.3).
"""
import argparse
import copy
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from cavgym_b200 import BatchedCAVEnv, splitting  # noqa: E402

# name -> (golden scenario, tester config, crude envs, crude episodes at least, splitting envs, repetitions, levels): the stock
# pedestrians scenario with RandomAgent testers that rarely act (tests/test_gpu_splitting.py), from a win rate crude Monte
# Carlo measures easily to one where it finds a few dozen hits.
RARE = {f"random tester, epsilon {eps:g}": ("pedestrians_rc_seed0", {"option": "random", "epsilon": eps}, 1 << 20, 16_000_000, 1 << 18, 16,
                                            levels) for eps, levels in ((3e-4, (-30.0, -10.0)), (1e-5, (-45.0, -25.0, -12.0, -4.0)),
                                                                        (1e-6, (-45.0, -25.0, -12.0, -4.0)))}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def compiled(golden, tester=None):
    from helpers import compile_from_meta, load_golden
    meta = copy.deepcopy(load_golden(golden)[0])
    if tester is not None:
        meta["config"]["tester_config"] = dict(tester)
        meta["config"]["ego_config"] = {"option": "noop"}
    return compile_from_meta(meta, mode="device")


def timed(fn, flush):
    flush.zero_()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop)


def cost(label, golden, n, dtype, steps, reps, flush):
    env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=compiled(golden), device="cuda:0", seed=1)
    start = env.save_envs()
    score = torch.empty(n, dtype=env.dtype, device=env.device)
    status = torch.empty(n, dtype=torch.uint8, device=env.device)
    calls = {"rollout": lambda: env.rollout(steps, auto_reset=False),
             "rollout_until": lambda: env.rollout_until(steps, math.inf, score, status=status)}
    for fn in calls.values():   # warm-up
        env.load_envs(start)
        score.fill_(-math.inf)
        fn()
    times = {key: [] for key in calls}
    for _ in range(reps):
        for key, fn in calls.items():
            env.load_envs(start)
            score.fill_(-math.inf)
            times[key].append(timed(fn, flush))
    ms = {key: float(np.median(v)) for key, v in times.items()}
    out = {"workload": label, "dtype": dtype, "envs": n, "bodies": env.num_bodies, "steps_per_launch": steps, "ms_per_launch": ms,
           "spread_ms": {key: [float(min(v)), float(max(v))] for key, v in times.items()},
           "until_over_rollout": ms["rollout_until"] / ms["rollout"]}
    env.close()
    return out


def gain(name, golden, tester, crude_envs, crude_episodes, n, reps, levels, seed=1):
    c = compiled(golden, tester)
    crude = BatchedCAVEnv(None, None, None, num_envs=crude_envs, compiled=c, device="cuda:0", seed=seed)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(-(-crude_episodes // crude_envs)):   # whole episodes: one per env and round (tests/test_gpu_splitting.py)
        crude.reset()
        crude.rollout(crude.max_timesteps, auto_reset=False)
    stop.record()
    stats = crude.stats()
    truncated = BatchedCAVEnv(None, None, None, num_envs=crude_envs, compiled=c, device="cuda:0", seed=seed)
    while truncated.stats()["episodes"] < crude_episodes:   # the count an auto-reset rollout stopped at a fixed step gives
        truncated.rollout(500, auto_reset=True)
    t_stats = truncated.stats()
    truncated.close()
    torch.cuda.synchronize()
    crude_s = start.elapsed_time(stop) / 1e3
    crude.close()
    env = BatchedCAVEnv(None, None, None, num_envs=n, compiled=c, device="cuda:0", seed=seed + 1)
    res = splitting.estimate(env, levels, reps, seed=seed)
    env.close()
    est = np.array(res.estimates)
    p_split = float(est.mean())
    split_var = float(est.var(ddof=1)) / reps
    e, hits = stats["episodes"], stats["interesting"]
    p_crude = hits / e
    p_for_crude = p_crude if hits else p_split
    crude_var = p_for_crude * (1 - p_for_crude) / e
    out = {"configuration": name, "scenario": golden, "tester": tester, "crude": {"envs": crude_envs, "episodes": e, "interesting": hits,
           "p": p_crude, "se": math.sqrt(crude_var), "variance_from": "own p" if hits else "splitting's p (no hit)",
           "device_s": crude_s, "env_steps": stats["env_steps"],
           "auto_reset_stopped_at_a_step": {"episodes": t_stats["episodes"], "p": t_stats["interesting"] / t_stats["episodes"]}},
           "splitting": {"envs": n, "repetitions": reps, "levels": [v if math.isfinite(v) else "inf" for v in res.levels],
                         "p": p_split, "se": math.sqrt(split_var), "mean_stage_fractions": np.mean(
                             [f + [0.0] * (len(res.levels) - len(f)) for f in res.fractions], axis=0).tolist(),
                         "device_s": res.device_seconds, "env_steps": res.env_steps}}
    if p_split > 0:
        out["work_normalised_relvar"] = {"crude": crude_var / p_for_crude ** 2 * crude_s, "splitting": split_var / p_split ** 2 * res.device_seconds}
        out["crude_over_splitting"] = out["work_normalised_relvar"]["crude"] / out["work_normalised_relvar"]["splitting"]
    if hits:
        out["agreement_in_combined_se"] = abs(p_split - p_crude) / math.sqrt(split_var + crude_var)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--out", default=None, help="also write the results here as JSON")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_splitting.py measures on a CUDA device; there is none")
    name, limit = card()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:0")
    costs, gains = [], []
    for dtype in ("float64", "float32"):
        for label, golden in (("pedestrians", "pedestrians_rc_seed0"), ("crossroads", "crossroads_random_all_seed6")):
            row = cost(label, golden, args.envs, dtype, args.steps, args.reps, flush)
            print(json.dumps(row), flush=True)
            costs.append(row)
    del flush
    torch.cuda.empty_cache()
    for key, spec in RARE.items():
        row = gain(key, *spec)
        print(json.dumps(row), flush=True)
        gains.append(row)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"card": name, "power_limit": limit, "cost": costs, "gain": gains}, f, indent=1)


if __name__ == "__main__":
    main()
