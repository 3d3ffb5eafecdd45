"""Fixed-level, fixed-effort multilevel splitting: estimates of the rate of "interesting" episodes (a tester wins,
reporting.py:227-243) too rare for crude Monte Carlo, whose cost grows as 1/p.

    python -m cavgym_b200.splitting config.json --envs N --levels L1,L2,... --repetitions R [--seed S]

A repetition resets all N envs and sets every score to -inf.  Stage j runs one `rollout_until(max_timesteps, L_j, score,
salt)`: every env either parks (its running-max danger reached L_j, or a tester won) or finishes, since an episode lasts at
most max_timesteps steps.  p_j = parked / N.  The N slots are then resampled from the H parked envs (each keeps its slot and
gets floor(N / H) copies in all; the N - H floor(N / H) left over go to parked envs drawn without replacement) with
BatchedCAVEnv.fork, the copies taking their source's score.  The last level is +inf, the tester win, and the repetition's
estimate is prod_j p_j (0 when a stage parks no env).  Each stage draws on fresh random streams (salt): a copy forked into
slot i would otherwise redraw the numbers of the trajectory slot i just discarded, which depend on that selection.

The levels are the caller's (DESIGN §3.3): a pilot `rollout_until(max_timesteps, inf, score)` over whole episodes leaves each
env's path-maximum danger in `score`, and levels at its quantiles that leave p_j around 0.1-0.5 are a reasonable start.

`estimate` is duck-typed over the env (num_envs, dtype, device, max_timesteps, timestep, reset, rollout_until, fork), so a
stand-in with the same methods can run it.
"""
import argparse
import json
import math
import time
from dataclasses import dataclass
from typing import List

import torch

from . import reporting

PARKED = 1
_MASK = (1 << 64) - 1


def _splitmix64(x):
    x = (x + 0x9E3779B97F4A7C15) & _MASK
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _MASK
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _MASK
    return x ^ (x >> 31)


def stage_salt(seed, repetition, stage):
    """Non-zero 64-bit salt of one stage (zero would mean the engine's own streams)."""
    salt = _splitmix64(_splitmix64(_splitmix64(int(seed) & _MASK) ^ int(repetition)) ^ int(stage))
    return salt or 1


def resample(parked, n, generator):
    """(src, dst) of the forks that refill n slots from the parked slots (CPU int64): every parked env keeps its own slot and
    is copied floor(n / H) - 1 more times, plus once more for each of the n - H floor(n / H) parked envs drawn without
    replacement; dst are the other slots in order."""
    h = parked.numel()
    q, r = divmod(n, h)
    copies = torch.full((h,), q - 1, dtype=torch.int64)
    if r:
        copies[torch.randperm(h, generator=generator)[:r]] += 1
    src = torch.repeat_interleave(parked, copies)
    keep = torch.zeros(n, dtype=torch.bool)
    keep[parked] = True
    dst = torch.nonzero(~keep).flatten()
    return src, dst


@dataclass(frozen=True)
class SplittingResult:
    estimates: List[float]        # prod_j p_j of each repetition
    fractions: List[List[float]]  # p_j of each repetition's stages (shorter when a stage parked nothing)
    levels: List[float]
    interval: reporting.Interval  # mean of the estimates and the half-width of its 95 % Student-t interval
    env_steps: int                # steps simulated over all envs, stages and repetitions
    device_seconds: float         # GPU time (CUDA events) of all repetitions; wall-clock time on a CPU device

    @property
    def mean(self):
        return self.interval.value


def estimate(env, levels, repetitions, seed=0):
    """Multilevel splitting estimate of P(a tester wins an episode) on `env`.  `levels`: increasing danger levels in px;
    +inf (the tester win) is appended when it is not the last."""
    levels = [float(v) for v in levels]
    if not levels or levels[-1] != math.inf:
        levels.append(math.inf)
    if any(math.isnan(v) for v in levels) or any(b <= a for a, b in zip(levels, levels[1:])):
        raise ValueError(f"levels must increase strictly: {levels}")
    if repetitions < 1:
        raise ValueError("repetitions must be >= 1")
    n, horizon, device = env.num_envs, env.max_timesteps, torch.device(env.device)
    score = torch.empty(n, dtype=env.dtype, device=device)
    steps = torch.zeros((), dtype=torch.int64, device=device)
    cuda = device.type == "cuda"
    if cuda:
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
    else:
        began = time.perf_counter()
    estimates, fractions = [], []
    for rep in range(repetitions):
        env.reset()
        score.fill_(-math.inf)
        p, fracs = 1.0, []
        for j, level in enumerate(levels):
            salt = stage_salt(seed, rep, j)
            before = env.timestep.to(torch.int64)
            status = env.rollout_until(horizon, level, score, salt=salt)
            steps += (env.timestep.to(torch.int64) - before).sum()
            parked = torch.nonzero(status == PARKED).flatten().cpu()
            fracs.append(parked.numel() / n)
            p *= fracs[-1]
            if parked.numel() == 0 or j + 1 == len(levels):
                break
            src, dst = resample(parked, n, torch.Generator().manual_seed(salt & (_MASK >> 1)))
            if dst.numel():
                src, dst = src.to(device), dst.to(device)
                score[dst] = score[src]
                env.fork(src, dst)
        estimates.append(p)
        fractions.append(fracs)
    if cuda:
        stop.record()
        stop.synchronize()
        seconds = start.elapsed_time(stop) / 1000.0
    else:
        seconds = time.perf_counter() - began
    if repetitions > 1:
        interval = reporting.confidence_interval(estimates)
    else:
        interval = reporting.Interval(estimates[0], math.nan)
    return SplittingResult(estimates, fractions, levels, interval, int(steps), seconds)


def main(argv=None):
    from .config import AgentType, make_config
    parser = argparse.ArgumentParser(description="Multilevel splitting estimate of the rate of episodes a tester wins.")
    parser.add_argument("config", help="the reference's config.json")
    parser.add_argument("--envs", type=int, default=1 << 20, help="envs per stage (the fixed effort N)")
    parser.add_argument("--levels", required=True, help="comma-separated increasing danger levels in px; +inf is appended")
    parser.add_argument("--repetitions", type=int, default=10)
    parser.add_argument("--seed", type=int, default=None, help="default: the config's seed")
    parser.add_argument("--dtype", default="float64", choices=("float64", "float32"))
    args = parser.parse_args(argv)
    with open(args.config, encoding="utf-8") as handle:
        config = make_config(json.load(handle))
    if config.ego_config.agent is AgentType.Q_LEARNING:
        parser.error("splitting needs every agent on the device: the Q-learning ego chooses its actions on the host")
    seed = (config.seed or 0) if args.seed is None else args.seed
    env = config.batched(args.envs, dtype=args.dtype, seed=seed)
    result = estimate(env, [float(v) for v in args.levels.split(",") if v.strip()], args.repetitions, seed=seed)
    env.close()
    print(json.dumps({"estimate": result.mean, "ci95": result.interval.error, "repetitions": args.repetitions, "envs": args.envs,
                      "levels": [v if math.isfinite(v) else "inf" for v in result.levels], "estimates": result.estimates,
                      "stage_fractions": result.fractions, "env_steps": result.env_steps, "device_seconds": result.device_seconds}))
    return result


if __name__ == "__main__":
    main()
