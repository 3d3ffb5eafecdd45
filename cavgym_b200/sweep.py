"""A sweep of one tester parameter (epsilon or distance threshold) as ONE batch: how the tester's setting changes the rate
of "interesting" episodes, those a tester wins (reporting.py:227-243).  The reference answers this with one process per grid
point (experiments.py); here point p owns the contiguous env slots [p * n_p, (p + 1) * n_p) of one engine, and every tester
body of those slots gets the point's value through BatchedCAVEnv.set_agent_params.  Philox is keyed by the global env id, so
the batch is exactly the K single-point engines laid side by side (tests/test_gpu_agent_params.py).

    python -m cavgym_b200.sweep config.json --epsilon 0.5,0.1,0.01 --envs-per-point 262144 --episodes 1000000 [--log-dir logs]
    python -m cavgym_b200.sweep config.json --threshold 400,500 ...     (proximity and election testers)

Each round is reset() followed by rollout(max_timesteps, auto_reset=False): every env plays exactly one whole episode per
round, so each episode is counted once and none is cut short by the end of the run (crude Monte Carlo over whole episodes,
DESIGN §3.3).  A point therefore gets rounds * n_p episodes, the first multiple of n_p at or above --episodes.  Per point the
results are reduced from the drained episode rows; the reference's config.json / episode.log / run.log are written under
<log-dir>/<name>=<value>/ in experiments.py's style.  --save-interesting K also writes the full trajectories of the first K
interesting episodes of each point there, as interesting.npz (BatchedCAVEnv.regenerate, trajectories.save_episodes).
"""
import argparse
import dataclasses
import json
import math
import os

import numpy as np

from . import _abi, reporting

PARAMETERS = {"epsilon": (_abi.CAV_AGENT_RANDOM, _abi.CAV_AGENT_RANDOM_CONSTRAINED),
              "threshold": (_abi.CAV_AGENT_PROXIMITY, _abi.CAV_AGENT_ELECTION)}


def with_round(rows, round_index):
    """Drained episode rows with a "round" field appended: the sweep round that played them.  An episode's rows carry no start
    time; round r of a sweep on a fresh engine starts at t_global = r * max_timesteps (start_steps)."""
    out = np.zeros(rows.shape, dtype=np.dtype(rows.dtype.descr + [("round", "<i4")]))
    for field in rows.dtype.names:
        out[field] = rows[field]
    out["round"] = round_index
    return out


def start_steps(rows, max_timesteps):
    """The t_global at the first step of each row's episode: every round is reset() + rollout(max_timesteps), so round r
    starts at r * max_timesteps."""
    return np.asarray(rows["round"], dtype=np.int64) * int(max_timesteps)


def interesting_rows(rows, k):
    """The first k rows (in drain order) of episodes a tester won (winner > 0)."""
    return rows[rows["winner"] > 0][:int(k)]


def point_slices(n_points, envs_per_point):
    """Env slots of each point: point p owns [p * n_p, (p + 1) * n_p)."""
    return [(p * envs_per_point, (p + 1) * envs_per_point) for p in range(n_points)]


def group_rows(rows, n_points, envs_per_point, env_offset=0):
    """Drained episode rows (CavEpisodeRow fields; `env` is the GLOBAL env id) split by point: row -> (env - env_offset) // n_p.
    Returns a list of n_points row arrays, each in drain order."""
    point = (np.asarray(rows["env"], dtype=np.int64) - int(env_offset)) // int(envs_per_point)
    if point.size and (point.min() < 0 or point.max() >= n_points):
        raise ValueError("an episode row belongs to no point of this sweep (wrong env_offset or envs_per_point)")
    return [rows[point == p] for p in range(n_points)]


@dataclasses.dataclass
class PointResult:
    name: str
    value: float
    episodes: int
    interesting: int
    env_steps: int
    confidence_timesteps: reporting.Interval
    confidence_score: reporting.Interval
    device_seconds: float   # of the whole batch: the points run concurrently in it

    def to_data(self):
        return {"name": self.name, "value": self.value, "episodes": self.episodes, "interesting": self.interesting,
                "env_steps": self.env_steps, "timesteps_interesting": list(self.confidence_timesteps),
                "score_interesting": list(self.confidence_score), "device_seconds": self.device_seconds}


def summarise(rows, name, value, device_seconds):
    """PointResult of one point's rows: the counts and, over the interesting episodes (winner > 0), mean +- 95 % CI of the
    timesteps and of the score (-liveness_sum), as reporting.RunSummary gives them."""
    hits = rows[rows["winner"] > 0]
    return PointResult(name, float(value), int(rows.size), int(hits.size), int(np.asarray(rows["timesteps"], dtype=np.int64).sum()),
                       reporting.confidence_interval([int(t) for t in hits["timesteps"]]),
                       reporting.confidence_interval([-int(s) for s in hits["liveness_sum"]]), float(device_seconds))


def parameter_grid(env, name, values, envs_per_point):
    """The [M, K * n_p] array of set_agent_params' `name` for this sweep: every tester body (b >= 1) whose agent reads the
    parameter gets its point's value; every other row keeps the scenario's own value."""
    import torch
    kinds = PARAMETERS[name]
    m = env.num_bodies
    bodies = env.compiled.struct.bodies
    own = [float(bodies[b].agent_epsilon if name == "epsilon" else bodies[b].agent_threshold) for b in range(m)]
    grid = torch.tensor(own, dtype=torch.float64).reshape(m, 1).repeat(1, len(values) * envs_per_point)
    testers = [b for b in range(1, m) if int(bodies[b].agent) in kinds]
    if not testers:
        raise ValueError(f"no tester body of this scenario reads {name} (agents {[int(bodies[b].agent) for b in range(m)]})")
    for p, (lo, hi) in enumerate(point_slices(len(values), envs_per_point)):
        grid[testers, lo:hi] = float(values[p])
    return grid


def run(env, name, values, envs_per_point, episodes, env_offset=0):
    """Sweep `name` over `values` on `env`, an engine of len(values) * envs_per_point envs (and global env ids from
    env_offset).  Rounds of reset() + rollout(max_timesteps, auto_reset=False) until every point has at least `episodes`
    episodes.  Returns (list of PointResult, list of per-point row arrays); the rows carry the round that played them
    (with_round)."""
    import torch
    n_points = len(values)
    if env.num_envs != n_points * envs_per_point:
        raise ValueError(f"the engine has {env.num_envs} envs, the sweep needs {n_points} x {envs_per_point}")
    grid = parameter_grid(env, name, values, envs_per_point)
    env.set_agent_params(**{name: grid})
    env.set_episode_log(env.num_envs)     # a round finishes each env's episode exactly once
    env.drain_episodes()
    rounds = max(1, math.ceil(episodes / envs_per_point))
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    seconds, parts = 0.0, [[] for _ in range(n_points)]
    for round_index in range(rounds):
        start.record()
        env.reset()
        env.rollout(env.max_timesteps, auto_reset=False)
        stop.record()
        stop.synchronize()
        seconds += start.elapsed_time(stop) / 1000.0
        rows, dropped = env.drain_episodes()
        if dropped or rows.size != env.num_envs:
            raise RuntimeError(f"a round drained {rows.size} episode rows ({dropped} dropped) from {env.num_envs} envs")
        for p, chunk in enumerate(group_rows(with_round(rows, round_index), n_points, envs_per_point, env_offset)):
            parts[p].append(chunk)
    per_point = [np.concatenate(chunks) for chunks in parts]
    return [summarise(rows, name, values[p], seconds) for p, rows in enumerate(per_point)], per_point


def write_logs(config, name, results, per_point, log_root, resolution):
    """experiments.py's files for each point: <log_root>/<name>=<value>/{config.json, episode.log, run.log} in the
    reference's row formats (reporting.py:157-158, 223-224)."""
    nan = float("nan")
    for result, rows in zip(results, per_point):
        log_dir = f"{log_root}/{name}={result.value:g}"
        tester = dataclasses.replace(config.tester_config, **{name: result.value})
        point_config = dataclasses.replace(config, tester_config=tester, episode_log=f"{log_dir}/episode.log", run_log=f"{log_dir}/run.log")
        os.makedirs(log_dir, exist_ok=True)
        point_config.write_json(f"{log_dir}/config.json")
        episode_file = reporting.get_episode_file_logger(point_config.episode_log)
        run_file = reporting.get_run_file_logger(point_config.run_log)
        for index, row in enumerate(rows, start=1):
            interesting = int(row["winner"]) > 0
            episode_file.info(reporting.EpisodeResults(index, reporting.TimeResults(int(row["timesteps"]), nan, nan, resolution),
                                                       completed=int(row["timesteps"]) == config.max_timesteps, interesting=interesting,
                                                       score=-int(row["liveness_sum"]) if interesting else nan).file_message())
        summary = reporting.RunSummary(result.episodes, result.env_steps, result.device_seconds * 1000.0, resolution, result.interesting,
                                       result.confidence_timesteps, result.confidence_score)
        run_file.info(summary.file_message())


def save_interesting(env, name, results, per_point, log_root, k, meta=None):
    """The first k interesting episodes of each point, regenerated on `env` (the sweep's engine, its parameters still set) with
    the start step of their round, written to <log_root>/<name>=<value>/interesting.npz (trajectories.save_episodes).  The
    file's meta is `meta` plus the point's parameter.  Returns the per-point lists of episodes."""
    from . import trajectories
    out = []
    for result, rows in zip(results, per_point):
        hits = interesting_rows(rows, k)
        episodes = env.regenerate(hits, t_global_start=start_steps(hits, env.max_timesteps)) if hits.size else []
        log_dir = f"{log_root}/{name}={result.value:g}"
        os.makedirs(log_dir, exist_ok=True)
        trajectories.save_episodes(f"{log_dir}/interesting.npz", episodes, dict(meta or {}, **{name: result.value}))
        out.append(episodes)
    return out


def main(argv=None):
    from .config import AgentType, make_config
    parser = argparse.ArgumentParser(description="Sweep a tester parameter across the envs of one batch.")
    parser.add_argument("config", help="the reference's config.json")
    which = parser.add_mutually_exclusive_group(required=True)
    which.add_argument("--epsilon", help="comma-separated epsilons of random / random-constrained testers")
    which.add_argument("--threshold", help="comma-separated distance thresholds (px) of proximity / election testers")
    parser.add_argument("--envs-per-point", type=int, default=1 << 18)
    parser.add_argument("--episodes", type=int, default=None, help="episodes per point (default: the config's)")
    parser.add_argument("--log-dir", default=None, help="write each point's config.json / episode.log / run.log under it")
    parser.add_argument("--seed", type=int, default=None, help="default: the config's seed")
    parser.add_argument("--dtype", default="float64", choices=("float64", "float32"))
    parser.add_argument("--save-interesting", type=int, default=0, metavar="K",
                        help="write the trajectories of the first K interesting episodes of each point to <log-dir>/<point>/interesting.npz")
    args = parser.parse_args(argv)
    if args.save_interesting < 0 or (args.save_interesting and not args.log_dir):
        parser.error("--save-interesting takes K >= 0 and needs --log-dir")
    name = "epsilon" if args.epsilon is not None else "threshold"
    values = [float(v) for v in (args.epsilon if name == "epsilon" else args.threshold).split(",") if v.strip()]
    with open(args.config, encoding="utf-8") as handle:
        config = make_config(json.load(handle))
    if config.ego_config.agent is AgentType.Q_LEARNING:
        parser.error("a sweep needs every agent on the device: the Q-learning ego chooses its actions on the host")
    if not hasattr(config.tester_config, name):
        parser.error(f"the config's tester ({config.tester_config.agent}) has no {name}")
    env = config.batched(len(values) * args.envs_per_point, dtype=args.dtype, seed=args.seed)
    results, per_point = run(env, name, values, args.envs_per_point, args.episodes or config.episodes)
    if args.log_dir:
        write_logs(config, name, results, per_point, args.log_dir, env.time_resolution)
    if args.save_interesting:
        save_interesting(env, name, results, per_point, args.log_dir, args.save_interesting,
                         {"config": config.to_data(), "dtype": args.dtype, "seed": (config.seed or 0) if args.seed is None else args.seed})
    env.close()
    for result in results:
        print(json.dumps(result.to_data()))
    return results


if __name__ == "__main__":
    main()
