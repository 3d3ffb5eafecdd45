"""Episodes out of a recorded rollout (BatchedCAVEnv.rollout(..., record=...)).

A record holds per-step slabs [T, ...] with the env index last.  The timestep row is the env's t_ep after the step and 0
where the env did not step, so an episode starts at a row with timestep 1 and ends at its last stepped row: one with
done == 1, or one cut off at max_timesteps (done stays 0 there; the next row of the env is 0 or 1, a new episode or a
frozen env).  complete_episodes returns the episodes that start and end inside the record, each in the per-episode layout
of the reference's fixtures (tests/golden/*.npz), so the replay path and the oracle take them as they take those.
save_episodes / load_episodes write and read such episodes as one .npz file in the fixtures' layout.
"""
import json

import numpy as np

NEEDED = ("observation", "action", "state", "reward", "done", "winner", "tangent", "timestep")


def _host(value):
    return value.cpu().numpy() if hasattr(value, "cpu") else np.asarray(value)


def complete_episodes(record, t_global_start, env_offset=0, max_timesteps=None):
    """Every episode of `record` that starts and ends inside it, as dicts: "env" (global env id = env_offset + index),
    "t_global_start" (the batch-wide step counter at its first step; t_global_start is the counter at the record's first
    row), "init_state" [M,4] (the observation of its first row), "actions" [L,M,2], "state" [L,M,4], "reward" [L,M],
    "done" [L], "winner" [L], "tangent" [L].  Ordered by env, then by start.

    An episode cut off at max_timesteps on the record's LAST row is only recognised with `max_timesteps` given (the
    scenario's); elsewhere the row after it tells.  Raises ValueError if a field it needs was not recorded."""
    missing = [name for name in NEEDED if record.get(name) is None]
    if missing:
        raise ValueError(f"complete_episodes needs the record fields {missing} (rollout(record=...))")
    rec = {name: _host(record[name]) for name in NEEDED}
    ts = rec["timestep"].astype(np.int64)
    n_rows, n_envs = ts.shape
    following = np.zeros_like(ts, dtype=bool)   # the next row is not the same episode's next step
    following[:-1] = ts[1:] <= 1
    ends = (ts > 0) & ((rec["done"] == 1) | following)
    if max_timesteps is not None:
        ends |= ts >= int(max_timesteps)
    episodes = []
    for e in range(n_envs):
        starts = np.flatnonzero(ts[:, e] == 1)
        stops = np.flatnonzero(ends[:, e])
        for s in starts:
            k = np.searchsorted(stops, s)
            if k == len(stops):
                break
            u = stops[k] + 1
            episodes.append({
                "env": int(env_offset) + e,
                "t_global_start": int(t_global_start) + int(s),
                "init_state": rec["observation"][s, :, :, e].copy(),
                "actions": np.ascontiguousarray(rec["action"][s:u, :, :, e]),
                "state": np.ascontiguousarray(rec["state"][s:u, :, :, e]),
                "reward": np.ascontiguousarray(rec["reward"][s:u, :, e]),
                "done": rec["done"][s:u, e].copy(),
                "winner": rec["winner"][s:u, e].copy(),
                "tangent": rec["tangent"][s:u, e].copy(),
            })
    return episodes


def save_episodes(path, episodes, meta):
    """Episodes (dicts of arrays and numbers, as complete_episodes or BatchedCAVEnv.regenerate return them) to one .npz in the
    layout of tests/golden: "meta" (JSON of `meta`, as uint8 bytes), "n_episodes", and "ep<i>_<field>" per episode.  A field
    that is None is left out."""
    arrays = {"meta": np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8), "n_episodes": np.int64(len(episodes))}
    for i, episode in enumerate(episodes):
        for key, value in episode.items():
            if value is not None:
                arrays[f"ep{i}_{key}"] = np.asarray(value)
    np.savez(path, **arrays)


def load_episodes(path):
    """(meta, episodes) of a file written by save_episodes (or a tests/golden fixture)."""
    with np.load(path) as data:
        meta = json.loads(bytes(data["meta"]).decode())
        episodes = []
        for i in range(int(data["n_episodes"])):
            prefix = f"ep{i}_"
            episodes.append({k[len(prefix):]: data[k] for k in data.files if k.startswith(prefix)})
    return meta, episodes
