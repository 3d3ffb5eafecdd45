"""Regenerating logged episodes (BatchedCAVEnv.regenerate, cavgym_regenerate_episodes) from their (env, episode) keys.

The contract: an episode played from a reset on the engine's own random streams is a pure function of the scenario, seed,
dtype, tau, its (global env id, episode number) and its slot's tester parameters, so regenerating it on a sibling engine in
any slot, any order and any batch size gives back every recorded field bit for bit; t_global adds only the time-out term of
one step's rewards; an episode that was not played that way is reported as not reproduced.

Scenarios run with max_timesteps lowered to 23 so that, in windows of 30 and 35 steps, episodes end and restart inside a
window, and the batch-wide t_global passes max_timesteps - 1 (the time-out reward).
"""
import copy
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import FAMILIES, MATRIX_M, compile_from_meta, load_golden, matrix_scenario, state_err

pytestmark = pytest.mark.gpu

MAX_T = 23
WINDOWS = (30, 35)
N = 203
OFFSET = 1000
FIELDS = ("observation", "action", "state", "reward", "done", "winner", "tangent", "timestep")
EPISODE_FIELDS = ("init_state", "actions", "state", "reward", "done", "winner", "tangent")
STOCK = ("pedestrians_rc_seed0", "pedestrians_proximity_seed3", "crossroads_random_all_seed6", "busstop_random_all_seed8",
         "pelican_random_all_seed10")
CASES = [("golden", name) for name in STOCK] + [("matrix", m, family) for m in MATRIX_M for family in FAMILIES]
DTYPES = ("float64", "float32")
CAV_EINVAL, CAV_ESTATE = -22, -1   # include/cavgym.h


def case_id(case):
    return case[1] if case[0] == "golden" else f"{case[2]}_{case[1]}_bodies"


def compiled(case, mode="device", max_t=MAX_T):
    if case[0] == "golden":
        meta = copy.deepcopy(load_golden(case[1])[0])
        meta["config"]["max_timesteps"] = max_t
        return compile_from_meta(meta, mode=mode)
    return matrix_scenario(case[1], case[2], mode, max_timesteps=max_t)


def make(case, dtype, n=N, offset=OFFSET, seed=5, mode="device"):
    from cavgym_b200 import BatchedCAVEnv
    return BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=compiled(case, mode), seed=seed, env_offset=offset)


def host(t):
    return t.cpu().numpy()


def numbered(episodes):
    """complete_episodes of a record that starts right after reset(): env e's j-th episode is its episode 1 + j."""
    seen = {}
    for ep in episodes:
        ep["episode"] = 1 + seen.get(ep["env"], 0)
        seen[ep["env"]] = ep["episode"]
    return episodes


_RUNS = {}


def original(case, dtype):
    """An auto-reset recorded rollout over WINDOWS on an engine of N envs at OFFSET: (engine, episodes, drained rows)."""
    from cavgym_b200.trajectories import complete_episodes
    key = (case, dtype)
    if key not in _RUNS:
        env = make(case, dtype)
        env.set_episode_log(1 << 14)
        env.reset()
        records = [{k: host(v) for k, v in env.rollout(w, auto_reset=True, record=FIELDS).items()} for w in WINDOWS]
        whole = {k: np.concatenate([r[k] for r in records]) for k in FIELDS}
        episodes = numbered(complete_episodes(whole, 0, env_offset=OFFSET, max_timesteps=MAX_T))
        rows, dropped = env.drain_episodes()
        assert dropped == 0
        _RUNS[key] = (env, episodes, rows)
    return _RUNS[key]


def rows_for(rows, episodes):
    index = {(int(r["env"]), int(r["episode"])): r for r in rows}
    return np.array([index[(ep["env"], ep["episode"])] for ep in episodes], dtype=rows.dtype)


def assert_same(got, want, fields=EPISODE_FIELDS):
    for name in fields:
        assert got[name].shape == want[name].shape, (name, got["env"], got["episode"])
        assert np.array_equal(got[name].view(np.uint8), want[name].view(np.uint8)), (name, got["env"], got["episode"])


# ------------------------------------------------------------------ 1. against the original run
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_regenerated_episodes_equal_the_recorded_ones_bitwise(case, dtype):
    env, episodes, rows = original(case, dtype)
    assert episodes and any(ep["episode"] > 1 for ep in episodes)   # restarts inside the run are covered
    order = np.random.default_rng(0).permutation(len(episodes))
    want = [episodes[i] for i in order]
    requested = rows_for(rows, want)
    before = env.launch_count()
    got = env.regenerate(requested, t_global_start=np.array([ep["t_global_start"] for ep in want]))
    assert env.launch_count() == before   # the original engine is not touched
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert (g["env"], g["episode"], g["t_global_start"]) == (w["env"], w["episode"], w["t_global_start"])
        assert g["reproduced"] is True
        assert_same(g, w)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", [("golden", "pedestrians_rc_seed0"), ("golden", "busstop_random_all_seed8"),
                                  ("matrix", 5, "homogeneous")], ids=case_id)
def test_the_regenerating_engine_logs_the_requested_rows(case, dtype):
    """The entry point itself: slots in another order on an engine of another size, whose drained rows are the requested
    rows, and whose record rows after an episode's end are frozen rows."""
    env, episodes, rows = original(case, dtype)
    requested = rows_for(rows, episodes)[::-1].copy()
    k = requested.size
    sib = make(case, dtype, n=k, offset=0)
    sib.set_episode_log(k)
    sib.set_global_timestep(MAX_T)
    rec = sib.regenerate_episodes(requested["env"], requested["episode"], MAX_T + 4, record=FIELDS)
    got, dropped = sib.drain_episodes()
    assert dropped == 0
    assert np.array_equal(np.sort(got, order=["env", "episode"]), np.sort(requested, order=["env", "episode"]))
    ts = host(rec["timestep"])
    for e in range(k):
        length = int(requested["timesteps"][e])
        assert np.array_equal(ts[:length, e], np.arange(1, length + 1)) and not ts[length:, e].any()
        assert not host(rec["reward"])[length:, :, e].any() and not host(rec["action"])[length:, :, :, e].any()
        assert (host(rec["state"])[length:, :, :, e] == host(rec["state"])[length - 1, :, :, e]).all()
    assert sib.state_dict()["t_global"] == MAX_T + MAX_T + 4
    assert sib.stats()["episodes"] == k


# ------------------------------------------------------------------ 2. the time-out term
@pytest.mark.parametrize("dtype", DTYPES)
def test_the_default_start_drops_exactly_the_time_out_term(dtype):
    case = ("golden", "pedestrians_rc_seed0")
    env, episodes, rows = original(case, dtype)
    spanning = [ep for ep in episodes if ep["t_global_start"] <= MAX_T - 1 < ep["t_global_start"] + len(ep["done"])
                and ep["done"][MAX_T - 1 - ep["t_global_start"]] == 0 and ep["winner"][MAX_T - 1 - ep["t_global_start"]] < 0]
    assert spanning
    got = env.regenerate(rows_for(rows, spanning))
    draw = env.compiled.struct.reward_draw
    for g, w in zip(got, spanning):
        assert g["reproduced"] is True and g["t_global_start"] == MAX_T
        assert_same(g, w, ("init_state", "actions", "state", "done", "winner", "tangent"))
        s = MAX_T - 1 - w["t_global_start"]
        differs = np.flatnonzero((g["reward"] != w["reward"]).any(axis=1))
        assert differs.tolist() == [s]
        want = (g["reward"][s] + g["reward"].dtype.type(draw)).astype(g["reward"].dtype)
        assert np.array_equal(want.view(np.uint8), w["reward"][s].view(np.uint8))


# ------------------------------------------------------------------ 3. sweeps
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name, case, values", [
    ("epsilon", ("golden", "pedestrians_rc_seed0"), (1.0, 0.3, 0.05)),
    ("threshold", ("golden", "pedestrians_proximity_seed3"), (150.0, 400.0, 900.0)),
], ids=["epsilon", "threshold"])
def test_sweep_episodes_regenerate_with_their_blocks_values(name, case, values, dtype):
    from cavgym_b200 import sweep
    from cavgym_b200.trajectories import complete_episodes
    from cavgym_b200 import BatchedCAVEnv
    n_p, max_t = 64, 60
    env = BatchedCAVEnv(None, None, None, num_envs=3 * n_p, dtype=dtype, compiled=compiled(case, max_t=max_t), seed=11,
                        env_offset=OFFSET)
    twin = BatchedCAVEnv(None, None, None, num_envs=3 * n_p, dtype=dtype, compiled=compiled(case, max_t=max_t), seed=11,
                         env_offset=OFFSET)
    _, per_point = sweep.run(env, name, values, n_p, episodes=2 * n_p, env_offset=OFFSET)
    twin.set_agent_params(**{name: sweep.parameter_grid(twin, name, values, n_p)})
    recorded = {}
    for round_index in range(2):
        twin.reset()
        record = twin.rollout(max_t, auto_reset=False, record=FIELDS)
        for ep in complete_episodes(record, round_index * max_t, env_offset=OFFSET, max_timesteps=max_t):
            recorded[(ep["env"], 1 + round_index)] = ep
    rows = np.concatenate(per_point)
    assert set(np.unique(rows["round"])) == {0, 1}
    hits = np.concatenate([sweep.interesting_rows(r, 1 << 30) for r in per_point])
    # every episode of the sweep, the interesting ones among them, regenerates bitwise with its block's values
    got = env.regenerate(rows, t_global_start=sweep.start_steps(rows, max_t))
    for g, row in zip(got, rows):
        assert g["reproduced"] is True
        assert_same(g, recorded[(int(row["env"]), int(row["episode"]))])
    print(f"{name}: {hits.size} interesting episodes of {rows.size}")
    # cleared parameters: the scenario's own value for every block, so the trajectories of the other blocks differ
    env.set_agent_params()
    cleared = env.regenerate(rows, t_global_start=sweep.start_steps(rows, max_t))
    changed = [not np.array_equal(c["actions"], g["actions"]) or not np.array_equal(c["state"], g["state"])
               for c, g in zip(cleared, got)]
    assert any(changed)


# ------------------------------------------------------------------ 4. replay
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", [("golden", name) for name in STOCK] + [("matrix", 6, "generic"), ("matrix", 8, "homogeneous")],
                         ids=case_id)
def test_regenerated_episodes_replay_on_external_actions_and_match_the_oracle(case, dtype):
    env, episodes, rows = original(case, dtype)
    got = env.regenerate(rows_for(rows, episodes), t_global_start=np.array([ep["t_global_start"] for ep in episodes]))
    for t0 in sorted({g["t_global_start"] for g in got}):
        group = [g for g in got if g["t_global_start"] == t0]
        k, length, m = len(group), max(len(g["done"]) for g in group), group[0]["init_state"].shape[0]
        actions = np.zeros((length, m, 2, k), dtype=group[0]["actions"].dtype)
        for j, g in enumerate(group):
            actions[:len(g["done"]), :, :, j] = g["actions"]
        ext = make(case, dtype, n=k, mode="external")
        ext.set_global_timestep(t0)
        ext.reset(init_state=np.stack([g["init_state"] for g in group], axis=-1))
        out = {name: host(v) for name, v in ext.replay(actions).items()}
        for j, g in enumerate(group):
            steps = len(g["done"])
            assert np.array_equal(out["state"][:steps, :, :, j], g["state"])
            assert np.array_equal(out["reward"][:steps, :, j], g["reward"])
            for name in ("done", "winner", "tangent"):
                assert np.array_equal(out[name][:steps, j], g[name])
        if dtype != "float64":
            continue
        from oracle.oracle import Oracle
        oracle = Oracle(compiled(case, "external"), k)
        oracle.set_global_timestep(t0)
        oracle.reset(init_state=np.stack([g["init_state"] for g in group], axis=-1))
        state, reward, done, winner, _ = oracle.replay(actions)
        for j, g in enumerate(group):
            steps = len(g["done"])
            flagged = np.flatnonzero(g["tangent"])
            upto = steps if flagged.size == 0 else flagged[0]
            assert state_err(state[:upto, :, :, j], g["state"][:upto]) <= 1e-9
            assert np.max(np.abs(reward[:upto, :, j] - g["reward"][:upto]) / np.maximum(1, np.abs(g["reward"][:upto])), initial=0) <= 1e-9
            assert np.array_equal(done[:upto, j], g["done"][:upto]) and np.array_equal(winner[:upto, j], g["winner"][:upto])


# ------------------------------------------------------------------ 5. rows that do not reproduce
def test_an_episode_continued_after_a_fork_is_reported_not_reproduced():
    """Slots 1..63 continue a copy of slot 0's episode from its step 5.  Their rows regenerate as what each slot would have
    played without the fork (a twin engine): reproduced exactly where that summary happens to equal the forked one's."""
    from cavgym_b200 import BatchedCAVEnv
    max_t, n = 300, 64
    engines = [BatchedCAVEnv(None, None, None, num_envs=n, dtype="float64", compiled=compiled(("golden", "pedestrians_random_all_seed4"),
                             max_t=max_t), seed=5, env_offset=OFFSET) for _ in range(2)]
    for env in engines:
        env.set_episode_log(1 << 12)
        env.reset()
        env.rollout(5, auto_reset=False)
    env, twin = engines
    env.fork(0, list(range(1, n)))
    for e in engines:
        e.rollout(max_t, auto_reset=False)
    rows = np.sort(env.drain_episodes()[0], order="env")
    plain = np.sort(twin.drain_episodes()[0], order="env")
    assert rows.size == plain.size == n
    got = env.regenerate(rows, t_global_start=0)
    summary = ("timesteps", "winner", "liveness_sum")
    for g, row, own in zip(got, rows, plain):
        assert g["reproduced"] == all(row[f] == own[f] for f in summary)
    assert got[0]["reproduced"] is True
    assert [g["reproduced"] for g in got[1:]].count(False) > 0


# ------------------------------------------------------------------ 6. refusals
def test_every_refusal_fires_before_any_launch():
    from cavgym_b200 import _native
    lib = _native.load()
    case = ("golden", "pedestrians_rc_seed0")

    def call(env, ids, eps, n_steps=MAX_T):
        return lib.cavgym_regenerate_episodes(env._handle, None if ids is None else C.c_void_p(ids.data_ptr()),
                                              None if eps is None else C.c_void_p(eps.data_ptr()), n_steps, None, env._stream())

    env = make(case, "float64", n=8)
    env.reset()
    ids = torch.arange(8, dtype=torch.int64, device=env.device)
    eps = torch.ones(8, dtype=torch.int32, device=env.device)
    def sections():
        snap = env.save_envs()
        return [snap[name].contiguous().view(torch.uint8).clone() for name in snap.NAMES]   # bytes: the agent rows hold NaN

    snap = sections()
    t_global = env.state_dict()["t_global"]
    before = env.launch_count()
    assert call(env, None, eps) == CAV_EINVAL and call(env, ids, None) == CAV_EINVAL
    assert call(env, ids, eps, -1) == CAV_EINVAL
    assert env.launch_count() == before
    for bad_ids, bad_eps in ((ids - 1, eps), (ids, eps - 2), (ids + (1 << 40), eps)):   # range-checked on the device
        assert call(env, bad_ids.contiguous(), bad_eps.contiguous()) == CAV_EINVAL
    assert all(torch.equal(a, b) for a, b in zip(sections(), snap)) and env.state_dict()["t_global"] == t_global
    before = env.launch_count()
    for bad in (dict(env_ids=np.arange(7), episodes=np.ones(7)), dict(env_ids=np.arange(8) - 1, episodes=np.ones(8)),
                dict(env_ids=np.arange(8), episodes=-np.ones(8))):
        with pytest.raises(ValueError):
            env.regenerate_episodes(**bad)
        assert env.launch_count() == before
    row = np.zeros(1, dtype=[("env", "<i8"), ("episode", "<i4")])
    for bad in (np.zeros(1, dtype=[("env", "<i8")]), np.array([(-1, 1)], dtype=row.dtype), np.array([(0, -1)], dtype=row.dtype)):
        with pytest.raises(ValueError):
            env.regenerate(bad)
    with pytest.raises(ValueError):
        env.regenerate(row, n_steps=-1)
    with pytest.raises(ValueError):
        env.regenerate(row, record=("nope",))
    env.set_agent_params(epsilon=torch.full((2, 8), 0.5, dtype=torch.float64))
    with pytest.raises(ValueError):   # a row outside this engine's slots has no parameters to gather
        env.regenerate(np.array([(0, 1)], dtype=row.dtype))
    env.set_agent_params()

    def refused(target):
        ids_t = torch.arange(target.num_envs, dtype=torch.int64, device=target.device)
        eps_t = torch.ones(target.num_envs, dtype=torch.int32, device=target.device)
        before = target.launch_count()
        assert call(target, ids_t, eps_t) == CAV_ESTATE
        assert target.launch_count() == before

    refused(make(case, "float64", n=8, mode="external"))
    refused(make(("golden", "learn_election3_seed22"), "float64", n=8))
    dense = make(case, "float64", n=8)
    dense.set_dense_path(True)
    refused(dense)
    over = make(case, "float64", n=8)
    over.set_uniform_override(torch.zeros((2, 3, 8), dtype=torch.float64))
    refused(over)
    over = make(case, "float64", n=8)
    over.set_spawn_override(torch.zeros((2, 5, 8), dtype=torch.float64))
    refused(over)


# ------------------------------------------------------------------ 7. CLI
def replays_bitwise(meta_config, dtype, episodes):
    from cavgym_b200 import BatchedCAVEnv
    meta = {"config": meta_config}
    for ep in episodes:
        ext = BatchedCAVEnv(None, None, None, num_envs=1, dtype=dtype, compiled=compile_from_meta(meta, mode="external"))
        ext.set_global_timestep(int(ep["t_global_start"]))
        ext.reset(init_state=ep["init_state"][:, :, None])
        out = ext.replay(ep["actions"][:, :, :, None])
        assert np.array_equal(host(out["state"])[:, :, :, 0], ep["state"])
        assert np.array_equal(host(out["reward"])[:, :, 0], ep["reward"])
        assert np.array_equal(host(out["winner"])[:, 0], ep["winner"])


def test_save_interesting_writes_loadable_episodes_that_replay(tmp_path):
    from cavgym_b200.config import make_config
    from cavgym_b200.trajectories import load_episodes
    meta = copy.deepcopy(load_golden("pedestrians_rc_seed0")[0])
    cfg = meta["config"]
    cfg.update(max_timesteps=60, episodes=512, seed=3, episode_log=str(tmp_path / "main" / "episode.log"),
               run_log=str(tmp_path / "main" / "run.log"))
    (tmp_path / "main").mkdir()
    path = tmp_path / "config.json"
    path.write_text(json.dumps(cfg))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run([sys.executable, "-m", "cavgym_b200.sweep", str(path), "--epsilon", "1.0,0.5", "--envs-per-point", "256",
                    "--episodes", "512", "--log-dir", str(tmp_path / "sweep"), "--save-interesting", "5"], check=True, cwd=root)
    subprocess.run([sys.executable, "-m", "cavgym_b200", str(path), "--envs", "256", "--save-interesting", "7"], check=True, cwd=root)
    files = [tmp_path / "sweep" / "epsilon=1" / "interesting.npz", tmp_path / "sweep" / "epsilon=0.5" / "interesting.npz",
             tmp_path / "main" / "interesting.npz"]
    for file, k in zip(files, (5, 5, 7)):
        saved_meta, episodes = load_episodes(file)
        assert len(episodes) <= k
        for ep in episodes:
            assert bool(ep["reproduced"]) and ep["winner"][-1] > 0
        assert make_config(saved_meta["config"]).max_timesteps == 60 and saved_meta["seed"] == 3
        replays_bitwise(cfg, saved_meta["dtype"], episodes)
        print(file, len(episodes))
