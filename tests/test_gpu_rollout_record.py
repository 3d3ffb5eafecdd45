"""Recorded rollouts (BatchedCAVEnv.rollout(..., record=...), cavgym_rollout_record) on every rollout path.

The contract: recording changes nothing else (engine bytes, counters, episode rows, t_global); every row equals what the
single-step path with device agents returns at that step, frozen rows included; the complete episodes of a record replay
bit for bit on external actions, and match the C oracle, on its replay and on its own device-agent run.

Scenarios run with max_timesteps lowered to 23 so that, in windows of 30 and 35 steps, episodes end (cut off, or done) and
restart inside a window, and the batch-wide t_global passes max_timesteps - 1 (the time-out reward, quirk 1).
"""
import copy
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from helpers import compile_from_meta, load_golden, matrix_scenario, state_err

pytestmark = pytest.mark.gpu

MAX_T = 23
WINDOWS = (30, 35)
FIELDS = ("observation", "action", "state", "reward", "done", "winner", "tangent", "timestep")
SNAP = ("state", "action", "agent", "cs", "liveness", "t_ep", "episode", "winner", "active", "done", "err")

# name -> (golden scenario, envs, knobs)
CASES = {
    "homogeneous_2_bodies": ("pedestrians_rc_eps05_seed1", 203, ()),
    "homogeneous_rolled_4_bodies": ("pedestrians3_rc_seed2", 203, ()),
    "synced_crossroads": ("crossroads_random_all_seed6", 203, ()),
    "synced_bus_stop": ("busstop_random_all_seed8", 203, ()),
    "synced_pelican_crossing": ("pelican_random_all_seed10", 203, ()),
    "election": ("learn_election3_seed22", 203, ()),
    "warp_per_env_forced": ("pedestrians_rc_eps05_seed1", 75, (("set_dense_path", True),)),
    "warp_per_env_320_bodies": ("dense320", 37, ()),
}
# the other cells of the (body count, family) matrix of helpers.matrix_scenario: every M = 1..8 of both families runs here
MATRIX_CELLS = [(1, "homogeneous"), (3, "homogeneous"), (5, "homogeneous"), (6, "homogeneous"), (7, "homogeneous"),
                (8, "homogeneous"), (1, "generic"), (2, "generic"), (4, "generic"), (6, "generic"), (7, "generic"), (8, "generic")]
CASES.update({f"matrix_{family}_{m}_bodies": (("matrix", m, family), 203, ()) for m, family in MATRIX_CELLS})


def compiled(name, mode):
    if isinstance(name, tuple):
        return matrix_scenario(name[1], name[2], mode, max_timesteps=MAX_T)
    if name == "dense320":
        from cavgym_b200.examples.environments import dense_traffic
        from cavgym_b200.library.bodies import Pedestrian
        from cavgym_b200.scenario import AgentSpec, compile_scenario
        road_map, constants = dense_traffic.make_world()
        bodies = dense_traffic.make_bodies(np_random=np.random.RandomState(0), road_map=road_map)
        cfg = SimpleNamespace(terminate_collisions="all", terminate_ego_zones=True, terminate_ego_offroad=False, max_timesteps=MAX_T,
                              reward_win=6000.0, reward_draw=2000.0, cost_step=4.0)
        specs = [AgentSpec("external") if mode == "external" else
                 AgentSpec("random-constrained", epsilon=0.01) if isinstance(b, Pedestrian) else AgentSpec("noop") for b in bodies]
        return compile_scenario(bodies, constants, cfg, specs)
    meta = copy.deepcopy(load_golden(name)[0])
    meta["config"]["max_timesteps"] = MAX_T
    return compile_from_meta(meta, mode=mode)


def engine(case, dtype, mode="device", n=None, knobs=None, seed=5):
    from cavgym_b200 import BatchedCAVEnv
    name, n_case, case_knobs = CASES[case]
    env = BatchedCAVEnv(None, None, None, num_envs=n or n_case, dtype=dtype, compiled=compiled(name, mode), seed=seed)
    for knob, value in (case_knobs if knobs is None else knobs):
        getattr(env, knob)(value)
    return env


def host(t):
    return t.cpu().numpy()


def snapshot_bytes(env):
    snap = env.save_envs()
    return torch.cat([snap[name].contiguous().view(torch.uint8).reshape(-1) for name in SNAP]).cpu()


_RUNS = {}


def run(case, dtype, auto_reset):
    """Twin engines over WINDOWS: `rec` records every field, `plain` does not, `steps` runs step() with device agents and
    action logging, resetting finished envs before a step when auto-resetting.  Returns the windows' records, t_global at
    their starts, the single-step rows and the three engines."""
    key = (case, dtype, auto_reset)
    if key in _RUNS:
        return _RUNS[key]
    rec, plain, steps = engine(case, dtype), engine(case, dtype), engine(case, dtype)
    for env in (rec, plain):
        env.set_episode_log(1 << 14)
    steps.set_action_logging(True)
    records, starts = [], []
    single = {name: [] for name in FIELDS}
    t_global = 0
    for window in WINDOWS:
        starts.append(t_global)
        records.append({k: host(v) for k, v in rec.rollout(window, auto_reset=auto_reset, record=FIELDS).items()})
        assert plain.rollout(window, auto_reset=auto_reset) is None
        for _ in range(window):
            if auto_reset:
                steps.reset(mask=steps.done_latch.clone())
            stepped = host(steps.done_latch) == 0
            single["observation"].append(host(steps.state).copy())
            state, reward, done, winner, tangent = steps.step(None)
            single["state"].append(host(state).copy())
            single["reward"].append(host(reward).copy())
            single["done"].append(host(done).copy())
            single["winner"].append(host(winner).copy())
            single["tangent"].append(host(tangent).copy())
            single["action"].append(np.where(stepped[None, None], host(steps.actions_taken), 0))
            single["timestep"].append(np.where(stepped, host(steps.timestep), 0))
        t_global += window
    torch.cuda.synchronize()
    single = {k: np.stack(v) for k, v in single.items()}
    _RUNS[key] = (records, starts, single, rec, plain, steps)
    return _RUNS[key]


def concat(records):
    return {k: np.concatenate([r[k] for r in records]) for k in FIELDS}


@pytest.mark.parametrize("auto_reset", [True, False], ids=["auto_reset", "no_reset"])
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_recording_changes_nothing_and_rows_equal_single_steps(case, dtype, auto_reset):
    records, starts, single, rec, plain, _ = run(case, dtype, auto_reset)
    # 1. the recorded engine is the plain one, byte for byte
    assert torch.equal(snapshot_bytes(rec), snapshot_bytes(plain))
    assert rec.stats() == plain.stats()
    rows_rec, dropped_rec = rec.drain_episodes()
    rows_plain, dropped_plain = plain.drain_episodes()
    assert dropped_rec == dropped_plain == 0 and len(rows_rec) > 0   # rows are appended in completion order: sort both
    assert np.array_equal(np.sort(rows_rec, order=["env", "episode"]), np.sort(rows_plain, order=["env", "episode"]))
    assert rec.state_dict()["t_global"] == plain.state_dict()["t_global"] == sum(WINDOWS)
    # 2. every row is the single-step path's, bitwise
    got = concat(records)
    for name in FIELDS:
        assert got[name].shape == single[name].shape, name
        assert np.array_equal(got[name].view(np.uint8), single[name].astype(got[name].dtype).view(np.uint8)), \
            f"{name}: first differing row {np.argwhere(got[name] != single[name])[:1]}"
    # the windows cover what they are meant to: episodes that end, restarts (or frozen rows) inside a window
    ts = got["timestep"]
    assert (ts == 1)[1:].any() if auto_reset else (ts == 0).any()
    assert ((ts > 0) & ((got["done"] == 1) | (ts == MAX_T))).any()


@pytest.mark.parametrize("auto_reset", [True, False], ids=["auto_reset", "no_reset"])
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_complete_episodes_replay_bitwise_on_external_actions(case, dtype, auto_reset):
    from cavgym_b200.trajectories import complete_episodes
    records, starts, *_ = run(case, dtype, auto_reset)
    episodes = [ep for record, t0 in zip(records, starts) for ep in complete_episodes(record, t0, max_timesteps=MAX_T)]
    assert episodes
    by_start = {}
    for ep in episodes:
        by_start.setdefault(ep["t_global_start"], []).append(ep)
    knobs = tuple(k for k in CASES[case][2] if k[0] == "set_dense_path")
    for t0, group in by_start.items():
        k, length = len(group), max(len(ep["done"]) for ep in group)
        m = group[0]["init_state"].shape[0]
        env = engine(case, dtype, mode="external", n=k, knobs=knobs)
        actions = np.zeros((length, m, 2, k), dtype=group[0]["actions"].dtype)
        for j, ep in enumerate(group):
            actions[:len(ep["done"]), :, :, j] = ep["actions"]
        env.set_global_timestep(t0)
        env.reset(init_state=np.stack([ep["init_state"] for ep in group], axis=-1))
        out = {name: host(v) for name, v in env.replay(actions).items()}
        for j, ep in enumerate(group):
            steps = len(ep["done"])
            assert np.array_equal(out["state"][:steps, :, :, j], ep["state"]), (t0, j)
            assert np.array_equal(out["reward"][:steps, :, j], ep["reward"]), (t0, j)
            for name in ("done", "winner", "tangent"):
                assert np.array_equal(out[name][:steps, j], ep[name]), (name, t0, j)


# the C oracle has no election agents; the warp-per-env cases are held to the thread-per-env rows by the tests above
ORACLE_CASES = ("homogeneous_2_bodies", "homogeneous_rolled_4_bodies", "synced_crossroads", "synced_bus_stop",
                "synced_pelican_crossing") + tuple(f"matrix_{family}_{m}_bodies" for m, family in MATRIX_CELLS)


@pytest.mark.parametrize("auto_reset", [True, False], ids=["auto_reset", "no_reset"])
@pytest.mark.parametrize("case", ORACLE_CASES)
def test_against_the_oracle_fp64(case, auto_reset):
    """The oracle replays the extracted episodes (state and rewards within 1e-9, events identical off flagged steps), and
    its own device-agent run, one step at a time on the same Philox streams, gives the recorded observation, action and
    state rows (1e-9) until an env's first flagged step."""
    from cavgym_b200.trajectories import complete_episodes
    from oracle.oracle import Oracle
    records, starts, *_ = run(case, "float64", auto_reset)
    name = CASES[case][0]
    for record, t0 in zip(records, starts):
        episodes = complete_episodes(record, t0, max_timesteps=MAX_T)
        for t_start in sorted({ep["t_global_start"] for ep in episodes}):
            group = [ep for ep in episodes if ep["t_global_start"] == t_start]
            length, m = max(len(ep["done"]) for ep in group), group[0]["init_state"].shape[0]
            actions = np.zeros((length, m, 2, len(group)))
            for j, ep in enumerate(group):
                actions[:len(ep["done"]), :, :, j] = ep["actions"]
            oracle = Oracle(compiled(name, "external"), len(group))
            oracle.set_global_timestep(t_start)
            oracle.reset(init_state=np.stack([ep["init_state"] for ep in group], axis=-1))
            state, reward, done, winner, _ = oracle.replay(actions)
            for j, ep in enumerate(group):
                steps = len(ep["done"])
                flagged = np.flatnonzero(ep["tangent"])
                upto = steps if flagged.size == 0 else flagged[0]
                assert state_err(state[:upto, :, :, j], ep["state"][:upto]) <= 1e-9
                assert np.max(np.abs(reward[:upto, :, j] - ep["reward"][:upto]) / np.maximum(1, np.abs(ep["reward"][:upto])), initial=0) <= 1e-9
                assert np.array_equal(done[:upto, j], ep["done"][:upto]) and np.array_equal(winner[:upto, j], ep["winner"][:upto])

    got = concat(records)
    n = got["timestep"].shape[1]
    oracle = Oracle(compiled(name, "device"), n, seed=5)
    live = np.ones(n, dtype=bool)   # envs not yet past a flagged step
    for t in range(got["timestep"].shape[0]):
        assert state_err(np.moveaxis(oracle.state[:, :, live], -1, 0), np.moveaxis(got["observation"][t][:, :, live], -1, 0)) <= 1e-9, t
        oracle.rollout(1, auto_reset=auto_reset)
        stepped = live & (got["timestep"][t] > 0)
        kept = stepped & ~(auto_reset & ((got["done"][t] == 1) | (got["timestep"][t] >= MAX_T)))   # not reset after the step
        assert state_err(np.moveaxis(oracle.state[:, :, kept], -1, 0), np.moveaxis(got["state"][t][:, :, kept], -1, 0)) <= 1e-9, t
        assert np.max(np.abs(oracle.actions_taken[:, :, kept] - got["action"][t][:, :, kept]), initial=0) <= 1e-9, t
        live &= got["tangent"][t] == 0
    assert live.sum() > n // 2


# ------------------------------------------------------------------ edges
def test_edges():
    env = engine("homogeneous_2_bodies", "float64", n=67)
    empty = env.rollout(0, record=FIELDS)
    assert all(v.shape[0] == 0 for v in empty.values()) and set(empty) == set(FIELDS)
    with pytest.raises(ValueError):
        env.rollout(5, record=("state", "observations"))
    twin = engine("homogeneous_2_bodies", "float64", n=67)
    assert env.rollout(17, record=()) == {}
    twin.rollout(17)
    from cavgym_b200 import _abi
    import ctypes
    assert env._lib.cavgym_rollout_record(env._handle, 9, 1, ctypes.byref(_abi.CavRolloutRecord()), env._stream()) == 0
    assert env._lib.cavgym_rollout_record(env._handle, 4, 1, None, env._stream()) == 0
    twin.rollout(9)   # the same launches: a launch that resets an env writes every row of it back, so the stored
    twin.rollout(4)   # actions of non-random agents depend on where the launches end
    assert torch.equal(snapshot_bytes(env), snapshot_bytes(twin)) and env.stats() == twin.stats()
    external = engine("homogeneous_2_bodies", "float64", mode="external", n=67)
    with pytest.raises(RuntimeError, match="on-device agent") as refused:
        external.rollout(3, record=("state",))
    assert refused.value.code == -1   # CAV_ESTATE
    from cavgym_b200.trajectories import complete_episodes
    record = {k: host(v) for k, v in env.rollout(40, record=("state", "done", "timestep")).items()}
    with pytest.raises(ValueError, match="observation"):
        complete_episodes(record, 0)


def test_slab_offsets_are_64_bit():
    """A state slab of more than 2^31 elements: its last row is the engine's state after the rollout (without auto-reset
    the finished envs stay frozen, so that is every env's last row)."""
    n, steps = 1 << 20, 520   # 520 x 2 x 4 x 2^20 = 4.4e9 elements
    env = engine("homogeneous_2_bodies", "float32", n=n)
    out = env.rollout(steps, auto_reset=False, record=("state",))["state"]
    assert out[-1].numel() * steps > 1 << 31
    assert torch.equal(out[-1], env.state)
    del out
