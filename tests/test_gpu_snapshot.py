"""Save, restore and fork environments on the device (cavgym_save_envs / load_envs / fork_envs) and engine checkpoints
(state_dict / load_state_dict).

The contract: an env loaded into a slot of the same global env id continues bit for bit on every kernel path; a fork is a
copy that continues on the target slot's own random stream; save, load and fork never touch the counters.  Agent state
holds NaN (None), so envs are compared as the bytes of a full save, next to the engine's exposed views and counters.
"""
import ctypes
import io
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from helpers import compile_from_meta, load_golden, soa

pytestmark = pytest.mark.gpu

NAMES = ("state", "action", "agent", "cs", "liveness", "t_ep", "episode", "winner", "active", "done", "err")


def dense_scenario():
    """The 320-body dense scenario of smoke(): 64 cars and 256 spawned pedestrians, all-pairs collisions."""
    from cavgym_b200.examples.environments import dense_traffic
    from cavgym_b200.library.bodies import Pedestrian
    from cavgym_b200.scenario import AgentSpec, compile_scenario
    road_map, constants = dense_traffic.make_world()
    bodies = dense_traffic.make_bodies(np_random=np.random.RandomState(0), road_map=road_map)
    cfg = SimpleNamespace(terminate_collisions="all", terminate_ego_zones=True, terminate_ego_offroad=False, max_timesteps=1000,
                          reward_win=6000.0, reward_draw=2000.0, cost_step=4.0)
    specs = [AgentSpec("random-constrained", epsilon=0.01) if isinstance(b, Pedestrian) else AgentSpec("noop") for b in bodies]
    return compile_scenario(bodies, constants, cfg, specs)


def engine(name, n, dtype, mode="external", seed=3, env_offset=0, knobs=()):
    from cavgym_b200 import BatchedCAVEnv
    compiled = dense_scenario() if name == "dense320" else compile_from_meta(load_golden(name)[0], mode=mode)
    env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=compiled, seed=seed, env_offset=env_offset)
    for knob, value in knobs:
        getattr(env, knob)(value)
    return env


def golden_actions(name, n, steps, bad_envs=()):
    """Joint actions [steps, M, 2, n]: the golden episodes tiled over the envs (zeros after an episode's end); envs in
    bad_envs get an out-of-range throttle at step 10 (the invalid-action flag)."""
    meta, episodes = load_golden(name)
    m, k = meta["n_bodies"], len(episodes)
    actions = np.zeros((steps, m, 2, n))
    for j, ep in enumerate(episodes):
        a = ep["actions"][:steps]
        actions[:a.shape[0], :, :, j::k] = a[..., None]
    for e in bad_envs:
        actions[10, 0, 0, e] = 1e6
    init = soa(np.stack([episodes[e % k]["init_state"] for e in range(n)]))
    return init, actions


def flat(snap):
    """Every row of a snapshot as bytes (the padding between its 256-byte aligned sections is not state)."""
    return torch.cat([section_bytes(snap, name).reshape(-1) for name in NAMES])


def blob(env, envs=None):
    return flat(env.save_envs(envs))


def counters(env):
    return env.state_dict()["counters"]


def section_bytes(snap, name):
    return snap[name].contiguous().view(torch.uint8).cpu()


# ------------------------------------------------------------------ 1. resume equals uninterrupted, on every path
# name -> (scenario, mode, n, steps before the save, knobs, driver, sections that must differ from a fresh engine at the save)
STEPPED = {"state", "cs", "liveness", "t_ep", "done", "winner", "err"}
CASES = {
    "tma_step": ("pedestrians_rc_seed0", "external", 692, 760, (("set_step_path", True),), "step", STEPPED),
    "plain_step": ("pedestrians_rc_seed0", "external", 692, 760, (("set_step_path", False),), "step", STEPPED),
    "tma_replay_chained": ("pedestrians_rc_seed0", "external", 692, 760, (("set_step_path", True),), "replay", STEPPED),
    "plain_replay": ("pedestrians_rc_seed0", "external", 692, 760, (("set_step_path", False),), "replay", STEPPED),
    "device_step_election": ("learn_election3_seed22", "device", 300, 250, (), "device_step",
                             {"state", "agent", "t_ep", "done", "winner", "active"}),
    "rollout_homogeneous": ("pedestrians_rc_eps05_seed1", "device", 1000, 500, (), "rollout", {"state", "cs", "agent", "t_ep", "episode"}),
    "rollout_heterogeneous": ("busstop_random_all_seed8", "device", 1000, 300, (), "rollout", {"state", "action", "t_ep", "episode"}),
    "rollout_election": ("learn_election3_seed22", "device", 300, 300, (), "rollout", {"state", "agent", "t_ep", "episode", "active"}),
    "warp_per_env_forced": ("pedestrians_rc_eps05_seed1", "device", 300, 500, (("set_dense_path", True),), "rollout",
                            {"state", "cs", "agent", "t_ep", "episode"}),
    "warp_per_env_320_bodies": ("dense320", "device", 37, 30, (), "rollout", {"state", "t_ep"}),
}
REPLAY_CHUNKS = (5, 20, 100, 300, 335)   # 760 steps: consecutive launches chain tile by tile


def test_the_cases_cover_every_section():
    assert set().union(*(case[-1] for case in CASES.values())) == set(NAMES)


def drive(env, driver, actions, t0, steps):
    if driver == "step":
        acts = torch.as_tensor(actions[t0:t0 + steps], dtype=env.dtype, device=env.device)
        for t in range(steps):
            env.step(acts[t])
    elif driver == "replay":
        acts = torch.as_tensor(actions[t0:t0 + steps], dtype=env.dtype, device=env.device)
        t = 0
        for chunk in REPLAY_CHUNKS:
            env.replay(acts[t:t + chunk], record=("state", "done") if chunk % 2 else ())
            t += chunk
        assert t == steps
    elif driver == "device_step":
        for _ in range(steps):
            env.step(None)
    else:
        env.rollout(steps, auto_reset=True)


@pytest.mark.parametrize("aligned", [False, True], ids=["ragged_n", "n_multiple_of_16"])
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_resume_equals_uninterrupted(case, dtype, aligned):
    """K steps, a checkpoint through torch.save / torch.load, a FRESH engine of the same seed and shard, K more steps: every
    per-env byte, the exposed views and the counters equal those of 2K uninterrupted steps.  A ragged N saves and loads
    row by row per element size; N a multiple of 16 takes the one-launch straight copy of every row."""
    name, mode, n, k, knobs, driver, must_differ = CASES[case]
    if aligned:
        n = (n + 15) // 16 * 16
    actions = None
    init = None
    if mode == "external":
        init, actions = golden_actions(name, n, 2 * k, bad_envs=(3, 100))
    envs = [engine(name, n, dtype, mode, knobs=knobs) for _ in range(3)]   # uninterrupted, saved, resumed
    for env in envs[:2]:
        env.reset(init_state=init)
    drive(envs[0], driver, actions, 0, k)
    drive(envs[0], driver, actions, k, k)
    drive(envs[1], driver, actions, 0, k)
    saved = envs[1].save_envs()
    buffer = io.BytesIO()
    torch.save(envs[1].state_dict(), buffer)
    buffer.seek(0)
    checkpoint = torch.load(buffer)
    fresh = envs[2].save_envs()
    differ = {s for s in NAMES if not torch.equal(section_bytes(saved, s), section_bytes(fresh, s))}
    assert must_differ <= differ, f"sections that differ from a fresh engine at the save: {sorted(differ)}"
    envs[2].load_state_dict(checkpoint)
    assert torch.equal(blob(envs[2]), flat(saved))
    drive(envs[2], driver, actions, k, k)
    want, got = envs[0], envs[2]
    assert torch.equal(blob(got), blob(want))
    for attr in ("state", "actions_taken", "agent_state", "episode_liveness", "timestep", "done_latch", "winner_latch", "error"):
        assert torch.equal(getattr(got, attr).contiguous().view(torch.uint8), getattr(want, attr).contiguous().view(torch.uint8)), attr
    assert torch.equal(counters(got), counters(want)) and got.stats() == want.stats()
    assert got.state_dict()["t_global"] == want.state_dict()["t_global"] == 2 * k


# ------------------------------------------------------------------ 2. state_dict round trip and refusals
def test_state_dict_refuses_another_scenario_dtype_env_count_or_seed():
    from cavgym_b200 import EnvSnapshot
    base = engine("pedestrians_rc_seed0", 96, "float64", mode="device", seed=3)
    base.reset()
    checkpoint = base.state_dict()
    for other in (engine("pedestrians_rc_eps05_seed1", 96, "float64", mode="device", seed=3),   # same bodies, tester epsilon differs
                  engine("pedestrians_rc_seed0", 96, "float32", mode="device", seed=3),
                  engine("pedestrians_rc_seed0", 97, "float64", mode="device", seed=3),
                  engine("pedestrians_rc_seed0", 96, "float64", mode="device", seed=4),
                  engine("pedestrians_rc_seed0", 96, "float64", mode="device", seed=3, env_offset=96)):
        with pytest.raises(ValueError):
            other.load_state_dict(checkpoint)
    engine("pedestrians_rc_seed0", 96, "float64", mode="device", seed=3).load_state_dict(checkpoint)
    snap = base.save_envs([0, 1, 2])
    for other in (engine("pedestrians_rc_eps05_seed1", 8, "float64", mode="device"), engine("pedestrians_rc_seed0", 8, "float32", mode="device"),
                  engine("pedestrians3_rc_seed2", 8, "float64", mode="device")):
        with pytest.raises(ValueError):
            other.load_envs(snap, [0, 1, 2])
    with pytest.raises(ValueError):
        base.load_envs(snap, [0, 1, 1])                       # repeated target
    with pytest.raises(ValueError):
        base.load_envs(snap, [0, 1, 96])                      # out of range
    with pytest.raises(ValueError):
        base.load_envs(snap, [0, 1])                          # count
    with pytest.raises(ValueError):
        base.fork([0, -1], [2, 3])
    with pytest.raises(ValueError):
        base.fork([0, 1], [2, 2])
    with pytest.raises(ValueError):
        base.save_envs([0, 96])
    with pytest.raises(ValueError):
        base.load_envs(EnvSnapshot(snap.data[:-1], snap.layout), [0, 1, 2])
    # the C entries refuse what they can check without reading device memory
    lib, h = base._lib, base._handle
    assert lib.cavgym_save_envs(h, None, 95, ctypes.c_void_p(snap.data.data_ptr()), None) == -22
    assert lib.cavgym_save_envs(h, None, 96, None, None) == -22
    assert lib.cavgym_load_envs(h, None, -1, None, None) == -22
    assert lib.cavgym_fork_envs(h, None, None, 4, None) == -22
    idx = torch.arange(97, device=base.device)
    assert lib.cavgym_fork_envs(h, ctypes.c_void_p(idx.data_ptr()), ctypes.c_void_p(idx.data_ptr()), 97, None) == -22
    assert lib.cavgym_snapshot_layout(h, -1, ctypes.byref(snap.layout)) == -22
    state = base._engine_state()
    state.fingerprint ^= 1
    assert lib.cavgym_load_engine(h, ctypes.byref(state)) == -22


def test_snapshot_views_and_layout():
    env = engine("pedestrians3_rc_seed2", 50, "float32", mode="device")
    env.reset()
    env.rollout(40)
    snap = env.save_envs([7, 3, 3])
    lay = snap.layout
    assert lay.k == 3 and lay.m == 4 and lay.real_rows == 4 * 13 and lay.i32_rows == 8 and lay.u8_rows == 2   # ego + 3 pedestrians
    assert lay.i32_offset % 256 == 0 and lay.u8_offset % 256 == 0 and snap.data.numel() == lay.total_bytes
    assert torch.equal(snap["state"], env.state[:, :, [7, 3, 3]])
    assert torch.equal(snap["liveness"], env.episode_liveness[:, [7, 3, 3]])
    assert torch.equal(snap["t_ep"], env.timestep[[7, 3, 3]]) and torch.equal(snap["done"], env.done_latch[[7, 3, 3]])
    assert torch.equal(snap["agent"].view(torch.int32), env.agent_state[:, :, [7, 3, 3]].view(torch.int32))
    host = snap.cpu()
    assert host.device.type == "cpu" and torch.equal(host["state"], snap["state"].cpu())
    assert host.to(env.device)["winner"].device == env.device


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_whole_engine_copy_equals_the_indexed_path(dtype):
    """With N a multiple of 16, saving or loading all envs in order is ONE launch that copies every row as 16-byte words.
    It must give the bytes of the per-element path (the same envs through an index list), match the engine's exposed views,
    and load back to the same engine state."""
    n = 1024 + 16 * 3
    env = engine("busstop_random_all_seed8", n, dtype, mode="device", seed=4)
    env.reset()
    env.rollout(260, auto_reset=True)                      # episodes ended and restarted: every row is far from its start
    order = torch.arange(n, device=env.device)
    before = env.launch_count()
    whole = env.save_envs()
    assert env.launch_count() == before + 1               # the straight copy
    indexed = env.save_envs(order)
    assert env.launch_count() == before + 1 + (2 if dtype == "float32" else 3)
    for name in NAMES:
        assert torch.equal(section_bytes(whole, name), section_bytes(indexed, name)), name
    views = {"state": env.state, "action": env.actions_taken, "agent": env.agent_state, "liveness": env.episode_liveness,
             "t_ep": env.timestep, "winner": env.winner_latch, "done": env.done_latch, "err": env.error}
    for name, view in views.items():
        assert torch.equal(section_bytes(whole, name), view.contiguous().view(torch.uint8).cpu()), name
    assert len(torch.unique(whole["episode"])) > 1
    # load: the straight copy into one engine, the indexed scatter into another, from the same snapshot of a third state
    other = engine("busstop_random_all_seed8", n, dtype, mode="device", seed=4)
    other.reset()
    other.rollout(37, auto_reset=True)
    target = other.save_envs()
    a, b = (engine("busstop_random_all_seed8", n, dtype, mode="device", seed=4) for _ in range(2))
    a.load_envs(target)
    b.load_envs(target, order)
    for e in (a, b):
        e.set_global_timestep(37)
        assert torch.equal(blob(e), flat(target))
        e.rollout(100, auto_reset=True)
    other.rollout(100, auto_reset=True)
    assert torch.equal(blob(a), blob(other)) and torch.equal(blob(b), blob(other))


def test_empty_selections_do_nothing_and_misaligned_snapshots_are_refused():
    env = engine("pedestrians_rc_seed0", 64, "float64", mode="device")
    env.reset()
    env.rollout(30)
    before = blob(env)
    empty = env.save_envs([])
    assert empty.k == 0 and empty.data.numel() == 0
    env.load_envs(empty, [])
    env.fork([], [])
    env.fork(torch.empty(0, dtype=torch.int64), torch.empty(0, dtype=torch.int64))
    assert torch.equal(blob(env), before)
    from cavgym_b200 import EnvSnapshot
    snap = env.save_envs([1, 2])
    room = torch.zeros(snap.data.numel() + 16, dtype=torch.uint8, device=env.device)
    shifted = room[8:8 + snap.data.numel()]
    shifted.copy_(snap.data)
    with pytest.raises(ValueError):
        env.load_envs(EnvSnapshot(shifted, snap.layout), [1, 2])
    lib, h = env._lib, env._handle
    idx = torch.tensor([1, 2], device=env.device)
    assert lib.cavgym_save_envs(h, ctypes.c_void_p(idx.data_ptr()), 2, ctypes.c_void_p(shifted.data_ptr()), None) == -22
    assert lib.cavgym_load_envs(h, ctypes.c_void_p(idx.data_ptr()), 2, ctypes.c_void_p(shifted.data_ptr()), None) == -22
    assert lib.cavgym_save_envs(h, None, 0, None, None) == 0 and lib.cavgym_fork_envs(h, None, None, 0, None) == 0
    assert torch.equal(blob(env), before)


# ------------------------------------------------------------------ 3. fork
def gather_columns(snap, src, dst):
    """The snapshot with column dst[j] replaced by column src[j] (numpy, section by section)."""
    lay = snap.layout
    data = snap.data.cpu().numpy().copy()
    for offset, rows, size in ((lay.real_offset, lay.real_rows, 8 if lay.dtype == 0 else 4), (lay.i32_offset, lay.i32_rows, 4),
                               (lay.u8_offset, lay.u8_rows, 1)):
        part = data[offset:offset + rows * lay.k * size].reshape(rows, lay.k, size)
        part[:, dst] = part[:, src].copy()
    from cavgym_b200 import EnvSnapshot
    return EnvSnapshot(torch.from_numpy(data), lay)


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_random_resample_equals_save_gather_load(dtype):
    n = 4000 + 13
    rng = np.random.default_rng(1)
    a, b = (engine("busstop_random_all_seed8", n, dtype, mode="device", seed=9) for _ in range(2))
    for env in (a, b):
        env.reset()
        env.rollout(200)
    before = counters(a)
    for src, dst in ((rng.integers(0, n, n), np.arange(n)),                                  # resample: repeats, dst = all
                     (rng.integers(0, 50, 700), rng.permutation(n)[:700])):                  # few sources into a random subset
        a.fork(torch.as_tensor(src), dst.tolist())
        b.load_envs(gather_columns(b.save_envs(), src, dst))
        assert torch.equal(blob(a), blob(b))
        for env in (a, b):
            env.rollout(60)
        assert torch.equal(blob(a), blob(b))
    assert torch.equal(counters(a), counters(b))
    # counters: fork and load leave the raw counters alone
    c = counters(a)
    a.fork(0, list(range(n)))
    a.load_envs(b.save_envs())
    assert torch.equal(counters(a), c) and not torch.equal(c, before)


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_broadcast_fork_under_identical_actions_gives_identical_columns(dtype):
    n = 224 * 3 + 20
    init, actions = golden_actions("pedestrians_rc_seed0", n, 300)
    env = engine("pedestrians_rc_seed0", n, dtype)
    env.reset(init_state=init)
    acts = torch.as_tensor(actions, dtype=env.dtype, device=env.device)
    env.replay(acts[:120], record=())
    env.fork(4, torch.arange(n))
    same = acts[120:, :, :, 4:5].expand(-1, -1, -1, n).contiguous()
    env.replay(same[:100], record=())
    for t in range(100, 180):
        env.step(same[t])
    snap = env.save_envs()
    for s in NAMES:
        col = snap[s]
        assert torch.equal(col.contiguous().view(torch.uint8).reshape(-1, n, col.element_size())[:, :1].expand(-1, n, -1),
                           col.contiguous().view(torch.uint8).reshape(-1, n, col.element_size())), s


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_forked_env_continues_on_its_own_key(dtype):
    """A fork with on-device agents is exactly the source's snapshot continued under the target's global id: a one-env engine
    whose shard offset gives its env 0 that id, loaded with the source's snapshot, runs the same bits."""
    n, src, k = 300, 5, 150
    targets = list(range(217, 237))
    env = engine("busstop_random_all_seed8", n, dtype, mode="device", seed=11, env_offset=1000)   # RandomAgents redraw with eps
    env.reset()
    env.rollout(k, auto_reset=True)
    source = env.save_envs([src])
    env.fork(src, targets)
    assert all(torch.equal(blob(env, [t]), flat(source)) for t in targets)
    single = engine("busstop_random_all_seed8", 1, dtype, mode="device", seed=11, env_offset=1000 + targets[0])
    single.load_envs(source)
    single.set_global_timestep(k)
    for e in (env, single):
        e.rollout(400, auto_reset=True)
    assert torch.equal(blob(env, [targets[0]]), blob(single))
    copies = {bytes(blob(env, [t]).numpy()) for t in [src] + targets}
    assert len(copies) > 1          # the copies diverged: each continues on its own slot's stream


# ------------------------------------------------------------------ 4. shards merge
@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_shard_snapshots_merge_into_one_engine(dtype):
    n, k = 1500, 400
    shards = [engine("pedestrians_rc_eps05_seed1", n, dtype, mode="device", seed=5, env_offset=r * n) for r in range(2)]
    for s in shards:
        s.reset()
        s.rollout(k, auto_reset=True)
    whole = engine("pedestrians_rc_eps05_seed1", 2 * n, dtype, mode="device", seed=5)
    for r, s in enumerate(shards):
        whole.load_envs(s.save_envs(), torch.arange(r * n, (r + 1) * n))
    whole.set_global_timestep(k)
    for e in shards + [whole]:
        e.rollout(k, auto_reset=True)
    merged = whole.save_envs()
    for r, s in enumerate(shards):
        part = s.save_envs()
        for name in NAMES:
            assert torch.equal(merged[name][..., r * n:(r + 1) * n].contiguous().view(torch.uint8), part[name].contiguous().view(torch.uint8)), name


# ------------------------------------------------------------------ 5. launch chaining
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("n", [224 * 300, 224 * 37 + 48])
def test_fork_and_load_inside_a_chained_replay_train(dtype, n):
    """A train of cavgym_replay launches issued without any host synchronisation, with a save, a fork and a load in the
    middle (through the C-ABI: the Python checks of the indices would synchronise), equals the same train on the plain
    kernels.  A snapshot launch ordered only programmatically behind replay_tma_kernel would read or overwrite env state
    under the running replay."""
    init, actions = golden_actions("pedestrians_rc_seed0", n, 260)
    envs = [engine("pedestrians_rc_seed0", n, dtype), engine("pedestrians_rc_seed0", n, dtype, knobs=(("set_step_path", False),))]
    rng = np.random.default_rng(2)
    src = torch.as_tensor(rng.integers(0, n, n // 2), device=envs[0].device)
    dst = torch.as_tensor(rng.permutation(n)[:n // 2], device=envs[0].device)
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731
    results = []
    for env in envs:
        acts = torch.as_tensor(actions, dtype=env.dtype, device=env.device)
        layout = env._layout(n)
        saved = torch.empty(int(layout.total_bytes), dtype=torch.uint8, device=env.device)
        lib, h, stream = env._lib, env._handle, env._stream()
        # the first fork allocates the engine's staging snapshot (and synchronises): do it before the train
        assert lib.cavgym_fork_envs(h, ptr(src), ptr(dst), src.numel(), stream) == 0
        env.reset(init_state=init)
        outs, t = [], 0
        for i, chunk in enumerate([5, 5, 20, 20, 20, 3, 20, 20, 20, 5, 40, 40, 20, 20]):
            if i == 3:
                assert lib.cavgym_save_envs(h, None, n, ptr(saved), stream) == 0
            if i == 6:
                assert lib.cavgym_fork_envs(h, ptr(src), ptr(dst), src.numel(), stream) == 0
            if i == 10:
                assert lib.cavgym_load_envs(h, None, n, ptr(saved), stream) == 0
            outs.append(env.replay(acts[t:t + chunk], record=("state", "reward", "done", "winner", "tangent") if i % 2 else ("state",)))
            t += chunk
        results.append(outs)
    torch.cuda.synchronize()
    for a, b in zip(*results):
        for key in a:
            if a[key] is not None:
                assert torch.equal(a[key], b[key]), key
    assert torch.equal(blob(envs[0]), blob(envs[1]))
    assert torch.equal(counters(envs[0]), counters(envs[1]))
