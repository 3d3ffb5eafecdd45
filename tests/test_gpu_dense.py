"""Warp-per-environment kernels (kernels_dense.cuh; scenarios with more than CAV_SMALL_M bodies, BASELINE config C4) through
the C-ABI:
  * against the thread-per-env kernels on the reference's own scenarios — BITWISE (state, rewards, events, near-tangent
    flags), replayed actions and on-device agents;
  * against the CPU oracle on the dense-traffic scenario (64 cars + 256 spawned pedestrians, terminate_collisions = "all",
    51,040 pairs per env-step): state 1e-9 (fp64) / 1e-4 (fp32), events identical off flagged steps;
  * the fp32 broad phase against an all-pairs separating-axis test written in torch, at scale (no pair may be lost).
"""
from types import SimpleNamespace

import numpy as np
import pytest

from helpers import check_against_oracle, compile_from_meta, load_golden, random_actions, soa, state_err

pytestmark = pytest.mark.gpu


def dense_config(collisions="all"):
    return SimpleNamespace(terminate_collisions=collisions, terminate_ego_zones=True, terminate_ego_offroad=False,
                           max_timesteps=1000, reward_win=6000.0, reward_draw=2000.0, cost_step=4.0)


def dense_scenario(mode, num_cars=64, num_pedestrians=256, epsilon=0.002, collisions="all"):
    from cavgym_b200.examples.environments import dense_traffic
    from cavgym_b200.library.bodies import Pedestrian
    from cavgym_b200.scenario import AgentSpec, compile_scenario
    road_map, constants = dense_traffic.make_world()
    bodies = dense_traffic.make_bodies(num_cars, num_pedestrians, np_random=np.random.RandomState(0), road_map=road_map)
    if mode == "external":
        specs = [AgentSpec("external") for _ in bodies]
    else:   # bodies are ordered along the road, cars and pedestrians interleaved: the agent follows the body's class
        specs = [AgentSpec("noop") if i == 0 else
                 AgentSpec("random-constrained", epsilon=epsilon) if isinstance(body, Pedestrian) else
                 AgentSpec("random", epsilon=epsilon) for i, body in enumerate(bodies)]
    comp = compile_scenario(bodies, constants, dense_config(collisions), specs)
    comp.is_car = np.array([not isinstance(body, Pedestrian) for body in bodies])
    return comp


def make(comp, n, dtype, **kw):
    from cavgym_b200 import BatchedCAVEnv
    return BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=comp, **kw)


def numpy_traj(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


# ------------------------------------------------------------------ dense path == small path, bit for bit
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("name", ["pedestrians_rc_seed0", "pedestrians3_rc_seed2", "busstop_random_all_seed8",
                                  "pelican_random_all_seed10", "crossroads_random_ego_seed7", "pedestrians_random_none_seed5"])
def test_dense_kernels_are_bitwise_equal_to_thread_per_env_kernels(name, dtype):
    import torch
    meta, episodes = load_golden(name)
    n, m = 67, meta["n_bodies"]          # ragged: not a multiple of the warps per CTA
    t_len = max(ep["actions"].shape[0] for ep in episodes)    # whole episodes: every env reaches its terminal step
    init = soa(np.stack([episodes[e % len(episodes)]["init_state"] for e in range(n)]))
    actions = np.zeros((t_len, m, 2, n))
    for e in range(n):
        a = episodes[e % len(episodes)]["actions"][:t_len]
        actions[:a.shape[0], :, :, e] = a
    outs = []
    for dense in (False, True):
        env = make(compile_from_meta(meta), n, dtype)
        env.set_dense_path(dense)
        env.reset(init_state=init)
        env.set_global_timestep(meta["config"]["max_timesteps"] - t_len // 4)   # the one-off time-out reward lands inside the window
        fused = numpy_traj(env.replay(actions[: t_len // 2]))
        stepped = {k: [] for k in ("state", "reward", "done", "winner", "tangent")}
        actions_t = torch.tensor(actions[t_len // 2:], dtype=env.dtype, device=env.device)
        for t in range(actions_t.shape[0]):
            for k, v in zip(stepped, env.step(actions_t[t])):
                stepped[k].append(v.cpu().numpy().copy())
        outs.append((fused, {k: np.stack(v) for k, v in stepped.items()}, env.episode_liveness.cpu().numpy(),
                     env.timestep.cpu().numpy(), env.stats()))
    for part in (0, 1):
        for key in ("state", "reward", "done", "winner", "tangent"):
            assert np.array_equal(outs[0][part][key], outs[1][part][key], equal_nan=True), (part, key)
    assert np.array_equal(outs[0][2], outs[1][2]) and np.array_equal(outs[0][3], outs[1][3])
    assert outs[0][4] == outs[1][4]
    if name not in ("crossroads_random_ego_seed7", "pedestrians_random_none_seed5"):   # those traces only time out
        assert outs[0][0]["done"].any() or outs[0][1]["done"].any()


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("name", ["pedestrians_rc_seed0", "pedestrians_proximity_seed3", "pelican_random_all_seed10",
                                  "busstop_random_all_seed8"])
def test_dense_rollout_with_device_agents_is_bitwise_equal_to_thread_per_env_rollout(name, dtype):
    meta, _ = load_golden(name)
    n = 130
    results = []
    for dense in (False, True):
        env = make(compile_from_meta(meta, mode="device"), n, dtype, seed=11, env_offset=5)
        env.set_dense_path(dense)
        env.set_action_logging(True)
        env.reset()
        env.rollout(700, auto_reset=True)
        env.rollout(650, auto_reset=True)
        results.append((env.state.cpu().numpy(), env.agent_state.cpu().numpy(), env.actions_taken.cpu().numpy(),
                        env.episode_liveness.cpu().numpy(), env.timestep.cpu().numpy(), env.stats()))
    for a, b in zip(results[0][:5], results[1][:5]):
        assert np.array_equal(a, b, equal_nan=True)
    assert results[0][5] == results[1][5]
    assert results[0][5]["episodes"] >= n


@pytest.mark.parametrize("name", ["busstop_random_all_seed8", "pelican_random_all_seed10", "crossroads_random_all_seed6"])
def test_rollout_without_auto_reset_on_a_ragged_batch(name):
    """The heterogeneous rollout kernels put block-wide barriers inside the step (kernels_small.cuh): lanes without an env
    (130 envs = four warps and two lanes) and envs that finished and stay finished (auto_reset off) must pass the same
    barriers as the lanes that are stepping.  Thread-per-env and warp-per-env paths must agree bitwise, and finished envs
    must stop where they ended."""
    meta, _ = load_golden(name)
    n = 130
    results = []
    for dense in (False, True):
        env = make(compile_from_meta(meta, mode="device"), n, "float64", seed=4)
        env.set_dense_path(dense)
        env.reset()
        env.rollout(500, auto_reset=False)
        frozen = env.state.clone()
        finished = env.done_latch.clone() != 0
        env.rollout(300, auto_reset=False)
        state = env.state.cpu().numpy()
        assert np.array_equal(state[:, :, finished.cpu().numpy()], frozen.cpu().numpy()[:, :, finished.cpu().numpy()])
        results.append((state, env.timestep.cpu().numpy(), env.done_latch.cpu().numpy(), env.stats()))
    assert np.array_equal(results[0][0], results[1][0]) and np.array_equal(results[0][1], results[1][1])
    assert np.array_equal(results[0][2], results[1][2]) and results[0][3] == results[1][3]
    assert results[0][2].any()


# ------------------------------------------------------------------ dense traffic (C4) vs the oracle
@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_dense_traffic_replay_matches_oracle(dtype):
    """64 cars + 256 pedestrians, random valid joint actions: cavgym_replay and cavgym_step vs the oracle."""
    import torch
    from oracle.oracle import Oracle
    n, t_len, cars, peds = 10, 120, 64, 256
    comp = dense_scenario("external")
    rng = np.random.RandomState(5)
    actions = random_actions(rng, t_len, n, comp.is_car)
    oracle = Oracle(dense_scenario("external"), n, seed=9, threads=8)
    oracle.reset()
    init = oracle.state.copy()          # the oracle's Philox spawn draws, replayed as initial states
    want = oracle.replay(actions)
    env = make(comp, n, dtype, seed=9)
    env.reset(init_state=init)
    fused = numpy_traj(env.replay(actions))
    fused = {k: (v.astype(np.float64) if v.dtype == np.float32 else v) for k, v in fused.items()}
    ended = check_against_oracle(fused, want, dtype)
    assert ended >= 3, "the action script should make several envs collide inside the window"
    if dtype == "float64":
        assert np.array_equal(env.episode_liveness.cpu().numpy(), oracle.liveness) or fused["tangent"].any()
    # the same through cavgym_step, one launch per timestep: bitwise the fused result
    env.reset(init_state=init)
    env.set_global_timestep(0)
    actions_t = torch.tensor(actions, dtype=env.dtype, device=env.device)
    for t in range(t_len):
        state, reward, done, winner, tangent = env.step(actions_t[t])
        if t % 17 == 0 or t == t_len - 1:
            assert np.array_equal(state.cpu().numpy().astype(np.float64), fused["state"][t])
            assert np.array_equal(reward.cpu().numpy().astype(np.float64), fused["reward"][t])
            assert np.array_equal(done.cpu().numpy(), fused["done"][t]) and np.array_equal(winner.cpu().numpy(), fused["winner"][t])


def test_dense_traffic_device_agents_match_oracle():
    """On-device agents on the shared Philox stream (spawns, RandomAgent cars, RandomConstrained pedestrians), auto-reset:
    engine and oracle must agree on every episode statistic and on the final state."""
    from oracle.oracle import Oracle
    n, steps = 12, 260
    env = make(dense_scenario("device", epsilon=0.004), n, "float64", seed=21, env_offset=3)
    env.reset()
    oracle = Oracle(dense_scenario("device", epsilon=0.004), n, seed=21, threads=8)
    oracle.set_shard(3)
    oracle.reset()
    assert np.array_equal(env.state.cpu().numpy(), oracle.state)
    env.rollout(steps, auto_reset=True)
    oracle.rollout(steps, auto_reset=True)
    got, want = env.stats(), oracle.stats()
    if got["tangent"] == 0 and want["tangent"] == 0:
        for key in ("episodes", "interesting", "sum_t", "sum_t2", "sum_score", "sum_score2", "env_steps", "sum_t_interesting", "sum_t2_interesting"):
            assert got[key] == want[key], key
        assert state_err(np.moveaxis(env.state.cpu().numpy(), 1, -1), np.moveaxis(oracle.state, 1, -1)) < 1e-9
    else:   # a flagged near-tangent decision may legitimately differ: episode counts stay close
        assert abs(got["episodes"] - want["episodes"]) <= max(2, want["episodes"] // 10)
    assert want["episodes"] >= n // 2, "the agents should end several episodes inside the window"


def test_dense_invalid_action_sets_error_flag_and_leaves_state():
    import torch
    n, cars, peds = 6, 64, 256
    env = make(dense_scenario("external"), n, "float64", seed=2)
    env.reset()
    before = env.state.clone()
    actions = torch.zeros((cars + peds, 2, n), dtype=torch.float64, device=env.device)
    actions[300, 1, 4] = 10.0    # steering far outside every body's limits, one body of one env
    state, reward, done, winner, _ = env.step(actions)
    torch.cuda.synchronize()
    err = env.error.cpu().numpy()
    assert err.tolist() == [0, 0, 0, 0, 1, 0]
    assert torch.equal(state[:, :, 4], before[:, :, 4]) and float(reward[:, 4].abs().max()) == 0.0
    assert not torch.equal(state[:, :, 3], before[:, :, 3])
    assert env.timestep.cpu().numpy().tolist() == [1, 1, 1, 1, 0, 1]


def all_pairs_reference(state, half_length, half_width, dynamic):
    """Closed separating-axis test of every pair of boxes, torch fp64 (test-side check of the kernel's broad + narrow
    phase): state [M, 4, N] -> bool [N] any pair intersects, and the smallest |margin| met."""
    import torch
    x, y, th = state[:, 0].T, state[:, 1].T, state[:, 3].T        # [N, M]
    c, s = torch.cos(th), torch.sin(th)
    hl, hw = half_length[None], half_width[None]
    tx, ty = x[:, None, :] - x[:, :, None], y[:, None, :] - y[:, :, None]     # centre_j - centre_i  [N, i, j]
    ci, si, cj, sj = c[:, :, None], s[:, :, None], c[:, None, :], s[:, None, :]
    hli, hwi, hlj, hwj = hl[:, :, None], hw[:, :, None], hl[:, None, :], hw[:, None, :]
    cd, sd = (ci * cj + si * sj).abs(), (ci * sj - si * cj).abs()
    m1 = (tx * ci + ty * si).abs() - (hli + (cd * hlj + sd * hwj))
    m2 = (ty * ci - tx * si).abs() - (hwi + (sd * hlj + cd * hwj))
    m3 = (tx * cj + ty * sj).abs() - (hlj + (cd * hli + sd * hwi))
    m4 = (ty * cj - tx * sj).abs() - (hwj + (sd * hli + cd * hwi))
    margin = torch.maximum(torch.maximum(m1, m2), torch.maximum(m3, m4))
    m = x.shape[1]
    upper = torch.triu(torch.ones((m, m), dtype=torch.bool, device=state.device), diagonal=1) & dynamic[:, None] & dynamic[None, :]
    margin = torch.where(upper[None], margin, torch.full_like(margin, float("inf")))
    flat = margin.reshape(margin.shape[0], -1)
    return (flat <= 0).any(dim=1), flat.abs().min(dim=1).values


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_dense_collision_flags_match_all_pairs_reference_at_scale(dtype):
    """8,192 envs x 320 bodies scattered at random (so that roughly half of the envs hold an overlapping pair): the done
    flag of one step with noop actions must equal an all-pairs separating-axis test in torch fp64 on the stepped state,
    for every env whose closest pair is not within the tolerance.  A pair lost by the fp32 broad phase would show here."""
    import torch
    n, cars, peds = 8192, 64, 256
    m = cars + peds
    comp = dense_scenario("external")
    env = make(comp, n, dtype, seed=4)
    gen = torch.Generator(device="cpu").manual_seed(17)
    init = torch.zeros((m, 4, n), dtype=torch.float64)
    init[:, 0] = torch.rand((m, n), generator=gen, dtype=torch.float64) * 6000.0 + 200.0
    init[:, 1] = (torch.rand((m, n), generator=gen, dtype=torch.float64) - 0.5) * 24000.0
    init[:, 3] = (torch.rand((m, n), generator=gen, dtype=torch.float64) - 0.5) * 2 * np.pi
    init[0, 0] = 100.0      # the ego: far from the finish line, on the road, heading along it
    init[0, 1] = 0.0
    init[0, 3] = 0.0
    env.reset(init_state=init.to(env.dtype))
    state, _, done, winner, tangent = env.step(torch.zeros((m, 2, n), dtype=env.dtype, device=env.device))
    types = comp.struct.types
    half_l = torch.tensor([types[comp.struct.bodies[b].type_id].length / 2 for b in range(m)], dtype=torch.float64, device=env.device)
    half_w = torch.tensor([types[comp.struct.bodies[b].type_id].width / 2 for b in range(m)], dtype=torch.float64, device=env.device)
    dynamic = torch.ones(m, dtype=torch.bool, device=env.device)
    want = torch.zeros(n, dtype=torch.bool, device=env.device)
    closest = torch.zeros(n, dtype=torch.float64, device=env.device)
    for lo in range(0, n, 256):
        want[lo:lo + 256], closest[lo:lo + 256] = all_pairs_reference(state[:, :, lo:lo + 256].double(), half_l, half_w, dynamic)
    tol = 1e-6 if dtype == "float64" else 0.2
    clear = closest > tol
    got = done.bool()
    # with velocity 0 pedestrians inside the ego's zones cannot end the episode first: zones are tested after collisions
    hits = want & clear
    assert hits.sum() > n // 8 and (~want & clear).sum() > n // 8, (int(hits.sum()), int((~want & clear).sum()))
    assert torch.equal(got[hits], want[hits])
    # envs without any overlapping pair may still end through the ego's zones / ego collisions: only a collision-free,
    # zone-free env must report not done -> compare on envs where no pedestrian is anywhere near the ego's lane ahead
    quiet = ~want & clear & (winner < 0)
    assert not got[quiet].any()


def test_maximum_body_count_matches_oracle():
    """CAV_MAX_BODIES = 512 bodies per env (128 cars + 384 pedestrians, 130,816 pairs per step), a ragged batch of 5 envs,
    on-device agents: engine vs oracle on every counter and on the final state."""
    from oracle.oracle import Oracle
    n, steps = 5, 120
    env = make(dense_scenario("device", num_cars=128, num_pedestrians=384, epsilon=0.003), n, "float64", seed=8)
    assert env.num_bodies == 512
    env.reset()
    oracle = Oracle(dense_scenario("device", num_cars=128, num_pedestrians=384, epsilon=0.003), n, seed=8, threads=8)
    oracle.reset()
    assert np.array_equal(env.state.cpu().numpy(), oracle.state)
    env.rollout(steps, auto_reset=True)
    oracle.rollout(steps, auto_reset=True)
    got, want = env.stats(), oracle.stats()
    if got["tangent"] == 0 and want["tangent"] == 0:
        for key in ("episodes", "interesting", "sum_t", "sum_t2", "sum_score", "sum_score2", "env_steps", "sum_t_interesting", "sum_t2_interesting"):
            assert got[key] == want[key], key
        assert state_err(np.moveaxis(env.state.cpu().numpy(), 1, -1), np.moveaxis(oracle.state, 1, -1)) < 1e-9
    assert want["episodes"] >= 2


def test_more_than_maximum_bodies_is_rejected():
    from cavgym_b200 import _native
    with pytest.raises((ValueError, _native.CavgymError)):
        make(dense_scenario("external", num_cars=130, num_pedestrians=384), 2, "float64")


def test_dense_step_host_equals_device_step():
    """cavgym_step_host on a 320-body scenario: pinned buffers (zero copy), pageable buffers (staged copies) and the device
    step give identical bits."""
    import torch
    n, steps = 6, 25
    comp = dense_scenario("external")
    m = comp.n_bodies
    actions = torch.tensor(random_actions(np.random.RandomState(2), steps, n, comp.is_car))
    envs = [make(dense_scenario("external"), n, "float64", seed=4) for _ in range(3)]
    def buffers(pin):
        shapes = {"actions": ((m, 2, n), torch.float64), "state": ((m, 4, n), torch.float64), "reward": ((m, n), torch.float64),
                  "done": ((n,), torch.uint8), "winner": ((n,), torch.int32), "tangent": ((n,), torch.uint8)}
        return {k: (torch.empty(s, dtype=d).pin_memory() if pin else torch.empty(s, dtype=d)) for k, (s, d) in shapes.items()}
    host = [buffers(True), buffers(False)]
    for env in envs:
        env.reset()
    for t in range(steps):
        for env, h in zip(envs[:2], host):
            h["actions"].copy_(actions[t])
            env.step_host(h["actions"], h["state"], h["reward"], h["done"], h["winner"], h["tangent"])
        out = envs[2].step(actions[t].to(envs[2].device))
        for key, dev in zip(("state", "reward", "done", "winner", "tangent"), out):
            assert torch.equal(host[0][key], dev.cpu()), (t, key)
            assert torch.equal(host[1][key], dev.cpu()), (t, key)
    assert envs[0].stats() == envs[1].stats() == envs[2].stats()


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("pedestrians", [5, 7])
def test_six_and_eight_body_scenarios_replay_and_step(pedestrians, dtype):
    """Pedestrians-v0 with 5 / 7 pedestrians (M = 6 / 8, the largest thread-per-env body counts; the TMA staging of the fp64
    replay kernel no longer fits shared memory there and the plain kernel takes over): a joint-action trace logged from the
    on-device agents, replayed through cavgym_replay and cavgym_step on both paths — bitwise equal — and against the oracle."""
    import torch
    from oracle.oracle import Oracle
    meta, _ = load_golden("pedestrians_rc_eps05_seed1")
    meta["config"]["scenario_config"]["num_pedestrians"] = pedestrians
    n, steps = 576, 120          # whole 16-env groups: the TMA kernels are eligible wherever their staging fits
    gen = make(compile_from_meta(meta, mode="device"), n, "float64", seed=6)
    gen.set_action_logging(True)
    gen.reset()
    init = gen.state.cpu().numpy().copy()
    actions = np.empty((steps, pedestrians + 1, 2, n))
    for t in range(steps):
        gen.step(None)
        actions[t] = gen.actions_taken.cpu().numpy()
    outs = []
    for dense in (False, True):
        env = make(compile_from_meta(meta), n, dtype)
        env.set_dense_path(dense)
        env.reset(init_state=init)
        fused = numpy_traj(env.replay(actions[:steps // 2]))
        act_t = torch.tensor(actions[steps // 2:], dtype=env.dtype, device=env.device)
        last = None
        for t in range(act_t.shape[0]):
            last = [v.cpu().numpy().copy() for v in env.step(act_t[t])]
        outs.append((fused, last, env.stats()))
    for key in ("state", "reward", "done", "winner", "tangent"):
        assert np.array_equal(outs[0][0][key], outs[1][0][key], equal_nan=True), key
    for a, b in zip(outs[0][1], outs[1][1]):
        assert np.array_equal(a, b, equal_nan=True)
    assert outs[0][2] == outs[1][2]
    if dtype == "float64":
        oracle = Oracle(compile_from_meta(meta), n, threads=8)
        oracle.reset(init_state=init)
        want = oracle.replay(actions[:steps // 2])
        check_against_oracle({k: v for k, v in outs[0][0].items()}, want, dtype)


# ------------------------------------------------------------------ the pair sweep at every tile shape, planted pairs
# kernels_dense.cuh pads M to Mp = (M + 31) & ~31 and sweeps pairs in passes of two 32-body tiles; these body counts give a
# ragged or full last tile, an odd or even tile count, and a final pass of one tile with tiles below it (65..96, 129..160)
SWEEP_M = (9, 31, 32, 33, 63, 64, 65, 96, 97, 128, 129, 160, 161, 320, 511, 512)
SPACING = 400.0     # lattice pitch: more than twice the sum of the largest half-diagonals (a car: 38.6 px) plus both lengths


def planted_pairs(m):
    """(i, j), i < j: every unordered pair up to 161 bodies; above, every within-tile offset 1..31 in every tile and every
    pair of tiles at three lane pairs (the lower tile against tile A and tile B of each pass)."""
    if m <= 161:
        i, j = np.triu_indices(m, 1)
        return np.stack([i, j], axis=1)
    tiles = (m + 31) // 32
    pairs = [(32 * t + (t * 5 + 3 * d) % (32 - d), 32 * t + (t * 5 + 3 * d) % (32 - d) + d) for t in range(tiles) for d in range(1, 32)]
    pairs += [(32 * a + la, 32 * b + lb) for a in range(tiles) for b in range(a + 1, tiles) for la, lb in ((0, 31), (31, 0), (13, 6))]
    return np.array([p for p in pairs if p[1] < m])


def planted_batch(comp, pairs, shuffled, x0, depth, rng):
    """Initial states [M, 4, N] of one env per pair plus 8 controls: the ego parked at (100, 0) heading along the road with
    v = 0 (no stopping zones), every other body still on a lattice of pitch SPACING from (x0, 3000) — in body order, or
    shuffled so that every tile's union box spans the lattice — at a random heading; then body j of the env's pair moved
    to overlap body i by `depth` px along i's axis, at i's heading (separating-axis margin -depth)."""
    m = comp.n_bodies
    types = comp.struct.types
    hl = np.array([types[comp.struct.bodies[b].type_id].length / 2 for b in range(m)])
    site = rng.permutation(m - 1) if shuffled else np.arange(m - 1)
    n = len(pairs) + 8
    state = np.zeros((m, 4, n))
    state[1:, 0] = (x0 + SPACING * (site % 40))[:, None]
    state[1:, 1] = (3000.0 + SPACING * (site // 40))[:, None]
    state[1:, 3] = rng.uniform(-np.pi, np.pi, m - 1)[:, None]
    state[0, 0] = 100.0
    e = np.arange(len(pairs))
    i, j = pairs[:, 0], pairs[:, 1]
    th = state[i, 3, e]
    reach = hl[i] + hl[j] - depth
    state[j, 0, e] = state[i, 0, e] + reach * np.cos(th)
    state[j, 1, e] = state[i, 1, e] + reach * np.sin(th)
    state[j, 3, e] = th
    return state


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("m", SWEEP_M)
def test_pair_sweep_finds_every_planted_pair(m, dtype):
    """Exactly one overlapping (or nearly touching) pair per env, every pair of bodies (or, from 320 bodies, every within-tile
    offset and every pair of tiles), the bodies in lattice order and shuffled, at depths -2 px, +-10 tau, and +-10 tau with
    the lattice translated to x = 2e4 px (one float32 ulp ~ 2e-3 px: an fp64 pair 1e-6 px deep must pass the float32 broad
    phase).  Every planted margin is more than 2 tau from 0, so `done` must be its exact decision and no env may be
    flagged; the 8 control envs of each batch, with no planted pair, must not end.  Noop actions, velocity 0."""
    import torch
    import exact_geometry as xg
    tau = {"float64": 1e-7, "float32": 5e-2}[dtype]
    cars = max(1, m // 5)
    comp = dense_scenario("external", num_cars=cars, num_pedestrians=m - cars)
    assert comp.n_bodies == m
    pairs = planted_pairs(m)
    rng = np.random.default_rng(m)
    batches, want = [], []
    for x0, depth in ((400.0, 2.0), (400.0, 10 * tau), (400.0, -10 * tau), (2e4, 10 * tau), (2e4, -10 * tau)):
        for shuffled in (False, True):
            batches.append(planted_batch(comp, pairs, shuffled, x0, depth, rng))
            want.append(np.concatenate([np.full(len(pairs), depth > 0), np.zeros(8, dtype=bool)]))
    init, want = np.concatenate(batches, axis=-1), np.concatenate(want)
    n = init.shape[-1]
    env = make(comp, n, dtype, seed=4)
    env.reset(init_state=init)
    state, _, done, _, tangent = env.step(torch.zeros((m, 2, n), dtype=env.dtype, device=env.device))
    done, tangent, state = done.cpu().numpy() != 0, tangent.cpu().numpy(), state.double().cpu().numpy()
    assert not tangent.any(), f"flagged without a margin within 2 tau: envs {np.flatnonzero(tangent)[:5]}"
    wrong = np.flatnonzero(done != want)
    if wrong.size:
        e = wrong[0] % (len(pairs) + 8)
        pytest.fail(f"{wrong.size} envs wrong, first {wrong[0]}: pair {tuple(pairs[e]) if e < len(pairs) else 'control'}, "
                    f"done {done[wrong[0]]}")
    # the construction against exact arithmetic on the stepped state, on a sample of planted envs of every batch
    types = comp.struct.types
    dims = [(types[comp.struct.bodies[b].type_id].length, types[comp.struct.bodies[b].type_id].width) for b in range(m)]
    per = len(pairs) + 8
    for b in range(len(batches)):
        for e in rng.choice(len(pairs), size=min(8, len(pairs)), replace=False):
            i, j = pairs[e]
            box = [xg.make_box(*dims[k], state[k, 3, b * per + e], state[k, 0, b * per + e], state[k, 1, b * per + e]) for k in (i, j)]
            margin = xg.sat_margin(*box)
            assert margin.cmp(0) == (-1 if want[b * per + e] else 1) and not margin.within(2 * tau), (b, i, j, float(margin))
    # the lattice: in a control env no two bodies come within reach of each other
    half_l = torch.tensor([d[0] / 2 for d in dims], dtype=torch.float64)
    half_w = torch.tensor([d[1] / 2 for d in dims], dtype=torch.float64)
    controls = [b * per + per - 1 for b in range(len(batches))]
    hit, closest = all_pairs_reference(torch.tensor(state[:, :, controls]), half_l, half_w, torch.ones(m, dtype=torch.bool))
    assert not hit.any() and float(closest.min()) > 100.0
