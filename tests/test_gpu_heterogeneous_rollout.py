"""cavgym_rollout of heterogeneous scenarios (crossroads, bus stop, pelican crossing) on the thread-per-env rollout kernel,
the default.  Its results — state, crossing-agent state, held actions, liveness, time steps, every episode counter and the
near-tangent count — must be bitwise those of the warp-per-env kernel (set_dense_path) on the same seeds, equal the same
global envs run as separate shards, and agree with the C oracle's restatement of environment.py:119-223 on the same Philox
streams."""
import numpy as np
import pytest

from helpers import agent_specs, bodies_and_constants, compile_from_meta, env_config_from, load_golden, state_err

pytestmark = pytest.mark.gpu

HETEROGENEOUS = ["crossroads_random_all_seed6", "crossroads_random_ego_seed7", "busstop_random_all_seed8", "busstop_noop_seed9",
                 "pelican_random_all_seed10", "pelican_random_ego_seed11"]


def make(comp, n, dtype, **kw):
    from cavgym_b200 import BatchedCAVEnv
    return BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=comp, **kw)


def snapshot(env):
    return (env.state.cpu().numpy(), env.agent_state.cpu().numpy(), env.actions_taken.cpu().numpy(), env.episode_liveness.cpu().numpy(),
            env.timestep.cpu().numpy(), env.done_latch.cpu().numpy(), env.stats())


def assert_same(a, b):
    for x, y in zip(a[:6], b[:6]):
        assert np.array_equal(x, y, equal_nan=True)
    assert a[6] == b[6]


def mixed_agents(meta):
    """The stock scenario with every kind of on-device agent a heterogeneous rollout takes: random cars (and crossing
    lights), a random-constrained and a proximity pedestrian.  (The reference's Config.setup cannot build this mix — quirk 10
    of SURVEY 8a — the engine's scenario tables can.)"""
    from cavgym_b200.scenario import AgentSpec, compile_scenario
    cfg = meta["config"]
    bodies, constants = bodies_and_constants(cfg)
    specs = agent_specs(cfg, bodies, "device")
    crossing = [AgentSpec("random-constrained", epsilon=0.02), AgentSpec("proximity", threshold=16.0 * 34)]
    k = 0
    for i, body in enumerate(bodies):
        if i > 0 and type(body).__name__ == "Pedestrian":
            specs[i] = crossing[k % 2]
            k += 1
    assert k > 0
    return compile_scenario(bodies, constants, env_config_from(cfg), specs)


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("name", HETEROGENEOUS)
def test_thread_per_env_rollout_is_bitwise_the_warp_per_env_rollout(name, dtype):
    meta, _ = load_golden(name)
    meta["config"]["tester_config"]["epsilon"] = 0.03
    n = 131                      # ragged: the last CTA has lanes without an env, the last warp a partial set of envs
    results = []
    for dense in (False, True):
        env = make(compile_from_meta(meta, mode="device"), n, dtype, seed=9, env_offset=3)
        env.set_dense_path(dense)
        env.set_action_logging(True)
        env.reset()
        env.rollout(450, auto_reset=True)
        env.rollout(1, auto_reset=True)
        env.rollout(649, auto_reset=True)
        results.append(snapshot(env))
    assert_same(results[0], results[1])
    if "noop" not in name:
        assert results[0][6]["episodes"] >= n // 2


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("name", ["crossroads_random_all_seed6", "pelican_random_all_seed10", "pelican_random_ego_seed11"])
def test_rollout_with_crossing_agents(name, dtype):
    meta, _ = load_golden(name)
    n = 200
    results = []
    for dense in (False, True):
        env = make(mixed_agents(meta), n, dtype, seed=21)
        env.set_dense_path(dense)
        env.set_action_logging(True)
        env.reset()
        for _ in range(4):
            env.rollout(300, auto_reset=True)
        results.append(snapshot(env))
    assert_same(results[0], results[1])
    assert np.isfinite(results[0][1]).any() or results[0][6]["episodes"] > 0   # some crossing was under way or episodes turned over


@pytest.mark.parametrize("name", ["busstop_random_all_seed8", "pelican_random_all_seed10", "crossroads_random_all_seed6"])
def test_rollout_matches_the_oracle(name):
    """Engine and oracle on their common Philox streams: every episode counter equal, final state within 1e-9."""
    from oracle.oracle import Oracle
    meta, _ = load_golden(name)
    meta["config"]["tester_config"]["epsilon"] = 0.03
    n, steps = 64, 700
    env = make(compile_from_meta(meta, mode="device"), n, "float64", seed=13)
    env.reset()
    env.rollout(steps, auto_reset=True)
    oracle = Oracle(compile_from_meta(meta, mode="device"), n, seed=13)
    oracle.reset()
    oracle.rollout(steps, auto_reset=True)
    got, want = env.stats(), oracle.stats()
    for key in ("episodes", "interesting", "sum_t", "sum_t2", "sum_score", "sum_score2", "env_steps", "body_steps"):
        assert got[key] == want[key], key
    assert state_err(np.moveaxis(env.state.cpu().numpy(), 1, -1), np.moveaxis(oracle.state, 1, -1)) < 1e-9


def test_split_batches_agree():
    """The same 96 global envs as one engine and as two shards (Philox is keyed by the global env id)."""
    meta, _ = load_golden("busstop_random_all_seed8")
    whole = make(compile_from_meta(meta, mode="device"), 96, "float64", seed=2)
    whole.reset(); whole.rollout(500, auto_reset=True)
    parts = []
    for offset, count in ((0, 40), (40, 56)):
        env = make(compile_from_meta(meta, mode="device"), count, "float64", seed=2, env_offset=offset)
        env.reset(); env.rollout(500, auto_reset=True)
        parts.append(env.state.cpu().numpy())
    assert np.array_equal(whole.state.cpu().numpy(), np.concatenate(parts, axis=-1))
