"""Every instantiation of the thread-per-env kernels: body count M = 1..8 x scenario family (homogeneous: the GENERIC = false
kernels; generic: GENERIC = true) x fp64 / fp32, on the cells of helpers.matrix_scenario.

The kernels change shape at compile time with M (TMA staging up to CAV_TMA_MAX_BODIES = 2 with a special case at M = 1,
the rolled transition, 256-thread CTAs and phase barriers of the generic rollout, election bookkeeping), so each cell is its
own code and is held here to
  * the C oracle: the first reset (bitwise in fp64), replayed random valid actions (fp64: state and rewards within 1e-9,
    events identical off flagged steps; fp32: the bars of helpers.check_against_oracle), and the on-device agents on the
    same Philox streams (observation, action and state within 1e-9 until an env's first flagged step, every counter equal
    when no step was flagged);
  * its own other paths, bitwise: fused replay with and without the TMA kernels and step() both ways; step() with device
    agents against rollout(auto_reset=True); the thread-per-env rollout against the warp-per-env one.
launch_count() shows the TMA step and replay kernels took whole tiles exactly where M <= 2.
"""
import numpy as np
import pytest
import torch

from helpers import (FAMILIES, MATRIX_M, check_against_oracle, expect_homogeneous, matrix_scenario, random_actions,
                     state_err)

pytestmark = pytest.mark.gpu

MAX_T = 60
T_REPLAY = 90             # replayed actions: every env times out inside the window, and planted pedestrians end some earlier
T_DEVICE = (50, 40)       # two rollout launches with on-device agents: episodes end and restart inside them
N_DEVICE = 203
CELLS = [pytest.param(m, family, id=f"{family}_m{m}") for family in FAMILIES for m in MATRIX_M]


def make(comp, n, dtype, **kw):
    from cavgym_b200 import BatchedCAVEnv
    return BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=comp, **kw)


def plant(init, comp, rng):
    """Initial states [M, 4, N] with, in about two envs of three, one pedestrian moved onto the road 40..400 px ahead of the
    ego, so that collisions and the ego's zones end episodes inside the window (spawned pedestrians alone rarely do)."""
    init = init.copy()
    n = init.shape[-1]
    peds = np.flatnonzero(~comp.is_car)
    if peds.size:
        envs = np.flatnonzero(rng.random(n) < 0.67)
        b = peds[rng.integers(0, peds.size, envs.size)]
        init[b, 0, envs] = init[0, 0, envs] + rng.uniform(40.0, 400.0, envs.size)
        init[b, 1, envs] = init[0, 1, envs] + rng.uniform(-60.0, 60.0, envs.size)
    return init


def host(out):
    return {k: v.cpu().numpy() for k, v in out.items() if v is not None}


# ------------------------------------------------------------------ replayed actions
@pytest.mark.parametrize("n", [128 * 5 + 52, 128 * 5 + 48])   # n % 16 != 0: whole TMA tiles + plain tail; == 0: ragged tile in-kernel
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("m, family", CELLS)
def test_replayed_actions_on_every_path_and_against_the_oracle(m, family, dtype, n):
    from oracle.oracle import Oracle
    comp = matrix_scenario(m, family, "external", max_timesteps=MAX_T)
    assert expect_homogeneous(comp, dtype) == (family == "homogeneous")
    oracle = Oracle(matrix_scenario(m, family, "external", max_timesteps=MAX_T), n, seed=9, threads=8)
    oracle.reset()
    # the first reset draws the same spawns
    first = make(comp, n, dtype, seed=9)
    first.reset()
    if dtype == "float64":
        assert np.array_equal(first.state.cpu().numpy(), oracle.state)
    else:
        assert state_err(np.moveaxis(first.state.cpu().numpy(), 1, -1), np.moveaxis(oracle.state, 1, -1)) < 1e-6
    rng = np.random.default_rng(100 * m + n)
    init = plant(oracle.state, comp, rng)
    actions = random_actions(rng, T_REPLAY, n, comp.is_car)
    oracle.reset(init_state=init)
    want = oracle.replay(actions)

    envs = [make(comp, n, dtype, seed=9), make(comp, n, dtype, seed=9)]
    envs[1].set_step_path(use_tma=False)
    fused, stepped, launches = [], [], []
    for env in envs:
        env.reset(init_state=init)
        before = env.launch_count()
        fused.append(host(env.replay(actions)))
        replayed = env.launch_count() - before
        # state / reward / winner only: no uint8 rows, so whole TMA tiles are eligible at n % 16 != 0 too
        env.reset(init_state=init)
        env.set_global_timestep(0)
        before = env.launch_count()
        partial = host(env.replay(actions, record=("state", "reward", "winner")))
        launches.append((replayed, env.launch_count() - before))
        for key in partial:
            assert np.array_equal(partial[key], fused[-1][key], equal_nan=True), key
        env.reset(init_state=init)
        env.set_global_timestep(0)
        acts = torch.tensor(actions, dtype=env.dtype, device=env.device)
        rows = {k: [] for k in ("state", "reward", "done", "winner", "tangent")}
        before = env.launch_count()
        for t in range(T_REPLAY):
            for k, v in zip(rows, env.step(acts[t])):
                rows[k].append(v.cpu().numpy().copy())
        launches[-1] += (env.launch_count() - before,)
        stepped.append({k: np.stack(v) for k, v in rows.items()})
    for key in ("state", "reward", "done", "winner", "tangent"):
        assert np.array_equal(fused[0][key], fused[1][key], equal_nan=True), ("replay", key)
        assert np.array_equal(stepped[0][key], fused[0][key], equal_nan=True), ("step, TMA", key)
        assert np.array_equal(stepped[1][key], fused[0][key], equal_nan=True), ("step, plain", key)
    for attr in ("episode_liveness", "timestep", "done_latch", "winner_latch"):
        assert torch.equal(getattr(envs[0], attr), getattr(envs[1], attr)), attr
    assert envs[0].stats() == envs[1].stats()
    # the TMA kernels took whole tiles (one more launch: tiles + plain tail) exactly where they exist; at n % 16 == 0 they
    # take every env, ragged tile included, in the one launch the plain kernel would make
    tma, plain = launches
    assert plain == (1, 1, T_REPLAY)
    if n % 16:
        assert tma == ((1, 2, 2 * T_REPLAY) if m <= 2 else plain), (tma, plain)
    else:
        assert tma == plain

    got = {k: (v.astype(np.float64) if v.dtype == np.float32 else v) for k, v in fused[0].items()}
    ended = check_against_oracle(got, want, dtype)
    assert ended > n // 10 if comp.is_car.sum() < m else ended == 0   # the ego alone, or with the car only, only times out
    assert envs[0].stats()["episodes"] >= n


# ------------------------------------------------------------------ on-device agents
def device_engine(m, family, dtype, dense=False):
    env = make(matrix_scenario(m, family, "device", max_timesteps=MAX_T), N_DEVICE, dtype, seed=5, env_offset=3)
    env.set_dense_path(dense)
    return env


def engine_bytes(env):
    return [env.state.cpu().numpy(), env.agent_state.cpu().numpy(), env.episode_liveness.cpu().numpy(),
            env.timestep.cpu().numpy(), env.done_latch.cpu().numpy(), env.winner_latch.cpu().numpy()]


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("m, family", CELLS)
def test_device_agents_step_rollout_and_warp_per_env_agree(m, family, dtype):
    """step() with action logging, resetting finished envs before each step, is rollout(auto_reset=True); the thread-per-env
    rollout is the warp-per-env one."""
    rollouts = []
    for dense in (False, True):
        env = device_engine(m, family, dtype, dense)
        env.reset()
        for window in T_DEVICE:
            env.rollout(window, auto_reset=True)
        rollouts.append((engine_bytes(env), env.stats()))
    steps = device_engine(m, family, dtype)
    steps.set_action_logging(True)
    steps.reset()
    for _ in range(sum(T_DEVICE)):
        steps.reset(mask=steps.done_latch.clone())
        steps.step(None)
    for got, name in ((rollouts[1], "warp-per-env rollout"), ((engine_bytes(steps), steps.stats()), "step()")):
        for a, b, what in zip(rollouts[0][0], got[0], ("state", "agent_state", "liveness", "timestep", "done", "winner")):
            assert np.array_equal(a, b, equal_nan=True), (name, what)
        assert rollouts[0][1] == got[1], name
    assert rollouts[0][1]["episodes"] >= N_DEVICE


@pytest.mark.parametrize("m, family", CELLS)
def test_device_agents_against_the_oracle_fp64(m, family):
    from oracle.oracle import Oracle
    env = device_engine(m, family, "float64")
    env.set_action_logging(True)
    env.reset()
    oracle = Oracle(matrix_scenario(m, family, "device", max_timesteps=MAX_T), N_DEVICE, seed=5, threads=8)
    oracle.set_shard(3)
    oracle.reset()
    assert np.array_equal(env.state.cpu().numpy(), oracle.state)
    live = np.ones(N_DEVICE, dtype=bool)   # envs not yet past a flagged step
    flagged = 0
    for t in range(sum(T_DEVICE)):
        env.reset(mask=env.done_latch.clone())
        assert state_err(np.moveaxis(oracle.state[:, :, live], -1, 0), np.moveaxis(env.state.cpu().numpy()[:, :, live], -1, 0)) <= 1e-9, t
        _, _, done, _, tangent = env.step(None)
        oracle.rollout(1, auto_reset=True)
        done, tangent, ts = done.cpu().numpy(), tangent.cpu().numpy(), env.timestep.cpu().numpy()
        kept = live & ~((done == 1) | (ts >= MAX_T))   # the oracle resets finished envs (and their held actions) after the step
        assert state_err(np.moveaxis(oracle.state[:, :, kept], -1, 0), np.moveaxis(env.state.cpu().numpy()[:, :, kept], -1, 0)) <= 1e-9, t
        assert np.max(np.abs(oracle.actions_taken[:, :, kept] - env.actions_taken.cpu().numpy()[:, :, kept]), initial=0) <= 1e-9, t
        live &= tangent == 0
        flagged += int(tangent.sum())
    got, want = env.stats(), oracle.stats()
    if got["tangent"] == 0 and want["tangent"] == 0:
        for key in ("episodes", "interesting", "sum_t", "sum_t2", "sum_score", "sum_score2", "env_steps", "sum_t_interesting",
                    "sum_t2_interesting"):
            assert got[key] == want[key], key
    assert live.sum() > N_DEVICE // 2
    assert want["episodes"] >= N_DEVICE
    print(f"{family} M={m}: {flagged} flagged env-steps of {N_DEVICE * sum(T_DEVICE)}")
