"""The parking rollout (BatchedCAVEnv.rollout_until, cavgym_rollout_until) and the splitting estimator on the GPU.

The contract: at level +inf and salt 0 the launch is rollout(auto_reset=False), byte for byte; the score is the running
maximum of the danger of the post-step states (px by which a pedestrian overlaps the ego's reaction zone), recomputed here
in torch fp64 from a recorded rollout, and +inf exactly where a tester won; a parked env holds the state of its first
crossing step and a repeated launch changes nothing; a non-zero salt draws fresh, reproducible streams; every refusal comes
before any launch; and the estimator agrees with crude Monte Carlo where both can measure.
"""
import copy
import ctypes
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from helpers import compile_from_meta, has_pedestrian, load_golden, matrix_scenario

pytestmark = pytest.mark.gpu

MAX_T = 40
N = 203   # ragged: not a multiple of any block size
SNAP = ("state", "action", "agent", "cs", "liveness", "t_ep", "episode", "winner", "active", "done", "err")
CASES = {
    "homogeneous_2_bodies": "pedestrians_rc_eps05_seed1",
    "homogeneous_rolled_4_bodies": "pedestrians3_rc_seed2",
    "crossroads": "crossroads_random_all_seed6",
    "pelican_crossing": "pelican_random_all_seed10",
    "election": "learn_election3_seed22",
}
# the cells of helpers.matrix_scenario that the recorded-rollout tests add, except those without a pedestrian (refused below)
MATRIX_CELLS = [(1, "homogeneous"), (3, "homogeneous"), (5, "homogeneous"), (6, "homogeneous"), (7, "homogeneous"),
                (8, "homogeneous"), (1, "generic"), (2, "generic"), (4, "generic"), (6, "generic"), (7, "generic"), (8, "generic")]
CASES.update({f"matrix_{family}_{m}_bodies": ("matrix", m, family) for m, family in MATRIX_CELLS if has_pedestrian(m, family)})
LIVE, PARKED, FINISHED = 0, 1, 2


def compiled(golden, mode="device", **config):
    if isinstance(golden, tuple):
        assert not config
        return matrix_scenario(golden[1], golden[2], mode, max_timesteps=MAX_T)
    meta = copy.deepcopy(load_golden(golden)[0])
    meta["config"]["max_timesteps"] = MAX_T
    meta["config"].update(config)
    return compile_from_meta(meta, mode=mode)


def engine(case, dtype="float64", n=N, seed=5, mode="device", **config):
    from cavgym_b200 import BatchedCAVEnv
    return BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=compiled(CASES.get(case, case), mode, **config), seed=seed)


def snapshot_bytes(env):
    snap = env.save_envs()
    return torch.cat([snap[name].contiguous().view(torch.uint8).reshape(-1) for name in SNAP]).cpu()


def fresh_score(env):
    return torch.full((env.num_envs,), -math.inf, dtype=env.dtype, device=env.device)


def t_global(env):
    return int(env._engine_state().t_global)


def danger_rows(env, state):
    """Danger of every recorded post-step state [T, M, 4, N], in fp64: -min over the pedestrians of the separating-axis
    margin of the body's box against the ego's reaction-zone rectangle."""
    sc = env.compiled.struct
    state = np.asarray(state, dtype=np.float64)
    ego = sc.types[sc.bodies[0].type_id]
    hl, hw = ego.length * 0.5, ego.width * 0.5
    x, y, v, th = (state[:, 0, c] for c in range(4))
    c, s = np.cos(th), np.sin(th)
    bd = (v * v) * (1.0 / (2.0 * -ego.min_throttle))
    hr = ((bd + v * 0.675) - bd) * 0.5
    centre, half = hl + bd + hr, hr
    out = np.full(x.shape, -np.inf)
    for b in range(1, sc.n_bodies):
        if not sc.bodies[b].flags & 1:   # CAV_FLAG_PEDESTRIAN
            continue
        k = sc.types[sc.bodies[b].type_id]
        hlb, hwb = k.length * 0.5, k.width * 0.5
        px, py, tb = state[:, b, 0], state[:, b, 1], state[:, b, 3]
        cb, sb = np.cos(tb), np.sin(tb)
        tx, ty = px - x, py - y
        cd, sd = c * cb + s * sb, c * sb - s * cb
        acd, asd = np.abs(cd), np.abs(sd)
        u, w = tx * c + ty * s, ty * c - tx * s
        tp, tq = tx * cb + ty * sb, ty * cb - tx * sb
        exb, eyb = acd * hlb + asd * hwb, asd * hlb + acd * hwb
        margin = np.maximum(np.maximum(np.abs(w) - (hw + eyb), np.abs(u - centre) - (half + exb)),
                            np.maximum(np.abs(tp - centre * cd) - ((hlb + asd * hw) + acd * half),
                                       np.abs(tq + centre * sd) - ((hwb + acd * hw) + asd * half)))
        out = np.maximum(out, -margin)
    return out


def recorded(case, dtype, steps, seed=5):
    env = engine(case, dtype, seed=seed)
    rec = {k: v.cpu().numpy() for k, v in env.rollout(steps, auto_reset=False, record=("state", "done", "winner", "timestep")).items()}
    return env, rec


def expected_scores(env, rec):
    """(running max of the danger over each env's scoring rows [T, N], tester won by row t [T, N]).  A scoring row is a step
    taken that does not end the episode without a tester win."""
    ts, done, winner = rec["timestep"], rec["done"], rec["winner"]
    stepped = ts > 0
    won = stepped & (winner > 0)
    ends = stepped & ((done == 1) | (ts >= MAX_T))
    scoring = stepped & ~ends
    running = np.maximum.accumulate(np.where(scoring, danger_rows(env, rec["state"]), -np.inf), axis=0)
    return running, np.logical_or.accumulate(won, axis=0)


# ------------------------------------------------------------------ level +inf, salt 0 is rollout(auto_reset=False)
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_at_level_inf_it_is_the_plain_rollout_bitwise(case, dtype):
    until, plain = engine(case, dtype), engine(case, dtype)
    for env in (until, plain):
        env.set_episode_log(1 << 12)
    score = fresh_score(until)
    for window in (17, 30):   # episodes of MAX_T = 40 steps end in the second window
        status = until.rollout_until(window, math.inf, score)
        plain.rollout(window, auto_reset=False)
    assert torch.equal(snapshot_bytes(until), snapshot_bytes(plain))
    assert until.stats() == plain.stats()
    rows_until, dropped_until = until.drain_episodes()
    rows_plain, dropped_plain = plain.drain_episodes()
    assert dropped_until == dropped_plain == 0 and len(rows_plain) == N
    assert np.array_equal(np.sort(rows_until, order=["env", "episode"]), np.sort(rows_plain, order=["env", "episode"]))
    assert t_global(until) == t_global(plain) == 47
    done, winner, st = (t.cpu().numpy() for t in (until.done_latch, until.winner_latch, status))
    assert (done != 0).all()
    assert np.array_equal(st, np.where(winner > 0, PARKED, FINISHED))
    assert np.array_equal(np.isposinf(score.cpu().numpy()), winner > 0)


# ------------------------------------------------------------------ the score is the running max of the danger
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_score_is_the_running_max_of_the_recomputed_danger(case, dtype):
    steps = MAX_T + 2
    twin, rec = recorded(case, dtype, steps)
    env = engine(case, dtype)
    score = fresh_score(env)
    env.rollout_until(steps, math.inf, score)
    running, won = expected_scores(twin, rec)
    got = score.double().cpu().numpy()
    assert np.array_equal(np.isposinf(got), won[-1])
    finite = ~won[-1]
    tol = 1e-9 if dtype == "float64" else 5e-3   # fp32: a few float ulps at the 1,000 px scale of the scene
    want = running[-1][finite]
    assert np.array_equal(np.isneginf(got[finite]), np.isneginf(want))
    both = np.isfinite(want)
    assert np.max(np.abs(got[finite][both] - want[both]), initial=0) <= tol


# ------------------------------------------------------------------ parking
@pytest.mark.parametrize("case", ["homogeneous_2_bodies", "crossroads", "election"])
def test_parked_envs_hold_their_first_crossing_state(case):
    steps = MAX_T + 2
    twin, rec = recorded(case, "float64", steps)
    running, won = expected_scores(twin, rec)
    finals = running[-1][np.isfinite(running[-1])]
    levels = [float(np.quantile(finals, q)) for q in (0.3, 0.6, 0.9)] + [math.inf]
    env = engine(case, "float64")
    score = fresh_score(env)
    parked_seen = 0
    for level in levels:
        for chunk in (5, 11, MAX_T):   # ragged launches: some envs stay live between them
            status = env.rollout_until(chunk, level, score).cpu().numpy()
            st, sc = status, score.cpu().numpy()
            k = env.timestep.cpu().numpy().astype(np.int64)        # each env's own steps (no reset since the start)
            done, winner = env.done_latch.cpu().numpy(), env.winner_latch.cpu().numpy()
            state = env.state.cpu().numpy()
            stepped = k > 0
            rows = rec["state"][np.maximum(k - 1, 0), :, :, np.arange(N)]   # [N, M, 4]
            assert np.array_equal(np.moveaxis(state, -1, 0)[stepped], rows[stepped])
            # status against the latches
            assert np.array_equal(st == FINISHED, (done != 0) & (winner <= 0))
            assert np.array_equal(st == PARKED, ((done != 0) & (winner > 0)) | ((done == 0) & (sc >= level)))
            assert np.array_equal(st == LIVE, (done == 0) & (sc < level))
            # a parked env (not a tester win) stopped at the first recorded row whose running max reaches the level
            crossed = (st == PARKED) & (done == 0)
            clear = np.all(np.abs(running - level) > 1e-6, axis=0)
            first = np.argmax(running >= level, axis=0)
            check = crossed & clear & stepped
            assert np.array_equal(k[check] - 1, first[check])
            parked_seen += int(check.sum())
            # a repeated launch at the same level changes nothing
            before, score_before = snapshot_bytes(env), score.clone()
            if (st == LIVE).any():
                continue
            again = env.rollout_until(7, level, score).cpu().numpy()
            assert torch.equal(snapshot_bytes(env), before) and torch.equal(score, score_before)
            assert np.array_equal(again, st)
    assert parked_seen > N // 4


# ------------------------------------------------------------------ salt
def test_salt_reproduces_and_changes_random_trajectories():
    a, b, c = (engine("homogeneous_2_bodies") for _ in range(3))
    scores = [fresh_score(e) for e in (a, b, c)]
    for env, score, salt in zip((a, b, c), scores, (0xC0FFEE, 0xC0FFEE, 0)):
        env.rollout_until(25, math.inf, score, salt=salt)
    assert torch.equal(snapshot_bytes(a), snapshot_bytes(b)) and torch.equal(scores[0], scores[1])
    moved = (a.state != c.state).any(dim=0).any(dim=0)
    assert moved.float().mean().item() > 0.5   # random-constrained testers draw every step
    d = engine("homogeneous_2_bodies")
    d.rollout_until(25, math.inf, fresh_score(d), salt=1)
    assert not torch.equal(snapshot_bytes(a), snapshot_bytes(d))
    assert int(a._engine_state().seed) == int(c._engine_state().seed) == 5


def dense320():
    from cavgym_b200 import BatchedCAVEnv
    from cavgym_b200.examples.environments import dense_traffic
    from cavgym_b200.library.bodies import Pedestrian
    from cavgym_b200.scenario import AgentSpec, compile_scenario
    road_map, constants = dense_traffic.make_world()
    bodies = dense_traffic.make_bodies(np_random=np.random.RandomState(0), road_map=road_map)
    cfg = SimpleNamespace(terminate_collisions="all", terminate_ego_zones=True, terminate_ego_offroad=False, max_timesteps=MAX_T,
                          reward_win=6000.0, reward_draw=2000.0, cost_step=4.0)
    specs = [AgentSpec("random-constrained", epsilon=0.01) if isinstance(b, Pedestrian) else AgentSpec("noop") for b in bodies]
    return BatchedCAVEnv(None, None, None, num_envs=8, compiled=compile_scenario(bodies, constants, cfg, specs))


def test_refusals_come_before_any_launch():
    EINVAL, ESTATE = -22, -1
    forced = engine("homogeneous_2_bodies")
    forced.set_dense_path(True)
    cases = [(engine("homogeneous_2_bodies"), {}, EINVAL, "score"), (engine("homogeneous_2_bodies"), {}, EINVAL, "status"),
             (engine("homogeneous_2_bodies"), {"n_steps": -1}, EINVAL, None),
             (engine("homogeneous_2_bodies"), {"level": math.nan}, EINVAL, None),
             (engine("homogeneous_2_bodies", terminate_ego_zones=False), {}, EINVAL, None),
             (engine("busstop_random_all_seed8"), {}, EINVAL, None),   # no Pedestrian body
             *[(engine(("matrix", m, family)), {}, EINVAL, None) for m, family in MATRIX_CELLS if not has_pedestrian(m, family)],
             (engine("homogeneous_2_bodies", mode="external"), {}, ESTATE, None),
             (forced, {}, ESTATE, None), (dense320(), {}, ESTATE, None)]
    for env, args, code, null in cases:
        n = env.num_envs
        score = fresh_score(env)
        status = torch.zeros(n, dtype=torch.uint8, device=env.device)
        launches, t0 = env.launch_count(), t_global(env)
        call = dict({"n_steps": 5, "level": 1.0}, **args)
        rc = env._lib.cavgym_rollout_until(env._handle, call["n_steps"], call["level"], 0, None if null == "score" else score.data_ptr(),
                                           None if null == "status" else status.data_ptr(), env._stream())
        assert rc == code, (env.compiled.body_classes, args, null, env._lib.cavgym_last_error())
        assert env.launch_count() == launches and t_global(env) == t0
        assert torch.equal(score, fresh_score(env)) and not status.any()
    env = engine("homogeneous_2_bodies")
    with pytest.raises(ValueError, match="score"):
        env.rollout_until(5, 1.0, torch.zeros(N, dtype=torch.float32, device=env.device))
    launches = env.launch_count()
    status = torch.full((N,), 7, dtype=torch.uint8, device=env.device)
    assert env.rollout_until(0, 1.0, fresh_score(env), status=status) is status and (status == 7).all()
    assert env.launch_count() == launches


# ------------------------------------------------------------------ the estimator
# RandomAgent testers that rarely act: measured on a B200 at 4.2 M episodes each, epsilon 0.002 gives a win rate of 1.4e-2
# and the pedestrian's path-maximum danger has quantiles -62 / -21 / -6.9 px at 0.5 / 0.9 / 0.99.  Smaller epsilons are rarer.
MODERATE, MODERATE_LEVELS = {"option": "random", "epsilon": 0.0003}, (-30.0, -10.0)
RARE, RARE_LEVELS = {"option": "random", "epsilon": 0.00001}, ((-30.0, -10.0), (-45.0, -25.0, -12.0, -4.0))
def stock(tester, seed, n):
    """The stock pedestrians scenario (one pedestrian, noop ego, max_timesteps 1000) with the given tester."""
    from cavgym_b200 import BatchedCAVEnv
    meta = copy.deepcopy(load_golden("pedestrians_rc_seed0")[0])
    meta["config"]["tester_config"] = dict(tester)
    meta["config"]["ego_config"] = {"option": "noop"}
    return BatchedCAVEnv(None, None, None, num_envs=n, compiled=compile_from_meta(meta, mode="device"), seed=seed)


def crude_monte_carlo(tester, seed, n=1 << 20, episodes=4_000_000):
    """interesting / episodes over whole episodes: each round runs every env through exactly one episode from a reset, so
    every episode is counted once and none is cut short (DESIGN §3.3)."""
    env = stock(tester, seed, n)
    for _ in range(-(-episodes // n)):
        env.reset()
        env.rollout(env.max_timesteps, auto_reset=False)
    stats = env.stats()
    assert stats["episodes"] >= episodes
    env.close()
    p = stats["interesting"] / stats["episodes"]
    return p, math.sqrt(p * (1 - p) / stats["episodes"])


def split(tester, seed, levels, n=1 << 18, repetitions=16):
    from cavgym_b200 import splitting
    env = stock(tester, seed, n)
    result = splitting.estimate(env, levels, repetitions, seed=seed)
    env.close()
    est = np.array(result.estimates)
    assert result.env_steps > 0 and result.device_seconds > 0
    return est.mean(), est.std(ddof=1) / math.sqrt(len(est)), result


def test_splitting_agrees_with_crude_monte_carlo():
    p_crude, se_crude = crude_monte_carlo(MODERATE, seed=21)
    assert 1e-3 <= p_crude <= 1e-2
    p_split, se_split, result = split(MODERATE, 22, MODERATE_LEVELS)
    assert all(0 < f < 1 for f in np.mean([r for r in result.fractions if len(r) == len(result.levels)], axis=0))
    assert abs(p_split - p_crude) <= 4 * math.hypot(se_crude, se_split), (p_split, se_split, p_crude, se_crude)


def test_two_level_schedules_agree_on_a_rarer_configuration():
    p_a, se_a, _ = split(RARE, 31, RARE_LEVELS[0])
    p_b, se_b, _ = split(RARE, 32, RARE_LEVELS[1])
    assert p_a > 0 and p_b > 0
    assert abs(p_a - p_b) <= 4 * math.hypot(se_a, se_b), (p_a, se_a, p_b, se_b)
