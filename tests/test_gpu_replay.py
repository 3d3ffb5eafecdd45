"""CUDA engine vs the reference traces and vs the CPU oracle on replayed joint actions (through the C-ABI).

Bar (north star): body state within 1e-9 relative in fp64 mode and 1e-4 in fp32 mode; done-step, winner and
liveness identical except on steps the engine flags as near-tangent.

"Relative" is |dp| / max(1 px, |p|) for a position, |dv| / max(1, |v|), and the angle difference modulo 2 pi over
max(1, |theta|) (helpers.state_err) — the STRICT per-step definition.  Measured on every fixture
(scripts/parity_report.py -> profiles/r2_parity_report.txt):

  fp64   strict 1.1e-13 worst, rewards 1.3e-11, no event or liveness difference at all, <= 0.18 % of steps flagged
  fp32   strict 3.0e-4 worst (a body whose coordinates were ~1,000 px and which later passes near the origin keeps the
         absolute error of the large coordinates: 3e-4 px against |p| ~ 1 px), 2.8e-5 when the error is taken relative to
         the largest |p| the body has reached so far (helpers.state_err_trajectory); rewards 2.7e-4; <= 4.2 % of steps
         flagged (tau = 0.05 px); every event difference is on a flagged step.

So fp32 mode meets 1e-4 on the trajectory scale and 5e-4 on the strict per-step scale; both are asserted below, next to the
flagged fractions (measured value + margin).  The comparison of an episode continues through flagged steps as long as the
events agree and ends at the first event difference (after it the two runs are different episodes).
"""
import numpy as np
import pytest

from helpers import (FAMILIES, GOLDEN_CASES, LEARN_CASES, MATRIX_M, compile_from_meta, load_golden, matrix_scenario, random_actions,
                     rel_err, soa, state_err, state_err_trajectory)

pytestmark = pytest.mark.gpu

REL = {"float64": 1e-9, "float32": 1e-4}
STRICT = {"float64": 1e-9, "float32": 5e-4}       # per-step |dp| / max(1, |p|): measured 1.1e-13 / 3.0e-4
REWARD = {"float64": 1e-9, "float32": 5e-4}       # relative to max(1, |r|): measured 1.3e-11 / 2.7e-4
FLAGGED = {"float64": 0.005, "float32": 0.06}     # fraction of steps flagged near-tangent: measured 0.0018 / 0.042


def make_env(meta, n, dtype, mode="external", **kw):
    from cavgym_b200 import BatchedCAVEnv
    comp = compile_from_meta(meta, mode=mode)
    return BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=comp, **kw)


def check_episode(traj, ep, col, dtype, liveness=None):
    """Compare one env column of a recorded trajectory with a golden episode; returns #flagged steps."""
    t_len = ep["actions"].shape[0]
    state = traj["state"][:t_len, :, :, col]
    reward = traj["reward"][:t_len, :, col]
    done = traj["done"][:t_len, col]
    winner = traj["winner"][:t_len, col]
    tangent = traj["tangent"][:t_len, col].astype(bool)
    mismatch = (done != ep["done"]) | (winner != ep["winner"])
    assert not np.any(mismatch & ~tangent), f"unflagged event mismatch at steps {np.nonzero(mismatch & ~tangent)[0][:5]}"
    if dtype == "float64":
        assert not mismatch.any(), "fp64: no fixture has an event difference, flagged or not"
    if np.any(mismatch):  # a flagged near-tangent divergence: the two runs are different episodes from here on
        t_len = int(np.nonzero(mismatch)[0][0])
    assert state_err(state[:t_len], ep["state"][:t_len]) < STRICT[dtype]
    assert state_err_trajectory(state[:t_len], ep["state"][:t_len]) < REL[dtype]
    assert rel_err(reward[:t_len], ep["reward"][:t_len]) < REWARD[dtype]
    if liveness is not None and not np.any(mismatch) and dtype == "float64":
        assert np.array_equal(liveness, ep["liveness"][-1])
    return int(tangent.sum())


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_step_by_step_matches_reference_fp64(name):
    """cavgym_step once per timestep, one env per golden episode (ragged lengths, zero-padded actions)."""
    import torch
    meta, episodes = load_golden(name)
    n, m = len(episodes), meta["n_bodies"]
    t_max = max(ep["actions"].shape[0] for ep in episodes)
    env = make_env(meta, n, "float64")
    init = np.stack([ep["init_state"] for ep in episodes])           # [N, M, 4]
    env.reset(init_state=soa(init))
    actions = np.zeros((t_max, m, 2, n))
    for e, ep in enumerate(episodes):
        actions[:ep["actions"].shape[0], :, :, e] = ep["actions"]
    # CAVEnv.current_timestep is per env object in the reference; replay each episode's own counter via the
    # engine-wide counter only when all episodes share it, else check the time-out reward separately below.
    starts = {int(ep["t_global_start"]) for ep in episodes}
    traj = {k: [] for k in ("state", "reward", "done", "winner", "tangent")}
    single_start = len(starts) == 1
    env.set_global_timestep(starts.pop() if single_start else -10 ** 9)
    actions_t = torch.tensor(actions, device=env.device)
    for t in range(t_max):
        state, reward, done, winner, tangent = env.step(actions_t[t])
        for k, v in zip(traj, (state, reward, done, winner, tangent)):
            traj[k].append(v.cpu().numpy().copy())
    traj = {k: np.stack(v) for k, v in traj.items()}
    live = env.episode_liveness.cpu().numpy()
    for e, ep in enumerate(episodes):
        want = dict(ep)
        if not single_start:  # remove the one-off time-out reward the reference adds at global step max_timesteps-1
            t_hit = meta["config"]["max_timesteps"] - 1 - int(ep["t_global_start"])
            if 0 <= t_hit < ep["reward"].shape[0] and not ep["done"][t_hit]:
                want["reward"] = ep["reward"].copy()
                want["reward"][t_hit] -= meta["config"]["reward_draw"]
        check_episode(traj, want, e, "float64", live[:, e])
    # frozen after the episode ended: reward 0, state unchanged
    for e, ep in enumerate(episodes):
        t_len = ep["actions"].shape[0]
        if t_len < t_max and ep["done"][-1]:
            assert np.all(traj["reward"][t_len:, :, e] == 0.0)
            assert np.array_equal(traj["state"][t_len, :, :, e], traj["state"][t_len - 1, :, :, e])


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("name", GOLDEN_CASES + LEARN_CASES)
def test_fused_replay_matches_reference(name, dtype):
    """cavgym_replay (T steps in one launch) per golden episode with the reference's own time-out counter."""
    meta, episodes = load_golden(name)
    env = make_env(meta, 1, dtype)
    flagged = 0
    for ep in episodes:
        env.reset(init_state=soa(ep["init_state"][None]))
        env.set_global_timestep(int(ep["t_global_start"]))
        out = env.replay(ep["actions"][..., None])
        traj = {k: v.double().cpu().numpy() if v.dtype.is_floating_point else v.cpu().numpy() for k, v in out.items()}
        flagged += check_episode(traj, ep, 0, dtype, env.episode_liveness.cpu().numpy()[:, 0])
    assert flagged <= sum(ep["actions"].shape[0] for ep in episodes) * FLAGGED[dtype]


def test_batched_replay_matches_oracle_65536_envs():
    """BASELINE config C2 shape: 65,536 envs, env e replays golden episode e mod K; engine vs CPU oracle over the
    whole batch (state 1e-9, events exact off flagged steps)."""
    from oracle.oracle import Oracle
    meta, episodes = load_golden("pedestrians_rc_seed0")
    n, m, t_len = 65536, meta["n_bodies"], 256
    k = len(episodes)
    init = np.stack([episodes[e % k]["init_state"] for e in range(k)])
    init = soa(init[np.arange(n) % k])
    actions = np.zeros((t_len, m, 2, n))
    for j, ep in enumerate(episodes):
        a = ep["actions"][:t_len]
        actions[:a.shape[0], :, :, j::k] = a[..., None]
    env = make_env(meta, n, "float64")
    env.reset(init_state=init)
    out = env.replay(actions, record=("state", "done", "winner", "tangent"))
    oracle = Oracle(compile_from_meta(meta), n, threads=8)
    oracle.reset(init_state=init)
    want_state, _, want_done, want_winner, _ = oracle.replay(actions)
    got_state = out["state"].cpu().numpy()
    assert state_err(np.moveaxis(got_state, 2, -1), np.moveaxis(want_state, 2, -1)) < 1e-9
    tangent = out["tangent"].cpu().numpy().astype(bool)
    mismatch = (out["done"].cpu().numpy() != want_done) | (out["winner"].cpu().numpy() != want_winner)
    assert not np.any(mismatch & ~tangent)
    assert np.array_equal(env.episode_liveness.cpu().numpy(), oracle.liveness)


def test_invalid_action_sets_error_flag_and_leaves_state():
    meta, episodes = load_golden("pedestrians_rc_seed0")
    env = make_env(meta, 4, "float64")
    env.reset(init_state=soa(np.stack([episodes[0]["init_state"]] * 4)))
    before = env.state.clone()
    actions = np.zeros((2, 2, 4))
    actions[0, 0, 1] = 1e6          # throttle out of Box bounds (environment.py:120)
    actions[1, 1, 3] = float("nan")
    state, reward, done, winner, _ = env.step(actions)
    err = env.error.cpu().numpy()
    assert err.tolist() == [0, 1, 0, 1]
    assert np.array_equal(state[:, :, 1].cpu().numpy(), before[:, :, 1].cpu().numpy())
    assert not np.array_equal(state[:, :, 0].cpu().numpy(), before[:, :, 0].cpu().numpy())
    assert env.stats()["errors"] == 2


def test_missing_actions_is_an_error():
    from cavgym_b200._native import CavgymError
    meta, _ = load_golden("pedestrians_rc_seed0")
    env = make_env(meta, 2, "float64")
    with pytest.raises(CavgymError):
        env.step(None)


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("n", [128 * 5 + 52, 128 * 5 + 48])   # n % 16 != 0: whole tiles + plain tail; n % 16 == 0: ragged tile in-kernel
@pytest.mark.parametrize("name", ["pedestrians_rc_seed0", "pedestrians3_rc_seed2", "crossroads_random_all_seed6", "pelican_random_all_seed10"])
def test_tma_step_kernel_is_bitwise_equal_to_plain_kernel(name, dtype, n):
    """cavgym_step on replayed actions runs the persistent TMA-staged kernel over whole 128-env tiles and the plain
    thread-per-env kernel over the ragged tail; both must produce the same bits as the plain kernel alone, every step,
    for every output (state, reward, done, winner, tangent, liveness, timestep)."""
    import torch
    meta, episodes = load_golden(name)
    m, k = meta["n_bodies"], len(episodes)
    t_max = min(400, max(ep["actions"].shape[0] for ep in episodes))
    init = soa(np.stack([episodes[e % k]["init_state"] for e in range(n)]))
    actions = np.zeros((t_max, m, 2, n))
    for j, ep in enumerate(episodes):
        a = ep["actions"][:t_max]
        actions[:a.shape[0], :, :, j::k] = a[..., None]
    envs = [make_env(meta, n, dtype), make_env(meta, n, dtype)]
    envs[1].set_step_path(use_tma=False)
    acts = torch.tensor(actions, dtype=envs[0].dtype, device=envs[0].device)
    for env in envs:
        env.reset(init_state=init)
    for t in range(t_max):
        outs = [env.step(acts[t]) for env in envs]
        if t % 7 == 0 or t == t_max - 1:
            for a, b in zip(*outs):
                assert torch.equal(a, b), f"step {t}"
    for attr in ("episode_liveness", "timestep", "done_latch", "winner_latch"):
        assert torch.equal(getattr(envs[0], attr), getattr(envs[1], attr)), attr
    assert envs[0].stats() == envs[1].stats()
    if n % 16 and m <= 2:   # the TMA-staged kernels serve scenarios of one or two bodies (CAV_TMA_MAX_BODIES)
        assert envs[0].launch_count() > envs[1].launch_count()  # two launches per step (tiles + tail) vs one
    else:
        assert envs[0].launch_count() == envs[1].launch_count()


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("n", [160 * 2 + 84, 160 * 2 + 96])   # n % 16 != 0 / == 0 (ragged last tile handled in-kernel)
@pytest.mark.parametrize("name", ["pedestrians_rc_seed0", "busstop_random_all_seed8"])
def test_tma_replay_kernel_is_bitwise_equal_to_plain_kernel(name, dtype, n):
    """cavgym_replay: the time-pipelined TMA kernel (whole tiles) + plain kernel (tail) against the plain kernel alone,
    in chunks of 1, 2, 3, 7 and 150 steps (fewer steps than pipeline stages included), with and without trajectories."""
    import torch
    meta, episodes = load_golden(name)
    m, k = meta["n_bodies"], len(episodes)
    t_max = min(320, max(ep["actions"].shape[0] for ep in episodes))
    init = soa(np.stack([episodes[e % k]["init_state"] for e in range(n)]))
    actions = np.zeros((t_max, m, 2, n))
    for j, ep in enumerate(episodes):
        a = ep["actions"][:t_max]
        actions[:a.shape[0], :, :, j::k] = a[..., None]
    envs = [make_env(meta, n, dtype), make_env(meta, n, dtype)]
    envs[1].set_step_path(use_tma=False)
    acts = torch.tensor(actions, dtype=envs[0].dtype, device=envs[0].device)
    for env in envs:
        env.reset(init_state=init)
    t = 0
    for chunk, record in ((1, ("state", "done")), (2, ()), (3, ("reward", "winner", "tangent")), (7, ("state",)),
                          (150, ("state", "reward", "done", "winner", "tangent")), (10 ** 6, ("state", "reward", "done"))):
        take = min(chunk, t_max - t)
        outs = [env.replay(acts[t:t + take], record=record) for env in envs]
        for key in record:
            assert torch.equal(outs[0][key], outs[1][key]), (chunk, key)
        assert torch.equal(envs[0].state, envs[1].state), chunk
        t += take
    for attr in ("episode_liveness", "timestep", "done_latch", "winner_latch"):
        assert torch.equal(getattr(envs[0], attr), getattr(envs[1], attr)), attr
    assert envs[0].stats() == envs[1].stats()


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("n", [224 * 300, 224 * 37 + 48, 224 * 900 + 16, 224 * 20 + 100])   # one wave and a bit, a ragged single wave, three waves, a tail for the plain kernel (n % 16 != 0)
def test_chained_replay_launches_are_bitwise_equal_to_the_plain_kernel(dtype, n):
    """Back-to-back cavgym_replay launches chain tile by tile (kernels_tma.cuh: a CTA waits for ITS tile's sequence number,
    not for the whole previous grid), so consecutive launches overlap on the device.  A train of launches issued without any
    synchronisation in between — chunks of different lengths, a whole-batch reset and a masked reset in the middle, which
    break the chain — must leave the same trajectories, state, latches and counters as the plain kernel."""
    import torch
    meta, episodes = load_golden("pedestrians_rc_seed0")
    m, k = meta["n_bodies"], len(episodes)
    t_max = 260
    init = soa(np.stack([episodes[e % k]["init_state"] for e in range(n)]))
    actions = np.zeros((t_max, m, 2, n))
    for j, ep in enumerate(episodes):
        a = ep["actions"][:t_max]
        actions[:a.shape[0], :, :, j::k] = a[..., None]
    envs = [make_env(meta, n, dtype), make_env(meta, n, dtype)]
    envs[1].set_step_path(use_tma=False)
    acts = torch.tensor(actions, dtype=envs[0].dtype, device=envs[0].device)
    mask = torch.zeros(n, dtype=torch.bool, device=envs[0].device)
    mask[::3] = True
    results = []
    for env in envs:
        env.reset(init_state=init)
        outs, t = [], 0
        for i, chunk in enumerate([5, 5, 5, 1, 2, 20, 20, 20, 3, 7, 20, 20, 5, 5, 40, 40, 20, 20]):
            if i == 8:
                env.reset(init_state=init)          # breaks the chain: the next launch waits for the whole stream again
            if i == 13:
                env.reset(mask=mask)
            outs.append(env.replay(acts[t:t + chunk], record=("state", "reward", "done", "winner", "tangent") if i % 2 else ("state",)))
            t += chunk
        results.append((outs, env))
    torch.cuda.synchronize()
    for a, b in zip(results[0][0], results[1][0]):
        for key in a:
            if a[key] is not None:
                assert torch.equal(a[key], b[key]), key
    for attr in ("state", "episode_liveness", "timestep", "done_latch", "winner_latch"):
        assert torch.equal(getattr(envs[0], attr), getattr(envs[1], attr)), attr
    assert envs[0].stats() == envs[1].stats()


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_road_kerb_and_corner_shares_match_oracle(dtype):
    """percentage_intersects (geometry.py:80-87) on the engine's closed-form paths: pedestrians are placed astride the
    kerbs and the four corners of the road with random headings (and a few clear of it / inside it), stepped with small
    steering so that the boxes rotate, and the road-share dependent outputs (reward, liveness) are compared with the
    CPU oracle, whose clipping is the reference's formulation with exact predicates."""
    from oracle.oracle import Oracle
    meta, _ = load_golden("pedestrians_rc_seed0")
    cfg = meta["config"]
    cfg["terminate_collisions"], cfg["terminate_ego_zones"] = "none", False   # keep every env alive: only shares matter
    comp = compile_from_meta(meta)
    n, steps = 4096, 12
    rng = np.random.default_rng(5)
    x0, x1, y0, y1 = 0.0, 1584.0, -58.4, 58.4                           # the stock road rectangle (SURVEY appendix A)
    where = rng.integers(0, 8, n)
    px = np.where(where % 4 == 0, x0, np.where(where % 4 == 1, x1, rng.uniform(x0 + 30, x1 - 30, n))) + rng.uniform(-9, 9, n)
    py = np.where(where < 6, np.where(rng.random(n) < 0.5, y0, y1), rng.uniform(-40, 40, n)) + rng.uniform(-9, 9, n)
    init = np.zeros((2, 4, n))
    init[0] = np.array([600.0, 29.2, 0.0, 0.0])[:, None]                # ego parked mid-road
    init[1, 0], init[1, 1], init[1, 2], init[1, 3] = px, py, 22.4, rng.uniform(-np.pi, np.pi, n)
    actions = np.zeros((steps, 2, 2, n))
    actions[:, 1, 1] = rng.uniform(-0.4 * np.pi, 0.4 * np.pi, (steps, n)) * (rng.random((steps, n)) < 0.5)
    from cavgym_b200 import BatchedCAVEnv
    env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=comp)
    oracle = Oracle(comp, n, threads=8)
    if dtype == "float32":
        init, actions = init.astype(np.float32).astype(np.float64), actions.astype(np.float32).astype(np.float64)
    env.reset(init_state=init)
    oracle.reset(init_state=init)
    out = env.replay(actions)
    want_state, want_reward, want_done, want_winner, _ = oracle.replay(actions)
    reward = out["reward"].double().cpu().numpy()
    tangent = out["tangent"].cpu().numpy().astype(bool)
    tol = 1e-9 if dtype == "float64" else 2e-3
    err = np.abs(reward - want_reward)
    assert err[:, 1].max() < tol * 4.0, err[:, 1].max()                 # reward = cost_step (4) * share terms
    live = env.episode_liveness.cpu().numpy()
    mism = live[1] != oracle.liveness[1]
    assert not np.any(mism & ~tangent.any(axis=0))                      # p > 0.5 events identical off flagged steps
    if dtype == "float64":
        assert mism.sum() == 0
    # the placement really exercises every class of case: share 0, share 1 and > 1000 distinct fractional shares
    share = ((1584.0 - 600.0) / 1584.0 * 4.0 - want_reward[0, 1]) / 4.0
    assert (share < 1e-12).sum() > 100 and (share > 1 - 1e-12).sum() > 100 and len(np.unique(np.round(share, 9))) > 1000


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_step_host_zero_copy_equals_staged_copies_and_device_step(dtype):
    """cavgym_step_host with pinned buffers (one launch reading / writing host memory over PCIe) against the staged
    path (chunked async copies) and against cavgym_step on device tensors: identical bits in every output."""
    import torch
    meta, episodes = load_golden("pedestrians_rc_seed0")
    n, m, k, t_max = 128 * 4 + 64, meta["n_bodies"], len(episodes), 60
    init = soa(np.stack([episodes[e % k]["init_state"] for e in range(n)]))
    actions = np.zeros((t_max, m, 2, n))
    for j, ep in enumerate(episodes):
        actions[:, :, :, j::k] = ep["actions"][:t_max, :, :, None]
    envs = [make_env(meta, n, dtype) for _ in range(3)]
    envs[1].set_host_path(zero_copy=False)
    tdtype = envs[0].dtype
    host = [{"actions": torch.empty((m, 2, n), dtype=tdtype).pin_memory(), "state": torch.empty((m, 4, n), dtype=tdtype).pin_memory(),
             "reward": torch.empty((m, n), dtype=tdtype).pin_memory(), "done": torch.empty(n, dtype=torch.uint8).pin_memory(),
             "winner": torch.empty(n, dtype=torch.int32).pin_memory(), "tangent": torch.empty(n, dtype=torch.uint8).pin_memory()}
            for _ in range(2)]
    acts = torch.tensor(actions, dtype=tdtype)
    for env in envs:
        env.reset(init_state=init)
    for t in range(t_max):
        for env, h in zip(envs[:2], host):
            h["actions"].copy_(acts[t])
            env.step_host(h["actions"], h["state"], h["reward"], h["done"], h["winner"], h["tangent"])
        state, reward, done, winner, tangent = envs[2].step(acts[t].to(envs[2].device))
        for key, dev in (("state", state), ("reward", reward), ("done", done), ("winner", winner), ("tangent", tangent)):
            assert torch.equal(host[0][key], host[1][key]), (t, key)
            assert torch.equal(host[0][key], dev.cpu()), (t, key)
    assert envs[0].stats() == envs[1].stats() == envs[2].stats()
    assert envs[0].launch_count() <= envs[1].launch_count()  # one launch per step; the staged path launches one per env-chunk


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_sharded_engines_match_one_engine(dtype):
    """Env-sharding (SURVEY §8e): two engines holding global envs [0, n) and [n, 2n) give exactly the states and episode
    counters of one engine holding [0, 2n) — Philox is keyed by the global env id (cavgym_set_shard).  The CPU twin with
    two gloo ranks and the all-reduce is tests/test_distributed.py."""
    meta, _ = load_golden("pedestrians_rc_eps05_seed1")
    n, steps = 3000, 700
    whole = make_env(meta, 2 * n, dtype, mode="device", seed=5)
    whole.reset()
    whole.rollout(steps, auto_reset=True)
    want_state, want = whole.state.cpu().numpy(), whole.stats()
    total = None
    for r in range(2):
        part = make_env(meta, n, dtype, mode="device", seed=5, env_offset=r * n)
        part.reset()
        part.rollout(steps, auto_reset=True)
        assert np.array_equal(part.state.cpu().numpy(), want_state[:, :, r * n:(r + 1) * n])
        got = part.stats()
        total = got if total is None else {k: total[k] + got[k] for k in got}
    assert total == want and want["episodes"] > n


def check_wire_format(compiled, init, actions):
    """cavgym_step_host_f32 on `actions` [T, M, 2, N] nudged off float32-representable values, against a second fp64 engine
    stepped on the device with the widened actions: the engine states are BITWISE equal, the outputs are their float32
    roundings, the events identical.  `compiled`: two CompiledScenario of the same scenario; `init`: initial states or None
    (both engines draw the same spawns).  Returns the wire engine's stats()."""
    import torch
    from cavgym_b200 import BatchedCAVEnv
    steps, m, _, n = actions.shape
    actions = actions * (1.0 - 1e-4 * np.random.RandomState(0).uniform(0.1, 1.0, actions.shape))   # inside the bounds
    wire = torch.tensor(actions, dtype=torch.float32).pin_memory()
    a, b = (BatchedCAVEnv(None, None, None, num_envs=n, dtype="float64", compiled=c) for c in compiled)
    a.reset(init_state=init)
    b.reset(init_state=init)
    h_state = torch.empty((m, 4, n), dtype=torch.float32).pin_memory()
    h_reward = torch.empty((m, n), dtype=torch.float32).pin_memory()
    h_done, h_winner = torch.empty(n, dtype=torch.uint8).pin_memory(), torch.empty(n, dtype=torch.int32).pin_memory()
    h_tangent = torch.empty(n, dtype=torch.uint8).pin_memory()
    for t in range(steps):
        a.step_host(wire[t], h_state, h_reward, h_done, h_winner, h_tangent)
        state, reward, done, winner, tangent = b.step(wire[t].double().cuda())
        assert torch.equal(a.state, b.state), t
        assert torch.equal(h_state, state.float().cpu()) and torch.equal(h_reward, reward.float().cpu()), t
        assert torch.equal(h_done, done.cpu()) and torch.equal(h_winner, winner.cpu()) and torch.equal(h_tangent, tangent.cpu()), t
    assert a.stats() == b.stats() and a.stats()["errors"] == 0
    with pytest.raises(Exception, match="page-locked"):
        a.step_host(wire[0].clone(), h_state, h_reward, h_done, h_winner, h_tangent)      # pageable actions
    return a.stats()


def test_float32_wire_format_is_the_fp64_engine_on_widened_actions():
    """cavgym_step_host_f32: float32 actions in, float32 state / rewards out, fp64 engine.  Against a second fp64 engine stepped
    on the device with the widened actions: the engine states are BITWISE equal, the outputs are their float32 roundings, the
    events identical."""
    meta, episodes = load_golden("learn_election3_seed22")      # four bodies; episodes of 116, 901, 218 and 79 steps
    k, n, steps = len(episodes), 4096, 250
    init = soa(np.stack([episodes[e % k]["init_state"] for e in range(n)]))
    actions = np.zeros((steps, meta["n_bodies"], 2, n))
    for j, ep in enumerate(episodes):
        a = ep["actions"][:steps]
        actions[:a.shape[0], :, :, j::k] = a[..., None]
    stats = check_wire_format([compile_from_meta(meta) for _ in range(2)], init, actions)
    assert stats["episodes"] > n // 2


@pytest.mark.parametrize("m, family", [pytest.param(m, family, id=f"{family}_m{m}") for family in FAMILIES for m in MATRIX_M])
def test_float32_wire_format_in_every_body_count_and_family(m, family):
    """The same on random valid actions in every (body count, family) cell of helpers.matrix_scenario, so that each
    instantiation of step_wire32_kernel runs: 692 envs, max_timesteps 60, every env times out inside the 90 steps."""
    n, steps = 692, 90
    compiled = [matrix_scenario(m, family, "external", max_timesteps=60) for _ in range(2)]
    actions = random_actions(np.random.RandomState(m), steps, n, compiled[0].is_car)
    stats = check_wire_format(compiled, None, actions)
    assert stats["episodes"] >= n


def test_sweep_totals_do_not_depend_on_the_split():
    """BASELINE config C5's claim: the seed sweep over a fixed GLOBAL env set gives identical totals however many GPUs share
    it.  The same 8,192 global envs are run as 1, 2, 4 and 8 shards (sharding.split_envs; one engine per shard, as one rank
    per GPU would hold them) for the same number of steps; every counter, summed over the shards, must be identical."""
    from cavgym_b200 import sharding
    meta, _ = load_golden("pedestrians_rc_eps05_seed1")
    total, steps = 8192, 1500
    want = None
    for world in (1, 2, 4, 8):
        summed = None
        for offset, count in sharding.split_envs(total, world):
            part = make_env(meta, count, "float64", mode="device", seed=0, env_offset=offset)
            part.reset()
            for _ in range(3):
                part.rollout(steps // 3, auto_reset=True)
            got = part.stats()
            summed = got if summed is None else {k: summed[k] + got[k] for k in got}
            part.close()
        if want is None:
            want = summed
            assert want["episodes"] > total and want["interesting"] > 0
        assert summed == want, world


def test_two_engines_on_two_devices_in_one_process():
    """The TMA kernels opt in to > 48 KB of shared memory per DEVICE: a second engine on another GPU of the same process must
    get its own opt-in (the launchers cache it per device)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    meta, episodes = load_golden("pedestrians_rc_seed0")
    ep = episodes[0]
    n = 256
    init = soa(np.repeat(ep["init_state"][None], n, axis=0))
    actions = np.repeat(ep["actions"][:40][..., None], n, axis=-1)
    outs = []
    for index in (0, 1):
        with torch.cuda.device(index):
            env = make_env(meta, n, "float64", device=f"cuda:{index}")
            env.reset(init_state=init)
            env.step(actions[0])
            out = env.replay(actions[1:])
            outs.append(out["state"].cpu().numpy())
            env.close()
    assert np.array_equal(outs[0], outs[1])
    assert state_err(np.moveaxis(outs[0][:, :, :, 0], 0, 0), ep["state"][1:40]) < 1e-9


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("name", __import__("helpers").INFO_CASES)
def test_info_matches_reference(name, dtype):
    """cavgym_info against env.info() recorded from the unmodified reference (environment.py:106-117): body polygons and road
    angles within the state tolerance, None (NaN) for exactly the same bodies — one env per recorded step."""
    from helpers import load_info_golden
    meta, state, polygons, angles = load_info_golden(name)
    t_len = state.shape[0]
    env = make_env(meta, t_len, dtype)
    env.reset(init_state=np.ascontiguousarray(np.transpose(state, (1, 2, 0))))
    out = env.info()
    got_polygons = np.transpose(out["body_polygons"].double().cpu().numpy(), (2, 0, 1))
    got_angles = out["road_angles"].double().cpu().numpy().T
    tol = REL[dtype]
    assert np.max(np.abs(got_polygons - polygons) / np.maximum(1.0, np.abs(polygons))) < tol
    # a body whose box edge lies within the tolerance of the road edge may be classified either way in fp32
    defined = np.isfinite(got_angles) & np.isfinite(angles)
    disagree = np.isfinite(got_angles) != np.isfinite(angles)
    assert disagree.sum() <= (0 if dtype == "float64" else max(2, angles.size // 200))
    d = got_angles[defined] - angles[defined]
    assert np.max(np.abs(np.arctan2(np.sin(d), np.cos(d)))) < (1e-9 if dtype == "float64" else 1e-4)
    assert defined.sum() > 100
    # polygons only / angles only
    only = env.info(road_angles=False)
    assert only["road_angles"] is None and only["body_polygons"].shape == (meta["n_bodies"], 8, t_len)


@pytest.mark.parametrize("name", ["pedestrians_rc_seed0", "pedestrians_rc_eps05_seed1", "pedestrians3_rc_seed2", "pedestrians_proximity_seed3",
                                  "pedestrians_random_all_seed4", "pelican_random_all_seed10", "crossroads_random_all_seed6"])
def test_device_agents_follow_reference_with_replayed_draws(name):
    """The ON-DEVICE agents (crossing state machine, steering inverse, RandomAgent; agents.cuh) fed with the MT19937 draws the
    reference consumed (cavgym_set_uniform_override): the actions they choose, the agents' internal state, the body state and
    the events must follow the reference's own run — one env per recorded episode, no replayed actions anywhere."""
    import torch
    meta, episodes = load_golden(name)
    n, m = len(episodes), meta["n_bodies"]
    t_max = max(ep["actions"].shape[0] for ep in episodes)
    env = make_env(meta, n, "float64", mode="device")
    env.set_action_logging(True)
    env.reset(init_state=soa(np.stack([ep["init_state"] for ep in episodes])))
    starts = {int(ep["t_global_start"]) for ep in episodes}
    env.set_global_timestep(starts.pop() if len(starts) == 1 else -10 ** 9)
    draws = np.full((t_max, m, 3, n), 0.5)
    for e, ep in enumerate(episodes):
        draws[:ep["draws"].shape[0], :, :, e] = np.nan_to_num(ep["draws"], nan=0.5)
    override = torch.zeros((m, 3, n), dtype=torch.float64, device=env.device)
    env.set_uniform_override(override)
    draws_t = torch.tensor(draws, device=env.device)
    flagged = 0
    for t in range(t_max):
        override.copy_(draws_t[t])
        state, reward, done, winner, tangent = env.step(None)
        state_h, taken, agent_h = state.cpu().numpy(), env.actions_taken.cpu().numpy(), env.agent_state.cpu().numpy()
        done_h, winner_h, tangent_h = done.cpu().numpy(), winner.cpu().numpy(), tangent.cpu().numpy()
        for e, ep in enumerate(episodes):
            if t >= ep["actions"].shape[0]:
                continue
            flagged += int(tangent_h[e])
            assert rel_err(taken[:, :, e], ep["actions"][t]) < 1e-9, (name, e, t)
            assert state_err(state_h[:, :, e], ep["state"][t]) < 1e-9, (name, e, t)
            if not tangent_h[e]:
                assert bool(done_h[e]) == bool(ep["done"][t]) and int(winner_h[e]) == int(ep["winner"][t]), (name, e, t)
            want = ep["agent_state"][t]
            crossing = ~np.isnan(want).all(axis=1)
            got = agent_h[:, :, e]
            assert np.array_equal(np.isnan(got[crossing]), np.isnan(want[crossing])), (name, e, t)
            g, w = np.nan_to_num(got[crossing]), np.nan_to_num(want[crossing])
            assert rel_err(g[:, :3], w[:, :3]) < 1e-9, (name, e, t)          # initial distance, waypoint x, y
            d = g[:, 3:] - w[:, 3:]                                            # target / prior orientation: angles, +pi == -pi
            assert np.max(np.abs(np.arctan2(np.sin(d), np.cos(d))), initial=0.0) < 1e-9, (name, e, t)
    assert flagged < 0.02 * sum(ep["actions"].shape[0] for ep in episodes)


def test_replay_on_pinned_host_tensors_equals_replay_on_device_tensors():
    """BatchedCAVEnv.replay_host: cavgym_replay reading its actions from and writing its trajectories to pinned host memory.
    Bitwise the device-buffer replay, over several calls (chunked like a caller would) and with optional outputs left out."""
    import torch
    meta, episodes = load_golden("pedestrians_rc_eps05_seed1")
    k, n, steps = len(episodes), 2048, 90
    init = soa(np.stack([episodes[e % k]["init_state"] for e in range(n)]))
    actions = np.zeros((steps, meta["n_bodies"], 2, n))
    for j, ep in enumerate(episodes):
        actions[:, :, :, j::k] = ep["actions"][:steps][..., None]
    a, b = make_env(meta, n, "float64"), make_env(meta, n, "float64")
    a.reset(init_state=init)
    b.reset(init_state=init)
    want = b.replay(actions)
    h_actions = torch.tensor(actions).pin_memory()
    m = meta["n_bodies"]
    out = {"state": torch.empty((steps, m, 4, n), dtype=torch.float64).pin_memory(), "reward": torch.empty((steps, m, n), dtype=torch.float64).pin_memory(),
           "done": torch.empty((steps, n), dtype=torch.uint8).pin_memory(), "winner": torch.empty((steps, n), dtype=torch.int32).pin_memory(),
           "tangent": torch.empty((steps, n), dtype=torch.uint8).pin_memory()}
    for at in range(0, steps, 30):
        a.replay_host(h_actions[at:at + 30], **{key: value[at:at + 30] for key, value in out.items()})
    for key in out:
        assert torch.equal(out[key], want[key].cpu()), key
    assert torch.equal(a.state, b.state) and a.stats() == b.stats()
    a.replay_host(h_actions[:5], reward=out["reward"][:5])                  # only the rewards
    with pytest.raises(ValueError, match="pinned"):
        a.replay_host(torch.tensor(actions[:5]), reward=out["reward"][:5])  # pageable actions
