"""Per-env tester parameters (BatchedCAVEnv.set_agent_params, cavgym_set_agent_params) on the thread-per-env kernels.

The contract: with every slot set to the scenario's own values the parameter kernels give exactly the plain kernels'
results; a batch whose blocks of slots carry different values is bitwise the engines built with each block's value in the
scenario and the block's global env ids (set_shard), laid side by side; the parameters belong to the slots (reset, fork and
checkpoints keep them where they are); and every path that does not read them refuses to run while they are set.

Scenarios run with max_timesteps lowered to 23 so that, in windows of 30 and 35 steps, episodes end and restart inside a
window.  Block edges (70 and 150 of 203 envs) fall inside a warp and inside a CTA of every rollout kernel.
"""
import copy

import numpy as np
import pytest
import torch

from helpers import FAMILIES, MATRIX_M, compile_from_meta, load_golden, matrix_scenario

pytestmark = pytest.mark.gpu

MAX_T = 23
WINDOWS = (30, 35)
N = 203
BLOCKS = ((0, 70), (70, 150), (150, 203))
SNAP = ("state", "action", "agent", "cs", "liveness", "t_ep", "episode", "winner", "active", "done", "err")
RECORD = ("observation", "action", "state", "reward", "done", "winner", "tangent", "timestep")
STOCK = ("pedestrians_rc_seed0", "crossroads_random_all_seed6", "busstop_random_all_seed8", "pelican_random_all_seed10",
         "pedestrians_proximity_seed3", "learn_election3_seed22", "pedestrians_random_all_seed4")
CASES = [("golden", name) for name in STOCK] + [("matrix", m, family) for m in MATRIX_M for family in FAMILIES]
DTYPES = ("float64", "float32")


def case_id(case):
    return case[1] if case[0] == "golden" else f"{case[2]}_{case[1]}_bodies"


def compiled(case, epsilon=None, threshold=None):
    """The scenario of `case` with on-device agents; epsilon / threshold: {body: value} written into its tables."""
    if case[0] == "golden":
        meta = copy.deepcopy(load_golden(case[1])[0])
        meta["config"]["max_timesteps"] = MAX_T
        comp = compile_from_meta(meta, mode="device")
    else:
        comp = matrix_scenario(case[1], case[2], "device", max_timesteps=MAX_T)
    for b, value in (epsilon or {}).items():
        comp.struct.bodies[b].agent_epsilon = value
    for b, value in (threshold or {}).items():
        comp.struct.bodies[b].agent_threshold = value
    return comp


def make(comp, n, dtype, offset=0, seed=5):
    from cavgym_b200 import BatchedCAVEnv
    env = BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=comp, seed=seed, env_offset=offset)
    env.set_episode_log(64 * n)
    return env


def own_values(env):
    """[M, N] epsilon and threshold holding the scenario's values in the rows that are read and NaN in every other row."""
    eps_rows, thr_rows = env.agent_rows()
    m, n = env.num_bodies, env.num_envs
    eps = torch.full((m, n), float("nan"), dtype=torch.float64)
    thr = torch.full((m, n), float("nan"), dtype=torch.float64)
    for b in eps_rows:
        eps[b] = env.compiled.struct.bodies[b].agent_epsilon
    for b in thr_rows:
        thr[b] = env.compiled.struct.bodies[b].agent_threshold
    return eps, thr


def snapshot(env, lo=0, hi=None):
    snap = env.save_envs()
    hi = env.num_envs if hi is None else hi
    return {name: snap[name][..., lo:hi].cpu() for name in SNAP}


def rows_by_env(rows):
    return np.sort(rows, order=("env", "episode"))


def run(env, path, auto_reset):
    """The same call sequence on any engine: two windows of rollout, of recorded rollout, or of step() with device agents
    (finished envs reset before every step with auto_reset, as rollout's auto-reset does).  Returns the records."""
    records = []
    env.reset()
    for window in WINDOWS:
        if path == "rollout":
            env.rollout(window, auto_reset=auto_reset)
        elif path == "record":
            records.append({k: v.cpu() for k, v in env.rollout(window, auto_reset=auto_reset, record=RECORD).items()})
        else:
            for _ in range(window):
                if auto_reset:
                    env.reset(mask=env.done_latch.clone())
                _, reward, done, winner, tangent = env.step(None)
                records.append({"reward": reward.cpu(), "done": done.cpu(), "winner": winner.cpu(), "tangent": tangent.cpu()})
    if path == "step" and auto_reset:
        env.reset(mask=env.done_latch.clone())
    return records


def results(env, records):
    rows, dropped = env.drain_episodes()
    assert dropped == 0
    return {"snap": snapshot(env), "stats": env.stats(), "rows": rows_by_env(rows), "t_global": env._engine_state().t_global,
            "records": records}


def assert_same(a, b, what=""):
    for name in SNAP:
        assert torch.equal(a["snap"][name].view(torch.uint8) if a["snap"][name].is_floating_point() else a["snap"][name],
                           b["snap"][name].view(torch.uint8) if b["snap"][name].is_floating_point() else b["snap"][name]), (what, name)
    assert a["stats"] == b["stats"], what
    assert np.array_equal(a["rows"], b["rows"]), what
    assert a["t_global"] == b["t_global"], what
    assert len(a["records"]) == len(b["records"])
    for ra, rb in zip(a["records"], b["records"]):
        for key in ra:
            assert torch.equal(ra[key].view(torch.uint8) if ra[key].is_floating_point() else ra[key],
                               rb[key].view(torch.uint8) if rb[key].is_floating_point() else rb[key]), (what, key)


# ------------------------------------------------------------------ 1. uniform equals plain
@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("path", ["rollout", "step", "record"])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_scenario_values_in_every_slot_give_the_plain_results(case, dtype, path, auto_reset):
    plain = make(compiled(case), N, dtype)
    want = results(plain, run(plain, path, auto_reset))
    env = make(compiled(case), N, dtype)
    eps, thr = own_values(env)
    env.set_agent_params(eps, thr)
    got = results(env, run(env, path, auto_reset))
    assert_same(got, want, "parameters = the scenario's values")
    assert want["stats"]["episodes"] > 0


# ------------------------------------------------------------------ 2. a sweep equals its parts
# (case, parameter, values per block): Random and RandomConstrained testers sweep epsilon, proximity and election thresholds
SWEEPS = {
    "rc_pedestrians": (("golden", "pedestrians_rc_seed0"), "epsilon", (0.5, 0.05, 0.01)),
    "random_pedestrians": (("golden", "pedestrians_random_all_seed4"), "epsilon", (0.5, 0.0, 0.05)),
    "random_bus_stop": (("golden", "busstop_random_all_seed8"), "epsilon", (0.3, 0.01, 0.1)),
    "random_pelican": (("golden", "pelican_random_all_seed10"), "epsilon", (0.5, 0.05, 0.2)),
    "proximity": (("golden", "pedestrians_proximity_seed3"), "threshold", (300.0, 544.0, 800.0)),
    "election": (("golden", "learn_election3_seed22"), "threshold", (700.0, 300.0, 544.0)),
}


def rows_of_testers(env, name):
    eps_rows, thr_rows = env.agent_rows()
    return [b for b in (eps_rows if name == "epsilon" else thr_rows) if b > 0]


def sweep_engine(case, name, per_block, dtype):
    """One engine of N envs whose block k carries per_block[k] = {body: value}; other rows NaN."""
    env = make(compiled(case), N, dtype)
    grid = torch.full((env.num_bodies, N), float("nan"), dtype=torch.float64)
    eps, thr = own_values(env)
    grid.copy_(eps if name == "epsilon" else thr)
    for (lo, hi), values in zip(BLOCKS, per_block):
        for b, value in values.items():
            grid[b, lo:hi] = value
    env.set_agent_params(**{name: grid})
    return env


def check_sweep(case, name, per_block, dtype, path, auto_reset):
    env = sweep_engine(case, name, per_block, dtype)
    whole = results(env, run(env, path, auto_reset))
    totals = {key: 0 for key in whole["stats"]}
    rows = []
    for (lo, hi), values in zip(BLOCKS, per_block):
        part = make(compiled(case, **{name: values}), hi - lo, dtype, offset=lo)
        got = results(part, run(part, path, auto_reset))
        for key in SNAP:
            a, b = got["snap"][key], whole["snap"][key][..., lo:hi]
            assert torch.equal(a.view(torch.uint8) if a.is_floating_point() else a,
                               b.contiguous().view(torch.uint8) if b.is_floating_point() else b.contiguous()), (lo, key)
        for ra, rb in zip(got["records"], whole["records"]):
            for key in ra:
                assert torch.equal(ra[key], rb[key][..., lo:hi]) or torch.equal(ra[key].nan_to_num(7.0), rb[key][..., lo:hi].nan_to_num(7.0)), (lo, key)
        assert got["t_global"] == whole["t_global"]
        rows.append(got["rows"])
        for key, value in got["stats"].items():
            totals[key] += value
    assert np.array_equal(rows_by_env(np.concatenate(rows)), whole["rows"])
    assert totals == whole["stats"]
    return whole


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("path", ["rollout", "record", "step"])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("sweep", sorted(SWEEPS))
def test_a_sweep_is_its_single_value_engines_side_by_side(sweep, dtype, path, auto_reset):
    case, name, values = SWEEPS[sweep]
    env = make(compiled(case), 1, dtype)
    bodies = rows_of_testers(env, name)
    env.close()
    per_block = [{b: v for b in bodies} for v in values]
    whole = check_sweep(case, name, per_block, dtype, path, auto_reset)
    assert whole["stats"]["episodes"] > 0


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("m", [3, 5])
def test_two_pedestrians_of_one_env_with_different_values(m, dtype):
    """Homogeneous cells (m = 5: the rolled kernels): every pedestrian of an env gets its own epsilon."""
    case = ("matrix", m, "homogeneous")
    values = [{b: (0.9, 0.01, 0.3, 0.6, 0.05, 0.2, 0.7)[(b + 2 * k) % 7] for b in range(1, m)} for k in range(len(BLOCKS))]
    check_sweep(case, "epsilon", values, dtype, "rollout", True)
    check_sweep(case, "epsilon", values, dtype, "record", False)


# ------------------------------------------------------------------ 3. limits
@pytest.mark.parametrize("dtype", DTYPES)
def test_epsilon_zero_is_a_noop_agent_and_one_acts_every_step(dtype):
    case = ("golden", "pedestrians_random_all_seed4")
    env = make(compiled(case), N, dtype)
    testers = rows_of_testers(env, "epsilon")
    eps, _ = own_values(env)
    eps[testers] = 0.0
    env.set_agent_params(eps)
    meta = copy.deepcopy(load_golden(case[1])[0])
    meta["config"]["max_timesteps"] = MAX_T
    meta["config"]["tester_config"] = {"option": "noop"}
    noop = make(compile_from_meta(meta, mode="device"), N, dtype)
    for e in (env, noop):
        e.reset()
        e.rollout(WINDOWS[0], auto_reset=True)
    a, b = snapshot(env), snapshot(noop)
    for key in ("state", "cs", "liveness", "t_ep", "episode", "winner", "done"):
        assert torch.equal(a[key], b[key]), key
    assert env.stats() == noop.stats()

    eps[testers] = 1.0
    env.set_agent_params(eps)
    env.reset()
    rec = env.rollout(WINDOWS[0], auto_reset=False, record=("action", "timestep"))
    action, ts = rec["action"][:, testers].cpu(), rec["timestep"].cpu()
    stepped = (ts[1:] > 1)   # a step after the first of an episode: its action must be a fresh draw
    assert stepped.any()
    changed = (action[1:] != action[:-1]).all(dim=2)   # both components redrawn
    assert changed[:, :, :][stepped.unsqueeze(1).expand_as(changed)].all()


# ------------------------------------------------------------------ 4. paths agree
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("sweep", ["rc_pedestrians", "random_bus_stop", "election"])
def test_step_equals_rollout_and_recording_changes_nothing(sweep, dtype):
    case, name, values = SWEEPS[sweep]
    probe = make(compiled(case), 1, dtype)
    per_block = [{b: v for b in rows_of_testers(probe, name)} for v in values]
    probe.close()
    out = {}
    for path in ("rollout", "step", "record"):
        env = sweep_engine(case, name, per_block, dtype)
        env.set_action_logging(True)
        out[path] = results(env, run(env, path, True))
        out[path]["records"] = []
    assert_same(out["step"], out["rollout"], "step() with device agents vs rollout(auto_reset=True)")
    assert_same(out["record"], out["rollout"], "recorded vs plain rollout")


# ------------------------------------------------------------------ 5. against the oracle
@pytest.mark.parametrize("m, family", [(3, "homogeneous"), (4, "generic")])
def test_blocks_against_the_oracle_fp64(m, family):
    """Each block of a sweep against the C oracle run with that block's scenario and global ids, step by step."""
    from oracle.oracle import Oracle
    from helpers import state_err
    case = ("matrix", m, family)
    probe = make(compiled(case), 1, "float64")
    testers = rows_of_testers(probe, "epsilon")
    probe.close()
    values = (0.9, 0.02, 0.3)
    env = sweep_engine(case, "epsilon", [{b: v for b in testers} for v in values], "float64")
    env.set_action_logging(True)
    env.reset()
    oracles = []
    for (lo, hi), v in zip(BLOCKS, values):
        oracle = Oracle(compiled(case, epsilon={b: v for b in testers}), hi - lo, seed=5, threads=8)
        oracle.set_shard(lo)
        oracle.reset()
        oracles.append(oracle)
    live = np.ones(N, dtype=bool)   # envs not yet past a flagged (near-tangent) step
    for t in range(WINDOWS[0]):
        env.reset(mask=env.done_latch.clone())
        before = env.state.cpu().numpy()
        for (lo, hi), oracle in zip(BLOCKS, oracles):
            keep = live[lo:hi]
            assert state_err(np.moveaxis(oracle.state[:, :, keep], -1, 0), np.moveaxis(before[:, :, lo:hi][:, :, keep], -1, 0)) <= 1e-9, (t, lo)
        _, _, done, _, tangent = env.step(None)
        done, tangent, ts = done.cpu().numpy(), tangent.cpu().numpy(), env.timestep.cpu().numpy()
        state, actions = env.state.cpu().numpy(), env.actions_taken.cpu().numpy()
        for (lo, hi), oracle in zip(BLOCKS, oracles):
            oracle.rollout(1, auto_reset=True)
            kept = live[lo:hi] & ~((done[lo:hi] == 1) | (ts[lo:hi] >= MAX_T))   # the oracle resets finished envs after the step
            assert state_err(np.moveaxis(oracle.state[:, :, kept], -1, 0), np.moveaxis(state[:, :, lo:hi][:, :, kept], -1, 0)) <= 1e-9, (t, lo)
            assert np.max(np.abs(oracle.actions_taken[:, :, kept] - actions[:, :, lo:hi][:, :, kept]), initial=0) <= 1e-9, (t, lo)
        live &= tangent == 0
    assert live.sum() > N // 2


# ------------------------------------------------------------------ 6. slots and checkpoints
@pytest.mark.parametrize("dtype", DTYPES)
def test_a_fork_continues_under_its_target_slot(dtype):
    case, name, values = SWEEPS["rc_pedestrians"]
    probe = make(compiled(case), 1, dtype)
    testers = rows_of_testers(probe, name)
    probe.close()
    per_block = [{b: v for b in testers} for v in values]
    env = sweep_engine(case, name, per_block, dtype)
    env.reset()
    env.rollout(10, auto_reset=True)
    src, dst = [3, 5, 66], [160, 170, 202]            # block 0 -> block 2
    source = env.save_envs(src)
    env.fork(src, dst)
    lo, hi = BLOCKS[2]
    ref = make(compiled(case, **{name: per_block[2]}), hi - lo, dtype, offset=lo)
    ref.reset()
    ref.set_global_timestep(env._engine_state().t_global)
    ref.load_envs(source, [d - lo for d in dst])
    env.rollout(WINDOWS[1], auto_reset=True)
    ref.rollout(WINDOWS[1], auto_reset=True)
    a, b = snapshot(env), snapshot(ref)
    for key in SNAP:
        x, y = a[key][..., dst].contiguous(), b[key][..., [d - lo for d in dst]].contiguous()
        assert torch.equal(x.view(torch.uint8), y.view(torch.uint8)) if x.is_floating_point() else torch.equal(x, y), key


@pytest.mark.parametrize("dtype", DTYPES)
def test_a_checkpoint_continues_and_clearing_restores_the_plain_kernels(dtype):
    case, name, values = SWEEPS["proximity"]
    probe = make(compiled(case), 1, dtype)
    per_block = [{b: v for b in rows_of_testers(probe, name)} for v in values]
    probe.close()
    env = sweep_engine(case, name, per_block, dtype)
    env.reset()
    env.rollout(WINDOWS[0], auto_reset=True)
    env.drain_episodes()
    checkpoint = env.state_dict()
    assert "agent_threshold" in checkpoint and "agent_epsilon" not in checkpoint
    fresh = make(compiled(case), N, dtype)
    fresh.load_state_dict(checkpoint)
    assert torch.equal(fresh.agent_params()[1].cpu().nan_to_num(-1.0), env.agent_params()[1].cpu().nan_to_num(-1.0))
    for e in (env, fresh):
        e.rollout(WINDOWS[1], auto_reset=True)
    assert_same(results(fresh, []), results(env, []), "checkpoint with parameters")

    # a checkpoint without parameters clears them
    plain = make(compiled(case), N, dtype)
    plain.reset()
    fresh.load_state_dict(plain.state_dict())
    assert fresh.agent_params() == (None, None)

    # clearing: the plain kernels again, launch for launch
    cleared = make(compiled(case), N, dtype)
    eps, thr = own_values(cleared)
    cleared.set_agent_params(threshold=thr * 2)
    cleared.set_agent_params()
    reference = make(compiled(case), N, dtype)
    counts = []
    for e in (cleared, reference):
        before = e.launch_count()
        out = results(e, run(e, "rollout", True))
        counts.append((e.launch_count() - before, out))
    assert counts[0][0] == counts[1][0]
    assert_same(counts[0][1], counts[1][1], "cleared parameters")


# ------------------------------------------------------------------ 7. refusals
def test_bad_values_are_refused_in_python_and_by_the_c_abi():
    import ctypes as C
    from cavgym_b200 import _native
    env = make(compiled(("golden", "pelican_random_all_seed10")), 37, "float64")
    m, n = env.num_bodies, env.num_envs
    eps, thr = own_values(env)
    rows, _ = env.agent_rows()
    lib = _native.load()
    with pytest.raises(ValueError):
        env.set_agent_params(eps[:, :5])
    for bad in (-0.1, 1.5, float("nan")):
        e = eps.clone()
        e[rows[-1], 7] = bad
        with pytest.raises(ValueError):
            env.set_agent_params(e)
        dev = e.cuda().contiguous()
        assert lib.cavgym_set_agent_params(env._handle, C.c_void_p(dev.data_ptr()), None, None) == -22
    assert env.agent_params() == (None, None)
    prox = make(compiled(("golden", "pedestrians_proximity_seed3")), 37, "float32")
    _, thr = own_values(prox)
    _, thr_rows = prox.agent_rows()
    for bad in (0.0, -3.0, float("inf"), float("nan")):
        t = thr.clone()
        t[thr_rows[0], 11] = bad
        with pytest.raises(ValueError):
            prox.set_agent_params(threshold=t)
        dev = t.to(device="cuda", dtype=torch.float32).contiguous()
        assert prox._lib.cavgym_set_agent_params(prox._handle, None, C.c_void_p(dev.data_ptr()), None) == -22
    # rows that are not read may hold anything
    e = eps.clone()
    e[0] = float("nan")
    env.set_agent_params(e)


@pytest.mark.parametrize("dtype", DTYPES)
def test_paths_that_do_not_read_parameters_refuse_while_they_are_set(dtype):
    from cavgym_b200._native import CavgymError
    env = make(compiled(("golden", "pedestrians_rc_seed0")), 64, dtype)
    eps, _ = own_values(env)
    env.set_agent_params(eps)
    with pytest.raises(CavgymError):
        env.rollout_until(5, 1.0, torch.zeros(64, dtype=env.dtype, device=env.device))
    if dtype == "float64":
        pinned = {k: torch.zeros(s, dtype=torch.float32).pin_memory() for k, s in (("state", (2, 4, 64)), ("reward", (2, 64)))}
        with pytest.raises(CavgymError):
            env.step_host(None, state_out=pinned["state"], reward_out=pinned["reward"])
    env.set_dense_path(True)
    for call in (lambda: env.step(None), lambda: env.rollout(3), lambda: env.rollout(3, record=("state",))):
        with pytest.raises(CavgymError):
            call()
    env.set_dense_path(False)
    env.rollout(3)

    from types import SimpleNamespace
    from cavgym_b200.examples.environments import dense_traffic
    from cavgym_b200.library.bodies import Pedestrian
    from cavgym_b200.scenario import AgentSpec, compile_scenario
    road_map, constants = dense_traffic.make_world()
    bodies = dense_traffic.make_bodies(np_random=np.random.RandomState(0), road_map=road_map)
    cfg = SimpleNamespace(terminate_collisions="all", terminate_ego_zones=True, terminate_ego_offroad=False, max_timesteps=MAX_T,
                          reward_win=6000.0, reward_draw=2000.0, cost_step=4.0)
    specs = [AgentSpec("random-constrained", epsilon=0.01) if isinstance(b, Pedestrian) else AgentSpec("noop") for b in bodies]
    big = make(compile_scenario(bodies, constants, cfg, specs), 8, dtype)
    eps, _ = own_values(big)
    with pytest.raises(CavgymError):
        big.set_agent_params(eps)
    big.set_agent_params()   # clearing is always allowed


# ------------------------------------------------------------------ 8. the sweep module
def test_sweep_module_matches_separate_engines_and_writes_the_reference_logs(tmp_path):
    from cavgym_b200 import reporting, sweep
    from cavgym_b200.config import make_config
    meta = copy.deepcopy(load_golden("pedestrians_rc_seed0")[0])
    meta["config"]["max_timesteps"] = 60
    config = make_config(meta["config"])
    values, n_p = (0.5, 0.05), 300
    env = config.batched(len(values) * n_p, seed=9)
    results_, per_point = sweep.run(env, "epsilon", values, n_p, episodes=2 * n_p)
    for p, value in enumerate(values):
        import dataclasses
        single = dataclasses.replace(config, tester_config=dataclasses.replace(config.tester_config, epsilon=value))
        part = single.batched(n_p, seed=9, env_offset=p * n_p)
        for _ in range(2):
            part.reset()
            part.rollout(part.max_timesteps, auto_reset=False)
        stats = part.stats()
        got = results_[p]
        assert (got.episodes, got.interesting, got.env_steps) == (stats["episodes"], stats["interesting"], stats["env_steps"])
        want_t = reporting.interval_from_sums(stats["interesting"], stats["sum_t_interesting"], stats["sum_t2_interesting"])
        want_s = reporting.interval_from_sums(stats["interesting"], stats["sum_score"], stats["sum_score2"])
        for a, b in ((got.confidence_timesteps, want_t), (got.confidence_score, want_s)):
            assert np.allclose(tuple(a), tuple(b), rtol=1e-9, equal_nan=True)
        assert got.episodes == 2 * n_p
    sweep.write_logs(config, "epsilon", results_, per_point, str(tmp_path), env.time_resolution)
    for result in results_:
        folder = tmp_path / f"epsilon={result.value:g}"
        assert make_config(__import__("json").loads((folder / "config.json").read_text())).tester_config.epsilon == result.value
        lines = (folder / "episode.log").read_text().splitlines()
        assert len(lines) == result.episodes and all(len(line.split(",")) == 5 for line in lines)
        run_line = (folder / "run.log").read_text().splitlines()
        assert len(run_line) == 1 and len(run_line[0].split(",")) == 10
        assert int(run_line[0].split(",")[3]) == result.interesting
