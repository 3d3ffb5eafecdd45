"""integration/batched.py — the binding INTEGRATION.md §A tells a CAV-Gym maintainer to add — run for real: against the
tables recorded for the unmodified reference's objects on CPU, and on the GPU against a reference trace."""
import copy
import importlib.util
import os

import numpy as np
import pytest

from helpers import load_golden, soa, state_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def binding():
    spec = importlib.util.spec_from_file_location("library_batched", os.path.join(ROOT, "integration", "batched.py"))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module


def test_binding_builds_its_tables_from_the_reference_env():
    """The walk integration/batched.py makes over an env (bodies, constants, env_config, time_resolution) gives the tables
    recorded for the reference's own pelican-crossing env (tests/golden/scenario_tables.npz, oracle/gen_tables_golden.py)."""
    from oracle import refload
    from cavgym_b200.config import make_config
    from cavgym_b200.scenario import AgentSpec, compile_scenario
    from helpers import load_scenario_tables
    data = refload.stock_config_dict(scenario="pelican-crossing", tester="random", seed=3, collisions="all")
    _, env, _, _ = make_config(copy.deepcopy(data)).setup()
    tables = compile_scenario(env.bodies, env.constants, env.env_config, [AgentSpec("external") for _ in env.bodies],
                              time_resolution=env.time_resolution).tables()
    assert len(tables["bodies"]) > 0 and tables["header"][:4] == (5).to_bytes(4, "little")
    assert tables == load_scenario_tables("binding_pelican-crossing")
    assert binding().BatchedCAVEnv.step.__doc__      # the module imports


@pytest.mark.gpu
def test_binding_steps_a_reference_trace_on_the_gpu():
    """The maintainer's binding (numpy in / out, cavgym_step_host) replays a recorded reference episode in 64 envs."""
    from cavgym_b200.config import make_config
    meta, episodes = load_golden("pedestrians_rc_seed0")
    ep = episodes[4]
    _, env, _, _ = make_config(copy.deepcopy(meta["config"])).setup()
    n = 64
    batch = binding().BatchedCAVEnv(env, n)
    state = batch.reset(init_state=soa(np.repeat(ep["init_state"][None], n, axis=0)))
    assert state_err(np.moveaxis(state, -1, 0), ep["init_state"]) == 0.0
    steps = ep["actions"].shape[0]
    for t in range(steps):
        actions = np.repeat(ep["actions"][t][..., None], n, axis=-1)
        state, reward, done, winner = batch.step(actions)
        assert state_err(np.moveaxis(state, -1, 0), ep["state"][t]) < 1e-9
        assert bool(done.all()) == bool(ep["done"][t]) and bool(done.any()) == bool(ep["done"][t])
    assert int(winner[0]) == int(ep["winner"][-1]) == 1 and batch.stats()["episodes"] == n
    again = batch.reset(mask=(np.arange(n) % 2).astype(np.uint8))      # half the envs re-spawn on the device, half stay finished
    assert state_err(np.moveaxis(again[:, :, 0::2], -1, 0), ep["state"][-1]) < 1e-9
    assert np.all(again[0, 0, 1::2] == 0.0) and np.all(np.abs(again[1, 1, 1::2]) > 60.0)   # ego back at x = 0, pedestrian on a pavement
    batch.close()
