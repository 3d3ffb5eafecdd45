"""config.json handling (reference config.py / config.json / schema.json): options, value checks, round trip, and which
on-device agent each body gets.  CPU only; the GPU side is tests/test_gpu_simulation.py."""
import copy
import json

import pytest

from cavgym_b200 import config as cfg

STOCK = {   # the keys and values of the reference's config.json, with the ego switched to noop and the mode to headless
    "verbosity": "silent", "episode_log": None, "run_log": None, "seed": 0, "episodes": 10, "max_timesteps": 1000,
    "terminate_collisions": "ego", "terminate_ego_zones": True, "terminate_ego_offroad": False,
    "reward_win": 6000.0, "reward_draw": 2000.0, "cost_step": 4.0,
    "scenario_config": {"option": "pedestrians", "num_pedestrians": 1, "outbound_pavement": 1.0, "inbound_pavement": 1.0},
    "ego_config": {"option": "noop"},
    "tester_config": {"option": "random-constrained", "epsilon": 0.01},
    "mode_config": {"option": "headless"},
}
Q_LEARNING = {"option": "q-learning", "alpha": {"start": 1.0, "stop": 0.1, "num_steps": 1000000}, "gamma": 0.9, "epsilon": 0.2,
              "feature_config": {"distance_x": False, "distance_y": False, "distance": True, "relative_angle": True,
                                 "heading": True, "on_road": False, "inverse_distance": False}, "log": None}


def stock(**changes):
    data = copy.deepcopy(STOCK)
    data.update(changes)
    return data


def test_round_trip_preserves_every_key(tmp_path):
    for data in (stock(), stock(ego_config=Q_LEARNING, mode_config={"option": "render", "episode_condition": 5, "video_dir": None}),
                 stock(scenario_config={"option": "bus-stop"}, tester_config={"option": "random", "epsilon": 0.5}, terminate_collisions="all"),
                 stock(tester_config={"option": "proximity", "threshold": 160.0}, seed=None)):
        config = cfg.make_config(copy.deepcopy(data))
        assert config.to_data() == data
        path = tmp_path / "nested" / "config.json"
        config.write_json(str(path))
        assert cfg.make_config(json.loads(path.read_text())) == config
    config = cfg.make_config(stock())
    assert str(config.scenario_config.scenario) == "pedestrians" and config.tester_config.agent is cfg.AgentType.RANDOM_CONSTRAINED
    assert config.terminate_collisions is cfg.CollisionType.EGO and config.mode_config.mode is cfg.Mode.HEADLESS


@pytest.mark.parametrize("changes, message", [
    ({"episodes": 0}, "must be > 0"), ({"max_timesteps": 0}, "must be > 0"), ({"seed": -1}, "seed must be >= 0"),
    ({"tester_config": {"option": "random-constrained", "epsilon": 1.5}}, "epsilon must be in [0, 1]"),
    ({"tester_config": {"option": "proximity", "threshold": 0.0}}, "threshold must be >= 0"),
    ({"scenario_config": {"option": "pedestrians", "num_pedestrians": -1, "outbound_pavement": 1.0, "inbound_pavement": 1.0}}, "num_pedestrians must be >= 0"),
    ({"scenario_config": {"option": "pedestrians", "num_pedestrians": 1, "outbound_pavement": 1.5, "inbound_pavement": 1.0}}, "outbound_pavement must be in [0,1]"),
    ({"scenario_config": {"option": "bus-stop", "lanes": 3}}, "unexpected parameters"),
    ({"mode_config": {"option": "render", "episode_condition": 0, "video_dir": None}}, "episode_condition must be >= 1"),
    ({"ego_config": dict(Q_LEARNING, alpha={"start": 0.1, "stop": 0.5, "num_steps": 10})}, "start must be greater than stop"),
])
def test_value_checks_raise_value_error(changes, message):
    with pytest.raises(ValueError, match=message.replace("[", r"\[").replace("]", r"\]")):
        cfg.make_config(stock(**changes))


def test_unknown_options_and_types():
    with pytest.raises(NotImplementedError):
        cfg.make_config(stock(scenario_config={"option": "roundabout"}))
    with pytest.raises(NotImplementedError):
        cfg.make_config(stock(ego_config={"option": "random-constrained", "epsilon": 0.1}))   # not an ego option
    with pytest.raises(ValueError):
        cfg.make_config(stock(terminate_collisions="some"))
    with pytest.raises(TypeError):
        cfg.make_config(stock(tester_config={"option": "random", "epsilon": "high"}))


def test_agent_specs_follow_the_reference_compatibility_rules():
    from cavgym_b200.examples.environments import bus_stop, pedestrians, pelican_crossing
    import numpy as np
    peds = pedestrians.make_bodies(3, 1.0, 1.0, np_random=np.random.RandomState(0))
    specs = cfg.make_config(stock()).agent_specs(peds)
    assert [s.kind for s in specs] == ["noop", "random-constrained", "random-constrained", "random-constrained"]
    assert specs[1].epsilon == 0.01
    specs = cfg.make_config(stock(ego_config={"option": "random", "epsilon": 0.3}, tester_config={"option": "proximity", "threshold": 99.0})).agent_specs(peds)
    assert [s.kind for s in specs] == ["random", "proximity", "proximity", "proximity"] and specs[2].threshold == 99.0
    # crossing agents cannot drive cars / buses / traffic lights (reference config.py:358-396)
    with pytest.raises(NotImplementedError):
        cfg.make_config(stock(scenario_config={"option": "bus-stop"})).agent_specs(bus_stop.make_bodies())
    specs = cfg.make_config(stock(scenario_config={"option": "pelican-crossing"}, tester_config={"option": "random", "epsilon": 0.1})).agent_specs(pelican_crossing.make_bodies())
    assert all(s.kind == "random" for s in specs[1:])
    render = {"option": "render", "episode_condition": 1, "video_dir": None}
    specs = cfg.make_config(stock(ego_config=Q_LEARNING, mode_config=render)).agent_specs(peds)
    assert specs[0].kind == "external"       # the tensor-API learner supplies the ego's action; testers stay on the device
    with pytest.raises(NotImplementedError, match="no on-device form"):
        cfg.make_config(stock(ego_config={"option": "keyboard"}, mode_config=render)).agent_specs(peds)
    specs = cfg.make_config(stock(tester_config={"option": "election", "threshold": 5.0})).agent_specs(peds)
    assert [s.kind for s in specs] == ["noop", "election", "election", "election"] and specs[1].threshold == 5.0


def test_package_level_names_resolve():
    import cavgym_b200
    assert cavgym_b200.Config is cfg.Config and cavgym_b200.make_config is cfg.make_config
    assert callable(cavgym_b200.make) and "Pedestrians-v0" in cavgym_b200.examples.registered()


@pytest.mark.parametrize("scenario,extra", [("pedestrians", {"num_pedestrians": 3}), ("crossroads", {}), ("bus-stop", {}),
                                            ("pelican-crossing", {})])
def test_reference_objects_compile_to_the_same_tables(scenario, extra):
    """compile_scenario reads reference-style objects by protocol (class names, attributes): this repo's mirrors of the
    modules behind the reference's Config.setup (library/environment.py:59-101, examples/environments/*.py) compile to the
    byte-identical CavScenario tables recorded for the UNMODIFIED reference's own objects (tests/golden/scenario_tables.npz,
    oracle/gen_tables_golden.py)."""
    import copy
    from helpers import load_scenario_tables
    from oracle import refload
    from cavgym_b200.scenario import AgentSpec, compile_scenario
    data = refload.stock_config_dict(scenario=scenario, tester="random", seed=5, collisions="all", offroad=True, **extra)
    mine_config = cfg.make_config(copy.deepcopy(data))
    _, my_env, _, _ = mine_config.setup()
    specs = [AgentSpec("noop")] + [AgentSpec("random", epsilon=0.01) for _ in my_env.bodies[1:]]
    mine = compile_scenario(my_env.bodies, my_env.constants, mine_config, specs).tables()
    assert mine == load_scenario_tables(scenario)


def test_experiments_grid_configs_are_the_reference_grid():
    """cavgym_b200.experiments builds, per grid point, the config the reference's experiments.py:40-82 builds (same scenario,
    rewards, feature set and tester settings), with a constant learning rate where the reference passes a float."""
    from cavgym_b200 import experiments
    from cavgym_b200.config import AgentType
    log_dir, config = experiments.make_config(AgentType.PROXIMITY, 0.5, 0.9, 0.1, log_root="out")
    assert log_dir == "out/tester=proximity/alpha=0.5/gamma=0.9/epsilon=0.1"
    data = config.to_data()
    assert data["ego_config"]["option"] == "q-learning" and data["ego_config"]["alpha"] == {"start": 0.5, "stop": 0.5, "num_steps": 2}
    assert data["ego_config"]["gamma"] == 0.9 and data["ego_config"]["epsilon"] == 0.1
    assert data["ego_config"]["feature_config"] == {"distance_x": False, "distance_y": False, "distance": True, "relative_angle": True,
                                                    "heading": True, "on_road": False, "inverse_distance": False}
    assert data["tester_config"] == {"option": "proximity", "threshold": 544.0}
    assert data["scenario_config"]["num_pedestrians"] == 1 and data["episodes"] == 10 and data["seed"] == 0
    assert cfg.make_config(data).to_data() == data            # round trip
    assert experiments.make_tester_config(AgentType.RANDOM).epsilon == 0.01
    assert experiments.make_tester_config(AgentType.RANDOM_CONSTRAINED).epsilon == 0.5
    assert len(experiments.ALPHAS) * len(experiments.GAMMAS) * len(experiments.EPSILONS) * len(experiments.TESTER_TYPES) == 81
