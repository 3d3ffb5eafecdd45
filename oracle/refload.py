"""Import the CAV-Gym reference VERBATIM from /root/reference with stand-ins for
its un-vendored dependencies.  TEST INFRASTRUCTURE ONLY — build container only.

The reference is not part of this repository, so nothing under tests/ (gpu or
not), bench.py or __graft_entry__.smoke() may call load(): it is used by
oracle/gen_*golden.py to produce the fixtures in tests/golden/, which the
tests compare with.

Stand-ins (oracle/standins/): gym 0.17.2 subset, shapely.geometry subset (exact
convex predicates), enforce_typing (identity), and `np.float = float` because
library/bodies.py:99-108 uses the alias numpy removed in 1.24.
"""
import os
import sys

REFERENCE_ROOT = os.environ.get("CAVGYM_REFERENCE", "/root/reference")
_STANDINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "standins")


def available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "library", "environment.py"))


def load():
    """Put the stand-ins and the reference on sys.path and return its key modules."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    import numpy as np
    if not hasattr(np, "float"):
        np.float = float  # bodies.py:99-108
    for path in (REFERENCE_ROOT, _STANDINS):
        if path not in sys.path:
            sys.path.insert(0, path)
    import config
    import reporting
    import simulation
    import examples  # registers the four env ids
    import library.bodies
    import library.environment
    import library.geometry
    import library.assets
    import examples.agents.pedestrian
    import examples.agents.dynamic_body
    import examples.agents.template
    return {
        "config": config,
        "reporting": reporting,
        "simulation": simulation,
        "examples": examples,
        "bodies": library.bodies,
        "environment": library.environment,
        "geometry": library.geometry,
        "assets": library.assets,
        "pedestrian_agents": examples.agents.pedestrian,
        "dynamic_body_agents": examples.agents.dynamic_body,
        "template_agents": examples.agents.template,
    }


def stock_config_dict(scenario="pedestrians", tester="random-constrained", epsilon=0.01, seed=0,
                      episodes=1, collisions="ego", zones=True, offroad=False, threshold=None,
                      num_pedestrians=1, ego="noop", ego_epsilon=0.01, max_timesteps=1000):
    """config.json (config.json:1-49) with ego->noop and mode->headless, as BASELINE C1 states."""
    scenario_config = {"option": scenario}
    if scenario == "pedestrians":
        scenario_config.update(num_pedestrians=num_pedestrians, outbound_pavement=1.0, inbound_pavement=1.0)
    tester_config = {"option": tester}
    if tester in ("random", "random-constrained"):
        tester_config["epsilon"] = epsilon
    if tester in ("proximity", "election"):
        tester_config["threshold"] = float(threshold)
    ego_config = {"option": ego}
    if ego == "random":
        ego_config["epsilon"] = ego_epsilon
    return {
        "verbosity": "silent",
        "episode_log": None,
        "run_log": None,
        "seed": seed,
        "episodes": episodes,
        "max_timesteps": max_timesteps,
        "terminate_collisions": collisions,
        "terminate_ego_zones": zones,
        "terminate_ego_offroad": offroad,
        "reward_win": 6000.0,
        "reward_draw": 2000.0,
        "cost_step": 4.0,
        "scenario_config": scenario_config,
        "ego_config": ego_config,
        "tester_config": tester_config,
        "mode_config": {"option": "headless"},
    }
