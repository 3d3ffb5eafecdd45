"""Generate tests/golden/scenario_tables.npz: the CavScenario tables (CompiledScenario.tables(): header, body rows, spawn
rows) that the stock scenarios compile to, as tests/test_config.py and tests/test_integration_binding.py compile them.

    python -m oracle.gen_tables_golden                        # record from this repository's mirrors of the reference modules
    python -m oracle.gen_tables_golden --check                # compile again and compare with the committed file
    python -m oracle.gen_tables_golden --reference --check    # compile the UNMODIFIED reference's own objects (oracle/refload.py)

The committed file was recorded from the mirrors (cavgym_b200.config / library / examples), whose tables had been checked
byte-identical to the ones the reference's own Config.setup objects compile to; `--reference --check` repeats that
comparison wherever the reference tree is available.
"""
import argparse
import copy
import os
import sys

import numpy as np

from . import refload

GOLDEN_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "scenario_tables.npz")
PARTS = ("header", "bodies", "spawns")
# case -> (refload.stock_config_dict kwargs, how the tables are compiled)
CASES = {
    # tests/test_config.py::test_reference_objects_compile_to_the_same_tables: noop ego, random testers, the Config as env_config
    "pedestrians": (dict(scenario="pedestrians", tester="random", seed=5, collisions="all", offroad=True, num_pedestrians=3), "config"),
    "crossroads": (dict(scenario="crossroads", tester="random", seed=5, collisions="all", offroad=True), "config"),
    "bus-stop": (dict(scenario="bus-stop", tester="random", seed=5, collisions="all", offroad=True), "config"),
    "pelican-crossing": (dict(scenario="pelican-crossing", tester="random", seed=5, collisions="all", offroad=True), "config"),
    # tests/test_integration_binding.py: what integration/batched.py compiles from an env (external agents, env.env_config)
    "binding_pelican-crossing": (dict(scenario="pelican-crossing", tester="random", seed=3, collisions="all"), "binding"),
}


def compile_case(name, make_config):
    from cavgym_b200.scenario import AgentSpec, compile_scenario
    kwargs, how = CASES[name]
    config = make_config(copy.deepcopy(refload.stock_config_dict(**kwargs)))
    _, env, _, _ = config.setup()
    if how == "binding":
        return compile_scenario(env.bodies, env.constants, env.env_config, [AgentSpec("external") for _ in env.bodies],
                                time_resolution=env.time_resolution).tables()
    specs = [AgentSpec("noop")] + [AgentSpec("random", epsilon=0.01) for _ in env.bodies[1:]]
    return compile_scenario(env.bodies, env.constants, config, specs).tables()


def main(argv=None):
    parser = argparse.ArgumentParser()
    parser.add_argument("--check", action="store_true")
    parser.add_argument("--reference", action="store_true", help="compile the reference's own objects instead of the mirrors")
    args = parser.parse_args(argv)
    if args.reference:
        make_config = refload.load()["config"].make_config
    else:
        from cavgym_b200.config import make_config
    payload = {}
    for name in CASES:
        for part, data in compile_case(name, make_config).items():
            payload[f"{name}/{part}"] = np.frombuffer(data, dtype=np.uint8)
    if not args.check:
        np.savez_compressed(GOLDEN_PATH, **payload)
        print(f"wrote {GOLDEN_PATH} ({os.path.getsize(GOLDEN_PATH) / 1024:.0f} KiB)")
        return 0
    old = dict(np.load(GOLDEN_PATH))
    failures = 0
    for name in CASES:
        ok = all(np.array_equal(old.get(f"{name}/{part}"), payload[f"{name}/{part}"]) for part in PARTS)
        failures += not ok
        print(("OK   " if ok else "DIFF ") + name)
    return 1 if failures else 0


if __name__ == "__main__":
    sys.exit(main())
