"""Shared test utilities: golden fixtures and scenario construction from their metadata."""
import json
import os
from types import SimpleNamespace

import numpy as np

from cavgym_b200.scenario import AgentSpec, compile_scenario

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_CASES = sorted(f[:-4] for f in os.listdir(GOLDEN_DIR)
                      if f.endswith(".npz") and f not in ("geometry_kat.npz", "scenario_tables.npz") and not f.startswith(("info_", "learn_")))
LEARN_CASES = sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.startswith("learn_") and f.endswith(".npz"))   # oracle/gen_learning_golden.py


def load_golden(name):
    data = np.load(os.path.join(GOLDEN_DIR, f"{name}.npz"))
    meta = json.loads(bytes(data["meta"]).decode())
    episodes = []
    for e in range(int(data["n_episodes"])):
        prefix = f"ep{e}_"
        episodes.append({k[len(prefix):]: data[k] for k in data.files if k.startswith(prefix)})
    return meta, episodes


INFO_CASES = sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.startswith("info_") and f.endswith(".npz"))


def load_info_golden(name):
    """(meta, state [T, M, 4], body_polygons [T, M, 8], road_angles [T, M]) recorded from the reference's env.info()."""
    data = np.load(os.path.join(GOLDEN_DIR, f"{name}.npz"))
    return json.loads(bytes(data["meta"]).decode()), data["state"], data["body_polygons"], data["road_angles"]


def load_scenario_tables(name):
    """CompiledScenario.tables() recorded for the reference's objects of one stock scenario (oracle/gen_tables_golden.py)."""
    data = np.load(os.path.join(GOLDEN_DIR, "scenario_tables.npz"))
    return {part: data[f"{name}/{part}"].tobytes() for part in ("header", "bodies", "spawns")}


def env_config_from(cfg):
    return SimpleNamespace(**{k: cfg[k] for k in ("terminate_collisions", "terminate_ego_zones", "terminate_ego_offroad",
                                                 "max_timesteps", "reward_win", "reward_draw", "cost_step")})


def bodies_and_constants(cfg):
    option = cfg["scenario_config"]["option"]
    if option == "pedestrians":
        from cavgym_b200.examples.environments import pedestrians as mod
        sc = cfg["scenario_config"]
        bodies = mod.make_bodies(sc["num_pedestrians"], sc["outbound_pavement"], sc["inbound_pavement"],
                                 np_random=np.random.RandomState(0))
    elif option == "crossroads":
        from cavgym_b200.examples.environments import crossroads as mod
        bodies = mod.make_bodies()
    elif option == "bus-stop":
        from cavgym_b200.examples.environments import bus_stop as mod
        bodies = mod.make_bodies()
    elif option == "pelican-crossing":
        from cavgym_b200.examples.environments import pelican_crossing as mod
        bodies = mod.make_bodies()
    else:
        raise KeyError(option)
    return bodies, mod.env_constants


def agent_specs(cfg, bodies, mode):
    """mode 'external': replayed joint actions.  mode 'device': the on-device agents Config.setup would build."""
    if mode == "external":
        return [AgentSpec("external") for _ in bodies]
    ego = cfg["ego_config"]
    tester = cfg["tester_config"]
    specs = [AgentSpec(ego["option"], epsilon=ego.get("epsilon", 0.0))]
    for _ in bodies[1:]:
        specs.append(AgentSpec(tester["option"], epsilon=tester.get("epsilon", 0.0), threshold=tester.get("threshold", 0.0)))
    return specs


def compile_from_meta(meta, mode="external"):
    cfg = meta["config"]
    bodies, constants = bodies_and_constants(cfg)
    return compile_scenario(bodies, constants, env_config_from(cfg), agent_specs(cfg, bodies, mode))


def soa(per_env):
    """[N][M][C] -> [M][C][N] contiguous."""
    return np.ascontiguousarray(np.transpose(np.asarray(per_env), (1, 2, 0)))


def rel_err(got, want):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    return float(np.max(np.abs(got - want) / np.maximum(1.0, np.abs(want)))) if got.size else 0.0


def state_err(got, want, dynamic=None):
    """Relative error of body state [..., M, 4] (component axis last): position as a vector,
    |dp| / max(1, |p|) (a coordinate that crosses zero has no meaningful scalar relative error), velocity
    |dv| / max(1, |v|), orientation as an angle modulo 2*pi — atan2(sin(t), cos(t)) may land on +pi in one
    libm and -pi in another for the same heading."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    if not got.size:
        return 0.0
    pos = np.hypot(got[..., 0] - want[..., 0], got[..., 1] - want[..., 1]) / np.maximum(1.0, np.hypot(want[..., 0], want[..., 1]))
    vel = np.abs(got[..., 2] - want[..., 2]) / np.maximum(1.0, np.abs(want[..., 2]))
    d = got[..., 3] - want[..., 3]
    plain = np.abs(d) / np.maximum(1.0, np.abs(want[..., 3]))
    ang = np.minimum(plain, np.abs(np.arctan2(np.sin(d), np.cos(d))) / np.maximum(1.0, np.abs(want[..., 3])))
    return float(max(pos.max(), vel.max(), ang.max()))


def state_err_trajectory(got, want):
    """state_err for a whole trajectory [T, M, 4] of an integration carried in float32: the position error is taken
    relative to the largest |position| the body has reached SO FAR in the episode (running maximum along T) instead of
    its current |position| (likewise the velocity, a running sum of throttle * dt).  A float32 coordinate is quantised relative to its magnitude when it is stored, so what an
    fp32 integration can preserve is digits of the trajectory's scale; dividing by the instantaneous |p| would demand
    absolute accuracy far below one ulp of the values that were summed whenever a body passes near the origin."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    if not got.size:
        return 0.0
    scale = np.maximum(1.0, np.maximum.accumulate(np.hypot(want[..., 0], want[..., 1]), axis=0))
    pos = np.hypot(got[..., 0] - want[..., 0], got[..., 1] - want[..., 1]) / scale
    vel = np.abs(got[..., 2] - want[..., 2]) / np.maximum(1.0, np.maximum.accumulate(np.abs(want[..., 2]), axis=0))
    d = got[..., 3] - want[..., 3]
    ang = np.abs(np.arctan2(np.sin(d), np.cos(d))) / np.maximum(1.0, np.abs(want[..., 3]))
    return float(max(pos.max(), vel.max(), ang.max()))
