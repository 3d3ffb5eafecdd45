"""Shared test utilities: golden fixtures and scenario construction from their metadata."""
import json
import math
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


# ------------------------------------------------------------------ the (body count, scenario family) matrix
def random_actions(rng, t_len, n, is_car):
    """Valid joint actions [T, M, 2, N]: cars brake / accelerate and steer a little, pedestrians wander."""
    m = len(is_car)
    car = np.asarray(is_car, dtype=bool)[None, :, None]
    actions = np.zeros((t_len, m, 2, n))
    hold = rng.random((t_len, m, n)) < 0.1
    throttle = rng.uniform(-140.0, 140.0, (t_len, m, n))
    steer_car = rng.uniform(-0.3, 0.3, (t_len, m, n))
    steer_ped = rng.uniform(-0.4 * np.pi, 0.4 * np.pi, (t_len, m, n))
    actions[:, :, 0] = np.where(hold & car, throttle, 0.0)
    actions[:, :, 1] = np.where(car, np.where(hold, steer_car, 0.0), np.where(rng.random((t_len, m, n)) < 0.3, steer_ped, 0.0))
    return actions


def check_against_oracle(got, want, dtype):
    """Trajectories [T, ...]: events identical off flagged steps; state / rewards compared up to the first flagged
    divergence of each env."""
    want_state, want_reward, want_done, want_winner, _ = want
    tangent = got["tangent"].astype(bool)
    mismatch = (got["done"] != want_done) | (got["winner"] != want_winner)
    assert not np.any(mismatch & ~tangent), f"unflagged event mismatch at {np.argwhere(mismatch & ~tangent)[:5]}"
    t_len, n = mismatch.shape
    err = state_err if dtype == "float64" else state_err_trajectory
    worst = 0.0
    for e in range(n):
        stop = int(np.nonzero(mismatch[:, e])[0][0]) if mismatch[:, e].any() else t_len
        worst = max(worst, err(np.moveaxis(got["state"][:stop, :, :, e], 2, -1), np.moveaxis(want_state[:stop, :, :, e], 2, -1)))
        assert rel_err(got["reward"][:stop, :, e], want_reward[:stop, :, e]) < (1e-9 if dtype == "float64" else 2e-3)
    assert worst < (1e-9 if dtype == "float64" else 1e-4), worst
    return int(want_done.any(axis=0).sum())


def custom_road_frames(snap):
    """(rear centre, orientation, length) of the roads of the custom-road scenario: the stock major road, one minor road
    rotated by 30 degrees, and two minor roads turned off the vertical by the angle that moves their far corners 0.5 and 2
    times `snap` (the axis snap, tau / 1000, engine.cu::convert) off their bounding box.  Every road is two lanes of 58.4 px."""
    return [((0.0, 0.0), 0.0, 1584.0), ((300.0, 58.4), math.pi / 6, 400.0),
            ((800.0, 58.4), math.pi / 2 + math.asin(0.5 * snap / 300.0), 300.0),
            ((1200.0, -58.4), -math.pi / 2 + math.asin(2.0 * snap / 300.0), 300.0)]


def custom_road_map(snap):
    from cavgym_b200.library import geometry
    from cavgym_b200.library.assets import Road, RoadConstants, RoadMap
    roads = [Road(RoadConstants(length=length, num_outbound_lanes=1, num_inbound_lanes=1, lane_width=58.4,
                                position=geometry.Point(*origin), orientation=phi)) for origin, phi, length in custom_road_frames(snap)]
    return RoadMap(major_road=roads[0], minor_roads=roads[1:])


MATRIX_M = tuple(range(1, 9))
FAMILIES = ("homogeneous", "generic")
TAU = {"float64": 1e-7, "float32": 5e-2}


def matrix_scenario(m, family, mode, max_timesteps=60):
    """One cell of the (body count, family) matrix of the thread-per-env kernels, M = 1..8.

    homogeneous: Pedestrians-v0, the ego and m - 1 spawned pedestrians (every road an axis-aligned rectangle, every body
                 after the ego a dynamic pedestrian: the GENERIC = false instantiations);
    generic:     the custom road map (the same major road, and minor roads that are not axis-aligned: one rotated by 30
                 degrees, two skewed off the vertical) with, for m >= 2, body 1 an oncoming car in the inbound lane, then
                 m - 2 pedestrians.  The car alone already makes the scenario generic, but the GENERIC = false kernels give
                 the same answers for it; bodies on the rotated roads are what only the generic kernels get right.
    mode 'external' replays joint actions; 'device' drives the ego with a noop agent (a RandomAgent when it is alone, so
    that envs differ), the car with a RandomAgent and the pedestrians with RandomConstrained agents.  `is_car` marks the
    bodies that take car actions."""
    from cavgym_b200.examples.environments import pedestrians as mod
    from cavgym_b200.examples.constants import car_constants
    from cavgym_b200.library.bodies import Car, DynamicBodyState
    assert m in MATRIX_M and family in FAMILIES
    constants = mod.env_constants
    car = family == "generic" and m >= 2
    bodies = mod.make_bodies(m - 1 - car, 1.0, 1.0, np_random=np.random.RandomState(0))
    if car:
        lane = mod.major_road.inbound.lanes[0]
        bodies.insert(1, Car(DynamicBodyState(lane.spawn, car_constants.max_velocity / 2, mod.major_road.inbound.orientation),
                             car_constants))
    if family == "generic":
        constants = SimpleNamespace(viewer_width=mod.env_constants.viewer_width, road_map=custom_road_map(TAU["float64"] * 1e-3))
    is_car = np.array([b == 0 or (car and b == 1) for b in range(m)])
    if mode == "external":
        specs = [AgentSpec("external") for _ in bodies]
    else:
        specs = [AgentSpec("random", epsilon=0.05) if m == 1 else AgentSpec("noop")]
        specs += [AgentSpec("random", epsilon=0.05) if is_car[b] else AgentSpec("random-constrained", epsilon=0.5) for b in range(1, m)]
    config = SimpleNamespace(terminate_collisions="ego", terminate_ego_zones=True, terminate_ego_offroad=False,
                             max_timesteps=max_timesteps, reward_win=6000.0, reward_draw=2000.0, cost_step=4.0)
    comp = compile_scenario(bodies, constants, config, specs)
    comp.is_car = is_car
    return comp


def expect_homogeneous(compiled, dtype="float64"):
    """engine.cu::convert's rule, restated on the compiled tables: at most CAV_SMALL_M bodies, every road an axis-aligned
    rectangle (every corner within tau / 1000 of its bounding box, in the engine's precision), every body dynamic and every
    body after the ego a pedestrian."""
    from cavgym_b200 import _abi
    s = compiled.struct
    if s.n_bodies > _abi.CAV_SMALL_M:
        return False
    to = np.float64 if dtype == "float64" else np.float32
    snap = float(to(TAU[dtype] * 1e-3))
    for r in range(s.n_roads):
        xs = [float(to(s.roads[r].x[i])) for i in range(4)]
        ys = [float(to(s.roads[r].y[i])) for i in range(4)]
        for vs in (xs, ys):
            lo, hi = min(vs), max(vs)
            if any(min(abs(v - lo), abs(v - hi)) > snap for v in vs) or not hi > lo:
                return False
    for b in range(s.n_bodies):
        if s.bodies[b].kind != _abi.CAV_BODY_DYNAMIC or (b > 0 and not s.bodies[b].flags & _abi.CAV_FLAG_PEDESTRIAN):
            return False
    return True


def has_pedestrian(m, family):
    """Whether the matrix cell (m, family) holds a pedestrian (the danger of the parking rollout needs one)."""
    return m - 1 - (family == "generic" and m >= 2) > 0
