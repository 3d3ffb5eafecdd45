"""The near-tangent contract, checked against exact arithmetic on every kernel path.

Every parity test of this repository compares events only off flagged steps.  That is sound only if

    a decision of a step (finish line, all-pairs and static collisions, off-road, ego collision, braking zone, reaction zone,
    liveness p > 0.5) may differ from the exact one only when the engine raises its near-tangent flag for that env-step,

and useful only if the flag is not raised without a cause.  Here a placement generator puts bodies at controlled distances
(multiples of tau) from every decision boundary and on every branch of `road_share` (one kerb, kerb touch, road corner:
axis-aligned shortcut, wedge, clipper, apart), each env of a batch one configuration stepped once with zero actions.  The
exact truth (tests/exact_geometry.py, rational arithmetic) is computed on the post-step state the engine returns, and every
kernel path (TMA / plain step, replay T = 1 and 3, warp-per-env, the thread-per-env rollout) must agree bitwise and
meet, in fp64 and fp32:
  soundness    a decision that differs from the exact one is flagged;
  sensitivity  a consulted margin with |m| <= tau/2, or a share with |p - 0.5| <= tau/2, is flagged;
  specificity  a flagged env has a consulted margin, a road-edge margin of a share, or the share of some road within 2 tau
               of 0.5;
  shares       p recovered from the reward is within a bound derived per branch (`share_bound`).
The CPU checks hold the exact reference to the reference's own known answers and the C oracle to the same contract.
"""
import math
from fractions import Fraction as F
from types import SimpleNamespace

import numpy as np
import pytest

import exact_geometry as xg
from helpers import GOLDEN_DIR, custom_road_frames, custom_road_map
from cavgym_b200 import _abi

TAU = {"float64": 1e-7, "float32": 5e-2}
AXIS_SHORTCUT = {"float64": 1e-9, "float32": 1e-5}     # corner_share_closed: min(|c|, |s|) below this is axis-aligned
EPS = {"float64": 2.0 ** -53, "float32": 2.0 ** -24}
KS = (-3.0, -1.0, -0.5, -0.125, 0.0, 0.125, 0.5, 1.0, 3.0)
DELTAS = (1e-12, 1e-10, 0.9e-9, 1.1e-9, 1e-7, 0.9e-5, 1.1e-5)
DT = 1.0 / 60


# ================================================================================================ scenarios
def env_config(collisions, offroad=False, zones=True):
    return SimpleNamespace(terminate_collisions=collisions, terminate_ego_zones=zones, terminate_ego_offroad=offroad,
                           max_timesteps=1000, reward_win=6000.0, reward_draw=2000.0, cost_step=4.0)


class QuadObstacle:
    """A road_map.obstacle that is not a rectangle: anything with bounding_box() -> four corners compiles."""

    def __init__(self, corners):
        self.corners = corners

    def bounding_box(self):
        return self.corners


# a convex quadrilateral with no right angle, on the stock pedestrians road
OBSTACLE = [(560.0, 20.0), (645.0, 34.0), (652.0, -27.0), (571.0, -41.0)]


def compile_category(cat, agents, dtype="float64"):
    from cavgym_b200.scenario import AgentSpec, compile_scenario
    if cat.scenario in ("pedestrians", "obstacle", "custom-roads"):
        from cavgym_b200.examples.environments import pedestrians as mod
        bodies = mod.make_bodies(cat.m - 1, 1.0, 1.0, np_random=np.random.RandomState(0))
    elif cat.scenario == "bus-stop":
        from cavgym_b200.examples.environments import bus_stop as mod
        bodies = mod.make_bodies()
    elif cat.scenario == "pelican":
        from cavgym_b200.examples.environments import pelican_crossing as mod
        bodies = mod.make_bodies()
    else:
        from cavgym_b200.examples.environments import crossroads as mod
        bodies = mod.make_bodies()
    constants = mod.env_constants
    if cat.scenario == "obstacle":
        from cavgym_b200.library.assets import RoadMap
        road_map = RoadMap(major_road=mod.road_map.major_road)
        road_map.set_obstacle(QuadObstacle(OBSTACLE))
        constants = SimpleNamespace(viewer_width=mod.env_constants.viewer_width, road_map=road_map)
    elif cat.scenario == "custom-roads":
        constants = SimpleNamespace(viewer_width=mod.env_constants.viewer_width, road_map=custom_road_map(TAU[dtype] * 1e-3))
    specs = [AgentSpec(agents) for _ in bodies]
    return compile_scenario(bodies, constants, env_config(cat.collisions, cat.offroad), specs)


class Desc:
    """What the exact cascade needs from the compiled scenario tables."""

    def __init__(self, comp, dtype="float64"):
        s = comp.struct
        self.m, self.W = s.n_bodies, s.viewer_width
        self.collisions, self.offroad, self.zones = s.terminate_collisions, bool(s.terminate_ego_offroad), bool(s.terminate_ego_zones)
        self.dims, self.ped, self.pelican = [], [], []
        for b in range(self.m):
            t = s.types[s.bodies[b].type_id]
            self.dims.append((t.length, t.width, t.min_throttle))
            self.ped.append(bool(s.bodies[b].flags & _abi.CAV_FLAG_PEDESTRIAN))
            self.pelican.append(s.bodies[b].kind == _abi.CAV_BODY_PELICAN)
        self.roads = [xg.quad([(s.roads[r].x[i], s.roads[r].y[i]) for i in range(4)]) for r in range(s.n_roads)]
        self.statics = [xg.quad([(s.statics[r].x[i], s.statics[r].y[i]) for i in range(4)]) for r in range(s.n_statics)]
        # a traffic light's share of the road is a constant of the scenario (environment.py:141), never flagged
        self.static_share = [max(xg.share(xg.quad([(s.bodies[b].static_box.x[i], s.bodies[b].static_box.y[i]) for i in range(4)]), q)
                                 for q in self.roads) if self.pelican[b] else None for b in range(self.m)]
        # engine.cu::convert: a road is axis-aligned when every corner, in the engine's precision, lies within tau / 1000 of
        # its bounding box; `skew` is how far the real corners are from the box the closed forms then use
        R = np.float64 if dtype == "float64" else np.float32
        snap = float(R(TAU[dtype] * 1e-3))
        self.road_axis, self.road_skew = [], []
        for r in range(s.n_roads):
            xs = [float(R(s.roads[r].x[i])) for i in range(4)]
            ys = [float(R(s.roads[r].y[i])) for i in range(4)]
            on = lambda v, lo, hi: min(abs(v - lo), abs(v - hi))
            dev = max(max(on(x, min(xs), max(xs)), on(y, min(ys), max(ys))) for x, y in zip(xs, ys))
            self.road_axis.append(dev <= snap)
            exact = [max(on(x, min(xs), max(xs)), on(y, min(ys), max(ys)))
                     for x, y in zip((s.roads[r].x[i] for i in range(4)), (s.roads[r].y[i] for i in range(4)))]
            self.road_skew.append(max(exact) + max(abs(float(R(s.roads[r].x[i])) - s.roads[r].x[i]) +
                                                   abs(float(R(s.roads[r].y[i])) - s.roads[r].y[i]) for i in range(4)))


# ================================================================================================ exact truth
def road_branch(box, road, c, s, hl, hw, tau, shortcut):
    """Which case of road_share (transition.cuh) this box takes on an axis-aligned road, from the exact geometry."""
    x0, x1, y0, y1 = xg.aabb(road)
    bx0, bx1, by0, by1 = xg.aabb(box)
    ex, ey = (bx1 - bx0) / 2, (by1 - by0) / 2
    m0, m1, m2, m3 = bx0 - x0, x1 - bx1, by0 - y0, y1 - by1
    mx, my = min(m0, m1), min(m2, m3)
    if mx < -(2 * ex + tau) or my < -(2 * ey + tau):
        return "zero"
    lo, hi = (mx, my) if mx < my else (my, mx)
    opposite = max(m0, m1) if mx < my else max(m2, m3)
    if lo >= tau:
        return "one"
    if lo > -tau and hi >= tau and opposite >= tau:
        return "touch"
    if lo <= -tau and hi >= tau and opposite >= tau:
        return "kerb"
    if not (mx < tau and my < tau and max(m0, m1) >= tau and max(m2, m3) >= tau):
        return "general"
    tx, ty = mx + ex, my + ey
    if not (ex - tx > 0 and ey - ty > 0):
        return "corner_open"             # the box does not reach into the quadrant outside both edges
    if min(abs(c), abs(s)) < shortcut:
        return "corner_axis"
    sx, sy = (-1 if m0 < m1 else 1), (-1 if m2 < m3 else 1)
    ux, uy, vx, vy = sx * c, sy * s, -(sx * s), sy * c
    pu, pv = ux * tx + uy * ty, vx * tx + vy * ty
    apart = ((ux >= 0 and uy >= 0 and pu >= hl + tau) or (ux <= 0 and uy <= 0 and -pu >= hl + tau) or
             (vx >= 0 and vy >= 0 and pv >= hw + tau) or (vx <= 0 and vy <= 0 and -pv >= hw + tau))
    if apart:
        return "corner_apart"
    return "corner_wedge" if abs(pu) < hl and abs(pv) < hw else "corner_clip"


def share_bound(label, dtype, x, y, c, s, length, width):
    """How far the engine's share may be from the exact one on each branch (derived from geometry.cuh):
      * kerb_share, kerb_touch_share, wedge_in_box_area work on box-relative distances: their inputs carry the rounding of
        the absolute position, ~eps * |x|, which moves the share by at most that over the smaller side;
      * corner_share / clip_area take shoelace sums of absolute coordinates: ~16 eps |x| |y| / (L W) (8 vertices, two
        products per term, plus the rounding of the clipped vertices);
      * the near-axis shortcut of corner_share_closed replaces box ∩ quadrant by its bounding rectangle: the two slivers
        it adds are at most delta (L^2 + W^2) / 2 with delta = min(|c|, |s|), over the box area L W.
    fp64 (eps = 2^-53): 1e-12 on the relative branches, ~1e-11 on the clipper near x = 1584; fp32 (eps = 2^-24): ~1e-4,
    below the 2e-3 the trace tests allow."""
    eps = EPS[dtype]
    ax, ay = abs(x) + (length + width), abs(y) + (length + width)
    relative = max(1e-12 if dtype == "float64" else 0.0, 8 * eps * max(ax, ay) / min(length, width))
    if label in ("zero", "one"):
        return 4 * eps
    if label == "corner_axis":
        return min(abs(c), abs(s)) * (length ** 2 + width ** 2) / (2 * length * width) + relative
    if label in ("corner_clip", "general"):
        return 16 * eps * ax * ay / (length * width) + relative
    return relative


def exact_truth(desc, st, tau, dtype):
    """The step's decisions on the post-step state st [M, 4] by the exact geometry, in the order of transition_body.inc:
    finish, then all-pairs and statics, then off-road, then ego and braking, then the reaction zone (lowest index wins).
    Returns the decisions, the margins consulted (`sens`: consulted by both the reference and the engine, so a margin
    within tau/2 must be flagged; `cause`: every margin or road-edge distance the engine may flag on), the shares, and
    the road_share branch of every body."""
    tau_q = F(tau)
    m = desc.m
    boxes, trig = [], []
    for b in range(m):
        if desc.pelican[b]:
            boxes.append(None)
            trig.append(None)
            continue
        x, y, _, th = (float(v) for v in st[b])
        length, width, _ = desc.dims[b]
        boxes.append(xg.make_box(length, width, th, x, y))
        trig.append((1.0, 0.0) if th == 0.0 else (math.cos(th), math.sin(th)))
    sens, cause, statics_near = [], [], set()

    def consult(d, sensitive=True):
        cause.append(d)
        if sensitive:
            sens.append(d)
        return d.num <= 0

    def pair(a, b):   # the engine evaluates a pair only when the bounding boxes are within tau
        d = xg.sat_margin(a, b)
        return consult(d, sensitive=xg.aabb_gap(a, b) <= tau_q * F(99, 100))

    fin = xg.Axis(min(p[0] for p in boxes[0]) - xg.fx(desc.W))
    consult(fin)
    terminate = win_ego = fin.num > 0
    win = -1
    if not terminate and desc.collisions == _abi.CAV_COLLISIONS_ALL:
        hit = False
        dyn = [b for b in range(m) if not desc.pelican[b]]
        for i in dyn:
            for j in dyn:
                if j > i:
                    hit |= pair(boxes[i], boxes[j])
            for k, q in enumerate(desc.statics):
                near_before = len(sens)
                hit |= pair(boxes[i], q)
                if len(sens) > near_before and sens[-1].within(F(tau) / 2):
                    statics_near.add(k)
        terminate = hit
    if not terminate and desc.offroad:
        on = False
        for q in desc.roads:
            on |= pair(boxes[0], q)
        terminate = not on
    if not terminate and (desc.collisions == _abi.CAV_COLLISIONS_EGO or desc.zones):
        x, y, v, th = (float(val) for val in st[0])
        length, width, min_throttle = desc.dims[0]
        zones = xg.stopping_zones(x, y, v, th, length, width, min_throttle)   # zero steering: zones exist iff td != 0
        ego_mode = desc.collisions == _abi.CAV_COLLISIONS_EGO
        peds = [b for b in range(1, m) if desc.ped[b]]
        hits = {}
        for b in peds:
            h = False
            if ego_mode:
                h = consult(xg.sat_margin(boxes[b], boxes[0]))
                if not h and zones is not None:
                    h = consult(xg.sat_margin(boxes[b], zones[0]))
            hits[b] = h
        if desc.zones and zones is not None:
            reaction = {b: xg.sat_margin(boxes[b], zones[1]) for b in peds}
            any_hit = any(hits.values())
            for b in peds:
                engine_consults = not any(hits[a] for a in peds if a <= b) and win < 0
                if engine_consults or not any_hit:
                    # the reference tests reaction zones only if nothing hit at all, the engine up to the first hit: a
                    # margin both evaluate must be flagged when near, either one may raise a flag on its own
                    consult(reaction[b], sensitive=engine_consults and not any_hit)
                if not any_hit and win < 0 and reaction[b].num <= 0:
                    win = b
            terminate = any_hit or win >= 0
        else:
            terminate = any(hits.values())
    shares, labels, bounds, near_half = [], [], [], []
    for b in range(1, m):
        if desc.pelican[b]:
            shares.append(desc.static_share[b])
            labels.append(["static"])
            bounds.append(1e-12 if dtype == "float64" else 1e-5)
            continue
        length, width, _ = desc.dims[b]
        x, y, _, th = (float(v) for v in st[b])
        c, s = trig[b]
        qs, lb = [], []
        for r, road in enumerate(desc.roads):
            qs.append(xg.share(boxes[b], road))
            # the engine compares rounded margins with tau: within rounding of a branch boundary it may take either side
            fuzz = F(8 * EPS[dtype] * (abs(x) + abs(y) + length + width))
            if desc.road_axis[r]:
                branch = lambda t: road_branch(boxes[b], road, xg.fx(c), xg.fx(s), F(length) / 2, F(width) / 2, t, F(AXIS_SHORTCUT[dtype]))
                labs, lab = {branch(t) for t in (tau_q, tau_q - fuzz, tau_q + fuzz)}, branch(tau_q)
                # the closed forms work on the road's bounding box, up to `skew` away from the road itself
                skew = desc.road_skew[r] * 2 * (length + width) / (length * width)
            else:   # only the bounding-box rejection comes before the general predicates
                lab = "zero" if road_branch(boxes[b], road, xg.fx(c), xg.fx(s), F(length) / 2, F(width) / 2, tau_q,
                                            F(AXIS_SHORTCUT[dtype])) == "zero" else "general"
                labs, skew = {lab, "general"}, 0.0
            lb.append((lab, max(share_bound(v, dtype, x, y, c, s, length, width) for v in labs) + skew))
            cause.extend((xg.contains_margin(road, boxes[b]), xg.sat_margin(boxes[b], road)))
        p = max(qs)
        near_half.extend(qs)    # the engine tests |q - 0.5| on every road's share, not only on the largest
        shares.append(p)
        labels.append([lab for lab, _ in lb])
        bounds.append(max(bd for (lab, bd), q in zip(lb, qs) if abs(float(q - p)) <= 1e-6))
    winner = 0 if win_ego else (win if win >= 0 else -1)
    return SimpleNamespace(terminate=terminate, winner=winner if terminate else -1, shares=shares, labels=labels,
                           bounds=bounds, sens=sens, cause=cause, road_shares=near_half, statics_near=statics_near)


# ================================================================================================ placements
def heading(rng):
    u = rng.random()
    if u < 0.2:
        return float(rng.choice([0.0, math.pi / 2, -math.pi / 2, math.pi]))
    if u < 0.7:
        base = float(rng.choice([0.0, math.pi / 2, -math.pi / 2, math.pi]))
        return base + float(rng.choice([-1.0, 1.0])) * float(rng.choice(DELTAS))
    return float(rng.uniform(-math.pi, math.pi))


def extents(length, width, th):
    c, s = abs(math.cos(th)), abs(math.sin(th))
    return c * length / 2 + s * width / 2, s * length / 2 + c * width / 2


def margin_k(rng, tau):
    return float(rng.choice(KS)) * tau


def kerb_place(rng, dims, tau, road, xband, edge=None):
    """A body across / touching / near one kerb of the axis-aligned road (x0, x1, y0, y1)."""
    length, width = dims[:2]
    th = heading(rng)
    ex, ey = extents(length, width, th)
    x0, x1, y0, y1 = road
    edge = edge if edge is not None else int(rng.integers(0, 4))
    mode = rng.integers(0, 4)
    # signed distance of the centre from the kerb, positive inside
    e_n = ey if edge < 2 else ex
    a = max(abs(math.cos(th)) * length / 2, abs(math.sin(th)) * width / 2) if edge < 2 else \
        max(abs(math.sin(th)) * length / 2, abs(math.cos(th)) * width / 2)
    if mode == 0:     # share near 0.5 + k tau (linear part of the trapezoid CDF: dp/dt = 1 / 2A)
        t = 2 * a * margin_k(rng, tau)
    elif mode == 1:   # touching the kerb from inside: edge margin k tau
        t = e_n + margin_k(rng, tau)
    elif mode == 2:   # touching from outside
        t = -e_n - margin_k(rng, tau)
    else:
        t = rng.uniform(-20, 20)
    if edge < 2:
        x = rng.uniform(*xband)
        y = (y1 - t) if edge == 0 else (y0 + t)
    else:
        y = rng.uniform(y0 + 25, y1 - 25)
        x = (x0 + t) if edge == 2 else (x1 - t)
    return [x, y, 0.0, th]


def corner_place(rng, dims, tau, corner, outward):
    """A body on a road corner: axis-aligned (shortcut), containing the corner (wedge), reaching into the quadrant
    outside both kerbs (clipper), or clear of it by (1 + k) tau along a box axis (apart)."""
    length, width = dims[:2]
    hl, hw = length / 2, width / 2
    (cx, cy), (sx, sy) = corner, outward
    mode = rng.integers(0, 5)
    if mode == 0:
        th = float(rng.choice([math.pi / 2, -math.pi / 2, 0.0, math.pi])) + float(rng.choice([-1.0, 0.0, 1.0])) * float(rng.choice(DELTAS))
        ex, ey = extents(length, width, th)
        a = rng.uniform(0, 2 * ex) if rng.random() < 0.7 else margin_k(rng, tau)
        b = rng.uniform(0, 2 * ey) if rng.random() < 0.7 else margin_k(rng, tau)
        return [cx - sx * (ex - a), cy - sy * (ey - b), 0.0, th]
    th = heading(rng) if rng.random() < 0.3 else float(rng.uniform(-math.pi, math.pi))
    c, s = math.cos(th), math.sin(th)
    if mode == 1:     # corner inside the box: corner = centre + pu u + pv v
        pu, pv = rng.uniform(-0.95, 0.95) * hl, rng.uniform(-0.95, 0.95) * hw
        return [cx - (pu * c - pv * s), cy - (pu * s + pv * c), 0.0, th]
    if mode == 2:
        ex, ey = extents(length, width, th)
        return [cx - sx * rng.uniform(-ex, ex), cy - sy * rng.uniform(-ey, ey), 0.0, th]
    if mode == 3:     # the box axis that points into the quadrant, the box before the corner by (1 + k) tau along it
        for (ax, ay), h, (px, py), hp in (((c, s), hl, (-s, c), hw), ((-c, -s), hl, (-s, c), hw), ((-s, c), hw, (c, s), hl),
                                          ((s, -c), hw, (c, s), hl)):
            if ax * sx >= 0 and ay * sy >= 0:
                break
        d = h + tau + margin_k(rng, tau)
        t = rng.uniform(-1.5, 1.5) * hp
        return [cx - d * ax + t * px, cy - d * ay + t * py, 0.0, th]
    return [cx + rng.uniform(-20, 20), cy + rng.uniform(-20, 20), 0.0, th]


def touching(rng, a_state, a_dims, b_dims, tau):
    """Body b placed so that its separating-axis margin to body a along one of a's edge normals is k tau."""
    xa, ya, _, tha = a_state
    hla, hwa = a_dims[0] / 2, a_dims[1] / 2
    thb = heading(rng)
    ca, sa = math.cos(tha), math.sin(tha)
    side = rng.integers(0, 4)
    n, h, perp, hp = [((ca, sa), hla, (-sa, ca), hwa), ((-ca, -sa), hla, (-sa, ca), hwa),
                      ((-sa, ca), hwa, (ca, sa), hla), ((sa, -ca), hwa, (ca, sa), hla)][side]
    cb, sb = math.cos(thb), math.sin(thb)
    rb = abs(n[0] * cb + n[1] * sb) * b_dims[0] / 2 + abs(-n[0] * sb + n[1] * cb) * b_dims[1] / 2
    d = h + rb + (margin_k(rng, tau) if rng.random() < 0.8 else rng.uniform(-20, 20))
    t = rng.uniform(-0.9, 0.9) * hp
    return [xa + d * n[0] + t * perp[0], ya + d * n[1] + t * perp[1], 0.0, thb]


def road_box(desc, r=0):
    return tuple(float(v) for v in xg.aabb(desc.roads[r]))


def gen_ped_share(desc, tau, rng):
    road = road_box(desc)
    x0, x1, y0, y1 = road
    corners = [((x, y), (1 if x == x1 else -1, 1 if y == y1 else -1)) for x in (x0, x1) for y in (y0, y1)]
    ped = desc.dims[1]
    if rng.random() < 0.5:
        body = kerb_place(rng, ped, tau, road, rng.choice([(60.0, 650.0), (950.0, 1520.0)]))
    else:
        corner, out = corners[rng.integers(0, 4)]
        body = corner_place(rng, ped, tau, corner, out)
    return [[800.0, 29.2, 0.0, 0.0], body]


def gen_bus_stop(desc, tau, rng):
    """Bus and cars on the kerbs and road corners, in separate stretches of the road so that they rarely meet."""
    road = road_box(desc)
    x0, x1, y0, y1 = road
    ego = [800.0, 0.0, 0.0, 0.0]
    out = [ego, None, None, None, None]

    def corner_at(x, b):
        y = y0 if rng.random() < 0.5 else y1
        return corner_place(rng, desc.dims[b], tau, (x, y), (1 if x == x1 else -1, 1 if y == y1 else -1))

    out[1] = corner_at(x0, 1) if rng.random() < 0.5 else kerb_place(rng, desc.dims[1], tau, road, (230.0, 420.0), int(rng.integers(0, 3)))
    out[2] = corner_at(x1, 2) if rng.random() < 0.7 else kerb_place(rng, desc.dims[2], tau, road, (1150.0, 1400.0),
                                                                     int(rng.choice([0, 1, 3])))
    out[3] = kerb_place(rng, desc.dims[3], tau, road, (560.0, 680.0), int(rng.integers(0, 2)))
    out[4] = kerb_place(rng, desc.dims[4], tau, road, (930.0, 1060.0), int(rng.integers(0, 2)))
    if rng.random() < 0.25:    # a car against the bus (bus-car pair of the all-pairs test)
        out[3] = touching(rng, out[1], desc.dims[1], desc.dims[3], tau)
    return out


def gen_collisions(desc, tau, rng):
    """Crossroads: car-car and car-pedestrian pairs at k tau (and static ego on the road, so off-road stays quiet)."""
    th = float(rng.choice([0.0, math.pi])) + (float(rng.choice([-1.0, 1.0])) * float(rng.choice(DELTAS)) if rng.random() < 0.5 else 0.0)
    ego = [float(rng.uniform(250, 600)), float(rng.uniform(-15, 15)), 0.0, th]
    car = touching(rng, ego, desc.dims[0], desc.dims[1], tau) if rng.random() < 0.6 else [float(rng.uniform(100, 1500)), float(rng.uniform(-50, 50)), 0.0, heading(rng)]
    target, dims = (ego, desc.dims[0]) if rng.random() < 0.5 else (car, desc.dims[1])
    ped = touching(rng, target, dims, desc.dims[2], tau) if rng.random() < 0.6 else [float(rng.uniform(100, 1500)), float(rng.uniform(-80, 80)), 0.0, heading(rng)]
    return [ego, car, ped]


def gen_offroad_finish(desc, tau, rng):
    """Ego with an edge or a corner at k tau from the road (top / bottom kerb, the far end) or from the finish line."""
    length, width, _ = desc.dims[0]
    x0, x1, y0, y1 = road_box(desc)
    th = heading(rng) if rng.random() < 0.7 else float(rng.uniform(-0.6, 0.6))
    ex, ey = extents(length, width, th)
    k = margin_k(rng, tau) if rng.random() < 0.85 else float(rng.uniform(-20, 20))
    where = rng.integers(0, 4)
    if where == 0:
        ego = [rng.uniform(200, 1300), y1 + ey + k, 0.0, th]
    elif where == 1:
        ego = [rng.uniform(200, 1300), y0 - ey - k, 0.0, th]
    elif where == 2:     # min corner x = W + k: the finish line
        ego = [desc.W + ex + k, rng.uniform(-40, 40), 0.0, th]
    else:                # the rear end of the road, from outside
        ego = [x0 - ex - k, rng.uniform(-40, 40), 0.0, th]
    return [[float(v) for v in ego], [700.0, -90.0, 0.0, 0.0]]


def gen_zones(desc, tau, rng):
    """Moving ego, two pedestrians at k tau from the ego box, the braking zone, the reaction zone and the split between
    them (post-step positions: the ego's v dt move is compensated)."""
    length, width, min_throttle = desc.dims[0]
    hl, hw = length / 2, width / 2
    th = heading(rng) if rng.random() < 0.5 else float(rng.uniform(-math.pi, math.pi))
    v = float(rng.uniform(1.0, 144.0)) if rng.random() < 0.9 else 0.0
    c, s = math.cos(th), math.sin(th)
    post = (float(rng.uniform(300, 900)), float(rng.uniform(-30, 30)))
    bd = v * v / (2 * -min_throttle)
    td = bd + v * xg.REACTION_TIME
    peds = []
    for b in (1, 2):
        pl, pw = desc.dims[b][:2]
        thb = heading(rng)
        cd, sd = abs(c * math.cos(thb) + s * math.sin(thb)), abs(c * math.sin(thb) - s * math.cos(thb))
        ru, rw = cd * pl / 2 + sd * pw / 2, sd * pl / 2 + cd * pw / 2     # pedestrian radii along the ego's axes
        k = margin_k(rng, tau)
        kind = rng.integers(0, 7) if b == 1 or rng.random() < 0.5 else 7
        w = float(rng.uniform(-hw, hw))
        if kind == 0:
            u = -(hl + ru + k)                        # behind the ego box
        elif kind == 1:
            u = hl + ru + k                           # ahead of the ego box (braking zone starts there)
        elif kind == 2:
            u = hl + bd - ru - k                      # inside the braking zone, k tau from the split
        elif kind == 3:
            u = hl + bd + ru + k                      # in the reaction zone, k tau beyond the split
        elif kind == 4:
            u = hl + td + ru + k                      # k tau beyond the far end of the reaction zone
        elif kind == 5:                               # beside the strip
            u = float(rng.uniform(-hl, hl + td))
            w = float(rng.choice([-1.0, 1.0])) * (hw + rw + k)
        elif kind == 6:
            u, w = float(rng.uniform(hl + bd, hl + td + ru)), float(rng.uniform(-hw - rw, hw + rw))
        else:
            u, w = float(rng.uniform(-hl - 20, hl + td + 20)), float(rng.uniform(-hw - 30, hw + 30))
        peds.append([post[0] + u * c - w * s, post[1] + u * s + w * c, 0.0, thb])
    ego = [post[0] - v * DT * c, post[1] - v * DT * s, v, th]
    return [ego] + peds


def in_frame(state, origin, phi):
    """A body state given in a road's frame (x along the road from its rear centre), in world coordinates."""
    x, y, v, th = state
    c, s = math.cos(phi), math.sin(phi)
    return [origin[0] + x * c - y * s, origin[1] + x * s + y * c, v, th + phi]


def gen_custom_roads(desc, tau, rng, dtype="float64"):
    """Pedestrians across the kerbs and far corners of the rotated road and of the two roads on either side of the axis
    snap; the ego at k tau from their edges, off the major road (off-road against a rotated road)."""
    frames = custom_road_frames(TAU[dtype] * 1e-3)
    out = []
    for b in range(3):
        r = int(rng.integers(1, 4))
        origin, phi, length = frames[r]
        road = (0.0, length, -58.4, 58.4)
        if b > 0 and rng.random() < 0.35:
            side = float(rng.choice([-1.0, 1.0]))
            local = corner_place(rng, desc.dims[b], tau, (length, 58.4 * side), (1, side))
        else:
            local = kerb_place(rng, desc.dims[b], tau, road, (0.35 * length, 0.9 * length), int(rng.choice([0, 1, 3])))
        out.append(in_frame(local, origin, phi))
    return out


def gen_pelican(desc, tau, rng):
    """Pelican crossing: the second car and the two pedestrians at k tau from the traffic lights and the obstacle
    (rectangular statics, tested with box_margin)."""
    statics = []
    for q in desc.statics:
        x0, x1, y0, y1 = (float(v) for v in xg.aabb(q))
        statics.append(([(x0 + x1) / 2, (y0 + y1) / 2, 0.0, 0.0], (x1 - x0, y1 - y0)))
    out = [[200.0, 29.2, 0.0, 0.0], None, [2.0, 0.0, 0.0, 0.0], None, None]   # body 2: the crossing, its light state
    for b in (1, 3, 4):
        pose, dims = statics[int(rng.integers(0, len(statics)))]
        out[b] = touching(rng, pose, dims, desc.dims[b], tau) if rng.random() < 0.85 else \
            [float(rng.uniform(650, 950)), float(rng.uniform(-110, 110)), 0.0, heading(rng)]
    return out


def gen_obstacle(desc, tau, rng):
    """A non-rectangular road_map.obstacle (sat_pose_quad): the ego and the pedestrians at k tau from its edges."""
    cx, cy = sum(p[0] for p in OBSTACLE) / 4, sum(p[1] for p in OBSTACLE) / 4
    out = []
    for b in range(3):
        if (b == 0 and rng.random() < 0.6) or (b > 0 and rng.random() < 0.15):
            out.append([float(rng.uniform(100, 400)) if b == 0 else float(rng.uniform(450, 750)), float(rng.uniform(-40, 40)), 0.0,
                        heading(rng)])
            continue
        i = int(rng.integers(0, 4))
        (ax, ay), (bx, by) = OBSTACLE[i], OBSTACLE[(i + 1) % 4]
        ln = math.hypot(bx - ax, by - ay)
        nx, ny = (by - ay) / ln, -(bx - ax) / ln
        if nx * (ax - cx) + ny * (ay - cy) < 0:
            nx, ny = -nx, -ny                                 # outward
        f = float(rng.uniform(0.25, 0.75))
        th = heading(rng) if rng.random() < 0.5 else math.atan2(by - ay, bx - ax) + float(rng.choice([0.0, 1e-10, -1.1e-5]))
        length, width = desc.dims[b][:2]
        c, s = math.cos(th), math.sin(th)
        rn = abs(nx * c + ny * s) * length / 2 + abs(-nx * s + ny * c) * width / 2
        d = rn + (margin_k(rng, tau) if rng.random() < 0.85 else float(rng.uniform(-20, 20)))
        out.append([ax + f * (bx - ax) + d * nx, ay + f * (by - ay) + d * ny, 0.0, th])
    return out


CATEGORIES = {
    # name: scenario, bodies, collisions, off-road, generator, envs (never a multiple of 16 or 224), seed
    "road_share_pedestrian": SimpleNamespace(scenario="pedestrians", m=2, collisions="ego", offroad=False, gen=gen_ped_share, n=1303, seed=1),
    "road_share_bus_stop": SimpleNamespace(scenario="bus-stop", m=5, collisions="all", offroad=False, gen=gen_bus_stop, n=701, seed=2),
    "collisions_crossroads": SimpleNamespace(scenario="crossroads", m=3, collisions="all", offroad=True, gen=gen_collisions, n=701, seed=3),
    "offroad_finish": SimpleNamespace(scenario="pedestrians", m=2, collisions="ego", offroad=True, gen=gen_offroad_finish, n=601, seed=4),
    "ego_zones": SimpleNamespace(scenario="pedestrians", m=3, collisions="ego", offroad=False, gen=gen_zones, n=901, seed=5),
    "custom_roads": SimpleNamespace(scenario="custom-roads", m=3, collisions="ego", offroad=True, gen=gen_custom_roads, n=757, seed=6),
    "statics_pelican": SimpleNamespace(scenario="pelican", m=5, collisions="all", offroad=False, gen=gen_pelican, n=523, seed=7),
    "statics_obstacle": SimpleNamespace(scenario="obstacle", m=3, collisions="all", offroad=False, gen=gen_obstacle, n=617, seed=8),
}
HETEROGENEOUS = ("bus-stop", "crossroads", "pelican", "custom-roads")   # tables the rollout kernels also run without unrolling


def placements(name, dtype):
    """[M, 4, N] initial states of a category; the same configurations for both dtypes, tau-scaled per dtype."""
    cat = CATEGORIES[name]
    desc = Desc(compile_category(cat, "external", dtype), dtype)
    rng = np.random.default_rng(cat.seed)
    extra = {"dtype": dtype} if cat.gen is gen_custom_roads else {}
    rows = [cat.gen(desc, TAU[dtype], rng, **extra) for _ in range(cat.n)]
    return np.ascontiguousarray(np.transpose(np.asarray(rows, dtype=np.float64), (1, 2, 0)))


# ================================================================================================ the contract
def recovered_share(state, reward, done, winner, W, dtype):
    """p from reward[b] = (ego_rel - p) * cost_step + terminal[b], with ego_rel = clamp((W - x0) / W) formed as the kernel
    forms it and the terminal reward of the engine's own decision (environment.py:208-220).  cost_step = 4 makes every
    product exact, so p carries only the rounding of the two additions: a few ulp of cost_step, and one ulp of
    |terminal| + cost_step where a terminal reward was added (returned as the second value, per body and env)."""
    R = np.float64 if dtype == "float64" else np.float32
    x0 = state[0, 0].astype(R)
    ego_rel = np.clip((R(W) - x0) * R(1.0 / W), R(0), R(1)).astype(np.float64)
    m = reward.shape[0]
    body = np.arange(1, m)[:, None]
    terminal = np.where(done[None, :] == 1, np.where(winner[None, :] == 0, -6000.0,
                                                     np.where(winner[None, :] == body, 6000.0, 2000.0)), 0.0)
    slack = np.where(terminal != 0, np.spacing(R(6004.0)).astype(np.float64), 0.0) / 4.0
    return ego_rel[None, :] - (reward[1:].astype(np.float64) - terminal) / 4.0, slack


def check_contract(name, desc, state, reward, done, winner, tangent, liveness, dtype, truths=None):
    """Assertions 2-5 of the module docstring on one step's outputs; returns the exact truths and summary counts."""
    tau = TAU[dtype]
    n = state.shape[-1]
    truths = truths or [exact_truth(desc, state[:, :, e], tau, dtype) for e in range(n)]
    p_got, slack = recovered_share(state, reward, done, winner, desc.W, dtype)
    flagged = tangent.astype(bool)
    unsound, insensitive, causeless, share_err = [], [], [], []
    for e, tr in enumerate(truths):
        p = [float(q) for q in tr.shares]
        live_exact = [q > F(1, 2) for q in tr.shares]
        differs = (bool(done[e] == 1) != tr.terminate) or (int(winner[e]) != tr.winner) or \
                  any(bool(liveness[b + 1, e]) != live_exact[b] for b in range(desc.m - 1))
        if differs and not flagged[e]:
            unsound.append(e)
        near = any(d.within(F(tau) / 2) for d in tr.sens) or any(abs(q - F(1, 2)) <= F(tau) / 2 for q in tr.shares)
        if near and not flagged[e]:
            insensitive.append(e)
        if flagged[e] and not (any(d.within(2 * F(tau)) for d in tr.cause) or any(abs(q - F(1, 2)) < 2 * F(tau) for q in tr.road_shares)):
            causeless.append(e)
        for b in range(desc.m - 1):
            err = abs(p_got[b, e] - p[b])
            if err > tr.bounds[b] + slack[b, e]:
                share_err.append((e, b + 1, tr.labels[b], err, tr.bounds[b] + slack[b, e]))

    def rows(es):
        return [(e, state[:, :, e].tolist(), int(done[e]), int(winner[e]), int(tangent[e])) for e in es[:4]]
    assert not unsound, f"{name}/{dtype}: decisions differ from the exact ones without a flag: {rows(unsound)}"
    assert not insensitive, f"{name}/{dtype}: a consulted margin within tau/2 was not flagged: {rows(insensitive)}"
    assert not causeless, f"{name}/{dtype}: flagged without a margin or share within 2 tau: {rows(causeless)}"
    worst = {}
    for e, tr in enumerate(truths):
        for b in range(desc.m - 1):
            lab = tr.labels[b][0] if len(tr.labels[b]) == 1 else "several roads"
            worst[lab] = max(worst.get(lab, 0.0), abs(p_got[b, e] - float(tr.shares[b])))
    print(f"{name}/{dtype}: {int(flagged.sum())} of {n} flagged; worst share error by branch:",
          {k: float(f"{v:.3g}") for k, v in sorted(worst.items())})
    share_err.sort(key=lambda r: -r[3] / max(r[4], 1e-300))
    assert not share_err, f"{name}/{dtype}: shares outside their bound (env, body, branch, err, bound): {share_err[:6]}"
    return truths


def coverage(name, desc, truths, flagged, done, dtype):
    """Both answers of every decision, flagged and unflagged envs, and a few dozen envs of every road_share branch (and
    every kind of static, and both sides of the road-axis snap) the category aims at, per body type."""
    n = len(truths)
    assert 0 < int(flagged.sum()) < n, f"{name}: flagged {int(flagged.sum())} of {n}"
    term = np.array([t.terminate for t in truths])
    if name in ("collisions_crossroads", "offroad_finish", "ego_zones", "custom_roads", "statics_pelican", "statics_obstacle"):
        assert 0 < term.sum() < n, f"{name}: terminated {term.sum()} of {n}"
    if name.startswith("statics"):   # margins within tau/2 against every static of the scenario
        for k in range(len(desc.statics)):
            hits = sum(k in t.statics_near for t in truths)
            assert hits >= 24, f"{name}: static {k} is within tau/2 in {hits} envs"
    if name == "custom_roads":
        if dtype == "float64":   # in fp32 the rounding of the corners to float is as large as the skews themselves
            assert desc.road_axis == [True, False, True, False], desc.road_axis
        for r, want_label in ((1, "general"), (2, "general" if not desc.road_axis[2] else None), (3, "general" if not desc.road_axis[3] else None)):
            labels = [t.labels[b][r] for t in truths for b in range(desc.m - 1)]
            crossing = sum(lab not in ("zero", "one") for lab in labels)
            assert crossing >= 24, f"{name}: road {r}: {crossing} bodies across its edges ({sorted(set(labels))})"
            if want_label:
                assert all(lab in ("zero", want_label) for lab in labels)
            else:
                assert sum(lab in ("touch", "kerb") or lab.startswith("corner") for lab in labels) >= 24, sorted(set(labels))
    if name == "ego_zones":
        winners = {t.winner for t in truths}
        assert {-1, 1, 2} <= winners, winners
    want = {"road_share_pedestrian": ("touch", "kerb", "corner_open", "corner_axis", "corner_wedge", "corner_clip", "corner_apart"),
            "road_share_bus_stop": ("touch", "kerb", "corner_axis", "corner_wedge", "corner_clip", "corner_apart")}.get(name, ())
    if not want:
        return
    kinds = sorted({tuple(desc.dims[b][:2]) for b in range(1, desc.m)})
    for dims in kinds:
        bodies = [b for b in range(1, desc.m) if tuple(desc.dims[b][:2]) == dims]
        counts = {}
        for t in truths:
            for b in bodies:
                for lab in t.labels[b - 1]:
                    counts[lab] = counts.get(lab, 0) + 1
        live = [t.shares[b - 1] > F(1, 2) for t in truths for b in bodies]
        assert any(live) and not all(live), (name, dims)
        corner_bodies = name == "road_share_pedestrian" or bodies[0] in (1, 2)   # the bus and the second car take corners
        for lab in want:
            if lab.startswith("corner") and not corner_bodies:
                continue
            assert counts.get(lab, 0) >= 24, f"{name}: body {dims}: branch {lab} has {counts.get(lab, 0)} envs ({counts})"


# ================================================================================================ CPU
def test_exact_reference_reproduces_the_reference_kat():
    """Shape.intersects / contains / percentage_intersects as the reference computed them on 240 pairs (geometry_kat.npz),
    from the reference's own corner lists; make_box reproduces those corners to the rounding of the doubles."""
    import os
    rows = np.load(os.path.join(GOLDEN_DIR, "geometry_kat.npz"))["pairs"]
    worst = 0.0
    for row in rows:
        la, wa, xa, ya, ta, lb, wb, xb, yb, tb, hit, inside, want = row[:13]
        a, b = xg.quad(row[13:21].reshape(4, 2)), xg.quad(row[21:29].reshape(4, 2))
        assert (xg.sat_margin(a, b).num <= 0) == bool(hit)
        assert (xg.contains_margin(b, a).num <= 0) == bool(inside)
        worst = max(worst, abs(float(xg.share(a, b)) - want))
        for box, ref in ((xg.make_box(la, wa, ta, xa, ya), row[13:21]), (xg.make_box(lb, wb, tb, xb, yb), row[21:29])):
            assert np.max(np.abs(np.array([float(c) for p in box for c in p]) - ref)) <= 1e-12 * max(1.0, np.abs(ref).max())
    assert worst < 1e-12
    assert rows[:, 10].any() and not rows[:, 10].all() and ((rows[:, 12] > 0) & (rows[:, 12] < 1)).any()


def test_exact_margins_and_shares_on_hand_made_cases():
    unit = xg.make_box(2.0, 2.0, 0.0, 0.0, 0.0)
    touching = xg.make_box(2.0, 2.0, 0.0, 2.0, 0.0)
    assert xg.sat_margin(unit, touching).num == 0                               # touching counts as a hit
    apart = xg.sat_margin(unit, xg.make_box(2.0, 2.0, 0.0, 2.5, 0.0))
    assert apart.cmp(0.5) == 0 and apart.within(0.5) and not apart.within(0.499)
    diamond = xg.make_box(math.sqrt(2.0), math.sqrt(2.0), math.pi / 4, 2.0, 0.0)   # corner at x ~ 1
    assert abs(float(xg.sat_margin(unit, diamond))) < 1e-15
    road = xg.quad([(0.0, 1.0), (10.0, 1.0), (10.0, -1.0), (0.0, -1.0)])
    assert xg.share(xg.make_box(2.0, 2.0, 0.0, 5.0, 1.0), road) == F(1, 2)
    assert xg.share(xg.make_box(2.0, 2.0, 0.0, 0.0, 1.0), road) == F(1, 4)        # on a road corner
    assert xg.contains_margin(road, xg.make_box(2.0, 2.0, 0.0, 5.0, 0.0)).num == 0
    braking, reaction = xg.stopping_zones(0.0, 0.0, 144.0, 0.0, 72.0, 28.0, -144.0)
    assert xg.aabb(braking) == (36, 36 + 72, -14, 14) and xg.aabb(reaction)[1] == 36 + 72 + F(144.0) * F(0.675)


@pytest.mark.parametrize("name", sorted(CATEGORIES))
def test_placements_reach_every_branch_and_both_answers(name):
    """The generator lands on every road_share branch the category aims at, for every body type, with both answers of
    its decisions (exact truth on the fp64 placements themselves)."""
    cat = CATEGORIES[name]
    desc = Desc(compile_category(cat, "external"))
    init = placements(name, "float64")
    truths = [exact_truth(desc, init[:, :, e], TAU["float64"], "float64") for e in range(cat.n)]
    near = np.array([any(d.within(F(TAU["float64"]) / 2) for d in t.sens) or
                     any(abs(q - F(1, 2)) <= F(TAU["float64"]) / 2 for q in t.shares) for t in truths])
    coverage(name, desc, truths, near, None, "float64")


@pytest.mark.parametrize("name", sorted(CATEGORIES))
def test_oracle_meets_the_exact_contract(name):
    """The C oracle — the reference every other GPU test compares with — on the fp64 placements: sound, sensitive,
    specific, shares within their bounds."""
    from oracle.oracle import Oracle
    cat = CATEGORIES[name]
    comp = compile_category(cat, "external")
    init = placements(name, "float64")
    oracle = Oracle(comp, cat.n, threads=8)
    oracle.reset(init_state=init)
    state, reward, done, winner, tangent = oracle.step(np.zeros((cat.m, 2, cat.n)))
    check_contract(name, Desc(comp), state, reward, done, winner, tangent, oracle.liveness.copy(), "float64")


# ================================================================================================ GPU
def make_env(comp, n, dtype):
    from cavgym_b200 import BatchedCAVEnv
    return BatchedCAVEnv(None, None, None, num_envs=n, dtype=dtype, compiled=comp)


def run_paths(name, dtype):
    """One zero-action step of the placements on every kernel path; asserts they agree bitwise and returns the outputs."""
    import torch
    cat = CATEGORIES[name]
    n, m = cat.n, cat.m
    init = placements(name, dtype)
    zeros = np.zeros((m, 2, n))
    outs = {}
    env = make_env(compile_category(cat, "external", dtype), n, dtype)

    def grab(step_out):
        return [v.cpu().numpy().copy() for v in step_out] + [env.episode_liveness.cpu().numpy().copy()]
    for path in ("tma", "plain", "dense"):
        env.set_step_path(path == "tma")
        env.set_dense_path(path == "dense")
        env.reset(init_state=init)
        outs[f"step_{path}"] = grab(env.step(zeros))
    env.set_step_path(True)
    env.set_dense_path(False)
    # three zero-action steps one launch each: what the fused replay of T = 3 must reproduce at every step
    env.reset(init_state=init)
    stepped = [grab(env.step(zeros)) for _ in range(3)]
    keys = ("state", "reward", "done", "winner", "tangent")
    for t_len in (1, 3):
        env.reset(init_state=init)
        rec = env.replay(np.zeros((t_len, m, 2, n)))
        live = env.episode_liveness.cpu().numpy().copy()
        for t in range(t_len):
            got = [rec[k][t].cpu().numpy() for k in keys]
            for key, a, b in zip(keys, stepped[t], got):
                assert np.array_equal(a, b, equal_nan=True), f"{name}/{dtype}: replay T = {t_len} step {t} differs from cavgym_step in {key}"
        assert np.array_equal(live, stepped[t_len - 1][5]), f"{name}/{dtype}: liveness after replay T = {t_len}"
    env.close()
    ref = outs["step_tma"]
    for path, got in outs.items():
        for key, a, b in zip(keys + ("liveness",), ref, got):
            assert np.array_equal(a, b, equal_nan=True), f"{name}/{dtype}: {path} differs from step_tma in {key}"
    for key, a, b in zip(keys + ("liveness",), ref, stepped[0]):
        assert np.array_equal(a, b, equal_nan=True), f"{name}/{dtype}: the first of three steps differs from step_tma in {key}"
    if cat.scenario in HETEROGENEOUS:   # thread-per-env rollout with noop agents
        agents = make_env(compile_category(cat, "noop", dtype), n, dtype)
        agents.reset(init_state=init)
        agents.rollout(1, auto_reset=False)
        torch.cuda.synchronize()
        assert np.array_equal(agents.state.cpu().numpy(), ref[0]), f"{name}/{dtype}: thread-per-env rollout state"
        assert np.array_equal(agents.episode_liveness.cpu().numpy(), ref[5]), f"{name}/{dtype}: thread-per-env rollout liveness"
        assert np.array_equal(agents.done_latch.cpu().numpy(), ref[2]), f"{name}/{dtype}: thread-per-env rollout done"
        assert np.array_equal(agents.winner_latch.cpu().numpy(), ref[3]), f"{name}/{dtype}: thread-per-env rollout winner"
        assert agents.stats()["tangent"] == int(ref[4].astype(bool).sum()), f"{name}/{dtype}: thread-per-env rollout tangent count"
        agents.close()
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("name", sorted(CATEGORIES))
def test_kernel_paths_meet_the_exact_contract(name, dtype):
    cat = CATEGORIES[name]
    desc = Desc(compile_category(cat, "external", dtype), dtype)
    state, reward, done, winner, tangent, liveness = run_paths(name, dtype)
    state = state.astype(np.float64)
    truths = check_contract(name, desc, state, reward, done, winner, tangent, liveness, dtype)
    coverage(name, desc, truths, tangent.astype(bool), done, dtype)
