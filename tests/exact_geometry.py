"""Exact restatement of the geometry one step decides on, for the near-tangent contract tests.

Everything here is rational arithmetic (fractions.Fraction) on the exact values of the doubles it is given (a float32 state
is widened to double first, which is exact).  Nothing is rounded until a result is turned into a float for reporting.

Body boxes are built as the reference builds them: make_rectangle(L, W).transform(theta, (x, y)) with c = math.cos(theta) and
s = math.sin(theta), the doubles the reference hands to Shapely, taken as exact rationals.  The engine's own cos / sin (host
libm values from its heading cache, or the device's sincos) may differ from those by about one ulp: a corner then moves by
|L| * 2**-53 ~ 1e-14 px in fp64 and |L| * 2**-24 ~ 1e-5 px in fp32 (L <= 192 px, the bus), far inside the near-tangent
tolerances tau = 1e-7 and 5e-2 px.

Margins are signed distances: for a separating-axis test, the largest over the edge normals of both polygons of the
smallest outward distance of the other polygon's vertices (> 0 disjoint, <= 0 intersecting, touching counts as a hit); for
`contains`, the largest outward distance of an inner vertex over the outer polygon's edges (<= 0 contained).  A distance is
kept as (numerator, |e|^2) with distance = numerator / |e|; it is compared with a threshold t by signs and by
numerator^2 against t^2 |e|^2, never through a square root (the engine's separation_bits does the same).
"""
import math
from fractions import Fraction as F
from functools import cmp_to_key

REACTION_TIME = 0.675   # library/bodies.py


def fx(v):
    """Exact rational value of a double (or of a float32 widened to double)."""
    return F(float(v))


# ------------------------------------------------------------------------------------------------ signed distances
class Dist:
    """num / sqrt(len2), exactly.  len2 > 0."""
    __slots__ = ("num", "len2")

    def __init__(self, num, len2):
        self.num, self.len2 = num, len2

    def cmp(self, t):
        """sign(self - t) for a rational threshold t."""
        a, t = self.num, F(t)
        if (a >= 0) != (t >= 0):
            return 1 if a >= 0 else -1
        lhs, rhs = a * a, t * t * self.len2
        if lhs == rhs:
            return 0
        bigger = lhs > rhs               # |self| > |t|
        return (1 if bigger else -1) * (1 if a >= 0 else -1)

    def within(self, t):
        """|self| <= t (t >= 0)."""
        return self.cmp(-t) >= 0 and self.cmp(t) <= 0

    def __float__(self):
        return float(self.num) / math.sqrt(float(self.len2))


def dist_cmp(a, b):
    """sign(a - b) of two Dist, exactly."""
    sa, sb = (a.num > 0) - (a.num < 0), (b.num > 0) - (b.num < 0)
    if sa != sb:
        return 1 if sa > sb else -1
    lhs, rhs = a.num * a.num * b.len2, b.num * b.num * a.len2
    if lhs == rhs:
        return 0
    bigger = lhs > rhs               # |a| > |b|
    return (1 if bigger else -1) * (1 if sa >= 0 else -1)


def dmax(items):
    return max(items, key=cmp_to_key(dist_cmp))


class Axis(Dist):
    """A distance measured along a coordinate axis (|e| = 1)."""

    def __init__(self, num):
        super().__init__(num, F(1))


# ------------------------------------------------------------------------------------------------ polygons
def make_box(length, width, theta, x, y):
    """make_rectangle(length, width).transform(theta, (x, y)) on exact rationals (geometry.py): corners rear_left,
    front_left, front_right, rear_right.  theta == 0 takes the reference's translate-only path."""
    hl, hw = fx(length) * F(1, 2), fx(width) * F(1, 2)
    local = [(-hl, hw), (hl, hw), (hl, -hw), (-hl, -hw)]
    x, y = fx(x), fx(y)
    if float(theta) == 0.0:
        return [(x + u, y + v) for u, v in local]
    c, s = fx(math.cos(float(theta))), fx(math.sin(float(theta)))
    return [(x + (c * u - s * v), y + (s * u + c * v)) for u, v in local]


def frame_box(x, y, theta, u0, u1, hw):
    """The rectangle [u0, u1] x [-hw, hw] of a body frame (x, y, theta) in world coordinates, exactly."""
    x, y = fx(x), fx(y)
    if float(theta) == 0.0:
        c, s = F(1), F(0)
    else:
        c, s = fx(math.cos(float(theta))), fx(math.sin(float(theta)))
    local = [(u0, hw), (u1, hw), (u1, -hw), (u0, -hw)]
    return [(x + (c * u - s * v), y + (s * u + c * v)) for u, v in local]


def quad(points):
    return [(fx(px), fx(py)) for px, py in points]


def area2(poly):
    return sum(poly[i][0] * poly[(i + 1) % len(poly)][1] - poly[(i + 1) % len(poly)][0] * poly[i][1] for i in range(len(poly)))


def _outward(poly):
    """(a, e, sign) per edge: outward distance of p is sign * cross(e, p - a) / |e|."""
    sign = -1 if area2(poly) > 0 else 1      # counter-clockwise: the inside is on the left (cross > 0)
    out = []
    for i in range(len(poly)):
        a, b = poly[i], poly[(i + 1) % len(poly)]
        e = (b[0] - a[0], b[1] - a[1])
        if e[0] or e[1]:
            out.append((a, e, sign))
    return out


def _cross(a, e, p):
    return e[0] * (p[1] - a[1]) - e[1] * (p[0] - a[0])


def sat_margin(A, B):
    """Largest separating-axis margin of two convex polygons: > 0 disjoint, <= 0 intersecting (closed)."""
    best = []
    for P, Q in ((A, B), (B, A)):
        for a, e, sign in _outward(P):
            best.append(Dist(min(sign * _cross(a, e, q) for q in Q), e[0] * e[0] + e[1] * e[1]))
    return dmax(best)


def contains_margin(outer, inner):
    """Largest outward distance of a vertex of `inner` over the edges of `outer`: <= 0 <=> outer contains inner."""
    return dmax([Dist(max(sign * _cross(a, e, q) for q in inner), e[0] * e[0] + e[1] * e[1]) for a, e, sign in _outward(outer)])


def clip(subject, clip_poly):
    """subject ∩ clip_poly for convex polygons, by Sutherland-Hodgman on rationals."""
    out = list(subject)
    for a, e, sign in _outward(clip_poly):
        if not out:
            break
        src, out = out, []
        for k in range(len(src)):
            p, q = src[k], src[(k + 1) % len(src)]
            dp, dq = -sign * _cross(a, e, p), -sign * _cross(a, e, q)   # >= 0 inside
            if dp >= 0:
                out.append(p)
            if (dp > 0 > dq) or (dp < 0 < dq):
                t = dp / (dp - dq)
                out.append((p[0] + t * (q[0] - p[0]), p[1] + t * (q[1] - p[1])))
    return out


def share(box, road):
    """Shape.percentage_intersects(box, road) (geometry.py:80-87): the exact area ratio.  Disjoint gives 0 and contained
    gives 1 through the same formula, so the reference's intersects / contains short cuts agree with it."""
    part = clip(box, road)
    return abs(area2(part)) / abs(area2(box)) if len(part) >= 3 else F(0)


def aabb(poly):
    xs, ys = [p[0] for p in poly], [p[1] for p in poly]
    return min(xs), max(xs), min(ys), max(ys)


def aabb_gap(a, b):
    """Largest axis-aligned gap between the bounding boxes of two polygons (> 0: disjoint along x or y)."""
    ax0, ax1, ay0, ay1 = aabb(a)
    bx0, bx1, by0, by1 = aabb(b)
    return max(ax0 - bx1, bx0 - ax1, ay0 - by1, by0 - ay1)


# ------------------------------------------------------------------------------------------------ stopping zones
def stopping_zones(x, y, v, theta, length, width, min_throttle):
    """DynamicBody.stopping_zones (bodies.py) and ConvexQuadrilateral.split_longitudinally (geometry.py) on the
    post-step state, exactly: the braking zone [hl, hl + bd] and the reaction zone [hl + bd, hl + td] of the body frame.
    None when the total stopping distance is zero (the caller handles steering)."""
    v = fx(v)
    bd = v * v / (2 * -fx(min_throttle))
    td = bd + v * fx(REACTION_TIME)
    if td == 0:
        return None
    hl, hw = fx(length) / 2, fx(width) / 2
    return frame_box(x, y, theta, hl, hl + bd, hw), frame_box(x, y, theta, hl + bd, hl + td, hw)
