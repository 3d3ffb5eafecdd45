// danger.cuh — how close a post-step state is to a tester win, for cavgym_rollout_until (kernels_until.cuh).
//
// A tester wins when a pedestrian's box meets the ego's reaction zone (environment.py:195-206).  The danger of a state is
// minus the smallest separating-axis margin of any pedestrian box against the reaction-zone rectangle, in px: positive
// when some pedestrian overlaps the rectangle.  The arithmetic is that of `margin(f.hl + f.bd + hr, hr)` in ego_margins
// (geometry.cuh), without its all_clear shortcut, so a clear pedestrian gets its true distance instead of the placeholder
// 1.  The rectangle is used whether or not the zones exist (f.have: the ego is not steering and moves): the danger only
// guides a splitting scheme between levels; the top level is the engine's own winner.
#pragma once
#include "transition.cuh"

namespace cav {

// Margin of a pedestrian box (centre px, py, heading cos cb / sin sb, half extents hlb, hwb) against the reaction zone of
// the ego frame f (pose, bd, td set as the transition sets them after body_step).
template <typename R>
__device__ __forceinline__ R reaction_margin(const EgoFrame<R>& f, R px, R py, R cb, R sb, R hlb, R hwb) {
  const R tx = px - f.x, ty = py - f.y;
  const R cd = f.c * cb + f.s * sb, sd = f.c * sb - f.s * cb;
  const R acd = rabs(cd), asd = rabs(sd);
  const R u = tx * f.c + ty * f.s, w = ty * f.c - tx * f.s;
  const R tp = tx * cb + ty * sb, tq = ty * cb - tx * sb;
  const R exb = acd * hlb + asd * hwb, eyb = asd * hlb + acd * hwb;
  const R lateral = rabs(w) - (f.hw + eyb);
  const R rp = hlb + asd * f.hw, rq = hwb + acd * f.hw;
  const R hr = (f.td - f.bd) * R(0.5);
  const R centre = f.hl + f.bd + hr, half = hr;
  const R mx = rabs(u - centre) - (half + exb);
  const R m3 = rabs(tp - centre * cd) - (rp + acd * half);
  const R m4 = rabs(tq + centre * sd) - (rq + asd * half);
  return rmax(rmax(lateral, mx), rmax(m3, m4));
}

// -min over the pedestrians b >= 1 of reaction_margin; -inf when there is none (the host refuses such scenarios).
// Pedestrians are the bodies the transition tests against the zones: every non-ego body in the homogeneous kernels
// (GENERIC = false), the CAV_FLAG_PEDESTRIAN bodies otherwise.
template <typename R, int M, bool GENERIC>
__device__ __forceinline__ R danger(const DevScenario<R>& sc, const EnvRegs<R, M>& env) {
  const DevType<R>& k0 = sc.bodies[0].k;
  EgoFrame<R> f;
  f.x = env.s[0][0]; f.y = env.s[0][1]; f.c = env.cs[0][0]; f.s = env.cs[0][1]; f.hl = k0.hl; f.hw = k0.hw;
  const R v0 = env.s[0][2];
  f.bd = (v0 * v0) * k0.inv_2brake;
  f.td = f.bd + v0 * R(0.675);
  f.have = true;
  R d = -INFINITY;
#pragma unroll
  for (int b = 1; b < M; ++b) {
    if (GENERIC && (sc.bodies[b].flags & CAV_FLAG_PEDESTRIAN) == 0) continue;
    d = rmax(d, -reaction_margin(f, env.s[b][0], env.s[b][1], env.cs[b][0], env.cs[b][1], sc.bodies[b].k.hl, sc.bodies[b].k.hw));
  }
  return d;
}

}  // namespace cav
