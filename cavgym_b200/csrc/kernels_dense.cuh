// kernels_dense.cuh — warp-per-environment kernels for scenarios with many bodies (CAV_SMALL_M < M <= CAV_MAX_BODIES),
// e.g. the dense-traffic stress configuration: 64 cars + 256 spawned pedestrians per env, terminate_collisions = "all",
// 51,040 box pairs per env-step (environment.py:156-177 is O(M^2)).
//
//   dense_kernel        n_steps of CAVEnv.step (environment.py:119-223) for one env per WARP: replayed actions or
//                       on-device agents, optional trajectory slabs, optional auto-reset (cavgym_step / _replay / _rollout)
//   dense_reset_kernel  CAVEnv.reset (environment.py:225-229) per warp
//
// Work split inside a warp: body b belongs to lane b % 32.  Per-body work (agents, DynamicBody.step, road share,
// reward, liveness, ego / stopping-zone tests) is a lane-strided loop; the per-environment reductions — any collision,
// any near-tangent decision, lowest-index pedestrian in the reaction zone (environment.py:198-200), action validity —
// are warp votes (__any_sync / __all_sync / __reduce_min_sync).  There is no block-wide barrier after the prologue.
//
// Shared memory (per env = per warp), resident for the whole launch: x, y, v, theta, cos, sin of every body in the
// engine's type R — staged once (dense_stage_env), stepped in place for every fused step, written back once
// (dense_writeback_env) — plus one float4 per body for the BROAD PHASE of the all-pairs test: the body's axis-aligned
// bounds {x lo, x hi, y lo, y hi} in fp32, rounded outward (broad_entry), so that a pair test is four fp32 compares and no
// arithmetic (broad_overlap) and passes a strict superset of the pairs the R-precision test passes.  Two levels: the union
// box of every 32-body tile (four REDUX each) lets whole tiles be skipped; inside, a lane meets the bodies below its own
// through broadcast LDS.128 reads, and the pairs within a tile by rotation.  Survivors (a few per env-step) take exactly
// the test sequence of the thread-per-env path (transition.cuh): R-precision AABB gap, then the four-axis margin, so
// results — including near-tangent flags — are bitwise those of the small-M kernels on the same scenario
// (tests/test_gpu_dense.py).  Per-body metadata (type, class flags, agent kind) is staged once per CTA and shared by its
// envs; which crossing agents are mid-crossing is a bit per body in a register (DenseEnv::busy).
//
// Bound: instruction fetch and fixed-latency dependencies at 8 warps per SM, not HBM and not a pipe: an env-step moves
// 88 B per body but runs ~11 k warp-instructions of branchy fp64 code (DESIGN.md 4.4, 4.5).  Rare paths are therefore
// out of line (body_turn_outlined, dense_road_share_edge, dense_random_sample, dense_*_candidates, dense_pair).
#pragma once
#include "transition.cuh"

namespace cav {

#ifndef CAV_DENSE_WARPS
#define CAV_DENSE_WARPS 4
#endif
#ifndef CAV_DENSE_MIN_BLOCKS
#define CAV_DENSE_MIN_BLOCKS 1
#endif
constexpr int kDenseWarps = CAV_DENSE_WARPS;
constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr int kDenseTiles = CAV_MAX_BODIES / 32;

enum { DM_TYPE_MASK = 7, DM_PELICAN = 8, DM_PEDESTRIAN = 16, DM_SPAWN = 32, DM_AGENT_SHIFT = 8, DM_AGENT_MASK = 7, DM_ABSENT = 1 << 15 };

template <typename R>
struct DenseBody {       // CavBody (include/cavgym.h) in the engine's type, 64 B
  int32_t meta;          // DM_* bits
  int32_t spawn_id;
  double epsilon;
  R threshold;
  R init[4];
  R static_share;        // PelicanCrossing: percentage_intersects(static box, road), a scenario constant
};

template <typename R>
struct DenseTables {
  DevType<R> types[CAV_MAX_TYPES];
  const DenseBody<R>* bodies;   // device, [M]
  int32_t has_external;         // some body takes its action from the `actions` buffer
  int32_t pad;
};

__device__ __forceinline__ int dm_agent(int32_t mt) { return (mt >> DM_AGENT_SHIFT) & DM_AGENT_MASK; }

template <typename R>
struct DenseSmem {
  float4* bp;              // [Mp] broad-phase entries
  float4* tu;              // [kDenseTiles] union of the entries of each 32-body tile
  R *x, *y, *v, *c, *s, *th;   // [Mp] bodies (resident for the whole launch)
  const int32_t* meta;     // [Mp], shared by the CTA
};

template <typename R>
__host__ __device__ inline size_t dense_smem_bytes(int m, int warps) {
  const size_t mp = (size_t)((m + 31) & ~31);
  return (size_t)warps * ((mp + kDenseTiles) * sizeof(float4) + mp * 6 * sizeof(R)) + mp * sizeof(int32_t);
}

// Broad-phase entry of a box: its axis-aligned bounds {x lo, x hi, y lo, y hi} in fp32, widened by the tangent tolerance and
// rounded OUTWARD (round-down for lo, round-up for hi, every operation), so that
//     R-precision test not "apart"  (|x_i - x_j| - (ex_i + ex_j) <= tau and the same in y)
//  => lo_i <= hi_j and lo_j <= hi_i in both axes            (four fp32 compares, no arithmetic, hence no rounding)
// i.e. the fp32 filter passes a superset of the pairs the exact stage wants to see.  An absent / static body gets the
// empty interval (+inf, -inf): it overlaps nothing.
__device__ __forceinline__ float4 broad_entry(double x, double y, double ex, double ey, double tau) {
  return make_float4(__double2float_rd(__dsub_rd(__dsub_rd(x, ex), tau)), __double2float_ru(__dadd_ru(__dadd_ru(x, ex), tau)),
                     __double2float_rd(__dsub_rd(__dsub_rd(y, ey), tau)), __double2float_ru(__dadd_ru(__dadd_ru(y, ey), tau)));
}
__device__ __forceinline__ float4 broad_entry(float x, float y, float ex, float ey, float tau) {
  return make_float4(__fsub_rd(__fsub_rd(x, ex), tau), __fadd_ru(__fadd_ru(x, ex), tau),
                     __fsub_rd(__fsub_rd(y, ey), tau), __fadd_ru(__fadd_ru(y, ey), tau));
}
__device__ __forceinline__ float4 broad_absent() { return make_float4(INFINITY, -INFINITY, INFINITY, -INFINITY); }
// float <-> int with the same order (for the warp-wide REDUX min / max, which exist for integers only)
__device__ __forceinline__ int ordered_int(float f) { const int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7FFFFFFF; }
__device__ __forceinline__ float ordered_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7FFFFFFF); }
__device__ __forceinline__ bool broad_overlap(const float4& a, const float4& b) {
  return a.x <= b.y && b.x <= a.y && a.z <= b.w && b.z <= a.w;
}

template <typename R>
__device__ __forceinline__ Box<R> dense_box(const DenseSmem<R>& sm, const DevType<R>& k, int b) {
  return {sm.x[b], sm.y[b], sm.c[b], sm.s[b], k.hl, k.hw};
}
template <typename R>
__device__ __forceinline__ Pose<R> dense_pose(const DenseSmem<R>& sm, const DevType<R>& k, int b) {
  return {sm.x[b], sm.y[b], sm.th[b], sm.c[b], sm.s[b], k.length, k.width};
}

// road_share of transition.cuh on an explicit pose (same cases, same order, same arithmetic), in two parts: the two
// answers almost every body gets — clear of the road's bounding box: 0; axis-aligned road, clearly inside: 1 — stay inline,
// kerbs, corners and general quads are one out-of-line function (the hot loop must stay small: the kernel is bound by
// instruction fetch, DESIGN.md 4.4).
template <typename R>
__device__ __noinline__ R dense_road_share_edge(const DevScenario<R>& sc, const DenseSmem<R>& sm, const DevType<R>& k, int b, int r,
                                                R ex, R ey, R tau, bool* near_out) {
  bool near = false;
  const Aabb<R> rd = sc.road_bb[r];
  const R px = sm.x[b], py = sm.y[b];
  const R m0 = (px - ex) - rd.x0, m1 = rd.x1 - (px + ex), m2 = (py - ey) - rd.y0, m3 = rd.y1 - (py + ey);
  const R mx = rmin(m0, m1), my = rmin(m2, m3);
  R result;
  bool settled = false;
  if (sc.road_axis[r]) {
    const bool x_edge = mx < my;
    const R lo = x_edge ? mx : my, hi = x_edge ? my : mx;
    const R opposite = x_edge ? rmax(m0, m1) : rmax(m2, m3);
    if (lo > -tau && hi >= tau && opposite >= tau) {   // (lo < tau here: the caller returned 1 otherwise)
      result = kerb_touch_share(sm.c[b], sm.s[b], k.hl, k.hw, lo, x_edge, ex, ey, near); settled = true;
    } else if (lo <= -tau && hi >= tau && opposite >= tau) {
      const R ac = rabs(sm.c[b]), as = rabs(sm.s[b]);
      const R p = kerb_share(lo + (x_edge ? ex : ey), (x_edge ? ac : as) * k.hl, (x_edge ? as : ac) * k.hw);
      if (rabs(p - R(0.5)) < tau) near = true;
      result = p; settled = true;
    } else if (mx < tau && my < tau && rmax(m0, m1) >= tau && rmax(m2, m3) >= tau) {
      const bool low_x = m0 < m1, low_y = m2 < m3;
      const R p = corner_share_closed(dense_pose(sm, k, b), mx + ex, my + ey, low_x ? R(-1) : R(1), low_x ? -rd.x0 : rd.x1,
                                      low_y ? R(-1) : R(1), low_y ? -rd.y0 : rd.y1, tau);
      if (rabs(p - R(0.5)) < tau) near = true;
      result = p; settled = true;
    }
  }
  if (!settled) {
    const Share<R> share = road_share_general(dense_pose(sm, k, b), &sc.quads[r], tau);
    near = (share.tangent != 0) || (rabs(share.value - R(0.5)) < tau);
    result = share.value;
  }
  *near_out = near;
  return result;
}

template <typename R>
__device__ __forceinline__ R dense_road_share(const DevScenario<R>& sc, const DenseSmem<R>& sm, const DevType<R>& k, int b, int r,
                                              R ex, R ey, R tau, bool& near) {
  const Aabb<R> rd = sc.road_bb[r];
  const R px = sm.x[b], py = sm.y[b];
  const R m0 = (px - ex) - rd.x0, m1 = rd.x1 - (px + ex), m2 = (py - ey) - rd.y0, m3 = rd.y1 - (py + ey);
  const R mx = rmin(m0, m1), my = rmin(m2, m3);
  if (mx < -((ex + ex) + tau) || my < -((ey + ey) + tau)) return R(0);
  if (sc.road_axis[r] && rmin(mx, my) >= tau) return R(1);
  bool edge_near = false;
  const R p = dense_road_share_edge(sc, sm, k, b, r, ex, ey, tau, &edge_near);
  near |= edge_near;
  return p;
}

// RandomAgent.choose_action when its epsilon test fires (template.py:52-56): Box.sample / Discrete.sample.  Out of line: rare.
template <typename R>
__device__ __noinline__ void dense_random_sample(const EnvBuffers<R>& buf, const DevType<R>& k, int64_t e, int b, bool pelican,
                                                 uint32_t episode, uint32_t t_ep, double u1, double u2, R* a0, R* a1) {
  if (pelican) {
    R v = R(floor(u1 * 4.0));
    if (v > R(3)) v = R(3);
    *a0 = v; *a1 = R(0);
    return;
  }
  if (!buf.uni_override) {
    double w[2];
    draw_block(buf.seed, (uint64_t)(buf.shard + e), b, KIND_AGENT1, episode, t_ep, w);
    u2 = w[0];
  }
  *a0 = R(double(k.amin) + (double(k.amax) - double(k.amin)) * u1);
  *a1 = R(double(k.smin) + (double(k.smax) - double(k.smin)) * u2);
}

// A vote of the pair sweep fired: look at the eight (or sixteen) folded tests one by one and run the exact stage on the
// candidates.  Out of line — a few calls per env-step — so that the sweep itself is a few hundred bytes of code.
template <typename R>
__device__ __noinline__ bool dense_sweep_candidates(const DenseSmem<R>& sm, const DenseTables<R>& tb, int i0, int jA, int jB, bool useA,
                                                    float4 pA, float4 pB, R tau, bool* tangent) {
  bool hit = false, tg = false;
  for (int u = 0; u < 8; ++u) {
    const int i = i0 + u;
    const float4 pi = sm.bp[i];
    if (useA && broad_overlap(pi, pA)) hit |= dense_pair(sm, tb, i, jA, tau, tg);
    if (broad_overlap(pi, pB)) hit |= dense_pair(sm, tb, i, jB, tau, tg);
  }
  *tangent |= tg;
  return hit;
}
template <typename R>
__device__ __noinline__ bool dense_within_candidates(const DenseSmem<R>& sm, const DenseTables<R>& tb, int base, int lane, int j, float4 pj,
                                                     R tau, bool* tangent) {
  bool hit = false, tg = false;
  for (int r = 1; r <= 16; ++r) {
    const int i = base + ((lane + r) & 31);
    if ((r < 16 || lane < 16) && broad_overlap(sm.bp[i], pj)) hit |= dense_pair(sm, tb, i < j ? i : j, i < j ? j : i, tau, tg);
  }
  *tangent |= tg;
  return hit;
}

// Warp-uniform per-env scalars.
struct DenseEnv {
  int32_t t_ep, episode, winner;
  uint8_t done;
  // lane-private, bit k = body lane + 32 k:
  uint32_t busy;      // its crossing agent has a waypoint or a target orientation (state words worth reading)
  uint32_t v_dirty;   // its velocity changed since it was staged
  uint32_t h_dirty;   // its heading (theta, cos, sin) changed since it was staged
  bool moved;         // some transition ran since the bodies were staged
};

// Bodies of env e, global -> shared, by their lanes (lane-private: the same lane reads them back).  Loads go out in
// batches of four bodies before any of them is used: 24 independent loads in flight per lane instead of one memory
// latency per body.  Also finds which crossing agents are mid-crossing (DenseEnv::busy).
template <typename R, bool AGENTS>
__device__ __noinline__ void dense_stage_env(const DevScenario<R>& sc, const EnvBuffers<R>& buf, int64_t e, int lane,
                                                const DenseSmem<R>& sm, DenseEnv& env) {
  __builtin_assume(__isShared(sm.bp)); __builtin_assume(__isShared(sm.tu)); __builtin_assume(__isShared(sm.x)); __builtin_assume(__isShared(sm.y));
  __builtin_assume(__isShared(sm.v)); __builtin_assume(__isShared(sm.c)); __builtin_assume(__isShared(sm.s));
  __builtin_assume(__isShared(sm.th)); __builtin_assume(__isShared(sm.meta));
  const int M = sc.n_bodies;
  const int64_t n = buf.n;
  env.busy = 0; env.v_dirty = 0; env.h_dirty = 0; env.moved = false;
  for (int b0 = lane, k0 = 0; b0 < M; b0 += 128, k0 += 4) {
    R tmp[4][8];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int b = b0 + 32 * u;
      if (b < M) {
#pragma unroll
        for (int w = 0; w < 4; ++w) tmp[u][w] = buf.state[((int64_t)b * 4 + w) * n + e];
        tmp[u][4] = buf.cs[((int64_t)b * 2 + 0) * n + e];
        tmp[u][5] = buf.cs[((int64_t)b * 2 + 1) * n + e];
        const int agent = dm_agent(sm.meta[b]);
        tmp[u][6] = tmp[u][7] = nan_<R>();
        if (AGENTS && (agent == CAV_AGENT_RANDOM_CONSTRAINED || agent == CAV_AGENT_PROXIMITY)) {
          tmp[u][6] = buf.agent[((int64_t)b * CAV_AGENT_WORDS + 1) * n + e];
          tmp[u][7] = buf.agent[((int64_t)b * CAV_AGENT_WORDS + 3) * n + e];
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int b = b0 + 32 * u;
      if (b < M) {
        sm.x[b] = tmp[u][0]; sm.y[b] = tmp[u][1]; sm.v[b] = tmp[u][2]; sm.th[b] = tmp[u][3]; sm.c[b] = tmp[u][4]; sm.s[b] = tmp[u][5];
        if (!isnan_(tmp[u][6]) || !isnan_(tmp[u][7])) env.busy |= 1u << (k0 + u);
      }
    }
  }
  __syncwarp();
}

// Shared -> global for what changed since staging.
template <typename R>
__device__ __noinline__ void dense_writeback_env(const DevScenario<R>& sc, const EnvBuffers<R>& buf, int64_t e, int lane,
                                                    const DenseSmem<R>& sm, DenseEnv& env) {
  __builtin_assume(__isShared(sm.bp)); __builtin_assume(__isShared(sm.tu)); __builtin_assume(__isShared(sm.x)); __builtin_assume(__isShared(sm.y));
  __builtin_assume(__isShared(sm.v)); __builtin_assume(__isShared(sm.c)); __builtin_assume(__isShared(sm.s));
  __builtin_assume(__isShared(sm.th)); __builtin_assume(__isShared(sm.meta));
  if (!env.moved) return;
  const int M = sc.n_bodies;
  const int64_t n = buf.n;
  for (int b = lane, k = 0; b < M; b += 32, ++k) {
    if (sm.meta[b] & DM_PELICAN) continue;   // its light state is written when it changes
    buf.state[((int64_t)b * 4 + 0) * n + e] = sm.x[b];
    buf.state[((int64_t)b * 4 + 1) * n + e] = sm.y[b];
    if (env.v_dirty >> k & 1u) buf.state[((int64_t)b * 4 + 2) * n + e] = sm.v[b];
    if (env.h_dirty >> k & 1u) {
      buf.state[((int64_t)b * 4 + 3) * n + e] = sm.th[b];
      buf.cs[((int64_t)b * 2 + 0) * n + e] = sm.c[b];
      buf.cs[((int64_t)b * 2 + 1) * n + e] = sm.s[b];
    }
  }
  env.v_dirty = 0; env.h_dirty = 0; env.moved = false;
}

// CAVEnv.reset for env e by its warp (reset_env of transition.cuh, lane-strided over bodies).
template <typename R>
__device__ __noinline__ void dense_reset_env(const DevScenario<R>& sc, const DenseTables<R>& tb, const EnvBuffers<R>& buf,
                                                const R* init, int64_t e, int lane, DenseEnv& env) {
  const int M = sc.n_bodies;
  const int64_t n = buf.n;
  env.episode += 1;
  for (int b = lane; b < M; b += 32) {
    const DenseBody<R>& body = tb.bodies[b];
    const int32_t mt = body.meta;
    R st[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) st[c] = body.init[c];
    if (init) {
#pragma unroll
      for (int c = 0; c < 4; ++c) st[c] = init[((int64_t)b * 4 + c) * n + e];
    } else if ((mt & DM_SPAWN) && body.spawn_id >= 0) {
      double u[5];
      if (buf.spawn_override) {
#pragma unroll
        for (int c = 0; c < 5; ++c) u[c] = buf.spawn_override[((int64_t)b * 5 + c) * n + e];
      } else {
        double w[2];
        const uint64_t g = (uint64_t)(buf.shard + e);
        draw_block(buf.seed, g, b, KIND_SPAWN0, (uint32_t)env.episode, 0u, w); u[0] = w[0]; u[1] = w[1];
        draw_block(buf.seed, g, b, KIND_SPAWN1, (uint32_t)env.episode, 0u, w); u[2] = w[0]; u[3] = w[1];
        draw_block(buf.seed, g, b, KIND_SPAWN2, (uint32_t)env.episode, 0u, w); u[4] = w[0];
      }
      spawn_body(buf.spawns[body.spawn_id], u, st);
    }
    R c = R(1), s = R(0);
    if (!(mt & DM_PELICAN)) heading_cs(sc, st[3], c, s);
#pragma unroll
    for (int w = 0; w < 4; ++w) buf.state[((int64_t)b * 4 + w) * n + e] = st[w];
    buf.action[((int64_t)b * 2 + 0) * n + e] = R(0);
    buf.action[((int64_t)b * 2 + 1) * n + e] = R(0);
    buf.cs[((int64_t)b * 2 + 0) * n + e] = c;
    buf.cs[((int64_t)b * 2 + 1) * n + e] = s;
#pragma unroll
    for (int w = 0; w < CAV_AGENT_WORDS; ++w) buf.agent[((int64_t)b * CAV_AGENT_WORDS + w) * n + e] = nan_<R>();
    buf.liveness[(int64_t)b * n + e] = 0;
  }
  env.t_ep = 0;
  env.done = 0;
  env.winner = -1;
  if (lane == 0) {
    buf.t_ep[e] = 0; buf.done[e] = 0; buf.winner[e] = -1; buf.episode[e] = env.episode;
  }
  __syncwarp();
}

// Exact stage of one candidate pair (i < j): the test sequence of transition.cuh's all-pairs loop.  Out of line: it runs a
// few times per env-step and is referenced from six places of the sweep, which must stay small enough for the
// instruction cache.
template <typename R>
__device__ __noinline__ bool dense_pair(const DenseSmem<R>& sm, const DenseTables<R>& tb, int i, int j, R tau, bool& tangent) {
  __builtin_assume(__isShared(sm.bp)); __builtin_assume(__isShared(sm.tu)); __builtin_assume(__isShared(sm.x)); __builtin_assume(__isShared(sm.y));
  __builtin_assume(__isShared(sm.v)); __builtin_assume(__isShared(sm.c)); __builtin_assume(__isShared(sm.s));
  __builtin_assume(__isShared(sm.th)); __builtin_assume(__isShared(sm.meta));
  const DevType<R>& ki = tb.types[sm.meta[i] & DM_TYPE_MASK];
  const DevType<R>& kj = tb.types[sm.meta[j] & DM_TYPE_MASK];
  R exi, eyi, exj, eyj;
  box_extents(sm.c[i], sm.s[i], ki.hl, ki.hw, exi, eyi);
  box_extents(sm.c[j], sm.s[j], kj.hl, kj.hw, exj, eyj);
  const bool apart = rabs(sm.x[i] - sm.x[j]) - (exi + exj) > tau || rabs(sm.y[i] - sm.y[j]) - (eyi + eyj) > tau;
  if (apart) return false;
  return margin_hit(box_margin(dense_box(sm, ki, i), dense_box(sm, kj, j)), tau, tangent);
}

// One joint transition of env e by its warp.  `actions` = this step's [M][2][N] rows (nullable when every body has an
// on-device agent).  Returns with env updated; outputs written through `io`.
// RECORD (dense_record_kernel): `act_rec` (nullable) receives this step's [M][2][N] joint action row.
template <typename R, bool AGENTS, bool RECORD = false>
__device__ __forceinline__ void dense_transition(const DevScenario<R>& sc, const DenseTables<R>& tb, const EnvBuffers<R>& buf,
                                                 const StepIO<R>& io, const R* actions, int64_t e, int64_t t_global, int lane,
                                                 const DenseSmem<R>& sm, DenseEnv& env, const bool phase_sync, R* act_rec = nullptr) {
  const int M = sc.n_bodies, Mp = (M + 31) & ~31;
  const int64_t n = buf.n;
  const R tau = sc.tau, dt = sc.dt;
  bool tangent = false;
  // the staging arrays reach this function through a struct of generic pointers: tell the compiler they are shared memory
  // (LDS / STS instead of generic LD / ST in the pair sweep)
  __builtin_assume(__isShared(sm.bp)); __builtin_assume(__isShared(sm.tu)); __builtin_assume(__isShared(sm.x)); __builtin_assume(__isShared(sm.y));
  __builtin_assume(__isShared(sm.v)); __builtin_assume(__isShared(sm.c)); __builtin_assume(__isShared(sm.s));
  __builtin_assume(__isShared(sm.th)); __builtin_assume(__isShared(sm.meta));

  // ---- action_space.contains for the replayed actions (environment.py:120): before any mutation
  if (!AGENTS || tb.has_external) {
    bool valid = true;
    for (int b = lane; b < M; b += 32) {
      const int32_t mt = sm.meta[b];
      if (AGENTS && dm_agent(mt) != CAV_AGENT_EXTERNAL) continue;
      const R a0 = actions[((int64_t)b * 2 + 0) * n + e], a1 = actions[((int64_t)b * 2 + 1) * n + e];
      if (mt & DM_PELICAN) {
        valid = valid && (a0 == R(0) || a0 == R(1) || a0 == R(2) || a0 == R(3));
      } else {
        const DevType<R>& k = tb.types[mt & DM_TYPE_MASK];
        valid = valid && (a0 >= k.amin && a0 <= k.amax && a1 >= k.smin && a1 <= k.smax);
      }
    }
    if (!__all_sync(kFull, valid)) {
      for (int b = lane; b < M; b += 32) {
        if (io.reward_out) io.reward_out[(int64_t)b * n + e] = R(0);
        if (io.state_out && io.state_out != buf.state) {
          io.state_out[((int64_t)b * 4 + 0) * n + e] = sm.x[b];
          io.state_out[((int64_t)b * 4 + 1) * n + e] = sm.y[b];
          io.state_out[((int64_t)b * 4 + 2) * n + e] = sm.v[b];
          io.state_out[((int64_t)b * 4 + 3) * n + e] = sm.th[b];
        }
      }
      if (lane == 0) {
        buf.err[e] = 1;
        if (io.done_out) io.done_out[e] = 0;
        if (io.winner_out) io.winner_out[e] = -1;
        if (io.tangent_out) io.tangent_out[e] = 0;
      }
      return;
    }
  }

  const R ego_pre_x = sm.x[0], ego_pre_y = sm.y[0];   // ProximityAgent looks at the ego BEFORE it moves
  __syncwarp();

  // ---- agents, body.step (environment.py:122-123), process_feedback (simulation.py:86-87: a function of the body's own
  //      new state only).  The bodies live in shared memory; a replayed action is fetched one iteration ahead; an idle
  //      crossing agent (DenseEnv::busy clear) that is not triggered touches no memory at all.
  R ego_steer = R(0), ego_v = R(0);
  bool agent_invalid = false;
  R w0_next = R(0), w1_next = R(0);
  auto prefetch = [&](int b) {
    if (b >= M) return;
    if (!AGENTS || dm_agent(sm.meta[b]) == CAV_AGENT_EXTERNAL) {
      w0_next = actions[((int64_t)b * 2 + 0) * n + e]; w1_next = actions[((int64_t)b * 2 + 1) * n + e];
    }
  };
  prefetch(lane);
  env.moved = true;
  for (int b = lane, kbit = 0; b < Mp; b += 32, ++kbit) {
    if (b >= M) { sm.bp[b] = broad_absent(); continue; }
    const int32_t mt = sm.meta[b];
    const int agent = dm_agent(mt);
    const bool pelican = (mt & DM_PELICAN) != 0;
    const DevType<R>& k = tb.types[mt & DM_TYPE_MASK];
    const R w0 = w0_next, w1 = w1_next;
    prefetch(b + 32);
    const R v_old = sm.v[b];
    R st[4] = {sm.x[b], sm.y[b], v_old, sm.th[b]};
    R a0 = R(0), a1 = R(0);
    R ag[CAV_AGENT_WORDS];
    bool ag_dirty = false, ag_loaded = false;
    const bool crossing = AGENTS && (agent == CAV_AGENT_RANDOM_CONSTRAINED || agent == CAV_AGENT_PROXIMITY);
    if (!AGENTS || agent == CAV_AGENT_EXTERNAL) {
      a0 = w0; a1 = w1;
    } else {
      const DenseBody<R>& body = tb.bodies[b];
      R held0 = R(0), held1 = R(0);
      if (agent == CAV_AGENT_RANDOM) {  // holds its last action (template.py:52-56)
        held0 = a0 = buf.action[((int64_t)b * 2 + 0) * n + e]; held1 = a1 = buf.action[((int64_t)b * 2 + 1) * n + e];
      }
      double u[CAV_DRAWS] = {0.0, 0.0, 0.0};
      if (agent == CAV_AGENT_RANDOM || agent == CAV_AGENT_RANDOM_CONSTRAINED) {
        if (buf.uni_override) {
#pragma unroll
          for (int c = 0; c < CAV_DRAWS; ++c) u[c] = buf.uni_override[((int64_t)b * CAV_DRAWS + c) * n + e];
        } else {
          draw_block(buf.seed, (uint64_t)(buf.shard + e), b, KIND_AGENT0, (uint32_t)env.episode, (uint32_t)env.t_ep, u);
        }
      }
      if (agent == CAV_AGENT_NOOP) {
        a0 = R(0); a1 = R(0);
      } else if (agent == CAV_AGENT_RANDOM) {
        if (u[0] < body.epsilon)
          dense_random_sample(buf, k, e, b, pelican, (uint32_t)env.episode, (uint32_t)env.t_ep, u[1], u[2], &a0, &a1);
      } else if (crossing) {
        const bool trigger = agent == CAV_AGENT_RANDOM_CONSTRAINED
                                 ? u[0] < body.epsilon
                                 : point_distance(st[0], st[1], ego_pre_x, ego_pre_y) < body.threshold;
        // An idle agent (no waypoint, no target orientation) that is not triggered chooses steering 0 and its
        // process_feedback is a no-op (pedestrian.py:36-69): its state words are read only when a crossing starts or is
        // under way.
        a0 = R(0); a1 = R(0);
        if (trigger || (env.busy >> kbit & 1u)) {
#pragma unroll
          for (int w = 0; w < CAV_AGENT_WORDS; ++w) ag[w] = buf.agent[((int64_t)b * CAV_AGENT_WORDS + w) * n + e];
          ag_loaded = true;
          a1 = choose_crossing_action(sc, k, st, ag, trigger, ag_dirty);
        } else {
          a1 = rmin(k.smax, rmax(k.smin, R(0)));   // make_steering_action with no target (dynamic_body.py:33-49)
        }
      }
      if (pelican) agent_invalid |= !(a0 == R(0) || a0 == R(1) || a0 == R(2) || a0 == R(3));
      else agent_invalid |= !(a0 >= k.amin && a0 <= k.amax && a1 >= k.smin && a1 <= k.smax);
      if (buf.log_actions || (agent == CAV_AGENT_RANDOM && (a0 != held0 || a1 != held1))) {
        buf.action[((int64_t)b * 2 + 0) * n + e] = a0; buf.action[((int64_t)b * 2 + 1) * n + e] = a1;
      }
    }
    if (pelican) {  // PelicanCrossing.step (bodies.py:450-461): the light state lives in the x slot
      const R light = st[0];
      if (a0 == R(1)) st[0] = R(0);
      else if (a0 == R(2)) st[0] = R(1);
      else if (a0 == R(3)) st[0] = R(2);
      if (!(st[0] == light)) buf.state[((int64_t)b * 4) * n + e] = st[0];
      sm.x[b] = st[0];
      sm.bp[b] = broad_absent();
    } else {
      R c = sm.c[b], s = sm.s[b], snapped;
      const bool turned = body_step<R, true>(k, st, a0, a1, dt, c, s, snapped);
      if (b == 0) { ego_steer = snapped; ego_v = st[2]; }
      if (ag_loaded) crossing_feedback(sc, st, ag, ag_dirty);
      sm.x[b] = st[0]; sm.y[b] = st[1];
      if (!(st[2] == v_old)) { sm.v[b] = st[2]; env.v_dirty |= 1u << kbit; }
      if (turned) { sm.c[b] = c; sm.s[b] = s; sm.th[b] = st[3]; env.h_dirty |= 1u << kbit; }
      R ex, ey;
      box_extents(c, s, k.hl, k.hw, ex, ey);
      sm.bp[b] = broad_entry(st[0], st[1], ex, ey, tau);
    }
    if (ag_loaded && ag_dirty) {
#pragma unroll
      for (int w = 0; w < CAV_AGENT_WORDS; ++w) buf.agent[((int64_t)b * CAV_AGENT_WORDS + w) * n + e] = ag[w];
      if (!isnan_(ag[1]) || !isnan_(ag[3])) env.busy |= 1u << kbit; else env.busy &= ~(1u << kbit);
    }
    if (io.state_out && io.state_out != buf.state) {
#pragma unroll
      for (int w = 0; w < 4; ++w) io.state_out[((int64_t)b * 4 + w) * n + e] = st[w];
    }
    if constexpr (RECORD) {
      if (act_rec) { act_rec[((int64_t)b * 2 + 0) * n + e] = a0; act_rec[((int64_t)b * 2 + 1) * n + e] = a1; }
    }
  }
  __syncwarp();
  ego_steer = __shfl_sync(kFull, ego_steer, 0);
  ego_v = __shfl_sync(kFull, ego_v, 0);
  if (AGENTS && __any_sync(kFull, agent_invalid) && lane == 0) buf.err[e] = 1;   // cannot happen with the stock agents

  // ---- termination cascade (environment.py:148-206)
  if (phase_sync) { __syncwarp(); __syncthreads(); }   // (launch-uniform) the warps of the CTA enter each phase together: shared instruction fetches
  const DevType<R>& k0 = tb.types[sm.meta[0] & DM_TYPE_MASK];
  const R x0 = sm.x[0], y0 = sm.y[0], c0 = sm.c[0], s0 = sm.s[0];
  R ex0, ey0;
  box_extents(c0, s0, k0.hl, k0.hw, ex0, ey0);
  const R W = sc.W;
  bool terminate = false, win_ego = false;
  int win_tester = -1;
  {
    const R margin = (x0 - ex0) - W;  // all four ego corners beyond the viewer width
    if (margin > -tau) {
      if (margin < tau) tangent = true;
      if (margin > R(0)) { terminate = true; win_ego = true; }
    }
  }
  if (!terminate && sc.collisions == CAV_COLLISIONS_ALL) {
    bool hit = false;
    // dynamic vs dynamic, two levels.
    // Tiles: the union of the entries of every 32-body tile (four warp-wide REDUX each).  A whole tile of i's is skipped
    // when no lane's body overlaps its union — exact, never changes a result; how much it saves depends on how
    // spatially coherent the body order is (dense_traffic.py orders bodies along the road).
    // Bodies: a lane owns two bodies per pass, jA = jt + lane and jB = jt + 32 + lane, and meets every i below them; the
    // entry of body i is one broadcast LDS.128 shared by both tests.
    // Candidates are rare (a few per env-step): eight tests are folded into one vote, and only a vote that fires looks at
    // them one by one.
    for (int tile = 0; tile * 32 < Mp; ++tile) {
      const float4 p = sm.bp[tile * 32 + lane];
      const int x0 = __reduce_min_sync(kFull, ordered_int(p.x)), x1 = __reduce_max_sync(kFull, ordered_int(p.y));
      const int y0 = __reduce_min_sync(kFull, ordered_int(p.z)), y1 = __reduce_max_sync(kFull, ordered_int(p.w));
      if (lane == 0) sm.tu[tile] = make_float4(ordered_float(x0), ordered_float(x1), ordered_float(y0), ordered_float(y1));
    }
    __syncwarp();
    for (int jt = 0; jt < Mp; jt += 64) {
      const int jA = jt + lane, jB = jt + 32 + lane;
      const bool haveB = jt + 32 < Mp;
      const float4 pA = sm.bp[jA], pB = haveB ? sm.bp[jB] : broad_absent();
      // every body of tiles [lo, hi) against this lane's jA and jB (all of them lie below both): broadcast reads
      auto sweep = [&](int lo, int hi, const bool useA) {
        for (int i0 = lo; i0 < hi; i0 += 8) {
          bool any = false;
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float4 pi = sm.bp[i0 + u];
            if (useA) any |= broad_overlap(pi, pA);
            any |= broad_overlap(pi, pB);
          }
          if (__any_sync(kFull, any)) {
            if (any) hit |= dense_sweep_candidates(sm, tb, i0, jA, jB, useA, pA, pB, tau, &tangent);
          }
        }
      };
      // the pairs INSIDE one tile, by rotation: in round r lane l meets the body of lane (l + r) mod 32, so rounds 1..15 meet
      // every unordered pair once and round 16 meets the remaining sixteen (lanes 0..15 only) — no index compare per test
      auto within = [&](int base, const float4& pj, int j) {
        bool any = false;
#pragma unroll
        for (int r = 1; r <= 16; ++r) {
          const float4 pi = sm.bp[base + ((lane + r) & 31)];
          any |= broad_overlap(pi, pj) && (r < 16 || lane < 16);
        }
        if (__any_sync(kFull, any)) {
          if (any) hit |= dense_within_candidates(sm, tb, base, lane, j, pj, tau, &tangent);
        }
      };
      for (int it = 0; it < jt; it += 32) {                      // tiles wholly below both of this pass's tiles
        const float4 ui = sm.tu[it >> 5];
        if (__any_sync(kFull, broad_overlap(ui, pA) || broad_overlap(ui, pB))) sweep(it, it + 32, true);
      }
      within(jt, pA, jA);
      if (haveB) {
        sweep(jt, jt + 32, false);                               // all of tile A is below tile B
        within(jt + 32, pB, jB);
      }
    }
    // dynamic vs static collidables (traffic lights, obstacle: environment.py:94-101)
    for (int i = lane; i < M; i += 32) {
      const int32_t mt = sm.meta[i];
      if (mt & DM_PELICAN) continue;
      const DevType<R>& ki = tb.types[mt & DM_TYPE_MASK];
      R exi, eyi;
      box_extents(sm.c[i], sm.s[i], ki.hl, ki.hw, exi, eyi);
      const R px = sm.x[i], py = sm.y[i];
      for (int s = 0; s < sc.n_statics; ++s) {
        const Aabb<R> sb = sc.static_bb[s];
        const bool apart = (px - exi) - sb.x1 > tau || sb.x0 - (px + exi) > tau || (py - eyi) - sb.y1 > tau || sb.y0 - (py + eyi) > tau;
        if (!apart) {
          if (sc.static_rect[s]) hit |= margin_hit(box_margin(dense_box(sm, ki, i), sc.static_box[s]), tau, tangent);
          else hit |= geo_hit(sat_pose_quad(dense_pose(sm, ki, i), &sc.quads[CAV_MAX_ROADS + s], tau), tangent);
        }
      }
    }
    terminate = __any_sync(kFull, hit);
  }
  if (!terminate && sc.offroad) {   // ego only: evaluated by every lane alike
    bool on_road = false;
    for (int r = 0; r < sc.n_roads; ++r) {
      const Aabb<R> rd = sc.road_bb[r];
      const bool apart = (x0 - ex0) - rd.x1 > tau || rd.x0 - (x0 + ex0) > tau || (y0 - ey0) - rd.y1 > tau || rd.y0 - (y0 + ey0) > tau;
      if (!apart) {
        if (sc.road_rect[r]) on_road |= margin_hit(box_margin(dense_box(sm, k0, 0), sc.road_box[r]), tau, tangent);
        else on_road |= geo_hit(sat_pose_quad(dense_pose(sm, k0, 0), &sc.quads[r], tau), tangent);
      }
    }
    terminate = !on_road;
  }
  if (!terminate && (sc.collisions == CAV_COLLISIONS_EGO || sc.zones)) {
    EgoFrame<R> f;
    f.x = x0; f.y = y0; f.c = c0; f.s = s0; f.hl = k0.hl; f.hw = k0.hw;
    f.bd = (ego_v * ego_v) * k0.inv_2brake;
    f.td = f.bd + ego_v * R(0.675);
    f.have = !(f.td == R(0)) && (ego_steer == R(0));
    const bool ego_mode = sc.collisions == CAV_COLLISIONS_EGO;
    // The reference walks the pedestrians in index order: ego box / braking zone for each (environment.py:183-193), and
    // the reaction zone only while nothing has hit and nobody has won yet (:195-206).  In parallel: every lane evaluates
    // its pedestrians, then the first hit and the first winner are warp minima, and a reaction-zone decision counts
    // towards the near-tangent flag only if the sequential walk would have made it.
    unsigned first_hit = 0xFFFFFFFFu, first_win = 0xFFFFFFFFu;
    uint32_t near_bits = 0;   // bit k: the reaction-zone margin of body lane + 32 k is within tau
    for (int b = lane; b < M; b += 32) {
      const int32_t mt = sm.meta[b];
      if (b == 0 || !(mt & DM_PEDESTRIAN) || (mt & DM_PELICAN)) continue;
      const DevType<R>& k = tb.types[mt & DM_TYPE_MASK];
      const EgoMargins<R> m = ego_margins(f, sm.x[b], sm.y[b], sm.c[b], sm.s[b], k.hl, k.hw, tau);
      if (m.all_clear) continue;
      if (ego_mode) {
        bool h = margin_hit(m.ego, tau, tangent);
        if (!h && f.have) h = margin_hit(m.braking, tau, tangent);
        if (h && (unsigned)b < first_hit) first_hit = (unsigned)b;
      }
      if (sc.zones && f.have) {
        if (rabs(m.reaction) < tau) near_bits |= 1u << (b >> 5);
        if (!(m.reaction > R(0)) && (unsigned)b < first_win) first_win = (unsigned)b;
      }
    }
    first_hit = __reduce_min_sync(kFull, first_hit);
    // The walk tests the reaction zone for body b iff nothing has hit among bodies <= b (b < first_hit) and nobody before
    // b has won (b <= first_win).  A lane's lowest winner is its only candidate: if that one is not below first_hit,
    // none of its later ones is.
    first_win = __reduce_min_sync(kFull, first_win < first_hit ? first_win : 0xFFFFFFFFu);
    for (int b = lane, kbit = 0; b < M; b += 32, ++kbit)
      if ((near_bits >> kbit & 1u) && (unsigned)b < first_hit && (unsigned)b <= first_win) tangent = true;
    if (first_hit != 0xFFFFFFFFu) { terminate = true; win_tester = -1; }
    else { win_tester = first_win == 0xFFFFFFFFu ? -1 : (int)first_win; terminate = win_tester >= 0; }
  }

  // ---- rewards, liveness (environment.py:131-146), terminal rewards and winner (:208-220)
  if (phase_sync) { __syncwarp(); __syncthreads(); }
  const R cstep = sc.cost_step;
  const R ego_rel = rmax(R(0), rmin(R(1), (W - x0) * sc.inv_W));
  const bool terminal = terminate || t_global == sc.max_timesteps - 1;
  for (int b = lane; b < M; b += 32) {
    R rb = R(0);
    if (b == 0) {
      const R voff = rabs(ego_v - sc.v_maint) * sc.inv_v_off;
      rb -= voff * cstep;
      rb += (R(1) - ego_rel) * cstep;
      if (terminal) rb += win_ego ? sc.reward_win : (win_tester >= 0 ? -sc.reward_win : sc.reward_draw);
    } else {
      const int32_t mt = sm.meta[b];
      R p = R(0);
      if (mt & DM_PELICAN) {
        p = tb.bodies[b].static_share;
      } else {
        const DevType<R>& k = tb.types[mt & DM_TYPE_MASK];
        R ex, ey;
        box_extents(sm.c[b], sm.s[b], k.hl, k.hw, ex, ey);
        for (int r = 0; r < sc.n_roads; ++r) {
          const R q = dense_road_share(sc, sm, k, b, r, ex, ey, tau, tangent);
          if (r == 0 || q > p) p = q;
        }
      }
      rb -= p * cstep;
      rb += ego_rel * cstep;
      if (p > R(0.5)) atomicAdd(&buf.liveness[(int64_t)b * n + e], 1);   // result unused: a fire-and-forget RED
      if (terminal) rb += win_ego ? -sc.reward_win : (win_tester < 0 ? sc.reward_draw : (win_tester == b ? sc.reward_win : sc.reward_draw));
    }
    if (io.reward_out) io.reward_out[(int64_t)b * n + e] = rb;
  }
  tangent = __any_sync(kFull, tangent);

  int32_t winner = -1;
  if (terminal) { if (win_ego) winner = 0; else if (win_tester >= 0) winner = win_tester; }
  env.t_ep += 1;
  env.winner = winner;
  if (terminate) env.done = 1;
  else if (env.t_ep >= sc.max_timesteps) env.done = 2;
  if (lane == 0) {
    buf.t_ep[e] = env.t_ep;
    if (env.done) { buf.done[e] = env.done; buf.winner[e] = env.winner; }
    if (tangent) count_tangent(buf.stats);
    if (io.done_out) io.done_out[e] = terminate ? 1 : 0;
    if (io.winner_out) io.winner_out[e] = winner;
    if (io.tangent_out) io.tangent_out[e] = tangent ? 1 : 0;
  }
  if (env.done) {   // reporting.analyse_episode (reporting.py:227-243)
    __syncwarp();   // liveness increments of this step are visible to the lanes that sum them
    long long sum = 0;
    for (int b = lane; b < M; b += 32) if (b > 0) sum += buf.liveness[(int64_t)b * n + e];
    sum = (long long)warp_sum((unsigned long long)sum);
    if (lane == 0) {
      EpisodeLog log{buf.ep_log, buf.ep_log_count, buf.ep_log_capacity, buf.shard + e, env.episode};
      if (buf.ep_log && !AGENTS) log.episode = buf.episode[e];
      score_episode<R, 1>(buf.stats, env.t_ep, env.winner, sum, log);
    }
  }
}

template <typename R>
__device__ __forceinline__ StepIO<R> io_at(const StepIO<R>& io, int64_t t, int64_t m, int64_t n) {
  const int64_t per_env = t * n;
  StepIO<R> at;
  at.actions = io.actions ? io.actions + per_env * m * 2 : nullptr;
  at.state_out = io.state_out ? io.state_out + per_env * m * 4 : nullptr;
  at.reward_out = io.reward_out ? io.reward_out + per_env * m : nullptr;
  at.done_out = io.done_out ? io.done_out + per_env : nullptr;
  at.winner_out = io.winner_out ? io.winner_out + per_env : nullptr;
  at.tangent_out = io.tangent_out ? io.tangent_out + per_env : nullptr;
  return at;
}

// traj != 0: io.* are [T] slabs (cavgym_replay); otherwise the same buffers are used by every step.
// CAV_DENSE_SYNC: 0 = warps run free, 1 = the warps of a CTA are re-aligned once per step, 2 = also at the phase boundaries
// inside the step (rollouts with on-device agents only).  The kernel is bound by instruction fetch (DESIGN 4.4): warps that
// walk the step code together share the fetches.  Measured on config C4 (100,000 envs x 320 bodies), M env-steps/s:
// pedestrians' eps = 2e-4: 22.5 (0) -> 26.6 (1) -> 27.6 (2); eps = 0.01 (the reference's): 13.4 (1) -> 16.2 (2).
#ifndef CAV_DENSE_SYNC
#define CAV_DENSE_SYNC 2
#endif
template <typename R, bool AGENTS>
__global__ void __launch_bounds__(kDenseWarps * 32, CAV_DENSE_MIN_BLOCKS) dense_kernel(const __grid_constant__ DevScenario<R> sc,
                                                                 const __grid_constant__ DenseTables<R> tb,
                                                                 const __grid_constant__ EnvBuffers<R> buf,
                                                                 const __grid_constant__ StepIO<R> io, int64_t t_global, int n_steps,
                                                                 int auto_reset, int traj) {
  extern __shared__ __align__(16) unsigned char dense_smem[];
  const int M = sc.n_bodies, Mp = (M + 31) & ~31;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float4* bp_all = reinterpret_cast<float4*>(dense_smem);
  R* geo_all = reinterpret_cast<R*>(dense_smem + sizeof(float4) * kDenseWarps * (Mp + kDenseTiles));
  int32_t* meta = reinterpret_cast<int32_t*>(geo_all + (size_t)kDenseWarps * 6 * Mp);
  for (int b = threadIdx.x; b < Mp; b += blockDim.x) meta[b] = b < M ? tb.bodies[b].meta : (int32_t)DM_ABSENT;
  __syncthreads();
  const int64_t e = buf.lo + (int64_t)blockIdx.x * kDenseWarps + warp;
  // Barriers inside the step need every warp of the CTA to run every step's transition: on-device agents for every body and
  // auto-reset (no frozen envs, no invalid-action exit).  Launch-uniform.
  const bool phase_sync = CAV_DENSE_SYNC >= 2 && AGENTS && auto_reset && !tb.has_external;
  if (e >= buf.hi) {   // a warp of the ragged last CTA without an env: keep the barriers below balanced
    if (CAV_DENSE_SYNC) for (int t = 0; t < n_steps * (phase_sync ? 3 : 1); ++t) __syncthreads();
    return;
  }
  DenseSmem<R> sm;
  sm.bp = bp_all + (size_t)warp * (Mp + kDenseTiles);
  sm.tu = sm.bp + Mp;
  R* geo = geo_all + (size_t)warp * 6 * Mp;
  sm.x = geo; sm.y = geo + Mp; sm.v = geo + 2 * Mp; sm.c = geo + 3 * Mp; sm.s = geo + 4 * Mp; sm.th = geo + 5 * Mp;
  sm.meta = meta;
  const int64_t n = buf.n;

  DenseEnv env;
  env.done = buf.done[e];
  env.t_ep = buf.t_ep[e];
  env.winner = env.done ? buf.winner[e] : -1;
  env.episode = AGENTS ? buf.episode[e] : 0;
  // The bodies are staged ONCE per launch and stay in shared memory across the fused steps; what changed goes back to
  // global memory at the end of the launch (or is discarded when the episode ends and the env is reset in-kernel).
  dense_stage_env<R, AGENTS>(sc, buf, e, lane, sm, env);
  for (int t = 0; t < n_steps; ++t) {
    if (CAV_DENSE_SYNC) __syncthreads();   // the warps of a CTA walk the (instruction-fetch bound) step code together
    const StepIO<R> at = traj ? io_at(io, (int64_t)t, (int64_t)M, n) : io;
    if (env.done && AGENTS && auto_reset) {
      dense_reset_env<R>(sc, tb, buf, nullptr, e, lane, env);
      dense_stage_env<R, AGENTS>(sc, buf, e, lane, sm, env);
    }
    if (env.done) {   // frozen until reset: reward 0, latched done / winner
      for (int b = lane; b < M; b += 32) {
        if (at.reward_out) at.reward_out[(int64_t)b * n + e] = R(0);
        if (at.state_out && at.state_out != buf.state) {
          at.state_out[((int64_t)b * 4 + 0) * n + e] = sm.x[b];
          at.state_out[((int64_t)b * 4 + 1) * n + e] = sm.y[b];
          at.state_out[((int64_t)b * 4 + 2) * n + e] = sm.v[b];
          at.state_out[((int64_t)b * 4 + 3) * n + e] = sm.th[b];
        }
      }
      if (lane == 0) {
        if (at.done_out) at.done_out[e] = env.done == 1 ? 1 : 0;
        if (at.winner_out) at.winner_out[e] = env.winner;
        if (at.tangent_out) at.tangent_out[e] = 0;
      }
      continue;
    }
    // (the actions pointer travels on its own: nvcc 12.9 folds `at.actions` back to `io.actions` when it is a member of the
    //  copied struct — seen in the PTX — while the output members are advanced correctly)
    const R* actions_t = io.actions;
    if (traj && actions_t) actions_t += (int64_t)t * M * 2 * n;
    dense_transition<R, AGENTS>(sc, tb, buf, at, actions_t, e, t_global + t, lane, sm, env, phase_sync);
    __syncwarp();
  }
  if (AGENTS && auto_reset && env.done) dense_reset_env<R>(sc, tb, buf, nullptr, e, lane, env);
  else dense_writeback_env<R>(sc, buf, e, lane, sm, env);
}

// cavgym_rollout_record on the warp-per-env path: dense_kernel<R, true>'s loop with traj = 1 (io = rec's state, reward, done,
// winner and tangent slabs) that also writes the observation before each step's transition, the executed action and t_ep
// after it; frozen rows get the frozen state, action 0 and timestep 0.  A kernel of its own so that dense_kernel's code
// stays as it is.
template <typename R>
__global__ void __launch_bounds__(kDenseWarps * 32, CAV_DENSE_MIN_BLOCKS) dense_record_kernel(const __grid_constant__ DevScenario<R> sc,
                                                                        const __grid_constant__ DenseTables<R> tb,
                                                                        const __grid_constant__ EnvBuffers<R> buf,
                                                                        const __grid_constant__ StepIO<R> io,
                                                                        const __grid_constant__ RolloutRecord<R> rec, int64_t t_global,
                                                                        int n_steps, int auto_reset) {
  extern __shared__ __align__(16) unsigned char dense_smem[];
  const int M = sc.n_bodies, Mp = (M + 31) & ~31;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float4* bp_all = reinterpret_cast<float4*>(dense_smem);
  R* geo_all = reinterpret_cast<R*>(dense_smem + sizeof(float4) * kDenseWarps * (Mp + kDenseTiles));
  int32_t* meta = reinterpret_cast<int32_t*>(geo_all + (size_t)kDenseWarps * 6 * Mp);
  for (int b = threadIdx.x; b < Mp; b += blockDim.x) meta[b] = b < M ? tb.bodies[b].meta : (int32_t)DM_ABSENT;
  __syncthreads();
  const int64_t e = buf.lo + (int64_t)blockIdx.x * kDenseWarps + warp;
  const bool phase_sync = CAV_DENSE_SYNC >= 2 && auto_reset && !tb.has_external;
  if (e >= buf.hi) {   // a warp of the ragged last CTA without an env: keep the barriers below balanced
    if (CAV_DENSE_SYNC) for (int t = 0; t < n_steps * (phase_sync ? 3 : 1); ++t) __syncthreads();
    return;
  }
  DenseSmem<R> sm;
  sm.bp = bp_all + (size_t)warp * (Mp + kDenseTiles);
  sm.tu = sm.bp + Mp;
  R* geo = geo_all + (size_t)warp * 6 * Mp;
  sm.x = geo; sm.y = geo + Mp; sm.v = geo + 2 * Mp; sm.c = geo + 3 * Mp; sm.s = geo + 4 * Mp; sm.th = geo + 5 * Mp;
  sm.meta = meta;
  const int64_t n = buf.n;

  DenseEnv env;
  env.done = buf.done[e];
  env.t_ep = buf.t_ep[e];
  env.winner = env.done ? buf.winner[e] : -1;
  env.episode = buf.episode[e];
  dense_stage_env<R, true>(sc, buf, e, lane, sm, env);
  for (int t = 0; t < n_steps; ++t) {
    if (CAV_DENSE_SYNC) __syncthreads();
    const StepIO<R> at = io_at(io, (int64_t)t, (int64_t)M, n);
    const int64_t row = (int64_t)t * n;
    R* act = rec.action ? rec.action + row * M * 2 : nullptr;
    if (env.done && auto_reset) {
      dense_reset_env<R>(sc, tb, buf, nullptr, e, lane, env);
      dense_stage_env<R, true>(sc, buf, e, lane, sm, env);
    }
    for (int b = lane; b < M; b += 32) {   // lane-private bodies: staged and stepped by this lane
      if (rec.observation) {
        R* o = rec.observation + row * M * 4;
        o[((int64_t)b * 4 + 0) * n + e] = sm.x[b];
        o[((int64_t)b * 4 + 1) * n + e] = sm.y[b];
        o[((int64_t)b * 4 + 2) * n + e] = sm.v[b];
        o[((int64_t)b * 4 + 3) * n + e] = sm.th[b];
      }
      if (env.done && act) { act[((int64_t)b * 2 + 0) * n + e] = R(0); act[((int64_t)b * 2 + 1) * n + e] = R(0); }
    }
    if (env.done) {   // frozen until reset: reward 0, latched done / winner, timestep 0
      for (int b = lane; b < M; b += 32) {
        if (at.reward_out) at.reward_out[(int64_t)b * n + e] = R(0);
        if (at.state_out) {
          at.state_out[((int64_t)b * 4 + 0) * n + e] = sm.x[b];
          at.state_out[((int64_t)b * 4 + 1) * n + e] = sm.y[b];
          at.state_out[((int64_t)b * 4 + 2) * n + e] = sm.v[b];
          at.state_out[((int64_t)b * 4 + 3) * n + e] = sm.th[b];
        }
      }
      if (lane == 0) {
        if (at.done_out) at.done_out[e] = env.done == 1 ? 1 : 0;
        if (at.winner_out) at.winner_out[e] = env.winner;
        if (at.tangent_out) at.tangent_out[e] = 0;
        if (rec.timestep) rec.timestep[row + e] = 0;
      }
      continue;
    }
    dense_transition<R, true, true>(sc, tb, buf, at, nullptr, e, t_global + t, lane, sm, env, phase_sync, act);
    if (lane == 0 && rec.timestep) rec.timestep[row + e] = env.t_ep;
    __syncwarp();
  }
  if (auto_reset && env.done) dense_reset_env<R>(sc, tb, buf, nullptr, e, lane, env);
  else dense_writeback_env<R>(sc, buf, e, lane, sm, env);
}

template <typename R>
__global__ void __launch_bounds__(kDenseWarps * 32) dense_reset_kernel(const __grid_constant__ DevScenario<R> sc,
                                                                       const __grid_constant__ DenseTables<R> tb,
                                                                       const __grid_constant__ EnvBuffers<R> buf, const uint8_t* mask,
                                                                       const R* init, int first_time) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t e = buf.lo + (int64_t)blockIdx.x * kDenseWarps + warp;
  if (e >= buf.hi || (mask && !mask[e])) return;
  DenseEnv env;
  env.episode = first_time ? -1 : buf.episode[e];
  if (!first_time && !buf.done[e] && lane == 0) {  // an unfinished episode is abandoned: keep its steps in the env-step total
    const int32_t t = buf.t_ep[e];
    if (t > 0) atomicAdd(&buf.stats[CAV_STAT_ENV_STEPS], (unsigned long long)t);
  }
  __syncwarp();
  dense_reset_env<R>(sc, tb, buf, init, e, lane, env);
  if (first_time && lane == 0) buf.err[e] = 0;
}

// ---------------------------------------------------------------- host-side launch table
template <typename R>
struct DenseLaunchers {
  // false = launch set-up failed (shared-memory opt-in)
  bool (*run)(const DevScenario<R>&, const DenseTables<R>&, const EnvBuffers<R>&, const StepIO<R>&, int64_t t_global, int n_steps,
              int auto_reset, int traj, bool agents, cudaStream_t);
  void (*reset)(const DevScenario<R>&, const DenseTables<R>&, const EnvBuffers<R>&, const uint8_t* mask, const R* init, int first_time,
                cudaStream_t);
  // cavgym_rollout_record; false = launch set-up failed
  bool (*rollout_record)(const DevScenario<R>&, const DenseTables<R>&, const EnvBuffers<R>&, const RolloutRecord<R>&, int64_t t_global,
                         int n_steps, int auto_reset, cudaStream_t);
};

template <typename R, bool AGENTS>
bool launch_dense_typed(const DevScenario<R>& sc, const DenseTables<R>& tb, const EnvBuffers<R>& buf, const StepIO<R>& io,
                        int64_t t_global, int n_steps, int auto_reset, int traj, cudaStream_t stream) {
  const size_t smem = dense_smem_bytes<R>(sc.n_bodies, kDenseWarps);
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(dense_kernel<R, AGENTS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return false;
  const unsigned grid = (unsigned)((buf.hi - buf.lo + kDenseWarps - 1) / kDenseWarps);
  dense_kernel<R, AGENTS><<<grid, kDenseWarps * 32, smem, stream>>>(sc, tb, buf, io, t_global, n_steps, auto_reset, traj);
  return true;
}

template <typename R>
bool launch_dense(const DevScenario<R>& sc, const DenseTables<R>& tb, const EnvBuffers<R>& buf, const StepIO<R>& io, int64_t t_global,
                  int n_steps, int auto_reset, int traj, bool agents, cudaStream_t stream) {
  return agents ? launch_dense_typed<R, true>(sc, tb, buf, io, t_global, n_steps, auto_reset, traj, stream)
                : launch_dense_typed<R, false>(sc, tb, buf, io, t_global, n_steps, auto_reset, traj, stream);
}

template <typename R>
bool launch_dense_record(const DevScenario<R>& sc, const DenseTables<R>& tb, const EnvBuffers<R>& buf, const RolloutRecord<R>& rec,
                         int64_t t_global, int n_steps, int auto_reset, cudaStream_t stream) {
  const size_t smem = dense_smem_bytes<R>(sc.n_bodies, kDenseWarps);
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(dense_record_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return false;
  const StepIO<R> io{nullptr, rec.state, rec.reward, rec.done, rec.winner, rec.tangent, 0};
  const unsigned grid = (unsigned)((buf.hi - buf.lo + kDenseWarps - 1) / kDenseWarps);
  dense_record_kernel<R><<<grid, kDenseWarps * 32, smem, stream>>>(sc, tb, buf, io, rec, t_global, n_steps, auto_reset);
  return true;
}

template <typename R>
void launch_dense_reset(const DevScenario<R>& sc, const DenseTables<R>& tb, const EnvBuffers<R>& buf, const uint8_t* mask, const R* init,
                        int first_time, cudaStream_t stream) {
  const unsigned grid = (unsigned)((buf.hi - buf.lo + kDenseWarps - 1) / kDenseWarps);
  dense_reset_kernel<R><<<grid, kDenseWarps * 32, 0, stream>>>(sc, tb, buf, mask, init, first_time);
}

template <typename R> const DenseLaunchers<R>* dense_launchers();   // defined in dense.cu

}  // namespace cav
