// transition.cuh — one joint transition of ONE environment, entirely in registers.
//
// Restates, in the reference's order (library/environment.py:119-223):
//   joint action        agents' choose_action on the pre-step state        simulation.py:71
//   validation          action_space.contains                              environment.py:120
//   body.step           kinematic bicycle / traffic-light state            environment.py:122-123
//   bounding boxes      info()['body_polygons']                            environment.py:107,125-127
//   rewards, liveness                                                      environment.py:131-146
//   termination cascade finish > all-collisions > off-road > ego-collision > reaction zone   :148-206
//   terminal rewards, winner                                               environment.py:208-220
//   process_feedback    crossing agents, post-step state                   simulation.py:86-87
// Used by the step, replay and rollout kernels (kernels_small.cuh), so the three share one
// definition of a transition.  Thread-per-environment: every array below is indexed by
// compile-time constants after unrolling and lives in registers.
//
// Boxes never become corner lists here: each body is (x, y, cos, sin, half length, half width) and every test is
// written on that form (geometry.cuh).  What stays out of line: general quads, road corners, libm.
#pragma once
#include <cooperative_groups.h>
#include <cooperative_groups/reduce.h>

#include "agents.cuh"

namespace cav {

template <typename R, int M>
struct EnvRegs {
  R s[M][4];         // x, y, v, theta (PelicanCrossing: light state in [0])
  R held[M][2];      // last action of on-device agents (RandomAgent holds it)
  R ag[M][CAV_AGENT_WORDS];
  R cs[M][2];        // cos, sin of the heading (EnvBuffers::cs)
  int32_t live[M];   // episode_liveness (environment.py:144-146); [0] unused
  int32_t t_ep, episode, winner;
  int32_t active;    // Election.active_player (0 = None); only kernels with on-device agents carry it
  uint32_t live_dirty;  // bit b: live[b] changed since it was loaded
  uint32_t cs_dirty;  // bit b: cs[b] changed since it was loaded
  uint32_t ag_dirty;  // bit b: ag[b] changed since it was loaded
  uint8_t done;
};

// Episode statistics (reporting.py:227-269) are updated with atomics at the moment an episode ends or a near-tangent
// step is flagged — about one env-step in a thousand — so no per-thread accumulators stay live through the step.
__device__ __forceinline__ void count_tangent(unsigned long long* stats) { atomicAdd(&stats[CAV_STAT_TANGENT], 1ull); }

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename R, int M>
__device__ __forceinline__ bool uses_agent_state(const DevScenario<R>& sc, int b) {
  return sc.bodies[b].agent == CAV_AGENT_RANDOM_CONSTRAINED || sc.bodies[b].agent == CAV_AGENT_PROXIMITY ||
         sc.bodies[b].agent == CAV_AGENT_ELECTION;
}

// Body b as a box / as a pose; b must be a compile-time constant at the call site (unrolled loops).
template <typename R, int M>
__device__ __forceinline__ Box<R> body_box(const DevScenario<R>& sc, const EnvRegs<R, M>& env, const int b) {
  return {env.s[b][0], env.s[b][1], env.cs[b][0], env.cs[b][1], sc.bodies[b].k.hl, sc.bodies[b].k.hw};
}
template <typename R, int M>
__device__ __forceinline__ Pose<R> body_pose(const DevScenario<R>& sc, const EnvRegs<R, M>& env, const int b) {
  const DevBody<R>& body = sc.bodies[b];
  return {env.s[b][0], env.s[b][1], env.s[b][3], env.cs[b][0], env.cs[b][1], body.k.length, body.k.width};
}

// closed predicate from a separating-axis margin; flags near-tangent decisions
template <typename R>
__device__ __forceinline__ bool margin_hit(R margin, R tau, bool& tangent) {
  if (rabs(margin) < tau) tangent = true;
  return !(margin > R(0));
}
__device__ __forceinline__ bool geo_hit(int r, bool& tangent) {
  if (r & GEO_TANGENT) tangent = true;
  return (r & GEO_HIT) != 0;
}

// One edge of the box TOUCHES a kerb (its margin lies within tau of zero, the other three edges are clearly inside): a car that
// starts half outside the end of its road is in this position for exactly one step of every episode, a tester that has braked
// to a stop there for the rest of it.  The reference's `contains` then decides between the exact 1 and the clipped share
// (geometry.py:81-86), both of which the one-kerb form gives (it is continuous through zero), and the decision is near-tangent
// by definition, so the flag is raised as the general predicates would raise it — without the polygon clipper, which cost the
// bus-stop rollout a tenth of its time at one active lane per warp.
template <typename R>
__device__ __forceinline__ R kerb_touch_share(R c, R s, R hl, R hw, R lo, bool x_edge, R ex, R ey, bool& near) {
  near = true;
  if (lo >= R(0)) return R(1);
  const R ac = rabs(c), as = rabs(s);
  return kerb_share(lo + (x_edge ? ex : ey), (x_edge ? ac : as) * hl, (x_edge ? as : ac) * hw);
}

// Shape.percentage_intersects(body box, road r) (environment.py:141, geometry.py:80-87).
//   AABB clear of the road            -> 0        (disjoint)
//   axis-aligned road, clearly inside -> 1        (contained)
//   axis-aligned road, one kerb       -> closed form (kerb_share)
//   anything else                     -> general predicates, out of line
// `near` is raised when the share is within tau of the liveness threshold 0.5 (environment.py:144) or a general
// predicate was near-tangent.  GENERIC = false: every road is known to be an axis-aligned rectangle.
template <typename R, int M, bool GENERIC>
__device__ __forceinline__ R road_share(const DevScenario<R>& sc, const EnvRegs<R, M>& env, const int b, int r, R ex, R ey,
                                        R tau, bool& near) {
  const Aabb<R> rd = sc.road_bb[r];
  const R px = env.s[b][0], py = env.s[b][1];
  const R m0 = (px - ex) - rd.x0, m1 = rd.x1 - (px + ex), m2 = (py - ey) - rd.y0, m3 = rd.y1 - (py + ey);
  const R mx = rmin(m0, m1), my = rmin(m2, m3);
  if (mx < -((ex + ex) + tau) || my < -((ey + ey) + tau)) return R(0);
  if (!GENERIC || sc.road_axis[r]) {
    const bool x_edge = mx < my;
    const R lo = x_edge ? mx : my, hi = x_edge ? my : mx;
    if (lo >= tau) return R(1);
    // one kerb: the smallest margin is clearly negative, the opposite edge and the other pair of edges clearly inside
    const R opposite = x_edge ? rmax(m0, m1) : rmax(m2, m3);
    if (lo > -tau && hi >= tau && opposite >= tau) return kerb_touch_share(env.cs[b][0], env.cs[b][1], sc.bodies[b].k.hl, sc.bodies[b].k.hw, lo, x_edge, ex, ey, near);
    if (lo <= -tau && hi >= tau && opposite >= tau) {
      const R ac = rabs(env.cs[b][0]), as = rabs(env.cs[b][1]);
      const R hl = sc.bodies[b].k.hl, hw = sc.bodies[b].k.hw;
      const R p = kerb_share(lo + (x_edge ? ex : ey), (x_edge ? ac : as) * hl, (x_edge ? as : ac) * hw);
      if (rabs(p - R(0.5)) < tau) near = true;
      return p;
    }
    // a corner of the road: one x-edge and one y-edge crossed (or touched), the opposite edges clearly inside
    if (mx < tau && my < tau && rmax(m0, m1) >= tau && rmax(m2, m3) >= tau) {
      const bool low_x = m0 < m1, low_y = m2 < m3;
      const R p = corner_share_closed(body_pose<R, M>(sc, env, b), mx + ex, my + ey, low_x ? R(-1) : R(1), low_x ? -rd.x0 : rd.x1,
                                      low_y ? R(-1) : R(1), low_y ? -rd.y0 : rd.y1, tau);
      if (rabs(p - R(0.5)) < tau) near = true;
      return p;
    }
  }
  const Share<R> share = road_share_general(body_pose<R, M>(sc, env, b), &sc.quads[r], tau);
  near |= (share.tangent != 0) || (rabs(share.value - R(0.5)) < tau);
  return share.value;
}

// Result of one transition besides the updated EnvRegs.
template <typename R, int M>
struct StepResult {
  R reward[M];
  bool terminate, tangent, invalid;
  int32_t winner;
};

// AGENTS = false compiles the replay-only variant: every body takes its action from `ext`.
// GENERIC = false compiles the homogeneous variant the engine selects when the scenario has no PelicanCrossing body,
// every non-ego body is a Pedestrian and every road is an axis-aligned rectangle (the Pedestrians-v0 family, any
// number of pedestrians): the per-body kind / flag tests disappear at compile time.
struct NoSink {
  template <typename E> __device__ __forceinline__ void operator()(const E&) const {}
};
// `phase()` is called at the three phase boundaries of a transition (after the joint action, after body.step, after the
// termination cascade) — by EVERY thread that enters the transition, on every path out of it.  CtaPhase makes each a
// block-wide barrier: a kernel whose threads all run one transition per step (the rollout kernels of the heterogeneous
// scenarios) keeps the warps of a CTA inside the same phase, so they share instruction fetches (DESIGN 4.5).
constexpr int kTransitionPhases = 3;
struct NoPhase { static constexpr bool kBarrier = false; __device__ __forceinline__ void operator()() const {} };
// The barrier is `bar.sync` (aligned): all 32 lanes of a warp must arrive together, so a kernel that uses CtaPhase makes
// EVERY lane run the transition on every step (lanes without an env of their own step a copy of a neighbour's with the side
// effects switched off, kernels_small.cuh) and re-converges the warp before each barrier.  `on` is launch-uniform.
struct CtaPhase {
  static constexpr bool kBarrier = true;
  bool on;
  __device__ __forceinline__ void operator()() const { if (on) { __syncwarp(); __syncthreads(); } }
};

// `tester` gives the transition the on-device agents' parameters: body b's RandomAgent / RandomConstrainedAgent epsilon
// (template.py:52-62, pedestrian.py:72-75) and ProximityAgent / ElectionAgent distance threshold (pedestrian.py:78-91) for
// env e.  SceneTester reads the scenario's values, the same for every env; EnvTester (kernels_params.cuh) reads per-env ones.
struct SceneTester {
  template <typename R> __device__ __forceinline__ double epsilon(const DevBody<R>& body, int, int64_t, int64_t) const { return body.epsilon; }
  template <typename R> __device__ __forceinline__ R threshold(const DevBody<R>& body, int, int64_t, int64_t) const { return body.threshold; }
};

// `key` gives the global env id that keys env e's Philox draws (spawns in reset_env, agents in the transition) and that its
// episode rows carry.  ShardKey is slot e of the engine's shard; SlotKey (kernels_regen.cuh) is an id the caller gave for the
// slot, so that a slot replays the episodes of another env.
struct ShardKey {
  template <typename R> __device__ __forceinline__ int64_t operator()(const EnvBuffers<R>& buf, int64_t e) const { return buf.shard + e; }
};

// `moved(env)` is called once, right after body.step: a kernel that stages state in shared memory writes the new
// state there at that point, so x, y, v, theta need not stay in registers through the geometry.
//
// Two instantiations of one body (transition_body.inc):
//   transition_unrolled   loops over bodies fully unrolled, every per-body array in registers — the homogeneous and the
//                         two-body kernels (the tuned paths of configs C2 / C5);
//   transition_rolled     loops over bodies kept as loops.  Heterogeneous scenarios with three or more bodies (crossroads,
//                         bus stop, pelican crossing): unrolled, one step of the M = 5 kernel is ~3,700 straight-line
//                         instructions — 60 KB of code per step against a 32 KB instruction cache — and ncu shows it waiting
//                         for instruction fetch 29 cycles for every cycle it issues (profiles/r1_rollout_kernels_ncu.txt).
//                         Rolled, the per-body code exists once; the per-body arrays are then indexed at run time and live in
//                         L1-resident local memory instead of registers.  Same arithmetic, same order: results are bitwise
//                         those of the unrolled form (and of the warp-per-env kernels, tests/test_gpu_dense.py).
#ifndef CAV_ROLLED_FROM_M
#define CAV_ROLLED_FROM_M 3
#endif
#ifndef CAV_ROLL_AGENTS
#define CAV_ROLL_AGENTS 0
#endif
// Homogeneous (Pedestrians-v0 family) kernels WITH on-device agents are rolled from this many bodies on (rollout at M = 4:
// 14.2 -> 8.8 ms per 100 steps of 262,144 envs, at M = 8: 78 -> 26 ms); on replayed actions they stay unrolled (the fused
// replay kernel keeps the state in registers across steps: 0.85 ms unrolled vs 1.42 ms rolled at M = 4).
#ifndef CAV_ROLLED_HOMOGENEOUS_REPLAY_FROM_M   // the same family on replayed actions (measured below)
#define CAV_ROLLED_HOMOGENEOUS_REPLAY_FROM_M 99
#endif
#ifndef CAV_ROLLED_HOMOGENEOUS_FROM_M
#define CAV_ROLLED_HOMOGENEOUS_FROM_M 4
#endif

#define CAV_BODY_LOOP _Pragma("unroll")
template <typename R, int M, bool AGENTS, bool GENERIC, typename Sink = NoSink, typename Phase = NoPhase,
          typename Tester = SceneTester, typename Key = ShardKey>
__device__ __forceinline__ void transition_unrolled(const DevScenario<R>& sc, const EnvBuffers<R>& buf, int64_t e, int64_t t_global,
                                                    EnvRegs<R, M>& env, const R (&ext)[M][2], StepResult<R, M>& out,
                                                    Sink moved = Sink(), Phase phase = Phase(), Tester tester = Tester(),
                                                    Key key = Key()) {
#include "transition_body.inc"
}
#undef CAV_BODY_LOOP

#define CAV_BODY_LOOP _Pragma("unroll 1")
template <typename R, int M, bool AGENTS, bool GENERIC, typename Sink = NoSink, typename Phase = NoPhase,
          typename Tester = SceneTester, typename Key = ShardKey>
__device__ __forceinline__ void transition_rolled(const DevScenario<R>& sc, const EnvBuffers<R>& buf, int64_t e, int64_t t_global,
                                                  EnvRegs<R, M>& env, const R (&ext)[M][2], StepResult<R, M>& out,
                                                  Sink moved = Sink(), Phase phase = Phase(), Tester tester = Tester(),
                                                  Key key = Key()) {
#include "transition_body.inc"
}
#undef CAV_BODY_LOOP

template <typename R, int M, bool AGENTS, bool GENERIC, typename Sink = NoSink, typename Phase = NoPhase,
          typename Tester = SceneTester, typename Key = ShardKey>
__device__ __forceinline__ void transition(const DevScenario<R>& sc, const EnvBuffers<R>& buf, int64_t e, int64_t t_global,
                                           EnvRegs<R, M>& env, const R (&ext)[M][2], StepResult<R, M>& out,
                                           Sink moved = Sink(), Phase phase = Phase(), Tester tester = Tester(), Key key = Key()) {
  if constexpr ((GENERIC && M >= CAV_ROLLED_FROM_M) || (!GENERIC && AGENTS && M >= CAV_ROLLED_HOMOGENEOUS_FROM_M) ||
                (!GENERIC && !AGENTS && M >= CAV_ROLLED_HOMOGENEOUS_REPLAY_FROM_M) ||
                (AGENTS && CAV_ROLL_AGENTS != 0 && M >= 2)) transition_rolled<R, M, AGENTS, GENERIC, Sink, Phase, Tester, Key>(sc, buf, e, t_global, env, ext, out, moved, phase, tester, key);
  else transition_unrolled<R, M, AGENTS, GENERIC, Sink, Phase, Tester, Key>(sc, buf, e, t_global, env, ext, out, moved, phase, tester, key);
}

// reporting.analyse_episode (reporting.py:227-243) for an env whose episode just ended.  The lanes of a warp that end their
// episodes in the same step (with a Noop ego EVERY env reaches the finish line at step 901 at once) first add up their
// contributions, so the ten global counters see one atomic per warp and counter instead of one per env.
struct EpisodeLog {
  CavEpisodeRow* rows;
  unsigned long long* count;
  int64_t capacity, env;   // env = global id of the env that finished
  int32_t episode;         // its per-env episode number (1 = the first episode after cavgym_create)
};

template <typename R, int M>
__device__ __noinline__ void score_episode(unsigned long long* stats, int32_t t_ep, int32_t winner, long long liveness_sum,
                                           const EpisodeLog log) {
  namespace cg = cooperative_groups;
  const cg::coalesced_group lanes = cg::coalesced_threads();
  const unsigned long long t = (unsigned long long)t_ep;
  const bool interesting = winner > 0;
  const long long score = interesting ? -liveness_sum : 0;
  const cg::plus<unsigned long long> add;
  const unsigned long long n_eps = lanes.size();
  const unsigned long long sum_t = cg::reduce(lanes, t, add), sum_t2 = cg::reduce(lanes, t * t, add);
  const unsigned long long n_int = cg::reduce(lanes, (unsigned long long)(interesting ? 1 : 0), add);
  unsigned long long sum_s = 0, sum_s2 = 0, sum_it = 0, sum_it2 = 0;
  if (n_int) {   // two's complement: the unsigned sums wrap to the signed ones
    sum_s = cg::reduce(lanes, (unsigned long long)score, add);
    sum_s2 = cg::reduce(lanes, (unsigned long long)(score * score), add);
    sum_it = cg::reduce(lanes, interesting ? t : 0ull, add);
    sum_it2 = cg::reduce(lanes, interesting ? t * t : 0ull, add);
  }
  unsigned long long slot = 0;
  if (lanes.thread_rank() == 0) {
    atomicAdd(&stats[CAV_STAT_EPISODES], n_eps);
    atomicAdd(&stats[CAV_STAT_SUM_T], sum_t);
    atomicAdd(&stats[CAV_STAT_SUM_T2], sum_t2);
    if (n_int) {
      atomicAdd(&stats[CAV_STAT_INTERESTING], n_int);
      atomicAdd(&stats[CAV_STAT_SUM_SCORE], sum_s);
      atomicAdd(&stats[CAV_STAT_SUM_SCORE2], sum_s2);
      atomicAdd(&stats[CAV_STAT_SUM_T_INTERESTING], sum_it);
      atomicAdd(&stats[CAV_STAT_SUM_T2_INTERESTING], sum_it2);
    }
    if (log.rows) slot = atomicAdd(log.count, n_eps);   // one reservation for all the rows of this warp
  }
  if (log.rows) {   // the reporting.EpisodeResults of this episode, one 24-byte row (file_message, reporting.py:157-158)
    slot = lanes.shfl(slot, 0) + lanes.thread_rank();
    if (slot < (unsigned long long)log.capacity) log.rows[slot] = {log.env, log.episode, t_ep, winner, (int32_t)liveness_sum};
  }
}

// `episode` = the env's episode number if the kernel carries it in registers (on-device agents), else -1: read it back.
template <typename R, int M, typename Key = ShardKey>
__device__ __forceinline__ void score_episode(const EnvBuffers<R>& buf, const EnvRegs<R, M>& env, int64_t e, int32_t episode = -1,
                                              Key key = Key()) {
  long long sum = 0;
#pragma unroll
  for (int b = 1; b < M; ++b) sum += env.live[b];
  EpisodeLog log{buf.ep_log, buf.ep_log_count, buf.ep_log_capacity, key(buf, e), episode};
  if (buf.ep_log && episode < 0) log.episode = buf.episode[e];
  score_episode<R, M>(buf.stats, env.t_ep, env.winner, sum, log);
}

// CAVEnv.reset for one env (environment.py:225-229): bodies back to init_state (SpawnPedestrians re-drawn),
// liveness zeroed, agents reset, on-device noop action.  `init` (nullable) replays given initial states.
template <typename R, int M, typename Key = ShardKey>
__device__ __forceinline__ void reset_env(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const R* init, int64_t e,
                                          EnvRegs<R, M>& env, Key key = Key()) {
  env.episode += 1;
#pragma unroll
  for (int b = 0; b < M; ++b) {
    const DevBody<R>& body = sc.bodies[b];
    R st[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) st[c] = body.init[c];
    if (init) {
#pragma unroll
      for (int c = 0; c < 4; ++c) st[c] = init[((int64_t)b * 4 + c) * buf.n + e];
    } else if ((body.flags & CAV_FLAG_SPAWN) && body.spawn_id >= 0) {
      double u[5];
      if (buf.spawn_override) {
#pragma unroll
        for (int c = 0; c < 5; ++c) u[c] = buf.spawn_override[((int64_t)b * 5 + c) * buf.n + e];
      } else {
        double w[2];
        const uint64_t g = (uint64_t)key(buf, e);
        draw_block(buf.seed, g, b, KIND_SPAWN0, (uint32_t)env.episode, 0u, w); u[0] = w[0]; u[1] = w[1];
        draw_block(buf.seed, g, b, KIND_SPAWN1, (uint32_t)env.episode, 0u, w); u[2] = w[0]; u[3] = w[1];
        draw_block(buf.seed, g, b, KIND_SPAWN2, (uint32_t)env.episode, 0u, w); u[4] = w[0];
      }
      spawn_body(buf.spawns[body.spawn_id], u, st);
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) env.s[b][c] = st[c];
    env.held[b][0] = R(0); env.held[b][1] = R(0);
    env.cs[b][0] = R(1); env.cs[b][1] = R(0);
    if (body.kind == CAV_BODY_DYNAMIC) heading_cs(sc, st[3], env.cs[b][0], env.cs[b][1]);
#pragma unroll
    for (int w = 0; w < CAV_AGENT_WORDS; ++w) env.ag[b][w] = nan_<R>();
    env.live[b] = 0;
  }
  env.t_ep = 0;
  env.done = 0;
  env.winner = -1;
  env.ag_dirty = 0xFFFFFFFFu;  // everything must be written back
  env.live_dirty = 0xFFFFFFFFu;
  env.cs_dirty = 0xFFFFFFFFu;
}

}  // namespace cav
