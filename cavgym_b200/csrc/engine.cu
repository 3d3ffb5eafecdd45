// engine.cu — the C-ABI of libcavgym_sm100.so (include/cavgym.h): engine lifetime, table
// conversion, kernel dispatch, the pipelined host-buffer step, statistics and the
// stand-alone per-function kernels.  No torch types; callers pass raw device pointers.
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#ifndef CAV_HOST_CTAS_PER_SM
#define CAV_HOST_CTAS_PER_SM 3
#endif


#include "kernels_dense.cuh"
#ifndef CAV_REPLAY_CHAIN   // 0: every replay launch waits for the whole previous grid (A/B)
#define CAV_REPLAY_CHAIN 1
#endif
#include "kernels_tma.cuh"   // (tma_span, kReplayTile for the replay launch chain; includes kernels_small.cuh)
#include "kernels_snapshot.cuh"
#include "kernels_until.cuh"
#include "kernels_params.cuh"
#include "kernels_regen.cuh"

namespace cav {

#define CAV_FOR_EACH_M(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8)
#define CAV_DECLARE(K)                                   \
  extern const SmallLaunchers<double> kSmallF64M##K;     \
  extern const SmallLaunchers<float> kSmallF32M##K;      \
  extern const RolloutRecordLauncher<double> kRecordF64M##K; \
  extern const RolloutRecordLauncher<float> kRecordF32M##K; \
  extern const RolloutUntilLauncher<double> kUntilF64M##K; \
  extern const RolloutUntilLauncher<float> kUntilF32M##K; \
  extern const ParamsLaunchers<double> kParamsF64M##K; \
  extern const ParamsLaunchers<float> kParamsF32M##K; \
  extern const RegenerateLauncher<double> kRegenF64M##K; \
  extern const RegenerateLauncher<float> kRegenF32M##K;
CAV_FOR_EACH_M(CAV_DECLARE)
#undef CAV_DECLARE

template <> const SmallLaunchers<double>* small_launchers<double>(int m) {
  switch (m) {
#define CAV_CASE(K) case K: return &kSmallF64M##K;
    CAV_FOR_EACH_M(CAV_CASE)
#undef CAV_CASE
    default: return nullptr;
  }
}
template <> const SmallLaunchers<float>* small_launchers<float>(int m) {
  switch (m) {
#define CAV_CASE(K) case K: return &kSmallF32M##K;
    CAV_FOR_EACH_M(CAV_CASE)
#undef CAV_CASE
    default: return nullptr;
  }
}

template <> RolloutRecordLauncher<double> rollout_record_launcher<double>(int m) {
  switch (m) {
#define CAV_CASE(K) case K: return kRecordF64M##K;
    CAV_FOR_EACH_M(CAV_CASE)
#undef CAV_CASE
    default: return nullptr;
  }
}
template <> RolloutRecordLauncher<float> rollout_record_launcher<float>(int m) {
  switch (m) {
#define CAV_CASE(K) case K: return kRecordF32M##K;
    CAV_FOR_EACH_M(CAV_CASE)
#undef CAV_CASE
    default: return nullptr;
  }
}

template <> RolloutUntilLauncher<double> rollout_until_launcher<double>(int m) {
  switch (m) {
#define CAV_CASE(K) case K: return kUntilF64M##K;
    CAV_FOR_EACH_M(CAV_CASE)
#undef CAV_CASE
    default: return nullptr;
  }
}
template <> RolloutUntilLauncher<float> rollout_until_launcher<float>(int m) {
  switch (m) {
#define CAV_CASE(K) case K: return kUntilF32M##K;
    CAV_FOR_EACH_M(CAV_CASE)
#undef CAV_CASE
    default: return nullptr;
  }
}

template <> const ParamsLaunchers<double>* params_launchers<double>(int m) {
  switch (m) {
#define CAV_CASE(K) case K: return &kParamsF64M##K;
    CAV_FOR_EACH_M(CAV_CASE)
#undef CAV_CASE
    default: return nullptr;
  }
}
template <> const ParamsLaunchers<float>* params_launchers<float>(int m) {
  switch (m) {
#define CAV_CASE(K) case K: return &kParamsF32M##K;
    CAV_FOR_EACH_M(CAV_CASE)
#undef CAV_CASE
    default: return nullptr;
  }
}

template <> RegenerateLauncher<double> regenerate_launcher<double>(int m) {
  switch (m) {
#define CAV_CASE(K) case K: return kRegenF64M##K;
    CAV_FOR_EACH_M(CAV_CASE)
#undef CAV_CASE
    default: return nullptr;
  }
}
template <> RegenerateLauncher<float> regenerate_launcher<float>(int m) {
  switch (m) {
#define CAV_CASE(K) case K: return kRegenF32M##K;
    CAV_FOR_EACH_M(CAV_CASE)
#undef CAV_CASE
    default: return nullptr;
  }
}

// cavgym_regenerate_episodes' range check of the caller's keys: bit 0 of *bad for a global env id outside [0, 2^40) (the ids
// cavgym_set_shard admits), bit 1 for a negative episode number.
__global__ void check_regen_keys_kernel(const int64_t* env_ids, const int32_t* episodes, int64_t n, unsigned int* bad) {
  unsigned int flags = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (env_ids[i] < 0 || env_ids[i] >= ((int64_t)1 << 40)) flags |= 1u;
    if (episodes[i] < 0) flags |= 2u;
  }
  if (flags) atomicOr(bad, flags);
}

static thread_local std::string g_error;

static int fail(int code, const std::string& message) {
  g_error = message;
  return code;
}

#define CUDA_TRY(call)                                                                             \
  do {                                                                                             \
    cudaError_t err_ = (call);                                                                     \
    if (err_ != cudaSuccess)                                                                       \
      return fail(CAV_ECUDA, std::string(#call) + ": " + cudaGetErrorString(err_));                \
  } while (0)

// ---------------------------------------------------------------- table conversion
template <typename R>
static Quad<R> to_quad(const CavQuad& q) {
  // Normalise to clockwise order; the predicates do not depend on which corner comes first.
  double twice_area = 0.0;
  for (int i = 0; i < 4; ++i) {
    const int j = (i + 1) & 3;
    twice_area += q.x[i] * q.y[j] - q.x[j] * q.y[i];
  }
  Quad<R> out;
  for (int i = 0; i < 4; ++i) {
    const int src = twice_area > 0 ? 3 - i : i;
    out.x[i] = (R)q.x[src];
    out.y[i] = (R)q.y[src];
  }
  return out;
}

template <typename R>
static Aabb<R> host_aabb(const Quad<R>& q) {
  Aabb<R> b{q.x[0], q.x[0], q.y[0], q.y[0]};
  for (int i = 1; i < 4; ++i) {
    b.x0 = std::fmin(b.x0, q.x[i]); b.x1 = std::fmax(b.x1, q.x[i]);
    b.y0 = std::fmin(b.y0, q.y[i]); b.y1 = std::fmax(b.y1, q.y[i]);
  }
  return b;
}

template <typename R>
static DevType<R> to_type(const CavBodyType& t) {
  DevType<R> k;
  k.length = (R)t.length; k.width = (R)t.width; k.wheelbase = (R)t.wheelbase;
  k.vmin = (R)t.min_velocity; k.vmax = (R)t.max_velocity; k.amin = (R)t.min_throttle; k.amax = (R)t.max_throttle;
  k.smin = (R)t.min_steering_angle; k.smax = (R)t.max_steering_angle;
  k.hl = (R)(t.length * 0.5); k.hw = (R)(t.width * 0.5); k.half_wb = (R)(t.wheelbase / 2.0);
  k.inv_2brake = (R)(1.0 / (2.0 * -t.min_throttle));
  const double half_wb = t.wheelbase / 2.0;
  const double kk_min = t.wheelbase / std::tan((double)k.smin), kk_max = t.wheelbase / std::tan((double)k.smax);
  k.kk_smin = kk_min; k.kk_smax = kk_max;
  k.inv_r_smin = 1.0 / std::sqrt(half_wb * half_wb + kk_min * kk_min);
  k.inv_r_smax = 1.0 / std::sqrt(half_wb * half_wb + kk_max * kk_max);
  auto turn_root = [&](double limit) {   // sqrt(wb^2 (1 + 4 / tan^2(limit))) in R, as steering_towards used to form it on the device
    const R wb = k.wheelbase, tn = (R)std::tan((double)(R)limit);
    return (R)std::sqrt((double)((wb * wb) * ((R)1 + (R)4 / (tn * tn))));
  };
  k.max_turn_smin = turn_root((double)k.smin);
  k.max_turn_smax = turn_root((double)k.smax);
  return k;
}

// Centre-extent form of a quad that is a rectangle (every road, traffic light and obstacle of the reference is one:
// make_rectangle(...).transform(...), assets.py / bodies.py); false for a general convex quad.
template <typename R>
static bool to_box(const Quad<R>& q, Box<R>& out) {
  const double ux = (double)q.x[1] - q.x[0], uy = (double)q.y[1] - q.y[0];   // rear_left -> front_left: the heading
  const double vx = (double)q.x[3] - q.x[0], vy = (double)q.y[3] - q.y[0];   // rear_left -> rear_right: across
  const double lu = std::sqrt(ux * ux + uy * uy), lv = std::sqrt(vx * vx + vy * vy);
  if (!(lu > 0.0) || !(lv > 0.0)) return false;
  const double scale = lu + lv, eps = (sizeof(R) == 8 ? 1e-12 : 1e-5) * scale;
  const double px = (double)q.x[0] + ux + vx - q.x[2], py = (double)q.y[0] + uy + vy - q.y[2];  // parallelogram closure
  if (std::fabs(px) > eps || std::fabs(py) > eps) return false;
  if (std::fabs(ux * vx + uy * vy) > eps * scale) return false;                                    // right angle
  out.px = (R)(((double)q.x[0] + q.x[1] + q.x[2] + q.x[3]) * 0.25);
  out.py = (R)(((double)q.y[0] + q.y[1] + q.y[2] + q.y[3]) * 0.25);
  out.c = (R)(ux / lu); out.s = (R)(uy / lu);
  out.hl = (R)(lu * 0.5); out.hw = (R)(lv * 0.5);
  return true;
}

template <typename R>
static void convert(const CavScenario& in, double tau, DevScenario<R>& out) {
  std::memset(&out, 0, sizeof(out));
  out.n_bodies = in.n_bodies; out.n_types = in.n_types; out.n_roads = in.n_roads; out.n_statics = in.n_statics;
  out.n_spawns = in.n_spawns;
  out.collisions = in.terminate_collisions; out.zones = in.terminate_ego_zones; out.offroad = in.terminate_ego_offroad;
  out.max_timesteps = in.max_timesteps;
  out.reward_win = (R)in.reward_win; out.reward_draw = (R)in.reward_draw; out.cost_step = (R)in.cost_step;
  out.W = (R)in.viewer_width; out.dt = (R)in.time_resolution;
  out.v_maint = (R)in.ego_maintenance_velocity; out.v_off = (R)in.ego_max_velocity_offset;
  out.inv_W = (R)(1.0 / in.viewer_width); out.inv_v_off = (R)(1.0 / in.ego_max_velocity_offset);
  out.tau = (R)tau;
  out.target_err = sizeof(R) == 8 ? (R)0.000000000000001 : (R)1e-6;  // dynamic_body.py:8; one float ulp at pi/2 is 1.2e-7
  for (int i = 0; i < 4; ++i) out.cl[i] = (R)in.centre_line[i];
  Quad<R> roads[CAV_MAX_ROADS];
  for (int i = 0; i < in.n_roads; ++i) {
    roads[i] = to_quad<R>(in.roads[i]);
    out.road_bb[i] = host_aabb(roads[i]);
    // Axis-aligned: every corner lies on a corner of the AABB — up to a thousandth of the near-tangent tolerance.  The side
    // roads of the crossroads scenario are make_rectangle(...).transform(+-pi/2, ...) (assets.py, crossroads.py:10-49): their
    // corners come out as 718.9999999999999 / 719.0, a skew of 1e-13 px that fp32 rounds away and fp64 does not.  Held to
    // exact equality, every body near those roads went through the general clipper (18 % of the rollout kernel's warp
    // instructions at 1.2 active lanes: crossroads ran twice as fast in fp32 as in fp64); the closed forms on the AABB differ
    // from the skewed quad by ~1e-13 px, four orders below what a decision may depend on without being flagged.
    const R snap = (R)(tau * 1e-3);
    auto on = [snap](R v, R bound) { return std::fabs((double)v - (double)bound) <= (double)snap; };
    bool axis = true;
    for (int c = 0; c < 4; ++c)
      axis = axis && (on(roads[i].x[c], out.road_bb[i].x0) || on(roads[i].x[c], out.road_bb[i].x1)) &&
             (on(roads[i].y[c], out.road_bb[i].y0) || on(roads[i].y[c], out.road_bb[i].y1));
    out.road_axis[i] = axis ? 1 : 0;
    out.road_rect[i] = to_box(roads[i], out.road_box[i]) ? 1 : 0;
  }
  for (int i = 0; i < in.n_statics; ++i) {
    const Quad<R> q = to_quad<R>(in.statics[i]);
    out.static_bb[i] = host_aabb(q);
    out.static_rect[i] = to_box(q, out.static_box[i]) ? 1 : 0;
  }
  for (int b = 0; b < in.n_bodies && b < CAV_SMALL_M; ++b) {
    const CavBody& src = in.bodies[b];
    DevBody<R>& dst = out.bodies[b];
    dst.kind = src.kind; dst.type_id = src.type_id; dst.flags = src.flags; dst.agent = src.agent; dst.spawn_id = src.spawn_id;
    dst.epsilon = src.agent_epsilon; dst.threshold = (R)src.agent_threshold;
    for (int c = 0; c < 4; ++c) dst.init[c] = (R)src.init_state[c];
    if (src.kind == CAV_BODY_DYNAMIC) dst.k = to_type<R>(in.types[src.type_id]);
    if (src.kind == CAV_BODY_PELICAN) {  // percentage_intersects(static box, road) never changes: environment.py:141
      const Quad<R> box = to_quad<R>(src.static_box);
      R share = (R)0;
      for (int r = 0; r < in.n_roads; ++r) {
        const R q = percentage_of(box, roads[r], (R)tau).value;
        if (r == 0 || q > share) share = q;
      }
      dst.static_share = share;
    }
  }
  bool homogeneous = in.n_bodies <= CAV_SMALL_M;
  for (int i = 0; i < in.n_roads; ++i) homogeneous = homogeneous && out.road_axis[i] && out.road_rect[i];
  for (int b = 0; b < in.n_bodies && b < CAV_SMALL_M; ++b) {
    homogeneous = homogeneous && in.bodies[b].kind == CAV_BODY_DYNAMIC;
    if (b > 0) homogeneous = homogeneous && (in.bodies[b].flags & CAV_FLAG_PEDESTRIAN);
  }
  out.homogeneous = homogeneous ? 1 : 0;
  out.has_election = 0;
  for (int b = 0; b < in.n_bodies && b < CAV_SMALL_M; ++b) if (in.bodies[b].agent == CAV_AGENT_ELECTION) out.has_election = 1;
  // heading cache: orientations bodies start with, cos/sin from the host C library (what math.cos/math.sin call)
  auto remember = [&out](double theta) {
    const R th = (R)theta;
    if (th == (R)0 || out.hc_n >= CAV_HEADING_CACHE) return;
    for (int i = 0; i < out.hc_n; ++i) if (out.hc_theta[i] == th) return;
    out.hc_theta[out.hc_n] = th;
    out.hc_cos[out.hc_n] = (R)std::cos((double)th);
    out.hc_sin[out.hc_n] = (R)std::sin((double)th);
    out.hc_n += 1;
  };
  for (int s = 0; s < in.n_spawns; ++s)
    for (int i = 0; i < in.spawns[s].n_orientations; ++i) remember(in.spawns[s].orientations[i]);
  for (int b = 0; b < in.n_bodies; ++b)
    if (in.bodies[b].kind == CAV_BODY_DYNAMIC) remember(in.bodies[b].init_state[3]);
}

// Per-body rows of the warp-per-env path (kernels_dense.cuh): any number of bodies, kept in device memory.
template <typename R>
static void convert_dense(const CavScenario& in, double tau, DenseTables<R>& tb, std::vector<DenseBody<R>>& rows) {
  std::memset(&tb, 0, sizeof(tb));
  for (int t = 0; t < in.n_types; ++t) tb.types[t] = to_type<R>(in.types[t]);
  Quad<R> roads[CAV_MAX_ROADS];
  for (int i = 0; i < in.n_roads; ++i) roads[i] = to_quad<R>(in.roads[i]);
  rows.assign((size_t)in.n_bodies, DenseBody<R>{});
  for (int b = 0; b < in.n_bodies; ++b) {
    const CavBody& src = in.bodies[b];
    DenseBody<R>& dst = rows[(size_t)b];
    dst.meta = (src.kind == CAV_BODY_DYNAMIC ? (src.type_id & DM_TYPE_MASK) : 0) | (src.kind == CAV_BODY_PELICAN ? DM_PELICAN : 0) |
               ((src.flags & CAV_FLAG_PEDESTRIAN) ? DM_PEDESTRIAN : 0) | ((src.flags & CAV_FLAG_SPAWN) ? DM_SPAWN : 0) |
               ((src.agent & DM_AGENT_MASK) << DM_AGENT_SHIFT);
    dst.spawn_id = src.spawn_id;
    dst.epsilon = src.agent_epsilon;
    dst.threshold = (R)src.agent_threshold;
    for (int c = 0; c < 4; ++c) dst.init[c] = (R)src.init_state[c];
    dst.static_share = (R)0;
    if (src.kind == CAV_BODY_PELICAN) {
      const Quad<R> box = to_quad<R>(src.static_box);
      for (int r = 0; r < in.n_roads; ++r) {
        const R q = percentage_of(box, roads[r], (R)tau).value;
        if (r == 0 || q > dst.static_share) dst.static_share = q;
      }
    }
    if (src.agent == CAV_AGENT_EXTERNAL) tb.has_external = 1;
  }
}

template <typename R>
static DevSpawn<R> to_spawn(const CavSpawn& in) {
  DevSpawn<R> out;
  std::memset(&out, 0, sizeof(out));
  out.n_boxes = in.n_boxes; out.n_orient = in.n_orientations;
  for (int i = 0; i < in.n_boxes; ++i)
    for (int c = 0; c < 4; ++c) { out.boxes[i].x[c] = (R)in.boxes[i].x[c]; out.boxes[i].y[c] = (R)in.boxes[i].y[c]; }
  for (int i = 0; i < in.n_orientations; ++i) out.orient[i] = (R)in.orientations[i];
  out.velocity = (R)in.velocity;
  return out;
}

// ---------------------------------------------------------------- small kernels living in this TU
__global__ void live_steps_kernel(const int32_t* t_ep, const uint8_t* done, const uint8_t* err, int64_t n,
                                  unsigned long long* out /* [2]: live steps, errors */) {
  unsigned long long steps = 0, errors = 0;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    if (!done[e]) steps += (unsigned long long)t_ep[e];
    errors += err[e];
  }
  steps = warp_sum(steps);
  errors = warp_sum(errors);
  if ((threadIdx.x & 31) == 0) {
    if (steps) atomicAdd(&out[0], steps);
    if (errors) atomicAdd(&out[1], errors);
  }
}

// DynamicBody.step alone (bodies.py:214-275): SoA state[4][n] in place, actions[2][n].
template <typename R>
__global__ void bodies_step_kernel(const __grid_constant__ DevType<R> k, R* state, const R* actions, int64_t n, R dt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  R st[4] = {state[i], state[n + i], state[2 * n + i], state[3 * n + i]};
  R c = R(1), s = st[3], snapped;
  if (!(st[3] == R(0))) sincos_(st[3], &s, &c);
  body_step(k, st, actions[i], actions[n + i], dt, c, s, snapped);
#pragma unroll
  for (int j = 0; j < 4; ++j) state[j * n + i] = st[j];
}

// DynamicBody.stopping_zones (bodies.py:122-135) written out from the EgoFrame the step kernels use (geometry.cuh): the
// braking rectangle spans [hl, hl + bd] and the reaction rectangle [hl + bd, hl + td] along the heading, the body's width across.
template <typename R>
__global__ void zones_probe_kernel(const __grid_constant__ DevType<R> k, const R* state, const R* steering, R* zones, uint8_t* have,
                                   int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const R x = state[i], y = state[n + i], v = state[2 * n + i], th = state[3 * n + i];
  R steer = steering[i];
  if (rabs(steer) < R(0.0000000000001)) steer = R(0);
  R c = R(1), s = th;
  if (!(th == R(0))) sincos_(th, &s, &c);
  EgoFrame<R> f;
  f.x = x; f.y = y; f.c = c; f.s = s; f.hl = k.hl; f.hw = k.hw;
  f.bd = (v * v) * k.inv_2brake;
  f.td = f.bd + v * R(0.675);
  f.have = !(f.td == R(0)) && (steer == R(0));
  have[i] = f.have ? 1 : 0;
  const R hb = f.bd * R(0.5), hr = (f.td - f.bd) * R(0.5);
  const R centre[2] = {f.hl + hb, f.hl + f.bd + hr}, half[2] = {hb, hr};
#pragma unroll
  for (int z = 0; z < 2; ++z) {
    const R along[4] = {centre[z] - half[z], centre[z] + half[z], centre[z] + half[z], centre[z] - half[z]};
    const R across[4] = {f.hw, f.hw, -f.hw, -f.hw};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      zones[(z * 8 + q) * n + i] = f.have ? x + (along[q] * c - across[q] * s) : nan_<R>();
      zones[(z * 8 + 4 + q) * n + i] = f.have ? y + (along[q] * s + across[q] * c) : nan_<R>();
    }
  }
}

// Shape.intersects / contains / percentage_intersects on n quad pairs (geometry.py:74-87).
template <typename R>
__global__ void geometry_probe_kernel(const R* qa, const R* qb, R* out, int64_t n, R tau) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Quad<R> A, B;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    A.x[c] = qa[c * n + i]; A.y[c] = qa[(4 + c) * n + i];
    B.x[c] = qb[c * n + i]; B.y[c] = qb[(4 + c) * n + i];
  }
  auto clockwise = [](Quad<R>& q) {  // the device predicates assume clockwise rings
    R twice_area = R(0);
#pragma unroll
    for (int c = 0; c < 4; ++c) twice_area += q.x[c] * q.y[(c + 1) & 3] - q.x[(c + 1) & 3] * q.y[c];
    if (twice_area > R(0)) {
      R t = q.x[0]; q.x[0] = q.x[3]; q.x[3] = t; t = q.x[1]; q.x[1] = q.x[2]; q.x[2] = t;
      t = q.y[0]; q.y[0] = q.y[3]; q.y[3] = t; t = q.y[1]; q.y[1] = q.y[2]; q.y[2] = t;
    }
  };
  clockwise(A);
  clockwise(B);
  bool tangent = false;
  const bool hit = intersects(A, aabb_of(A), B, aabb_of(B), tau, tangent);
  bool inside = false;
  R share = R(0);
  if (hit) inside = contains(B, A, tau, tangent);
  if (!(aabb_gap(aabb_of(A), aabb_of(B)) > tau)) {
    const Share<R> sh = percentage_of(A, B, tau);
    share = sh.value;
    tangent |= sh.tangent != 0;
  }
  out[i] = hit ? R(1) : R(0);
  out[n + i] = inside ? R(1) : R(0);
  out[2 * n + i] = share;
  out[3 * n + i] = tangent ? R(1) : R(0);
}

// CAVEnv.info (environment.py:106-117): body_polygons and road_angles of the current state, one thread per env.
// road angle = DynamicBody.line_anchor_relative_angle (bodies.py:206-212): direction from the body to the closest point of
// the major road's centre line (geometry.py:412-421) minus the heading, normalised into (-pi, pi] (geometry.py:380-385);
// NaN stands for the reference's None (the body's box intersects the major road).
template <typename R>
__global__ void info_kernel(const __grid_constant__ DevScenario<R> sc, const __grid_constant__ DenseTables<R> tb,
                            const __grid_constant__ EnvBuffers<R> buf, const Quad<R>* static_quads, R* polygons, R* angles) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, n = buf.n;
  if (e >= n) return;
  const R pi = R(3.14159265358979323846), two_pi = R(6.28318530717958647692);
  for (int b = 0; b < sc.n_bodies; ++b) {
    const int32_t mt = tb.bodies[b].meta;
    const DevType<R>& k = tb.types[mt & DM_TYPE_MASK];
    const R x = buf.state[((int64_t)b * 4 + 0) * n + e], y = buf.state[((int64_t)b * 4 + 1) * n + e];
    const R th = buf.state[((int64_t)b * 4 + 3) * n + e];
    Quad<R> q;
    bool on_road;
    if (mt & DM_PELICAN) {
      q = static_quads[b];
      on_road = (sat_bits(q, sc.quads[0], sc.tau) & GEO_HIT) != 0;
    } else {
      const R c = buf.cs[((int64_t)b * 2 + 0) * n + e], s = buf.cs[((int64_t)b * 2 + 1) * n + e];
      make_box(k.length, k.width, th, c, s, x, y, q);
      if (sc.road_rect[0]) on_road = !(box_margin(Box<R>{x, y, c, s, k.hl, k.hw}, sc.road_box[0]) > R(0));
      else on_road = (sat_bits(q, sc.quads[0], sc.tau) & GEO_HIT) != 0;
    }
    if (polygons) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        polygons[((int64_t)b * 8 + c) * n + e] = q.x[c];
        polygons[((int64_t)b * 8 + 4 + c) * n + e] = q.y[c];
      }
    }
    if (angles) {
      R angle = nan_<R>();
      if (!on_road) {
        const R dx = sc.cl[2] - sc.cl[0], dy = sc.cl[3] - sc.cl[1];
        const R a = (dy * (y - sc.cl[1]) + dx * (x - sc.cl[0])) / ((dx * dx) + (dy * dy));
        const R cx = sc.cl[0] + a * dx, cy = sc.cl[1] + a * dy;
        R radians = atan2_(cy - y, cx - x) - th;
        while (radians <= -pi) radians += two_pi;
        while (radians > pi) radians -= two_pi;
        angle = radians == R(0) ? radians + R(0) : radians;
      }
      angles[(int64_t)b * n + e] = angle;
    }
  }
}

}  // namespace cav

using namespace cav;

// ---------------------------------------------------------------- engine object
struct CavEngine {
  int dtype = CAV_F64, device = 0, m = 0;
  int64_t n = 0, t_global = 0, launches = 0;
  uint64_t seed = 0;
  bool has_external = false, has_device_agents = false;
  bool use_tma = true;  // cavgym_set_step_path: 0 = plain thread-per-env kernel only
  bool zero_copy_host = true;  // cavgym_set_host_path: 0 = always stage host buffers through device copies
  bool dense = false;          // warp-per-env kernels (kernels_dense.cuh): always for m > CAV_SMALL_M, cavgym_set_dense_path otherwise
  DenseTables<double> tb64;
  DenseTables<float> tb32;
  void* d_dense_bodies = nullptr;
  void* d_static_quads = nullptr;   // Quad<R>[m]: PelicanCrossing.static_bounding_box per body (cavgym_info)
  double tau = 1e-7;
  CavScenario host{};
  std::vector<CavBody> bodies;
  std::vector<CavSpawn> spawns;
  DevScenario<double> sc64;
  DevScenario<float> sc32;
  EnvBuffers<double> buf64;
  EnvBuffers<float> buf32;
  std::vector<void*> allocations;
  // host-buffer pipeline (cavgym_step_host)
  static constexpr int kPipe = 3;
  cudaStream_t pipe[kPipe] = {nullptr, nullptr, nullptr};
  int step_ctas_per_sm = 0;       // cap on resident CTAs per SM of the persistent step kernel for the next launch (0 = occupancy)
  int host_ctas_per_sm = CAV_HOST_CTAS_PER_SM;   // the same for the zero-copy host path (cavgym_set_host_path)
  bool host_ready = false;        // streams and staging buffers of the host-buffer entry points all exist
  // launch chaining of the TMA replay kernel (kernels_tma.cuh): sequence number of the last launch, the API call it was made
  // in, its stream and env range; the next cavgym_replay chains to it iff it is the very next API call on this engine
  int32_t* d_tile_gen = nullptr;
  int32_t replay_seq = 0;
  int64_t api_calls = 0, chain_call = -2, chain_lo = 0, chain_span = 0;
  cudaStream_t chain_stream = nullptr;
  bool caller_work_pending = true;   // a call queued work on a caller stream since the last host-buffer call synchronised
  const void* host_seen[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // caller buffers of the last zero-copy call ...
  void* host_mapped[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};       // ... and their device addresses
  void* d_init = nullptr;         // staging for cavgym_reset_host's init_state / mask
  uint8_t* d_mask = nullptr;
  void *d_actions = nullptr, *d_reward = nullptr;
  uint8_t *d_done = nullptr, *d_tangent = nullptr;
  int32_t* d_winner = nullptr;
  unsigned long long* d_scratch = nullptr;
  void* d_quads = nullptr;  // Quad<R>[CAV_MAX_ROADS + CAV_MAX_STATICS] in the engine's type: corner lists for the general fallbacks
  uint64_t fingerprint = 0;      // of the scenario tables' contents (scenario_fingerprint)
  void* d_stage = nullptr;       // cavgym_fork_envs: snapshot of the sources, grown on demand, freed by cavgym_destroy
  size_t stage_bytes = 0;
  // cavgym_set_agent_params: per-env tester parameters [m][n] (epsilon double, threshold real), allocated on first use
  double* d_epsilon = nullptr;
  void* d_threshold = nullptr;
  unsigned int* d_param_flags = nullptr;
  bool epsilon_set = false, threshold_set = false;
  unsigned int* d_regen_flags = nullptr;   // cavgym_regenerate_episodes' key check, allocated on first use

  bool agent_params_set() const { return epsilon_set || threshold_set; }
  size_t real_size() const { return dtype == CAV_F64 ? 8 : 4; }
};

template <typename T>
static int dev_alloc(CavEngine* eng, T** ptr, size_t count, bool zero = true) {
  void* p = nullptr;
  CUDA_TRY(cudaMalloc(&p, count * sizeof(T) > 0 ? count * sizeof(T) : sizeof(T)));
  eng->allocations.push_back(p);
  if (zero) CUDA_TRY(cudaMemset(p, 0, count * sizeof(T)));
  *ptr = (T*)p;
  return CAV_OK;
}

template <typename R>
static int setup_buffers(CavEngine* eng, EnvBuffers<R>& buf) {
  const int64_t n = eng->n, m = eng->m;
  std::memset(&buf, 0, sizeof(buf));
  buf.n = n; buf.lo = 0; buf.hi = n; buf.shard = 0; buf.seed = eng->seed;
  int rc;
  if ((rc = dev_alloc(eng, &buf.state, (size_t)m * 4 * n))) return rc;
  if ((rc = dev_alloc(eng, &buf.action, (size_t)m * 2 * n))) return rc;
  if ((rc = dev_alloc(eng, &buf.agent, (size_t)m * CAV_AGENT_WORDS * n))) return rc;
  if ((rc = dev_alloc(eng, &buf.cs, (size_t)m * 2 * n))) return rc;
  if ((rc = dev_alloc(eng, &buf.liveness, (size_t)m * n))) return rc;
  if ((rc = dev_alloc(eng, &buf.t_ep, (size_t)n))) return rc;
  if ((rc = dev_alloc(eng, &buf.episode, (size_t)n))) return rc;
  if ((rc = dev_alloc(eng, &buf.winner, (size_t)n))) return rc;
  if ((rc = dev_alloc(eng, &buf.active, (size_t)n))) return rc;
  if ((rc = dev_alloc(eng, &buf.done, (size_t)n))) return rc;
  if ((rc = dev_alloc(eng, &buf.err, (size_t)n))) return rc;
  if ((rc = dev_alloc(eng, &buf.stats, (size_t)CAV_N_STATS))) return rc;
  if (!eng->d_tile_gen && (rc = dev_alloc(eng, &eng->d_tile_gen, (size_t)(n / kReplayTile + 2)))) return rc;
  std::vector<DevSpawn<R>> spawns;
  for (const CavSpawn& s : eng->spawns) spawns.push_back(to_spawn<R>(s));
  DevSpawn<R>* d_spawns = nullptr;
  if ((rc = dev_alloc(eng, &d_spawns, spawns.size() ? spawns.size() : 1))) return rc;
  if (!spawns.empty()) CUDA_TRY(cudaMemcpy(d_spawns, spawns.data(), spawns.size() * sizeof(DevSpawn<R>), cudaMemcpyHostToDevice));
  buf.spawns = d_spawns;
  Quad<R> quads[CAV_MAX_ROADS + CAV_MAX_STATICS];
  std::memset(quads, 0, sizeof(quads));
  for (int i = 0; i < eng->host.n_roads; ++i) quads[i] = to_quad<R>(eng->host.roads[i]);
  for (int i = 0; i < eng->host.n_statics; ++i) quads[CAV_MAX_ROADS + i] = to_quad<R>(eng->host.statics[i]);
  Quad<R>* d_quads = nullptr;
  if ((rc = dev_alloc(eng, &d_quads, CAV_MAX_ROADS + CAV_MAX_STATICS))) return rc;
  CUDA_TRY(cudaMemcpy(d_quads, quads, sizeof(quads), cudaMemcpyHostToDevice));
  eng->d_quads = d_quads;
  return CAV_OK;
}

static int rebuild_tables(CavEngine* eng) {
  convert<double>(eng->host, eng->tau, eng->sc64);
  convert<float>(eng->host, eng->tau, eng->sc32);
  eng->sc64.quads = (const Quad<double>*)eng->d_quads;  // only the table of the engine's own type is dereferenced
  eng->sc32.quads = (const Quad<float>*)eng->d_quads;
  std::vector<DenseBody<double>> rows64;
  std::vector<DenseBody<float>> rows32;
  convert_dense<double>(eng->host, eng->tau, eng->tb64, rows64);
  convert_dense<float>(eng->host, eng->tau, eng->tb32, rows32);
  if (eng->d_dense_bodies) {   // allocated by cavgym_create once the device is selected
    if (eng->dtype == CAV_F64) CUDA_TRY(cudaMemcpy(eng->d_dense_bodies, rows64.data(), rows64.size() * sizeof(DenseBody<double>), cudaMemcpyHostToDevice));
    else CUDA_TRY(cudaMemcpy(eng->d_dense_bodies, rows32.data(), rows32.size() * sizeof(DenseBody<float>), cudaMemcpyHostToDevice));
  }
  eng->tb64.bodies = (const DenseBody<double>*)eng->d_dense_bodies;
  eng->tb32.bodies = (const DenseBody<float>*)eng->d_dense_bodies;
  return CAV_OK;
}

static int check_engine(CavEngine* eng) {
  if (!eng) return fail(CAV_EINVAL, "engine is NULL");
  cudaError_t err = cudaSetDevice(eng->device);
  if (err != cudaSuccess) return fail(CAV_ECUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(err));
  eng->api_calls += 1;   // every entry point passes here once: replay launches chain only across ADJACENT calls
  return CAV_OK;
}

static int launch_check(CavEngine* eng, const char* what, int n_launches = 1) {
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(CAV_ECUDA, std::string(what) + ": " + cudaGetErrorString(err));
  eng->launches += n_launches;
  eng->caller_work_pending = true;
  return CAV_OK;
}

template <typename R>
static AgentParams<R> agent_params(const CavEngine* eng) {
  return {eng->epsilon_set ? eng->d_epsilon : nullptr, eng->threshold_set ? (const R*)eng->d_threshold : nullptr};
}

// Per-env tester parameters are honoured by the thread-per-env step, rollout and recording kernels only.
static int refuse_dense_with_params(CavEngine* eng, const char* what) {
  if (eng->dense && eng->agent_params_set())
    return fail(CAV_ESTATE, std::string(what) + ": per-env agent parameters are set (cavgym_set_agent_params) and the warp-per-env "
                            "kernels do not read them; clear them or turn cavgym_set_dense_path off");
  return CAV_OK;
}

static int do_reset(CavEngine* eng, const uint8_t* mask, const void* init, int first_time, cudaStream_t stream) {
  if (eng->dense) {
    if (eng->dtype == CAV_F64) dense_launchers<double>()->reset(eng->sc64, eng->tb64, eng->buf64, mask, (const double*)init, first_time, stream);
    else dense_launchers<float>()->reset(eng->sc32, eng->tb32, eng->buf32, mask, (const float*)init, first_time, stream);
    return launch_check(eng, "dense reset kernel");
  }
  if (eng->dtype == CAV_F64) small_launchers<double>(eng->m)->reset(eng->sc64, eng->buf64, mask, (const double*)init, first_time, stream);
  else small_launchers<float>(eng->m)->reset(eng->sc32, eng->buf32, mask, (const float*)init, first_time, stream);
  return launch_check(eng, "reset kernel");
}

template <typename R> static const DenseTables<R>& dense_tables(const CavEngine* eng);
template <> const DenseTables<double>& dense_tables<double>(const CavEngine* eng) { return eng->tb64; }
template <> const DenseTables<float>& dense_tables<float>(const CavEngine* eng) { return eng->tb32; }

template <typename R>
static int dense_run(CavEngine* eng, const DevScenario<R>& sc, const EnvBuffers<R>& buf, const StepIO<R>& io, int n_steps, int auto_reset,
                     int traj, cudaStream_t stream) {
  if (!dense_launchers<R>()->run(sc, dense_tables<R>(eng), buf, io, eng->t_global, n_steps, auto_reset, traj, eng->has_device_agents, stream))
    return fail(CAV_ECUDA, "dense kernel set-up failed (shared memory opt-in)");
  return launch_check(eng, "dense kernel");
}

template <typename R>
static int step_range_typed(CavEngine* eng, const DevScenario<R>& sc, EnvBuffers<R> buf, const StepIO<R>& io, cudaStream_t stream) {
  if (eng->dense) return dense_run(eng, sc, buf, io, 1, 0, 0, stream);
  if (eng->has_device_agents && eng->agent_params_set()) {
    params_launchers<R>(eng->m)->step(sc, buf, io, agent_params<R>(eng), eng->t_global, stream);
    return launch_check(eng, "step kernel (agent parameters)");
  }
  const SmallLaunchers<R>* k = small_launchers<R>(eng->m);
  int launches = 0;
  if (!eng->has_device_agents && eng->use_tma) {   // replayed actions: persistent TMA-staged kernel over the whole tiles
    int64_t taken = 0;
    if (!k->step_tma(sc, buf, io, eng->t_global, stream, &taken)) return fail(CAV_ECUDA, "TMA step kernel set-up failed");
    if (taken > 0) { buf.lo += taken; ++launches; }
  }
  if (buf.lo < buf.hi) { k->step(sc, buf, io, eng->t_global, eng->has_device_agents, stream); ++launches; }
  return launch_check(eng, "step kernel", launches);
}

// Replayed actions, T fused steps: whole 128-env tiles through the TMA-pipelined kernel, the ragged tail through the
// plain one.  The trajectory pointers of the tail launch are the same (env-indexed rows), only the env range differs.
template <typename R>
static int replay_typed(CavEngine* eng, const DevScenario<R>& sc, EnvBuffers<R> buf, const StepIO<R>& io, int n_steps,
                        cudaStream_t stream, int* launches) {
  if (eng->dense) return dense_run(eng, sc, buf, io, n_steps, 0, 1, stream);
  const SmallLaunchers<R>* k = small_launchers<R>(eng->m);
  if (eng->use_tma) {
    int64_t taken = 0;
    StepIO<R> chain = io;
    chain.tile_gen = eng->d_tile_gen;
    chain.seq = eng->replay_seq + 1;
    // chained to the previous launch iff that was the previous API call on this engine, on this stream, over these envs
    const int64_t span = tma_span(buf, io, kReplayTile, io.done_out != nullptr || io.tangent_out != nullptr);
    chain.chained = eng->d_tile_gen && CAV_REPLAY_CHAIN && eng->chain_call == eng->api_calls - 1 && eng->chain_stream == stream &&
                    eng->chain_lo == buf.lo && eng->chain_span == span;
    if (!k->replay_tma(sc, buf, chain, eng->t_global, n_steps, stream, &taken)) return fail(CAV_ECUDA, "TMA replay kernel set-up failed");
    if (taken > 0) {
      eng->replay_seq += 1;
      eng->chain_call = eng->api_calls; eng->chain_stream = stream; eng->chain_lo = buf.lo; eng->chain_span = taken;
      buf.lo += taken; ++*launches;
    }
  }
  if (buf.lo < buf.hi) { k->replay(sc, buf, io, eng->t_global, n_steps, stream); ++*launches; }
  return CAV_OK;
}

// ---------------------------------------------------------------- snapshots (kernels_snapshot.cuh)
// 64-bit FNV-1a over the scenario's contents: the CavScenario header up to its two pointers, then the spawn and body rows.
// None of the three structs has padding, so equal tables give equal bytes wherever they were compiled.
static uint64_t scenario_fingerprint(const CavScenario& sc) {
  uint64_t h = 0xcbf29ce484222325ull;
  auto mix = [&h](const void* p, size_t bytes) {
    const unsigned char* c = static_cast<const unsigned char*>(p);
    for (size_t i = 0; i < bytes; ++i) { h ^= c[i]; h *= 0x100000001b3ull; }
  };
  mix(&sc, offsetof(CavScenario, spawns));
  if (sc.n_spawns > 0) mix(sc.spawns, sizeof(CavSpawn) * (size_t)sc.n_spawns);
  mix(sc.bodies, sizeof(CavBody) * (size_t)sc.n_bodies);
  return h;
}

static void snapshot_layout(const CavEngine* eng, int64_t k, CavSnapshotLayout* out) {
  auto align = [](int64_t bytes) { return (bytes + 255) & ~(int64_t)255; };
  std::memset(out, 0, sizeof(*out));
  out->version = CAV_SNAPSHOT_VERSION;
  out->dtype = eng->dtype;
  out->m = eng->m;
  out->k = k;
  out->real_rows = (int64_t)eng->m * (4 + 2 + CAV_AGENT_WORDS + 2);   // state, action, agent, cs
  out->i32_rows = (int64_t)eng->m + 4;                                 // liveness, t_ep, episode, winner, active
  out->u8_rows = 2;                                                    // done, err
  out->real_offset = 0;
  out->i32_offset = align(out->real_rows * k * (int64_t)eng->real_size());
  out->u8_offset = out->i32_offset + align(out->i32_rows * k * 4);
  out->total_bytes = out->u8_offset + align(out->u8_rows * k);
  out->fingerprint = eng->fingerprint;
}

template <typename T>
static void add_rows(SnapTable<T>& t, void* engine, char* snap, int64_t rows) {
  const int s = t.n_seg++;
  t.eng[s] = static_cast<T*>(engine);
  t.snap[s] = reinterpret_cast<T*>(snap);
  t.row_end[s] = (s ? t.row_end[s - 1] : 0) + rows;
}

// Every row of the k selected envs between the engine and `snap` (laid out by snapshot_layout): 3 launches in fp64 (8-, 4-
// and 1-byte rows), 2 in fp32 (the 4-byte reals share a launch with the int32 rows).
template <typename R>
static int move_envs(CavEngine* eng, const EnvBuffers<R>& buf, const int64_t* idx, int64_t k, char* snap, bool to_snapshot,
                     cudaStream_t stream) {
  using W = typename std::conditional<sizeof(R) == 8, unsigned long long, uint32_t>::type;
  CavSnapshotLayout L;
  snapshot_layout(eng, k, &L);
  const int64_t m = eng->m;
  SnapTable<W> reals{};
  SnapTable<uint32_t> words{};
  SnapTable<uint8_t> bytes{};
  char* p = snap + L.real_offset;
  const int64_t real_row = k * (int64_t)sizeof(R);
  add_rows(reals, buf.state, p, m * 4);                  p += m * 4 * real_row;
  add_rows(reals, buf.action, p, m * 2);                 p += m * 2 * real_row;
  add_rows(reals, buf.agent, p, m * CAV_AGENT_WORDS);    p += m * CAV_AGENT_WORDS * real_row;
  add_rows(reals, buf.cs, p, m * 2);
  auto add_ints = [&](SnapTable<uint32_t>& ints) {
    char* q = snap + L.i32_offset;
    add_rows(ints, buf.liveness, q, m);                  q += m * k * 4;
    add_rows(ints, buf.t_ep, q, 1);                      q += k * 4;
    add_rows(ints, buf.episode, q, 1);                   q += k * 4;
    add_rows(ints, buf.winner, q, 1);                    q += k * 4;
    add_rows(ints, buf.active, q, 1);
  };
  if constexpr (sizeof(R) == 4) add_ints(reals);   // fp32: the int32 rows continue the 4-byte table
  else add_ints(words);
  add_rows(bytes, buf.done, snap + L.u8_offset, 1);
  add_rows(bytes, buf.err, snap + L.u8_offset + k, 1);
  const char* what = to_snapshot ? "snapshot gather kernel" : "snapshot scatter kernel";
  if (!idx && k % 16 == 0) {
    SnapTable<uint4> wide{};
    append_wide(wide, reals);
    append_wide(wide, words);
    append_wide(wide, bytes);
    wide.n = wide.k = k / 16;
    wide.idx = nullptr;
    wide.to_snapshot = to_snapshot ? 1 : 0;
    launch_snapshot(wide, stream);
    return launch_check(eng, what);
  }
  auto run = [&](auto& t) {
    t.n = eng->n; t.k = k; t.idx = idx; t.to_snapshot = to_snapshot ? 1 : 0;
    launch_snapshot(t, stream);
  };
  run(reals);
  if (words.n_seg) run(words);
  run(bytes);
  return launch_check(eng, what, words.n_seg ? 3 : 2);
}

static int move_envs(CavEngine* eng, const int64_t* idx, int64_t k, void* snap, bool to_snapshot, cudaStream_t stream) {
  return eng->dtype == CAV_F64 ? move_envs(eng, eng->buf64, idx, k, (char*)snap, to_snapshot, stream)
                               : move_envs(eng, eng->buf32, idx, k, (char*)snap, to_snapshot, stream);
}

// ---------------------------------------------------------------- recorded rollouts
template <typename R>
static int rollout_record_typed(CavEngine* eng, const DevScenario<R>& sc, const EnvBuffers<R>& buf, const CavRolloutRecord& r,
                                int n_steps, int auto_reset, cudaStream_t stream) {
  const RolloutRecord<R> rec{(R*)r.observation, (R*)r.action, (R*)r.state, (R*)r.reward, r.done, r.winner, r.tangent, r.timestep};
  if (eng->dense) {
    if (!dense_launchers<R>()->rollout_record(sc, dense_tables<R>(eng), buf, rec, eng->t_global, n_steps, auto_reset, stream))
      return fail(CAV_ECUDA, "dense kernel set-up failed (shared memory opt-in)");
    return launch_check(eng, "dense record kernel");
  }
  if (eng->agent_params_set()) {
    params_launchers<R>(eng->m)->rollout_record(sc, buf, rec, agent_params<R>(eng), eng->t_global, n_steps, auto_reset, stream);
    return launch_check(eng, "rollout record kernel (agent parameters)");
  }
  rollout_record_launcher<R>(eng->m)(sc, buf, rec, eng->t_global, n_steps, auto_reset, stream);
  return launch_check(eng, "rollout record kernel");
}

extern "C" {

const char* cavgym_last_error(void) { return g_error.c_str(); }
const char* cavgym_version(void) { return "cavgym_b200 0.1.0 (sm_100a)"; }

int cavgym_host_alloc(size_t bytes, int write_combined, void** out) {
  if (!out || bytes == 0) return fail(CAV_EINVAL, "out is NULL or bytes is 0");
  *out = nullptr;
  CUDA_TRY(cudaHostAlloc(out, bytes, cudaHostAllocMapped | cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0)));
  return CAV_OK;
}

int cavgym_host_free(void* ptr) {
  if (!ptr) return CAV_OK;
  CUDA_TRY(cudaFreeHost(ptr));
  return CAV_OK;
}

int cavgym_create(const CavScenario* tables, int64_t n_envs, int dtype, int device, uint64_t seed, CavEngine** out) {
  if (!tables || !out) return fail(CAV_EINVAL, "tables/out is NULL");
  *out = nullptr;
  if (n_envs <= 0) return fail(CAV_EINVAL, "n_envs must be positive");
  if (dtype != CAV_F64 && dtype != CAV_F32) return fail(CAV_EINVAL, "dtype must be CAV_F64 or CAV_F32");
  if (tables->n_bodies < 1 || !tables->bodies) return fail(CAV_EINVAL, "scenario has no bodies");
  if (tables->n_bodies > CAV_MAX_BODIES) return fail(CAV_EINVAL, "more than CAV_MAX_BODIES bodies");
  if (tables->n_bodies <= CAV_SMALL_M && (dtype == CAV_F64 ? (const void*)small_launchers<double>(tables->n_bodies)->step : (const void*)small_launchers<float>(tables->n_bodies)->step) == nullptr)
    return fail(CAV_EINVAL, "this development build of the library was compiled without this body count (CAVGYM_ONLY_M)");
  if (tables->n_roads < 1 || tables->n_roads > CAV_MAX_ROADS || tables->n_statics < 0 || tables->n_statics > CAV_MAX_STATICS ||
      tables->n_types < 0 || tables->n_types > CAV_MAX_TYPES)
    return fail(CAV_EINVAL, "road/static/type counts out of range");
  if (tables->n_spawns < 0 || (tables->n_spawns > 0 && !tables->spawns)) return fail(CAV_EINVAL, "n_spawns < 0 or spawns is NULL");
  for (int k = 0; k < tables->n_spawns; ++k) {   // spawn_body indexes fixed arrays with these counts
    const CavSpawn& sp = tables->spawns[k];
    if (sp.n_boxes < 1 || sp.n_boxes > CAV_MAX_SPAWN_BOXES || sp.n_orientations < 1 || sp.n_orientations > CAV_MAX_SPAWN_ORIENT)
      return fail(CAV_EINVAL, "spawn n_boxes / n_orientations out of range");
  }
  if (!(tables->time_resolution > 0) || !(tables->viewer_width > 0)) return fail(CAV_EINVAL, "time_resolution and viewer_width must be > 0");
  if (tables->max_timesteps < 1) return fail(CAV_EINVAL, "max_timesteps must be >= 1");
  if (tables->bodies[0].kind != CAV_BODY_DYNAMIC) return fail(CAV_EINVAL, "the ego (body 0) must be a dynamic body");
  for (int b = 0; b < tables->n_bodies; ++b) {
    const CavBody& body = tables->bodies[b];
    if (body.kind == CAV_BODY_DYNAMIC && (body.type_id < 0 || body.type_id >= tables->n_types))
      return fail(CAV_EINVAL, "body type_id out of range");
    if ((body.flags & CAV_FLAG_SPAWN) && (body.spawn_id < 0 || body.spawn_id >= tables->n_spawns || !tables->spawns))
      return fail(CAV_EINVAL, "spawn_id out of range");
    if (body.agent < CAV_AGENT_EXTERNAL || body.agent > CAV_AGENT_ELECTION) return fail(CAV_EINVAL, "unknown agent kind");
    if (body.agent == CAV_AGENT_ELECTION && tables->n_bodies > CAV_SMALL_M)
      return fail(CAV_EINVAL, "election agents are arbitrated in the thread-per-env kernels: at most CAV_SMALL_M bodies");
    if ((body.agent == CAV_AGENT_RANDOM_CONSTRAINED || body.agent == CAV_AGENT_PROXIMITY || body.agent == CAV_AGENT_ELECTION) &&
        !(body.kind == CAV_BODY_DYNAMIC && (body.flags & CAV_FLAG_PEDESTRIAN)))
      return fail(CAV_EINVAL, "crossing agents need a Pedestrian body (config.py:358-396)");
  }
  CUDA_TRY(cudaSetDevice(device));
  CavEngine* eng = new (std::nothrow) CavEngine();
  if (!eng) return fail(CAV_ENOMEM, "out of host memory");
  eng->dtype = dtype; eng->device = device; eng->m = tables->n_bodies; eng->n = n_envs; eng->seed = seed;
  eng->tau = dtype == CAV_F64 ? 1e-7 : 5e-2;
  eng->host = *tables;
  eng->bodies.assign(tables->bodies, tables->bodies + tables->n_bodies);
  if (tables->n_spawns > 0) eng->spawns.assign(tables->spawns, tables->spawns + tables->n_spawns);
  eng->host.bodies = eng->bodies.data();
  eng->host.spawns = eng->spawns.data();
  eng->fingerprint = scenario_fingerprint(eng->host);
  for (const CavBody& body : eng->bodies) {
    if (body.agent == CAV_AGENT_EXTERNAL) eng->has_external = true; else eng->has_device_agents = true;
  }
  eng->dense = eng->m > CAV_SMALL_M;
  int rc = dtype == CAV_F64 ? setup_buffers(eng, eng->buf64) : setup_buffers(eng, eng->buf32);
  if (rc == CAV_OK) {
    char* rows = nullptr;
    rc = dev_alloc(eng, &rows, (size_t)eng->m * (dtype == CAV_F64 ? sizeof(DenseBody<double>) : sizeof(DenseBody<float>)));
    eng->d_dense_bodies = rows;
  }
  if (rc == CAV_OK) rc = rebuild_tables(eng);
  if (rc == CAV_OK) {   // static boxes of PelicanCrossing bodies, in the engine's type
    const size_t quad_bytes = dtype == CAV_F64 ? sizeof(Quad<double>) : sizeof(Quad<float>);
    char* quads = nullptr;
    rc = dev_alloc(eng, &quads, (size_t)eng->m * quad_bytes);
    eng->d_static_quads = quads;
    if (rc == CAV_OK) {
      std::vector<char> host((size_t)eng->m * quad_bytes, 0);
      for (int b = 0; b < eng->m; ++b) {
        if (eng->bodies[(size_t)b].kind != CAV_BODY_PELICAN) continue;
        if (dtype == CAV_F64) { const Quad<double> q = to_quad<double>(eng->bodies[(size_t)b].static_box); std::memcpy(&host[(size_t)b * quad_bytes], &q, quad_bytes); }
        else { const Quad<float> q = to_quad<float>(eng->bodies[(size_t)b].static_box); std::memcpy(&host[(size_t)b * quad_bytes], &q, quad_bytes); }
      }
      cudaError_t err = cudaMemcpy(quads, host.data(), host.size(), cudaMemcpyHostToDevice);
      if (err != cudaSuccess) rc = fail(CAV_ECUDA, std::string("static quads: ") + cudaGetErrorString(err));
    }
  }
  if (rc == CAV_OK) rc = dev_alloc(eng, &eng->d_scratch, 2);
  if (rc == CAV_OK) rc = do_reset(eng, nullptr, nullptr, 1, nullptr);  // constructor-time spawn (bodies.py:296)
  if (rc == CAV_OK) {
    cudaError_t err = cudaDeviceSynchronize();
    if (err != cudaSuccess) rc = fail(CAV_ECUDA, std::string("create: ") + cudaGetErrorString(err));
  }
  if (rc != CAV_OK) { cavgym_destroy(eng); return rc; }
  *out = eng;
  return CAV_OK;
}

int cavgym_destroy(CavEngine* eng) {
  if (!eng) return CAV_OK;
  cudaSetDevice(eng->device);
  cudaDeviceSynchronize();
  for (void* p : eng->allocations) cudaFree(p);
  if (eng->d_stage) cudaFree(eng->d_stage);
  for (cudaStream_t s : eng->pipe) if (s) cudaStreamDestroy(s);
  delete eng;
  return CAV_OK;
}

int cavgym_set_shard(CavEngine* eng, int64_t offset) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (offset < 0 || offset + eng->n > ((int64_t)1 << 40)) return fail(CAV_EINVAL, "global env ids must fit 40 bits");
  eng->buf64.shard = offset; eng->buf32.shard = offset;
  rc = do_reset(eng, nullptr, nullptr, 1, nullptr);  // redo the constructor-time spawn with the global ids
  if (rc) return rc;
  CUDA_TRY(cudaDeviceSynchronize());
  return CAV_OK;
}

int cavgym_reset(CavEngine* eng, const uint8_t* mask, const void* init_state, cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  return do_reset(eng, mask, init_state, 0, stream);
}

static int step_range(CavEngine* eng, int64_t lo, int64_t hi, const void* actions, void* state_out, void* reward_out,
                      uint8_t* done_out, int32_t* winner_out, uint8_t* tangent_out, cudaStream_t stream) {
  if (eng->dtype == CAV_F64) {
    EnvBuffers<double> buf = eng->buf64; buf.lo = lo; buf.hi = hi;
    StepIO<double> io{(const double*)actions, (double*)state_out, (double*)reward_out, done_out, winner_out, tangent_out, eng->step_ctas_per_sm};
    return step_range_typed(eng, eng->sc64, buf, io, stream);
  }
  EnvBuffers<float> buf = eng->buf32; buf.lo = lo; buf.hi = hi;
  StepIO<float> io{(const float*)actions, (float*)state_out, (float*)reward_out, done_out, winner_out, tangent_out, eng->step_ctas_per_sm};
  return step_range_typed(eng, eng->sc32, buf, io, stream);
}

int cavgym_step(CavEngine* eng, const void* actions, void* state_out, void* reward_out, uint8_t* done_out, int32_t* winner_out,
                uint8_t* tangent_flag_out, cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!actions && eng->has_external) return fail(CAV_EINVAL, "actions is NULL but a body has CAV_AGENT_EXTERNAL");
  if ((rc = refuse_dense_with_params(eng, "cavgym_step"))) return rc;
  rc = step_range(eng, 0, eng->n, actions, state_out, reward_out, done_out, winner_out, tangent_flag_out, stream);
  if (rc) return rc;
  eng->t_global += 1;
  return CAV_OK;
}

int cavgym_rollout(CavEngine* eng, int n_steps, int auto_reset, cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (n_steps < 0) return fail(CAV_EINVAL, "n_steps must be >= 0");
  if (eng->has_external) return fail(CAV_ESTATE, "cavgym_rollout needs an on-device agent for every body");
  if ((rc = refuse_dense_with_params(eng, "cavgym_rollout"))) return rc;
  if (n_steps == 0) return CAV_OK;
  if (eng->dense) {
    const StepIO<double> io64{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0};
    const StepIO<float> io32{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0};
    rc = eng->dtype == CAV_F64 ? dense_run(eng, eng->sc64, eng->buf64, io64, n_steps, auto_reset, 0, stream)
                               : dense_run(eng, eng->sc32, eng->buf32, io32, n_steps, auto_reset, 0, stream);
    if (rc) return rc;
    eng->t_global += n_steps;
    return CAV_OK;
  }
  if (eng->agent_params_set()) {
    if (eng->dtype == CAV_F64)
      params_launchers<double>(eng->m)->rollout(eng->sc64, eng->buf64, agent_params<double>(eng), eng->t_global, n_steps, auto_reset, stream);
    else
      params_launchers<float>(eng->m)->rollout(eng->sc32, eng->buf32, agent_params<float>(eng), eng->t_global, n_steps, auto_reset, stream);
  } else if (eng->dtype == CAV_F64) {
    small_launchers<double>(eng->m)->rollout(eng->sc64, eng->buf64, eng->t_global, n_steps, auto_reset, stream);
  } else {
    small_launchers<float>(eng->m)->rollout(eng->sc32, eng->buf32, eng->t_global, n_steps, auto_reset, stream);
  }
  rc = launch_check(eng, "rollout kernel");
  if (rc) return rc;
  eng->t_global += n_steps;
  return CAV_OK;
}

int cavgym_rollout_record(CavEngine* eng, int n_steps, int auto_reset, const CavRolloutRecord* rec, cudaStream_t stream) {
  if (!rec || !(rec->observation || rec->action || rec->state || rec->reward || rec->done || rec->winner || rec->tangent || rec->timestep))
    return cavgym_rollout(eng, n_steps, auto_reset, stream);
  int rc = check_engine(eng);
  if (rc) return rc;
  if (n_steps < 0) return fail(CAV_EINVAL, "n_steps must be >= 0");
  if (eng->has_external) return fail(CAV_ESTATE, "cavgym_rollout_record needs an on-device agent for every body");
  if ((rc = refuse_dense_with_params(eng, "cavgym_rollout_record"))) return rc;
  if (n_steps == 0) return CAV_OK;
  rc = eng->dtype == CAV_F64 ? rollout_record_typed(eng, eng->sc64, eng->buf64, *rec, n_steps, auto_reset, stream)
                             : rollout_record_typed(eng, eng->sc32, eng->buf32, *rec, n_steps, auto_reset, stream);
  if (rc) return rc;
  eng->t_global += n_steps;
  return CAV_OK;
}

int cavgym_rollout_until(CavEngine* eng, int n_steps, double level, uint64_t salt, void* score, uint8_t* status, cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!score || !status) return fail(CAV_EINVAL, "score/status is NULL");
  if (n_steps < 0) return fail(CAV_EINVAL, "n_steps must be >= 0");
  if (std::isnan(level)) return fail(CAV_EINVAL, "level is NaN");
  bool pedestrian = false;
  for (int b = 1; b < eng->m; ++b) pedestrian = pedestrian || (eng->bodies[(size_t)b].flags & CAV_FLAG_PEDESTRIAN) != 0;
  if (!eng->host.terminate_ego_zones || !pedestrian)
    return fail(CAV_EINVAL, "no tester can win this scenario: cavgym_rollout_until needs terminate_ego_zones and a Pedestrian body");
  if (eng->has_external) return fail(CAV_ESTATE, "cavgym_rollout_until needs an on-device agent for every body");
  if (eng->dense) return fail(CAV_ESTATE, "cavgym_rollout_until runs on the thread-per-environment path only (at most CAV_SMALL_M bodies, "
                                          "cavgym_set_dense_path off)");
  if (eng->agent_params_set())
    return fail(CAV_ESTATE, "cavgym_rollout_until does not read per-env agent parameters: clear them (cavgym_set_agent_params) first");
  if (n_steps == 0) return CAV_OK;
  if (eng->dtype == CAV_F64)
    rollout_until_launcher<double>(eng->m)(eng->sc64, eng->buf64, (double*)score, status, level, salt, eng->t_global, n_steps, stream);
  else
    rollout_until_launcher<float>(eng->m)(eng->sc32, eng->buf32, (float*)score, status, level, salt, eng->t_global, n_steps, stream);
  rc = launch_check(eng, "rollout until kernel");
  if (rc) return rc;
  eng->t_global += n_steps;
  return CAV_OK;
}

int cavgym_regenerate_episodes(CavEngine* eng, const int64_t* env_ids, const int32_t* episodes, int n_steps, const CavRolloutRecord* rec,
                               cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!env_ids || !episodes) return fail(CAV_EINVAL, "env_ids/episodes is NULL");
  if (n_steps < 0) return fail(CAV_EINVAL, "n_steps must be >= 0");
  if (eng->has_external)
    return fail(CAV_ESTATE, "cavgym_regenerate_episodes needs an on-device agent for every body (external actions came from the caller)");
  for (int b = 0; b < eng->m; ++b)
    if (eng->bodies[(size_t)b].agent == CAV_AGENT_ELECTION)
      return fail(CAV_ESTATE, "cavgym_regenerate_episodes: an election outlives episodes, so an episode depends on the ones before it");
  if (eng->dense)
    return fail(CAV_ESTATE, "cavgym_regenerate_episodes runs on the thread-per-environment path only (at most CAV_SMALL_M bodies, "
                            "cavgym_set_dense_path off)");
  if (eng->buf64.uni_override || eng->buf64.spawn_override)
    return fail(CAV_ESTATE, "cavgym_regenerate_episodes draws from the engine's random streams: clear the uniform / spawn overrides");
  if (!eng->d_regen_flags && (rc = dev_alloc(eng, &eng->d_regen_flags, 1))) return rc;
  CUDA_TRY(cudaMemsetAsync(eng->d_regen_flags, 0, sizeof(unsigned int), stream));
  check_regen_keys_kernel<<<148 * 4, 256, 0, stream>>>(env_ids, episodes, eng->n, eng->d_regen_flags);
  if ((rc = launch_check(eng, "regeneration key check kernel"))) return rc;
  unsigned int bad = 0;
  CUDA_TRY(cudaMemcpyAsync(&bad, eng->d_regen_flags, sizeof(bad), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  if (bad & 1u) return fail(CAV_EINVAL, "env id outside [0, 2^40)");
  if (bad & 2u) return fail(CAV_EINVAL, "negative episode number");
  const CavRolloutRecord none{};
  const CavRolloutRecord& r = rec ? *rec : none;
  if (eng->dtype == CAV_F64) {
    const RolloutRecord<double> slabs{(double*)r.observation, (double*)r.action, (double*)r.state, (double*)r.reward, r.done, r.winner,
                                      r.tangent, r.timestep};
    regenerate_launcher<double>(eng->m)(eng->sc64, eng->buf64, slabs, agent_params<double>(eng), env_ids, episodes, eng->t_global,
                                        n_steps, stream);
  } else {
    const RolloutRecord<float> slabs{(float*)r.observation, (float*)r.action, (float*)r.state, (float*)r.reward, r.done, r.winner,
                                     r.tangent, r.timestep};
    regenerate_launcher<float>(eng->m)(eng->sc32, eng->buf32, slabs, agent_params<float>(eng), env_ids, episodes, eng->t_global,
                                       n_steps, stream);
  }
  if ((rc = launch_check(eng, "regeneration kernel"))) return rc;
  eng->t_global += n_steps;
  return CAV_OK;
}

int cavgym_set_agent_params(CavEngine* eng, const double* epsilon, const void* threshold, cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!epsilon && !threshold) {
    eng->epsilon_set = eng->threshold_set = false;
    return CAV_OK;
  }
  if (eng->m > CAV_SMALL_M)
    return fail(CAV_ESTATE, "per-env agent parameters are read by the thread-per-environment kernels only (at most CAV_SMALL_M bodies)");
  uint32_t eps_rows = 0, thr_rows = 0;   // bit b: body b's agent reads that row
  for (int b = 0; b < eng->m; ++b) {
    const int agent = eng->bodies[(size_t)b].agent;
    if (agent == CAV_AGENT_RANDOM || agent == CAV_AGENT_RANDOM_CONSTRAINED) eps_rows |= 1u << b;
    if (agent == CAV_AGENT_PROXIMITY || agent == CAV_AGENT_ELECTION) thr_rows |= 1u << b;
  }
  const size_t count = (size_t)eng->m * (size_t)eng->n;
  if (!eng->d_param_flags) {
    if ((rc = dev_alloc(eng, &eng->d_param_flags, 1))) return rc;
    if ((rc = dev_alloc(eng, &eng->d_epsilon, count, false))) return rc;
    char* thr = nullptr;
    if ((rc = dev_alloc(eng, &thr, count * eng->real_size(), false))) return rc;
    eng->d_threshold = thr;
  }
  // the caller's arrays are checked before they are copied: a refused call leaves the engine's parameters as they were
  CUDA_TRY(cudaMemsetAsync(eng->d_param_flags, 0, sizeof(unsigned int), stream));
  if (eng->dtype == CAV_F64)
    check_agent_params_kernel<double><<<148 * 4, 256, 0, stream>>>(epsilon, (const double*)threshold, eng->n, eng->m, eps_rows, thr_rows,
                                                                  eng->d_param_flags);
  else
    check_agent_params_kernel<float><<<148 * 4, 256, 0, stream>>>(epsilon, (const float*)threshold, eng->n, eng->m, eps_rows, thr_rows,
                                                                 eng->d_param_flags);
  if ((rc = launch_check(eng, "agent parameter check kernel"))) return rc;
  unsigned int bad = 0;
  CUDA_TRY(cudaMemcpyAsync(&bad, eng->d_param_flags, sizeof(bad), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  if (bad & 1u) return fail(CAV_EINVAL, "epsilon outside [0, 1] (or NaN) in a row a RandomAgent / RandomConstrainedAgent reads");
  if (bad & 2u) return fail(CAV_EINVAL, "threshold not finite and > 0 in a row a ProximityAgent / ElectionAgent reads");
  if (epsilon) CUDA_TRY(cudaMemcpyAsync(eng->d_epsilon, epsilon, count * sizeof(double), cudaMemcpyDeviceToDevice, stream));
  if (threshold) CUDA_TRY(cudaMemcpyAsync(eng->d_threshold, threshold, count * eng->real_size(), cudaMemcpyDeviceToDevice, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  eng->epsilon_set = epsilon != nullptr;
  eng->threshold_set = threshold != nullptr;
  return CAV_OK;
}

int cavgym_replay(CavEngine* eng, int n_steps, const void* actions, void* state_traj, void* reward_traj, uint8_t* done_traj,
                  int32_t* winner_traj, uint8_t* tangent_traj, cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (n_steps < 0) return fail(CAV_EINVAL, "n_steps must be >= 0");
  if (!actions) return fail(CAV_EINVAL, "actions is NULL");
  if (eng->has_device_agents) return fail(CAV_ESTATE, "cavgym_replay needs CAV_AGENT_EXTERNAL for every body");
  if (n_steps == 0) return CAV_OK;
  int launches = 0;
  if (eng->dtype == CAV_F64) {
    StepIO<double> io{(const double*)actions, (double*)state_traj, (double*)reward_traj, done_traj, winner_traj, tangent_traj, 0};
    rc = replay_typed(eng, eng->sc64, eng->buf64, io, n_steps, stream, &launches);
  } else {
    StepIO<float> io{(const float*)actions, (float*)state_traj, (float*)reward_traj, done_traj, winner_traj, tangent_traj, 0};
    rc = replay_typed(eng, eng->sc32, eng->buf32, io, n_steps, stream, &launches);
  }
  if (rc) return rc;
  if (!eng->dense) rc = launch_check(eng, "replay kernel", launches);
  if (rc) return rc;
  eng->t_global += n_steps;
  return CAV_OK;
}

// Streams and staging buffers of the host-buffer entry points, created on first use.  `host_ready` is only set once every
// allocation has succeeded; a failure part-way leaves the pieces on eng->allocations (freed by cavgym_destroy) and the
// next call starts over instead of running with null staging pointers.
static int host_setup(CavEngine* eng) {
  if (eng->host_ready) return CAV_OK;
  int rc = CAV_OK;
  const int64_t n = eng->n, m = eng->m;
  const size_t rs = eng->real_size();
  for (auto& s : eng->pipe)
    if (!s) CUDA_TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  void* p = nullptr;
  CUDA_TRY(cudaMalloc(&p, (size_t)m * 2 * n * rs)); eng->allocations.push_back(p); eng->d_actions = p;
  CUDA_TRY(cudaMalloc(&p, (size_t)m * n * rs)); eng->allocations.push_back(p); eng->d_reward = p;
  CUDA_TRY(cudaMalloc(&p, (size_t)m * 4 * n * rs)); eng->allocations.push_back(p); eng->d_init = p;
  if ((rc = dev_alloc(eng, &eng->d_done, (size_t)n))) return rc;
  if ((rc = dev_alloc(eng, &eng->d_tangent, (size_t)n))) return rc;
  if ((rc = dev_alloc(eng, &eng->d_winner, (size_t)n))) return rc;
  if ((rc = dev_alloc(eng, &eng->d_mask, (size_t)n))) return rc;
  eng->host_ready = true;
  return CAV_OK;
}

// Host buffers: env range split into chunks, each chunk's H2D copy -> kernel -> D2H copies queued on one of
// kPipe streams so that copies of one chunk overlap the kernel and copies of the others (PCIe is full duplex).
int cavgym_step_host(CavEngine* eng, const void* actions, void* state_out, void* reward_out, uint8_t* done_out,
                     int32_t* winner_out, uint8_t* tangent_flag_out) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!actions && eng->has_external) return fail(CAV_EINVAL, "actions is NULL but a body has CAV_AGENT_EXTERNAL");
  if ((rc = refuse_dense_with_params(eng, "cavgym_step_host"))) return rc;
  const int64_t n = eng->n, m = eng->m;
  const size_t rs = eng->real_size();
  if ((rc = host_setup(eng))) return rc;
  // Order after whatever the caller queued on its own streams (a reset on torch's stream, say) — only when some call has
  // queued such work since this entry point last synchronised: back-to-back host steps pay no device-wide synchronise.
  if (eng->caller_work_pending) CUDA_TRY(cudaDeviceSynchronize());

  // Zero-copy path: when every caller buffer is pinned (page-locked, mapped) host memory, the step kernel reads the
  // actions and writes the results over PCIe itself — the TMA producer warp's bulk copies take host addresses just as
  // they take HBM addresses — so the whole call is ONE launch with transfers and arithmetic overlapped tile by tile,
  // instead of a chain of chunked cudaMemcpyAsync calls whose launch overheads dominate at this batch size.
  if (eng->zero_copy_host) {
    const void* host[6] = {actions, state_out, reward_out, done_out, winner_out, tangent_flag_out};
    bool all_mapped = true;
    if (memcmp(host, eng->host_seen, sizeof(host)) != 0) {   // new buffers: ask the driver once, remember the answer
      for (int i = 0; i < 6; ++i) eng->host_seen[i] = nullptr;
      void* dev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
      for (int i = 0; i < 6 && all_mapped; ++i) {
        if (!host[i]) continue;
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, host[i]) != cudaSuccess) { cudaGetLastError(); all_mapped = false; break; }
        if (attr.type == cudaMemoryTypeHost && attr.devicePointer) dev[i] = attr.devicePointer;
        else all_mapped = false;
      }
      if (all_mapped)
        for (int i = 0; i < 6; ++i) { eng->host_seen[i] = host[i]; eng->host_mapped[i] = dev[i]; }
    }
    if (all_mapped) {
      void** dev = eng->host_mapped;
      cudaStream_t s = eng->pipe[0];
      // (the CTA count is a tuning knob of cavgym_set_host_path; measured at 65,536 envs: 157 / 155 / 155 us per call with
      //  1 / 2 / 3 CTAs per SM, 157 us with the plain kernel on the same mapped buffers, 161-173 us with the actions brought
      //  in by chunked DMA copies instead — the call is bound by the PCIe link, scripts/e2e_breakdown.py)
      eng->step_ctas_per_sm = eng->host_ctas_per_sm;
      rc = step_range(eng, 0, n, dev[0], dev[1], dev[2], (uint8_t*)dev[3], (int32_t*)dev[4], (uint8_t*)dev[5], s);
      eng->step_ctas_per_sm = 0;
      if (rc) return rc;
      CUDA_TRY(cudaStreamSynchronize(s));
      eng->caller_work_pending = false;
      eng->t_global += 1;
      return CAV_OK;
    }
  }
  const int64_t chunks = n >= (1 << 16) ? 8 : (n >= (1 << 12) ? 2 : 1);
  char* d_state = (char*)(eng->dtype == CAV_F64 ? (void*)eng->buf64.state : (void*)eng->buf32.state);
  for (int64_t c = 0; c < chunks; ++c) {
    const int64_t lo = n * c / chunks, hi = n * (c + 1) / chunks, w = hi - lo;
    if (w <= 0) continue;
    cudaStream_t s = eng->pipe[c % CavEngine::kPipe];
    if (actions)
      CUDA_TRY(cudaMemcpy2DAsync((char*)eng->d_actions + lo * rs, n * rs, (const char*)actions + lo * rs, n * rs, w * rs, m * 2,
                                 cudaMemcpyHostToDevice, s));
    rc = step_range(eng, lo, hi, actions ? eng->d_actions : nullptr, nullptr, reward_out ? eng->d_reward : nullptr,
                    done_out ? eng->d_done : nullptr, winner_out ? eng->d_winner : nullptr,
                    tangent_flag_out ? eng->d_tangent : nullptr, s);
    if (rc) return rc;
    if (state_out)
      CUDA_TRY(cudaMemcpy2DAsync((char*)state_out + lo * rs, n * rs, d_state + lo * rs, n * rs, w * rs, m * 4, cudaMemcpyDeviceToHost, s));
    if (reward_out)
      CUDA_TRY(cudaMemcpy2DAsync((char*)reward_out + lo * rs, n * rs, (char*)eng->d_reward + lo * rs, n * rs, w * rs, m,
                                 cudaMemcpyDeviceToHost, s));
    if (done_out) CUDA_TRY(cudaMemcpyAsync(done_out + lo, eng->d_done + lo, w, cudaMemcpyDeviceToHost, s));
    if (winner_out) CUDA_TRY(cudaMemcpyAsync(winner_out + lo, eng->d_winner + lo, w * 4, cudaMemcpyDeviceToHost, s));
    if (tangent_flag_out) CUDA_TRY(cudaMemcpyAsync(tangent_flag_out + lo, eng->d_tangent + lo, w, cudaMemcpyDeviceToHost, s));
  }
  for (auto& s : eng->pipe) CUDA_TRY(cudaStreamSynchronize(s));
  eng->caller_work_pending = false;
  eng->t_global += 1;
  return CAV_OK;
}

int cavgym_step_host_f32(CavEngine* eng, const float* actions, float* state_out, float* reward_out, uint8_t* done_out,
                         int32_t* winner_out, uint8_t* tangent_flag_out) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (eng->dtype != CAV_F64) return fail(CAV_ESTATE, "the float32 wire format is for fp64 engines; a float32 engine uses cavgym_step_host");
  if (eng->dense) return fail(CAV_ESTATE, "the float32 wire format is implemented by the thread-per-environment kernels (at most CAV_SMALL_M bodies)");
  if (eng->agent_params_set())
    return fail(CAV_ESTATE, "the float32 wire format does not read per-env agent parameters: clear them (cavgym_set_agent_params) first");
  if (!actions && eng->has_external) return fail(CAV_EINVAL, "actions is NULL but a body has CAV_AGENT_EXTERNAL");
  if ((rc = host_setup(eng))) return rc;
  if (eng->caller_work_pending) CUDA_TRY(cudaDeviceSynchronize());
  const void* host[6] = {actions, state_out, reward_out, done_out, winner_out, tangent_flag_out};
  void* dev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  for (int i = 0; i < 6; ++i) {
    if (!host[i]) continue;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, host[i]) != cudaSuccess || attr.type != cudaMemoryTypeHost || !attr.devicePointer) {
      cudaGetLastError();
      return fail(CAV_ESTATE, "cavgym_step_host_f32 needs page-locked, device-mapped buffers (cavgym_host_alloc / pin_memory)");
    }
    dev[i] = attr.devicePointer;
  }
  const WireIO32 wire{(const float*)dev[0], (float*)dev[1], (float*)dev[2], (uint8_t*)dev[3], (int32_t*)dev[4], (uint8_t*)dev[5]};
  cudaStream_t s = eng->pipe[0];
  if (!small_launchers<double>(eng->m)->step_wire32(eng->sc64, eng->buf64, wire, eng->t_global, eng->has_device_agents, s))
    return fail(CAV_ESTATE, "float32 wire kernels are not compiled for this engine type");
  rc = launch_check(eng, "step kernel (float32 wire)");
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize(s));
  eng->caller_work_pending = false;
  eng->t_global += 1;
  return CAV_OK;
}

// CAVEnv.reset with HOST buffers (the host-buffer twin of cavgym_reset, for callers that hold no device memory):
// mask u8[N] and init_state real[M][4][N] are copied in (each nullable), the post-reset state is copied out (nullable).
int cavgym_reset_host(CavEngine* eng, const uint8_t* mask, const void* init_state, void* state_out) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if ((rc = host_setup(eng))) return rc;
  if (eng->caller_work_pending) CUDA_TRY(cudaDeviceSynchronize());
  const size_t state_bytes = (size_t)eng->m * 4 * eng->n * eng->real_size();
  cudaStream_t s = eng->pipe[0];
  if (mask) CUDA_TRY(cudaMemcpyAsync(eng->d_mask, mask, (size_t)eng->n, cudaMemcpyHostToDevice, s));
  if (init_state) CUDA_TRY(cudaMemcpyAsync(eng->d_init, init_state, state_bytes, cudaMemcpyHostToDevice, s));
  rc = do_reset(eng, mask ? eng->d_mask : nullptr, init_state ? eng->d_init : nullptr, 0, s);
  if (rc) return rc;
  if (state_out) {
    const void* d_state = eng->dtype == CAV_F64 ? (const void*)eng->buf64.state : (const void*)eng->buf32.state;
    CUDA_TRY(cudaMemcpyAsync(state_out, d_state, state_bytes, cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  eng->caller_work_pending = false;
  return CAV_OK;
}

int cavgym_info(CavEngine* eng, void* polygons_out, void* road_angle_out, cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!polygons_out && !road_angle_out) return CAV_OK;
  const unsigned grid = (unsigned)((eng->n + 127) / 128);
  if (eng->dtype == CAV_F64)
    info_kernel<double><<<grid, 128, 0, stream>>>(eng->sc64, eng->tb64, eng->buf64, (const Quad<double>*)eng->d_static_quads,
                                                  (double*)polygons_out, (double*)road_angle_out);
  else
    info_kernel<float><<<grid, 128, 0, stream>>>(eng->sc32, eng->tb32, eng->buf32, (const Quad<float>*)eng->d_static_quads,
                                                 (float*)polygons_out, (float*)road_angle_out);
  return launch_check(eng, "info kernel");
}

int cavgym_snapshot_layout(CavEngine* eng, int64_t k, CavSnapshotLayout* out) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!out || k < 0) return fail(CAV_EINVAL, "out is NULL or k < 0");
  snapshot_layout(eng, k, out);
  return CAV_OK;
}

// The kernels read and write a snapshot in 8-byte (fp64 reals) and, for all envs in order, 16-byte words.
static int check_snapshot(const void* snapshot) {
  if (!snapshot) return fail(CAV_EINVAL, "snapshot is NULL");
  if (reinterpret_cast<uintptr_t>(snapshot) & 15u) return fail(CAV_EINVAL, "snapshot is not 16-byte aligned");
  return CAV_OK;
}

int cavgym_save_envs(CavEngine* eng, const int64_t* envs, int64_t k, void* snapshot, cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (k < 0) return fail(CAV_EINVAL, "k < 0");
  if (k == 0) return CAV_OK;   // an empty selection (whose device pointer may well be NULL) moves nothing
  if (!envs && k != eng->n) return fail(CAV_EINVAL, "envs is NULL and k is not the engine's env count");
  if ((rc = check_snapshot(snapshot))) return rc;
  return move_envs(eng, envs, k, snapshot, true, stream);
}

int cavgym_load_envs(CavEngine* eng, const int64_t* envs, int64_t k, const void* snapshot, cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (k < 0) return fail(CAV_EINVAL, "k < 0");
  if (k == 0) return CAV_OK;
  if (!envs && k != eng->n) return fail(CAV_EINVAL, "envs is NULL and k is not the engine's env count");
  if (k > eng->n) return fail(CAV_EINVAL, "more target envs than the engine holds: targets must be unique");
  if ((rc = check_snapshot(snapshot))) return rc;
  return move_envs(eng, envs, k, const_cast<void*>(snapshot), false, stream);
}

int cavgym_fork_envs(CavEngine* eng, const int64_t* src, const int64_t* dst, int64_t k, cudaStream_t stream) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (k < 0) return fail(CAV_EINVAL, "k < 0");
  if (k == 0) return CAV_OK;
  if (!src || !dst) return fail(CAV_EINVAL, "src/dst is NULL");
  if (k > eng->n) return fail(CAV_EINVAL, "more target envs than the engine holds: targets must be unique");
  CavSnapshotLayout L;
  snapshot_layout(eng, k, &L);
  if ((size_t)L.total_bytes > eng->stage_bytes) {
    CUDA_TRY(cudaDeviceSynchronize());   // an earlier fork may still be reading the old staging buffer
    if (eng->d_stage) CUDA_TRY(cudaFree(eng->d_stage));
    eng->d_stage = nullptr;
    eng->stage_bytes = 0;
    CUDA_TRY(cudaMalloc(&eng->d_stage, (size_t)L.total_bytes));
    eng->stage_bytes = (size_t)L.total_bytes;
  }
  // every read (the gather into the staging snapshot) precedes every write: src may overlap dst and repeat
  if ((rc = move_envs(eng, src, k, eng->d_stage, true, stream))) return rc;
  return move_envs(eng, dst, k, eng->d_stage, false, stream);
}

int cavgym_save_engine(CavEngine* eng, CavEngineState* out) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!out) return fail(CAV_EINVAL, "out is NULL");
  std::memset(out, 0, sizeof(*out));
  out->version = CAV_SNAPSHOT_VERSION;
  out->dtype = eng->dtype;
  out->m = eng->m;
  out->n = eng->n;
  out->shard = eng->buf64.shard;
  out->t_global = eng->t_global;
  out->seed = eng->seed;
  out->fingerprint = eng->fingerprint;
  out->tau = eng->tau;
  CUDA_TRY(cudaDeviceSynchronize());
  const unsigned long long* stats = eng->dtype == CAV_F64 ? eng->buf64.stats : eng->buf32.stats;
  CUDA_TRY(cudaMemcpy(out->counters, stats, sizeof(out->counters), cudaMemcpyDeviceToHost));
  return CAV_OK;
}

int cavgym_load_engine(CavEngine* eng, const CavEngineState* in) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!in) return fail(CAV_EINVAL, "in is NULL");
  if (in->version != CAV_SNAPSHOT_VERSION) return fail(CAV_EINVAL, "engine state of another version");
  if (in->fingerprint != eng->fingerprint) return fail(CAV_EINVAL, "engine state of another scenario (fingerprint)");
  if (in->dtype != eng->dtype || in->m != eng->m || in->n != eng->n)
    return fail(CAV_EINVAL, "engine state of another dtype, body count or env count");
  if (in->seed != eng->seed || in->shard != eng->buf64.shard) return fail(CAV_EINVAL, "engine state of another seed or shard");
  if (!(in->tau >= 0)) return fail(CAV_EINVAL, "tau must be >= 0");
  CUDA_TRY(cudaDeviceSynchronize());   // the counters and (for another tau) the tables are rewritten under no running kernel
  const unsigned long long* stats = eng->dtype == CAV_F64 ? eng->buf64.stats : eng->buf32.stats;
  CUDA_TRY(cudaMemcpy((void*)stats, in->counters, sizeof(in->counters), cudaMemcpyHostToDevice));
  eng->t_global = in->t_global;
  if (in->tau != eng->tau) {
    eng->tau = in->tau;
    return rebuild_tables(eng);
  }
  return CAV_OK;
}

int cavgym_stats(CavEngine* eng, int64_t* out10 /* [CAV_N_STATS] */) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!out10) return fail(CAV_EINVAL, "out10 is NULL");
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemset(eng->d_scratch, 0, 2 * sizeof(unsigned long long)));
  const int32_t* t_ep = eng->dtype == CAV_F64 ? eng->buf64.t_ep : eng->buf32.t_ep;
  const uint8_t* done = eng->dtype == CAV_F64 ? eng->buf64.done : eng->buf32.done;
  const uint8_t* err = eng->dtype == CAV_F64 ? eng->buf64.err : eng->buf32.err;
  const unsigned long long* stats = eng->dtype == CAV_F64 ? eng->buf64.stats : eng->buf32.stats;
  live_steps_kernel<<<148 * 4, 256>>>(t_ep, done, err, eng->n, eng->d_scratch);
  rc = launch_check(eng, "stats kernel");
  if (rc) return rc;
  unsigned long long raw[CAV_N_STATS], extra[2];
  CUDA_TRY(cudaMemcpy(raw, stats, sizeof(raw), cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(extra, eng->d_scratch, sizeof(extra), cudaMemcpyDeviceToHost));
  for (int i = 0; i < CAV_N_STATS; ++i) out10[i] = (int64_t)raw[i];
  // finished episodes + episodes abandoned by a reset + episodes in flight
  out10[CAV_STAT_ENV_STEPS] = (int64_t)(raw[CAV_STAT_SUM_T] + raw[CAV_STAT_ENV_STEPS] + extra[0]);
  out10[CAV_STAT_BODY_STEPS] = out10[CAV_STAT_ENV_STEPS] * eng->m;
  out10[CAV_STAT_ERRORS] = (int64_t)extra[1];
  return CAV_OK;
}

int cavgym_set_episode_log(CavEngine* eng, int64_t capacity) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (capacity < 0) return fail(CAV_EINVAL, "capacity must be >= 0");
  CUDA_TRY(cudaDeviceSynchronize());   // kernels in flight carry the old ring in their parameters
  CavEpisodeRow* rows = nullptr;
  unsigned long long* count = eng->dtype == CAV_F64 ? eng->buf64.ep_log_count : eng->buf32.ep_log_count;
  if (capacity > 0) {
    if ((rc = dev_alloc(eng, &rows, (size_t)capacity, false))) return rc;
    if (!count && (rc = dev_alloc(eng, &count, 1))) return rc;
    CUDA_TRY(cudaMemset(count, 0, sizeof(*count)));
  }
  for (int k = 0; k < 2; ++k) {   // both typed views of the buffers carry the ring
    CavEpisodeRow*& r = k ? eng->buf32.ep_log : eng->buf64.ep_log;
    (k ? eng->buf32.ep_log_count : eng->buf64.ep_log_count) = count;
    (k ? eng->buf32.ep_log_capacity : eng->buf64.ep_log_capacity) = capacity;
    r = rows;
  }
  return CAV_OK;
}

int cavgym_drain_episodes(CavEngine* eng, CavEpisodeRow* out, int64_t max_rows, int64_t* n_rows, int64_t* dropped) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!n_rows || max_rows < 0 || (max_rows > 0 && !out)) return fail(CAV_EINVAL, "bad argument");
  *n_rows = 0;
  if (dropped) *dropped = 0;
  const CavEpisodeRow* rows = eng->dtype == CAV_F64 ? eng->buf64.ep_log : eng->buf32.ep_log;
  unsigned long long* count = eng->dtype == CAV_F64 ? eng->buf64.ep_log_count : eng->buf32.ep_log_count;
  const int64_t capacity = eng->dtype == CAV_F64 ? eng->buf64.ep_log_capacity : eng->buf32.ep_log_capacity;
  if (!rows) return fail(CAV_ESTATE, "the episode log is off (cavgym_set_episode_log)");
  CUDA_TRY(cudaDeviceSynchronize());
  unsigned long long appended = 0;
  CUDA_TRY(cudaMemcpy(&appended, count, sizeof(appended), cudaMemcpyDeviceToHost));
  const int64_t held = (int64_t)appended < capacity ? (int64_t)appended : capacity;
  const int64_t take = held < max_rows ? held : max_rows;
  if (take > 0) CUDA_TRY(cudaMemcpy(out, rows, (size_t)take * sizeof(CavEpisodeRow), cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemset(count, 0, sizeof(*count)));
  *n_rows = take;
  if (dropped) *dropped = (int64_t)appended - take;
  return CAV_OK;
}

int cavgym_error_count(CavEngine* eng, int64_t* out) {
  int64_t stats[CAV_N_STATS];
  int rc = cavgym_stats(eng, stats);
  if (rc) return rc;
  if (!out) return fail(CAV_EINVAL, "out is NULL");
  *out = stats[CAV_STAT_ERRORS];
  return CAV_OK;
}

int cavgym_launch_count(CavEngine* eng, int64_t* out) {
  if (!eng || !out) return fail(CAV_EINVAL, "engine/out is NULL");
  *out = eng->launches;
  return CAV_OK;
}

#define CAV_PTR(field) (eng ? (eng->dtype == CAV_F64 ? (void*)eng->buf64.field : (void*)eng->buf32.field) : nullptr)
void* cavgym_state_ptr(CavEngine* eng) { return CAV_PTR(state); }
int32_t* cavgym_liveness_ptr(CavEngine* eng) { return (int32_t*)CAV_PTR(liveness); }
void* cavgym_agent_state_ptr(CavEngine* eng) { return CAV_PTR(agent); }
void* cavgym_action_ptr(CavEngine* eng) { return CAV_PTR(action); }
int32_t* cavgym_timestep_ptr(CavEngine* eng) { return (int32_t*)CAV_PTR(t_ep); }
uint8_t* cavgym_done_ptr(CavEngine* eng) { return (uint8_t*)CAV_PTR(done); }
int32_t* cavgym_winner_ptr(CavEngine* eng) { return (int32_t*)CAV_PTR(winner); }
uint8_t* cavgym_error_ptr(CavEngine* eng) { return (uint8_t*)CAV_PTR(err); }
#undef CAV_PTR

int cavgym_set_uniform_override(CavEngine* eng, const double* uniforms) {
  if (!eng) return fail(CAV_EINVAL, "engine is NULL");
  eng->buf64.uni_override = uniforms; eng->buf32.uni_override = uniforms;
  return CAV_OK;
}

int cavgym_set_spawn_override(CavEngine* eng, const double* draws) {
  if (!eng) return fail(CAV_EINVAL, "engine is NULL");
  eng->buf64.spawn_override = draws; eng->buf32.spawn_override = draws;
  return CAV_OK;
}

int cavgym_set_action_logging(CavEngine* eng, int enabled) {
  if (!eng) return fail(CAV_EINVAL, "engine is NULL");
  eng->buf64.log_actions = enabled; eng->buf32.log_actions = enabled;
  return CAV_OK;
}

int cavgym_set_step_path(CavEngine* eng, int use_tma) {
  if (!eng) return fail(CAV_EINVAL, "engine is NULL");
  eng->use_tma = use_tma != 0;
  return CAV_OK;
}

int cavgym_set_dense_path(CavEngine* eng, int force) {
  if (!eng) return fail(CAV_EINVAL, "engine is NULL");
  if (eng->m > CAV_SMALL_M && !force) return fail(CAV_EINVAL, "more than CAV_SMALL_M bodies: only the warp-per-environment kernels apply");
  if (force && eng->sc64.has_election) return fail(CAV_EINVAL, "election agents run in the thread-per-environment kernels only");
  eng->dense = force != 0 || eng->m > CAV_SMALL_M;
  return CAV_OK;
}

int cavgym_set_host_path(CavEngine* eng, int zero_copy) {
  if (!eng) return fail(CAV_EINVAL, "engine is NULL");
  eng->zero_copy_host = zero_copy != 0;
  // tuning: 1 = zero copy with the default CTA count, 2..8 = zero copy with (value - 1) CTAs per SM
  if (zero_copy >= 1 && zero_copy <= 8) eng->host_ctas_per_sm = zero_copy == 1 ? CAV_HOST_CTAS_PER_SM : zero_copy - 1;
  return CAV_OK;
}

int cavgym_set_global_timestep(CavEngine* eng, int64_t t) {
  if (!eng) return fail(CAV_EINVAL, "engine is NULL");
  eng->t_global = t;
  return CAV_OK;
}

int cavgym_set_tangent_tolerance(CavEngine* eng, double tau) {
  int rc = check_engine(eng);
  if (rc) return rc;
  if (!(tau >= 0)) return fail(CAV_EINVAL, "tau must be >= 0");
  CUDA_TRY(cudaDeviceSynchronize());   // the device tables are rewritten: no kernel of this engine may still be reading them
  eng->tau = tau;
  return rebuild_tables(eng);
}

int cavgym_bodies_step(const CavBodyType* type, void* state, const void* actions, int64_t n, double time_resolution, int dtype,
                       cudaStream_t stream) {
  if (!type || !state || !actions || n < 0) return fail(CAV_EINVAL, "bad argument");
  if (n == 0) return CAV_OK;
  const unsigned grid = (unsigned)((n + 127) / 128);
  if (dtype == CAV_F64) bodies_step_kernel<double><<<grid, 128, 0, stream>>>(to_type<double>(*type), (double*)state, (const double*)actions, n, time_resolution);
  else if (dtype == CAV_F32) bodies_step_kernel<float><<<grid, 128, 0, stream>>>(to_type<float>(*type), (float*)state, (const float*)actions, n, (float)time_resolution);
  else return fail(CAV_EINVAL, "dtype must be CAV_F64 or CAV_F32");
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(CAV_ECUDA, std::string("bodies_step kernel: ") + cudaGetErrorString(err));
  return CAV_OK;
}

int cavgym_zones_probe(const CavBodyType* type, const void* state, const void* steering, void* zones_out, uint8_t* have_out,
                       int64_t n, int dtype, cudaStream_t stream) {
  if (!type || !state || !steering || !zones_out || !have_out || n < 0) return fail(CAV_EINVAL, "bad argument");
  if (n == 0) return CAV_OK;
  const unsigned grid = (unsigned)((n + 127) / 128);
  if (dtype == CAV_F64) zones_probe_kernel<double><<<grid, 128, 0, stream>>>(to_type<double>(*type), (const double*)state, (const double*)steering, (double*)zones_out, have_out, n);
  else if (dtype == CAV_F32) zones_probe_kernel<float><<<grid, 128, 0, stream>>>(to_type<float>(*type), (const float*)state, (const float*)steering, (float*)zones_out, have_out, n);
  else return fail(CAV_EINVAL, "dtype must be CAV_F64 or CAV_F32");
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(CAV_ECUDA, std::string("zones_probe kernel: ") + cudaGetErrorString(err));
  return CAV_OK;
}

int cavgym_geometry_probe(const void* quads_a, const void* quads_b, void* out, int64_t n, int dtype, cudaStream_t stream) {
  if (!quads_a || !quads_b || !out || n < 0) return fail(CAV_EINVAL, "bad argument");
  if (n == 0) return CAV_OK;
  const unsigned grid = (unsigned)((n + 127) / 128);
  if (dtype == CAV_F64) geometry_probe_kernel<double><<<grid, 128, 0, stream>>>((const double*)quads_a, (const double*)quads_b, (double*)out, n, 1e-7);
  else if (dtype == CAV_F32) geometry_probe_kernel<float><<<grid, 128, 0, stream>>>((const float*)quads_a, (const float*)quads_b, (float*)out, n, 5e-2f);
  else return fail(CAV_EINVAL, "dtype must be CAV_F64 or CAV_F32");
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(CAV_ECUDA, std::string("geometry_probe kernel: ") + cudaGetErrorString(err));
  return CAV_OK;
}

}  // extern "C"
