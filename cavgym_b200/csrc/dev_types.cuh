// dev_types.cuh — device-side tables and per-environment register state.
//
// The scenario (include/cavgym.h CavScenario) is converted once on the host into
// DevScenario<R> in the engine's arithmetic type R and passed to every kernel BY VALUE
// as a __grid_constant__ parameter: all threads read it through the constant bank
// (uniform loads), no global traffic.
//
// Rectangles (body boxes, roads, traffic lights, the obstacle, stopping zones) are kept in
// CENTRE-EXTENT form — centre, unit heading (c, s), half length, half width — because every
// test of the step (separating axes, road share, finish line) is a handful of dot products in
// that form; corner lists (Quad) exist only for the general-polygon fallbacks.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/cavgym.h"

namespace cav {

template <typename R>
struct Quad {
  R x[4], y[4];  // rear_left, front_left, front_right, rear_right — clockwise (y up)
};

template <typename R>
struct Box {  // make_rectangle(2*hl, 2*hw).transform(theta, (px, py)) with c, s = cos/sin(theta)  (geometry.py:241-251)
  R px, py, c, s, hl, hw;
};

#define CAV_HEADING_CACHE 4

template <typename R>
struct DevType {
  R length, width, wheelbase, vmin, vmax, amin, amax, smin, smax;
  R hl, hw;            // half length / half width
  R half_wb;           // wheelbase / 2 (bodies.py:246: rear axle offset)
  R inv_2brake;        // 1 / (2 * -min_throttle): braking distance = v*v * inv_2brake (bodies.py:123)
  // Full-lock turns (what a crossing agent commands for all but the last step of a turn): wheelbase / tan(limit)
  // and 1 / turn radius of the body centre, host libm values.
  double kk_smin, kk_smax, inv_r_smin, inv_r_smax;  // double in both modes (see body_step)
  // Largest heading change per unit of travelled distance at full lock, 2 / sqrt(wb^2 (1 + 4 / tan^2(limit))), host libm
  // values in the reference's operation order (dynamic_body.py:40-41): make_steering_action only ever asks for the two limits.
  R max_turn_smin, max_turn_smax;
};

template <typename R>
struct Aabb {
  R x0, x1, y0, y1;
};

template <typename R>
struct DevBody {
  int32_t kind, type_id, flags, agent, spawn_id, pad;
  double epsilon;  // compared against a 53-bit draw in double in both modes
  R threshold;
  R init[4];       // init_state (bodies.py:27); PelicanCrossing: light state in [0]
  DevType<R> k;    // this body's DynamicBodyConstants row, resolved on the host
  R static_share;  // PelicanCrossing: max over roads of percentage_intersects(static box, road) — a scenario constant
};

template <typename R>
struct DevSpawn {
  int32_t n_boxes, n_orient;
  Quad<R> boxes[CAV_MAX_SPAWN_BOXES];
  R orient[CAV_MAX_SPAWN_ORIENT];
  R velocity;
  R init[4];  // unused padding for alignment / future use
};

template <typename R>
struct DevScenario {
  int32_t n_bodies, n_types, n_roads, n_statics, n_spawns;
  int32_t collisions, zones, offroad;
  int32_t homogeneous;  // no PelicanCrossing body, bodies 1.. all Pedestrians, roads axis-aligned: GENERIC = false kernels
  int64_t max_timesteps;
  R reward_win, reward_draw, cost_step, W, dt, v_maint, v_off;
  R inv_W, inv_v_off;  // reciprocals of the two constant divisors on the always-executed path
  R tau;         // near-tangent tolerance (px)
  R target_err;  // TARGET_ERROR (dynamic_body.py:8); widened for float
  R cl[4];       // centre line start x,y end x,y
  // Headings bodies are created with (spawn orientations, init orientations): cos/sin evaluated ON THE HOST
  // with the C library the reference's math.cos/math.sin use.
  int32_t hc_n, has_election;   // has_election: some body is driven by CAV_AGENT_ELECTION (Election.result runs every step)
  R hc_theta[CAV_HEADING_CACHE], hc_cos[CAV_HEADING_CACHE], hc_sin[CAV_HEADING_CACHE];
  Aabb<R> road_bb[CAV_MAX_ROADS];
  Box<R> road_box[CAV_MAX_ROADS];
  int32_t road_axis[CAV_MAX_ROADS];   // 1 if the road rectangle is exactly axis-aligned (road == its AABB)
  int32_t road_rect[CAV_MAX_ROADS];   // 1 if the road quad is a rectangle (road_box valid)
  Aabb<R> static_bb[CAV_MAX_STATICS];
  Box<R> static_box[CAV_MAX_STATICS];
  int32_t static_rect[CAV_MAX_STATICS];
  const Quad<R>* quads;  // device: roads[CAV_MAX_ROADS] then statics[CAV_MAX_STATICS] as corner lists (general fallbacks)
  DevBody<R> bodies[CAV_SMALL_M];
};

// Per-env buffers owned by the engine (SoA, env fastest) + optional per-call I/O.
template <typename R>
struct EnvBuffers {
  int64_t n;            // envs in this engine (= stride of every per-env array)
  int64_t lo, hi;       // env range this launch covers (chunked host pipeline); normally [0, n)
  int64_t shard;        // global id of env 0
  uint64_t seed;
  R* state;             // [M][4][N]
  R* action;            // [M][2][N] last joint action (RandomAgent's held action)
  R* agent;             // [M][5][N] crossing-agent state, NaN = None
  R* cs;                // [M][2][N] cos/sin of each body's heading; refreshed only when the heading changes
  int32_t* liveness;    // [M][N]
  int32_t* t_ep;        // [N]
  int32_t* episode;     // [N]
  int32_t* winner;      // [N]
  int32_t* active;      // [N] Election.active_player (election.py:12), 0 = None; survives resets like the reference's object
  uint8_t* done;        // [N] 0 live, 1 done, 2 cut off at max_timesteps
  uint8_t* err;         // [N]
  unsigned long long* stats;  // [CAV_N_STATS]
  const DevSpawn<R>* spawns;
  const double* uni_override;    // [M][3][N] or null
  const double* spawn_override;  // [M][5][N] or null
  int32_t log_actions;           // store every on-device agent's action in `action` (default: RandomAgent only)
  // per-episode rows (reporting.py:157-158 episode.log), appended by score_episode when enabled (cavgym_set_episode_log)
  CavEpisodeRow* ep_log;              // [ep_log_capacity] or null
  unsigned long long* ep_log_count;   // rows appended since the last drain (may exceed the capacity: the excess was dropped)
  int64_t ep_log_capacity;
};

template <typename R>
struct StepIO {
  const R* actions;  // [M][2][N] or null
  R* state_out;      // nullable; == state means in place
  R* reward_out;
  uint8_t* done_out;
  int32_t* winner_out;
  uint8_t* tangent_out;
  int32_t ctas_per_sm;   // host side only: cap on resident CTAs per SM of the persistent step kernel (0 = as many as fit)
  // replay_tma_kernel, launch chaining (kernels_tma.cuh): tile_gen[i] = sequence number of the last replay launch that has
  // written tile i's env state back; a launch with `chained` set waits for its own tiles' seq - 1 instead of for the whole
  // previous grid.  Engine-owned; null = no chaining.
  int32_t* tile_gen;
  int32_t seq, chained;
};

// cavgym_rollout_record: the per-step [T] slabs of a recorded rollout (CavRolloutRecord), each nullable; row t of a slab
// has the per-step shape with the env index fastest.  Only the recording kernels take it, so StepIO, EnvBuffers and
// DevScenario — parameters of every kernel — keep their layout.
template <typename R>
struct RolloutRecord {
  R* observation;      // [T][M][4][N] state the agents saw at step t (after the auto-reset)
  R* action;           // [T][M][2][N] joint action executed at step t
  R* state;            // [T][M][4][N] state after step t
  R* reward;           // [T][M][N]
  uint8_t* done;       // [T][N]
  int32_t* winner;     // [T][N]
  uint8_t* tangent;    // [T][N]
  int32_t* timestep;   // [T][N] t_ep after step t, 0 where the env did not step
};

// cavgym_set_agent_params: per-env tester parameters, [M][N] with the env index fastest, each nullable (null = the scenario's
// DevBody value).  Given by value to the parameter kernels only (kernels_params.cuh), for the reason RolloutRecord is.
template <typename R>
struct AgentParams {
  const double* epsilon;   // RandomAgent / RandomConstrainedAgent epsilon, double in both modes as DevBody::epsilon
  const R* threshold;      // ProximityAgent / ElectionAgent distance threshold
};

// cavgym_step_host_f32: joint actions and results cross the host link as float32 while the engine steps in its own type.
struct WireIO32 {
  const float* actions;  // [M][2][N]
  float* state_out;      // [M][4][N], nullable
  float* reward_out;     // [M][N], nullable
  uint8_t* done_out;
  int32_t* winner_out;
  uint8_t* tangent_out;
};

}  // namespace cav
