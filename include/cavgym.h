/* cavgym.h — C-ABI of libcavgym_sm100.so, the B200 batched stepping engine for CAV-Gym.
 *
 * The reference (TSL-UOB/CAV-Gym) has no FFI: its boundary is the Python protocol
 *   CAVEnv(bodies, constants, env_config, np_random)        library/environment.py:59
 *   CAVEnv.reset() -> joint_obs                              library/environment.py:225-229
 *   CAVEnv.step(joint_action) -> (obs, reward, done, info)   library/environment.py:119-223
 * Every entry point below names the reference interface it replaces.  Plain
 * pointers and sizes only; no torch types.  Device buffers are raw device
 * pointers (torch.Tensor.data_ptr()); the caller owns every I/O buffer, the
 * engine owns its tables, body state, agent state, RNG counters and liveness.
 *
 * Layout (all per-env arrays are SoA with the environment index fastest):
 *   state    [M][4][N]  x, y, velocity, orientation          (bodies.py:48-60)
 *   actions  [M][2][N]  throttle, steering_angle             (bodies.py:104-109)
 *                       PelicanCrossing body: TrafficLightAction value in [.][0]
 *   reward   [M][N]     joint reward                          (environment.py:131-146,208-213)
 *   done     [N] u8, winner [N] i32 (-1 = no 'winner' key)    (environment.py:148-220)
 *   liveness [M][N] i32 episode_liveness                      (environment.py:144-146)
 * real = double (dtype 0) or float (dtype 1).
 *
 * Errors: every call returns 0 or a negative CAV_E* code and never throws;
 * cavgym_last_error() gives the message of the calling thread's last failure.
 * One engine per device; an engine is not thread-safe.  No call synchronises the
 * host with the device except cavgym_stats, cavgym_error_count, cavgym_set_agent_params
 * and the *_host calls.
 */
#ifndef CAVGYM_H
#define CAVGYM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __DRIVER_TYPES_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define CAV_MAX_ROADS 4         /* road_map.roads: major + minor roads (assets.py:115-120) */
#define CAV_MAX_STATICS 8       /* traffic lights + obstacle (environment.py:94-101) */
#define CAV_MAX_SPAWN_BOXES 2   /* pedestrians.py:45-68 */
#define CAV_MAX_SPAWN_ORIENT 4
#define CAV_MAX_TYPES 8
#define CAV_SMALL_M 8           /* thread-per-env fused kernels up to this many bodies */
#define CAV_MAX_BODIES 512      /* warp-per-env dense kernels (bodies staged in shared memory) up to this many bodies */
#define CAV_AGENT_WORDS 5       /* CrossingAgent state (pedestrian.py:14-31); NaN = None */
#define CAV_DRAWS 3             /* [0,1) draws an agent may consume per step */

enum { CAV_F64 = 0, CAV_F32 = 1 };

enum {                          /* negative return codes */
  CAV_OK = 0,
  CAV_EINVAL = -22,             /* bad argument / unsupported scenario */
  CAV_ENOMEM = -12,
  CAV_ECUDA = -5,               /* a CUDA runtime call failed */
  CAV_ESTATE = -1               /* call not valid in the engine's current state */
};

enum { CAV_BODY_DYNAMIC = 0,    /* DynamicBody and subclasses (bodies.py:78-346) */
       CAV_BODY_PELICAN = 1 };  /* PelicanCrossing (bodies.py:409-461) */

enum { CAV_FLAG_PEDESTRIAN = 1, /* isinstance(body, Pedestrian) (environment.py:192,199) */
       CAV_FLAG_SPAWN = 2 };    /* SpawnPedestrian: re-drawn on reset (bodies.py:290-312) */

enum { CAV_AGENT_EXTERNAL = 0,            /* action comes from the `actions` buffer */
       CAV_AGENT_NOOP = 1,                /* NoopAgent            (template.py:24-37) */
       CAV_AGENT_RANDOM = 2,              /* RandomAgent          (template.py:40-62) */
       CAV_AGENT_RANDOM_CONSTRAINED = 3,  /* RandomConstrainedAgent (pedestrian.py:72-75) */
       CAV_AGENT_PROXIMITY = 4,           /* ProximityAgent       (pedestrian.py:78-91) */
       CAV_AGENT_ELECTION = 5 };          /* ElectionAgent arbitrated by Election (pedestrian.py:94-116, election.py:4-57);
                                             scenarios of at most CAV_SMALL_M bodies */

enum { CAV_COLLISIONS_NONE = 0, CAV_COLLISIONS_EGO = 1, CAV_COLLISIONS_ALL = 2 }; /* config.py:237-240 */

/* Convex quadrilateral, corners in the reference's order rear_left, front_left,
 * front_right, rear_right (geometry.py:96-107). */
typedef struct CavQuad { double x[4]; double y[4]; } CavQuad;

/* DynamicBodyConstants (bodies.py:63-75); track is cosmetic and omitted. */
typedef struct CavBodyType {
  double length, width, wheelbase;
  double min_velocity, max_velocity;
  double min_throttle, max_throttle;
  double min_steering_angle, max_steering_angle;
} CavBodyType;

/* SpawnPedestrianState (bodies.py:283-287). */
typedef struct CavSpawn {
  int32_t n_boxes, n_orientations;
  CavQuad boxes[CAV_MAX_SPAWN_BOXES];
  double orientations[CAV_MAX_SPAWN_ORIENT];
  double velocity;
} CavSpawn;

typedef struct CavBody {
  int32_t kind;              /* CAV_BODY_* */
  int32_t type_id;           /* row of CavScenario.types (dynamic bodies) */
  int32_t flags;             /* CAV_FLAG_* */
  int32_t spawn_id;          /* row of CavScenario.spawns, or -1 */
  int32_t agent;             /* CAV_AGENT_* */
  int32_t reserved;
  double agent_epsilon;      /* RandomAgent / RandomConstrainedAgent epsilon */
  double agent_threshold;    /* ProximityAgent distance_threshold */
  double init_state[4];      /* x, y, v, theta; PelicanCrossing: TrafficLightState in [0] */
  CavQuad static_box;        /* PelicanCrossing.static_bounding_box (bodies.py:415) */
} CavBody;

/* Everything CAVEnv.__init__ receives, flattened (environment.py:59-92). */
typedef struct CavScenario {
  int32_t n_bodies, n_types, n_roads, n_statics, n_spawns;
  int32_t terminate_collisions;      /* CAV_COLLISIONS_* (config.json "terminate_collisions") */
  int32_t terminate_ego_zones;       /* bool */
  int32_t terminate_ego_offroad;     /* bool */
  int64_t max_timesteps;
  double reward_win, reward_draw, cost_step;
  double viewer_width;               /* CAVEnvConstants.viewer_width (environment.py:47-51) */
  double time_resolution;            /* 1/frequency = 1/60 (environment.py:65-66) */
  double ego_maintenance_velocity;   /* environment.py:87 */
  double ego_max_velocity_offset;    /* environment.py:88 */
  double centre_line[4];             /* major road longitudinal_line(): start x,y, end x,y (config.py:363) */
  CavQuad roads[CAV_MAX_ROADS];      /* roads[0] = major road */
  CavQuad statics[CAV_MAX_STATICS];  /* collidable traffic lights, then the obstacle */
  CavBodyType types[CAV_MAX_TYPES];
  const CavSpawn* spawns;            /* host pointer, n_spawns rows (copied by cavgym_create) */
  const CavBody* bodies;             /* host pointer, n_bodies rows (copied by cavgym_create) */
} CavScenario;

typedef struct CavEngine CavEngine;

/* One finished episode as reporting.analyse_episode scores it (reporting.py:227-243) — the fields of an episode.log
 * row (reporting.py:157-158) that exist for an environment of a batch.  interesting <=> winner > 0, score = -liveness_sum
 * when interesting (else NaN), completed <=> timesteps == max_timesteps. */
typedef struct CavEpisodeRow {
  int64_t env;           /* global env id (shard offset included) */
  int32_t episode;       /* the env's own episode count, 1 = its first episode */
  int32_t timesteps;
  int32_t winner;        /* info['winner'] of the last step, -1 when absent */
  int32_t liveness_sum;  /* sum(env.episode_liveness[1:]) */
} CavEpisodeRow;

/* Indices of cavgym_stats' twelve int64 counters (reporting.py:227-269 definitions).  SUM_T / SUM_T2 run over every
 * finished episode; SUM_T_INTERESTING / SUM_T2_INTERESTING only over episodes with winner > 0, which is what the reference's
 * run summary reports as the timesteps of its "interesting" tests (reporting.py:246-255). */
enum { CAV_STAT_EPISODES = 0, CAV_STAT_INTERESTING = 1, CAV_STAT_SUM_T = 2, CAV_STAT_SUM_T2 = 3,
       CAV_STAT_SUM_SCORE = 4, CAV_STAT_SUM_SCORE2 = 5, CAV_STAT_ENV_STEPS = 6, CAV_STAT_BODY_STEPS = 7,
       CAV_STAT_TANGENT = 8, CAV_STAT_ERRORS = 9, CAV_STAT_SUM_T_INTERESTING = 10, CAV_STAT_SUM_T2_INTERESTING = 11,
       CAV_N_STATS = 12 };

#define CAV_SNAPSHOT_VERSION 1

/* Layout of a snapshot of k envs (cavgym_save_envs): three sections, each starting on 256 bytes, of rows of k elements
 * (env j of row r at r * k + j).  Reals (dtype): state [M][4], action [M][2], agent [M][CAV_AGENT_WORDS], cs [M][2] (the
 * cos/sin heading cache); int32: liveness [M], t_ep, episode, winner, active; u8: done, err.  That is everything the
 * kernels read or write per env.  fingerprint: 64-bit FNV-1a over the scenario tables' contents (the CavScenario header up
 * to its pointers, then the spawn and body rows), so two engines of the same scenario agree wherever they were built. */
typedef struct CavSnapshotLayout {
  int32_t version, dtype, m, reserved;
  int64_t k;
  int64_t real_rows, i32_rows, u8_rows;
  int64_t real_offset, i32_offset, u8_offset;   /* bytes from the start of the snapshot */
  int64_t total_bytes;
  uint64_t fingerprint;
} CavSnapshotLayout;

/* Engine-wide state of a checkpoint (cavgym_save_engine): the raw device counters (before cavgym_stats adds the steps of
 * episodes in flight), the batch-wide step counter and what an engine must share with the saved one to continue it. */
typedef struct CavEngineState {
  int32_t version, dtype, m, reserved;
  int64_t n, shard, t_global;
  uint64_t seed, fingerprint;
  double tau;
  int64_t counters[CAV_N_STATS];
} CavEngineState;

/* ---- lifecycle ------------------------------------------------------------------- */

/* CAVEnv.__init__ x n_envs (environment.py:59-92; Config.setup config.py:272-415).
 * Copies the tables to `device`, allocates per-env storage and performs the
 * constructor-time spawn of every SpawnPedestrian (bodies.py:296).  `seed` keys
 * the Philox streams of the on-device agents and spawners. */
int cavgym_create(const CavScenario* tables, int64_t n_envs, int dtype, int device, uint64_t seed, CavEngine** out);
int cavgym_destroy(CavEngine* engine);

/* Env-sharding (experiments.py:121-122 analogue): this engine holds global env ids
 * [offset, offset + n_envs).  Philox is keyed by the GLOBAL id, so results do not
 * depend on how envs are split across GPUs.  Call before the first reset. */
int cavgym_set_shard(CavEngine* engine, int64_t global_env_offset);

/* CAVEnv.reset (environment.py:225-229; Body.reset bodies.py:32-33,111-114;
 * SpawnPedestrian.reset bodies.py:298-300; Agent.reset pedestrian.py:27-31).
 * mask  : device u8[N] or NULL (= all); envs with mask!=0 are reset.
 * init_state: device real[M][4][N] or NULL; when given it REPLACES the spawn draw
 *         (replay of reference-generated initial states). */
int cavgym_reset(CavEngine* engine, const uint8_t* mask, const void* init_state, cudaStream_t stream);

/* ---- stepping -------------------------------------------------------------------- */

/* CAVEnv.step (environment.py:119-223) over all N envs, one fused launch.
 * actions : device real[M][2][N]; may be NULL iff no body has CAV_AGENT_EXTERNAL
 *           (bodies with an on-device agent ignore their rows).
 * state_out, reward_out, done_out, winner_out, tangent_flag_out: device, each
 *           nullable.  state_out may be cavgym_state_ptr() (no extra write).
 * An env whose episode has ended stays frozen (reward 0, done 1) until it is reset.
 * Invalid actions (environment.py:120) set the env's error flag instead of aborting
 * the batch; see cavgym_error_count. */
int cavgym_step(CavEngine* engine, const void* actions, void* state_out, void* reward_out,
                uint8_t* done_out, int32_t* winner_out, uint8_t* tangent_flag_out, cudaStream_t stream);

/* Simulation.run's inner loop (simulation.py:70-97) on device: n_steps fused
 * transitions with the on-device agents; with auto_reset, an env whose episode ends
 * (done, or max_timesteps reached, simulation.py:69-70) is scored
 * (reporting.py:227-243) and reset in the same kernel. */
int cavgym_rollout(CavEngine* engine, int n_steps, int auto_reset, cudaStream_t stream);

/* The per-step returns of env.step inside Simulation.run's loop (simulation.py:38-118), for a cavgym_rollout: device slabs
 * [T] x the per-step shape, env index fastest (as cavgym_replay's), each nullable.  Row t holds
 *   observation real[T][M][4][N]  the state the agents saw when they chose step t's actions: AFTER any auto-reset at the top
 *                                 of step t (the reference's observation, environment.py:223-229)
 *   action      real[T][M][2][N]  the joint action executed at step t, for every agent kind (what
 *                                 cavgym_set_action_logging stores)
 *   state       real[T][M][4][N]  the state after step t
 *   reward      real[T][M][N], done u8[T][N], winner i32[T][N], tangent u8[T][N]   as cavgym_replay's
 *   timestep    i32[T][N]         the env's t_ep after step t: 1 on the first step of an episode
 * A row where the env does not step (finished, auto_reset = 0) is a frozen row, as in cavgym_replay: state and observation
 * unchanged, reward 0, done / winner latched, tangent 0, action 0, timestep 0.  So an episode starts at a row with
 * timestep == 1; it ends at a row with done == 1 and timestep > 0, or — cut off at max_timesteps (done stays 0) — at a row
 * with timestep == max_timesteps. */
typedef struct CavRolloutRecord {
  void* observation;
  void* action;
  void* state;
  void* reward;
  uint8_t* done;
  int32_t* winner;
  uint8_t* tangent;
  int32_t* timestep;
} CavRolloutRecord;

/* cavgym_rollout that also writes `rec` (HOST struct of device pointers; NULL or all-NULL = cavgym_rollout).  The launches,
 * engine state, counters, episode-log rows and t_global afterwards are exactly those of cavgym_rollout. */
int cavgym_rollout_record(CavEngine* engine, int n_steps, int auto_reset, const CavRolloutRecord* rec, cudaStream_t stream);

/* One stage of a multilevel splitting estimate of the rate of "interesting" episodes, those a tester wins (winner > 0,
 * reporting.py:227-243): Simulation.run's loop (simulation.py:38-118) as cavgym_rollout with auto_reset = 0, that also
 * carries a caller-owned score per env and PARKS an env at the first step where its score reaches `level`.
 *   danger of a post-step state: -min over the Pedestrian bodies of the separating-axis margin of the body's box against
 *     the ego's reaction-zone rectangle (environment.py:195-206), in px, positive on overlap; the rectangle is taken whether
 *     or not the zones exist (the ego steering, or standing still).
 *   at entry: an env with done != 0 is not stepped: parked with score = +inf if its latched winner is > 0, finished
 *     otherwise.  A live env with score >= level is parked without a step (so a repeated launch changes nothing, and a
 *     launch at a higher level resumes it).
 *   per step: a step that ends the episode with winner > 0 sets score = +inf (parked); one that ends it otherwise (done, or
 *     cut off at max_timesteps) finishes the env and leaves its score; any other step sets score = max(score, danger) and
 *     parks the env once score >= level.  A parked env keeps the state of that step, as a finished env is frozen.
 * score   device real[N], read and written.  status  device u8[N]: 0 = live below the level after n_steps, 1 = parked
 *         (tester wins included), 2 = finished without reaching the level.
 * Every step taken is scored, logged and counted as cavgym_rollout's; t_global advances by n_steps.
 * salt = 0 draws the engine's Philox streams bit for bit; any other salt keys this launch's draws with
 * seed ^ splitmix64(salt) instead (the engine's seed, cavgym_save_engine included, is unchanged): the fresh randomness a
 * copy made by cavgym_fork_envs needs, since its slot's own stream at the same (episode, t) drew the trajectory that was
 * just discarded.  An ordinary launch on `stream`.  n_steps = 0 does nothing.
 * CAV_EINVAL: NULL engine, score or status, n_steps < 0, NaN level, a scenario no tester can win (terminate_ego_zones off
 * or no Pedestrian body).  CAV_ESTATE: a body with CAV_AGENT_EXTERNAL, or the warp-per-environment path (more than
 * CAV_SMALL_M bodies, or cavgym_set_dense_path(1)), or per-env agent parameters set (cavgym_set_agent_params). */
int cavgym_rollout_until(CavEngine* engine, int n_steps, double level, uint64_t salt, void* score, uint8_t* status,
                         cudaStream_t stream);

/* Per-env tester parameters, so that one batch can sweep them: env e's body b uses epsilon[b][e] where the scenario's
 * RandomAgent / RandomConstrainedAgent epsilon (CavBody.agent_epsilon; template.py:52-62, pedestrian.py:72-75) would be used,
 * and threshold[b][e] where its ProximityAgent / ElectionAgent distance_threshold (CavBody.agent_threshold;
 * pedestrian.py:78-91) would be.
 *   epsilon    device double[M][N] (double in both engine types, as agent_epsilon), nullable
 *   threshold  device real[M][N], nullable
 * A NULL array means the scenario's value; both NULL clears the parameters and returns the engine to its plain kernels.
 * Row b of epsilon is read only where body b's agent is CAV_AGENT_RANDOM or CAV_AGENT_RANDOM_CONSTRAINED, row b of threshold
 * only where it is CAV_AGENT_PROXIMITY or CAV_AGENT_ELECTION; other rows may hold anything (NaN included).  The rows that are
 * read must hold epsilon in [0, 1] and threshold > 0 and finite (config.py's ranges): CAV_EINVAL otherwise, and the engine's
 * parameters are left as they were.  The arrays are copied into engine-owned buffers; agent kinds stay the scenario's.
 * The parameters belong to the env SLOTS: cavgym_reset, auto-reset, cavgym_load_envs and cavgym_fork_envs do not move them,
 * and cavgym_save_engine does not carry them.  Philox streams are unchanged: only the decisions draw < epsilon and
 * distance < threshold differ.  Honoured by cavgym_step and cavgym_step_host with on-device agents, cavgym_rollout and
 * cavgym_rollout_record.  While parameters are set, cavgym_step_host_f32 and cavgym_rollout_until return CAV_ESTATE, and
 * so does any stepping call on the warp-per-environment path (cavgym_set_dense_path(1)).
 * CAV_ESTATE also for parameters on a scenario of more than CAV_SMALL_M bodies.  Synchronises `stream`. */
int cavgym_set_agent_params(CavEngine* engine, const double* epsilon, const void* threshold, cudaStream_t stream);

/* Regenerate logged episodes: every slot e of the engine (all N) becomes episode episodes[e] of global env env_ids[e] —
 * the (env, episode) of a CavEpisodeRow, from this engine or any other of the same scenario, seed, dtype and tau — and then
 * steps n_steps times without auto-reset.  With on-device agents an episode's states, actions, done, winner, tangent flags
 * and liveness are a pure function of those, of its (env, episode) key (which keys its spawn and agent draws) and of the
 * slot's tester parameters (cavgym_set_agent_params where set, the scenario's values otherwise).  So an episode played
 * from a reset on the engine's own streams is reproduced bit for bit, K of them side by side in one launch.  t_global
 * only adds the time-out term (quirk 1) to the rewards of one step: it is read at the first step and advances by n_steps,
 * so set it (cavgym_set_global_timestep) to the step at which the episode started.
 *   env_ids   device int64[N], each in [0, 2^40)     episodes  device int32[N], each >= 0
 *   rec       as cavgym_rollout_record's (HOST struct of device pointers), NULL allowed: row 0 is the episode's first
 *             step, rows after it ends are frozen rows.
 * The slot's unfinished episode, if any, is abandoned as cavgym_reset counts it; counters, the episode log and t_global
 * then behave as for cavgym_rollout_record, and an episode row carries env_ids[e], so draining this engine's log gives
 * back the requested rows of the episodes that reproduce.  Episodes that were not played from a reset on the engine's
 * own streams (cavgym_fork_envs or cavgym_load_envs mid-episode, cavgym_rollout_until with a salt) are not reproduced.
 * The keys are range-checked on the device before any state changes: synchronises `stream`.
 * CAV_EINVAL: NULL engine, env_ids or episodes, n_steps < 0, an id or episode out of range.  CAV_ESTATE: a body with
 * CAV_AGENT_EXTERNAL (its actions came from the caller), election testers (the active player outlives episodes, so an
 * episode depends on the ones before it), the warp-per-environment path (more than CAV_SMALL_M bodies, or
 * cavgym_set_dense_path(1)), a uniform or spawn override set. */
int cavgym_regenerate_episodes(CavEngine* engine, const int64_t* env_ids, const int32_t* episodes, int n_steps,
                               const CavRolloutRecord* rec, cudaStream_t stream);

/* Replayed joint actions, n_steps transitions in one launch:
 * actions real[T][M][2][N]; trajectory outputs (each nullable) state real[T][M][4][N],
 * reward real[T][M][N], done u8[T][N], winner i32[T][N], tangent u8[T][N].
 * Every pointer may also be page-locked, device-mapped HOST memory (cavgym_host_alloc, tensor.pin_memory()): the kernel
 * then streams actions in and trajectories out over PCIe inside the launch (BatchedCAVEnv.replay_host).
 * Calls that follow one another directly (no other call on this engine in between) on the same stream are ordered env tile
 * by env tile rather than grid by grid, so their launches overlap on the device; to everything else in the stream — and to
 * the host — they complete in order as usual.  Engine state (cavgym_state_ptr etc.) must not be written by other work of the
 * stream between two such calls without an API call on the engine in between (cavgym_reset, cavgym_step ... all qualify). */
int cavgym_replay(CavEngine* engine, int n_steps, const void* actions, void* state_traj, void* reward_traj,
                  uint8_t* done_traj, int32_t* winner_traj, uint8_t* tangent_traj, cudaStream_t stream);

/* cavgym_step with HOST buffers (same shapes); returns when the outputs are on the host.  Pinned buffers
 * (cudaHostAlloc / cudaHostRegister / torch pin_memory) are read and written by the step kernel itself, zero copy;
 * pageable buffers are copied in and out in env-chunks pipelined over internal streams. */
int cavgym_step_host(CavEngine* engine, const void* actions, void* state_out, void* reward_out,
                     uint8_t* done_out, int32_t* winner_out, uint8_t* tangent_flag_out);

/* cavgym_step_host for an fp64 engine with a float32 WIRE format: actions, state_out and reward_out are float32 host
 * arrays (same shapes); the engine widens the actions, steps in double and narrows the results, so half the bytes cross
 * PCIe.  What the caller gives up is the last 29 bits of every action and observation, nothing else: the engine's state and
 * all events stay those of the fp64 engine fed the widened actions.  Buffers must be page-locked and device-mapped
 * (cavgym_host_alloc, tensor.pin_memory()); scenarios of at most CAV_SMALL_M bodies; CAV_ESTATE otherwise. */
int cavgym_step_host_f32(CavEngine* engine, const float* actions, float* state_out, float* reward_out, uint8_t* done_out,
                         int32_t* winner_out, uint8_t* tangent_flag_out);

/* CAVEnv.reset (environment.py:225-229) with HOST buffers, for callers that hold no device memory (the host-buffer twin
 * of cavgym_reset, as cavgym_step_host is of cavgym_step): mask host u8[N] or NULL, init_state host real[M][4][N] or NULL
 * are copied in; the post-reset state is copied to state_out (host real[M][4][N], nullable).  Synchronises. */
int cavgym_reset_host(CavEngine* engine, const uint8_t* mask, const void* init_state, void* state_out);

/* CAVEnv.info (environment.py:106-117) for the current state of every env, on demand (nothing on the step path reads it):
 * polygons_out   device real[M][8][N]: body_polygons, x of rear_left, front_left, front_right, rear_right, then y
 *                (bodies.py:116-117; PelicanCrossing: its static box), nullable;
 * road_angle_out device real[M][N]: road_angles — DynamicBody.line_anchor_relative_angle towards the major road's centre line
 *                (bodies.py:206-212), NaN where the reference gives None (the body's box intersects the major road), nullable. */
int cavgym_info(CavEngine* engine, void* polygons_out, void* road_angle_out, cudaStream_t stream);

/* ---- snapshots: save, restore and fork environments; checkpoint an engine ---------- */
/* The reference-side equivalent is copy.deepcopy(CAVEnv), whose copies share one MT19937 stream; here an env's random
 * stream is keyed by (global env id, kind, body, episode, t), so an env loaded into a slot of the same global id continues
 * bit for bit, and a copy in another slot continues from the same situation on that slot's own stream.
 * Save, load and fork never touch the counters of cavgym_stats: an overwritten episode is neither scored nor counted as
 * abandoned.  t_global is batch-wide (cavgym_save_engine), so a loaded env times out at the loading engine's t_global.
 * Snapshot rows are not meant to be edited: the cs rows must match the headings; new states go through cavgym_reset.
 * A snapshot is only valid for an engine of the same scenario (fingerprint), dtype and body count.
 * The kernels are ordinary launches on `stream`; a cavgym_replay that follows waits for them like for any other call. */

/* Layout of a snapshot of k envs of this engine; out is HOST memory. */
int cavgym_snapshot_layout(CavEngine* engine, int64_t k, CavSnapshotLayout* out);
/* Copies envs[0..k) (device int64, NULL = all N in order with k = N) into `snapshot` (device, layout total_bytes, 16-byte
 * aligned: CAV_EINVAL otherwise; cudaMalloc and torch allocations are).  k = 0 does nothing.  Indices outside [0, N) are
 * skipped. */
int cavgym_save_envs(CavEngine* engine, const int64_t* envs, int64_t k, void* snapshot, cudaStream_t stream);
/* Writes snapshot column j into env envs[j] (device int64, unique, NULL = all N in order); snapshot as for
 * cavgym_save_envs.  k = 0 does nothing. */
int cavgym_load_envs(CavEngine* engine, const int64_t* envs, int64_t k, const void* snapshot, cudaStream_t stream);
/* Env dst[j] becomes a copy of env src[j] (device int64, dst unique; src may repeat and overlap dst): every source is read,
 * into an engine-owned staging snapshot, before any target is written.  k = 0 does nothing.  All forks of one engine share
 * that staging snapshot, so they must be ordered on one stream.  A fork of more envs than any fork before it on the engine
 * grows the staging snapshot, which synchronises the device (and so cannot be captured into a CUDA graph). */
int cavgym_fork_envs(CavEngine* engine, const int64_t* src, const int64_t* dst, int64_t k, cudaStream_t stream);
/* Engine-wide state; out is HOST memory.  Synchronises. */
int cavgym_save_engine(CavEngine* engine, CavEngineState* out);
/* Restores t_global, the raw counters and tau after checking fingerprint, dtype, m, n, seed and shard (CAV_EINVAL on a
 * mismatch).  The episode-log ring, the replay launch chain and every knob are not part of the state.  Synchronises. */
int cavgym_load_engine(CavEngine* engine, const CavEngineState* in);

/* ---- accounting ------------------------------------------------------------------ */

/* reporting.analyse_episode / analyse_run (reporting.py:227-269) sums over episodes
 * scored so far; out is a HOST int64[CAV_N_STATS].  Synchronises. */
int cavgym_stats(CavEngine* engine, int64_t* out);
int cavgym_error_count(CavEngine* engine, int64_t* out);   /* envs with the invalid-action flag set */
int cavgym_launch_count(CavEngine* engine, int64_t* out);  /* kernels launched by this engine so far */

/* Per-episode rows (Simulation.run's episode.log, simulation.py:103-105): with capacity > 0 every episode scored from
 * now on is also appended to a device ring of `capacity` rows (0 switches it off and frees nothing).  An episode that finds
 * the ring full is still counted in cavgym_stats but its row is dropped; drain often enough. */
int cavgym_set_episode_log(CavEngine* engine, int64_t capacity);
/* Copies the rows appended since the last drain to `out` (HOST, room for max_rows) in append order, empties the ring,
 * *n_rows = rows copied, *dropped = rows lost to a full ring or to max_rows.  Synchronises. */
int cavgym_drain_episodes(CavEngine* engine, CavEpisodeRow* out, int64_t max_rows, int64_t* n_rows, int64_t* dropped);

/* ---- engine-owned device buffers (zero-copy views for the host shim) --------------- */
void* cavgym_state_ptr(CavEngine* engine);          /* real[M][4][N] */
int32_t* cavgym_liveness_ptr(CavEngine* engine);    /* i32[M][N] episode_liveness */
void* cavgym_agent_state_ptr(CavEngine* engine);    /* real[M][5][N] CrossingAgent state, NaN = None */
void* cavgym_action_ptr(CavEngine* engine);         /* real[M][2][N] last joint action taken */
int32_t* cavgym_timestep_ptr(CavEngine* engine);    /* i32[N] timesteps into the current episode */
uint8_t* cavgym_done_ptr(CavEngine* engine);        /* u8[N] latched done */
int32_t* cavgym_winner_ptr(CavEngine* engine);      /* i32[N] latched winner */
uint8_t* cavgym_error_ptr(CavEngine* engine);       /* u8[N] invalid-action flag */

/* ---- knobs ----------------------------------------------------------------------- */

/* Replace the Philox draws by caller-provided [0,1) numbers (replay of the
 * reference's MT19937 draws): device f64[M][CAV_DRAWS][N] read by every later
 * step, NULL restores Philox.  Slot 0 = epsilon test (template.py:61-62), slots
 * 1,2 = Box.sample components / Discrete.sample. */
int cavgym_set_uniform_override(CavEngine* engine, const double* uniforms);

/* Replace the five spawn draws (box, triangle, u, v, orientation) of every
 * SpawnPedestrian by caller-provided [0,1) numbers: device f64[M][5][N], NULL restores Philox. */
int cavgym_set_spawn_override(CavEngine* engine, const double* draws);

/* cavgym_action_ptr normally holds only what a RandomAgent must remember; with logging on,
 * every on-device agent's chosen action is stored there each step (parity tests, compat view). */
int cavgym_set_action_logging(CavEngine* engine, int enabled);

/* cavgym_step with replayed actions normally runs the persistent TMA-staged kernel (whole 128-env tiles, 16-byte
 * aligned buffers) and the plain thread-per-env kernel for whatever is left; use_tma = 0 forces the plain kernel
 * everywhere (A/B measurements, parity of the two paths). */
int cavgym_set_step_path(CavEngine* engine, int use_tma);

/* Scenarios with more than CAV_SMALL_M bodies always run the warp-per-environment kernels (one env per warp, bodies
 * staged in shared memory, fp32 broad phase + exact narrow phase for the all-pairs collision test of
 * environment.py:156-177); force = 1 selects them for a small scenario too (parity of the two paths), 0 goes back. */
int cavgym_set_dense_path(CavEngine* engine, int force);

/* cavgym_step_host with pinned (page-locked, mapped) buffers runs as one launch that reads and writes host memory
 * directly over PCIe; zero_copy = 0 forces the staged path (chunked async copies through device buffers), which is also
 * what pageable buffers get.  Tuning values: 2..8 = zero copy with (zero_copy - 1) resident CTAs per SM. */
int cavgym_set_host_path(CavEngine* engine, int zero_copy);

/* CAVEnv.current_timestep (environment.py:90,222) is never reset by the reference;
 * the engine keeps ONE counter of step calls for the whole batch. */
int cavgym_set_global_timestep(CavEngine* engine, int64_t t);

/* Near-tangent tolerance in pixels (default 1e-7 for f64, 5e-2 for f32). */
int cavgym_set_tangent_tolerance(CavEngine* engine, double tau);

/* ---- stand-alone kernels (per-function parity and the Body.step plugin hook) --------- */

/* DynamicBody.step (bodies.py:214-275) for n independent bodies of one type:
 * state real[4][n] in place, actions real[2][n], device pointers. */
int cavgym_bodies_step(const CavBodyType* type, void* state, const void* actions, int64_t n, double time_resolution,
                       int dtype, cudaStream_t stream);

/* Shape.intersects / contains / percentage_intersects (geometry.py:74-87) for n quad pairs:
 * quads_a, quads_b real[8][n] (x0..x3, y0..y3); out real[4][n] = a.intersects(b), b.contains(a),
 * a.percentage_intersects(b), near-tangent flag. */
int cavgym_geometry_probe(const void* quads_a, const void* quads_b, void* out, int64_t n, int dtype, cudaStream_t stream);

/* DynamicBody.stopping_zones (bodies.py:122-135, geometry.py:176-191) for n independent bodies of one type, from the
 * representation the step kernels test against (braking and reaction rectangles laid end to end in the body's frame):
 * state real[4][n], steering real[n] (the body's current steering angle) -> zones real[16][n] = braking x0..x3, y0..y3,
 * reaction x0..x3, y0..y3 in the reference's corner order (rear left, front left, front right, rear right), and
 * have u8[n] = 0 where the reference returns (None, None): total distance 0 or steering != 0. */
int cavgym_zones_probe(const CavBodyType* type, const void* state, const void* steering, void* zones_out, uint8_t* have_out,
                       int64_t n, int dtype, cudaStream_t stream);

const char* cavgym_last_error(void);
/* Page-locked, device-mapped host memory for the buffers of cavgym_step_host / cavgym_reset_host (what a caller without
 * PyTorch uses instead of tensor.pin_memory()).  write_combined != 0 allocates write-combined memory: meant for buffers the
 * host only WRITES and the GPU reads (the joint actions) — GPU reads of it do not snoop the CPU caches; host reads of it are
 * slow.  Free with cavgym_host_free. */
int cavgym_host_alloc(size_t bytes, int write_combined, void** out);
int cavgym_host_free(void* ptr);

const char* cavgym_version(void);

#ifdef __cplusplus
}
#endif
#endif /* CAVGYM_H */
