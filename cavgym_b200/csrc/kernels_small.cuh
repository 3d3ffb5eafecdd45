// kernels_small.cuh — thread-per-environment kernels for scenarios with M <= CAV_SMALL_M bodies.
//
//   step_kernel     one CAVEnv.step over all N envs                 (cavgym_step)
//   replay_kernel   T steps on replayed joint actions, state kept in registers   (cavgym_replay)
//   rollout_kernel  T steps with on-device agents, scoring and auto-reset in-kernel  (cavgym_rollout)
//   rollout_record_kernel  the same, writing per-step [T] slabs                    (cavgym_rollout_record)
//   reset_kernel    CAVEnv.reset for masked envs                    (cavgym_reset / cavgym_create)
//
// HBM layout is SoA with the environment index fastest, so lane i of a warp touches
// consecutive 8-byte (fp64) / 4-byte (fp32) words: every global access is a fully
// coalesced 256 B / 128 B warp transaction.  All loads of a thread are issued before the
// first dependent use (memory-level parallelism = 6M+2 independent loads per thread).
// Roofline: HBM-bound streaming; algorithmic bytes per body-step 88 B (fp64) / 44 B (fp32)
// on replayed actions (SURVEY §8d).  No shared memory: there is no reuse across envs.
#pragma once
#include <type_traits>
#include "transition.cuh"

namespace cav {

constexpr int kThreads = 128;
// The multi-step kernels (replay, rollout) are ONE wave of long-running blocks: with 224-thread blocks, two per SM, the
// 65,536-env configuration is 293 blocks on 296 slots, every env resident from the first step to the last.
#ifndef CAV_LOOP_THREADS
#define CAV_LOOP_THREADS 224
#endif
constexpr int kLoopThreads = CAV_LOOP_THREADS;
// The rollout kernel (on-device agents, auto-reset) usually runs over many more envs than one wave: 128-thread blocks,
// four per SM (pedestrians rollout at 1M envs: 7.2 -> 6.8 ms per 100 steps against 224 x 2).
#ifndef CAV_ROLLOUT_THREADS
#define CAV_ROLLOUT_THREADS 128
#endif
#ifndef CAV_MIN_BLOCKS_ROLLOUT
#define CAV_MIN_BLOCKS_ROLLOUT 4
#endif
constexpr int kRolloutThreads = CAV_ROLLOUT_THREADS;
// The heterogeneous kernels of four or more bodies synchronise their warps at every phase boundary (CtaPhase): the more warps
// walk the code together, the more instruction fetches are shared.  Measured, 1,048,576 envs x 100 steps (ms per launch, four
// launches): bus stop 128 threads 39 / 50 / 52 / 52, 256 threads 37 / 43 / 44 / 44, 512 threads 40 / 42 / 42 / 43; pelican
// crossing 128: 28 / 27 / 29 / 30, 256: 27 / 28 / 31 / 31; crossroads (three bodies) is best at 128.
#ifndef CAV_ROLLOUT_THREADS_SYNCED
#define CAV_ROLLOUT_THREADS_SYNCED 256
#endif
template <bool GENERIC, int M> __host__ __device__ constexpr int rollout_threads() { return GENERIC && M >= 4 ? CAV_ROLLOUT_THREADS_SYNCED : kRolloutThreads; }
template <bool GENERIC, int M> __host__ __device__ constexpr int rollout_min_blocks() {
  return GENERIC && M >= 4 ? (CAV_MIN_BLOCKS_ROLLOUT * kRolloutThreads) / CAV_ROLLOUT_THREADS_SYNCED : CAV_MIN_BLOCKS_ROLLOUT;
}
#ifndef CAV_MIN_BLOCKS_STEP
#define CAV_MIN_BLOCKS_STEP 4
#endif
#ifndef CAV_MIN_BLOCKS_LOOP
#define CAV_MIN_BLOCKS_LOOP 2
#endif

template <typename R, int M, bool AGENTS>
__device__ __forceinline__ void load_env(const DevScenario<R>& sc, const EnvBuffers<R>& buf, int64_t e, EnvRegs<R, M>& env) {
  const int64_t n = buf.n;
  env.done = buf.done[e];
  env.t_ep = buf.t_ep[e];
  env.winner = env.done ? buf.winner[e] : -1;
  env.ag_dirty = 0;
  env.cs_dirty = 0;
  env.live_dirty = 0;
  env.live[0] = 0;
#pragma unroll
  for (int b = 1; b < M; ++b) env.live[b] = buf.liveness[(int64_t)b * n + e];
  env.episode = AGENTS ? buf.episode[e] : 0;
  env.active = AGENTS && M >= 3 && sc.has_election ? buf.active[e] : 0;
#pragma unroll
  for (int b = 0; b < M; ++b) {
#pragma unroll
    for (int c = 0; c < 4; ++c) env.s[b][c] = buf.state[((int64_t)b * 4 + c) * n + e];
    env.held[b][0] = R(0); env.held[b][1] = R(0);
    env.cs[b][0] = R(1); env.cs[b][1] = R(0);
    if (sc.bodies[b].kind == CAV_BODY_DYNAMIC) {
      env.cs[b][0] = buf.cs[((int64_t)b * 2 + 0) * n + e];
      env.cs[b][1] = buf.cs[((int64_t)b * 2 + 1) * n + e];
    }
    if (AGENTS && sc.bodies[b].agent == CAV_AGENT_RANDOM) {
      env.held[b][0] = buf.action[((int64_t)b * 2 + 0) * n + e];
      env.held[b][1] = buf.action[((int64_t)b * 2 + 1) * n + e];
    }
    if (AGENTS && uses_agent_state<R, M>(sc, b)) {
#pragma unroll
      for (int w = 0; w < CAV_AGENT_WORDS; ++w) env.ag[b][w] = buf.agent[((int64_t)b * CAV_AGENT_WORDS + w) * n + e];
    }
  }
}

// Write back what a kernel changed.  `all` forces every per-env word (after a reset).
template <typename R, int M, bool AGENTS>
__device__ __forceinline__ void store_env(const DevScenario<R>& sc, const EnvBuffers<R>& buf, int64_t e, const EnvRegs<R, M>& env,
                                          bool all) {
  const int64_t n = buf.n;
#pragma unroll
  for (int b = 0; b < M; ++b) {
#pragma unroll
    for (int c = 0; c < 4; ++c) buf.state[((int64_t)b * 4 + c) * n + e] = env.s[b][c];
    if (all || (AGENTS && sc.bodies[b].agent != CAV_AGENT_EXTERNAL && (buf.log_actions || sc.bodies[b].agent == CAV_AGENT_RANDOM))) {
      buf.action[((int64_t)b * 2 + 0) * n + e] = env.held[b][0];
      buf.action[((int64_t)b * 2 + 1) * n + e] = env.held[b][1];
    }
    if (all || (env.live_dirty >> b & 1u)) buf.liveness[(int64_t)b * n + e] = env.live[b];
    if (all || (env.cs_dirty >> b & 1u)) {
      buf.cs[((int64_t)b * 2 + 0) * n + e] = env.cs[b][0];
      buf.cs[((int64_t)b * 2 + 1) * n + e] = env.cs[b][1];
    }
    if (all || (AGENTS && uses_agent_state<R, M>(sc, b) && (env.ag_dirty >> b & 1u))) {
#pragma unroll
      for (int w = 0; w < CAV_AGENT_WORDS; ++w) buf.agent[((int64_t)b * CAV_AGENT_WORDS + w) * n + e] = env.ag[b][w];
    }
  }
  buf.t_ep[e] = env.t_ep;
  if (all || env.done) { buf.done[e] = env.done; buf.winner[e] = env.winner; }
  if (all) buf.episode[e] = env.episode;
  if (AGENTS && M >= 3 && sc.has_election) buf.active[e] = env.active;
}

template <typename R, int M>
__device__ __forceinline__ void write_outputs(const EnvBuffers<R>& buf, const StepIO<R>& io, int64_t e, const EnvRegs<R, M>& env,
                                              const R (&reward)[M], bool done, int32_t winner, bool tangent) {
  const int64_t n = buf.n;
  if (io.state_out && io.state_out != buf.state) {
#pragma unroll
    for (int b = 0; b < M; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) io.state_out[((int64_t)b * 4 + c) * n + e] = env.s[b][c];
  }
  if (io.reward_out) {
#pragma unroll
    for (int b = 0; b < M; ++b) io.reward_out[(int64_t)b * n + e] = reward[b];
  }
  if (io.done_out) io.done_out[e] = done ? 1 : 0;
  if (io.winner_out) io.winner_out[e] = winner;
  if (io.tangent_out) io.tangent_out[e] = tangent ? 1 : 0;
}

// One transition of env e held in `env`, with all the bookkeeping shared by the three kernels: frozen envs, invalid
// actions, outputs, latching and scoring.  Returns true if the episode ended in this step.  One output site: frozen
// (finished, not yet reset) envs report reward 0 and their latched done / winner through the same stores.
// `ghost`: the lane steps a COPY of env e to keep its warp whole (rollout_kernel); nothing it does may be seen.
template <typename R, int M, bool AGENTS, bool GENERIC, typename Phase = NoPhase, typename Tester = SceneTester, typename Key = ShardKey>
__device__ __forceinline__ bool advance(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const StepIO<R>& io, int64_t e,
                                        int64_t t_global, EnvRegs<R, M>& env, const R (&ext)[M][2], Phase phase = Phase(),
                                        const bool ghost = false, R* reward_sink = nullptr, const Tester tester = Tester(),
                                        const Key key = Key()) {
  StepResult<R, M> res;
  bool ended = false;
  if (CAV_UNLIKELY(env.done != 0)) {  // frozen until reset
#pragma unroll
    for (int b = 0; b < M; ++b) res.reward[b] = R(0);
    res.terminate = env.done == 1;
    res.winner = env.winner;
    res.tangent = false;
  } else {
    transition<R, M, AGENTS, GENERIC, NoSink, Phase, Tester, Key>(sc, buf, e, t_global, env, ext, res, NoSink(), phase, tester, key);
    if (!ghost) {
      if (CAV_UNLIKELY(res.invalid)) buf.err[e] = 1;
      if (CAV_UNLIKELY(res.tangent)) count_tangent(buf.stats);
      if (CAV_UNLIKELY(env.done != 0)) score_episode<R, M, Key>(buf, env, e, AGENTS ? env.episode : -1, key);
    }
    ended = env.done != 0;
  }
  if (!ghost) write_outputs<R, M>(buf, io, e, env, res.reward, res.terminate, res.winner, res.tangent);
  if (reward_sink) {
#pragma unroll
    for (int b = 0; b < M; ++b) reward_sink[b] = res.reward[b];
  }
  return ended;
}

template <typename R, int M>
__device__ __forceinline__ void load_actions(const R* actions, int64_t n, int64_t e, R (&ext)[M][2]) {
#pragma unroll
  for (int b = 0; b < M; ++b) {
    ext[b][0] = actions ? actions[((int64_t)b * 2 + 0) * n + e] : R(0);
    ext[b][1] = actions ? actions[((int64_t)b * 2 + 1) * n + e] : R(0);
  }
}

template <typename R, int M, bool AGENTS, bool GENERIC>
__global__ void __launch_bounds__(kThreads, CAV_MIN_BLOCKS_STEP) step_kernel(const __grid_constant__ DevScenario<R> sc,
                                                        const __grid_constant__ EnvBuffers<R> buf,
                                                        const __grid_constant__ StepIO<R> io, int64_t t_global) {
  const int64_t e = buf.lo + (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (e < buf.hi) {
    EnvRegs<R, M> env;
    R ext[M][2];
    load_env<R, M, AGENTS>(sc, buf, e, env);
    load_actions<R, M>(io.actions, buf.n, e, ext);
    const bool was_live = env.done == 0;
    advance<R, M, AGENTS, GENERIC>(sc, buf, io, e, t_global, env, ext);
    if (was_live) store_env<R, M, AGENTS>(sc, buf, e, env, false);
  }
}

// cavgym_step_host_f32: the step of an engine of type R with float32 buffers on the host side of the link — actions are
// widened on load, state and rewards narrowed on store; the engine's own state stays in R.
template <typename R, int M, bool AGENTS, bool GENERIC>
__global__ void __launch_bounds__(kThreads, CAV_MIN_BLOCKS_STEP) step_wire32_kernel(const __grid_constant__ DevScenario<R> sc,
                                                               const __grid_constant__ EnvBuffers<R> buf,
                                                               const __grid_constant__ WireIO32 wire, int64_t t_global) {
  const int64_t e = buf.lo + (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (e >= buf.hi) return;
  const int64_t n = buf.n;
  EnvRegs<R, M> env;
  R ext[M][2], reward[M];
  load_env<R, M, AGENTS>(sc, buf, e, env);
#pragma unroll
  for (int b = 0; b < M; ++b) {
    ext[b][0] = wire.actions ? R(wire.actions[((int64_t)b * 2 + 0) * n + e]) : R(0);
    ext[b][1] = wire.actions ? R(wire.actions[((int64_t)b * 2 + 1) * n + e]) : R(0);
  }
  const bool was_live = env.done == 0;
  const StepIO<R> io = {nullptr, nullptr, nullptr, wire.done_out, wire.winner_out, wire.tangent_out, 0};
  advance<R, M, AGENTS, GENERIC>(sc, buf, io, e, t_global, env, ext, NoPhase(), false, reward);
  if (was_live) store_env<R, M, AGENTS>(sc, buf, e, env, false);
#pragma unroll
  for (int b = 0; b < M; ++b) {
    if (wire.state_out) {
#pragma unroll
      for (int c = 0; c < 4; ++c) wire.state_out[((int64_t)b * 4 + c) * n + e] = (float)env.s[b][c];
    }
    if (wire.reward_out) wire.reward_out[(int64_t)b * n + e] = (float)reward[b];
  }
}

// Trajectory outputs are [T][...] slabs of the per-step shapes; io.* point at step 0.
template <typename R, int M, bool GENERIC>
__global__ void __launch_bounds__(kLoopThreads, CAV_MIN_BLOCKS_LOOP) replay_kernel(const __grid_constant__ DevScenario<R> sc,
                                                          const __grid_constant__ EnvBuffers<R> buf,
                                                          const __grid_constant__ StepIO<R> io, int64_t t_global, int n_steps) {
  const int64_t e = buf.lo + (int64_t)blockIdx.x * kLoopThreads + threadIdx.x;
  const int64_t n = buf.n;
  if (e < buf.hi) {
    EnvRegs<R, M> env;
    load_env<R, M, false>(sc, buf, e, env);
    const bool was_live = env.done == 0;
    R ext[M][2], nxt[M][2];
    load_actions<R, M>(io.actions, n, e, ext);
    for (int t = 0; t < n_steps; ++t) {
      // software prefetch: issue step t+1's action loads before step t's arithmetic
      if (t + 1 < n_steps) load_actions<R, M>(io.actions + (int64_t)(t + 1) * M * 2 * n, n, e, nxt);
      StepIO<R> at = io;
      at.actions = nullptr;
      if (io.state_out) at.state_out = io.state_out + (int64_t)t * M * 4 * n;
      if (io.reward_out) at.reward_out = io.reward_out + (int64_t)t * M * n;
      if (io.done_out) at.done_out = io.done_out + (int64_t)t * n;
      if (io.winner_out) at.winner_out = io.winner_out + (int64_t)t * n;
      if (io.tangent_out) at.tangent_out = io.tangent_out + (int64_t)t * n;
      advance<R, M, false, GENERIC>(sc, buf, at, e, t_global + t, env, ext);
#pragma unroll
      for (int b = 0; b < M; ++b) { ext[b][0] = nxt[b][0]; ext[b][1] = nxt[b][1]; }
    }
    if (was_live) store_env<R, M, false>(sc, buf, e, env, false);
  }
}

// The heterogeneous scenarios (crossroads, bus stop, pelican crossing) re-align the warps of a CTA once per step (bar.sync):
// their transition is 5,000 warp-instructions of branchy code per step and the path is bound by instruction fetch
// (DESIGN 4.5) — warps that drift apart over the fused steps each stream the code through the 32 KB instruction cache on
// their own, warps that walk it together share the fetches.  Measured at 1,048,576 envs, 100 steps per launch, with the
// barrier at the top of the step and at the three phase boundaries inside the transition (CtaPhase): bus stop
// 1.69 -> 2.03 G env-steps/s, crossroads 3.39 -> 3.60, pelican crossing 3.39 -> 3.55; the two-body pedestrians kernel loses
// 11 % with a per-step barrier (its loop fits the cache), so it keeps running free.
#ifndef CAV_ROLLOUT_SYNC_FROM_M
#define CAV_ROLLOUT_SYNC_FROM_M 3
#endif
#ifndef CAV_ROLLOUT_SYNC_HOMOGENEOUS   // tuning: barriers in the homogeneous (pedestrians family) rollout kernels too
#define CAV_ROLLOUT_SYNC_HOMOGENEOUS 0
#endif

template <typename R, int M, bool GENERIC>
__global__ void __launch_bounds__((rollout_threads<GENERIC, M>()), (rollout_min_blocks<GENERIC, M>())) rollout_kernel(const __grid_constant__ DevScenario<R> sc,
                                                           const __grid_constant__ EnvBuffers<R> buf, int64_t t_global,
                                                           int n_steps, int auto_reset) {
  const int64_t e_raw = buf.lo + (int64_t)blockIdx.x * rollout_threads<GENERIC, M>() + threadIdx.x;
  const bool in_range = e_raw < buf.hi;
  constexpr bool kSync = (GENERIC && M >= CAV_ROLLOUT_SYNC_FROM_M) || (CAV_ROLLOUT_SYNC_HOMOGENEOUS != 0 && !GENERIC);
  using Phase = typename std::conditional<kSync, CtaPhase, NoPhase>::type;
  // Barriers need every lane of every warp of the CTA to run every step: auto-reset (no env stays finished) and, for the
  // lanes of a ragged last CTA that have no env, a copy of the batch's last env stepped as a ghost.
  const bool sync_on = kSync && auto_reset != 0;
  if (!in_range && !sync_on) return;
  const bool ghost = !in_range;
  const int64_t e = in_range ? e_raw : buf.hi - 1;
  Phase phase;
  if constexpr (kSync) phase.on = sync_on;
  EnvRegs<R, M> env;
  load_env<R, M, true>(sc, buf, e, env);
  const StepIO<R> io = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0};
  R ext[M][2];
  load_actions<R, M>(nullptr, buf.n, e, ext);
  bool was_reset = false;
  for (int t = 0; t < n_steps; ++t) {
    if (sync_on) { __syncwarp(); __syncthreads(); }
    if (CAV_UNLIKELY(env.done != 0)) {
      if (!auto_reset) break;
      reset_env<R, M>(sc, buf, nullptr, e, env);
      was_reset = true;
    }
    advance<R, M, true, GENERIC, Phase>(sc, buf, io, e, t_global + t, env, ext, phase, ghost);
  }
  if (ghost) return;
  if (auto_reset && env.done) { reset_env<R, M>(sc, buf, nullptr, e, env); was_reset = true; }
  store_env<R, M, true>(sc, buf, e, env, was_reset);
}

// cavgym_rollout_record: rollout_kernel's loop, writing row t of every slab of `rec` for each env — the observation after
// the auto-reset at the top of step t, then through advance() the post-step state, reward, done, winner and tangent, then
// the executed action and t_ep.  An env that does not step (finished, auto_reset = 0) keeps filling its rows as a frozen
// env (state unchanged, reward 0, latched done / winner, action 0, timestep 0) where rollout_kernel leaves its loop.  Ghost
// lanes write nothing.  A kernel of its own rather than a flag of rollout_kernel, so that rollout_kernel's code stays as it
// is; the rewards, which rollout_kernel never stores, are formed only here.
template <typename R, int M, bool GENERIC>
__global__ void __launch_bounds__((rollout_threads<GENERIC, M>()), (rollout_min_blocks<GENERIC, M>())) rollout_record_kernel(
    const __grid_constant__ DevScenario<R> sc, const __grid_constant__ EnvBuffers<R> buf, const __grid_constant__ RolloutRecord<R> rec,
    int64_t t_global, int n_steps, int auto_reset) {
  const int64_t e_raw = buf.lo + (int64_t)blockIdx.x * rollout_threads<GENERIC, M>() + threadIdx.x;
  const bool in_range = e_raw < buf.hi;
  constexpr bool kSync = (GENERIC && M >= CAV_ROLLOUT_SYNC_FROM_M) || (CAV_ROLLOUT_SYNC_HOMOGENEOUS != 0 && !GENERIC);
  using Phase = typename std::conditional<kSync, CtaPhase, NoPhase>::type;
  const bool sync_on = kSync && auto_reset != 0;
  if (!in_range && !sync_on) return;
  const bool ghost = !in_range;
  const int64_t e = in_range ? e_raw : buf.hi - 1;
  const int64_t n = buf.n;
  Phase phase;
  if constexpr (kSync) phase.on = sync_on;
  EnvRegs<R, M> env;
  load_env<R, M, true>(sc, buf, e, env);
  R ext[M][2];
  load_actions<R, M>(nullptr, n, e, ext);
  bool was_reset = false;
  for (int t = 0; t < n_steps; ++t) {
    if (sync_on) { __syncwarp(); __syncthreads(); }
    if (CAV_UNLIKELY(env.done != 0) && auto_reset) {
      reset_env<R, M>(sc, buf, nullptr, e, env);
      was_reset = true;
    }
    const int64_t row = (int64_t)t * n;
    const bool stepped = env.done == 0;
    if (!ghost && rec.observation) {
#pragma unroll
      for (int b = 0; b < M; ++b)
#pragma unroll
        for (int c = 0; c < 4; ++c) rec.observation[row * (M * 4) + ((int64_t)b * 4 + c) * n + e] = env.s[b][c];
    }
    const StepIO<R> at = {nullptr, rec.state ? rec.state + row * (M * 4) : nullptr, rec.reward ? rec.reward + row * M : nullptr,
                          rec.done ? rec.done + row : nullptr, rec.winner ? rec.winner + row : nullptr,
                          rec.tangent ? rec.tangent + row : nullptr, 0};
    advance<R, M, true, GENERIC, Phase>(sc, buf, at, e, t_global + t, env, ext, phase, ghost);
    if (!ghost && rec.action) {
#pragma unroll
      for (int b = 0; b < M; ++b) {
        rec.action[row * (M * 2) + ((int64_t)b * 2 + 0) * n + e] = stepped ? env.held[b][0] : R(0);
        rec.action[row * (M * 2) + ((int64_t)b * 2 + 1) * n + e] = stepped ? env.held[b][1] : R(0);
      }
    }
    if (!ghost && rec.timestep) rec.timestep[row + e] = stepped ? env.t_ep : 0;
  }
  if (ghost) return;
  if (auto_reset && env.done) { reset_env<R, M>(sc, buf, nullptr, e, env); was_reset = true; }
  store_env<R, M, true>(sc, buf, e, env, was_reset);
}

template <typename R, int M>
__global__ void __launch_bounds__(kThreads) reset_kernel(const __grid_constant__ DevScenario<R> sc,
                                                         const __grid_constant__ EnvBuffers<R> buf, const uint8_t* mask,
                                                         const R* init, int first_time) {
  const int64_t e = buf.lo + (int64_t)blockIdx.x * kThreads + threadIdx.x;
  const bool mine = e < buf.hi && (!mask || mask[e]);
  // an unfinished episode is abandoned: keep its steps in the env-step total.  One atomic per warp, not per env: a reset of
  // a whole batch mid-episode would otherwise queue 65,536 atomics on one counter (35 us for a 5 us kernel).
  unsigned long long abandoned = 0;
  if (mine && !first_time && !buf.done[e]) abandoned = (unsigned long long)buf.t_ep[e];
  abandoned = warp_sum(abandoned);
  if ((threadIdx.x & 31) == 0 && abandoned) atomicAdd(&buf.stats[CAV_STAT_ENV_STEPS], abandoned);
  if (!mine) return;
  EnvRegs<R, M> env;
  env.episode = first_time ? -1 : buf.episode[e];
  env.active = first_time || !sc.has_election ? 0 : buf.active[e];   // the Election object outlives episodes (election.py:12)
  reset_env<R, M>(sc, buf, init, e, env);
  store_env<R, M, true>(sc, buf, e, env, true);
  if (first_time) buf.err[e] = 0;
}

// ---------------------------------------------------------------- host-side launch table
template <typename R>
struct SmallLaunchers {
  void (*step)(const DevScenario<R>&, const EnvBuffers<R>&, const StepIO<R>&, int64_t t_global, bool agents, cudaStream_t);
  void (*replay)(const DevScenario<R>&, const EnvBuffers<R>&, const StepIO<R>&, int64_t t_global, int n_steps, cudaStream_t);
  void (*rollout)(const DevScenario<R>&, const EnvBuffers<R>&, int64_t t_global, int n_steps, int auto_reset, cudaStream_t);
  void (*reset)(const DevScenario<R>&, const EnvBuffers<R>&, const uint8_t* mask, const R* init, int first_time, cudaStream_t);
  // TMA-staged step for replayed actions (kernels_tma.cuh): steps the whole tiles of [lo, hi) it can take and reports how
  // many envs that was (0 = buffers not 16-byte aligned: use `step`); false = launch set-up failed.
  bool (*step_tma)(const DevScenario<R>&, const EnvBuffers<R>&, const StepIO<R>&, int64_t t_global, cudaStream_t, int64_t* envs_done);
  bool (*replay_tma)(const DevScenario<R>&, const EnvBuffers<R>&, const StepIO<R>&, int64_t t_global, int n_steps, cudaStream_t,
                     int64_t* envs_done);
  // step with float32 host-side buffers (cavgym_step_host_f32); false = not compiled for this engine type
  bool (*step_wire32)(const DevScenario<R>&, const EnvBuffers<R>&, const WireIO32&, int64_t t_global, bool agents, cudaStream_t);
};

template <typename R> inline unsigned grid_for(const EnvBuffers<R>& buf, int threads = kThreads) {
  return (unsigned)((buf.hi - buf.lo + threads - 1) / threads);
}

// sc.homogeneous (set by the host when the scenario qualifies) selects the GENERIC = false instantiation.
template <typename R, int M>
void launch_step(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const StepIO<R>& io, int64_t t_global, bool agents,
                 cudaStream_t stream) {
  const unsigned grid = grid_for(buf);
  if (sc.homogeneous) {
    if (agents) step_kernel<R, M, true, false><<<grid, kThreads, 0, stream>>>(sc, buf, io, t_global);
    else step_kernel<R, M, false, false><<<grid, kThreads, 0, stream>>>(sc, buf, io, t_global);
  } else {
    if (agents) step_kernel<R, M, true, true><<<grid, kThreads, 0, stream>>>(sc, buf, io, t_global);
    else step_kernel<R, M, false, true><<<grid, kThreads, 0, stream>>>(sc, buf, io, t_global);
  }
}
template <typename R, int M>
bool launch_step_wire32(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const WireIO32& wire, int64_t t_global, bool agents,
                        cudaStream_t stream) {
  if constexpr (!std::is_same<R, double>::value) {
    return false;   // a float32 engine already has float32 buffers: cavgym_step_host
  } else {
    const unsigned grid = grid_for(buf);
    if (sc.homogeneous) {
      if (agents) step_wire32_kernel<R, M, true, false><<<grid, kThreads, 0, stream>>>(sc, buf, wire, t_global);
      else step_wire32_kernel<R, M, false, false><<<grid, kThreads, 0, stream>>>(sc, buf, wire, t_global);
    } else {
      if (agents) step_wire32_kernel<R, M, true, true><<<grid, kThreads, 0, stream>>>(sc, buf, wire, t_global);
      else step_wire32_kernel<R, M, false, true><<<grid, kThreads, 0, stream>>>(sc, buf, wire, t_global);
    }
    return true;
  }
}
template <typename R, int M>
void launch_replay(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const StepIO<R>& io, int64_t t_global, int n_steps,
                   cudaStream_t stream) {
  if (sc.homogeneous) replay_kernel<R, M, false><<<grid_for(buf, kLoopThreads), kLoopThreads, 0, stream>>>(sc, buf, io, t_global, n_steps);
  else replay_kernel<R, M, true><<<grid_for(buf, kLoopThreads), kLoopThreads, 0, stream>>>(sc, buf, io, t_global, n_steps);
}
template <typename R, int M>
void launch_rollout(const DevScenario<R>& sc, const EnvBuffers<R>& buf, int64_t t_global, int n_steps, int auto_reset,
                    cudaStream_t stream) {
  constexpr int plain = rollout_threads<false, M>(), synced = rollout_threads<true, M>();
  if (sc.homogeneous) rollout_kernel<R, M, false><<<grid_for(buf, plain), plain, 0, stream>>>(sc, buf, t_global, n_steps, auto_reset);
  else rollout_kernel<R, M, true><<<grid_for(buf, synced), synced, 0, stream>>>(sc, buf, t_global, n_steps, auto_reset);
}
template <typename R, int M>
void launch_rollout_record(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const RolloutRecord<R>& rec, int64_t t_global,
                           int n_steps, int auto_reset, cudaStream_t stream) {
  constexpr int plain = rollout_threads<false, M>(), synced = rollout_threads<true, M>();
  if (sc.homogeneous) rollout_record_kernel<R, M, false><<<grid_for(buf, plain), plain, 0, stream>>>(sc, buf, rec, t_global, n_steps, auto_reset);
  else rollout_record_kernel<R, M, true><<<grid_for(buf, synced), synced, 0, stream>>>(sc, buf, rec, t_global, n_steps, auto_reset);
}
template <typename R, int M>
void launch_reset(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const uint8_t* mask, const R* init, int first_time,
                  cudaStream_t stream) {
  reset_kernel<R, M><<<grid_for(buf), kThreads, 0, stream>>>(sc, buf, mask, init, first_time);
}

// Defined in small_mK.cu (one translation unit per body count so they compile in parallel).
template <typename R> const SmallLaunchers<R>* small_launchers(int m);

// cavgym_rollout_record (launch_rollout_record), defined in record_mK.cu: translation units apart from small_mK.cu, where a
// further caller of the transition's out-of-line helpers would change how they are compiled for the existing kernels.
template <typename R>
using RolloutRecordLauncher = void (*)(const DevScenario<R>&, const EnvBuffers<R>&, const RolloutRecord<R>&, int64_t t_global,
                                       int n_steps, int auto_reset, cudaStream_t);
template <typename R> RolloutRecordLauncher<R> rollout_record_launcher(int m);

}  // namespace cav
