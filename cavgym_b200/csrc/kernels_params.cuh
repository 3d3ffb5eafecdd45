// kernels_params.cuh — the thread-per-environment step, rollout and recording kernels with per-env tester parameters
// (cavgym_set_agent_params): body b of env e compares its draw with epsilon[b][e] where the scenario's RandomAgent /
// RandomConstrainedAgent would compare it with its one epsilon (template.py:52-62, pedestrian.py:72-75), and its distance to
// the ego with threshold[b][e] where ProximityAgent / ElectionAgent would use their one distance_threshold
// (pedestrian.py:78-91).  Everything else — Philox streams and keys included — is the plain kernels' code: the same
// transition (transition.cuh), given EnvTester instead of SceneTester.
//
// The parameters are read where the decision is taken, once per step and tester body, coalesced (env index fastest) and
// L2-resident for any batch a B200 holds.  Only the bodies whose agent kind reads a row ever load from it.  A ghost lane of the
// synced kernels steps a copy of env hi - 1 and so reads that env's parameters.
//
// Compiled in params_mK.cu, apart from small_mK.cu, for the reason record_mK.cu is (kernels_small.cuh).
#pragma once
#include "kernels_small.cuh"

namespace cav {

template <typename R>
struct EnvTester {
  AgentParams<R> p;
  __device__ __forceinline__ double epsilon(const DevBody<R>& body, int b, int64_t e, int64_t n) const {
    return p.epsilon ? p.epsilon[(int64_t)b * n + e] : body.epsilon;
  }
  __device__ __forceinline__ R threshold(const DevBody<R>& body, int b, int64_t e, int64_t n) const {
    return p.threshold ? p.threshold[(int64_t)b * n + e] : body.threshold;
  }
};

// step_kernel<R, M, true, GENERIC>, rollout_kernel and rollout_record_kernel (kernels_small.cuh) line for line, with `tester`
// given to advance().  Copies rather than one body shared through an inline function: the plain kernels compiled from such
// a shared body were no longer instruction-for-instruction what they were.
template <typename R, int M, bool GENERIC>
__global__ void __launch_bounds__(kThreads, CAV_MIN_BLOCKS_STEP) step_params_kernel(const __grid_constant__ DevScenario<R> sc,
                                                                const __grid_constant__ EnvBuffers<R> buf,
                                                                const __grid_constant__ StepIO<R> io,
                                                                const __grid_constant__ AgentParams<R> params, int64_t t_global) {
  const int64_t e = buf.lo + (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (e < buf.hi) {
    EnvRegs<R, M> env;
    R ext[M][2];
    load_env<R, M, true>(sc, buf, e, env);
    load_actions<R, M>(io.actions, buf.n, e, ext);
    const bool was_live = env.done == 0;
    advance<R, M, true, GENERIC, NoPhase, EnvTester<R>>(sc, buf, io, e, t_global, env, ext, NoPhase(), false, nullptr, EnvTester<R>{params});
    if (was_live) store_env<R, M, true>(sc, buf, e, env, false);
  }
}

template <typename R, int M, bool GENERIC>
__global__ void __launch_bounds__((rollout_threads<GENERIC, M>()), (rollout_min_blocks<GENERIC, M>())) rollout_params_kernel(
    const __grid_constant__ DevScenario<R> sc, const __grid_constant__ EnvBuffers<R> buf, const __grid_constant__ AgentParams<R> params,
    int64_t t_global, int n_steps, int auto_reset) {
  const int64_t e_raw = buf.lo + (int64_t)blockIdx.x * rollout_threads<GENERIC, M>() + threadIdx.x;
  const bool in_range = e_raw < buf.hi;
  constexpr bool kSync = (GENERIC && M >= CAV_ROLLOUT_SYNC_FROM_M) || (CAV_ROLLOUT_SYNC_HOMOGENEOUS != 0 && !GENERIC);
  using Phase = typename std::conditional<kSync, CtaPhase, NoPhase>::type;
  const bool sync_on = kSync && auto_reset != 0;
  if (!in_range && !sync_on) return;
  const bool ghost = !in_range;
  const int64_t e = in_range ? e_raw : buf.hi - 1;   // a ghost steps env hi - 1, with env hi - 1's parameters
  Phase phase;
  if constexpr (kSync) phase.on = sync_on;
  const EnvTester<R> tester{params};
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
    advance<R, M, true, GENERIC, Phase, EnvTester<R>>(sc, buf, io, e, t_global + t, env, ext, phase, ghost, nullptr, tester);
  }
  if (ghost) return;
  if (auto_reset && env.done) { reset_env<R, M>(sc, buf, nullptr, e, env); was_reset = true; }
  store_env<R, M, true>(sc, buf, e, env, was_reset);
}

template <typename R, int M, bool GENERIC>
__global__ void __launch_bounds__((rollout_threads<GENERIC, M>()), (rollout_min_blocks<GENERIC, M>())) rollout_record_params_kernel(
    const __grid_constant__ DevScenario<R> sc, const __grid_constant__ EnvBuffers<R> buf, const __grid_constant__ RolloutRecord<R> rec,
    const __grid_constant__ AgentParams<R> params, int64_t t_global, int n_steps, int auto_reset) {
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
  const EnvTester<R> tester{params};
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
    advance<R, M, true, GENERIC, Phase, EnvTester<R>>(sc, buf, at, e, t_global + t, env, ext, phase, ghost, nullptr, tester);
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

template <typename R>
struct ParamsLaunchers {
  // step with on-device agents (cavgym_step, cavgym_step_host) over [buf.lo, buf.hi)
  void (*step)(const DevScenario<R>&, const EnvBuffers<R>&, const StepIO<R>&, const AgentParams<R>&, int64_t t_global, cudaStream_t);
  void (*rollout)(const DevScenario<R>&, const EnvBuffers<R>&, const AgentParams<R>&, int64_t t_global, int n_steps, int auto_reset,
                  cudaStream_t);
  void (*rollout_record)(const DevScenario<R>&, const EnvBuffers<R>&, const RolloutRecord<R>&, const AgentParams<R>&, int64_t t_global,
                         int n_steps, int auto_reset, cudaStream_t);
};

template <typename R, int M>
void launch_step_params(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const StepIO<R>& io, const AgentParams<R>& params,
                        int64_t t_global, cudaStream_t stream) {
  const unsigned grid = grid_for(buf);
  if (sc.homogeneous) step_params_kernel<R, M, false><<<grid, kThreads, 0, stream>>>(sc, buf, io, params, t_global);
  else step_params_kernel<R, M, true><<<grid, kThreads, 0, stream>>>(sc, buf, io, params, t_global);
}
template <typename R, int M>
void launch_rollout_params(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const AgentParams<R>& params, int64_t t_global,
                           int n_steps, int auto_reset, cudaStream_t stream) {
  constexpr int plain = rollout_threads<false, M>(), synced = rollout_threads<true, M>();
  if (sc.homogeneous)
    rollout_params_kernel<R, M, false><<<grid_for(buf, plain), plain, 0, stream>>>(sc, buf, params, t_global, n_steps, auto_reset);
  else
    rollout_params_kernel<R, M, true><<<grid_for(buf, synced), synced, 0, stream>>>(sc, buf, params, t_global, n_steps, auto_reset);
}
template <typename R, int M>
void launch_rollout_record_params(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const RolloutRecord<R>& rec,
                                  const AgentParams<R>& params, int64_t t_global, int n_steps, int auto_reset, cudaStream_t stream) {
  constexpr int plain = rollout_threads<false, M>(), synced = rollout_threads<true, M>();
  if (sc.homogeneous)
    rollout_record_params_kernel<R, M, false><<<grid_for(buf, plain), plain, 0, stream>>>(sc, buf, rec, params, t_global, n_steps,
                                                                                        auto_reset);
  else
    rollout_record_params_kernel<R, M, true><<<grid_for(buf, synced), synced, 0, stream>>>(sc, buf, rec, params, t_global, n_steps,
                                                                                         auto_reset);
}

template <typename R, int M>
constexpr ParamsLaunchers<R> make_params_launchers() {
  return {&launch_step_params<R, M>, &launch_rollout_params<R, M>, &launch_rollout_record_params<R, M>};
}

// Defined in engine.cu from the params_mK.cu tables.
template <typename R> const ParamsLaunchers<R>* params_launchers(int m);

// cavgym_set_agent_params' range check of the rows that are read (bit b of eps_rows / thr_rows: body b's agent reads that row):
// bit 0 of *bad for an epsilon outside [0, 1] or NaN, bit 1 for a threshold that is not finite and > 0.
template <typename R>
__global__ void check_agent_params_kernel(const double* epsilon, const R* threshold, int64_t n, int m, uint32_t eps_rows,
                                          uint32_t thr_rows, unsigned int* bad) {
  const int64_t total = (int64_t)m * n;
  unsigned int flags = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / n);
    if (epsilon && (eps_rows >> b & 1u)) {
      const double v = epsilon[i];
      if (!(v >= 0.0 && v <= 1.0)) flags |= 1u;
    }
    if (threshold && (thr_rows >> b & 1u)) {
      const R v = threshold[i];
      if (!(v > R(0) && v < R(INFINITY))) flags |= 2u;
    }
  }
  if (flags) atomicOr(bad, flags);
}

}  // namespace cav
