// kernels_regen.cuh — cavgym_regenerate_episodes: slot e of the engine replays episode episodes[e] of global env env_id[e],
// whichever run logged it, and records it.
//
// With the stock on-device agents an episode is a pure function of the scenario, seed, dtype and tau, of the key (global env
// id, episode number) of its Philox draws, and of the slot's tester parameters; t_global only adds the time-out term to the
// rewards of one step.  So the kernel keys slot e's draws with env_id[e] (SlotKey) instead of its own global id, resets the
// env in registers exactly as reset_env numbers episodes (the episode counter is episodes[e] - 1 before the increment), then
// runs rollout_record_kernel's loop with auto_reset = 0: the same RolloutRecord rows, frozen rows after the episode ends, the
// same counters, and an episode row that carries env_id[e].  EnvTester reads the engine's per-env parameters where they are
// set and the scenario's otherwise.
//
// An ordinary launch, thread per env: no barriers, no ghost lanes, never programmatically dependent.
// Compiled in regen_mK.cu, apart from small_mK.cu, for the reason record_mK.cu is (kernels_small.cuh).
#pragma once
#include "kernels_params.cuh"

namespace cav {

// Global id given per slot: read once by the kernel, held in a register.
struct SlotKey {
  int64_t id;
  template <typename R> __device__ __forceinline__ int64_t operator()(const EnvBuffers<R>&, int64_t) const { return id; }
};

template <typename R, int M, bool GENERIC>
__global__ void __launch_bounds__((rollout_threads<GENERIC, M>()), (rollout_min_blocks<GENERIC, M>())) regenerate_kernel(
    const __grid_constant__ DevScenario<R> sc, const __grid_constant__ EnvBuffers<R> buf, const __grid_constant__ RolloutRecord<R> rec,
    const __grid_constant__ AgentParams<R> params, const int64_t* env_id, const int32_t* episodes, int64_t t_global, int n_steps) {
  const int64_t e = buf.lo + (int64_t)blockIdx.x * rollout_threads<GENERIC, M>() + threadIdx.x;
  if (e >= buf.hi) return;
  const int64_t n = buf.n;
  const SlotKey key{env_id[e]};
  const EnvTester<R> tester{params};
  // the slot's unfinished episode is abandoned, as cavgym_reset counts it
  if (!buf.done[e] && buf.t_ep[e] > 0) atomicAdd(&buf.stats[CAV_STAT_ENV_STEPS], (unsigned long long)buf.t_ep[e]);
  EnvRegs<R, M> env;
  env.episode = episodes[e] - 1;   // reset_env increments it
  env.active = 0;                  // election testers are refused
  reset_env<R, M, SlotKey>(sc, buf, nullptr, e, env, key);
  R ext[M][2];
  load_actions<R, M>(nullptr, n, e, ext);
  for (int t = 0; t < n_steps; ++t) {
    const int64_t row = (int64_t)t * n;
    const bool stepped = env.done == 0;
    if (rec.observation) {
#pragma unroll
      for (int b = 0; b < M; ++b)
#pragma unroll
        for (int c = 0; c < 4; ++c) rec.observation[row * (M * 4) + ((int64_t)b * 4 + c) * n + e] = env.s[b][c];
    }
    const StepIO<R> at = {nullptr, rec.state ? rec.state + row * (M * 4) : nullptr, rec.reward ? rec.reward + row * M : nullptr,
                          rec.done ? rec.done + row : nullptr, rec.winner ? rec.winner + row : nullptr,
                          rec.tangent ? rec.tangent + row : nullptr, 0};
    advance<R, M, true, GENERIC, NoPhase, EnvTester<R>, SlotKey>(sc, buf, at, e, t_global + t, env, ext, NoPhase(), false, nullptr,
                                                                  tester, key);
    if (rec.action) {
#pragma unroll
      for (int b = 0; b < M; ++b) {
        rec.action[row * (M * 2) + ((int64_t)b * 2 + 0) * n + e] = stepped ? env.held[b][0] : R(0);
        rec.action[row * (M * 2) + ((int64_t)b * 2 + 1) * n + e] = stepped ? env.held[b][1] : R(0);
      }
    }
    if (rec.timestep) rec.timestep[row + e] = stepped ? env.t_ep : 0;
  }
  store_env<R, M, true>(sc, buf, e, env, true);
}

template <typename R>
using RegenerateLauncher = void (*)(const DevScenario<R>&, const EnvBuffers<R>&, const RolloutRecord<R>&, const AgentParams<R>&,
                                    const int64_t* env_id, const int32_t* episodes, int64_t t_global, int n_steps, cudaStream_t);

template <typename R, int M>
void launch_regenerate(const DevScenario<R>& sc, const EnvBuffers<R>& buf, const RolloutRecord<R>& rec, const AgentParams<R>& params,
                       const int64_t* env_id, const int32_t* episodes, int64_t t_global, int n_steps, cudaStream_t stream) {
  constexpr int plain = rollout_threads<false, M>(), synced = rollout_threads<true, M>();
  if (sc.homogeneous)
    regenerate_kernel<R, M, false><<<grid_for(buf, plain), plain, 0, stream>>>(sc, buf, rec, params, env_id, episodes, t_global, n_steps);
  else
    regenerate_kernel<R, M, true><<<grid_for(buf, synced), synced, 0, stream>>>(sc, buf, rec, params, env_id, episodes, t_global, n_steps);
}

// Defined in engine.cu from the regen_mK.cu tables.
template <typename R> RegenerateLauncher<R> regenerate_launcher(int m);

}  // namespace cav
