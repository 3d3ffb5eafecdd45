// kernels_until.cuh — cavgym_rollout_until: rollout_kernel's loop without auto-reset, carrying one caller-owned score per env
// and parking an env at the first step where its score reaches a level (the stage of a multilevel splitting scheme).
//
// Per env, at entry: a finished env (done != 0) is not stepped — parked with score +inf when its latched winner is a tester
// (> 0), finished otherwise; a live env whose score is already >= level is parked without a step.  Then per step: a step that
// ends the episode with a tester win sets score = +inf (parked); one that ends it otherwise (done, or cut off at
// max_timesteps) finishes the env with its score unchanged; any other step sets score = max(score, danger) (danger.cuh) and
// parks the env once score >= level.  A parked env leaves the loop as a frozen env leaves rollout_kernel's, so its state is
// the state after that step.  Everything a step does besides (store_env, scoring through advance, error flags, tangent
// counter) is rollout_kernel's.
//
// Thread per env with no barriers and no ghost lanes: without auto-reset rollout_kernel does not synchronise either.
// Compiled in until_mK.cu, apart from small_mK.cu, for the reason record_mK.cu is (kernels_small.cuh).
#pragma once
#include "danger.cuh"
#include "kernels_small.cuh"

namespace cav {

enum : uint8_t { UNTIL_LIVE = 0, UNTIL_PARKED = 1, UNTIL_FINISHED = 2 };

template <typename R, int M, bool GENERIC>
__global__ void __launch_bounds__((rollout_threads<GENERIC, M>()), (rollout_min_blocks<GENERIC, M>())) rollout_until_kernel(
    const __grid_constant__ DevScenario<R> sc, const __grid_constant__ EnvBuffers<R> buf, R* score, uint8_t* status, double level,
    int64_t t_global, int n_steps) {
  const int64_t e = buf.lo + (int64_t)blockIdx.x * rollout_threads<GENERIC, M>() + threadIdx.x;
  if (e >= buf.hi) return;
  EnvRegs<R, M> env;
  load_env<R, M, true>(sc, buf, e, env);
  R s = score[e];
  uint8_t st = UNTIL_LIVE;
  if (env.done != 0) {
    st = env.winner > 0 ? UNTIL_PARKED : UNTIL_FINISHED;
    if (env.winner > 0) s = R(INFINITY);
  } else if ((double)s >= level) {
    st = UNTIL_PARKED;
  }
  if (st == UNTIL_LIVE) {
    const StepIO<R> io = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0};
    R ext[M][2];
    load_actions<R, M>(nullptr, buf.n, e, ext);
    for (int t = 0; t < n_steps; ++t) {
      if (advance<R, M, true, GENERIC>(sc, buf, io, e, t_global + t, env, ext)) {
        if (env.winner > 0) { s = R(INFINITY); st = UNTIL_PARKED; }
        else st = UNTIL_FINISHED;
        break;
      }
      s = rmax(s, danger<R, M, GENERIC>(sc, env));
      if ((double)s >= level) { st = UNTIL_PARKED; break; }
    }
    store_env<R, M, true>(sc, buf, e, env, false);
  }
  score[e] = s;
  status[e] = st;
}

// SplitMix64's output function (Steele, Lea and Flood 2014): a salt of a few bits still changes about half the key's bits.
inline uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

template <typename R>
using RolloutUntilLauncher = void (*)(const DevScenario<R>&, const EnvBuffers<R>&, R* score, uint8_t* status, double level,
                                      uint64_t salt, int64_t t_global, int n_steps, cudaStream_t);

// salt != 0 keys this launch's Philox draws with seed ^ splitmix64(salt), in the by-value copy of the buffers only: the
// engine's seed (and so every other call and every checkpoint) is unchanged.
template <typename R, int M>
void launch_rollout_until(const DevScenario<R>& sc, const EnvBuffers<R>& engine_buf, R* score, uint8_t* status, double level,
                          uint64_t salt, int64_t t_global, int n_steps, cudaStream_t stream) {
  EnvBuffers<R> buf = engine_buf;
  if (salt != 0) buf.seed ^= splitmix64(salt);
  constexpr int plain = rollout_threads<false, M>(), synced = rollout_threads<true, M>();
  if (sc.homogeneous)
    rollout_until_kernel<R, M, false><<<grid_for(buf, plain), plain, 0, stream>>>(sc, buf, score, status, level, t_global, n_steps);
  else
    rollout_until_kernel<R, M, true><<<grid_for(buf, synced), synced, 0, stream>>>(sc, buf, score, status, level, t_global, n_steps);
}

// Defined in engine.cu from the until_mK.cu tables.
template <typename R> RolloutUntilLauncher<R> rollout_until_launcher(int m);

}  // namespace cav
