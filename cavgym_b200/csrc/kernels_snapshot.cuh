// kernels_snapshot.cuh — moves the per-env rows of selected environments between the engine's SoA buffers and a packed
// snapshot (cavgym_save_envs / cavgym_load_envs / cavgym_fork_envs, include/cavgym.h).
//
// A snapshot of k envs holds, per section, rows of k elements (snapshot row r, env j at r * k + j); the engine holds the
// same rows with n elements (env e at r * n + e).  One launch moves every row of one element size (8, 4 or 1 bytes; fp32
// reals share the 4-byte launch with the int32 rows): the segment table names, for each engine buffer of that size, its
// base, the base of its rows in the snapshot and its row count.  A thread owns one snapshot column j and kSnapRows
// consecutive rows, so it reads its index once and the snapshot side of every row is coalesced across the warp; the
// engine side follows the index list (gathered or scattered).  All envs in order is a straight copy (append_wide).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace cav {

constexpr int kSnapMaxSegments = 11;  // every per-env buffer: state, action, agent, cs, liveness, t_ep, episode, winner, active, done, err
constexpr int kSnapRows = 8;          // rows per thread (loads in flight per thread)
constexpr int kSnapThreads = 256;

template <typename T>
struct SnapTable {
  T* eng[kSnapMaxSegments];         // engine buffer: rows of n elements
  T* snap[kSnapMaxSegments];        // the same rows in the snapshot: rows of k elements
  int64_t row_end[kSnapMaxSegments];  // cumulative row count up to and including segment s
  int32_t n_seg;
  int32_t to_snapshot;              // 1: engine -> snapshot (save, gather); 0: snapshot -> engine (load, scatter)
  int64_t n, k;
  const int64_t* idx;               // [k] engine env of snapshot column j; null: column j is env j (k == n)
};

// Never launched with the programmatic-dependent-launch attribute: replay_tma_kernel releases its dependents at entry, and
// a dependent snapshot launch would then read or overwrite env state under a running replay.
template <typename T>
__global__ void __launch_bounds__(kSnapThreads) snapshot_kernel(const __grid_constant__ SnapTable<T> t) {
  const int64_t j = (int64_t)blockIdx.x * kSnapThreads + threadIdx.x;
  if (j >= t.k) return;
  const int64_t e = t.idx ? t.idx[j] : j;
  if (e < 0 || e >= t.n) return;   // the API validates indices; an out-of-range one is skipped, never followed
  const int64_t rows = t.row_end[t.n_seg - 1];
  const int64_t row0 = (int64_t)blockIdx.y * kSnapRows;
  const T* src[kSnapRows];
  T* dst[kSnapRows];
  int s = 0;
#pragma unroll
  for (int i = 0; i < kSnapRows; ++i) {
    const int64_t row = row0 + i;
    src[i] = nullptr;
    dst[i] = nullptr;
    if (row < rows) {
      while (row >= t.row_end[s]) ++s;   // block-uniform
      const int64_t r = row - (s ? t.row_end[s - 1] : 0);
      T* engine = t.eng[s] + r * t.n + e;
      T* snap = t.snap[s] + r * t.k + j;
      src[i] = t.to_snapshot ? engine : snap;
      dst[i] = t.to_snapshot ? snap : engine;
    }
  }
  T v[kSnapRows];
#pragma unroll
  for (int i = 0; i < kSnapRows; ++i)
    if (src[i]) v[i] = *src[i];
#pragma unroll
  for (int i = 0; i < kSnapRows; ++i)
    if (dst[i]) *dst[i] = v[i];
}

// Host side: one launch over every row of the table (grid: 256 columns x kSnapRows rows per block).
template <typename T>
inline void launch_snapshot(const SnapTable<T>& t, cudaStream_t stream) {
  if (t.k <= 0 || t.n_seg <= 0) return;
  const int64_t rows = t.row_end[t.n_seg - 1];
  const dim3 grid((unsigned)((t.k + kSnapThreads - 1) / kSnapThreads), (unsigned)((rows + kSnapRows - 1) / kSnapRows));
  snapshot_kernel<T><<<grid, kSnapThreads, 0, stream>>>(t);
}

// All envs in order (no index list, k == n) with k a multiple of 16: every segment of every element size is then one
// contiguous, 16-byte aligned block on both sides, and a row of `elem`-byte words is `elem` rows of k / 16 16-byte words.
// The whole save or load becomes ONE straight copy in 16-byte words.
template <typename T>
inline void append_wide(SnapTable<uint4>& w, const SnapTable<T>& t) {
  for (int s = 0; s < t.n_seg; ++s) {
    const int i = w.n_seg++;
    w.eng[i] = reinterpret_cast<uint4*>(t.eng[s]);
    w.snap[i] = reinterpret_cast<uint4*>(t.snap[s]);
    w.row_end[i] = (i ? w.row_end[i - 1] : 0) + (t.row_end[s] - (s ? t.row_end[s - 1] : 0)) * (int64_t)sizeof(T);
  }
}

}  // namespace cav
