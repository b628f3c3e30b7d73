// The window normalisers of utils/preprocessor.py:53-107, shared by the window materialiser (mdg_aux.cu) and the
// replay rows gather (mdg_replay.cuh): one implementation, so a window normalised at sample time is bit-identical to
// the one env.window() writes.
#pragma once
#include <float.h>

#include "mdg_common.cuh"
#include "mdg_math.cuh"

namespace mdg {

__device__ __forceinline__ double nan_to_num(double x) {  // np.nan_to_num
  if (x != x) return 0.;
  if (isinf(x)) return x > 0 ? DBL_MAX : -DBL_MAX;
  return x;
}

// Sum over the time axis of one column, in numpy's order (the reference's mean/std are numpy reductions of the
// window the normaliser sees):
//   * that array has more than one column, (k, F>1): numpy reduces axis 0 row by row -> a left-to-right fold;
//   * it has one column, (k, 1): numpy coalesces it to 1-D and sums it pairwise (`pairwise`):
//       n < 8          left to right;
//       8 <= n <= 128  eight interleaved accumulators, combined ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the
//                      n % 8 tail left to right;
//       n > 128        split at n2 = n/2 - (n/2) % 8 and add the sums of [0, n2) and [n2, n), each by these rules.
// MODE 0: x   1: (x-c)^2   2: x with NaN -> 0 (nansum)   3: (x-c)^2 with NaN -> 0
template <int MODE>
__device__ __forceinline__ double col_term(const double* col, int s, int sstride, double c) {
  const double x = col[s * sstride];
  if (MODE == 0) return x;
  if (MODE == 2) return (x == x) ? x : 0.;
  const double d = x - c;
  if (MODE == 3 && !(x == x)) return 0.;
  return d * d;
}
// numpy's pairwise block, 8 <= n <= 128
template <int MODE>
__device__ __forceinline__ double col_block8(const double* col, int n, int sstride, double c) {
  double r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = col_term<MODE>(col, j, sstride, c);
  int i = 8;
  for (; i < n - (n % 8); i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = r[j] + col_term<MODE>(col, i + j, sstride, c);
  }
  double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
  for (; i < n; ++i) res = res + col_term<MODE>(col, i, sstride, c);
  return res;
}
// n > 128, pairwise: out of line, so that the halving walk does not weigh on the common case's register allocation
template <int MODE>
__device__ __noinline__ double col_sum_halving(const double* col, int n, int sstride, double c) {
  // The halving recursion (no device recursion), walked block by block from the left.  The current node is the path
  // from the whole column: bit i of `path` set = it lies in the right half at halving i, and left[i] then holds the
  // sum of that left half.  A halving leaves at most m/2 + 8 rows, so any int n reaches a block within 25 halvings.
  double left[25];
  unsigned path = 0;
  int d = 0;
  for (;;) {
    int s = 0, m = n;  // the current node: rows [s, s + m)
    for (int i = 0; i < d; ++i) {
      const int h = m / 2 - (m / 2) % 8;
      if ((path >> i) & 1u) { s += h; m -= h; } else { m = h; }
    }
    while (m > 128) { m = m / 2 - (m / 2) % 8; ++d; }  // down the left halves to a block
    double v = col_block8<MODE>(col + s * sstride, m, sstride, c);
    while (d > 0 && ((path >> (d - 1)) & 1u)) {  // a right half is done: so is its parent
      --d;
      path &= ~(1u << d);
      v = left[d] + v;
    }
    if (d == 0) return v;
    left[d - 1] = v;  // a left half is done: go to its sibling
    path |= 1u << (d - 1);
  }
}
template <int MODE>
__device__ __forceinline__ double col_sum(const double* col, int n, int sstride, double c, bool pairwise) {
  if (!pairwise || n < 8) {
    double s = col_term<MODE>(col, 0, sstride, c);
    for (int i = 1; i < n; ++i) s = s + col_term<MODE>(col, i, sstride, c);
    return s;
  }
  if (n <= 128) return col_block8<MODE>(col, n, sstride, c);
  return col_sum_halving<MODE>(col, n, sstride, c);
}

// Normalise, in place, the windows of a shared-memory tile: window w starts at tile + w * a.estride, its row s at
// + s * a.sstride, feature f at + f; nv rows, the normaliser a.norm sees features [0, Fe).  The tile holds windows
// e0 ... e0 + a.envs - 1 of a.N; those past the end are skipped.  The calling thread owns the column `col` (feature f of
// one window) together with Z - 1 others (z = 0..Z-1 split its rows); `mine` = the column is real and f < Fe.  cpar: the column's (shift, scale) pair in shared memory.
// `pairwise`: the array the reference normalises has this one column (col_sum).
// Every thread of the block calls it (barriers inside); the caller synchronises before reading the tile.
// The element-wise parts (logs, the final scale/shift) are spread over the Z threads of a column; only the column
// statistics (sums in numpy's order) are one thread per column.  Divisions by a per-column constant are
// multiplications by its reciprocal, logs are mdg_math's fast_log (observations carry the 1e-9 bar).
template <class Tile>
__device__ __forceinline__ void normalise_windows(const Tile& a, double* tile, double* col, double* cpar, int nv, int Fe,
                                                  bool pairwise, int64_t e0, bool mine, int z, int Z) {
  // 2a: element-wise pre-transform
  if (mine && (a.norm == MDG_NORM_LOG || a.norm == MDG_NORM_LOG_STANDARD)) {
    for (int s = z; s < nv; s += Z) {
      double x = col[s * a.sstride];
      if (a.norm == MDG_NORM_LOG) x = (x != x) ? x : (x < 1e-5 ? 1e-5 : x);  // log(max(x, 1e-5))
      col[s * a.sstride] = fast_log(x);
    }
  }
  if (a.norm == MDG_NORM_LOG_STANDARD) __syncthreads();
  // 2b: column statistics
  if (mine && z == 0) {
    double shift = 0., scale = 1.;
    switch (a.norm) {
      case MDG_NORM_LOOKBACK:      // x / x[-1]
      case MDG_NORM_LOOKBACK_LOG:  // log(x / x[-1])
        scale = 1. / col[(nv - 1) * a.sstride];
        break;
      case MDG_NORM_STANDARD: {  // nan_to_num((x - mean(0)) / std(0))
        shift = col_sum<0>(col, nv, a.sstride, 0., pairwise) / nv;
        scale = 1. / sqrt(col_sum<1>(col, nv, a.sstride, shift, pairwise) / nv);
        break;
      }
      case MDG_NORM_LOG_STANDARD: {  // x = log(x); nan_to_num((x - nanmean) / nanstd)
        int cnt = 0;
        for (int s = 0; s < nv; ++s) cnt += (col[s * a.sstride] == col[s * a.sstride]) ? 1 : 0;
        shift = col_sum<2>(col, nv, a.sstride, 0., pairwise) / cnt;
        scale = 1. / sqrt(col_sum<3>(col, nv, a.sstride, shift, pairwise) / cnt);
        break;
      }
      default:
        break;
    }
    cpar[0] = shift; cpar[1] = scale;
  }
  const bool scaled = a.norm == MDG_NORM_LOOKBACK || a.norm == MDG_NORM_LOOKBACK_LOG ||
                      a.norm == MDG_NORM_STANDARD || a.norm == MDG_NORM_LOG_STANDARD;
  if (scaled) {
    __syncthreads();
    // 2c: element-wise finish
    if (mine) {
      const double shift = cpar[0], scale = cpar[1];
      const bool zs = a.norm == MDG_NORM_STANDARD || a.norm == MDG_NORM_LOG_STANDARD;
      for (int s = z; s < nv; s += Z) {
        double x = col[s * a.sstride];
        if (zs) {
          // (x - mean) / sd with sd == 0: 0/0 -> nan -> 0, c/0 -> +-inf -> +-DBL_MAX, as np.nan_to_num
          const double d = x - shift;
          x = nan_to_num(d * scale);
        } else {
          x = x * scale;
          if (a.norm == MDG_NORM_LOOKBACK_LOG) x = fast_log(x);
        }
        col[s * a.sstride] = x;
      }
    }
  }
  if (a.norm == MDG_NORM_EXPANDING) {
    // x / _expanding_mean(x): the gufunc runs over the LAST axis (features), preprocessor.py:72-73,472-491
    const int tid = (threadIdx.z * blockDim.y + threadIdx.y) * blockDim.x + threadIdx.x;
    const int nthr = blockDim.x * blockDim.y * blockDim.z;
    for (int r = tid; r < a.envs * nv; r += nthr) {
      const int re = r / nv, rs = r - re * nv;
      if (e0 + re >= a.N) continue;
      double* row = tile + (int64_t)re * a.estride + (int64_t)rs * a.sstride;
      double acc = (row[0] == row[0]) ? row[0] : 0.;
      int w = 1;
      double prev = row[0];
      row[0] = prev / acc;
      for (int i = 1; i < Fe; ++i) {
        const double x = row[i];
        if (x == x) { acc = acc + x; w += 1; }
        row[i] = x / (acc / w);
      }
    }
  }
}

}  // namespace mdg
