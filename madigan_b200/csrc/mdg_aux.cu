// Kernels around the step path (sm_100a): Portfolio's derived accounting, the
// StackerDiscrete window materialiser with its normalisers, and per-slab episode
// statistics.  All HBM-bound streaming work; the window kernel stages one tile of
// the observation ring through shared memory to turn [slot][feat][env] rows into
// contiguous (env, k, feat) windows with coalesced traffic on both sides.
#include <float.h>
#include <math.h>
#include <stdio.h>

#include <stdlib.h>

#include <cuda.h>  // CUtensorMap and its enums (types only: the driver entry point is looked up at run time)

#include "mdg_common.cuh"
#include "mdg_window_norm.cuh"

namespace mdg {

constexpr int kBlockA = 128;

// ---------------------------------------------------------------------------
// derived accounting  (Portfolio.cpp:140-235, 243-252)
// ---------------------------------------------------------------------------
struct DerivedArgs {
  MdgParams P;
  MdgState S;
  MdgDerived D;
  int64_t N;
};
// ... with broker sets: the margins of every env from its set
struct DerivedBrokerArgs : DerivedArgs {
  MdgParamSets ps;
  const double* broker;
};

template <bool BROKER>
__device__ __forceinline__ void derived_body(const DerivedArgs& a, int64_t e) {
  const int64_t N = a.N;
  if (e >= N) return;
  const int na = a.P.n_assets;
  const MdgState& S = a.S;
  const MdgDerived& D = a.D;
  const double cash = S.cash[e];
  double av, ml, bms, se, um, bav;
  {
    const double l = S.ledger[e], p = S.price[e], m = S.mean_entry[e];
    const double mask = l < 0. ? 1. : 0.;
    av = l * p; ml = m * l; bms = S.borrowed[e]; se = l * (m * mask);
    um = fabs(l) * m; bav = l * (p * mask);
  }
  for (int j = 1; j < na; ++j) {
    const double l = S.ledger[(int64_t)j * N + e], p = S.price[(int64_t)j * N + e],
                 m = S.mean_entry[(int64_t)j * N + e];
    const double mask = l < 0. ? 1. : 0.;
    av = av + l * p; ml = ml + m * l; bms = bms + S.borrowed[(int64_t)j * N + e];
    se = se + l * (m * mask); um = um + fabs(l) * m; bav = bav + l * (p * mask);
  }
  const double equity = cash + av - bms;  // :211-213
  const double pnl = av - ml;             // :184-186
  const double balance = cash + se;       // :192-197
  if (D.equity) D.equity[e] = equity;
  if (D.asset_value) D.asset_value[e] = av;
  if (D.pnl) D.pnl[e] = pnl;
  if (D.balance) D.balance[e] = balance;
  double reqM = a.P.required_margin, maintM = a.P.maintenance_margin;
  if constexpr (BROKER) {
    const DerivedBrokerArgs& b = static_cast<const DerivedBrokerArgs&>(a);
    const int64_t set = env_set(b.ps, e);
    reqM = broker_value(b.broker, b.ps.n_sets, set, MDG_BROKER_REQUIRED_MARGIN);
    maintM = broker_value(b.broker, b.ps.n_sets, set, MDG_BROKER_MAINTENANCE_MARGIN);
  }
  if (D.available_margin) D.available_margin[e] = (balance + pnl) / reqM;  // :229-231
  if (D.used_margin) D.used_margin[e] = reqM * um;                          // :199-201
  if (D.borrowed_margin) D.borrowed_margin[e] = bms;
  if (D.borrowed_asset_value) D.borrowed_asset_value[e] = bav;  // :219-223
  if (D.risk) D.risk[e] = margin_call(cash, av, ml, bms, se, maintM) ? MDG_RISK_MARGIN_CALL : MDG_RISK_GREEN;
  const double w0 = (cash - bms) / equity;
  // abs-normalisers: sum |.| left to right (:144-148, :164-168)
  double sabs = 0., sabs_full = fabs(w0);
  for (int j = 0; j < na; ++j) {
    const double l = S.ledger[(int64_t)j * N + e], p = S.price[(int64_t)j * N + e];
    const double w = (l * p) / equity;
    sabs = (j == 0) ? fabs(w) : sabs + fabs(w);
    sabs_full = sabs_full + fabs(w);
  }
  if (D.ledger_normed_full) D.ledger_normed_full[e] = w0;
  if (D.ledger_abs_normed_full) D.ledger_abs_normed_full[e] = w0 / sabs_full;
  if (D.position_values_full) D.position_values_full[e] = cash - bms;
  if (D.ledger_full) D.ledger_full[e] = cash - bms;
  for (int j = 0; j < na; ++j) {
    const double l = S.ledger[(int64_t)j * N + e], p = S.price[(int64_t)j * N + e],
                 m = S.mean_entry[(int64_t)j * N + e];
    const double pv = l * p;
    const double w = pv / equity;
    if (D.position_values) D.position_values[(int64_t)j * N + e] = pv;          // :170-172
    if (D.pnl_positions) D.pnl_positions[(int64_t)j * N + e] = pv - m * l;      // :188-190
    if (D.ledger_normed) D.ledger_normed[(int64_t)j * N + e] = w;               // :140-142
    if (D.ledger_abs_normed) D.ledger_abs_normed[(int64_t)j * N + e] = w / sabs;
    if (D.ledger_normed_full) D.ledger_normed_full[(int64_t)(j + 1) * N + e] = w;  // :150-155
    if (D.ledger_abs_normed_full) D.ledger_abs_normed_full[(int64_t)(j + 1) * N + e] = w / sabs_full;
    if (D.position_values_full) D.position_values_full[(int64_t)(j + 1) * N + e] = pv;  // :174-178
    if (D.ledger_full) D.ledger_full[(int64_t)(j + 1) * N + e] = l;                      // :157-161
  }
}
__global__ void __launch_bounds__(kBlockA) derived_kernel(const __grid_constant__ DerivedArgs a) {
  derived_body<false>(a, (int64_t)blockIdx.x * kBlockA + threadIdx.x);
}
__global__ void __launch_bounds__(kBlockA) derived_broker_kernel(const __grid_constant__ DerivedBrokerArgs a) {
  derived_body<true>(a, (int64_t)blockIdx.x * kBlockA + threadIdx.x);
}

// ---------------------------------------------------------------------------
// window materialiser  (utils/preprocessor.py:183-189 current_data, :53-107 normalisers)
// ---------------------------------------------------------------------------
struct WindowArgs {
  const double* ring;        // [k][F][N]
  const double* prefix;      // [N][k][F] rows of the last reset's history fill, or nullptr
  const int64_t* timestamp;  // [N] (nullptr: every row comes from the ring)
  const int64_t* reset_ts;   // [N]
  void* out;
  int64_t N;
  int F, k, head, n_valid, norm, out_dtype, layout, flat_prefix;
  int xform, Feff, Fout;  // Feff: features the normaliser sees; Fout: features written
  int stride, age0;       // window row s = ring row of age age0 + (n_valid-1-s)*stride (MultiStackerDiscrete dilations)
  int Ftot, foff;         // out has Ftot features per row; this window fills columns [foff, foff + Fout)
  int envs;     // envs per block (blockDim.x)
  int sstride;  // smem stride between rows s (doubles)
  int estride;  // smem stride between envs   (doubles)
};

// blockDim = (envs, F): thread (x=e_local, y=f) owns one (env, feature) column.
__global__ void window_kernel(const __grid_constant__ WindowArgs a) {
  extern __shared__ double tile[];  // [envs][n_valid][F] with padded strides
  const int el = threadIdx.x, f = threadIdx.y;
  const int64_t e0 = (int64_t)blockIdx.x * a.envs;
  const int64_t e = e0 + el;
  const int nv = a.n_valid, F = a.F, k = a.k;
  const bool live = e < a.N;
  double* col = tile + (int64_t)el * a.estride + f;
  // phase 1: coalesced ring reads (consecutive envs), column into smem.  Rows older than the env's last
  // reset are not in the ring: they come from the env-major prefix buffer (prices) or are flat (portfolio).
  if (live) {
    long long since = 0x7fffffff;  // ring rows written since the last reset (the newest row always is one)
    if (a.timestamp) since = a.timestamp[e] - a.reset_ts[e] + 1;
    // 16 independent loads in flight per thread (a one-load-per-iteration loop made the kernel latency-bound:
    // 1.1 ms per 65,536 x 64 x 16 window, profiles/r1_notes.md)
    constexpr int U = 16;
    const int Z = blockDim.z, z = threadIdx.z;  // the column's rows are dealt round-robin to Z threads
    const int max_age = a.age0 + (nv - 1) * a.stride;
    const int isince = since > max_age + 1 ? max_age + 1 : (int)since;  // rows with age < isince come from the ring
    const double* rbase = a.ring + (int64_t)f * a.N + e;         // + slot * rstride
    const int64_t rstride = (int64_t)F * a.N;
    // prefix row of age `age`: k - 1 - (age - (since - 1)) = (k - 2 + since) - age
    const double* pbase = a.prefix ? a.prefix + ((int64_t)e * k + (k - 2 + isince)) * F + f : nullptr;
    const double flat = (f == 0) ? 1. : 0.;  // flat portfolio: ledgerNormedFull == [1, 0, ..., 0]
    for (int j0 = 0; z + Z * j0 < nv; j0 += U) {
      double v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int s = z + Z * (j0 + u);
        v[u] = 0.;
        if (s < nv) {
          const int age = a.age0 + (nv - 1 - s) * a.stride;
          int slot = a.head - age;  // age <= k - 1 (checked by the launcher): one wrap at most
          if (slot < 0) slot += k;
          if (age < isince) v[u] = rbase[slot * rstride];
          else if (pbase) v[u] = *(pbase - (int64_t)age * F);
          else v[u] = flat;
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int s = z + Z * (j0 + u);
        if (s < nv) col[s * a.sstride] = v[u];
      }
    }
  }
  __syncthreads();
  const int Fe = a.Feff;
  if (a.xform == MDG_XFORM_PAIR_RATIO) {  // price[:, 0] / price[:, 1]  (preprocessor.py:314-315)
    if (live && f == 0 && threadIdx.z == 0)
      for (int s = 0; s < nv; ++s) col[s * a.sstride] = col[s * a.sstride] / col[s * a.sstride + 1];
    __syncthreads();
  }

  // phase 2: normalise in place
  {
    const int Z = blockDim.z, z = threadIdx.z;
    double* cpar = tile + (int64_t)a.envs * a.estride + ((int64_t)el * F + f) * 2;  // (shift, scale) per column
    // a window written as a column block of a wider output is normalised as part of that (k, Ftot) array
    normalise_windows(a, tile, col, cpar, nv, Fe, Fe == 1 && a.Ftot == a.Fout, e0, live && f < Fe, z, Z);
  }
  __syncthreads();

  // phase 3: contiguous write-out of the block's windows
  const int tid = (threadIdx.z * blockDim.y + threadIdx.y) * blockDim.x + threadIdx.x;
  const int nthr = blockDim.x * blockDim.y * blockDim.z;
  const int Fo = a.Fout;
  const int per_env = nv * Fo;
  const int rows = (int)((a.N - e0) < a.envs ? (a.N - e0) : a.envs);
  const bool f32 = a.out_dtype == MDG_DTYPE_F32, diff = a.xform == MDG_XFORM_RETURNS;
  if (a.Ftot != Fo) {  // this window is a column block of a wider output (concatenation over dilations)
    const int Ft = a.Ftot;
    for (int re = 0; re < rows; ++re) {
      for (int r = tid; r < per_env; r += nthr) {
        const int sr = r / Fo, ff = r - sr * Fo;
        const double* q = tile + (int64_t)re * a.estride + (int64_t)sr * a.sstride + ff;
        const double v = diff ? q[1] - q[0] : q[0];
        const int64_t o = (a.layout == MDG_LAYOUT_NKF) ? ((e0 + re) * nv + sr) * Ft + a.foff + ff
                                                        : ((e0 + re) * Ft + a.foff + ff) * nv + sr;
        if (f32) ((float*)a.out)[o] = (float)v; else ((double*)a.out)[o] = v;
      }
    }
  } else if (a.layout == MDG_LAYOUT_NKF && nthr % Fo == 0) {
    // thread -> fixed feature, rows advance by nthr / Fo: consecutive threads write consecutive elements and no
    // index needs a division (a 64-bit div/mod per element made this phase instruction-bound)
    const int ff = tid % Fo, sstep = nthr / Fo;
    for (int re = 0; re < rows; ++re) {
      const double* tp = tile + (int64_t)re * a.estride + ff;
      const int64_t o0 = (e0 + re) * per_env + ff;
      for (int sr = tid / Fo; sr < nv; sr += sstep) {
        const double* q = tp + sr * a.sstride;
        const double v = diff ? q[1] - q[0] : q[0];  // np.diff(price): last axis (:330)
        if (f32) ((float*)a.out)[o0 + sr * Fo] = (float)v; else ((double*)a.out)[o0 + sr * Fo] = v;
      }
    }
  } else {
    for (int re = 0; re < rows; ++re) {
      for (int r = tid; r < per_env; r += nthr) {
        int sr, ff;
        if (a.layout == MDG_LAYOUT_NKF) { sr = r / Fo; ff = r - sr * Fo; } else { ff = r / nv; sr = r - ff * nv; }
        const double* q = tile + (int64_t)re * a.estride + (int64_t)sr * a.sstride + ff;
        const double v = diff ? q[1] - q[0] : q[0];
        const int64_t o = (e0 + re) * per_env + r;
        if (f32) ((float*)a.out)[o] = (float)v; else ((double*)a.out)[o] = v;
      }
    }
  }
}

// ---------------------------------------------------------------------------
// window materialiser, TMA variant (sm_90+/sm_100a): the common case -- StackerDiscrete's price window, (N, k, F)
// layout, every normaliser but `expanding` -- as a tile-movement kernel.
//
//   load   the ring is a 2-D tensor [k*F rows][N envs] of fp64; a tile is 8 consecutive envs.  One elected thread
//          issues one `cp.async.bulk.tensor.2d` per window row-group (box = F rows x 8 envs = F x 64 bytes) against an
//          mbarrier: the whole tile (64 KB at 64 x 16) is in flight at once with no registers and no issue slots
//          spent on it, and lands as T[row = s*F + f][env] in LOGICAL time order (the ring wrap is resolved by the
//          box coordinates).
//   patch  rows older than an env's last reset are replaced from the env-major prefix buffer (contiguous per env).
//   math   one thread per (env, feature, half-column): lane = env fastest, so the column reads are at most 2-way
//          bank-conflicted without padding or swizzle.
//   store  fp32: the block's windows are staged as O[env][k*F] (env stride + 16 bytes: conflict-free) and written
//          with one `cp.async.bulk.global.shared::cta` per env (4 KB contiguous); fp64: 32-byte pieces, direct.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// tile = E consecutive envs x FT consecutive features (a.envs, a.sstride carry E and FT; blockIdx.x = env tile * nq +
// feature group, so that the feature groups of one env tile run together and their partial lines merge in L2)
__global__ void window_tma_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ WindowArgs a) {
  extern __shared__ __align__(128) unsigned char wsm[];
  const int nv = a.n_valid, F = a.F, k = a.k, E = a.envs, FT = a.sstride;
  const int nq = F / FT;
  const int f0 = (int)(blockIdx.x % nq) * FT;
  const int64_t e0 = (int64_t)(blockIdx.x / nq) * E;
  const int rows = nv * FT;
  double* T = reinterpret_cast<double*>(wsm);                                   // [rows][E]
  unsigned char* O = wsm + (size_t)rows * E * sizeof(double);                  // [E][ostride] (fp32 staging)
  const int ostride = a.estride;                                                // bytes per env in O (0: no staging)
  double* cpar = reinterpret_cast<double*>(O + (size_t)E * ostride);            // [E*FT][2] (shift, scale)
  int* s_since = reinterpret_cast<int*>(cpar + E * FT * 2);                     // [E]
  uint64_t* mbar = reinterpret_cast<uint64_t*>(s_since + E);                    // 8-byte aligned by construction
  const int tid = threadIdx.x, nthr = blockDim.x;
  int slot0 = (a.head - (nv - 1)) % k;
  if (slot0 < 0) slot0 += k;

  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mbar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)),
                 "r"((uint32_t)(rows * E * sizeof(double)))
                 : "memory");
    const uint64_t desc = reinterpret_cast<uint64_t>(&tmap);
    for (int s = 0; s < nv; ++s) {
      int slot = slot0 + s;
      if (slot >= k) slot -= k;
      asm volatile(
          "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
              "r"(smem_u32(T + (size_t)s * FT * E)),
          "l"(desc), "r"(smem_u32(mbar)), "r"((int)e0), "r"(slot * F + f0)
          : "memory");
    }
  }
  // rows written to the ring since each env's last reset (the newest row always is one)
  if (tid < E) {
    long long since = 0x7fffffff;
    const int64_t e = e0 + tid;
    if (a.timestamp && e < a.N) since = a.timestamp[e] - a.reset_ts[e] + 1;
    s_since[tid] = since > nv ? nv : (int)since;
  }
  {  // wait for the tile (phase 0); a tile that never lands is a bug, not a hang
    uint32_t done = 0;
    for (unsigned spin = 0; !done; ++spin) {
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(done)
          : "r"(smem_u32(mbar))
          : "memory");
      if (spin > (1u << 24)) __trap();
    }
  }
  __syncthreads();  // s_since visible
  // patch: window rows s < nv - since of env e come from the prefix buffer (contiguous there) or are flat.
  // Per patched env, every thread keeps up to four independent loads in flight (the run is contiguous in the prefix
  // buffer when the tile holds all features).
#pragma unroll 1
  for (int el = 0; el < E; ++el) {
    const int isince = s_since[el];
    const int64_t e = e0 + el;
    if (isince >= nv || e >= a.N) continue;
    const int cnt = (nv - isince) * FT;
    const double* pb = a.prefix ? a.prefix + ((int64_t)e * k + (k - 1 + isince - nv)) * F + f0 : nullptr;
    constexpr int U = 4;
    for (int r0 = tid; r0 < cnt; r0 += nthr * U) {
      double v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int r = r0 + u * nthr;
        v[u] = 0.;
        if (r < cnt) {
          if (FT == F) {
            v[u] = pb ? pb[r] : ((r % F == 0) ? 1. : 0.);
          } else {
            const int s = r / FT, f_ = r - s * FT;
            v[u] = pb ? pb[s * F + f_] : ((f0 + f_ == 0) ? 1. : 0.);  // flat portfolio: ledgerNormedFull == [1, 0, ..., 0]
          }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int r = r0 + u * nthr;
        if (r < cnt) T[(size_t)r * E + el] = v[u];
      }
    }
  }
  __syncthreads();

  // math: thread (e, f, z), env fastest; column = T + f*E + e, stride between samples FT*E
  const int el = tid & (E - 1), f = (tid / E) % FT, z = tid / (E * FT), Z = nthr / (E * FT);
  const int SS = FT * E;
  double* col = T + f * E + el;
  const bool live = (e0 + el) < a.N;
  if (live && (a.norm == MDG_NORM_LOG || a.norm == MDG_NORM_LOG_STANDARD)) {
    for (int s = z; s < nv; s += Z) {
      double x = col[s * SS];
      if (a.norm == MDG_NORM_LOG) x = (x != x) ? x : (x < 1e-5 ? 1e-5 : x);  // log(max(x, 1e-5))
      col[s * SS] = fast_log(x);
    }
  }
  if (a.norm == MDG_NORM_LOG_STANDARD) __syncthreads();
  double* cp = cpar + (el * FT + f) * 2;
  if (live && z == 0) {
    double shift = 0., scale = 1.;
    const bool pw = (F == 1);
    switch (a.norm) {
      case MDG_NORM_LOOKBACK:
      case MDG_NORM_LOOKBACK_LOG:
        scale = 1. / col[(nv - 1) * SS];
        break;
      case MDG_NORM_STANDARD:
        shift = col_sum<0>(col, nv, SS, 0., pw) / nv;
        scale = 1. / sqrt(col_sum<1>(col, nv, SS, shift, pw) / nv);
        break;
      case MDG_NORM_LOG_STANDARD: {
        int cnt = 0;
        for (int s = 0; s < nv; ++s) cnt += (col[s * SS] == col[s * SS]) ? 1 : 0;
        shift = col_sum<2>(col, nv, SS, 0., pw) / cnt;
        scale = 1. / sqrt(col_sum<3>(col, nv, SS, shift, pw) / cnt);
        break;
      }
      default:
        break;
    }
    cp[0] = shift; cp[1] = scale;
  }
  __syncthreads();
  const bool scaled = a.norm == MDG_NORM_LOOKBACK || a.norm == MDG_NORM_LOOKBACK_LOG ||
                      a.norm == MDG_NORM_STANDARD || a.norm == MDG_NORM_LOG_STANDARD;
  const bool zs = a.norm == MDG_NORM_STANDARD || a.norm == MDG_NORM_LOG_STANDARD;
  const bool f32 = a.out_dtype == MDG_DTYPE_F32;
  if (live) {
    const double shift = cp[0], scale = cp[1];
    float* orow = reinterpret_cast<float*>(O + (size_t)el * ostride);
    for (int s = z; s < nv; s += Z) {
      double x = col[s * SS];
      if (scaled) {
        if (zs) {
          x = nan_to_num((x - shift) * scale);
        } else {
          x = x * scale;
          if (a.norm == MDG_NORM_LOOKBACK_LOG) x = fast_log(x);
        }
      }
      if (f32) orow[s * FT + f] = (float)x; else col[s * SS] = x;
    }
  }
  if (f32 && FT == F) {  // whole windows: one bulk store per env
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic writes of O -> visible to the bulk copy
    __syncthreads();
    if (tid < E && (e0 + tid) < a.N) {
      const uint32_t bytes = (uint32_t)(rows * sizeof(float));
      float* dst = reinterpret_cast<float*>(a.out) + (e0 + tid) * rows;
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst),
                   "r"(smem_u32(O + (size_t)tid * ostride)), "r"(bytes)
                   : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // shared memory may go away after this
    }
  } else if (f32) {  // a feature group: FT consecutive fp32 per (env, sample), linear reads of O
    __syncthreads();
    float* out = reinterpret_cast<float*>(a.out);
    for (int el_ = 0; el_ < E; ++el_) {
      if (e0 + el_ >= a.N) break;
      const float* orow = reinterpret_cast<const float*>(O + (size_t)el_ * ostride);
      float* dst = out + (e0 + el_) * (int64_t)nv * F + f0;
      for (int r = tid; r < rows; r += nthr) {
        const int s = r / FT, f_ = r - s * FT;
        dst[s * F + f_] = orow[r];
      }
    }
  } else {
    __syncthreads();
    double* out = reinterpret_cast<double*>(a.out);
    const int per = 32 / E > 0 ? 32 / E : 1;  // consecutive elements of one env handled by one warp
    (void)per;
    for (int idx = tid; idx < rows * E; idx += nthr) {  // lanes: env fastest
      const int e_ = idx & (E - 1), r = idx / E;
      const int s = r / FT, f_ = r - s * FT;
      if (e0 + e_ < a.N) out[((e0 + e_) * (int64_t)nv + s) * F + f0 + f_] = T[(size_t)r * E + e_];
    }
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
  static const EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

// launch the TMA variant when the case qualifies; returns 1 when it did, 0 when the caller should fall back, <0 on error
static int launch_window_tma(const MdgWindow* w, WindowArgs a) {
  // OPT-IN (MDG_WIN_TMA=1): measured on B200 at 65,536 x 64 x 16 -> fp32 the TMA tile kernel takes 423 us (None) /
  // 512 us (standard_normal) against 232 / 351 us for the register-staged kernel below (profiles/r2_notes.md): the
  // ring is env-minor, so a tile of 8 envs is 1,024 rows of 64 bytes for the TMA engine, and 18 % of the envs need
  // their pre-reset rows patched in afterwards.  Parity-tested either way (tests/test_gpu_window.py).
  const char* en = getenv("MDG_WIN_TMA");  // read per call: the parity tests switch it on and off in one process
  const int enabled = en ? atoi(en) : 0;
  if (!enabled) return 0;
  const char* vE = getenv("MDG_WIN_TMA_E");
  const char* vF = getenv("MDG_WIN_TMA_FT");
  const int env_E = vE ? atoi(vE) : 8, env_FT = vF ? atoi(vF) : 16;
  if (!enabled) return 0;
  const int F = a.F, nv = a.n_valid;
  if (a.xform != MDG_XFORM_NONE || a.layout != MDG_LAYOUT_NKF || a.norm == MDG_NORM_EXPANDING) return 0;
  if (a.stride != 1 || a.age0 != 0 || a.Ftot != a.Fout) return 0;
  int E = env_E, FT = env_FT;
  if (E != 8 && E != 16 && E != 32) return 0;
  if (FT > F) FT = F;
  if (F % FT) return 0;
  if ((a.N & 1) || a.N < E || (reinterpret_cast<uintptr_t>(a.ring) & 15)) return 0;
  if (((size_t)FT * E * sizeof(double)) % 128) return 0;  // every box lands on a 128-byte boundary
  const bool f32 = a.out_dtype == MDG_DTYPE_F32;
  const size_t rows = (size_t)nv * FT;
  if (f32 && FT == F && (((rows * sizeof(float)) & 15) || (reinterpret_cast<uintptr_t>(a.out) & 15))) return 0;
  const int ostride = f32 ? (int)(rows * sizeof(float) + 16) : 0;
  const size_t smem = rows * E * sizeof(double) + (size_t)E * ostride + (size_t)E * FT * 2 * sizeof(double) +
                      E * sizeof(int) + 16;
  if (smem > 110 * 1024) return 0;
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) return 0;
  CUtensorMap tmap;
  const cuuint64_t gdim[2] = {(cuuint64_t)a.N, (cuuint64_t)a.k * (cuuint64_t)F};
  const cuuint64_t gstride[1] = {(cuuint64_t)a.N * sizeof(double)};
  const cuuint32_t box[2] = {(cuuint32_t)E, (cuuint32_t)FT};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult cr = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(a.ring), gdim, gstride, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) return 0;
  static size_t smem_allowed = 48 * 1024;
  if (smem > smem_allowed) {
    cudaError_t ce = cudaFuncSetAttribute(window_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return cuda_err(ce, "window (tma) smem attr");
    smem_allowed = smem;
  }
  a.estride = ostride;
  a.envs = E;
  a.sstride = FT;
  int Z = 256 / (E * FT);
  if (Z < 1) Z = 1;
  const unsigned grid = (unsigned)(((a.N + E - 1) / E) * (F / FT));
  window_tma_kernel<<<grid, E * FT * Z, smem, (cudaStream_t)w->stream>>>(tmap, a);
  const int rc = cuda_err(cudaGetLastError(), "mdg_materialise_window (tma) launch");
  return rc ? rc : 1;
}

__global__ void time_kernel(const int64_t* timestamp, int64_t N, int nv, int64_t* out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * nv) return;
  const int64_t e = idx / nv;
  const int s = (int)(idx - e * nv);
  out[idx] = timestamp[e] - (nv - 1 - s);  // every window row is exactly one generator tick
}

// ---------------------------------------------------------------------------
// episode statistics: one vector per slab, all-reduced across GPUs by the host (NCCL)
// ---------------------------------------------------------------------------
__device__ __forceinline__ void atomic_min_double(double* addr, double v) {
  unsigned long long* a = (unsigned long long*)addr;
  unsigned long long old = *a, assumed;
  do {
    assumed = old;
    if (!(v < __longlong_as_double((long long)assumed))) break;
    old = atomicCAS(a, assumed, (unsigned long long)__double_as_longlong(v));
  } while (assumed != old);
}
__device__ __forceinline__ void atomic_max_double(double* addr, double v) {
  unsigned long long* a = (unsigned long long*)addr;
  unsigned long long old = *a, assumed;
  do {
    assumed = old;
    if (!(v > __longlong_as_double((long long)assumed))) break;
    old = atomicCAS(a, assumed, (unsigned long long)__double_as_longlong(v));
  } while (assumed != old);
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

struct StatsArgs {
  MdgParams P;
  MdgState S;
  MdgStepIO IO;
  int64_t N;
  double* out;
};

__global__ void stats_init_kernel(double* out, int n) {
  const int i = threadIdx.x;
  if (i < n) out[i] = (i == 3) ? INFINITY : (i == 4 ? -INFINITY : 0.);
}

// grid-stride, per-thread partials -> warp shuffles -> one atomic per warp per statistic
__global__ void __launch_bounds__(256) stats_kernel(const __grid_constant__ StatsArgs a) {
  const int64_t N = a.N;
  const int na = a.P.n_assets;
  double cnt = 0., seq = 0., ssq = 0., mn = INFINITY, mx = -INFINITY, srew = 0., scost = 0., ndone = 0.;
  double expo[MDG_MAX_ASSETS], held[MDG_MAX_ASSETS];
#pragma unroll
  for (int j = 0; j < MDG_MAX_ASSETS; ++j) { expo[j] = 0.; held[j] = 0.; }
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < N; e += (int64_t)gridDim.x * blockDim.x) {
    double av = 0., bms = 0.;
    for (int j = 0; j < na; ++j) {
      av = av + a.S.ledger[(int64_t)j * N + e] * a.S.price[(int64_t)j * N + e];
      bms = bms + a.S.borrowed[(int64_t)j * N + e];
    }
    const double eq = a.S.cash[e] + av - bms;
    cnt += 1.; seq += eq; ssq += eq * eq; mn = fmin(mn, eq); mx = fmax(mx, eq);
    if (a.IO.reward) srew += a.IO.reward[e];
    if (a.IO.done) ndone += a.IO.done[e] ? 1. : 0.;
#pragma unroll
    for (int j = 0; j < MDG_MAX_ASSETS; ++j) {
      if (j < na) {
        const double l = a.S.ledger[(int64_t)j * N + e];
        if (a.IO.trans_cost) scost += a.IO.trans_cost[(int64_t)j * N + e];
        expo[j] += fabs(l * a.S.price[(int64_t)j * N + e]) / eq;
        held[j] += (l != 0.) ? 1. : 0.;
      }
    }
  }
  const bool lead = (threadIdx.x & 31) == 0;
  cnt = warp_sum(cnt); seq = warp_sum(seq); ssq = warp_sum(ssq); srew = warp_sum(srew);
  scost = warp_sum(scost); ndone = warp_sum(ndone); mn = warp_min(mn); mx = warp_max(mx);
  if (lead) {
    atomicAdd(&a.out[0], cnt); atomicAdd(&a.out[1], seq); atomicAdd(&a.out[2], ssq);
    atomic_min_double(&a.out[3], mn); atomic_max_double(&a.out[4], mx);
    atomicAdd(&a.out[5], srew); atomicAdd(&a.out[6], scost); atomicAdd(&a.out[7], ndone);
  }
#pragma unroll
  for (int j = 0; j < MDG_MAX_ASSETS; ++j) {
    if (j < na) {
      const double x = warp_sum(expo[j]), h = warp_sum(held[j]);
      if (lead) {
        atomicAdd(&a.out[MDG_STATS_NSCALAR + j], x);
        atomicAdd(&a.out[MDG_STATS_NSCALAR + na + j], h);
      }
    }
  }
}

}  // namespace mdg

using namespace mdg;

extern "C" int mdg_derived(const MdgParams* P, const MdgState* S, const MdgDerived* D, const MdgLaunch* L) {
  if (!P || !S || !D || !L) return set_err(MDG_E_INVALID, "null argument");
  if (P->n_assets < 1 || P->n_assets > MDG_MAX_ASSETS) return set_err(MDG_E_UNSUPPORTED, "n_assets out of range");
  if (L->n_envs <= 0) return L->n_envs == 0 ? MDG_OK : set_err(MDG_E_INVALID, "n_envs < 0");
  DerivedArgs a;
  a.P = *P; a.S = *S; a.D = *D; a.N = L->n_envs;
  const unsigned grid = (unsigned)((a.N + kBlockA - 1) / kBlockA);
  derived_kernel<<<grid, kBlockA, 0, (cudaStream_t)L->stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_derived launch");
}

extern "C" int mdg_derived_sets_broker(const MdgParams* P, const MdgState* S, const MdgDerived* D, const MdgLaunch* L,
                                       const MdgParamSets* sets, const double* broker) {
  if (!P || !S || !D || !L) return set_err(MDG_E_INVALID, "null argument");
  if (P->n_assets < 1 || P->n_assets > MDG_MAX_ASSETS) return set_err(MDG_E_UNSUPPORTED, "n_assets out of range");
  const int rc = check_sets(P, sets);
  if (rc) return rc;
  if (!broker) return mdg_derived(P, S, D, L);
  if (L->n_envs <= 0) return L->n_envs == 0 ? MDG_OK : set_err(MDG_E_INVALID, "n_envs < 0");
  DerivedBrokerArgs a;
  a.P = *P; a.S = *S; a.D = *D; a.N = L->n_envs;
  a.ps = *sets;
  a.broker = broker;
  const unsigned grid = (unsigned)((a.N + kBlockA - 1) / kBlockA);
  derived_broker_kernel<<<grid, kBlockA, 0, (cudaStream_t)L->stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_derived launch");
}

extern "C" int mdg_materialise_window(const MdgWindow* w) {
  if (!w || !w->ring || !w->out) return set_err(MDG_E_INVALID, "null window/ring/out");
  const int n_feats = w->n_feats, window = w->window, head = w->head, n_valid = w->n_valid;
  if (n_feats < 1 || n_feats > 64) return set_err(MDG_E_UNSUPPORTED, "n_feats must be in 1..64");
  if (window < 1 || head < 0 || head >= window || n_valid < 1 || n_valid > window)
    return set_err(MDG_E_INVALID, "bad window/head/n_valid");
  if (w->norm_type < MDG_NORM_NONE || w->norm_type > MDG_NORM_EXPANDING) return set_err(MDG_E_INVALID, "bad norm_type");
  if (w->out_dtype != MDG_DTYPE_F64 && w->out_dtype != MDG_DTYPE_F32) return set_err(MDG_E_INVALID, "bad out_dtype");
  if (w->out_layout != MDG_LAYOUT_NKF && w->out_layout != MDG_LAYOUT_NFK) return set_err(MDG_E_INVALID, "bad layout");
  if (w->timestamp && !w->reset_ts) return set_err(MDG_E_INVALID, "timestamp given without reset_ts");
  if (w->timestamp && !w->prefix && !w->flat_prefix) return set_err(MDG_E_INVALID, "no prefix source for rows older than the reset");
  if (w->transform < MDG_XFORM_NONE || w->transform > MDG_XFORM_RETURNS) return set_err(MDG_E_INVALID, "bad transform");
  if (w->transform == MDG_XFORM_PAIR_RATIO && n_feats != 2)
    return set_err(MDG_E_INVALID, "the pair-ratio window needs exactly 2 features");  // preprocessor.py:301 assert
  if (w->n_envs <= 0) return w->n_envs == 0 ? MDG_OK : set_err(MDG_E_INVALID, "n_envs < 0");
  if (w->transform == MDG_XFORM_RETURNS && n_feats == 1) return MDG_OK;  // np.diff of one feature: (k, 0), nothing to write
  WindowArgs a;
  a.xform = w->transform;
  a.Feff = (w->transform == MDG_XFORM_PAIR_RATIO) ? 1 : n_feats;
  a.Fout = (w->transform == MDG_XFORM_PAIR_RATIO) ? 1 : (w->transform == MDG_XFORM_RETURNS ? n_feats - 1 : n_feats);
  a.ring = w->ring; a.prefix = w->prefix; a.timestamp = w->timestamp; a.reset_ts = w->reset_ts;
  a.out = w->out; a.N = w->n_envs; a.F = n_feats; a.k = window; a.head = head; a.n_valid = n_valid;
  a.norm = w->norm_type; a.out_dtype = w->out_dtype; a.layout = w->out_layout; a.flat_prefix = w->flat_prefix;
  a.stride = w->stride > 1 ? w->stride : 1;
  a.age0 = w->age0 > 0 ? w->age0 : 0;
  if (a.age0 + (int64_t)(n_valid - 1) * a.stride >= window)
    return set_err(MDG_E_INVALID, "dilated window reaches beyond the ring (need window >= age0 + (n_valid-1)*stride + 1)");
  a.Ftot = w->out_feats_total > 0 ? w->out_feats_total : a.Fout;
  a.foff = w->out_feats_total > 0 ? w->out_feat_offset : 0;
  if (a.foff < 0 || a.foff + a.Fout > a.Ftot) return set_err(MDG_E_INVALID, "bad out_feat_offset / out_feats_total");
  {
    const int t = launch_window_tma(w, a);
    if (t != 0) return t < 0 ? t : MDG_OK;
  }
  // envs per block: a power of two with about 64 columns per block and two threads per column -- small tiles
  // (35 KB at 64 x 16), six blocks per SM: measured best at 65,536 x 64 x 16 (profiles/window_cost.py)
  int envs = 32;
  while (envs > 1 && envs * n_feats > 64) envs >>= 1;
  static const int env_override = [] { const char* v = getenv("MDG_WIN_ENVS"); return v ? atoi(v) : 0; }();
  static const int z_override = [] { const char* v = getenv("MDG_WIN_Z"); return v ? atoi(v) : 0; }();
  if (env_override) envs = env_override;
  a.sstride = n_feats + 1;  // odd-ish row stride: conflict-free (N,F,k) reads
  for (;;) {
    int es = n_valid * a.sstride;
    es += ((2 - es) % 16 + 16) % 16;  // env stride == 2 (mod 16 doubles): conflict-free column writes
    a.estride = es;
    if (((size_t)envs * es + (size_t)envs * n_feats * 2) * sizeof(double) <= 96 * 1024 || envs == 1) break;
    envs >>= 1;
  }
  a.envs = envs;
  const size_t smem = ((size_t)envs * a.estride + (size_t)envs * n_feats * 2) * sizeof(double);
  if (smem > 200 * 1024) return set_err(MDG_E_UNSUPPORTED, "window tile does not fit shared memory");
  static size_t smem_allowed = 48 * 1024;  // raise the opt-in limit only when a larger tile is first needed
  if (smem > smem_allowed) {
    cudaError_t ce = cudaFuncSetAttribute(window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return cuda_err(ce, "window smem attr");
    smem_allowed = smem;
  }
  const unsigned grid = (unsigned)((w->n_envs + envs - 1) / envs);
  int zdim = 2;  // threads per column for the data-movement and element-wise phases
  if (z_override) zdim = z_override;
  window_kernel<<<grid, dim3(envs, n_feats, zdim), smem, (cudaStream_t)w->stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_materialise_window launch");
}

extern "C" int mdg_materialise_time(const int64_t* timestamp, int64_t n_envs, int32_t n_valid, int64_t* out,
                                    void* stream) {
  if (!timestamp || !out) return set_err(MDG_E_INVALID, "null timestamp/out");
  if (n_valid < 1) return set_err(MDG_E_INVALID, "bad n_valid");
  if (n_envs <= 0) return n_envs == 0 ? MDG_OK : set_err(MDG_E_INVALID, "n_envs < 0");
  const int64_t total = n_envs * n_valid;
  time_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(timestamp, n_envs, n_valid, out);
  return cuda_err(cudaGetLastError(), "mdg_materialise_time launch");
}

extern "C" int mdg_episode_stats(const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgLaunch* L,
                                 double* out) {
  if (!P || !S || !L || !out) return set_err(MDG_E_INVALID, "null argument");
  if (P->n_assets < 1 || P->n_assets > MDG_MAX_ASSETS) return set_err(MDG_E_UNSUPPORTED, "n_assets out of range");
  StatsArgs a;
  a.P = *P; a.S = *S;
  if (IO) a.IO = *IO; else memset(&a.IO, 0, sizeof(a.IO));
  a.N = L->n_envs; a.out = out;
  cudaStream_t st = (cudaStream_t)L->stream;
  stats_init_kernel<<<1, 64, 0, st>>>(out, MDG_STATS_NSCALAR + 2 * P->n_assets);
  if (a.N > 0) {
    int grid = (int)((a.N + 255) / 256);
    if (grid > 148 * 4) grid = 148 * 4;  // a few resident CTAs per SM, grid-stride over the slab
    stats_kernel<<<grid, 256, 0, st>>>(a);
  }
  return cuda_err(cudaGetLastError(), "mdg_episode_stats launch");
}
