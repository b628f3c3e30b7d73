// On-device episode tearsheet (reference: madigan/utils/metrics.py:83-171 test_summary, helpers :334-421).
// One thread per env; [rows][N] accumulators, coalesced.  See include/madigan_b200.h (MdgTearsheet) for the contract.
// Episode results (MdgEpisodeResults): the same recorder, harvested into an exact per-set table when an episode ends.
#include <math.h>
#include <stdio.h>

#include "mdg_common.cuh"

namespace mdg {

// ---------------------------------------------------------------------------------------------------------------
// The tearsheet arithmetic, shared by the tearsheet kernels and the episode-results kernel.
// Re-arm env e: empty accumulators, recording from the next update.
__device__ __forceinline__ void ts_rearm(const MdgTearsheet& t, int64_t e) {
  const int64_t N = t.n_envs;
  t.nsteps[e] = 0;
  t.active[e] = 1;
  t.sum_equity[e] = 0.; t.last_equity[e] = 0.; t.sum_reward[e] = 0.; t.sum_cost[e] = 0.;
  t.peak[e] = -INFINITY;
  t.min_valley[e] = INFINITY;
  for (int j = 0; j < t.n_assets; ++j) t.in_pos[(int64_t)j * N + e] = 0.;
  for (int j = 0; j < t.n_offsets; ++j) {
    t.ret_n[(int64_t)j * N + e] = 0;
    t.ret_mean[(int64_t)j * N + e] = 0.;
    t.ret_m2[(int64_t)j * N + e] = 0.;
    t.ret_down[(int64_t)j * N + e] = 0.;
  }
}

// Record the step env e has just taken (the env is active).
__device__ __forceinline__ void ts_update(const MdgTearsheet& t, const MdgState& S, const MdgStepIO& IO, int na,
                                          int64_t e) {
  const int64_t N = t.n_envs;
  const int J = t.n_offsets;
  // equity of the portfolio as the step left it: cash + assetValue - borrowedMargin from the folds the step kernel
  // keeps in state (Portfolio.cpp:211-213; bit-identical to the derived-accounting kernel's equity)
  const double eq = S.cash[e] + S.folds[0 * N + e] - S.folds[2 * N + e];
  const int64_t n = t.nsteps[e];  // steps recorded before this one
  t.sum_equity[e] += eq;
  t.last_equity[e] = eq;
  t.sum_reward[e] += IO.reward[e];
  double cost = 0.;
  for (int j = 0; j < na; ++j) {
    cost += IO.trans_cost[(int64_t)j * N + e];
    if (S.ledger[(int64_t)j * N + e] != 0.) t.in_pos[(int64_t)j * N + e] += 1.;  // metrics.py:119
  }
  t.sum_cost[e] += cost;
  const double pk = fmax(t.peak[e], eq);  // expanding max incl. the current point (metrics.py:419)
  t.peak[e] = pk;
  t.min_valley[e] = fmin(t.min_valley[e], eq / pk);
  // log returns at offsets 2^j (metrics.py:367-411 with unit timestamps: out[r] = log(arr[r] / arr[r - tf]), r >= tf)
  const int R = J > 0 ? (1 << (J - 1)) : 0;
  for (int j = 0; j < J; ++j) {
    const int64_t tf = (int64_t)1 << j;
    if (n >= tf) {
      const double prev = t.eq_ring[(int64_t)((n - tf) & (R - 1)) * N + e];
      const double r = log(eq / prev);
      if (r == r) {  // nanmean / nanstd skip NaN
        const int64_t o = (int64_t)j * N + e;
        const int c = t.ret_n[o] + 1;
        const double d = r - t.ret_mean[o];
        const double m = t.ret_mean[o] + d / c;
        t.ret_n[o] = c;
        t.ret_mean[o] = m;
        t.ret_m2[o] += d * (r - m);
        if (r < 0.) t.ret_down[o] += r * r;
      }
    }
  }
  if (R > 0) t.eq_ring[(int64_t)(n & (R - 1)) * N + e] = eq;
  t.nsteps[e] = n + 1;
}

// The tearsheet fields of env e, in output order: emit(field, value) for field 0 .. MDG_TS_NFIXED + 3J + nA - 1.
template <class Emit>
__device__ __forceinline__ void ts_summary(const MdgTearsheet& t, int64_t e, Emit&& emit) {
  const int64_t N = t.n_envs;
  const int na = t.n_assets, J = t.n_offsets;
  const int64_t n = t.nsteps[e];
  const double dn = (double)n;
  emit(0, dn);
  emit(1, t.sum_equity[e] / dn);
  emit(2, n ? t.last_equity[e] : NAN);
  emit(3, t.sum_reward[e] / dn);
  emit(4, n ? t.min_valley[e] : NAN);
  emit(5, t.sum_cost[e] / (dn * na));
  emit(6, t.sum_cost[e]);
  const int64_t max_tf = n ? (n - 1) / 10 : -1;  // (timestamps[-1] - timestamps[0]) // 10, metrics.py:108
  for (int j = 0; j < J; ++j) {
    const int64_t q = (int64_t)j * N + e;
    double mean = NAN, sharpe = NAN, sortino = NAN;
    if (((int64_t)1 << j) <= max_tf) {
      const int c = t.ret_n[q];
      mean = c ? t.ret_mean[q] : NAN;
      const double sd = sqrt(t.ret_m2[q] / (c - 1));  // np.nanstd(ddof=1)
      sharpe = (sd == 0.) ? 0. : mean / sd;           // metrics.py:345-348
      const double downside = t.ret_down[q] / (dn - 1);  // len(diff) counts the NaN head too, :359
      if (downside == 0.) sortino = (mean > 0.) ? 50. : 0.;  // :361-365
      else sortino = fmin(mean / downside, 50.);
    }
    emit(MDG_TS_NFIXED + 3 * j, mean);
    emit(MDG_TS_NFIXED + 3 * j + 1, sharpe);
    emit(MDG_TS_NFIXED + 3 * j + 2, sortino);
  }
  for (int i = 0; i < na; ++i) emit(MDG_TS_NFIXED + 3 * J + i, t.in_pos[(int64_t)i * N + e] / dn);
}

// ---------------------------------------------------------------------------------------------------------------
struct TsResetArgs {
  MdgTearsheet ts;
  const uint8_t* mask;
};

__global__ void __launch_bounds__(256) tearsheet_reset_kernel(const __grid_constant__ TsResetArgs a) {
  const MdgTearsheet& t = a.ts;
  const int64_t N = t.n_envs, e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (e >= N || (a.mask && !a.mask[e])) return;
  ts_rearm(t, e);
}

struct TsUpdateArgs {
  MdgTearsheet ts;
  MdgState S;
  MdgStepIO IO;
  int na;
};

__global__ void __launch_bounds__(256) tearsheet_update_kernel(const __grid_constant__ TsUpdateArgs a) {
  const MdgTearsheet& t = a.ts;
  const int64_t N = t.n_envs, e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (e >= N || !t.active[e]) return;
  ts_update(t, a.S, a.IO, a.na, e);
  if (a.IO.done && a.IO.done[e]) t.active[e] = 0;  // the step that reports done is the last one of the episode
}

struct TsSummaryArgs {
  MdgTearsheet ts;
  double* out;
};

__global__ void __launch_bounds__(256) tearsheet_summary_kernel(const __grid_constant__ TsSummaryArgs a) {
  const MdgTearsheet& t = a.ts;
  const int64_t N = t.n_envs, e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (e >= N) return;
  double* o = a.out + e;
  ts_summary(t, e, [&](int f, double v) { o[(int64_t)f * N] = v; });
}

// ---------------------------------------------------------------------------------------------------------------
// Episode results: the exact per-set table (include/madigan_b200.h, MdgEpisodeResults).
constexpr int kResDigits = 5;                     // base-2^30 digits of a quantised value, the top one signed
constexpr int kResFieldStride = 1 + 2 * kResDigits;  // count, sum digits, sum-of-squares digits
constexpr int kResHead = 2;                       // n_episodes, n_margin_call

// The five two's-complement base-2^30 digits of X = rint(v 2^64), |v| < 2^31 (so |X| < 2^126 for a square too).
// |X| is split with floor and exact power-of-two scalings: every remainder is a multiple of the ulp of the value it
// is taken from and no larger, so no step rounds.  A negative X is then negated in the digits: ~|X| + 1.
__device__ __forceinline__ void res_digits(double v, int32_t d[kResDigits]) {
  const double x = rint(v * 0x1p64);
  double r = fabs(x);
  const double d4 = floor(r * 0x1p-120); r -= d4 * 0x1p120;
  const double d3 = floor(r * 0x1p-90); r -= d3 * 0x1p90;
  const double d2 = floor(r * 0x1p-60); r -= d2 * 0x1p60;
  const double d1 = floor(r * 0x1p-30); r -= d1 * 0x1p30;
  d[0] = (int32_t)r; d[1] = (int32_t)d1; d[2] = (int32_t)d2; d[3] = (int32_t)d3; d[4] = (int32_t)d4;
  if (x < 0.) {
    int32_t carry = 1;
    for (int k = 0; k < kResDigits - 1; ++k) {
      const int32_t c = ((1 << 30) - 1 - d[k]) + carry;
      d[k] = c & ((1 << 30) - 1);
      carry = c >> 30;
    }
    d[kResDigits - 1] = ~d[kResDigits - 1] + carry;
  }
}

// order-preserving int64 image of an fp64 value (an involution: the same map decodes it)
__device__ __forceinline__ long long res_image(double v) {
  const long long b = __double_as_longlong(v);
  return b < 0 ? b ^ 0x7fffffffffffffffLL : b;
}

// Add value v of every lane of group `grp` (lanes of one set) into one field of the set's row: the lanes' digits are
// summed exactly in int64 registers at the group's lowest lane, which issues the atomics.
__device__ __forceinline__ void res_add(double v, unsigned grp, bool lead, unsigned long long* acc, long long* mn,
                                        long long* mx) {
  const bool ok = fabs(v) < 0x1p31;  // false for NaN and +-inf
  int32_t q[kResDigits] = {0, 0, 0, 0, 0}, s[kResDigits] = {0, 0, 0, 0, 0};
  if (ok) {
    res_digits(v, q);
    res_digits(v * v, s);
  }
  long long cnt = ok, lo = ok ? res_image(v) : 0x7fffffffffffffffLL, hi = ok ? res_image(v) : (-0x7fffffffffffffffLL - 1);
  long long Q[kResDigits], Sq[kResDigits];
  for (int k = 0; k < kResDigits; ++k) { Q[k] = q[k]; Sq[k] = s[k]; }
  for (unsigned m = grp & (grp - 1); m; m &= m - 1) {  // the group's other lanes, into every lane's registers
    const int src = __ffs(m) - 1;
    cnt += __shfl_sync(grp, (int)ok, src);
    for (int k = 0; k < kResDigits; ++k) {
      Q[k] += __shfl_sync(grp, q[k], src);
      Sq[k] += __shfl_sync(grp, s[k], src);
    }
    const long long l = __shfl_sync(grp, lo, src), h = __shfl_sync(grp, hi, src);
    lo = l < lo ? l : lo;
    hi = h > hi ? h : hi;
  }
  if (!lead || cnt == 0) return;
  atomicAdd(acc, (unsigned long long)cnt);
  for (int k = 0; k < kResDigits; ++k) {
    if (Q[k]) atomicAdd(acc + 1 + k, (unsigned long long)Q[k]);
    if (Sq[k]) atomicAdd(acc + 1 + kResDigits + k, (unsigned long long)Sq[k]);
  }
  atomicMin(mn, lo);
  atomicMax(mx, hi);
}

struct ResRecordArgs {
  MdgEpisodeResults r;
  MdgState S;
  MdgStepIO IO;
  const int32_t* set_of_env;  // nullptr: one set
  const double* broker;       // nullptr: every episode starts with init_cash
  double init_cash;
  int na;
};

// One thread per env: the tearsheet update; for an env whose step reported done, its tearsheet row (the money fields
// over the starting cash) into its set's row of the table, then the re-arm.
__global__ void __launch_bounds__(256) results_record_kernel(const __grid_constant__ ResRecordArgs a) {
  const MdgTearsheet& t = a.r.ts;
  const int64_t N = t.n_envs, e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  bool harvest = false;
  if (e < N && t.active[e]) {
    ts_update(t, a.S, a.IO, a.na, e);
    harvest = a.IO.done[e] != 0;
  }
  const unsigned D = __ballot_sync(0xffffffffu, harvest);
  if (!harvest) return;
  const int32_t S = a.r.n_sets, F = a.r.n_fields;
  int64_t set = 0;
  if (a.set_of_env) {
    const unsigned s = (unsigned)a.set_of_env[e], last = (unsigned)(S - 1);
    set = (int64_t)(s < last ? s : last);
  }
  const double cash = a.broker ? broker_value(a.broker, S, set, MDG_BROKER_INIT_CASH) : a.init_cash;
  const unsigned grp = __match_any_sync(D, (int)set);
  const bool lead = (int)(threadIdx.x & 31) == __ffs(grp) - 1;
  unsigned long long* row = reinterpret_cast<unsigned long long*>(a.r.acc) + set * (kResHead + kResFieldStride * F);
  long long* mn = reinterpret_cast<long long*>(a.r.ext) + set * F;
  long long* mx = mn + (int64_t)S * F;
  const unsigned mc = __ballot_sync(grp, a.IO.margin_call[e] != 0);
  if (lead) {
    atomicAdd(row, (unsigned long long)__popc(grp));
    if (mc) atomicAdd(row + 1, (unsigned long long)__popc(mc));
  }
  ts_summary(t, e, [&](int f, double v) {
    if (f == 1 || f == 2 || f == 5 || f == 6) v /= cash;  // mean / final equity, mean / total transaction cost
    res_add(v, grp, lead, row + kResHead + kResFieldStride * f, mn + f, mx + f);
  });
  ts_rearm(t, e);
}

static int check_ts(const MdgTearsheet* t) {
  if (!t) return set_err(MDG_E_INVALID, "null tearsheet");
  if (t->n_assets < 1 || t->n_assets > MDG_MAX_ASSETS) return set_err(MDG_E_INVALID, "tearsheet: bad n_assets");
  if (t->n_offsets < 0 || t->n_offsets > MDG_TS_MAX_OFFSETS) return set_err(MDG_E_INVALID, "tearsheet: bad n_offsets");
  if (!t->nsteps || !t->active || !t->sum_equity || !t->last_equity || !t->sum_reward || !t->peak || !t->min_valley ||
      !t->sum_cost || !t->in_pos)
    return set_err(MDG_E_INVALID, "tearsheet: null accumulator");
  if (t->n_offsets > 0 && (!t->eq_ring || !t->ret_n || !t->ret_mean || !t->ret_m2 || !t->ret_down))
    return set_err(MDG_E_INVALID, "tearsheet: null return accumulator");
  return MDG_OK;
}

int check_results(const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgParamSets* sets,
                  const MdgEpisodeResults* r) {
  if (!r) return set_err(MDG_E_INVALID, "null episode results");
  int rc = check_ts(&r->ts);
  if (rc) return rc;
  if (!P || !S || !IO) return set_err(MDG_E_INVALID, "null params/state/io");
  if (!S->cash || !S->folds || !S->ledger || !IO->reward || !IO->trans_cost || !IO->done || !IO->margin_call)
    return set_err(MDG_E_INVALID, "episode results: null state/io pointer");
  if (P->n_assets != r->ts.n_assets) return set_err(MDG_E_INVALID, "episode results: n_assets mismatch");
  if (!r->acc || !r->ext) return set_err(MDG_E_INVALID, "episode results: null table");
  if (r->n_fields != MDG_TS_NFIXED + 3 * r->ts.n_offsets + r->ts.n_assets)
    return set_err(MDG_E_INVALID, "episode results: n_fields is not MDG_TS_NFIXED + 3 n_offsets + n_assets");
  if (r->n_sets != (sets ? sets->n_sets : 1))
    return set_err(MDG_E_INVALID, "episode results: n_sets differs from the parameter sets (1 without)");
  if (r->ts.n_envs < 0) return set_err(MDG_E_INVALID, "n_envs < 0");
  return MDG_OK;
}

int launch_results_record(const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgParamSets* sets,
                          const double* broker, const MdgEpisodeResults* r, void* stream) {
  if (r->ts.n_envs == 0) return MDG_OK;
  ResRecordArgs a;
  a.r = *r; a.S = *S; a.IO = *IO;
  a.set_of_env = sets ? sets->set_of_env : nullptr;
  a.broker = sets ? broker : nullptr;
  a.init_cash = P->init_cash;
  a.na = P->n_assets;
  results_record_kernel<<<(unsigned)((r->ts.n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
  return cuda_err(cudaGetLastError(), "episode results record launch");
}

}  // namespace mdg

using namespace mdg;

extern "C" int mdg_tearsheet_reset(const MdgTearsheet* ts, const uint8_t* mask, void* stream) {
  int rc = check_ts(ts);
  if (rc) return rc;
  if (ts->n_envs <= 0) return ts->n_envs == 0 ? MDG_OK : set_err(MDG_E_INVALID, "n_envs < 0");
  TsResetArgs a;
  a.ts = *ts; a.mask = mask;
  tearsheet_reset_kernel<<<(unsigned)((ts->n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_tearsheet_reset launch");
}

extern "C" int mdg_tearsheet_update(const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgTearsheet* ts,
                                    void* stream) {
  int rc = check_ts(ts);
  if (rc) return rc;
  if (!P || !S || !IO) return set_err(MDG_E_INVALID, "null params/state/io");
  if (!S->cash || !S->folds || !S->ledger || !IO->reward || !IO->trans_cost)
    return set_err(MDG_E_INVALID, "tearsheet update: null state/io pointer");
  if (P->n_assets != ts->n_assets) return set_err(MDG_E_INVALID, "tearsheet: n_assets mismatch");
  if (ts->n_envs <= 0) return ts->n_envs == 0 ? MDG_OK : set_err(MDG_E_INVALID, "n_envs < 0");
  TsUpdateArgs a;
  a.ts = *ts; a.S = *S; a.IO = *IO; a.na = P->n_assets;
  tearsheet_update_kernel<<<(unsigned)((ts->n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_tearsheet_update launch");
}

extern "C" int mdg_tearsheet_summary(const MdgTearsheet* ts, double* out, void* stream) {
  int rc = check_ts(ts);
  if (rc) return rc;
  if (!out) return set_err(MDG_E_INVALID, "null out");
  if (ts->n_envs <= 0) return ts->n_envs == 0 ? MDG_OK : set_err(MDG_E_INVALID, "n_envs < 0");
  TsSummaryArgs a;
  a.ts = *ts; a.out = out;
  tearsheet_summary_kernel<<<(unsigned)((ts->n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_tearsheet_summary launch");
}

extern "C" int mdg_episode_results_record(const MdgParams* P, const MdgState* S, const MdgStepIO* IO,
                                          const MdgParamSets* sets, const double* broker,
                                          const MdgEpisodeResults* res, void* stream) {
  int rc = check_results(P, S, IO, sets, res);
  if (rc) return rc;
  if (sets && (rc = check_sets(P, sets))) return rc;
  if (!sets && broker) return set_err(MDG_E_INVALID, "episode results: a broker table needs parameter sets");
  return launch_results_record(P, S, IO, sets, broker, res, stream);
}
