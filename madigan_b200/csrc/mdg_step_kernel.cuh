// Fused Env.step / Env.reset kernels for N independent environments (sm_100a).
//
// One thread per env STREAMS over its assets in a rolled loop: state tensors are
// [rows][N], so every load/store is one coalesced 256-byte run per warp, each value is
// read once, and the kernel is a few thousand instructions (an earlier fully unrolled,
// register-resident version was I-cache bound, profiles/r1_notes.md).  One launch does what the
// reference does across Env.h:189-256, Broker.cpp:124-178, Portfolio.cpp:140-323,
// the DataSource.cpp getData family, offpolicy_q.py:140-164 and nstep_buffer.py:
//   transact (sequential over assets, risk-gated) -> generator tick -> equity,
//   reward, done -> newest observation-ring row -> agent reward -> shaped reward.
// HBM-bound integer/fp64 work: no tensor cores.
#pragma once
#include <cuda.h>
#include <math.h>
#include <stdio.h>

#include "mdg_common.cuh"

namespace mdg {

struct StepArgs {
  MdgParams P;
  MdgReward R;
  MdgState S;
  MdgStepIO IO;
  MdgLaunch L;
  int units_v2;     // set by launch_step: the units matrix can be read with 16-byte loads (aligned base, even nA)
  // constants of the risk gates, filled by launch_step: as kernel parameters they are constant-bank operands of the
  // instructions that use them instead of ten live registers per thread (the one-wave variant spills at 128)
  double c_reqM, c_maintM, c_band_scale, c_g1, c_g2;
  int c_reqM_ok, c_force_exact;
  int bulk;  // set by launch_step: the pairs' state rows reach the block through cp.async.bulk + mbarrier (see step_body)
  int* done_count;  // nullable (auto-reset): number of envs that finished this step ...
  int* done_list;   // ... and their indices, appended warp by warp in the kernel's tail
  // bulk == 2: tensor maps of the state slab (N x nA x {price, ledger, mean entry, borrowed}) and of the caller's units
  // matrix (nA x N), filled by launch_step; tma_units: the units come through the ring too
  int tma_units;
  alignas(64) CUtensorMap tm_state;
  alignas(64) CUtensorMap tm_units;
};

// the launches with parameter sets (mdg_step_sets): the table and the assignment, after everything the other launches
// read, so that their kernels' parameters are unchanged
struct StepSetsArgs : StepArgs {
  MdgParamSets ps;
};
// ... and with broker sets (mdg_step_sets_broker): the broker table, [MDG_BROKER_NPARAM][n_sets]
struct StepSetsBrokerArgs : StepSetsArgs {
  const double* broker;
};

constexpr int kBlock = 128;

// experiment knobs (MDG_EXTRA_NVCC_FLAGS + MDG_LIB_VARIANT, see build.py); the defaults are the measured best
#ifndef MDG_PFDIST
#define MDG_PFDIST 1    // prefetch distance in pairs
#endif
#ifndef MDG_RNG_UNROLL
#define MDG_RNG_UNROLL 4
#endif
#ifndef MDG_TAIL_UNROLL
#define MDG_TAIL_UNROLL 2
#endif
#ifndef MDG_UNITS_CG
#define MDG_UNITS_CG 0  // 1: units read as 16-byte vectors that bypass L1 (measured slower at 65,536 envs)
#endif
#ifndef MDG_ST
#define MDG_ST 0        // 0: plain stores, 1: st.global.cg (no L1 allocation) for state and outputs
#endif
#ifndef MDG_AB_L1
#define MDG_AB_L1 0
#endif
constexpr int kRngUnroll = MDG_RNG_UNROLL, kTailUnroll = MDG_TAIL_UNROLL;  // #pragma unroll does not expand macros

// ---- bulk-copy staging of the state rows (sm_90+: cp.async.bulk + mbarrier, SASS UBLKCP / SYNCS)
constexpr int kStageRows = 11;  // per stage: nine rows of BS doubles + the pair's units (2 per env)
constexpr int kBulkRows = 9;    // per pair: price x2, ledger x2, mean entry x2, borrowed margin x2, the pair's mean
constexpr int kBulkStages = 2;
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  for (unsigned spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (spin > (1u << 24)) __trap();  // a row that never lands is a bug, not a hang
  }
}

template <class T> __device__ __forceinline__ void gst(T* p, T v) {
  if (MDG_ST) __stcg(p, v); else *p = v;
}

// ---------------------------------------------------------------------------
// reward shapers (utils/buffers/nstep_buffer.py), one scalar component
// ---------------------------------------------------------------------------
__device__ __forceinline__ double clip(double x, double lo, double hi) {
  if (x != x) return x;
  return x < lo ? lo : (x > hi ? hi : x);
}
constexpr double kEps32 = 1.1920928955078125e-07;  // np.finfo(np.float32).eps, nstep_buffer.py:20

__device__ __forceinline__ double dsr_value(double A, double B, double r) {  // :80-85
  const double dA = r - A, dB = r * r - B;
  const double v = B - A * A;
  // (v^2)^(3/4) = |v|^(3/2), as |v| sqrt|v| (2 ulp; pow() costs ~250 instructions per call)
  const double av = fabs(v);
  return (B * dA - (A * dB) / 2) / (av * sqrt(av) + kEps32);
}
__device__ __forceinline__ double ddr_value(double A, double B, double r) {  // :146-156
  if (r > 0.) return (r - A / 2) / (sqrt(B) + kEps32);
  return (B * (r - A / 2) - (A * (r * r)) / 2) / (B * sqrt(B) + kEps32);  // B^(3/2)
}

// entry j (0 = oldest) of this env's n-step buffer, component c
struct NStepView {
  const double* ring;  // [nstep][ra][N]
  int64_t N, e;
  int n, ra, c, base;  // base = physical slot of entry 0
  double newest;       // the entry added this step (also stored in the ring when n>1)
  int len;             // entries including the newest
  __device__ __forceinline__ double at(int j) const {
    if (j == len - 1) return newest;
    int slot = base + j;
    if (slot >= n) slot -= n;
    return ring[((int64_t)slot * ra + c) * N + e];
  }
};

// shaped reward of one pop over entries [first, len) ; updates A,B for DSR/DDR
static __device__ __noinline__ double shaper_pop(const MdgReward& R, const NStepView& v, int first, double& A,
                                          double& B) {
  const int n = v.len - first;
  const double* disc = R.discounts;
  switch (R.shaper) {
    case MDG_SHAPER_SUM:
    case MDG_SHAPER_COSINE: {  // :23-27, :182-204
      double s = 0.;
      for (int j = 0; j < n; j += 4) {  // four ring loads in flight, summed in entry order
        const int m = n - j;
        const double x0 = v.at(first + j), x1 = m > 1 ? v.at(first + j + 1) : 0.,
                     x2 = m > 2 ? v.at(first + j + 2) : 0., x3 = m > 3 ? v.at(first + j + 3) : 0.;
        s = s + disc[j] * x0;
        if (m > 1) s = s + disc[j + 1] * x1;
        if (m > 2) s = s + disc[j + 2] * x2;
        if (m > 3) s = s + disc[j + 3] * x3;
      }
      return s;
    }
    case MDG_SHAPER_DSR: {  // :62-78
      double s = disc[0] * dsr_value(A, B, v.at(first));
      for (int j = 1; j < n; ++j) s = s + disc[j] * dsr_value(A, B, v.at(first + j));
      s = s / n;
      const double r0 = v.at(first), dA = r0 - A, dB = r0 * r0 - B;  // :87-91
      A += R.adaptation_rate * dA;
      B += R.adaptation_rate * dB;
      return clip(s, -1., 1.);
    }
    case MDG_SHAPER_DDR: {  // :128-162
      double s = disc[0] * ddr_value(A, B, v.at(first));
      for (int j = 1; j < n; ++j) s = s + disc[j] * ddr_value(A, B, v.at(first + j));
      s = s / n;
      const double r0 = v.at(first), dA = r0 - A;
      double m = r0 < 0. ? r0 : 0.;
      if (r0 != r0) m = r0;
      const double dB = m * m - B;
      A += R.adaptation_rate * dA;
      B += R.adaptation_rate * dB;
      return clip(s, -1., 1.);
    }
    case MDG_SHAPER_SHARPE: {  // :207-239
      if (n == 1) {
        double diff = v.at(first) - 0.;
        diff = (diff != 0.) ? diff : 0.;
        return diff / sqrt(diff * diff);
      }
      double sum = 0., ssq = 0.;
      for (int j = 0; j < n; ++j) {
        const double dj = (v.at(first + j) - 0.) * disc[j];
        if (j == 0) { sum = dj; ssq = dj * dj; } else { sum = sum + dj; ssq = ssq + dj * dj; }
      }
      const double num = sum / n;
      const double denom = sqrt(ssq / (n - 1));
      const double out = (denom != 0.) ? num / denom : 0.;
      return clip(.1 * out, -1., 1.);
    }
    case MDG_SHAPER_SORTINO_A: {  // :242-272
      const double ex = R.sortino_exp;
      if (n == 1) {
        const double diff = v.at(first) - 0.;
        const double downside = pow(pow(fabs(diff), ex), 1 / ex);
        return clip(0.1 * ((diff != 0.) ? diff / downside : 0.), -1., 1.);
      }
      double sum = 0., den = 0.;
      for (int j = 0; j < n; ++j) {
        const double dj = (v.at(first + j) - 0.) * disc[j];
        double down = dj < 0. ? dj : 0.;
        if (dj != dj) down = dj;
        if (down < -1.) down = -1.;
        const double t = pow(pow(fabs(down), ex) / (n - 1), 1 / ex);
        if (j == 0) { sum = dj; den = t; } else { sum = sum + dj; den = den + t; }
      }
      const double num = sum / n;
      const double zero_case = (num == 0.) ? 0. : 1.;
      const double normal = clip(.1 * (num / den), -1., 1.);
      return (den != 0.) ? normal : zero_case;
    }
    case MDG_SHAPER_SORTINO_B: {  // :276-312
      const double ex = R.sortino_exp;
      if (n == 1) {
        double diff = v.at(first) - 0.;
        if (diff < -1.) diff = -1.;
        if (diff < 0.) diff = -pow(-diff, 1 / ex);
        return clip(diff, -1., 1.);
      }
      double s = 0.;
      for (int j = 0; j < n; ++j) {
        double dj = (v.at(first + j) - 0.) * disc[j];
        if (dj < -1.) dj = -1.;
        if (dj < 0.) dj = -pow(-dj, 1 / ex);
        s = (j == 0) ? dj : s + dj;
      }
      return clip(s, -1., 1.);
    }
  }
  return 0.;
}

// ReplayBuffer.add (replay_buffer.py:68-80) + NStepBuffer.pop_nstep_sarsd (nstep_buffer.py:342-361)
// for component c of env e: add `raw`, pop once when full, drain on done.
static __device__ __noinline__ void shaper_add(const StepArgs& a, int64_t e, int c, int ra, double raw, bool done,
                                           int len_before, int& len_after, int& n_popped) {
  const MdgReward& R = a.R;
  const int64_t N = a.L.n_envs;
  const int n = R.nstep;
  double A = 0., B = 0.;
  const bool moments = (R.shaper == MDG_SHAPER_DSR || R.shaper == MDG_SHAPER_DDR);
  if (moments) {
    A = a.S.shaper_A[(int64_t)c * N + e];
    B = a.S.shaper_B[(int64_t)c * N + e];
  }
  NStepView v;
  v.ring = a.S.nstep_ring;
  v.N = N; v.e = e; v.n = n; v.ra = ra; v.c = c;
  v.newest = raw;
  v.len = len_before + 1;
  int base = a.L.nstep_pos - len_before;
  if (base < 0) base += n;
  v.base = base;
  if (n > 1) a.S.nstep_ring[((int64_t)a.L.nstep_pos * ra + c) * N + e] = raw;
  int first = 0, k = 0;
  if (v.len >= n) {
    a.IO.shaped_reward[((int64_t)k * ra + c) * N + e] = shaper_pop(R, v, first, A, B);
    ++first; ++k;
  }
  if (done) {
#pragma unroll 1
    while (first < v.len) {
      a.IO.shaped_reward[((int64_t)k * ra + c) * N + e] = shaper_pop(R, v, first, A, B);
      ++first; ++k;
    }
  }
  if (moments) {
    a.S.shaper_A[(int64_t)c * N + e] = A;
    a.S.shaper_B[(int64_t)c * N + e] = B;
  }
  len_after = v.len - first;
  n_popped = k;
}

// ---------------------------------------------------------------------------
// the step kernel
// ---------------------------------------------------------------------------
// rows of MdgState.folds
#define MDG_FOLD_AV 0
#define MDG_FOLD_ML 1
#define MDG_FOLD_BM 2
#define MDG_FOLD_SE 3
#define MDG_FOLD_G 4

// Exact risk gate of asset i (Portfolio::checkRisk(i, units), Portfolio.cpp:254-279): every accounting
// quantity is a left-to-right fold over the assets, exactly as in the oracle.  COLD path, called only when
// the cheap bound in step_kernel cannot decide.  (pav..pse) are the folds over the already processed
// assets 0..i-1 (final values); assets i.. are untouched so far and are re-read from global memory.
static __device__ __noinline__ int exact_gate(const MdgState& S, int64_t N, int64_t e, int na, double cash,
                                              double reqM, double maintM, int i, double units, double av,
                                              double ml, double bms, double se) {
#pragma unroll 1
  for (int j = i; j < na; ++j) {
    const double l = S.ledger[(int64_t)j * N + e], p = S.price[(int64_t)j * N + e],
                 m = S.mean_entry[(int64_t)j * N + e], b = S.borrowed[(int64_t)j * N + e];
    const double t_se = l * (m * (l < 0. ? 1. : 0.));
    if (j == 0) { av = l * p; ml = m * l; bms = b; se = t_se; }
    else { av = av + l * p; ml = ml + m * l; bms = bms + b; se = se + t_se; }
  }
  const double price = S.price[(int64_t)i * N + e], cur = S.ledger[(int64_t)i * N + e];
  const bool opposite = (signbit(units) != 0) != (signbit(cur) != 0);
  const double pnl = av - ml;        // :184-186
  const double balance = cash + se;  // :192-197
  const double availableMargin = (balance + pnl) / reqM;  // :229-231
  if (opposite) {
    const double excess = units + cur;
    if (availableMargin <= fabs(price * excess) || balance <= 0.) return MDG_RISK_INSUFF_MARGIN;
    return MDG_RISK_GREEN;
  }
  if (margin_call(cash, av, ml, bms, se, maintM)) return MDG_RISK_MARGIN_CALL;
  if (availableMargin <= fabs(price * units) || balance <= 0.) return MDG_RISK_INSUFF_MARGIN;
  return MDG_RISK_GREEN;
}

// Registers of one env while it streams over its assets
struct StepAcc {
  double cash;
  double rAV, rML, rBM, rSE, G;  // running sums (cheap risk bound) and their magnitude bound
  double pav, pml, pbm, pse;     // exact left-to-right folds over the processed assets, old prices
  double nav, gsum;              // exact fold of ledger*new price; magnitude sum for the next step
  double rprod, inv_prev;        // reduced agent reward accumulated in the asset loop (post_tick)
  bool reduce_inloop;
  bool bad_risk;
};

// The broker settings the step kernel reads, and the risk-gate constants made from them.
// StepConsts: kernel parameters (MdgParams, and StepArgs.c_* that launch_step computes from it); `c` is only a tag.
struct StepConsts {
  __device__ __forceinline__ double init_cash(const StepArgs& a) const { return a.P.init_cash; }
  __device__ __forceinline__ double reqM(const StepArgs& a) const { return a.c_reqM; }
  __device__ __forceinline__ double maintM(const StepArgs& a) const { return a.c_maintM; }
  __device__ __forceinline__ double slip_rel(const StepArgs& a) const { return a.P.slippage_rel; }
  __device__ __forceinline__ double slip_abs(const StepArgs& a) const { return a.P.slippage_abs; }
  __device__ __forceinline__ double tcost_rel(const StepArgs& a) const { return a.P.tcost_rel; }
  __device__ __forceinline__ double tcost_abs(const StepArgs& a) const { return a.P.tcost_abs; }
  __device__ __forceinline__ int reqM_ok(const StepArgs& a) const { return a.c_reqM_ok; }
  __device__ __forceinline__ double band_scale(const StepArgs& a) const { return a.c_band_scale; }
  __device__ __forceinline__ double g1(const StepArgs& a) const { return a.c_g1; }
  __device__ __forceinline__ double g2(const StepArgs& a) const { return a.c_g2; }
};
// BrokerConsts (broker sets): the env's entry of the broker table, loaded next to each use (the table is a few hundred
// bytes and stays in L1 / L2; only the 32-bit set index is live), and the gate constants computed per env with
// launch_step's expressions, so that every decision is the one a launch with these values in MdgParams takes
struct BrokerConsts {
  uint32_t set;
  __device__ __forceinline__ double at(const StepArgs& a, int k) const {
    const StepSetsBrokerArgs& b = static_cast<const StepSetsBrokerArgs&>(a);
    return broker_value(b.broker, b.ps.n_sets, set, k);
  }
  __device__ __forceinline__ double init_cash(const StepArgs& a) const { return at(a, MDG_BROKER_INIT_CASH); }
  __device__ __forceinline__ double reqM(const StepArgs& a) const { return at(a, MDG_BROKER_REQUIRED_MARGIN); }
  __device__ __forceinline__ double maintM(const StepArgs& a) const { return at(a, MDG_BROKER_MAINTENANCE_MARGIN); }
  __device__ __forceinline__ double slip_rel(const StepArgs& a) const { return at(a, MDG_BROKER_SLIPPAGE_REL); }
  __device__ __forceinline__ double slip_abs(const StepArgs& a) const { return at(a, MDG_BROKER_SLIPPAGE_ABS); }
  __device__ __forceinline__ double tcost_rel(const StepArgs& a) const { return at(a, MDG_BROKER_TCOST_REL); }
  __device__ __forceinline__ double tcost_abs(const StepArgs& a) const { return at(a, MDG_BROKER_TCOST_ABS); }
  __device__ __forceinline__ int reqM_ok(const StepArgs& a) const {
    const double r = reqM(a);
    return (r > 0. && r <= 1e6) ? 1 : 0;
  }
  __device__ __forceinline__ double band_scale(const StepArgs& a) const {
    const double r = reqM(a);
    return 1e-9 * (1. + fabs(maintM(a))) * (r > 1. ? r : 1.);
  }
  __device__ __forceinline__ double g1(const StepArgs& a) const { return 6. + 3. * fabs(slip_rel(a)) + fabs(tcost_rel(a)); }
  __device__ __forceinline__ double g2(const StepArgs& a) const { return 3. * fabs(slip_abs(a)); }
};

// Broker::handleTransaction(port, i, units) (Broker.cpp:124-142) for one asset whose state is in registers:
// risk gate (Portfolio.cpp:254-279), slippage/cost (Broker.cpp:171-178), ledger update (Portfolio.cpp:284-323).
//
// The gate compares folds over the whole portfolio with thresholds.  Recomputing the folds per asset is
// O(nA^2) fp64 work, so the gate first uses RUNNING sums (O(1) update per transaction, hence rounded
// differently from a fresh fold) with a rigorous bound: running and exact folds differ by < 1e-13 * G
// (G = sum of magnitudes); a decision is taken from the running sums only when it clears its threshold by
// 1e-9 * G.  Otherwise -- a knife-edge, NaN/Inf, a non-positive required margin -- the exact left-to-right
// folds decide (exact_gate).  Decisions, and therefore ledgers, are bit-identical to the oracle's either way.
template <bool TX2, class C>
__device__ __forceinline__ void tx_asset(const StepArgs& a, const C& c, StepAcc& A, int64_t N, int64_t e,
                                         int na, int i, double price, double& cur, double& mep, double& bm,
                                         double units, double& tp, double& tu, double& tc, int& risk,
                                         double& prev_val) {
  const MdgState& S = a.S;
  prev_val = cur * price;  // offpolicy_q.py:141
  tp = 0.; tu = 0.; tc = 0.;
  risk = MDG_RISK_GREEN;
  if (units != 0.) {  // Broker.cpp:126 (NaN units do enter, as in the reference)
    const bool opposite = (signbit(units) != 0) != (signbit(cur) != 0);
    if (!opposite || units > -1 * cur) {  // Portfolio.cpp:257-258: only these orders are gated
      const double amt = fabs(price * (opposite ? units + cur : units));
      const double bal = A.cash + A.rSE, pnl = A.rAV - A.rML, x = bal + pnl;
      const double band = c.band_scale(a) * (A.G + amt);
      const double d1 = x - amt * c.reqM(a);  // availableMargin <= |amount|  <=>  d1 <= 0
      bool certain;
      int r_fast;
      if constexpr (TX2) {
        // multi-wave variant (168 registers): predicate arithmetic instead of short-circuit branches, the same
        // decisions; 3.5 % faster at 1 M envs, but it costs registers the one-wave variant does not have
        const double m = c.maintM(a) * pnl;
        const double d3 = (A.cash + A.rAV - A.rBM) + m, d4 = x + m;  // Portfolio::checkRisk() first (:268), :243-252
        const bool ok1 = (fabs(d1) > band) & (fabs(bal) > band);
        const bool ok2 = (fabs(d3) > band) & (fabs(d4) > band);
        certain = c.reqM_ok(a) & ok1 & (opposite | ok2);
        const bool insuff = (d1 <= 0.) | (bal <= 0.);
        const bool mcall = !opposite & ((d3 <= 0.) | (d4 <= 0.));
        r_fast = mcall ? MDG_RISK_MARGIN_CALL : (insuff ? MDG_RISK_INSUFF_MARGIN : MDG_RISK_GREEN);
      } else {
        certain = c.reqM_ok(a) && fabs(d1) > band && fabs(bal) > band;
        r_fast = (d1 <= 0. || bal <= 0.) ? MDG_RISK_INSUFF_MARGIN : MDG_RISK_GREEN;
        if (!opposite) {  // Portfolio::checkRisk() first (:268), :243-252
          const double m = c.maintM(a) * pnl;
          const double d3 = (A.cash + A.rAV - A.rBM) + m, d4 = x + m;
          certain = certain && fabs(d3) > band && fabs(d4) > band;
          if (d3 <= 0. || d4 <= 0.) r_fast = MDG_RISK_MARGIN_CALL;
        }
      }
      risk = (certain && !a.c_force_exact)
                 ? r_fast
                 : exact_gate(S, N, e, na, A.cash, c.reqM(a), c.maintM(a), i, units, A.pav, A.pml, A.pbm, A.pse);
    }
    if (risk == MDG_RISK_GREEN) {
      // Broker::applySlippage / getTransactionCost  Broker.cpp:171-178
      const double slippage = (price * c.slip_rel(a)) + c.slip_abs(a);
      const double transactionPrice = units < 0 ? (price - slippage) : (price + slippage);
      const double transactionCost = fabs(units * price) * c.tcost_rel(a) + c.tcost_abs(a);
      tp = transactionPrice; tu = units; tc = transactionCost;
      // Portfolio::handleTransaction  Portfolio.cpp:284-323
      const double o_ml = mep * cur, o_bm = bm;
      const double o_se = (cur < 0.) ? o_ml : 0.;
      if (opposite) {
        if (fabs(units) > fabs(cur)) {
          units += cur;
          A.cash += cur * transactionPrice;
          cur = 0.;
          mep = transactionPrice;
        }
      } else {
        mep += (transactionPrice - mep) * (units / (units + cur));
      }
      const double amount = transactionPrice * units;
      const double marginToUse = amount * c.reqM(a);
      const double marginToBorrow = amount - marginToUse;
      bm += marginToBorrow;
      A.cash -= (marginToUse + transactionCost);
      cur += units;
      if constexpr (TX2) {
        const bool flat = fabs(cur) < 0.000001;
        mep = flat ? 0. : mep;
        const bool ra_ = flat & (bm > 0.);
        A.cash = ra_ ? A.cash - bm : A.cash;
        bm = ra_ ? 0. : bm;
        const bool rb_ = bm < 0.;
        A.cash = rb_ ? A.cash - bm : A.cash;
        bm = rb_ ? 0. : bm;
      } else {
        if (fabs(cur) < 0.000001) {
          mep = 0.;
          if (bm > 0.) { A.cash -= bm; bm = 0.; }
        }
        if (bm < 0.) { A.cash -= bm; bm = 0.; }
      }
      gst(&S.ledger[(int64_t)i * N + e], cur);
      gst(&S.mean_entry[(int64_t)i * N + e], mep);
      gst(&S.borrowed[(int64_t)i * N + e], bm);
      // running sums and their magnitude bound
      const double n_av = cur * price, n_ml = mep * cur;
      A.rAV += n_av - prev_val;
      A.rML += n_ml - o_ml;
      A.rBM += bm - o_bm;
      A.rSE += ((cur < 0.) ? n_ml : 0.) - o_se;
      // every new term's magnitude is at most its old magnitude (already in G) plus |units|*(|price|+|tp|), three
      // terms, plus the cost; with |tp| <= |price|(1+|slip_rel|)+|slip_abs| and |cost| <= |units price||tc_rel|+|tc_abs|
      // that is |units| * (|price| * g1 + g2) (+ |tc_abs|, added once per asset in the prologue)
      A.G += fabs(tu) * (fabs(price) * c.g1(a) + c.g2(a));
    } else if (risk != MDG_RISK_INSUFF_MARGIN) {
      A.bad_risk = true;
    }
  }
  if (a.L.mode != MDG_MODE_HOLD) {
    gst(&a.IO.trans_price[(int64_t)i * N + e], tp);
    gst(&a.IO.trans_units[(int64_t)i * N + e], tu);
    gst(&a.IO.trans_cost[(int64_t)i * N + e], tc);
    a.IO.risk[(int64_t)i * N + e] = (uint8_t)risk;
  }
  // exact folds of the final ledger, old prices (Portfolio.cpp:180-197,207-209)
  const double t_ml = mep * cur;
  const double t_se = (cur < 0.) ? t_ml : 0. * t_ml;
  if (i == 0) { A.pav = cur * price; A.pml = t_ml; A.pbm = bm; A.pse = t_se; }
  else { A.pav = A.pav + cur * price; A.pml = A.pml + t_ml; A.pbm = A.pbm + bm; A.pse = A.pse + t_se; }
  A.gsum += fabs(t_ml) + fabs(bm);
}

// Shared-memory stash of the all-OU-pairs kernel, one column per thread, four rows per pair p:
//   before the pair is processed: rows 4p..4p+2 hold its three normals (noise slots 3p..3p+2);
//   afterwards: rows 4p, 4p+1 = position values after the tick, rows 4p+2, 4p+3 = prev value + mar_diff.
__device__ __forceinline__ int stash_normal_row(int slot) { const int p = slot / 3; return 4 * p + (slot - 3 * p); }
template <bool PAIRS> __device__ __forceinline__ int stash_cur_row(int j, int na) {
  return PAIRS ? 4 * (j >> 1) + (j & 1) : j;
}
template <bool PAIRS> __device__ __forceinline__ int stash_pm_row(int j, int na) {
  return PAIRS ? 4 * (j >> 1) + 2 + (j & 1) : na + j;
}

// dqn.py:165-178: centred action times (unit_size * availableMargin / price); action 0 closes an open position
__device__ __forceinline__ double action_units(int act, int half, double scale, double price, double cur) {
  if (act == 0) return (cur != 0.) ? -cur : 0.;
  return (double)(act - half) * (scale / price);
}

// ddpg.py:182-207: target weights -> units.  desired = w / sum(w) in fp32 (what torch computes on the actor's
// output), widened; units = ((desired - ledgerNormedFull_i) * equity) / price, ledgerNormedFull_i =
// (ledger_i * price_i) / equity (Portfolio.cpp:150-155).  w_sum == 0: the weights are taken as they are (:193-194).
__device__ __forceinline__ double weight_units(float w, float w_sum, double price, double cur, double equity) {
  const float d = (w_sum == 0.f) ? w : w / w_sum;
  const double cur_w = (cur * price) / equity;
  return (((double)d - cur_w) * equity) / price;
}

// after the tick of asset i: state/observation stores, fold of the new position value, reward stash
template <bool PAIRS, int BS>
__device__ __forceinline__ void post_tick(const StepArgs& a, StepAcc& A, int64_t N, int64_t e, int na, int i,
                                          double cur, double newp, double prev_val, double tp, double tu,
                                          double tc, double* st) {
  gst(&a.S.price[(int64_t)i * N + e], newp);
  gst(&a.IO.obs_price[((int64_t)a.L.head * na + i) * N + e], newp);  // State.price row (Env.h:202,228,254)
  const double cur_val = cur * newp;
  A.nav = (i == 0) ? cur_val : A.nav + cur_val;
  A.gsum += fabs(cur_val);
  st[stash_cur_row<PAIRS>(i, na) * BS] = cur_val;
  const double pm = prev_val + (tu * tp + tc);  // prev_val + mar_diff, offpolicy_q.py:153-156
  if (A.reduce_inloop) {
    // reduced agent reward (offpolicy_q.py:152-164): sum_j log(max(1 + (cur_j - pm_j)/prevEq, .35)) accumulated as the
    // log of a product (see the tail) right here, so that pm_j needs no stash row
    double x = (cur_val - pm) * A.inv_prev;
    x += 1;
    x = (x != x) ? x : ((x < .35) ? .35 : x);
    A.rprod = (i == 0) ? x : A.rprod * x;
  } else {
    st[stash_pm_row<PAIRS>(i, na) * BS] = pm;
  }
}

// One Philox block -> two standard normals (Box-Muller), the same (block, lane) addressing as draw_normal:
// slot s = block s>>1, lane s&1.
__device__ __forceinline__ void normal_block(uint32_t gid, uint32_t blk, uint32_t t_lo, uint32_t t_hi, uint32_t k0,
                                             uint32_t k1, double& z_lane0, double& z_lane1) {
  uint64_t x0, x1;
  philox4x32_10(gid, blk, t_lo, t_hi, k0, k1, x0, x1);
  const double u1 = ((double)(x0 >> 12) + 0.5) * 0x1.0p-52;
  const double u2 = (double)(x1 >> 11) * 0x1.0p-53;
  const double r = fast_sqrt_pos(-2.0 * fast_log_pos(u1));
  double sn, cs;
  fast_sincos_2pi(u2, sn, cs);
  z_lane0 = r * cs;
  z_lane1 = r * sn;
}

// generator-state rows owned by asset i (see MdgAssetGen)
__device__ __forceinline__ int gen_state_rows(const MdgAssetGen& g) {
  if (g.gslot < 0) return 0;
  switch (g.type) {
    case MDG_GEN_TRENDYOU: return 4;
    case MDG_GEN_TRENDOU: return 3;
    case MDG_GEN_SIMPLETREND: return 2;
    case MDG_GEN_SINEADDER: return (int)g.p[0];
    case MDG_GEN_SINEDYNAMIC: return 4 * (int)g.p[0];
    case MDG_GEN_SINEDYNAMICTREND: return 4 * (int)g.p[0] + 1 + (int)g.p[4];
    default: return 1;
  }
}

// Two register budgets of the same kernel, chosen by the number of envs per launch (profiles/largeN.py):
//   128 registers -> 4 blocks of 128 per SM: the 443 envs per SM of a 65,536-env launch are resident in ONE
//     wave (that launch is latency-bound: a second wave would cost as much as the first);
//   168 registers -> 3 blocks per SM, no spills: best throughput when there are many waves (>= 262,144 envs).
// (64-thread blocks x 7 per SM at 144 registers were measured slower than either.)
// -DMDG_PHASE_CLOCKS (profiling builds only, profiles/phase_clocks.py): thread MDG_PCLK_TID of the first 64 blocks
// records clock64() at the phase boundaries of its step
#ifdef MDG_PHASE_CLOCKS
#ifndef MDG_PCLK_TID
#define MDG_PCLK_TID 0
#endif
#ifndef MDG_PCLK_B0
#define MDG_PCLK_B0 0  // first of the 64 blocks that record
#endif
__device__ long long g_phase_clk[64 * 64];
__device__ unsigned long long g_block_ns[1024 * 4];  // per block: %globaltimer at entry / exit of thread 0, %smid
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define MDG_PCLK(slot)                                                                                     \
  do {                                                                                                     \
    if (threadIdx.x == MDG_PCLK_TID && blockIdx.x >= MDG_PCLK_B0 && blockIdx.x < MDG_PCLK_B0 + 64)         \
      g_phase_clk[(blockIdx.x - MDG_PCLK_B0) * 64 + (slot)] = clock64();                                   \
  } while (0)
#else
#define MDG_PCLK(slot)
#endif

template <bool PAIRS, int BS, bool ACTIONS, bool TX2, bool BULK, bool SETS = false, bool BROKER = false>
__device__ __forceinline__ void step_body(const StepArgs& a) {
  static_assert(SETS || !BROKER, "broker sets index the parameter sets' assignment");
  MDG_PCLK(0);
#ifdef MDG_PHASE_CLOCKS
  if (threadIdx.x == 0 && blockIdx.x < 1024) {
    unsigned smid;
    asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
    g_block_ns[blockIdx.x * 4] = global_ns();
    g_block_ns[blockIdx.x * 4 + 2] = smid;
  }
#endif
  // per-thread stash, [2*nA][BS]: position value after the tick, and prev value + mar_diff (and, in the
  // all-pairs kernel, this step's normals before they are consumed; see stash_normal_row)
  extern __shared__ __align__(128) double stash[];
  const MdgParams& P = a.P;
  const MdgState& S = a.S;
  const int64_t N = a.L.n_envs;
  const int na = P.n_assets;
  const int tid = threadIdx.x;
  const int64_t e = (int64_t)blockIdx.x * BS + tid;
  const int mode = a.L.mode;
  double* st = stash + tid;  // this thread's column, [row * BS]
  // the caller's units matrix is (N, nA) env-major: a thread's row is one 128-byte line.  Read as 16-byte
  // vectors (one per pair) that bypass L1, so that the 64 KB of unit lines per SM do not evict the prefetched state
  const bool units_v2 = MDG_UNITS_CG && PAIRS && mode == MDG_MODE_MULTI && a.units_v2;
  if (e >= N) return;
  // parameter sets: this env's set (SETS only; the table's address and n_sets stay kernel-parameter operands)
  uint32_t set = 0;
  if constexpr (SETS) set = (uint32_t)env_set(static_cast<const StepSetsArgs&>(a).ps, e);
  // Bulk staging (all-pairs kernel, whole blocks only): the nine 1-KB state rows a block needs for a pair are
  // contiguous in the [rows][N] tensors, so one elected thread fetches them with nine cp.async.bulk copies into a
  // two-stage shared-memory ring, two pairs ahead, completion on an mbarrier per stage.  The bytes are in flight
  // without holding registers (the register prefetch of round 1 spilled at the 128-register budget) and arrive in
  // shared memory instead of L2 (the prefetch.global.L1 hints still left an L2 round trip on every first use).
  constexpr bool bulk = PAIRS && BULK;
  double* ring = stash + 2 * na * BS;
  uint64_t* full = reinterpret_cast<uint64_t*>(ring + kBulkStages * kStageRows * BS);
  const int64_t e0 = (int64_t)blockIdx.x * BS;
  const bool tma = bulk && a.bulk == 2;
  const bool tma_units = tma && a.tma_units;
  // bulk == 2: ONE 3-D tensor copy brings the pair's eight state rows (box 128 envs x 2 assets x 4 tensors), one
  // 2-D tensor copy gathers the pair's 16 bytes of every env's units row (box 2 x 128), one bulk copy the mean row
  auto tma_issue = [&](int pp, int stage) {  // one thread
    const uint32_t mb = smem_u32(&full[stage]);
    double* sb = ring + stage * kStageRows * BS;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb),
                 "r"((uint32_t)((kBulkRows + (tma_units ? 2 : 0)) * BS * sizeof(double)))
                 : "memory");
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            smem_u32(sb)),
        "l"(&a.tm_state), "r"((int)e0), "r"(2 * pp), "r"(0), "r"(mb)
        : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(sb + 8 * BS)),
                 "l"(S.gstate + (int64_t)P.gen[2 * pp].gslot * N + e0), "r"((uint32_t)(BS * sizeof(double))), "r"(mb)
                 : "memory");
    if (tma_units)
      asm volatile(
          "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
              smem_u32(sb + kBulkRows * BS)),
          "l"(&a.tm_units), "r"(2 * pp), "r"((int)e0), "r"(mb)
          : "memory");
  };
  auto bulk_issue = [&](int pp, int stage) {  // one thread
    // The copies below write the stage through the async proxy; it was last accessed through the generic proxy (read
    // by this block's threads, ordered by the barrier before the issue).  PTX orders the two proxies only through a
    // proxy fence.  Without it, runs with slabs on concurrent streams (tests/test_bench_dump.py) differed from run
    // to run in thousands of envs.
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (tma) { tma_issue(pp, stage); return; }
    const uint32_t mb = smem_u32(&full[stage]);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb),
                 "r"((uint32_t)(kBulkRows * BS * sizeof(double)))
                 : "memory");
    const int64_t o0 = (int64_t)(2 * pp) * N + e0, o1 = o0 + N;
    const double* src[kBulkRows] = {S.price + o0, S.price + o1, S.ledger + o0, S.ledger + o1, S.mean_entry + o0,
                                    S.mean_entry + o1, S.borrowed + o0, S.borrowed + o1,
                                    S.gstate + (int64_t)P.gen[2 * pp].gslot * N + e0};
#pragma unroll
    for (int r = 0; r < kBulkRows; ++r)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       smem_u32(ring + stage * kStageRows * BS + r * BS)),
                   "l"(src[r]), "r"((uint32_t)(BS * sizeof(double))), "r"(mb)
                   : "memory");
  };
  const bool shaping = (a.R.shaper != MDG_SHAPER_OFF) && (mode != MDG_MODE_HOLD);
  const double* urow = a.IO.units ? a.IO.units + (mode == MDG_MODE_MULTI ? e * na : e) : nullptr;  // unused with actions
  const bool moments = shaping && (a.R.shaper == MDG_SHAPER_DSR || a.R.shaper == MDG_SHAPER_DDR);
  auto prefetch_hint = [&](int pp) {
    const int64_t o0 = (int64_t)(2 * pp) * N + e, o1 = o0 + N;
    asm volatile("prefetch.global.L1 [%0];" ::"l"(S.price + o0));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(S.price + o1));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(S.ledger + o0));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(S.ledger + o1));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(S.mean_entry + o0));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(S.mean_entry + o1));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(S.borrowed + o0));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(S.borrowed + o1));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(S.gstate + (int64_t)P.gen[2 * pp].gslot * N + e));
  };
  if (PAIRS && !bulk) {
    // The next pair's lines are pulled into L1 with prefetch hints and loaded when needed.  (Holding the next
    // pair in registers instead made the compiler spill it at the 128-register budget -- a local store right
    // behind the load, i.e. a full-latency stall; cp.async stages in shared memory were slower too:
    // profiles/r1_notes.md.)
    prefetch_hint(0);
    if (MDG_PFDIST > 1 && na > 2) prefetch_hint(1);
    if (mode == MDG_MODE_MULTI && urow) asm volatile("prefetch.global.L1 [%0];" ::"l"(urow));
  }
  // The reduced reward's n-step shaper with nstep == 1 (add, pop at once: the common case) runs inline in the tail;
  // its moments are loaded here, at the start, so that no load latency is left at the end of the thread's chain.
  // The env's tick is the first thing requested: it is all the normals need, and they are generated below while the
  // rest of the prologue's loads (and everybody else's: every block of a one-wave launch starts at the same moment,
  // profiles/phase_clocks.py: the youngest block of an SM left the prologue 6,000 cycles after the oldest) arrive.
  const int64_t ts = S.timestamp[e];
  const bool inline_shaper = shaping && a.R.reduce_rewards && a.R.shaper != MDG_SHAPER_COSINE && a.R.nstep == 1 &&
                             (moments || a.R.shaper == MDG_SHAPER_SUM);
  double shA = 0., shB = 0.;
  if (moments && inline_shaper) {
    shA = a.S.shaper_A[e];
    shB = a.S.shaper_B[e];
  } else if (moments) {  // read at the very end of the kernel: have the lines in L2 by then
    asm volatile("prefetch.global.L2 [%0];" ::"l"(a.S.shaper_A + e));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(a.S.shaper_B + e));
  }

  StepAcc A;
  A.cash = S.cash[e];
  // Folds of the incoming portfolio.  They are exactly the folds this kernel (or reset/init/refresh)
  // computed at the end of the previous call -- same values, same left-to-right order -- so they are
  // carried in state instead of re-reading the whole portfolio before the first transaction.
  A.rAV = S.folds[(int64_t)MDG_FOLD_AV * N + e];
  A.rML = S.folds[(int64_t)MDG_FOLD_ML * N + e];
  A.rBM = S.folds[(int64_t)MDG_FOLD_BM * N + e];
  A.rSE = S.folds[(int64_t)MDG_FOLD_SE * N + e];
  A.G = S.folds[(int64_t)MDG_FOLD_G * N + e];
  // The ring is set up AFTER the loads above have been issued: the first copy instructions of a kernel keep their
  // thread busy for ~4,000 cycles (profiles/phase_clocks.py: the issuing warp left the prologue 4,000 cycles after
  // the others, and they waited for it at the first pair), which now overlaps the latency of these loads.  Only the
  // first pair's rows are requested here, the second pair's after the normals.
  if (bulk) {
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&full[0])) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&full[1])) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) bulk_issue(0, 0);
  }
  const uint32_t gid = (uint32_t)(a.L.env_offset + e);
  const uint32_t k0 = (uint32_t)a.L.seed, k1 = (uint32_t)(a.L.seed >> 32);
  const uint32_t t_lo = (uint32_t)(uint64_t)ts, t_hi = (uint32_t)((uint64_t)ts >> 32);
  if (PAIRS) {
    const int np = na >> 1;
    // This step's normals, all at once: the Philox + Box-Muller blocks are independent of each other and of
    // the ledger, so they are generated four at a time (four interleaved dependency chains per thread --
    // the kernel is latency-bound at one thread per env) while the first loads are in flight.
    if (!a.IO.normals) {
      const int nslots = 3 * np, nblk = (nslots + 1) >> 1;
#pragma unroll kRngUnroll
      for (int b = 0; b < nblk; ++b) {
        double za, zb;
        normal_block(gid, (uint32_t)b, t_lo, t_hi, k0, k1, za, zb);
        st[stash_normal_row(2 * b) * BS] = za;
        if (2 * b + 1 < nslots) st[stash_normal_row(2 * b + 1) * BS] = zb;
      }
    }
  }
  MDG_PCLK(2);
  A.pav = A.pml = A.pbm = A.pse = A.nav = A.gsum = 0.;
  A.bad_risk = false;
  const double prevEq = A.cash + A.rAV - A.rBM;  // Env.h:190,208,234
  A.inv_prev = 1. / prevEq;
  A.rprod = 1.;
  A.reduce_inloop = shaping && a.R.reduce_rewards && a.R.shaper != MDG_SHAPER_COSINE;
  // DQN.action_to_transaction (dqn.py:160-179) fused in front of the step: units from discrete actions and the
  // availableMargin of the incoming portfolio (Portfolio.cpp:229-231), one scale for every asset
  // (a template parameter: the three extra live values cost 3 % in the units kernel at its 128-register budget)
  const int8_t* arow = (ACTIONS && mode == MDG_MODE_MULTI && a.IO.actions) ? a.IO.actions + e * na : nullptr;
  const auto c = [&] {  // the broker settings: kernel parameters, or this env's set (BROKER)
    if constexpr (BROKER) return BrokerConsts{set};
    else return StepConsts{};
  }();
  const double act_scale = arow ? a.L.unit_size * (((A.cash + A.rSE) + (A.rAV - A.rML)) / c.reqM(a)) : 0.;
  const int act_half = a.L.action_atoms / 2;
  // DDPG.action_to_transaction (ddpg.py:182-207), likewise: target weights (cash first) -> units
  const float* wrow = (ACTIONS && mode == MDG_MODE_MULTI && a.IO.weights) ? a.IO.weights + e * (na + 1) : nullptr;
  float w_sum = 0.f;
  if (wrow) {
    w_sum = wrow[0];
    for (int j = 1; j <= na; ++j) w_sum = w_sum + wrow[j];
  }

  A.G += na * fabs(c.tcost_abs(a));  // the absolute cost of up to nA transactions

  MDG_PCLK(1);
  if (PAIRS) {
    // ---- headline path: every asset belongs to an OU pair.  One iteration = one pair; the next pair's
    // state and units are loaded while the current pair is processed (software prefetch).
    const int np = na >> 1;
    if (bulk && tid == 0 && na > 2) bulk_issue(1, 1);
#pragma unroll 1
    for (int p = 0; p < np; ++p) {
      double price[2], cur[2], mep[2], bm[2], units[2], prev_val[2], tp[2], tu[2], tc[2];
      int risk[2];
      // the pair's state arrived through the prefetch stage p & 1 (group p; at most group p+1 is still in flight)
      double mean;
      if (bulk) {
        const int stage = p & 1;
        mbar_wait(&full[stage], (uint32_t)((p >> 1) & 1));
        if (p == 0) MDG_PCLK(41);
        if (p == 3) MDG_PCLK(43);
        const double* rg = ring + stage * kStageRows * BS + tid;
        price[0] = rg[0]; price[1] = rg[BS]; cur[0] = rg[2 * BS]; cur[1] = rg[3 * BS];
        mep[0] = rg[4 * BS]; mep[1] = rg[5 * BS]; bm[0] = rg[6 * BS]; bm[1] = rg[7 * BS];
        mean = rg[8 * BS];
        if (tma_units) {
          const double2 u2 = *reinterpret_cast<const double2*>(ring + stage * kStageRows * BS + kBulkRows * BS + 2 * tid);
          units[0] = u2.x; units[1] = u2.y;
        }
        __syncthreads();  // every thread has taken its values: the stage is free for the pair after next
        if (p == 0) MDG_PCLK(42);
        if (p == 3) MDG_PCLK(44);
        if (tid == 0 && p + kBulkStages < np) bulk_issue(p + kBulkStages, stage);
      } else {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int64_t o = (int64_t)(2 * p + q) * N + e;
          price[q] = S.price[o]; cur[q] = S.ledger[o]; mep[q] = S.mean_entry[o]; bm[q] = S.borrowed[o];
        }
      }
      if (tma_units) {
        // (taken from the ring above)
      } else if (units_v2) {
        const double2 u2 = __ldcg(reinterpret_cast<const double2*>(urow + 2 * p));
        units[0] = u2.x; units[1] = u2.y;
      } else {
        units[0] = (mode == MDG_MODE_MULTI && !arow && !wrow) ? urow[2 * p] : 0.;
        units[1] = (mode == MDG_MODE_MULTI && !arow && !wrow) ? urow[2 * p + 1] : 0.;
      }
      if (wrow) {
#pragma unroll
        for (int q = 0; q < 2; ++q) units[q] = weight_units(wrow[2 * p + q + 1], w_sum, price[q], cur[q], prevEq);
      } else if (arow) {
#pragma unroll
        for (int q = 0; q < 2; ++q) units[q] = action_units(arow[2 * p + q], act_half, act_scale, price[q], cur[q]);
      }
      if (!bulk) {
        mean = S.gstate[(int64_t)P.gen[2 * p].gslot * N + e];
        if (p + MDG_PFDIST < np) prefetch_hint(p + MDG_PFDIST);
      }
#if defined(MDG_PHASE_CLOCKS) && defined(MDG_PCLK_USE)
      {  // force the operands to have arrived before the clock is read: 1 = state values, 2 = units, 3 = both
        double chk = 0.;
        if (MDG_PCLK_USE & 1) chk += price[0] + cur[0] + mep[0] + bm[0] + price[1] + cur[1] + mep[1] + bm[1] + mean;
        if (MDG_PCLK_USE & 2) chk += units[0] + units[1];
        if (chk == 1.2345e300) __trap();
      }
#endif
      MDG_PCLK(3 + 4 * p);
      {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int i = 2 * p + q;
          if (mode == MDG_MODE_SINGLE) units[q] = (i == a.L.asset_idx) ? urow[0] : 0.;
          tx_asset<TX2>(a, c, A, N, e, na, i, price[q], cur[q], mep[q], bm[q], units[q], tp[q], tu[q], tc[q], risk[q],
                        prev_val[q]);
          MDG_PCLK(4 + 4 * p + q);
        }
      }
      // OUPair::getData, DataSource.cpp:1232-1240 (draw order rw, x0, x1)
      const MdgAssetGen& g0 = P.gen[2 * p];
      const MdgAssetGen& g1 = P.gen[2 * p + 1];
      double z_rw, z0, z1;
      if (a.IO.normals) {
        z_rw = a.IO.normals[(int64_t)g0.nslot_aux * N + e];
        z0 = a.IO.normals[(int64_t)g0.nslot * N + e];
        z1 = a.IO.normals[(int64_t)g1.nslot * N + e];
      } else {
        z_rw = st[(4 * p) * BS];
        z0 = st[(4 * p + 1) * BS];
        z1 = st[(4 * p + 2) * BS];
      }
      double newp0, newp1;
      if constexpr (SETS) {  // the pair's five values of this env's set
        const MdgParamSets& ps = static_cast<const StepSetsArgs&>(a).ps;
        const SetParams q0 = set_params(ps, set, 2 * p), q1 = set_params(ps, set, 2 * p + 1);
        const double s_theta0 = q0[0], s_phi0 = q0[1], s_noise = q0[2], s_theta1 = q1[0], s_phi1 = q1[1];
        mean += mean * (z_rw * s_noise);
        gst(&S.gstate[(int64_t)g0.gslot * N + e], mean);
        newp0 = price[0] + ((s_theta0 * (mean - price[0])) + mean * (z0 * s_phi0));
        newp1 = price[1] + ((s_theta1 * (mean - price[1])) + mean * (z1 * s_phi1));
      } else {
        mean += mean * (z_rw * g0.p[2]);
        gst(&S.gstate[(int64_t)g0.gslot * N + e], mean);
        newp0 = price[0] + ((g0.p[0] * (mean - price[0])) + mean * (z0 * g0.p[1]));
        newp1 = price[1] + ((g1.p[0] * (mean - price[1])) + mean * (z1 * g1.p[1]));
      }
      post_tick<true, BS>(a, A, N, e, na, 2 * p, cur[0], newp0, prev_val[0], tp[0], tu[0], tc[0], st);
      post_tick<true, BS>(a, A, N, e, na, 2 * p + 1, cur[1], newp1, prev_val[1], tp[1], tu[1], tc[1], st);
      MDG_PCLK(6 + 4 * p);
    }
  } else {
    // ---- generic path (Composite / sine / trend sources): one asset per iteration
    LazyDraws dr;
    dr.N = N; dr.e = e; dr.gstride = N;
    dr.gid = gid; dr.k0 = k0; dr.k1 = k1; dr.t_lo = t_lo; dr.t_hi = t_hi;
    dr.cached_block = -1;
    dr.normals = a.IO.normals; dr.uniforms = a.IO.uniforms;
    double pair_mean = 0.;
#pragma unroll 1
    for (int i = 0; i < na; ++i) {
      const double price = S.price[(int64_t)i * N + e];
      double cur = S.ledger[(int64_t)i * N + e];
      double mep = S.mean_entry[(int64_t)i * N + e];
      double bm = S.borrowed[(int64_t)i * N + e];
      double units = 0.;
      if (wrow) units = weight_units(wrow[i + 1], w_sum, price, cur, prevEq);
      else if (arow) units = action_units(arow[i], act_half, act_scale, price, cur);
      else if (mode == MDG_MODE_MULTI) units = urow[i];
      else if (mode == MDG_MODE_SINGLE && i == a.L.asset_idx) units = urow[0];
      double tp, tu, tc, prev_val;
      int risk;
      tx_asset<TX2>(a, c, A, N, e, na, i, price, cur, mep, bm, units, tp, tu, tc, risk, prev_val);
      // generator tick of this asset (DataSource.cpp getData family)
      const MdgAssetGen& g = P.gen[i];
      double newp;
      if constexpr (SETS) {  // the same bodies, parameters from this env's set
        const SetParams sp = set_params(static_cast<const StepSetsArgs&>(a).ps, set, i);
        if (g.type == MDG_GEN_OUPAIR) {
          if (g.role == 0) {
            double* mrow = S.gstate + (int64_t)g.gslot * N + e;
            double m = *mrow;
            m += m * (draw_normal(dr, g.nslot_aux) * sp[2]);
            *mrow = m;
            pair_mean = m;
          }
          newp = price + ((sp[0] * (pair_mean - price)) + pair_mean * (draw_normal(dr, g.nslot) * sp[1]));
        } else if (g.type == MDG_GEN_OU) {
          newp = price + ((sp[1] * (sp[0] - price)) + sp[0] * sp[2] * draw_normal(dr, g.nslot));
        } else {
          double* gs = S.gstate + (int64_t)(g.gslot < 0 ? 0 : g.gslot) * N + e;
          newp = gen_tick_sets(g, sp, price, gs, dr, pair_mean);
        }
      } else if (g.type == MDG_GEN_OUPAIR) {  // OUPair::getData :1232-1240 (draw order rw, x0, x1)
        if (g.role == 0) {
          double* mrow = S.gstate + (int64_t)g.gslot * N + e;
          double m = *mrow;
          m += m * (draw_normal(dr, g.nslot_aux) * g.p[2]);
          *mrow = m;
          pair_mean = m;
        }
        newp = price + ((g.p[0] * (pair_mean - price)) + pair_mean * (draw_normal(dr, g.nslot) * g.p[1]));
      } else if (g.type == MDG_GEN_OU) {  // OU::getData :1173-1180
        newp = price + ((g.p[1] * (g.p[0] - price)) + g.p[0] * g.p[2] * draw_normal(dr, g.nslot));
      } else {
        double* gs = S.gstate + (int64_t)(g.gslot < 0 ? 0 : g.gslot) * N + e;
        newp = gen_tick(g, price, gs, dr, pair_mean, P.gen_ext);
      }
      post_tick<false, BS>(a, A, N, e, na, i, cur, newp, prev_val, tp, tu, tc, st);
    }
  }

  const double cash = A.cash, nav = A.nav, pml = A.pml, pbm = A.pbm, pse = A.pse, maintM = c.maintM(a);
  MDG_PCLK(39);
  const int head = a.L.head;
  // BrokerResponse.marginCall (Broker.cpp:135,156): Portfolio::checkRisk() after the last transaction
  if (mode != MDG_MODE_HOLD) a.IO.margin_call[e] = margin_call(cash, A.pav, pml, pbm, pse, maintM) ? 1 : 0;
  gst(&S.cash[e], cash);
  gst(&S.timestamp[e], ts + 1);
  gst(&S.folds[(int64_t)MDG_FOLD_AV * N + e], nav);
  gst(&S.folds[(int64_t)MDG_FOLD_ML * N + e], pml);
  gst(&S.folds[(int64_t)MDG_FOLD_BM * N + e], pbm);
  gst(&S.folds[(int64_t)MDG_FOLD_SE * N + e], pse);
  gst(&S.folds[(int64_t)MDG_FOLD_G * N + e], fabs(cash) + A.gsum);
  const bool bad_risk = A.bad_risk;

  // ---- equity, reward, done (Env.h:192-198, 211-223, 237-249)
  const double currentEq = cash + nav - pbm;
  const double clampv = (mode == MDG_MODE_SINGLE) ? 0.01 : 0.3;
  gst(&a.IO.reward[e], fast_log(dmax(currentEq / prevEq, clampv)));
  const bool mc = margin_call(cash, nav, pml, pbm, pse, maintM);
  bool done = mc || (currentEq < 0.1 * c.init_cash(a));
  if (mode != MDG_MODE_HOLD) done = done || bad_risk;
  a.IO.done[e] = done ? 1 : 0;
  if (a.done_count) {  // auto-reset: finished envs append themselves to the reset list (warp-aggregated)
    const unsigned am = __activemask();
    const unsigned ballot = __ballot_sync(am, done);
    if (ballot) {
      const int lane = tid & 31, leader_lane = __ffs(ballot) - 1;
      int base = 0;
      if (lane == leader_lane) base = atomicAdd(a.done_count, __popc(ballot));
      base = __shfl_sync(am, base, leader_lane);
      if (done) a.done_list[base + __popc(ballot & ((1u << lane) - 1u))] = (int)e;
    }
  }

  // ---- State.portfolio row = ledgerNormedFull (Portfolio.cpp:150-155).  Observations carry a 1e-9 bar
  // (not bit-exactness): the nA+1 divisions by equity are one reciprocal and nA+1 multiplies.
  const double inv_eq = 1. / currentEq;
  const bool cosine = shaping && a.R.shaper == MDG_SHAPER_COSINE;
  double cosv_pp = 0., cosv_qq = 0., cosv_pq = 0.;
  {
    const double w0 = (cash - pbm) * inv_eq;
    gst(&a.IO.obs_port[((int64_t)head * (na + 1)) * N + e], w0);
    if (cosine) {
      const double d0 = a.R.desired_portfolio[0];
      cosv_pp = w0 * w0; cosv_qq = d0 * d0; cosv_pq = w0 * d0;
    }
  }
  const int ra = a.R.reduce_rewards ? 1 : na;
  const double inv_prev = A.inv_prev;
  const int len_before = (shaping && a.R.nstep > 1) ? S.nstep_len[e] : 0;
  int len_after = 0, n_popped = 0;
  double rsum = 0., rprod = 1.;
#pragma unroll kTailUnroll
  for (int j = 0; j < na; ++j) {
    const double cur_val = st[stash_cur_row<PAIRS>(j, na) * BS];
    const double w = cur_val * inv_eq;
    gst(&a.IO.obs_port[((int64_t)head * (na + 1) + j + 1) * N + e], w);
    if (cosine) {
      const double dj = a.R.desired_portfolio[j + 1];
      cosv_pp = cosv_pp + w * w; cosv_qq = cosv_qq + dj * dj; cosv_pq = cosv_pq + w * dj;
    }
    if (shaping && !cosine && !A.reduce_inloop) {  // per-asset agent rewards (offpolicy_q.py:152-164); cosine: below
      double x = (cur_val - st[stash_pm_row<PAIRS>(j, na) * BS]) * inv_prev;
      x += 1;
      const double r = fast_log((x != x) ? x : ((x < .35) ? .35 : x));
      gst(&a.IO.agent_reward[(int64_t)j * N + e], r);
      shaper_add(a, e, j, ra, r, done, len_before, len_after, n_popped);
    }
  }
  // reduced reward: sum_j log(x_j) as log(prod_j x_j) -- one log instead of nA (each x_j is in [.35, ~1.x] and
  // nA <= 16, so the product neither overflows nor underflows; the two differ by ~1e-15 absolute, rewards carry
  // the 1e-9 bar)
  if (A.reduce_inloop) rsum = fast_log(A.rprod);
  if (cosine) {  // the PPC term needs the whole portfolio row first (nstep_buffer.py:173-191)
    const double extra = a.R.cosine_temp * (cosv_pq / (sqrt(cosv_pp) * sqrt(cosv_qq)));
#pragma unroll 1
    for (int j = 0; j < na; ++j) {
      double x = (st[stash_cur_row<PAIRS>(j, na) * BS] - st[stash_pm_row<PAIRS>(j, na) * BS]) * inv_prev;
      x += 1;
      x = (x != x) ? x : ((x < .35) ? .35 : x);
      if (a.R.reduce_rewards) {
        rprod = (j == 0) ? x : rprod * x;
      } else {
        const double r = fast_log(x);
        gst(&a.IO.agent_reward[(int64_t)j * N + e], r);
        shaper_add(a, e, j, ra, r + extra, done, len_before, len_after, n_popped);
      }
    }
    if (a.R.reduce_rewards) {
      rsum = fast_log(rprod);
      gst(&a.IO.agent_reward[e], rsum);
      shaper_add(a, e, 0, 1, rsum + extra, done, len_before, len_after, n_popped);
    }
  } else if (inline_shaper) {  // nstep == 1: add, pop at once (shaper_add / shaper_pop with len == n == 1, same arithmetic)
    gst(&a.IO.agent_reward[e], rsum);
    double sh;
    const double d0 = a.R.discounts[0];
    if (a.R.shaper == MDG_SHAPER_DSR) {         // nstep_buffer.py:62-91
      sh = d0 * dsr_value(shA, shB, rsum);
      sh = sh / 1;
      const double dA = rsum - shA, dB = rsum * rsum - shB;
      shA += a.R.adaptation_rate * dA;
      shB += a.R.adaptation_rate * dB;
      sh = clip(sh, -1., 1.);
    } else if (a.R.shaper == MDG_SHAPER_DDR) {  // :128-162
      sh = d0 * ddr_value(shA, shB, rsum);
      sh = sh / 1;
      const double dA = rsum - shA;
      double mneg = rsum < 0. ? rsum : 0.;
      if (rsum != rsum) mneg = rsum;
      const double dB = mneg * mneg - shB;
      shA += a.R.adaptation_rate * dA;
      shB += a.R.adaptation_rate * dB;
      sh = clip(sh, -1., 1.);
    } else {                                     // sum_default :23-27
      sh = 0.;
      sh = sh + d0 * rsum;
    }
    gst(&a.IO.shaped_reward[e], sh);
    n_popped = 1;
    if (moments) { gst(&a.S.shaper_A[e], shA); gst(&a.S.shaper_B[e], shB); }
  } else if (shaping && a.R.reduce_rewards) {
    gst(&a.IO.agent_reward[e], rsum);
    shaper_add(a, e, 0, 1, rsum, done, len_before, len_after, n_popped);
  }
  if (shaping) {
    if (a.R.nstep > 1) S.nstep_len[e] = len_after;
    a.IO.n_popped[e] = n_popped;
  }
  MDG_PCLK(40);
#ifdef MDG_PHASE_CLOCKS
  if (threadIdx.x == 0 && blockIdx.x < 1024) g_block_ns[blockIdx.x * 4 + 1] = global_ns();
#endif
}

template <bool PAIRS, int BS, int MINB, bool ACTIONS, bool BULK = false>
__global__ void __launch_bounds__(BS, MINB) step_kernel(const __grid_constant__ StepArgs a) {
#ifndef MDG_BULK_TX2
#define MDG_BULK_TX2 0
#endif
  step_body<PAIRS, BS, ACTIONS, (MINB < 4) || (BULK && MDG_BULK_TX2), BULK>(a);  // MINB 3 = the multi-wave register budget
}

// the same instantiations for the launches with parameter sets (mdg_step_sets): 128-thread blocks only
template <bool PAIRS, int BS, int MINB, bool ACTIONS, bool BULK = false>
__global__ void __launch_bounds__(BS, MINB) step_sets_kernel(const __grid_constant__ StepSetsArgs a) {
  step_body<PAIRS, BS, ACTIONS, (MINB < 4) || (BULK && MDG_BULK_TX2), BULK, true>(a);
}
// ... and with broker sets (mdg_step_sets_broker)
template <bool PAIRS, int BS, int MINB, bool ACTIONS, bool BULK = false>
__global__ void __launch_bounds__(BS, MINB) step_sets_broker_kernel(const __grid_constant__ StepSetsBrokerArgs a) {
  step_body<PAIRS, BS, ACTIONS, (MINB < 4) || (BULK && MDG_BULK_TX2), BULK, true, true>(a);
}

// 64-thread blocks, seven per SM (one-wave launches): at 128 registers (registers are granted per warp in units that make 136 or 144 x 14 warps overflow the file: measured two waves)
#ifndef MDG_BS64_REGS
#define MDG_BS64_REGS 128
#endif
template <bool ACTIONS, bool BULK>
__global__ void __maxnreg__(MDG_BS64_REGS) step_kernel64(const __grid_constant__ StepArgs a) {
  step_body<true, 64, ACTIONS, false, BULK>(a);
}

// host side: is every asset part of an OUPair laid out (role0, role1) with in-order noise slots?
static inline bool all_ou_pairs(const MdgParams& P) {
  if (P.n_assets % 2) return false;
  for (int i = 0; i < P.n_assets; i += 2) {
    const MdgAssetGen &g0 = P.gen[i], &g1 = P.gen[i + 1];
    const int s = 3 * (i / 2);
    if (g0.type != MDG_GEN_OUPAIR || g1.type != MDG_GEN_OUPAIR || g0.role != 0 || g1.role != 1 ||
        g1.partner != i || g0.gslot < 0 || g0.nslot_aux != s || g0.nslot != s + 1 || g1.nslot != s + 2)
      return false;
  }
  return P.n_normals == 3 * (P.n_assets / 2);
}

// generator groups of a parameter set: an OUPair (role 0 followed by its role 1) is one group, every other asset its own
static inline int fill_groups(const MdgParams& P, int8_t* leader) {
  int n = 0;
  for (int i = 0; i < P.n_assets; ++i)
    if (!(P.gen[i].type == MDG_GEN_OUPAIR && P.gen[i].role == 1)) leader[n++] = (int8_t)i;
  return n;
}

// ---- tensor maps of the TMA staging path (driver entry point through the runtime: no -lcuda) --------------
typedef CUresult (*StepEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static inline StepEncodeTiledFn step_tensor_map_encoder() {
  static const StepEncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (StepEncodeTiledFn)p;
  }();
  return fn;
}
// Encoding a map costs about a microsecond of host time: a launch's maps depend only on (base, spacing, N, nA), which
// repeat from step to step, so the last few are kept per host thread.
struct StepMapKey {
  const void* base;
  int64_t spacing, N;
  int nA, kind, bs;
  bool operator==(const StepMapKey& o) const {
    return base == o.base && spacing == o.spacing && N == o.N && nA == o.nA && kind == o.kind && bs == o.bs;
  }
};
static inline bool step_tensor_map(const StepMapKey& k, CUtensorMap* out) {
  constexpr int kSlots = 32;
  thread_local StepMapKey keys[kSlots];
  thread_local CUtensorMap maps[kSlots];
  thread_local int used = 0, next = 0;
  for (int i = 0; i < used; ++i)
    if (keys[i] == k) { *out = maps[i]; return true; }
  StepEncodeTiledFn enc = step_tensor_map_encoder();
  if (!enc) return false;
  CUtensorMap m;
  CUresult cr;
  if (k.kind == 0) {  // state slab: N x nA x 4 tensors, box 128 x 2 x 4
    const cuuint64_t gdim[3] = {(cuuint64_t)k.N, (cuuint64_t)k.nA, 4};
    const cuuint64_t gstr[2] = {(cuuint64_t)k.N * sizeof(double), (cuuint64_t)k.spacing};
    const cuuint32_t box[3] = {(cuuint32_t)k.bs, 2, 4}, estr[3] = {1, 1, 1};
    cr = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<void*>(k.base), gdim, gstr, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  } else {  // units (N, nA) env-major: nA x N, box 2 x 128
    const cuuint64_t gdim[2] = {(cuuint64_t)k.nA, (cuuint64_t)k.N};
    const cuuint64_t gstr[1] = {(cuuint64_t)k.nA * sizeof(double)};
    const cuuint32_t box[2] = {2, (cuuint32_t)k.bs}, estr[2] = {1, 1};
    cr = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void*>(k.base), gdim, gstr, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (cr != CUDA_SUCCESS) return false;
  const int slot = used < kSlots ? used++ : (next = (next + 1) % kSlots);
  keys[slot] = k;
  maps[slot] = m;
  *out = m;
  return true;
}

// one 128-thread instantiation of the step kernel, with or without parameter sets (and broker sets)
template <bool SETS, bool BROKER, bool PAIRS, int MINB, bool ACT, bool BULK, class Args>
static inline void launch_step128(const Args& a, unsigned grid, size_t smem, cudaStream_t st) {
  if constexpr (BROKER) step_sets_broker_kernel<PAIRS, 128, MINB, ACT, BULK><<<grid, 128, smem, st>>>(a);
  else if constexpr (SETS) step_sets_kernel<PAIRS, 128, MINB, ACT, BULK><<<grid, 128, smem, st>>>(a);
  else step_kernel<PAIRS, 128, MINB, ACT, BULK><<<grid, 128, smem, st>>>(a);
}

// Args: StepArgs, StepSetsArgs with SETS, or StepSetsBrokerArgs with SETS and BROKER
template <bool SETS = false, bool BROKER = false, class Args = StepArgs>
static inline int launch_step(Args& a) {
  const int64_t N = a.L.n_envs;
  cudaStream_t st = (cudaStream_t)a.L.stream;
  const bool pairs = all_ou_pairs(a.P);
  a.c_reqM = a.P.required_margin;
  a.c_maintM = a.P.maintenance_margin;
  a.c_reqM_ok = (a.c_reqM > 0. && a.c_reqM <= 1e6) ? 1 : 0;
  a.c_band_scale = 1e-9 * (1. + fabs(a.c_maintM)) * (a.c_reqM > 1. ? a.c_reqM : 1.);
  a.c_g1 = 6. + 3. * fabs(a.P.slippage_rel) + fabs(a.P.tcost_rel);
  a.c_g2 = 3. * fabs(a.P.slippage_abs);
  a.c_force_exact = (a.L.flags & MDG_FLAG_FORCE_EXACT_GATE) ? 1 : 0;

  a.units_v2 = (a.IO.units && (reinterpret_cast<uintptr_t>(a.IO.units) & 15) == 0 && a.P.n_assets % 2 == 0) ? 1 : 0;
  static const int bulk_off = [] { const char* v = getenv("MDG_NO_BULK"); return v ? atoi(v) : 0; }();
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  const bool small = N <= 148 * 512 * 2;  // up to two waves at 4 blocks per SM
  // Staging of the pairs' state through shared memory (see step_body).  bulk = 2 (TMA tensor copies: one 3-D box for
  // the eight state rows, one 2-D box for the units, needs the four state tensors equally spaced): 37.2 us against
  // 39.4 us at 65,536 envs per launch, 426 against 437 us at 1,048,576.  bulk = 1 (nine row copies, any layout):
  // neutral in the one-wave variant, 4 % slower in the multi-wave one, so only used in the former.
  // MDG_BS64=1 (profiling knob): one-wave launches with 64-thread blocks, seven per SM.  65,536 envs are 2,048 warps,
  // 13.8 per SM; 128-thread blocks put 16 warps on 68 of the SMs and 12 on the rest, 64-thread blocks 14 on nearly all.
  // Measured (profiles/block_times.py, r2_notes.md): the launch still ends with the youngest block of the fullest SMs
  // at ~30.5 us either way; 36.2 against 37.1 us for a lone launch, no difference inside bench.py -- not the default.
  static const int bs64_on = [] { const char* v = getenv("MDG_BS64"); return v ? atoi(v) : 0; }();
  const int bs = (!SETS && pairs && bs64_on && N <= 148 * 7 * 64) ? 64 : 128;  // no 64-thread sets instantiation
  const unsigned grid = (unsigned)((N + bs - 1) / bs);
  a.bulk = (pairs && !bulk_off && N % bs == 0 && al16(a.S.price) && al16(a.S.ledger) && al16(a.S.mean_entry) &&
            al16(a.S.borrowed) && al16(a.S.gstate)) ? 1 : 0;
  a.tma_units = 0;
  static const int tma_off = [] { const char* v = getenv("MDG_NO_TMA"); return v ? atoi(v) : 0; }();
  if (a.bulk && !tma_off) {
    // the four state tensors as ONE 3-D tensor: they have to be equally spaced (Env allocates them as one slab)
    const char *p0 = (const char*)a.S.price, *p1 = (const char*)a.S.ledger, *p2 = (const char*)a.S.mean_entry,
               *p3 = (const char*)a.S.borrowed;
    const int64_t sp = p1 - p0;
    if (sp >= (int64_t)a.P.n_assets * N * 8 && (sp & 15) == 0 && p2 - p1 == sp && p3 - p2 == sp && N <= 0x7fffffff &&
        step_tensor_map(StepMapKey{a.S.price, sp, N, a.P.n_assets, 0, bs}, &a.tm_state)) {
      a.bulk = 2;
      const bool by_units = a.L.mode == MDG_MODE_MULTI && a.IO.units && !a.IO.actions && !a.IO.weights;
      if (by_units && a.units_v2 && step_tensor_map(StepMapKey{a.IO.units, 0, N, a.P.n_assets, 1, bs}, &a.tm_units))
        a.tma_units = 1;
    }
  }
  if (a.bulk == 1 && !small) a.bulk = 0;
  const size_t smem = sizeof(double) * 2 * (size_t)a.P.n_assets * bs +
                      (a.bulk ? sizeof(double) * kBulkStages * kStageRows * bs + 16 : 0);
  if (smem > 48 * 1024) {  // the bulk ring lifts the all-pairs kernels above the default dynamic shared-memory limit
    static const cudaError_t attr = [] {
      cudaError_t e_ = cudaSuccess;
      auto set = [&](const void* f) {
        const cudaError_t r_ = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, 56 * 1024);
        if (r_ != cudaSuccess) e_ = r_;
      };
      if constexpr (BROKER) {
        set((const void*)step_sets_broker_kernel<true, 128, 4, true, true>);
        set((const void*)step_sets_broker_kernel<true, 128, 4, false, true>);
        set((const void*)step_sets_broker_kernel<true, 128, 3, true, true>);
        set((const void*)step_sets_broker_kernel<true, 128, 3, false, true>);
      } else if constexpr (SETS) {
        set((const void*)step_sets_kernel<true, 128, 4, true, true>);
        set((const void*)step_sets_kernel<true, 128, 4, false, true>);
        set((const void*)step_sets_kernel<true, 128, 3, true, true>);
        set((const void*)step_sets_kernel<true, 128, 3, false, true>);
      } else {
        set((const void*)step_kernel<true, 128, 4, true, true>); set((const void*)step_kernel<true, 128, 4, false, true>);
        set((const void*)step_kernel<true, 128, 3, true, true>); set((const void*)step_kernel<true, 128, 3, false, true>);
      }
      return e_;
    }();
    if (attr != cudaSuccess) return cuda_err(attr, "mdg_step shared-memory opt-in");
  }
  const bool acts = a.L.mode == MDG_MODE_MULTI && (a.IO.actions || a.IO.weights);
#define MDG_LAUNCH(PAIRS_, MINB_, ACT_, BULK_) launch_step128<SETS, BROKER, PAIRS_, MINB_, ACT_, BULK_>(a, grid, smem, st)
  if (bs == 64) {
    if constexpr (!SETS) {
      if (a.bulk) {
        if (acts) step_kernel64<true, true><<<grid, 64, smem, st>>>(a);
        else step_kernel64<false, true><<<grid, 64, smem, st>>>(a);
      } else {
        if (acts) step_kernel64<true, false><<<grid, 64, smem, st>>>(a);
        else step_kernel64<false, false><<<grid, 64, smem, st>>>(a);
      }
    }
  } else if (small && a.bulk) {
    if (acts) MDG_LAUNCH(true, 4, true, true);
    else MDG_LAUNCH(true, 4, false, true);
  } else if (a.bulk) {
    if (acts) MDG_LAUNCH(true, 3, true, true);
    else MDG_LAUNCH(true, 3, false, true);
  } else if (small) {
    if (pairs) { if (acts) MDG_LAUNCH(true, 4, true, false); else MDG_LAUNCH(true, 4, false, false); }
    else { if (acts) MDG_LAUNCH(false, 4, true, false); else MDG_LAUNCH(false, 4, false, false); }
  } else {
    if (pairs) { if (acts) MDG_LAUNCH(true, 3, true, false); else MDG_LAUNCH(true, 3, false, false); }
    else { if (acts) MDG_LAUNCH(false, 3, true, false); else MDG_LAUNCH(false, 3, false, false); }
  }
#undef MDG_LAUNCH
  return cuda_err(cudaGetLastError(), "mdg_step launch");
}

}  // namespace mdg
