// extern "C" entry points of the step path + the (rare, non-unrolled) reset / init kernels.
#include <stdlib.h>

#include <atomic>

#include "mdg_step_kernel.cuh"

namespace mdg {

char* err_buf() {
  thread_local static char buf[512] = "";
  return buf;
}

// ---------------------------------------------------------------------------
// reset: Env::reset (Env.h:181-187) + StackerDiscrete.initialize_history (preprocessor.py:191-194)
// ---------------------------------------------------------------------------
struct ResetArgs {
  MdgParams P;
  MdgState S;
  MdgStepIO IO;
  MdgLaunch L;
  const uint8_t* mask;
  int fill_ticks;
  int clear_nstep;
};

// Envs that reset are rare and scattered, and each must fast-forward fill_ticks generator ticks
// (A17: a reset consumes k ticks).  One thread per env would leave 31 lanes idle for 64 ticks in
// almost every warp, so the block (a) compacts the indices of its resetting envs in shared memory
// and (b) spreads (generator group, env) items over ALL its threads: an OU pair or a single
// asset is an independent stochastic process, and Philox draws are addressed by (env, tick, slot),
// so any lane can compute any group's path.
constexpr int kResetBlock = 256;

__global__ void __launch_bounds__(kResetBlock) reset_kernel(const __grid_constant__ ResetArgs a) {
  __shared__ int s_list[kResetBlock];
  __shared__ long long s_ts[kResetBlock];
  __shared__ int s_leader[MDG_MAX_ASSETS];
  __shared__ int s_count, s_nlead;
  const MdgParams& P = a.P;
  const int64_t N = a.L.n_envs;
  const int tid = threadIdx.x;
  const int64_t e0 = (int64_t)blockIdx.x * kResetBlock;
  const int na = P.n_assets;
  const int k = a.L.window;
  const int fill = a.fill_ticks;
  if (tid == 0) {
    s_count = 0;
    int n = 0;
    for (int i = 0; i < na; ++i)
      if (!(P.gen[i].type == MDG_GEN_OUPAIR && P.gen[i].role == 1)) s_leader[n++] = i;
    s_nlead = n;
  }
  __syncthreads();
  {  // (a) warp-aggregated compaction of the resetting envs of this block
    const int64_t e = e0 + tid;
    const bool flag = (e < N) && (!a.mask || a.mask[e]);
    const unsigned ballot = __ballot_sync(0xffffffffu, flag);
    int base = 0;
    if ((tid & 31) == 0 && ballot) base = atomicAdd(&s_count, __popc(ballot));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (flag) s_list[base + __popc(ballot & ((1u << (tid & 31)) - 1u))] = tid;
  }
  __syncthreads();
  const int nd = s_count;
  if (nd == 0) return;
  const double cash = P.init_cash;
  const double eq = cash + 0. - 0.;  // flat portfolio: equity == cash
  // per-env scalars: fresh Broker/Account/Portfolio (Env.h:150-165), cash weight and timestamps of the rows
  for (int it = tid; it < nd; it += kResetBlock) {
    const int64_t e = e0 + s_list[it];
    if (a.clear_nstep && a.S.nstep_len) a.S.nstep_len[e] = 0;  // offpolicy_q.py:94
    a.S.cash[e] = cash;
    if (a.S.folds) {  // flat portfolio: every fold is a sum of zeros
      a.S.folds[(int64_t)MDG_FOLD_AV * N + e] = 0.;
      a.S.folds[(int64_t)MDG_FOLD_ML * N + e] = 0.;
      a.S.folds[(int64_t)MDG_FOLD_BM * N + e] = 0.;
      a.S.folds[(int64_t)MDG_FOLD_SE * N + e] = 0.;
      a.S.folds[(int64_t)MDG_FOLD_G * N + e] = fabs(cash);
    }
    const long long ts = a.S.timestamp[e];
    s_ts[it] = ts;
    a.S.timestamp[e] = ts + fill;
    a.S.reset_ts[e] = ts + fill;
    a.IO.obs_port[((int64_t)a.L.head * (na + 1)) * N + e] = (cash - 0.) / eq;  // newest row = current state
  }
  __syncthreads();
  // (b) items ordered leader-major so that neighbouring lanes run the same generator type
  const int nitems = nd * s_nlead;
  for (int item = tid; item < nitems; item += kResetBlock) {
    const int l = item / nd, d = item - l * nd;
    const int64_t e = e0 + s_list[d];
    const int i0 = s_leader[l];
    const int cnt = (P.gen[i0].type == MDG_GEN_OUPAIR) ? 2 : 1;
    double pr[2];
    for (int c = 0; c < cnt; ++c) {  // dataSource_->reset() and the empty ledger
      const MdgAssetGen& g = P.gen[i0 + c];
      double* gs = a.S.gstate + (int64_t)(g.gslot < 0 ? 0 : g.gslot) * N + e;
      const CtorDraws cd = ctor_draws((uint32_t)(a.L.env_offset + e), a.L.seed, s_ts[d], 2, i0 + c);
      pr[c] = gen_reset(g, a.S.price[(int64_t)(i0 + c) * N + e], gs, N, P.gen_ext, &cd);
      a.S.ledger[(int64_t)(i0 + c) * N + e] = 0.;
      a.S.mean_entry[(int64_t)(i0 + c) * N + e] = 0.;
      a.S.borrowed[(int64_t)(i0 + c) * N + e] = 0.;
    }
    LazyDraws dr;
    dr.N = N; dr.e = e; dr.gstride = N;
    dr.gid = (uint32_t)(a.L.env_offset + e);
    dr.k0 = (uint32_t)a.L.seed; dr.k1 = (uint32_t)(a.L.seed >> 32);
    const long long ts0 = s_ts[d];
#pragma unroll 1
    for (int t = 0; t < fill; ++t) {
      const long long tick = ts0 + t;
      dr.t_lo = (uint32_t)(unsigned long long)tick;
      dr.t_hi = (uint32_t)((unsigned long long)tick >> 32);
      dr.cached_block = -1;
      dr.normals = a.IO.normals ? a.IO.normals + (int64_t)t * P.n_normals * N : nullptr;
      dr.uniforms = a.IO.uniforms ? a.IO.uniforms + (int64_t)t * P.n_uniforms * N : nullptr;
      double pair_mean = 0.;
#pragma unroll 1
      for (int c = 0; c < cnt; ++c) {
        const MdgAssetGen& g = P.gen[i0 + c];
        double* gs = a.S.gstate + (int64_t)(g.gslot < 0 ? 0 : g.gslot) * N + e;
        pr[c] = gen_tick(g, pr[c], gs, dr, pair_mean, P.gen_ext);
        a.IO.pre_price[((int64_t)e * k + (k - fill + t)) * na + i0 + c] = pr[c];
        if (t == fill - 1) {  // newest row = current state, also in the ring
          a.IO.obs_price[((int64_t)a.L.head * na + i0 + c) * N + e] = pr[c];
          a.IO.obs_port[((int64_t)a.L.head * (na + 1) + i0 + c + 1) * N + e] = (0. * pr[c]) / eq;
        }
      }
    }
    for (int c = 0; c < cnt; ++c) a.S.price[(int64_t)(i0 + c) * N + e] = pr[c];
  }
}

// ---------------------------------------------------------------------------
// reset with a workspace: a list of the resetting envs + ONE refill kernel.
//   list  : built by reset_scan_kernel from a mask (explicit Env.reset) or, on the auto-reset path, by the
//           step kernel itself (its last warp appends the envs whose `done` it has just computed).
//   refill: one block of 128 threads per listed env (grid-stride; the host sizes the grid without knowing the
//           count, blocks past the end of the list exit at once).  Per chunk of <= 64 ticks:
//             phase 1  the dependence-free part -- Philox + Box-Muller of every (tick, block) -- packed over
//                      the 128 threads into shared memory (the normals never touch global memory);
//             phase 2  the serial recurrence of each generator group on neighbouring lanes of warp 0, reading
//                      the normals from shared memory, writing the env's contiguous pre_price rows.
//           Then the fresh Broker/Account/Portfolio (Env.h:150-165), timestamps and the newest ring row.
//   The workspace header {count, ticket} is self-cleaning: the last block to leave zeroes it.
// ---------------------------------------------------------------------------
struct ResetWsArgs {
  MdgParams P;
  MdgState S;
  MdgStepIO IO;
  MdgLaunch L;
  const uint8_t* mask;
  int fill_ticks;
  int clear_nstep;
  int* count;   // workspace header: number of listed envs
  int* ticket;  // workspace header: blocks of the refill kernel that have left
  int* list;    // workspace: env index of each listed env
  int chunk;    // ticks per shared-memory chunk
  int n_groups;
  int8_t leader[MDG_MAX_ASSETS];
  // refill kernel: generator group run by each thread (-1: none).  Groups of one generator type share a warp,
  // different types go to different warps, so that a Composite's 64-tick recurrences do not serialise by type.
  int8_t group_of_thread[128];
};

// the refills of the launches with parameter sets: the table and the assignment after everything the others read
struct ResetWsSetsArgs : ResetWsArgs {
  MdgParamSets ps;
};
// ... with broker sets: the broker table, [MDG_BROKER_NPARAM][n_sets]
struct ResetWsBrokerArgs : ResetWsSetsArgs {
  const double* broker;
};

__global__ void __launch_bounds__(256) reset_scan_kernel(const __grid_constant__ ResetWsArgs a) {
  const int64_t N = a.L.n_envs;
  const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool flag = (e < N) && (!a.mask || a.mask[e]);
  const unsigned ballot = __ballot_sync(0xffffffffu, flag);
  if (!ballot) return;
  int base = 0;
  if (lane == (__ffs(ballot) - 1)) base = atomicAdd(a.count, __popc(ballot));
  base = __shfl_sync(0xffffffffu, base, __ffs(ballot) - 1);
  if (flag) a.list[base + __popc(ballot & ((1u << lane) - 1u))] = (int)e;
}

constexpr int kFillBlock = 128;

template <bool SETS, bool BROKER = false>
__device__ __forceinline__ void reset_fill_body(const ResetWsArgs& a) {
  extern __shared__ double zs[];  // [chunk][n_normals]
  const MdgParams& P = a.P;
  const int tid = threadIdx.x;
  const int na = P.n_assets, nn = P.n_normals, nb = (nn + 1) >> 1;
  const int fill = a.fill_ticks, k = a.L.window, chunk = a.chunk, nlead = a.n_groups;
  const int64_t N = a.L.n_envs;
  const int count = *(volatile int*)a.count;
  const double cash0 = P.init_cash;
  const double eq0 = cash0 + 0. - 0.;              // flat portfolio: equity == cash
  const bool eq_plain0 = eq0 > 0. && eq0 < 1e300;  // then (0*p)/eq == 0*p exactly
  const uint32_t k0 = (uint32_t)a.L.seed, k1 = (uint32_t)(a.L.seed >> 32);
  const uint32_t magic = (uint32_t)((0x100000000ull + (uint32_t)nb - 1) / (uint32_t)(nb > 0 ? nb : 1));  // ceil(2^32 / nb)
  for (int d = blockIdx.x; d < count; d += gridDim.x) {
    const int64_t e = a.list[d];
    const long long ts0 = a.S.timestamp[e];
    int64_t set = 0;  // parameter sets: the listed env's set
    if constexpr (SETS) set = env_set(static_cast<const ResetWsSetsArgs&>(a).ps, e);
    double cash = cash0, eq = eq0;
    bool eq_plain = eq_plain0;
    if constexpr (BROKER) {  // the fresh portfolio's cash from the listed env's set
      const ResetWsBrokerArgs& b = static_cast<const ResetWsBrokerArgs&>(a);
      cash = broker_value(b.broker, b.ps.n_sets, set, MDG_BROKER_INIT_CASH);
      eq = cash + 0. - 0.;
      eq_plain = eq > 0. && eq < 1e300;
    }
    __syncthreads();  // every thread has read the old timestamp (and the previous env's normals are consumed)
    if (tid == 32) {  // fresh Broker/Account/Portfolio (Env.h:150-165): per-env scalars
      if (a.clear_nstep && a.S.nstep_len) a.S.nstep_len[e] = 0;  // offpolicy_q.py:94
      a.S.cash[e] = cash;
      if (a.S.folds) {  // flat portfolio: every fold is a sum of zeros
        a.S.folds[(int64_t)MDG_FOLD_AV * N + e] = 0.;
        a.S.folds[(int64_t)MDG_FOLD_ML * N + e] = 0.;
        a.S.folds[(int64_t)MDG_FOLD_BM * N + e] = 0.;
        a.S.folds[(int64_t)MDG_FOLD_SE * N + e] = 0.;
        a.S.folds[(int64_t)MDG_FOLD_G * N + e] = fabs(cash);
      }
      a.S.timestamp[e] = ts0 + fill;
      a.S.reset_ts[e] = ts0 + fill;
      a.IO.obs_port[((int64_t)a.L.head * (na + 1)) * N + e] = (cash - 0.) / eq;  // newest row = current state
    }
    // generator state of group `tid` (warp 0, lanes < nlead) in registers for the whole fast-forward
    const int grp = a.group_of_thread[tid];
    const bool worker = grp >= 0 && grp < nlead;
    const int i0 = worker ? a.leader[grp] : 0;
    const MdgAssetGen& g0 = P.gen[i0];
    const bool is_pair = g0.type == MDG_GEN_OUPAIR;
    const int cnt = is_pair ? 2 : 1;
    const int ngs_all = gen_state_rows(g0);
    const bool big = ngs_all > 4;  // SINE* sources: the state stays in global memory
    const int ngs = big ? 0 : ngs_all;
    double pr[2] = {0., 0.}, gsl[4] = {0., 0., 0., 0.};
    double* gsg = a.S.gstate + (int64_t)(g0.gslot < 0 ? 0 : g0.gslot) * N + e;
    if (worker) {
      for (int r = 0; r < ngs; ++r) gsl[r] = a.S.gstate[(int64_t)(g0.gslot + r) * N + e];
      for (int c = 0; c < cnt; ++c) pr[c] = a.S.price[(int64_t)(i0 + c) * N + e];
      for (int c = 0; c < cnt; ++c) {  // dataSource_->reset() and the empty ledger
        const CtorDraws cd = ctor_draws((uint32_t)(a.L.env_offset + e), a.L.seed, ts0, 2, i0 + c);
        if constexpr (SETS)  // no SINE* source here: the state is in registers
          pr[c] = gen_reset_p(P.gen[i0 + c], set_params(static_cast<const ResetWsSetsArgs&>(a).ps, set, i0 + c), pr[c],
                              gsl, 1, P.gen_ext, &cd);
        else
          pr[c] = big ? gen_reset(P.gen[i0 + c], pr[c], gsg, N, P.gen_ext, &cd)
                      : gen_reset(P.gen[i0 + c], pr[c], gsl, 1, P.gen_ext, &cd);
        a.S.ledger[(int64_t)(i0 + c) * N + e] = 0.;
        a.S.mean_entry[(int64_t)(i0 + c) * N + e] = 0.;
        a.S.borrowed[(int64_t)(i0 + c) * N + e] = 0.;
      }
    }
    const uint32_t gid = (uint32_t)(a.L.env_offset + e);
    double* prow = a.IO.pre_price + ((int64_t)e * k + (k - fill)) * na + i0;
    for (int t0 = 0; t0 < fill; t0 += chunk) {
      const int nt = (fill - t0) < chunk ? (fill - t0) : chunk;
      if (t0 > 0) __syncthreads();  // the previous chunk's normals are consumed
      // ---- phase 1: this chunk's normals into shared memory
      if (a.IO.normals) {  // validation mode: the injected stream [tick][slot][env]
        for (int j = tid; j < nt * nn; j += kFillBlock) {
          const int t = j / nn, s_ = j - t * nn;
          zs[j] = a.IO.normals[((int64_t)(t0 + t) * nn + s_) * N + e];
        }
      } else {
        for (uint32_t j = tid; j < (uint32_t)(nt * nb); j += kFillBlock) {
          const uint32_t t = (nb == 1) ? j : __umulhi(j, magic);  // j / nb, exact for j < 2^16
          const uint32_t b = j - t * (uint32_t)nb;
          const unsigned long long tick = (unsigned long long)(ts0 + t0) + t;
          double za, zb;
          normal_block(gid, b, (uint32_t)tick, (uint32_t)(tick >> 32), k0, k1, za, zb);
          double* z = zs + t * (uint32_t)nn + 2 * b;
          z[0] = za;
          if (2 * (int)b + 1 < nn) z[1] = zb;
        }
      }
      __syncthreads();
      // ---- phase 2: the serial recurrences, one generator group per lane
      if (worker) {
        if (is_pair) {  // OUPair::getData (DataSource.cpp:1232-1240) inlined
          const MdgAssetGen& g1 = P.gen[i0 + 1];
          double theta0 = g0.p[0], phi0 = g0.p[1], noise = g0.p[2], theta1 = g1.p[0], phi1 = g1.p[1];
          if constexpr (SETS) {
            const MdgParamSets& ps = static_cast<const ResetWsSetsArgs&>(a).ps;
            const SetParams q0 = set_params(ps, set, i0), q1 = set_params(ps, set, i0 + 1);
            theta0 = q0[0]; phi0 = q0[1]; noise = q0[2]; theta1 = q1[0]; phi1 = q1[1];
          }
          const int s_rw = g0.nslot_aux, s_0 = g0.nslot, s_1 = g1.nslot;
          double m = gsl[0];
#pragma unroll 4
          for (int t = 0; t < nt; ++t) {
            const double* zn = zs + t * nn;
            m += m * (zn[s_rw] * noise);
            pr[0] += (theta0 * (m - pr[0])) + m * (zn[s_0] * phi0);
            pr[1] += (theta1 * (m - pr[1])) + m * (zn[s_1] * phi1);
            double* dst = prow + (int64_t)(t0 + t) * na;
            if ((na & 1) == 0) {  // 16-byte aligned: the env's pairs fill whole 128-byte lines together
              *reinterpret_cast<double2*>(dst) = make_double2(pr[0], pr[1]);
            } else {
              dst[0] = pr[0];
              dst[1] = pr[1];
            }
          }
          gsl[0] = m;
        } else {
          TickDraws dr;
          dr.N = N; dr.e = e; dr.gstride = big ? N : 1;
          dr.gid = gid; dr.k0 = k0; dr.k1 = k1;
#pragma unroll 1
          for (int t = 0; t < nt; ++t) {
            const long long tick = ts0 + t0 + t;
            dr.t_lo = (uint32_t)(unsigned long long)tick;
            dr.t_hi = (uint32_t)((unsigned long long)tick >> 32);
            dr.z = zs + t * nn;
            dr.uniforms = a.IO.uniforms ? a.IO.uniforms + (int64_t)(t0 + t) * P.n_uniforms * N : nullptr;
            double pair_mean = 0.;
            if constexpr (SETS)
              pr[0] = gen_tick_sets(g0, set_params(static_cast<const ResetWsSetsArgs&>(a).ps, set, i0), pr[0], gsl, dr,
                                    pair_mean);
            else
              pr[0] = gen_tick(g0, pr[0], big ? gsg : gsl, dr, pair_mean, P.gen_ext);
            prow[(int64_t)(t0 + t) * na] = pr[0];
          }
        }
      }
    }
    if (worker) {
      for (int c = 0; c < cnt; ++c) {  // newest row = current state, also in the ring
        a.IO.obs_price[((int64_t)a.L.head * na + i0 + c) * N + e] = pr[c];
        a.IO.obs_port[((int64_t)a.L.head * (na + 1) + i0 + c + 1) * N + e] = eq_plain ? 0. * pr[c] : (0. * pr[c]) / eq;
      }
      for (int r = 0; r < ngs; ++r) a.S.gstate[(int64_t)(g0.gslot + r) * N + e] = gsl[r];
      for (int c = 0; c < cnt; ++c) a.S.price[(int64_t)(i0 + c) * N + e] = pr[c];
    }
  }
  // self-cleaning header: the last block to leave zeroes the count for the next step kernel
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    const int t = atomicAdd(a.ticket, 1);
    if (t == (int)gridDim.x - 1) {
      *a.count = 0;
      *a.ticket = 0;
      __threadfence();
    }
  }
}
__global__ void __launch_bounds__(kFillBlock) reset_fill_kernel(const __grid_constant__ ResetWsArgs a) {
  reset_fill_body<false>(a);
}
__global__ void __launch_bounds__(kFillBlock) reset_fill_sets_kernel(const __grid_constant__ ResetWsSetsArgs a) {
  reset_fill_body<true>(a);
}
__global__ void __launch_bounds__(kFillBlock) reset_fill_sets_broker_kernel(const __grid_constant__ ResetWsBrokerArgs a) {
  reset_fill_body<true, true>(a);
}

// The refill of the all-OU-pairs parameter sets (all_ou_pairs(P)) when the normals come from Philox: one lane per
// (listed env, pair), np = nA/2 lanes per env, 128/np envs per block.  A pair is an independent process whose three
// normals per tick (slots 3p, 3p+1, 3p+2) are two Philox blocks, so every lane draws its own normals in registers and
// runs its pair's recurrence without shared memory or a barrier inside the tick loop; the tick loop is unrolled so that
// the next ticks' Philox overlaps the current tick's dependent chain.  (Pairs 2q and 2q+1 share block 3q+1: measured,
// swapping its halves between the two lanes beats drawing it twice, profiles/r3_notes.md.)  The draws, the recurrence
// and the stores are reset_fill_kernel's expression for expression (same translation unit, same -fmad=false), so the
// two kernels write bit-identical results.
// -DMDG_FILL_PAIRS_UNROLL / -DMDG_FILL_PAIRS_MINB (profiling builds): tick-loop unroll and the minimum resident blocks
// per SM the register budget is sized for
#ifndef MDG_FILL_PAIRS_UNROLL
#define MDG_FILL_PAIRS_UNROLL 4
#endif
#ifndef MDG_FILL_PAIRS_MINB
#define MDG_FILL_PAIRS_MINB 1
#endif
constexpr int kFillPairsUnroll = MDG_FILL_PAIRS_UNROLL;
template <bool SETS, bool BROKER = false>
__device__ __forceinline__ void reset_fill_pairs_body(const ResetWsArgs& a) {
  const MdgParams& P = a.P;
  const int tid = threadIdx.x;
  const int na = P.n_assets, np = na >> 1, epb = kFillBlock / np;
  const int slot = tid / np, p = tid - slot * np;  // env of the group, pair of the env
  const int fill = a.fill_ticks, k = a.L.window;
  const int64_t N = a.L.n_envs;
  const int listed = *(volatile int*)a.count;
  const int count = (int64_t)listed < N ? listed : (int)N;  // a stale header cannot index past the list
  const double cash0 = P.init_cash;
  const double eq0 = cash0 + 0. - 0.;              // flat portfolio: equity == cash
  const bool eq_plain0 = eq0 > 0. && eq0 < 1e300;  // then (0*p)/eq == 0*p exactly
  const uint32_t k0 = (uint32_t)a.L.seed, k1 = (uint32_t)(a.L.seed >> 32);
  const int i0 = 2 * p;
  const MdgAssetGen &g0 = P.gen[i0], &g1 = P.gen[i0 + 1];
  double theta0 = g0.p[0], phi0 = g0.p[1], noise = g0.p[2], theta1 = g1.p[0], phi1 = g1.p[1];  // SETS: per env below
  // slot s = Philox block s>>1, output s&1: pair p reads blocks b and b+1, b = 3p>>1
  const uint32_t blk = (uint32_t)(3 * p) >> 1;
  const bool odd = p & 1;
  for (int d0 = blockIdx.x * epb; d0 < count; d0 += gridDim.x * epb) {
    const int d = d0 + slot;
    const bool active = slot < epb && d < count;
    const int64_t e = active ? a.list[d] : 0;
    const long long ts0 = active ? a.S.timestamp[e] : 0;
    double cash = cash0, eq = eq0;
    bool eq_plain = eq_plain0;
    if constexpr (SETS) {  // this lane's pair in the listed env's set (idle lanes read env 0's, and store nothing)
      const MdgParamSets& ps = static_cast<const ResetWsSetsArgs&>(a).ps;
      const int64_t set = env_set(ps, e);
      const SetParams q0 = set_params(ps, set, i0), q1 = set_params(ps, set, i0 + 1);
      theta0 = q0[0]; phi0 = q0[1]; noise = q0[2]; theta1 = q1[0]; phi1 = q1[1];
      if constexpr (BROKER) {  // the fresh portfolio's cash from the set too
        cash = broker_value(static_cast<const ResetWsBrokerArgs&>(a).broker, ps.n_sets, set, MDG_BROKER_INIT_CASH);
        eq = cash + 0. - 0.;
        eq_plain = eq > 0. && eq < 1e300;
      }
    }
    __syncthreads();  // every lane of an env has read the old timestamp before its pair-0 lane writes the new one
    // idle lanes run the tick loop too (without storing): the loop's shuffles take every lane of the warp
    if (active && p == 0) {  // fresh Broker/Account/Portfolio (Env.h:150-165): per-env scalars
      if (a.clear_nstep && a.S.nstep_len) a.S.nstep_len[e] = 0;  // offpolicy_q.py:94
      a.S.cash[e] = cash;
      if (a.S.folds) {  // flat portfolio: every fold is a sum of zeros
        a.S.folds[(int64_t)MDG_FOLD_AV * N + e] = 0.;
        a.S.folds[(int64_t)MDG_FOLD_ML * N + e] = 0.;
        a.S.folds[(int64_t)MDG_FOLD_BM * N + e] = 0.;
        a.S.folds[(int64_t)MDG_FOLD_SE * N + e] = 0.;
        a.S.folds[(int64_t)MDG_FOLD_G * N + e] = fabs(cash);
      }
      a.S.timestamp[e] = ts0 + fill;
      a.S.reset_ts[e] = ts0 + fill;
      a.IO.obs_port[((int64_t)a.L.head * (na + 1)) * N + e] = (cash - 0.) / eq;  // newest row = current state
    }
    for (int c = 0; c < 2 && active; ++c) {  // the empty ledger
      a.S.ledger[(int64_t)(i0 + c) * N + e] = 0.;
      a.S.mean_entry[(int64_t)(i0 + c) * N + e] = 0.;
      a.S.borrowed[(int64_t)(i0 + c) * N + e] = 0.;
    }
    // OUPair::reset (gen_reset, DataSource.cpp:1242-1246) draws nothing: the shared mean and both prices restart at 10
    double m = 10., pr0 = 10., pr1 = 10.;
    const uint32_t gid = (uint32_t)(a.L.env_offset + e);
    double2* prow = reinterpret_cast<double2*>(a.IO.pre_price + ((int64_t)e * k + (k - fill)) * na) + p;
    auto tick = [&](int t, double z_rw, double z_0, double z_1) {  // OUPair::getData (DataSource.cpp:1232-1240)
      m += m * (z_rw * noise);
      pr0 += (theta0 * (m - pr0)) + m * (z_0 * phi0);
      pr1 += (theta1 * (m - pr1)) + m * (z_1 * phi1);
      if (active) prow[(int64_t)t * np] = make_double2(pr0, pr1);  // a warp's tick: 128 contiguous bytes per env
    };
    int t = 0;
    if ((np & 1) == 0) {
      // pairs 2q and 2q+1 sit on neighbouring lanes of one warp and share Philox block 3q+1: of two ticks, the even
      // lane draws it for the first and the odd lane for the second, and each hands the other the half it needs
      const uint32_t b_own = odd ? blk + 1 : blk, b_sh = odd ? blk : blk + 1;
#pragma unroll kFillPairsUnroll / 2
      for (; t + 1 < fill; t += 2) {
        const unsigned long long ta = (unsigned long long)ts0 + (unsigned)t, tb = ta + 1, tsh = odd ? tb : ta;
        double oa0, oa1, ob0, ob1, s0, s1;
        normal_block(gid, b_own, (uint32_t)ta, (uint32_t)(ta >> 32), k0, k1, oa0, oa1);
        normal_block(gid, b_own, (uint32_t)tb, (uint32_t)(tb >> 32), k0, k1, ob0, ob1);
        normal_block(gid, b_sh, (uint32_t)tsh, (uint32_t)(tsh >> 32), k0, k1, s0, s1);
        const double recv = __shfl_xor_sync(0xffffffffu, odd ? s0 : s1, 1);
        const double sa = odd ? recv : s0, sb = odd ? s1 : recv;  // this lane's half of the shared block
        tick(t, odd ? sa : oa0, odd ? oa0 : oa1, odd ? oa1 : sa);
        tick(t + 1, odd ? sb : ob0, odd ? ob0 : ob1, odd ? ob1 : sb);
      }
    }
#pragma unroll kFillPairsUnroll
    for (; t < fill; ++t) {  // an odd number of pairs, or the last of an odd number of ticks: both blocks per lane
      const unsigned long long tk = (unsigned long long)ts0 + (unsigned)t;
      double l0, l1, h0, h1;
      normal_block(gid, blk, (uint32_t)tk, (uint32_t)(tk >> 32), k0, k1, l0, l1);
      normal_block(gid, blk + 1, (uint32_t)tk, (uint32_t)(tk >> 32), k0, k1, h0, h1);
      tick(t, odd ? l1 : l0, odd ? h0 : l1, odd ? h1 : h0);
    }
    if (!active) continue;
    a.IO.obs_price[((int64_t)a.L.head * na + i0) * N + e] = pr0;  // newest row = current state, also in the ring
    a.IO.obs_price[((int64_t)a.L.head * na + i0 + 1) * N + e] = pr1;
    a.IO.obs_port[((int64_t)a.L.head * (na + 1) + i0 + 1) * N + e] = eq_plain ? 0. * pr0 : (0. * pr0) / eq;
    a.IO.obs_port[((int64_t)a.L.head * (na + 1) + i0 + 2) * N + e] = eq_plain ? 0. * pr1 : (0. * pr1) / eq;
    a.S.gstate[(int64_t)g0.gslot * N + e] = m;
    a.S.price[(int64_t)i0 * N + e] = pr0;
    a.S.price[(int64_t)(i0 + 1) * N + e] = pr1;
  }
  // self-cleaning header: the last block to leave zeroes the count for the next step kernel
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    const int t = atomicAdd(a.ticket, 1);
    if (t == (int)gridDim.x - 1) {
      *a.count = 0;
      *a.ticket = 0;
      __threadfence();
    }
  }
}
__global__ void __launch_bounds__(kFillBlock, MDG_FILL_PAIRS_MINB) reset_fill_pairs_kernel(const __grid_constant__ ResetWsArgs a) {
  reset_fill_pairs_body<false>(a);
}
__global__ void __launch_bounds__(kFillBlock, MDG_FILL_PAIRS_MINB)
    reset_fill_pairs_sets_kernel(const __grid_constant__ ResetWsSetsArgs a) {
  reset_fill_pairs_body<true>(a);
}
__global__ void __launch_bounds__(kFillBlock, MDG_FILL_PAIRS_MINB)
    reset_fill_pairs_sets_broker_kernel(const __grid_constant__ ResetWsBrokerArgs a) {
  reset_fill_pairs_body<true, true>(a);
}

// constructor state (Env.h:139-165 before the first tick)
struct InitArgs {
  MdgParams P;
  MdgReward R;
  MdgState S;
  MdgLaunch L;
};
struct InitSetsArgs : InitArgs {
  MdgParamSets ps;
};
struct InitBrokerArgs : InitSetsArgs {
  const double* broker;
};
// e: computed in the kernels, where the compiler knows the range of threadIdx.x
template <bool SETS, bool BROKER = false>
__device__ __forceinline__ void init_body(const InitArgs& a, int64_t e) {
  const int64_t N = a.L.n_envs;
  if (e >= N) return;
  const int na = a.P.n_assets;
  for (int i = 0; i < na; ++i) {
    const MdgAssetGen& g = a.P.gen[i];
    double* gs = a.S.gstate + (int64_t)(g.gslot < 0 ? 0 : g.gslot) * N + e;
    const CtorDraws cd = ctor_draws((uint32_t)(a.L.env_offset + e), a.L.seed, 0, 3, i);
    if constexpr (SETS) {  // start values (OU mean, Synth phase, trend start) from the env's set
      const MdgParamSets& ps = static_cast<const InitSetsArgs&>(a).ps;
      a.S.price[(int64_t)i * N + e] = gen_start_p(g, set_params(ps, env_set(ps, e), i), gs, N, a.P.gen_ext, &cd);
    } else {
      a.S.price[(int64_t)i * N + e] = gen_start(g, gs, N, a.P.gen_ext, &cd);
    }
    a.S.ledger[(int64_t)i * N + e] = 0.;
    a.S.mean_entry[(int64_t)i * N + e] = 0.;
    a.S.borrowed[(int64_t)i * N + e] = 0.;
  }
  double cash = a.P.init_cash;
  if constexpr (BROKER) {  // the env's set's starting cash
    const InitBrokerArgs& b = static_cast<const InitBrokerArgs&>(a);
    cash = broker_value(b.broker, b.ps.n_sets, env_set(b.ps, e), MDG_BROKER_INIT_CASH);
  }
  a.S.cash[e] = cash;
  a.S.timestamp[e] = 0;
  if (a.S.reset_ts) a.S.reset_ts[e] = 0;
  if (a.S.folds) {
    for (int r = 0; r < 4; ++r) a.S.folds[(int64_t)r * N + e] = 0.;
    a.S.folds[(int64_t)MDG_FOLD_G * N + e] = fabs(cash);
  }
  const int ra = a.R.reduce_rewards ? 1 : na;
  for (int c = 0; c < ra; ++c) {
    if (a.S.shaper_A) a.S.shaper_A[(int64_t)c * N + e] = 0.;
    if (a.S.shaper_B) a.S.shaper_B[(int64_t)c * N + e] = 0.;
  }
  if (a.S.nstep_len) a.S.nstep_len[e] = 0;
}
__global__ void __launch_bounds__(128) init_kernel(const __grid_constant__ InitArgs a) {
  init_body<false>(a, (int64_t)blockIdx.x * 128 + threadIdx.x);
}
__global__ void __launch_bounds__(128) init_sets_kernel(const __grid_constant__ InitSetsArgs a) {
  init_body<true>(a, (int64_t)blockIdx.x * 128 + threadIdx.x);
}
__global__ void __launch_bounds__(128) init_sets_broker_kernel(const __grid_constant__ InitBrokerArgs a) {
  init_body<true, true>(a, (int64_t)blockIdx.x * 128 + threadIdx.x);
}

// exact left-to-right folds of the portfolio as stored (after external writes into the state tensors)
struct FoldArgs {
  MdgParams P;
  MdgState S;
  int64_t N;
};
__global__ void __launch_bounds__(128) refresh_folds_kernel(const __grid_constant__ FoldArgs a) {
  const int64_t N = a.N;
  const int64_t e = (int64_t)blockIdx.x * 128 + threadIdx.x;
  if (e >= N) return;
  double av = 0., ml = 0., bms = 0., se = 0., g = fabs(a.S.cash[e]);
  for (int j = 0; j < a.P.n_assets; ++j) {
    const double l = a.S.ledger[(int64_t)j * N + e], p = a.S.price[(int64_t)j * N + e],
                 m = a.S.mean_entry[(int64_t)j * N + e], b = a.S.borrowed[(int64_t)j * N + e];
    const double t_ml = m * l;
    const double t_se = (l < 0.) ? t_ml : 0. * t_ml;
    if (j == 0) { av = l * p; ml = t_ml; bms = b; se = t_se; }
    else { av = av + l * p; ml = ml + t_ml; bms = bms + b; se = se + t_se; }
    g += fabs(l * p) + fabs(t_ml) + fabs(b);
  }
  a.S.folds[(int64_t)MDG_FOLD_AV * N + e] = av;
  a.S.folds[(int64_t)MDG_FOLD_ML * N + e] = ml;
  a.S.folds[(int64_t)MDG_FOLD_BM * N + e] = bms;
  a.S.folds[(int64_t)MDG_FOLD_SE * N + e] = se;
  a.S.folds[(int64_t)MDG_FOLD_G * N + e] = g;
}

static int check_common(const MdgParams* P, const MdgLaunch* L) {
  if (!P || !L) return set_err(MDG_E_INVALID, "null params/launch");
  if (P->n_assets < 1 || P->n_assets > MDG_MAX_ASSETS)
    return set_err(MDG_E_UNSUPPORTED, "n_assets must be in 1..MDG_MAX_ASSETS (thread-per-env kernels)");
  if (L->n_envs < 0) return set_err(MDG_E_INVALID, "n_envs < 0");
  if (L->n_envs > (int64_t)2147483647 * 32) return set_err(MDG_E_UNSUPPORTED, "n_envs too large");
  for (int i = 0; i < P->n_assets; ++i) {
    const MdgAssetGen& g = P->gen[i];
    if (g.type < MDG_GEN_SINEADDER) continue;
    if (g.type > MDG_GEN_SINEDYNAMICTREND) return set_err(MDG_E_INVALID, "unknown generator type");
    const int K = (int)g.p[0];
    const int64_t off = (int64_t)g.p[1], rec = g.type == MDG_GEN_SINEADDER ? 4 : 12;
    if (K < 1 || K > MDG_MAX_SINE_COMPONENTS) return set_err(MDG_E_UNSUPPORTED, "sine components must be in 1..MDG_MAX_SINE_COMPONENTS");
    if (!P->gen_ext || off < 0 || off + rec * K > P->n_gen_ext) return set_err(MDG_E_INVALID, "gen_ext is null or too short for a SINE* generator");
    if (g.type == MDG_GEN_SINEDYNAMICTREND) {
      const int T = (int)g.p[4];
      const int64_t toff = (int64_t)g.p[5];
      if (T < 0 || T > MDG_MAX_SINE_TRENDS) return set_err(MDG_E_UNSUPPORTED, "trends must be in 0..MDG_MAX_SINE_TRENDS");
      if (toff < 0 || toff + 4 * T > P->n_gen_ext) return set_err(MDG_E_INVALID, "gen_ext too short for the trend list");
    }
    if (g.type != MDG_GEN_SINEADDER && !(g.p[2] >= 1.)) return set_err(MDG_E_INVALID, "sampleRate must be >= 1");
  }
  return MDG_OK;
}

}  // namespace mdg

using namespace mdg;

static int step_impl(const MdgParams* P, const MdgReward* R, const MdgState* S, const MdgStepIO* IO,
                     const MdgLaunch* L, int* done_count, int* done_list, const MdgParamSets* sets = nullptr,
                     const double* broker = nullptr) {
  int rc = check_common(P, L);
  if (rc) return rc;
  if (!S || !IO) return set_err(MDG_E_INVALID, "null state/io");
  if (!S->folds) return set_err(MDG_E_INVALID, "state.folds is null");
  if (L->window < 1 || L->head < 0 || L->head >= L->window) return set_err(MDG_E_INVALID, "bad window/head");
  if (L->mode < MDG_MODE_HOLD || L->mode > MDG_MODE_SINGLE) return set_err(MDG_E_INVALID, "bad mode");
  const bool by_weights = L->mode == MDG_MODE_MULTI && IO->weights;
  const bool by_actions = L->mode == MDG_MODE_MULTI && IO->actions && !by_weights;
  if (L->mode != MDG_MODE_HOLD && !IO->units && !by_actions && !by_weights) return set_err(MDG_E_INVALID, "units is null");
  if (by_actions && (L->action_atoms < 1 || L->action_atoms > 127))
    return set_err(MDG_E_INVALID, "action_atoms must be in [1, 127] with io.actions");
  if (L->mode == MDG_MODE_SINGLE && (L->asset_idx < 0 || L->asset_idx >= P->n_assets))
    return set_err(MDG_E_INVALID, "asset index out of range");  // std::out_of_range -> IndexError
  if (L->n_envs == 0) return MDG_OK;
  StepArgs a;
  a.P = *P;
  if (R) a.R = *R; else { memset(&a.R, 0, sizeof(a.R)); a.R.shaper = MDG_SHAPER_OFF; a.R.nstep = 1; }
  a.S = *S;
  a.IO = *IO;
  a.L = *L;
  if (a.R.shaper != MDG_SHAPER_OFF) {
    if (a.R.nstep < 1 || a.R.nstep > MDG_MAX_NSTEP) return set_err(MDG_E_INVALID, "nstep out of range");
    if (!IO->agent_reward || !IO->shaped_reward || !IO->n_popped)
      return set_err(MDG_E_INVALID, "shaper on but agent_reward/shaped_reward/n_popped is null");
    if ((a.R.shaper == MDG_SHAPER_DSR || a.R.shaper == MDG_SHAPER_DDR) && (!S->shaper_A || !S->shaper_B))
      return set_err(MDG_E_INVALID, "DSR/DDR need shaper_A/shaper_B");
    if (a.R.nstep > 1 && (!S->nstep_ring || !S->nstep_len))
      return set_err(MDG_E_INVALID, "nstep>1 needs nstep_ring/nstep_len");
    if (L->nstep_pos < 0 || L->nstep_pos >= a.R.nstep) return set_err(MDG_E_INVALID, "bad nstep_pos");
  }
  a.done_count = done_count;
  a.done_list = done_list;
  if (!sets) return launch_step(a);
  StepSetsBrokerArgs b;
  static_cast<StepArgs&>(b) = a;
  b.ps = *sets;
  b.broker = broker;
  if (!broker) return launch_step<true>(static_cast<StepSetsArgs&>(b));
  return launch_step<true, true>(b);
}

extern "C" int mdg_step(const MdgParams* P, const MdgReward* R, const MdgState* S, const MdgStepIO* IO,
                        const MdgLaunch* L) {
  return step_impl(P, R, S, IO, L, nullptr, nullptr);
}

extern "C" int mdg_step_sets_broker(const MdgParams* P, const MdgReward* R, const MdgState* S, const MdgStepIO* IO,
                                    const MdgLaunch* L, const MdgParamSets* sets, const double* broker) {
  int rc = check_common(P, L);
  if (rc) return rc;
  rc = check_sets(P, sets);
  if (rc) return rc;
  return step_impl(P, R, S, IO, L, nullptr, nullptr, sets, broker);
}

extern "C" int mdg_step_sets(const MdgParams* P, const MdgReward* R, const MdgState* S, const MdgStepIO* IO,
                             const MdgLaunch* L, const MdgParamSets* sets) {
  return mdg_step_sets_broker(P, R, S, IO, L, sets, nullptr);
}

extern "C" int mdg_reset(const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgLaunch* L,
                         const uint8_t* mask, int fill_ticks, int clear_nstep) {
  int rc = check_common(P, L);
  if (rc) return rc;
  if (!S || !IO) return set_err(MDG_E_INVALID, "null state/io");
  if (!S->reset_ts || !IO->pre_price) return set_err(MDG_E_INVALID, "state.reset_ts / io.pre_price is null");
  if (L->window < 1 || L->head < 0 || L->head >= L->window) return set_err(MDG_E_INVALID, "bad window/head");
  if (fill_ticks < 1) fill_ticks = 1;
  if (fill_ticks > L->window) return set_err(MDG_E_INVALID, "fill_ticks > window");
  if (L->n_envs == 0) return MDG_OK;
  ResetArgs a;
  a.P = *P; a.S = *S; a.IO = *IO; a.L = *L;
  a.mask = mask; a.fill_ticks = fill_ticks; a.clear_nstep = clear_nstep;
  const unsigned grid = (unsigned)((L->n_envs + kResetBlock - 1) / kResetBlock);
  reset_kernel<<<grid, kResetBlock, 0, (cudaStream_t)L->stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_reset launch");
}

extern "C" int64_t mdg_reset_workspace_bytes(const MdgParams* P, int64_t n_envs, int fill_ticks) {
  if (!P || n_envs < 0) return -1;
  (void)fill_ticks;
  return 256 + 4 * ((n_envs + 63) / 64 * 64);  // header {count, ticket} + list
}

namespace mdg {
static int fill_ws_args(ResetWsArgs& a, const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgLaunch* L,
                        int fill_ticks, int clear_nstep, void* workspace, int64_t workspace_bytes) {
  const int64_t N = L->n_envs;
  if (N > 2147483647) return set_err(MDG_E_UNSUPPORTED, "n_envs too large for the reset list");
  if (workspace_bytes < 256 + 4 * N) return set_err(MDG_E_INVALID, "reset workspace too small (see mdg_reset_workspace_bytes)");
  a.P = *P; a.S = *S; a.IO = *IO; a.L = *L;
  a.mask = nullptr; a.fill_ticks = fill_ticks; a.clear_nstep = clear_nstep;
  a.count = (int*)workspace;
  a.ticket = (int*)workspace + 1;
  a.list = (int*)((char*)workspace + 256);
  a.chunk = fill_ticks < 64 ? fill_ticks : 64;
  if (P->n_normals > 64) {  // many SineAdder components: keep the normals chunk within 32 KB of shared memory
    const int cap = 4096 / P->n_normals;
    a.chunk = a.chunk < cap ? a.chunk : (cap > 0 ? cap : 1);
  }
  a.n_groups = fill_groups(*P, a.leader);
  static_assert(kFillBlock == 128, "group_of_thread is sized for 128 threads");
  for (int t = 0; t < kFillBlock; ++t) a.group_of_thread[t] = -1;
  int types[MDG_MAX_ASSETS], n_types = 0, used[kFillBlock / 32] = {0, 0, 0, 0};
  for (int g = 0; g < a.n_groups; ++g) {
    const int ty = P->gen[a.leader[g]].type;
    int k = 0;
    while (k < n_types && types[k] != ty) ++k;
    if (k == n_types) types[n_types++] = ty;
    const int w = k % (kFillBlock / 32);
    a.group_of_thread[32 * w + used[w]++] = (int8_t)g;  // at most MDG_MAX_ASSETS groups: a warp never overflows
  }
  return MDG_OK;
}
// SM count of the current device, looked up once per device ordinal
static int64_t sm_count() {
  constexpr int kMaxDevices = 64;
  static std::atomic<int> cached[kMaxDevices];
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) dev = 0;
  if (dev < kMaxDevices) n = cached[dev].load(std::memory_order_relaxed);
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    if (dev < kMaxDevices) cached[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}
// all-OU-pairs refill: blocks per SM of its grid (grid-stride over groups of envs beyond that)
constexpr int kFillPairsBlocksPerSm = 2;
// ... and the fewest assets it is taken for: a lane runs its pair's 64 ticks in series (~20 us), where the generic kernel
// spreads an env's draws over a block (~12 us).  With few pairs per env that latency is not paid back: one OU pair per
// env (C3, 65,536 envs, one stream) measured 20.5 us per step with the generic refill, 34.9 with this one.
constexpr int kFillPairsMinAssets = 8;
// Args: ResetWsArgs, ResetWsSetsArgs with SETS, or ResetWsBrokerArgs with SETS and BROKER (the same kernel choice)
template <bool SETS = false, bool BROKER = false, class Args = ResetWsArgs>
static int launch_fill(const Args& a, int64_t max_listed) {
  // the count is on the device: size the grid for the most the list can hold, capped at a few blocks per SM
  // (grid-stride; blocks past the end of the list only read the count and take their exit ticket)
  static const int64_t knob = []() {  // MDG_FILL_GRID: profiling knob
    const char* v = getenv("MDG_FILL_GRID");
    const long n = v ? atol(v) : 0;
    return (int64_t)(n > 0 ? n : 0);
  }();
  cudaStream_t st = (cudaStream_t)a.L.stream;
  if (!(a.L.flags & MDG_FLAG_GENERIC_FILL) && !a.IO.normals && !a.IO.uniforms && a.P.n_assets >= kFillPairsMinAssets &&
      all_ou_pairs(a.P) &&
      (reinterpret_cast<uintptr_t>(a.IO.pre_price) & 15) == 0) {
    const int64_t epb = kFillBlock / (a.P.n_assets / 2);
    const int64_t groups = (max_listed + epb - 1) / epb;
    const int64_t cap = knob ? knob : kFillPairsBlocksPerSm * sm_count();
    const unsigned grid = (unsigned)(groups < cap ? (groups > 0 ? groups : 1) : cap);
    if constexpr (BROKER) reset_fill_pairs_sets_broker_kernel<<<grid, kFillBlock, 0, st>>>(a);
    else if constexpr (SETS) reset_fill_pairs_sets_kernel<<<grid, kFillBlock, 0, st>>>(a);
    else reset_fill_pairs_kernel<<<grid, kFillBlock, 0, st>>>(a);
    return cuda_err(cudaGetLastError(), "reset_fill_pairs launch");
  }
  const int64_t cap = knob ? knob : 148 * 8;
  const unsigned grid = (unsigned)(max_listed < cap ? (max_listed > 0 ? max_listed : 1) : cap);
  const size_t smem = sizeof(double) * (size_t)a.chunk * (size_t)(a.P.n_normals > 0 ? a.P.n_normals : 1);
  if constexpr (BROKER) reset_fill_sets_broker_kernel<<<grid, kFillBlock, smem, st>>>(a);
  else if constexpr (SETS) reset_fill_sets_kernel<<<grid, kFillBlock, smem, st>>>(a);
  else reset_fill_kernel<<<grid, kFillBlock, smem, st>>>(a);
  return cuda_err(cudaGetLastError(), "reset_fill launch");
}
}  // namespace mdg

static int reset_ws_impl(const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgLaunch* L,
                         const uint8_t* mask, int fill_ticks, int clear_nstep, void* workspace, int64_t workspace_bytes,
                         const MdgParamSets* sets, const double* broker = nullptr) {
  int rc = check_common(P, L);
  if (rc) return rc;
  if (sets && (rc = check_sets(P, sets))) return rc;
  if (!S || !IO) return set_err(MDG_E_INVALID, "null state/io");
  if (!S->reset_ts || !IO->pre_price) return set_err(MDG_E_INVALID, "state.reset_ts / io.pre_price is null");
  if (L->window < 1 || L->head < 0 || L->head >= L->window) return set_err(MDG_E_INVALID, "bad window/head");
  if (fill_ticks < 1) fill_ticks = 1;
  if (fill_ticks > L->window) return set_err(MDG_E_INVALID, "fill_ticks > window");
  const int64_t N = L->n_envs;
  if (N == 0) return MDG_OK;
  ResetWsBrokerArgs a;
  rc = fill_ws_args(a, P, S, IO, L, fill_ticks, clear_nstep, workspace, workspace_bytes);
  if (rc) return rc;
  a.mask = mask;
  cudaStream_t st = (cudaStream_t)L->stream;
  cudaError_t ce = cudaMemsetAsync(workspace, 0, 256, st);  // an explicit reset does not rely on the header's state
  if (ce != cudaSuccess) return cuda_err(ce, "mdg_reset_ws memset");
  reset_scan_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(a);
  if (!sets) return launch_fill(static_cast<const ResetWsArgs&>(a), N);
  a.ps = *sets;
  a.broker = broker;
  if (!broker) return launch_fill<true>(static_cast<const ResetWsSetsArgs&>(a), N);
  return launch_fill<true, true>(a, N);
}

extern "C" int mdg_reset_ws(const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgLaunch* L,
                            const uint8_t* mask, int fill_ticks, int clear_nstep, void* workspace,
                            int64_t workspace_bytes) {
  if (!workspace) return mdg_reset(P, S, IO, L, mask, fill_ticks, clear_nstep);
  return reset_ws_impl(P, S, IO, L, mask, fill_ticks, clear_nstep, workspace, workspace_bytes, nullptr);
}

extern "C" int mdg_reset_ws_sets_broker(const MdgParams* P, const MdgState* S, const MdgStepIO* IO,
                                        const MdgLaunch* L, const uint8_t* mask, int fill_ticks, int clear_nstep,
                                        void* workspace, int64_t workspace_bytes, const MdgParamSets* sets,
                                        const double* broker) {
  if (!sets) return set_err(MDG_E_INVALID, "null parameter sets");
  if (!workspace) return set_err(MDG_E_INVALID, "mdg_reset_ws_sets needs a workspace");
  return reset_ws_impl(P, S, IO, L, mask, fill_ticks, clear_nstep, workspace, workspace_bytes, sets, broker);
}

extern "C" int mdg_reset_ws_sets(const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgLaunch* L,
                                 const uint8_t* mask, int fill_ticks, int clear_nstep, void* workspace,
                                 int64_t workspace_bytes, const MdgParamSets* sets) {
  return mdg_reset_ws_sets_broker(P, S, IO, L, mask, fill_ticks, clear_nstep, workspace, workspace_bytes, sets, nullptr);
}

static int step_autoreset_impl(const MdgParams* P, const MdgReward* R, const MdgState* S, const MdgStepIO* IO,
                               const MdgLaunch* L, int fill_ticks, int clear_nstep, void* workspace,
                               int64_t workspace_bytes, const MdgParamSets* sets, const double* broker = nullptr) {
  int rc = check_common(P, L);
  if (rc) return rc;
  if (sets && (rc = check_sets(P, sets))) return rc;
  if (!workspace) return set_err(MDG_E_INVALID, "mdg_step_autoreset needs a workspace");
  if (!S || !IO) return set_err(MDG_E_INVALID, "null state/io");
  if (!S->reset_ts || !IO->pre_price) return set_err(MDG_E_INVALID, "state.reset_ts / io.pre_price is null");
  if (fill_ticks < 1) fill_ticks = 1;
  if (fill_ticks > L->window) return set_err(MDG_E_INVALID, "fill_ticks > window");
  if (L->n_envs == 0) return MDG_OK;
  ResetWsBrokerArgs a;
  MdgStepIO io = *IO;  // the reset draws from Philox (no injected stream) and takes no units
  io.units = nullptr; io.normals = nullptr; io.uniforms = nullptr; io.actions = nullptr; io.weights = nullptr;
  rc = fill_ws_args(a, P, S, &io, L, fill_ticks, clear_nstep, workspace, workspace_bytes);
  if (rc) return rc;
  rc = step_impl(P, R, S, IO, L, a.count, a.list, sets, broker);  // the step kernel appends the finished envs to the list
  if (rc) return rc;
  if (!sets) return launch_fill(static_cast<const ResetWsArgs&>(a), L->n_envs);
  a.ps = *sets;
  a.broker = broker;
  if (!broker) return launch_fill<true>(static_cast<const ResetWsSetsArgs&>(a), L->n_envs);
  return launch_fill<true, true>(a, L->n_envs);
}

extern "C" int mdg_step_autoreset(const MdgParams* P, const MdgReward* R, const MdgState* S, const MdgStepIO* IO,
                                  const MdgLaunch* L, int fill_ticks, int clear_nstep, void* workspace,
                                  int64_t workspace_bytes) {
  return step_autoreset_impl(P, R, S, IO, L, fill_ticks, clear_nstep, workspace, workspace_bytes, nullptr);
}

extern "C" int mdg_step_autoreset_sets_broker(const MdgParams* P, const MdgReward* R, const MdgState* S,
                                              const MdgStepIO* IO, const MdgLaunch* L, int fill_ticks, int clear_nstep,
                                              void* workspace, int64_t workspace_bytes, const MdgParamSets* sets,
                                              const double* broker) {
  if (!sets) return set_err(MDG_E_INVALID, "null parameter sets");
  return step_autoreset_impl(P, R, S, IO, L, fill_ticks, clear_nstep, workspace, workspace_bytes, sets, broker);
}

extern "C" int mdg_step_autoreset_sets(const MdgParams* P, const MdgReward* R, const MdgState* S, const MdgStepIO* IO,
                                       const MdgLaunch* L, int fill_ticks, int clear_nstep, void* workspace,
                                       int64_t workspace_bytes, const MdgParamSets* sets) {
  return mdg_step_autoreset_sets_broker(P, R, S, IO, L, fill_ticks, clear_nstep, workspace, workspace_bytes, sets,
                                        nullptr);
}

static int init_state_impl(const MdgParams* P, const MdgReward* R, const MdgState* S, const MdgLaunch* L,
                           const MdgParamSets* sets, const double* broker = nullptr) {
  int rc = check_common(P, L);
  if (rc) return rc;
  if (sets && (rc = check_sets(P, sets))) return rc;
  if (!S) return set_err(MDG_E_INVALID, "null state");
  if (L->n_envs == 0) return MDG_OK;
  InitBrokerArgs a;
  a.P = *P;
  if (R) a.R = *R; else { memset(&a.R, 0, sizeof(a.R)); a.R.nstep = 1; }
  a.S = *S; a.L = *L;
  const unsigned grid = (unsigned)((L->n_envs + 128 - 1) / 128);
  if (sets && broker) {
    a.ps = *sets;
    a.broker = broker;
    init_sets_broker_kernel<<<grid, 128, 0, (cudaStream_t)L->stream>>>(a);
  } else if (sets) {
    a.ps = *sets;
    init_sets_kernel<<<grid, 128, 0, (cudaStream_t)L->stream>>>(static_cast<const InitSetsArgs&>(a));
  } else {
    init_kernel<<<grid, 128, 0, (cudaStream_t)L->stream>>>(static_cast<const InitArgs&>(a));
  }
  return cuda_err(cudaGetLastError(), "mdg_init_state launch");
}

extern "C" int mdg_init_state(const MdgParams* P, const MdgReward* R, const MdgState* S, const MdgLaunch* L) {
  return init_state_impl(P, R, S, L, nullptr);
}

extern "C" int mdg_init_state_sets_broker(const MdgParams* P, const MdgReward* R, const MdgState* S,
                                          const MdgLaunch* L, const MdgParamSets* sets, const double* broker) {
  if (!sets) return set_err(MDG_E_INVALID, "null parameter sets");
  return init_state_impl(P, R, S, L, sets, broker);
}

extern "C" int mdg_init_state_sets(const MdgParams* P, const MdgReward* R, const MdgState* S, const MdgLaunch* L,
                                   const MdgParamSets* sets) {
  return mdg_init_state_sets_broker(P, R, S, L, sets, nullptr);
}

extern "C" int mdg_refresh_folds(const MdgParams* P, const MdgState* S, const MdgLaunch* L) {
  int rc = check_common(P, L);
  if (rc) return rc;
  if (!S || !S->folds) return set_err(MDG_E_INVALID, "null state/folds");
  if (L->n_envs == 0) return MDG_OK;
  FoldArgs a;
  a.P = *P; a.S = *S; a.N = L->n_envs;
  const unsigned grid = (unsigned)((L->n_envs + 128 - 1) / 128);
  refresh_folds_kernel<<<grid, 128, 0, (cudaStream_t)L->stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_refresh_folds launch");
}

#ifdef MDG_PHASE_CLOCKS
// profiling builds only: copies the 64 x 64 phase clocks of the last step launch to the host
extern "C" int mdg_debug_phase_clocks(long long* out) {
  return cuda_err(cudaMemcpyFromSymbol(out, mdg::g_phase_clk, sizeof(long long) * 64 * 64), "phase clocks");
}
extern "C" int mdg_debug_block_times(unsigned long long* out) {
  return cuda_err(cudaMemcpyFromSymbol(out, mdg::g_block_ns, sizeof(unsigned long long) * 1024 * 4), "block times");
}
#endif

extern "C" int mdg_abi_version(void) { return MDG_ABI_VERSION; }
extern "C" const char* mdg_last_error(void) { return err_buf(); }
extern "C" int mdg_sizeof(int which) {
  switch (which) {
    case 0: return (int)sizeof(MdgAssetGen);
    case 1: return (int)sizeof(MdgParams);
    case 2: return (int)sizeof(MdgReward);
    case 3: return (int)sizeof(MdgState);
    case 4: return (int)sizeof(MdgStepIO);
    case 5: return (int)sizeof(MdgLaunch);
    case 6: return (int)sizeof(MdgDerived);
    case 7: return (int)sizeof(MdgWindow);
    case 8: return (int)sizeof(MdgReplay);
    case 9: return (int)sizeof(MdgReplayBatch);
    case 10: return (int)sizeof(MdgRewardNorm);
    case 11: return (int)sizeof(MdgTearsheet);
    case 12: return (int)sizeof(MdgPrioritized);
    case 13: return (int)sizeof(MdgReplayRows);
    case 14: return (int)sizeof(MdgParamSets);
  }
  return -1;
}
