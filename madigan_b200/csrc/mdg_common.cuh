// Device-side building blocks of the batched Madigan environment (sm_100a).
//
// Everything here mirrors, per env, the arithmetic of the reference's C++ env
// (file:line citations are relative to /root/reference/madigan/environments/cpp/).
// The translation unit is compiled with -fmad=false: the ledger must not contract
// a*b+c into an FMA, because branch decisions (risk gates) and therefore the
// bit-exact ledger depend on the rounding of every intermediate.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/madigan_b200.h"
#include "mdg_math.cuh"

#define MDG_PI2 (3.141592653589793238463 * 2)  // DataSource.h:24

namespace mdg {

char* err_buf();  // thread-local, 512 bytes, defined in mdg_step.cu

inline int set_err(int code, const char* msg) {
  snprintf(err_buf(), 512, "%s", msg);
  return code;
}
inline int cuda_err(cudaError_t e, const char* where) {
  if (e == cudaSuccess) return MDG_OK;
  snprintf(err_buf(), 512, "%s: %s", where, cudaGetErrorString(e));
  return MDG_E_CUDA;
}

// ---------------------------------------------------------------------------
// Philox4x32-10, counter = (env id, stream<<16|block, tick lo, tick hi), key = seed.
// One block -> two 64-bit words -> two draws.  Same conventions as oracle/mdg_oracle.c.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint64_t& x0, uint64_t& x1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  x0 = ((uint64_t)c1 << 32) | c0;
  x1 = ((uint64_t)c3 << 32) | c2;
}

// Draw conventions (shared with oracle/mdg_oracle.c): normal slot s lives in Philox block s>>1 of
// stream 0 (Box-Muller: lane 0 = r*cos, lane 1 = r*sin), uniform slot s in block s>>1 of stream 1.
constexpr int kMaxNormals = (3 * MDG_MAX_ASSETS) / 2;  // 3 per OU pair, 1 per other asset

// Draw source of the reset kernel: normals computed on demand (one Box-Muller block cached), so that
// different lanes can fast-forward different generator groups of different envs.
struct LazyDraws {
  const double* normals;   // [n_normals][N] for this tick (validation mode) or nullptr
  const double* uniforms;  // [n_uniforms][N] for this tick (validation mode) or nullptr
  int64_t N, e, gstride;
  uint32_t gid, k0, k1, t_lo, t_hi;
  int cached_block;
  double z0, z1;
};
static __device__ __noinline__ double draw_normal(LazyDraws& c, int slot) {
  if (c.normals) return c.normals[(int64_t)slot * c.N + c.e];
  const int blk = slot >> 1;
  if (blk != c.cached_block) {
    uint64_t x0, x1;
    philox4x32_10(c.gid, (uint32_t)blk, c.t_lo, c.t_hi, c.k0, c.k1, x0, x1);
    const double u1 = ((double)(x0 >> 12) + 0.5) * 0x1.0p-52;
    const double u2 = (double)(x1 >> 11) * 0x1.0p-53;
    const double r = fast_sqrt_pos(-2.0 * fast_log_pos(u1));
    double sn, cs;
    fast_sincos_2pi(u2, sn, cs);
    c.z0 = r * cs;
    c.z1 = r * sn;
    c.cached_block = blk;
  }
  return (slot & 1) ? c.z1 : c.z0;
}
static __device__ __noinline__ double draw_uniform(LazyDraws& c, int slot) {
  if (c.uniforms) return c.uniforms[(int64_t)slot * c.N + c.e];
  uint64_t x0, x1;
  philox4x32_10(c.gid, (1u << 16) | (uint32_t)(slot >> 1), c.t_lo, c.t_hi, c.k0, c.k1, x0, x1);
  return (double)(((slot & 1) ? x1 : x0) >> 11) * 0x1.0p-53;
}

// Draw source of the reset kernel's recurrence phase: this (env, tick)'s normals were generated into
// shared memory by all lanes of the block beforehand; uniforms (trend generators only) stay on demand.
struct TickDraws {
  const double* z;         // z[slot]
  const double* uniforms;  // [n_uniforms][N] for this tick (validation mode) or nullptr
  int64_t N, e, gstride;
  uint32_t gid, k0, k1, t_lo, t_hi;
};
__device__ __forceinline__ double draw_normal(TickDraws& c, int slot) { return c.z[slot]; }
static __device__ __noinline__ double draw_uniform(TickDraws& c, int slot) {
  if (c.uniforms) return c.uniforms[(int64_t)slot * c.N + c.e];
  uint64_t x0, x1;
  philox4x32_10(c.gid, (1u << 16) | (uint32_t)(slot >> 1), c.t_lo, c.t_hi, c.k0, c.k1, x0, x1);
  return (double)(((slot & 1) ? x1 : x0) >> 11) * 0x1.0p-53;
}

// ---------------------------------------------------------------------------
// generator state flags (bit0 trending, bit1 direction +1, bits 32.. remaining length)
// ---------------------------------------------------------------------------
__device__ __forceinline__ double pack_flags(int trending, int dir, int len) {
  const long long b = (long long)(trending ? 1 : 0) | (long long)(dir > 0 ? 2 : 0) |
                      (long long)((unsigned long long)(unsigned int)len << 32);
  return __longlong_as_double(b);
}
__device__ __forceinline__ void unpack_flags(double f, int& trending, int& dir, int& len) {
  const long long b = __double_as_longlong(f);
  trending = (int)(b & 1);
  dir = (b & 2) ? 1 : -1;
  len = (int)((unsigned long long)b >> 32);
}
__device__ __forceinline__ double dmax(double a, double b) { return (a < b) ? b : a; }  // std::max
__device__ __forceinline__ int u_int(double u, double a, double b) { return (int)(a + floor(u * (b - a + 1.))); }
__device__ __forceinline__ double u_real(double u, double a, double b) { return a + u * (b - a); }

// uniform draws of the SINEDYNAMIC* constructor (stream 3) and reset() (stream 2): slot 64*asset + 3c + {0,1,2}
struct CtorDraws {
  uint32_t gid, k0, k1, t_lo, t_hi;
  int stream;
  int asset;
};
static __device__ __noinline__ double draw_ctor_uniform(const CtorDraws& c, int slot) {
  uint64_t x0, x1;
  philox4x32_10(c.gid, ((uint32_t)c.stream << 16) | (uint32_t)(slot >> 1), c.t_lo, c.t_hi, c.k0, c.k1, x0, x1);
  return (double)(((slot & 1) ? x1 : x0) >> 11) * 0x1.0p-53;
}
__device__ __forceinline__ CtorDraws ctor_draws(uint32_t gid, uint64_t seed, long long tick, int stream, int asset) {
  CtorDraws c;
  c.gid = gid; c.k0 = (uint32_t)seed; c.k1 = (uint32_t)(seed >> 32);
  c.t_lo = (uint32_t)(unsigned long long)tick; c.t_hi = (uint32_t)((unsigned long long)tick >> 32);
  c.stream = stream; c.asset = asset;
  return c;
}
// freq, mu, amp of every component ~ uniform_real(lo, hi) (DataSource.cpp:771-773 / 783-787, :972-974 / 992-996)
static __device__ __noinline__ void sine_dynamic_sample(const MdgAssetGen& g, double* __restrict__ gs, int64_t N,
                                                        const double* __restrict__ ext, const CtorDraws& c) {
  const int K = (int)g.p[0];
  const double* cp = ext + (int64_t)g.p[1];
  for (int i = 0; i < K; ++i, cp += 12)
    for (int j = 0; j < 3; ++j)
      gs[(int64_t)(4 * i + j) * N] = u_real(draw_ctor_uniform(c, 64 * c.asset + 3 * i + j), cp[3 * j], cp[3 * j + 1]);
}

// random boolean b of this tick (randomBoolGenerator.h:8-14): bit 52-b of floor(u 2^53)
__device__ __forceinline__ bool u_bool(unsigned long long bits, int b) { return (bits >> (52 - b)) & 1ull; }
__device__ __forceinline__ double dmin(double a, double b) { return (b < a) ? b : a; }  // std::min
// bounded +-step walk of updateParams (DataSource.cpp:804-812)
__device__ __forceinline__ double sine_walk(double v, bool up, const double* r) {
  return dmax(r[0], dmin(r[1], v + (up ? r[2] : -r[2])));
}
// WaveTableOsc::setFreq + process (WaveTableOsc.h:77-110) of the component with record cp
__device__ __forceinline__ double osc_process(const double* __restrict__ ext, const double* __restrict__ cp,
                                              double incr, double& phasor) {
  const int nt = (int)cp[9];
  const double* tl = ext + (int64_t)cp[10];
  int idx = 0;
  while (incr >= tl[3 * idx] && idx < nt - 1) ++idx;
  phasor += incr;
  if (phasor >= 1.) phasor -= 1.;
  const int len = (int)tl[3 * idx + 1];
  const double* tab = ext + (int64_t)tl[3 * idx + 2];
  const double temp = phasor * len;
  const int ip = (int)temp;
  const double frac = temp - ip;
  const double s0 = tab[ip], s1 = tab[ip + 1];
  return s0 + (s1 - s0) * frac;
}

// Parameter accessors of the generator bodies.  AssetParams: p[j] is MdgAssetGen.p[j] (launches without parameter
// sets).  SetParams: p[j] of the asset is the env's entry of a parameter-set table (MdgParamSets, set-minor),
// q = &table[(i * MDG_GEN_NPARAM) * n_sets + set].
struct AssetParams {
  const MdgAssetGen& g;
  __device__ __forceinline__ double operator[](int j) const { return g.p[j]; }
};
struct SetParams {
  const double* q;
  int64_t S;
  __device__ __forceinline__ double operator[](int j) const { return q[j * S]; }
};
__device__ __forceinline__ SetParams set_params(const MdgParamSets& ps, int64_t set, int asset) {
  return SetParams{ps.p + (int64_t)asset * MDG_GEN_NPARAM * ps.n_sets + set, (int64_t)ps.n_sets};
}
// the env's set: an index outside [0, n_sets) is clamped, as unsigned, to n_sets - 1 (never read outside the table)
__device__ __forceinline__ int64_t env_set(const MdgParamSets& ps, int64_t e) {
  const unsigned s = (unsigned)ps.set_of_env[e], last = (unsigned)(ps.n_sets - 1);
  return (int64_t)(s < last ? s : last);
}
// broker sets: slot k (MdgBrokerSlot) of set `set` in a broker table, [MDG_BROKER_NPARAM][n_sets] set-minor
__device__ __forceinline__ double broker_value(const double* __restrict__ broker, int32_t n_sets, int64_t set, int k) {
  return __ldg(broker + (int64_t)k * n_sets + set);
}
// per-episode set draw (MdgSetDraw): u from Philox stream 4 of (env id, tick), then the number of cdf entries <= u,
// an upper-bound binary search of ceil(log2 n_sets) + 1 loads (clamped: a cdf whose last entry is not 1 reads no
// further than set n_sets - 1)
__device__ __forceinline__ int32_t draw_set(const double* __restrict__ cdf, int32_t n_sets, uint32_t gid,
                                            unsigned long long tick, uint32_t k0, uint32_t k1) {
  uint64_t x0, x1;
  philox4x32_10(gid, 4u << 16, (uint32_t)tick, (uint32_t)(tick >> 32), k0, k1, x0, x1);
  const double u = (double)(x0 >> 11) * 0x1.0p-53;
  int32_t lo = 0, len = n_sets;
  while (len > 0) {
    const int32_t half = len >> 1;
    if (__ldg(cdf + lo + half) <= u) {
      lo += half + 1;
      len -= half + 1;
    } else {
      len = half;
    }
  }
  return lo < n_sets ? lo : n_sets - 1;
}

// parameter sets (host): a table and an assignment, and only generators whose p slots are plain numbers
static inline int check_sets(const MdgParams* P, const MdgParamSets* ps) {
  if (!ps) return set_err(MDG_E_INVALID, "null parameter sets");
  if (ps->n_sets < 1) return set_err(MDG_E_INVALID, "parameter sets: n_sets < 1");
  if (!ps->p || !ps->set_of_env) return set_err(MDG_E_INVALID, "parameter sets: null table / set_of_env");
  for (int i = 0; i < P->n_assets; ++i)
    if (P->gen[i].type >= MDG_GEN_SINEADDER)
      return set_err(MDG_E_UNSUPPORTED, "parameter sets do not support SINE* generators");
  return MDG_OK;
}

// episode results (mdg_tearsheet.cu): the argument checks and the record + harvest launch, which the fused
// step + auto-reset (mdg_api.cu) issues between its step kernel and its refill
int check_results(const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgParamSets* sets,
                  const MdgEpisodeResults* res);
int launch_results_record(const MdgParams* P, const MdgState* S, const MdgStepIO* IO, const MdgParamSets* sets,
                          const double* broker, const MdgEpisodeResults* res, void* stream);

// One getData() of asset i (DataSource.cpp).  `price` is the asset's current price
// (== generator value for every synthetic source), gs points at gstate row gslot for
// this env (stride N), pair_mean carries OUPair's shared mean from role 0 to role 1.
// D provides N, draw_normal(d, slot), draw_uniform(d, slot); p[j] (PP: a pointer or SetParams) the parameter slots.
template <class D, class PP>
__device__ __forceinline__ double gen_tick_p(const MdgAssetGen& g, const PP& p, double price, double* __restrict__ gs,
                                             D& d, double& pair_mean, const double* __restrict__ ext) {
  const int64_t N = d.gstride;  // distance between this asset's generator-state rows
  switch (g.type) {
    case MDG_GEN_SYNTH: {  // DataSource.cpp:535-543
      const double x = gs[0];
      price = draw_normal(d, g.nslot) * p[5] + p[1] + p[2] * sin(MDG_PI2 * x * p[0]);
      gs[0] = x + p[4];
      break;
    }
    case MDG_GEN_SAWTOOTH: {  // :558-567
      const double x = gs[0];
      double ip;
      price = draw_normal(d, g.nslot) * p[5] + p[1] + p[2] * modf(x * p[0], &ip);
      gs[0] = x + p[4];
      break;
    }
    case MDG_GEN_TRIANGLE: {  // :569-578
      const double x = gs[0];
      price = draw_normal(d, g.nslot) * p[5] + p[1] + 4 * p[2] / MDG_PI2 * asin(sin(MDG_PI2 * x / p[0]));
      gs[0] = x + p[4];
      break;
    }
    case MDG_GEN_GAUSSIAN:  // :1108-1114
      price = draw_normal(d, g.nslot) * p[1] + p[0];
      break;
    case MDG_GEN_OU:  // :1173-1180
      price += (p[1] * (p[0] - price)) + p[0] * p[2] * draw_normal(d, g.nslot);
      break;
    case MDG_GEN_OUPAIR: {  // :1232-1240
      if (g.role == 0) {
        double m = gs[0];
        m += m * (draw_normal(d, g.nslot_aux) * p[2]);
        gs[0] = m;
        pair_mean = m;
      }
      const double m = pair_mean;
      price += (p[0] * (m - price)) + m * (draw_normal(d, g.nslot) * p[1]);
      break;
    }
    case MDG_GEN_SIMPLETREND: {  // :1324-1350
      double y = price;
      int trending, dir, len;
      unpack_flags(gs[N], trending, dir, len);
      if (trending) {
        y += y * gs[0] * dir;
        if (--len == 0) trending = 0;
      } else {
        const double r = draw_uniform(d, g.uslot);
        if (r < p[0]) {
          trending = 1;
          dir = (draw_uniform(d, g.uslot + 1) < 0.5) ? -1 : 1;
          len = u_int(draw_uniform(d, g.uslot + 2), p[1], p[2]);
          gs[0] = u_real(draw_uniform(d, g.uslot + 3), p[5], p[6]);
        }
      }
      if (y <= .1) dir = 1;
      y += y * (draw_normal(d, g.nslot) * p[3]);
      y = dmax(0.01, y);
      price = y;
      gs[N] = pack_flags(trending, dir, len);
      break;
    }
    case MDG_GEN_TRENDOU: {  // :1457-1493
      double y = price;
      int trending, dir, len;
      unpack_flags(gs[2 * N], trending, dir, len);
      if (trending) {
        y += y * (gs[N] * dir + draw_normal(d, g.nslot) * p[8]);
        len -= 1;
        if (len == 0) {
          trending = 0;
          gs[0] = y;
        }
        y = dmax(0.01, y);
        if (y <= .1) dir = 1;
      } else {
        const double ou_noise = y * (draw_normal(d, g.nslot) * p[7]);
        const double rev = p[6] * (gs[0] - y);
        y += rev + ou_noise;
        const double r = draw_uniform(d, g.uslot);
        if (r < p[0]) {
          trending = 1;
          dir = (draw_uniform(d, g.uslot + 1) < 0.5) ? -1 : 1;
          len = u_int(draw_uniform(d, g.uslot + 2), p[1], p[2]);
          gs[N] = u_real(draw_uniform(d, g.uslot + 3), p[3], p[4]);
        }
      }
      price = y;
      gs[2 * N] = pack_flags(trending, dir, len);
      break;
    }
    case MDG_GEN_TRENDYOU: {  // :1602-1642
      int trending, dir, len;
      unpack_flags(gs[3 * N], trending, dir, len);
      double ou = gs[0], tr = gs[N];
      const double ou_noise = tr * (draw_normal(d, g.nslot) * p[7]);
      const double rev = p[6] * (-ou);
      ou += rev + ou_noise;
      if (trending) {
        tr += tr * (gs[2 * N] * dir);
        tr = dmax(0.1, tr);
        if (tr <= .1) {
          dir = 1;
          trending = 1;
          len = u_int(draw_uniform(d, g.uslot + 2), p[1], p[2]);
        }
        if (--len == 0) trending = 0;
      } else {
        const double r = draw_uniform(d, g.uslot);
        if (r < p[0]) {
          trending = 1;
          dir = (draw_uniform(d, g.uslot + 1) < 0.5) ? -1 : 1;
          len = u_int(draw_uniform(d, g.uslot + 2), p[1], p[2]);
          gs[2 * N] = u_real(draw_uniform(d, g.uslot + 3), p[3], p[4]);
        }
      }
      gs[0] = ou;
      gs[N] = tr;
      price = ou + tr;
      gs[3 * N] = pack_flags(trending, dir, len);
      break;
    }
    case MDG_GEN_SINEADDER: {  // :663-673
      const int K = (int)p[0];
      const double* cp = ext + (int64_t)p[1];
      double sum = 0.;
      for (int i = 0; i < K; ++i, cp += 4) {
        const double x = gs[(int64_t)i * N];
        sum = sum + ((draw_normal(d, g.nslot + i) * p[3] + cp[1]) + cp[2] * sin(MDG_PI2 * x * cp[0]));
        gs[(int64_t)i * N] = x + p[2];
      }
      price = sum;
      break;
    }
    case MDG_GEN_SINEDYNAMIC:
    case MDG_GEN_SINEDYNAMICTREND: {  // :802-841, :1002-1047
      const bool trend = g.type == MDG_GEN_SINEDYNAMICTREND;
      const int K = (int)p[0];
      const double* cp = ext + (int64_t)p[1];
      const unsigned long long bits = (unsigned long long)(draw_uniform(d, g.uslot) * 0x1.0p53);
      double tcmp = trend ? gs[(int64_t)(4 * K) * N] : 1.;
      double sum = 0.;
      for (int i = 0; i < K; ++i, cp += 12) {
        double* s = gs + (int64_t)(4 * i) * N;
        const double mu = sine_walk(s[N], u_bool(bits, 3 * i), cp + 3);
        const double amp = sine_walk(s[2 * N], u_bool(bits, 3 * i + 1), cp + 6);
        const double freq = sine_walk(s[0], u_bool(bits, 3 * i + 2), cp);
        double phasor = s[3 * N];
        const double o = osc_process(ext, cp, freq / p[2], phasor);
        s[0] = freq; s[N] = mu; s[2 * N] = amp; s[3 * N] = phasor;
        sum = trend ? sum + tcmp * (mu + amp * o) : sum + (mu + amp * o);
      }
      const double z = draw_normal(d, g.nslot) * p[3] + 0.;
      if (!trend) {
        price = sum + z;
        break;
      }
      const int T = (int)p[4];
      const double* tp = ext + (int64_t)p[5];
      for (int j = 0; j < T; ++j, tp += 4) {
        double* fl = gs + (int64_t)(4 * K + 1 + j) * N;
        int trending, dir, len;
        unpack_flags(fl[0], trending, dir, len);
        if (trending) {
          tcmp += tcmp * tp[2] * dir;
          if (--len == 0) trending = 0;
        } else {
          const double r = draw_uniform(d, g.uslot + 1 + 2 * j);
          if (r < tp[3]) {
            trending = 1;
            dir = u_bool(bits, 3 * K + j) ? -1 : 1;
            len = u_int(draw_uniform(d, g.uslot + 2 + 2 * j), tp[0], tp[1]);
          }
        }
        if (tcmp <= .1) dir = 1;
        tcmp = dmax(0.01, tcmp);
        fl[0] = pack_flags(trending, dir, len);
      }
      gs[(int64_t)(4 * K) * N] = tcmp;
      price = sum + tcmp + tcmp * z;
      break;
    }
  }
  return price;
}
// NOT inlined: one copy of the nine generator bodies per kernel and draw source (generic / Composite path).
template <class D>
static __device__ __noinline__ double gen_tick(const MdgAssetGen& g, double price, double* __restrict__ gs,
                                               D& d, double& pair_mean, const double* __restrict__ ext = nullptr) {
  const double* p = g.p;
  return gen_tick_p(g, p, price, gs, d, pair_mean, ext);
}
// ... and the parameter-set launches' copy (SINE* sources are not accepted there: p[] is a plain number everywhere)
template <class D>
static __device__ __noinline__ double gen_tick_sets(const MdgAssetGen& g, SetParams p, double price,
                                                    double* __restrict__ gs, D& d, double& pair_mean) {
  return gen_tick_p(g, p, price, gs, d, pair_mean, nullptr);
}

// DataSource::reset() of asset i; returns the new price (Synth/OU/Gaussian: unchanged).
template <class PP>
__device__ __forceinline__ double gen_reset_p(const MdgAssetGen& g, const PP& p, double price, double* __restrict__ gs,
                                              int64_t N, const double* __restrict__ ext, const CtorDraws* cd) {
  switch (g.type) {
    case MDG_GEN_SINEDYNAMIC:
    case MDG_GEN_SINEDYNAMICTREND:  // :783-787, :992-996: new freq, mu, amp; phasors and trend state stay
      sine_dynamic_sample(g, gs, N, ext, *cd);
      return price;
    case MDG_GEN_OUPAIR:  // DataSource.cpp:1242-1246
      if (g.role == 0) gs[0] = 10.;
      return 10.;
    case MDG_GEN_SIMPLETREND:  // :1352-1359
      gs[N] = pack_flags(0, 1, 0);
      return p[4];
    case MDG_GEN_TRENDOU: {  // :1495-1502 (direction, dY untouched)
      int trending, dir, len;
      unpack_flags(gs[2 * N], trending, dir, len);
      gs[0] = p[5];
      gs[2 * N] = pack_flags(0, dir, 0);
      return p[5];
    }
    case MDG_GEN_TRENDYOU: {  // :1644-1657
      int trending, dir, len;
      unpack_flags(gs[3 * N], trending, dir, len);
      gs[0] = 0.;
      gs[N] = p[5];
      gs[3 * N] = pack_flags(0, dir, 0);
      return p[5];
    }
    default:
      return price;
  }
}

__device__ __forceinline__ double gen_reset(const MdgAssetGen& g, double price, double* __restrict__ gs,
                                            int64_t N, const double* __restrict__ ext = nullptr,
                                            const CtorDraws* cd = nullptr) {
  return gen_reset_p(g, AssetParams{g}, price, gs, N, ext, cd);
}

// constructor state of asset i (initParams of each source); returns the start price
template <class PP>
__device__ __forceinline__ double gen_start_p(const MdgAssetGen& g, const PP& p, double* __restrict__ gs, int64_t N,
                                              const double* __restrict__ ext, const CtorDraws* cd) {
  switch (g.type) {
    case MDG_GEN_SINEADDER: {  // x = phase, DataSource.cpp:652
      const int K = (int)g.p[0];
      const double* cp = ext + (int64_t)g.p[1];
      for (int i = 0; i < K; ++i) gs[(int64_t)i * N] = cp[4 * i + 3];
      return 0.;
    }
    case MDG_GEN_SINEDYNAMIC:
    case MDG_GEN_SINEDYNAMICTREND: {  // :741-780, :938-989
      const int K = (int)g.p[0];
      sine_dynamic_sample(g, gs, N, ext, *cd);
      for (int i = 0; i < K; ++i) gs[(int64_t)(4 * i + 3) * N] = 0.;  // phasor, WaveTableOsc.h:62
      if (g.type == MDG_GEN_SINEDYNAMICTREND) {
        const int T = (int)g.p[4];
        gs[(int64_t)(4 * K) * N] = 1.;  // trendComponent :982
        for (int j = 0; j < T; ++j) gs[(int64_t)(4 * K + 1 + j) * N] = pack_flags(0, 1, 0);
      }
      return 0.;
    }
    case MDG_GEN_SYNTH:
    case MDG_GEN_SAWTOOTH:
    case MDG_GEN_TRIANGLE:
      gs[0] = p[3];  // DataSource.cpp:463
      return 0.;
    case MDG_GEN_OU:
    case MDG_GEN_GAUSSIAN:
      return p[0];  // :1129, :1066
    case MDG_GEN_OUPAIR:
      if (g.role == 0) gs[0] = 10.;  // :1194
      return 10.;                    // :1192
    case MDG_GEN_SIMPLETREND:
      gs[0] = 0.;
      gs[N] = pack_flags(0, 1, 0);
      return p[4];  // :1273
    case MDG_GEN_TRENDOU:
      gs[0] = p[5];
      gs[N] = 0.;
      gs[2 * N] = pack_flags(0, 1, 0);
      return p[5];
    case MDG_GEN_TRENDYOU:
      gs[0] = 0.;
      gs[N] = p[5];
      gs[2 * N] = 0.;
      gs[3 * N] = pack_flags(0, 1, 0);
      return p[5];
  }
  return 0.;
}

__device__ __forceinline__ double gen_start(const MdgAssetGen& g, double* __restrict__ gs, int64_t N,
                                            const double* __restrict__ ext = nullptr, const CtorDraws* cd = nullptr) {
  return gen_start_p(g, AssetParams{g}, gs, N, ext, cd);
}

// Portfolio::checkRisk() :243-252 from the folds
__device__ __forceinline__ bool margin_call(double cash, double av, double ml, double bms, double se,
                                            double maintM) {
  const double pnl = av - ml;
  const double marginRequired = maintM * pnl;
  const double equity = cash + av - bms;
  if (equity <= -marginRequired) return true;
  const double balance = cash + se;
  if ((balance + pnl) <= -marginRequired) return true;
  return false;
}

}  // namespace mdg
