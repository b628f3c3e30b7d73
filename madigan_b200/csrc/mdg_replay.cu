// Device-side n-step replay ingest and sampling (include/madigan_b200.h, "Device-side n-step replay ingest").
#include <stdio.h>

#include "mdg_replay.cuh"

namespace mdg {

struct AppendArgs {
  MdgReplay rp;
  int64_t N, step;
  const double* action;
  const double* shaped;
  const int32_t* n_popped;
  const int32_t* nstep_len;
  const uint8_t* done;
};

// one thread per env: store this step's action in the action ring, then append the popped transitions
// (ReplayBuffer.add, replay_buffer.py:68-80; pop_nstep_sarsd, nstep_buffer.py:342-361)
__global__ void __launch_bounds__(256) replay_append_kernel(const __grid_constant__ AppendArgs a) {
  const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const MdgReplay& r = a.rp;
  const int n = r.nstep, A = r.n_action, ra = r.ra;
  const int lane = threadIdx.x & 31;
  int pops = 0;
  if (e < a.N) {
    double* dst = r.act_ring + ((int64_t)(a.step % n) * a.N + e) * A;
    for (int j = 0; j < A; ++j) dst[j] = a.action[e * A + j];
    pops = a.n_popped[e];
  }
  // warp-aggregated reservation of ring slots
  int incl = pops;
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  const int total = __shfl_sync(0xffffffffu, incl, 31);
  unsigned long long base = 0;
  if (lane == 31 && total > 0) base = atomicAdd(r.cursor, (unsigned long long)total);
  base = __shfl_sync(0xffffffffu, base, 31);
  if (e >= a.N || pops == 0) return;
  const int len_after = (n > 1 && a.nstep_len) ? a.nstep_len[e] : 0;
  const int L0 = len_after + pops;  // entries in the n-step buffer right after this step's add
  unsigned long long pos = base + (unsigned long long)(incl - pops);
  for (int k = 0; k < pops; ++k, ++pos) {
    const int L = L0 - k;  // entries when this pop happens: the popped one is step - L + 1
    const int64_t slot = (int64_t)(pos % (unsigned long long)r.capacity);
    const int64_t s_state = a.step - L, s_act = a.step - L + 1;
    r.t_env[slot] = (int32_t)e;
    r.t_state_slot[slot] = (int32_t)(((s_state % r.depth) + r.depth) % r.depth);
    r.t_next_slot[slot] = (int32_t)(a.step % r.depth);
    r.t_state_step[slot] = s_state;
    r.t_done[slot] = a.done[e];
    for (int c = 0; c < ra; ++c) r.t_reward[slot * ra + c] = a.shaped[((int64_t)k * ra + c) * a.N + e];
    const double* src = r.act_ring + ((int64_t)(((s_act % n) + n) % n) * a.N + e) * A;
    for (int j = 0; j < A; ++j) r.t_action[slot * A + j] = src[j];
  }
}

// Sample b's draw (ReplayBuffer._sample_idxs, replay_buffer.py:107-108: uniform over the filled part), redrawn until
// `resident` accepts the record, 64 attempts at most (-1: none found).
template <class Resident>
__device__ __forceinline__ long long replay_draw(const MdgReplay& r, int64_t b, uint64_t seed, uint64_t draw,
                                                 Resident resident) {
  const unsigned long long cur = *r.cursor;
  const unsigned long long filled = cur < (unsigned long long)r.capacity ? cur : (unsigned long long)r.capacity;
  long long pick = -1;
  for (uint32_t attempt = 0; attempt < 64 && filled > 0; ++attempt) {
    uint64_t x0, x1;
    philox4x32_10((uint32_t)b, (uint32_t)(b >> 32) ^ (attempt << 8), (uint32_t)draw, (uint32_t)(draw >> 32),
                  (uint32_t)seed, (uint32_t)(seed >> 32), x0, x1);
    const unsigned long long j = (unsigned long long)(((x0 >> 11) * 0x1.0p-53) * (double)filled);
    const long long cand = (long long)(j < filled ? j : filled - 1);
    if (resident(cand)) { pick = cand; break; }
  }
  return pick;
}

struct SampleArgs {
  MdgReplay rp;
  int64_t cur_step, batch;
  uint64_t seed, draw;
  GatherArgs g;
};

// one block per sample: thread 0 draws a non-stale transition (ReplayBuffer._sample_idxs, replay_buffer.py:107-108:
// uniform over the filled part), then the block copies the two windows and the small fields
__global__ void __launch_bounds__(kGatherThreads) replay_sample_kernel(const __grid_constant__ SampleArgs a) {
  __shared__ long long s_idx;
  const MdgReplay& r = a.rp;
  const int64_t b = blockIdx.x;
  if (threadIdx.x == 0)
    s_idx = replay_draw(r, b, a.seed, a.draw, [&](long long c) { return replay_resident(r, c, a.cur_step); });
  __syncthreads();
  const long long idx = s_idx;
  if (threadIdx.x == 0) a.g.out.idx[b] = idx;
  replay_gather(r, a.g, b, idx);
}

struct RowsIngestArgs {
  MdgReplayRows rw;
  const double* ring;        // [k][F][N] obs_price
  const double* prefix;      // [N][k][F] pre_price
  const int64_t* timestamp;  // [N]
  const int64_t* reset_ts;   // [N]
  int64_t N, slot;
  int head, whole;
};

constexpr int kIngestEnvs = 64;  // envs per block of the rows ingest (256 threads)

// The ingest rule (include/madigan_b200.h, "Replay row store") for kIngestEnvs envs per block: one thread per env
// decides and counts; the newest ring rows are read coalesced over envs into shared memory and written back as one
// contiguous run of F doubles per env (per-thread row writes, 32 KB apart at the bench shape, were far slower); each
// env that appends its whole window is copied by one warp.  The window's rows are read as window_kernel (mdg_aux.cu)
// reads them: ring rows for ages < since, prefix rows otherwise.
__global__ void __launch_bounds__(256) replay_rows_ingest_kernel(const __grid_constant__ RowsIngestArgs a) {
  __shared__ double s_row[kIngestEnvs][65];  // newest ring row per env (F <= 64), padded
  __shared__ long long s_pos[kIngestEnvs];  // ring position of the first row the env appends
  __shared__ int s_since[kIngestEnvs], s_whole[kIngestEnvs];
  const MdgReplayRows& w = a.rw;
  const int t = threadIdx.x, k = w.window, F = w.n_feats;
  const int64_t R = w.n_rows, e0 = (int64_t)blockIdx.x * kIngestEnvs;
  const int ne = (int)(a.N - e0 < kIngestEnvs ? a.N - e0 : kIngestEnvs);
  if (t < ne) {
    const int64_t e = e0 + t;
    const int64_t ts = a.timestamp[e];
    const long long since = ts - a.reset_ts[e] + 1;  // ring rows written since the last reset
    const bool whole = a.whole || since == 1 || ts != w.last_ts[e] + 1;
    const long long cnt = w.row_count[e], added = whole ? k : 1;
    s_pos[t] = (cnt + 1) % R;
    s_since[t] = since > k ? k : (int)since;
    s_whole[t] = whole;
    w.row_count[e] = cnt + added;
    w.row_end[a.slot * a.N + e] = cnt + added;
    w.last_ts[e] = ts;
  }
  for (int i = t; i < kIngestEnvs * F; i += 256) {
    const int el = i % kIngestEnvs, f = i / kIngestEnvs;
    if (el < ne) s_row[el][f] = a.ring[((int64_t)a.head * F + f) * a.N + e0 + el];
  }
  __syncthreads();
  for (int i = t; i < ne * F; i += 256) {
    const int el = i / F, f = i - el * F;
    if (!s_whole[el]) w.rows[((e0 + el) * R + s_pos[el]) * F + f] = s_row[el][f];
  }
  // whole windows: U independent loads in flight per lane (one load per iteration left each copy latency-bound)
  const int lane = t & 31;
  for (int el = t >> 5; el < ne; el += 256 / 32) {
    if (!s_whole[el]) continue;
    const int64_t e = e0 + el, p0 = s_pos[el];
    const int is = s_since[el];
    double* dst = w.rows + e * R * F;
    const double* rb = a.ring + e;
    const double* pb = a.prefix + (e * k + (k - 2 + is)) * F;  // prefix row of age `age`: (k - 2 + since) - age
    constexpr int U = 8;
    for (int i0 = lane; i0 < k * F; i0 += 32 * U) {
      double v[U];
      int64_t o[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = i0 + 32 * u;
        o[u] = -1;
        v[u] = 0.;
        if (i < k * F) {
          const int s = i / F, f = i - s * F;
          const int age = k - 1 - s;
          int slot = a.head - age;
          if (slot < 0) slot += k;
          v[u] = age < is ? rb[((int64_t)slot * F + f) * a.N] : pb[f - (int64_t)age * F];
          int64_t p = p0 + s;  // k <= R: one wrap at most
          if (p >= R) p -= R;
          o[u] = p * F + f;
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (o[u] >= 0) dst[o[u]] = v[u];
    }
  }
}

struct SampleRowsArgs {
  MdgReplay rp;
  int64_t cur_step;
  uint64_t seed, draw;
  RowsGatherArgs g;
};

// replay_sample_kernel over the row store: the same draws, with the row store's residency test added
__global__ void __launch_bounds__(kGatherThreads) replay_sample_rows_kernel(const __grid_constant__ SampleRowsArgs a) {
  __shared__ long long s_idx;
  const MdgReplay& r = a.rp;
  const int64_t b = blockIdx.x;
  if (threadIdx.x == 0) {
    const int64_t cur = a.cur_step, N = a.g.N;
    s_idx = replay_draw(r, b, a.seed, a.draw, [&](long long c) {
      return replay_resident(r, c, cur) && rows_resident(r, a.g.rw, N, c);
    });
  }
  __syncthreads();
  const long long idx = s_idx;
  if (threadIdx.x == 0) a.g.out.idx[b] = idx;
  replay_gather_rows(r, a.g, b, idx);
}

}  // namespace mdg

using namespace mdg;

extern "C" int mdg_replay_append(const MdgReplay* rp, int64_t n_envs, int64_t step, const double* action,
                                 const double* shaped_reward, const int32_t* n_popped, const int32_t* nstep_len,
                                 const uint8_t* done, void* stream) {
  int rc = check_replay(rp);
  if (rc) return rc;
  if (!action || !shaped_reward || !n_popped || !done) return set_err(MDG_E_INVALID, "null append input");
  if (rp->nstep > 1 && !nstep_len) return set_err(MDG_E_INVALID, "nstep > 1 needs nstep_len");
  if (step < 0) return set_err(MDG_E_INVALID, "negative step");
  if (n_envs <= 0) return n_envs == 0 ? MDG_OK : set_err(MDG_E_INVALID, "n_envs < 0");
  AppendArgs a;
  a.rp = *rp; a.N = n_envs; a.step = step; a.action = action; a.shaped = shaped_reward; a.n_popped = n_popped;
  a.nstep_len = nstep_len; a.done = done;
  replay_append_kernel<<<(unsigned)((n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_replay_append launch");
}

extern "C" int mdg_replay_sample(const MdgReplay* rp, int64_t n_envs, int64_t cur_step, const void* obs_price,
                                 const double* obs_port, int32_t window_elems, int32_t n_port, int32_t obs_dtype,
                                 int64_t batch, uint64_t seed, uint64_t draw, const MdgReplayBatch* out,
                                 void* stream) {
  int rc = check_replay(rp);
  if (rc) return rc;
  rc = check_gather(obs_price, obs_port, window_elems, n_port, obs_dtype, out);
  if (rc) return rc;
  if (batch <= 0) return batch == 0 ? MDG_OK : set_err(MDG_E_INVALID, "batch < 0");
  SampleArgs a;
  a.rp = *rp; a.cur_step = cur_step; a.batch = batch; a.seed = seed; a.draw = draw;
  a.g.N = n_envs; a.g.obs_price = obs_price; a.g.obs_port = obs_port; a.g.welems = window_elems; a.g.n_port = n_port;
  a.g.dtype = obs_dtype; a.g.out = *out;
  replay_sample_kernel<<<(unsigned)batch, kGatherThreads, 0, (cudaStream_t)stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_replay_sample launch");
}

extern "C" int mdg_replay_rows_ingest(const MdgReplayRows* rows, const MdgWindow* w, int64_t slot,
                                      int32_t whole_window) {
  int rc = check_rows(rows, 1);
  if (rc) return rc;
  if (!w || !w->ring || !w->prefix || !w->timestamp || !w->reset_ts)
    return set_err(MDG_E_INVALID, "null window ring/prefix/timestamp/reset_ts");
  if (w->n_feats != rows->n_feats || w->window != rows->window)
    return set_err(MDG_E_INVALID, "window shape != replay rows shape");
  if (w->n_valid != w->window) return set_err(MDG_E_INVALID, "replay rows need a full window (n_valid == window)");
  if (w->head < 0 || w->head >= w->window) return set_err(MDG_E_INVALID, "bad head");
  if (slot < 0) return set_err(MDG_E_INVALID, "negative slot");
  if (w->n_envs <= 0) return w->n_envs == 0 ? MDG_OK : set_err(MDG_E_INVALID, "n_envs < 0");
  RowsIngestArgs a;
  a.rw = *rows; a.ring = w->ring; a.prefix = w->prefix; a.timestamp = w->timestamp; a.reset_ts = w->reset_ts;
  a.N = w->n_envs; a.slot = slot; a.head = w->head; a.whole = whole_window != 0;
  replay_rows_ingest_kernel<<<(unsigned)((a.N + kIngestEnvs - 1) / kIngestEnvs), 256, 0, (cudaStream_t)w->stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_replay_rows_ingest launch");
}

extern "C" int mdg_replay_sample_rows(const MdgReplay* rp, const MdgReplayRows* rows, int64_t n_envs, int64_t cur_step,
                                      const double* obs_port, int32_t n_port, int32_t norm_type, int32_t out_dtype,
                                      int64_t batch, uint64_t seed, uint64_t draw, const MdgReplayBatch* out,
                                      void* stream) {
  int rc = check_replay(rp);
  if (!rc) rc = check_rows_sample(rows, rp, obs_port, n_port, norm_type, out_dtype, out);
  if (rc) return rc;
  if (batch <= 0) return batch == 0 ? MDG_OK : set_err(MDG_E_INVALID, "batch < 0");
  const size_t smem = rows_gather_smem(*rows);
  static size_t smem_allowed = 48 * 1024;
  rc = rows_gather_smem_attr(replay_sample_rows_kernel, smem, &smem_allowed);
  if (rc) return rc;
  SampleRowsArgs a;
  a.rp = *rp; a.cur_step = cur_step; a.seed = seed; a.draw = draw;
  a.g.N = n_envs; a.g.rw = *rows; a.g.obs_port = obs_port; a.g.n_port = n_port; a.g.dtype = out_dtype;
  a.g.norm = norm_type; a.g.out = *out;
  replay_sample_rows_kernel<<<(unsigned)batch, kGatherThreads, smem, (cudaStream_t)stream>>>(a);
  return cuda_err(cudaGetLastError(), "mdg_replay_sample_rows launch");
}
