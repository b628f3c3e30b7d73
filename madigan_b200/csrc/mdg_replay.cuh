// The replay gathers shared by the uniform (mdg_replay.cu) and the prioritized (mdg_per.cu) samplers: stored windows
// (replay_gather) and the row store (replay_gather_rows).
#pragma once
#include "mdg_common.cuh"
#include "mdg_window_norm.cuh"

namespace mdg {

constexpr int kGatherThreads = 128;  // block size of every kernel that calls replay_gather

// Where the gather reads the observations and writes the batch (include/madigan_b200.h, mdg_replay_sample).
struct GatherArgs {
  int64_t N;
  const void* obs_price;
  const double* obs_port;
  int welems, n_port, dtype;
  MdgReplayBatch out;
};

// The record's fields but the windows: portfolio rows, action, reward and done of record idx (env e, state slot ss,
// next slot sn) into row b of the batch.
__device__ __forceinline__ void gather_record(const MdgReplay& r, int64_t N, const double* obs_port, int n_port,
                                              const MdgReplayBatch& out, int64_t b, long long idx, int64_t e,
                                              int64_t ss, int64_t sn) {
  constexpr int NT = kGatherThreads;
  for (int i = threadIdx.x; i < n_port; i += NT) {
    out.state_port[b * n_port + i] = obs_port[(ss * N + e) * n_port + i];
    out.next_port[b * n_port + i] = obs_port[(sn * N + e) * n_port + i];
  }
  for (int i = threadIdx.x; i < r.n_action; i += NT) out.action[b * r.n_action + i] = r.t_action[idx * r.n_action + i];
  for (int i = threadIdx.x; i < r.ra; i += NT) out.reward[b * r.ra + i] = r.t_reward[idx * r.ra + i];
  if (threadIdx.x == 0) out.done[b] = r.t_done[idx];
}

// Row b of the batch, written by the kGatherThreads threads of the calling block: record idx's two windows,
// portfolio rows, action, reward and done; idx < 0 (no resident transition found) gives a zero row with done = 1.
// out.idx is the caller's.
__device__ __forceinline__ void replay_gather(const MdgReplay& r, const GatherArgs& a, int64_t b, long long idx) {
  constexpr int NT = kGatherThreads;
  if (idx < 0) {
    const int64_t o_b = b * a.welems;
    if (a.dtype == MDG_DTYPE_F32) {
      float* d0 = (float*)a.out.state_price; float* d1 = (float*)a.out.next_price;
      for (int i = threadIdx.x; i < a.welems; i += NT) { d0[o_b + i] = 0.f; d1[o_b + i] = 0.f; }
    } else {
      double* d0 = (double*)a.out.state_price; double* d1 = (double*)a.out.next_price;
      for (int i = threadIdx.x; i < a.welems; i += NT) { d0[o_b + i] = 0.; d1[o_b + i] = 0.; }
    }
    for (int i = threadIdx.x; i < a.n_port; i += NT) { a.out.state_port[b * a.n_port + i] = 0.; a.out.next_port[b * a.n_port + i] = 0.; }
    for (int i = threadIdx.x; i < r.n_action; i += NT) a.out.action[b * r.n_action + i] = 0.;
    for (int i = threadIdx.x; i < r.ra; i += NT) a.out.reward[b * r.ra + i] = 0.;
    if (threadIdx.x == 0) a.out.done[b] = 1;
    return;
  }
  const int64_t e = r.t_env[idx];
  const int64_t ss = r.t_state_slot[idx], sn = r.t_next_slot[idx];
  const int64_t o_s = (ss * a.N + e) * a.welems, o_n = (sn * a.N + e) * a.welems, o_b = b * a.welems;
  if (a.dtype == MDG_DTYPE_F32) {
    const float* src = (const float*)a.obs_price;
    float* d0 = (float*)a.out.state_price;
    float* d1 = (float*)a.out.next_price;
    for (int i = threadIdx.x; i < a.welems; i += NT) { d0[o_b + i] = src[o_s + i]; d1[o_b + i] = src[o_n + i]; }
  } else {
    const double* src = (const double*)a.obs_price;
    double* d0 = (double*)a.out.state_price;
    double* d1 = (double*)a.out.next_price;
    for (int i = threadIdx.x; i < a.welems; i += NT) { d0[o_b + i] = src[o_s + i]; d1[o_b + i] = src[o_n + i]; }
  }
  gather_record(r, a.N, a.obs_port, a.n_port, a.out, b, idx, e, ss, sn);
}

// The staleness test of both samplers: the observation slot of the record's state has not been overwritten (a slot
// survives `depth` steps).  t_state_step = INT64_MIN marks a slot never written (step -1 is observe_start's slot).
__device__ __forceinline__ bool replay_resident(const MdgReplay& r, long long slot, int64_t cur_step) {
  const long long sstep = r.t_state_step[slot];
  return sstep != (-9223372036854775807LL - 1) && sstep > cur_step - r.depth;
}

// Where the rows gather reads the row store and writes the batch (include/madigan_b200.h, mdg_replay_sample_rows).
struct RowsGatherArgs {
  int64_t N;
  MdgReplayRows rw;
  const double* obs_port;
  int n_port, dtype, norm;
  MdgReplayBatch out;
};

// Dynamic shared memory of a block that runs replay_gather_rows: the two raw windows and a (shift, scale) per column.
static inline size_t rows_gather_smem(const MdgReplayRows& w) {
  return ((size_t)2 * w.window * w.n_feats + (size_t)4 * w.n_feats) * sizeof(double);
}

// The extra residency test of the row store: the state's k rows are still in its env's row ring (the next state's
// rows are newer).  row_end < k: the slot was never written.
__device__ __forceinline__ bool rows_resident(const MdgReplay& r, const MdgReplayRows& w, int64_t N, long long idx) {
  const int64_t e = r.t_env[idx];
  const int64_t end = w.row_end[(int64_t)r.t_state_slot[idx] * N + e];
  return end >= w.window && end - w.window + 1 > w.row_count[e] - w.n_rows;
}

// replay_gather over the row store: the two raw windows of record idx are loaded into shared memory (the rows of a
// window are one contiguous run of the env-major ring, or two where it wraps: coalesced 8-byte loads, eight in
// flight per thread), normalised there by normalise_windows -- thread (window, feature, z) owns one column, Z threads
// per column -- and written out in the output dtype.  idx < 0 gives replay_gather's zero row.
static __device__ __noinline__ void replay_gather_rows(const MdgReplay& r, const RowsGatherArgs& a, int64_t b,
                                                   long long idx) {
  constexpr int NT = kGatherThreads;
  extern __shared__ double rtile[];  // [2][k][F] raw windows (state, next), then [2][F] (shift, scale)
  const int k = a.rw.window, F = a.rw.n_feats, W = k * F;
  if (idx < 0) {  // uniform over the block
    GatherArgs g;
    g.N = a.N; g.obs_price = nullptr; g.obs_port = a.obs_port; g.welems = W; g.n_port = a.n_port; g.dtype = a.dtype;
    g.out = a.out;
    replay_gather(r, g, b, idx);
    return;
  }
  const int64_t e = r.t_env[idx];
  const int64_t ss = r.t_state_slot[idx], sn = r.t_next_slot[idx];
  const int64_t R = a.rw.n_rows, RF = R * F;
  // element offset of each window's oldest row in the env's ring
  const int64_t p_s = ((a.rw.row_end[ss * a.N + e] - k + 1) % R) * F;
  const int64_t p_n = ((a.rw.row_end[sn * a.N + e] - k + 1) % R) * F;
  const double* src = a.rw.rows + e * RF;
  constexpr int U = 8;
  for (int i0 = threadIdx.x; i0 < 2 * W; i0 += NT * U) {
    double v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * NT;
      v[u] = 0.;
      if (i < 2 * W) {
        int64_t j = i < W ? p_s + i : p_n + (i - W);
        if (j >= RF) j -= RF;
        v[u] = src[j];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * NT;
      if (i < 2 * W) rtile[i] = v[u];
    }
  }
  __syncthreads();
  {
    const int t = threadIdx.x, f = t % F, el = (t / F) & 1, z = t / (2 * F), Z = NT / (2 * F);
    struct { int norm, sstride, estride, envs; int64_t N; } tl = {a.norm, F, W, 2, 2};  // two windows, both real
    normalise_windows(tl, rtile, rtile + el * W + f, rtile + 2 * W + (el * F + f) * 2, k, F, F == 1, 0, z < Z, z,
                      Z);
  }
  __syncthreads();
  const int64_t o_b = b * W;
  if (a.dtype == MDG_DTYPE_F32) {
    float* d0 = (float*)a.out.state_price; float* d1 = (float*)a.out.next_price;
    for (int i = threadIdx.x; i < W; i += NT) { d0[o_b + i] = (float)rtile[i]; d1[o_b + i] = (float)rtile[W + i]; }
  } else {
    double* d0 = (double*)a.out.state_price; double* d1 = (double*)a.out.next_price;
    for (int i = threadIdx.x; i < W; i += NT) { d0[o_b + i] = rtile[i]; d1[o_b + i] = rtile[W + i]; }
  }
  gather_record(r, a.N, a.obs_port, a.n_port, a.out, b, idx, e, ss, sn);
}

static inline int check_replay(const MdgReplay* rp) {
  if (!rp) return set_err(MDG_E_INVALID, "null replay");
  if (!rp->t_env || !rp->t_state_slot || !rp->t_next_slot || !rp->t_state_step || !rp->t_done || !rp->t_reward ||
      !rp->t_action || !rp->cursor || !rp->act_ring)
    return set_err(MDG_E_INVALID, "replay storage pointer is null");
  if (rp->capacity < 1 || rp->depth < 2 || rp->nstep < 1 || rp->nstep > MDG_MAX_NSTEP || rp->ra < 1 || rp->n_action < 1)
    return set_err(MDG_E_INVALID, "bad replay dimensions");
  if (rp->depth <= rp->nstep) return set_err(MDG_E_INVALID, "replay depth must exceed nstep");
  return MDG_OK;
}

// Validation of a sample call's observation and batch arguments, shared by both samplers.
static inline int check_gather(const void* obs_price, const double* obs_port, int32_t window_elems, int32_t n_port,
                               int32_t obs_dtype, const MdgReplayBatch* out) {
  if (!obs_price || !obs_port || !out) return set_err(MDG_E_INVALID, "null sample input");
  if (!out->idx || !out->state_price || !out->next_price || !out->state_port || !out->next_port || !out->action ||
      !out->reward || !out->done)
    return set_err(MDG_E_INVALID, "null sample output");
  if (obs_dtype != MDG_DTYPE_F64 && obs_dtype != MDG_DTYPE_F32) return set_err(MDG_E_INVALID, "bad obs dtype");
  if (window_elems < 1 || n_port < 1) return set_err(MDG_E_INVALID, "bad window/portfolio size");
  return MDG_OK;
}

// Validation of the row store and of a rows sample call's window arguments.  depth: the observation slots the rows
// must outlive (MdgReplay.depth; 1 where the caller has none).
static inline int check_rows(const MdgReplayRows* w, int64_t depth) {
  if (!w) return set_err(MDG_E_INVALID, "null replay rows");
  if (!w->rows || !w->row_end || !w->row_count || !w->last_ts) return set_err(MDG_E_INVALID, "replay rows pointer is null");
  if (w->window < 1 || w->n_feats < 1) return set_err(MDG_E_INVALID, "bad replay rows dimensions");
  if (w->n_feats > 64) return set_err(MDG_E_UNSUPPORTED, "replay rows: n_feats must be in 1..64");
  if (w->n_rows < depth + w->window - 1) return set_err(MDG_E_INVALID, "replay rows: n_rows < depth + window - 1");
  return MDG_OK;
}

static inline int check_rows_sample(const MdgReplayRows* w, const MdgReplay* rp, const double* obs_port,
                                    int32_t n_port, int32_t norm_type, int32_t out_dtype, const MdgReplayBatch* out) {
  int rc = check_rows(w, rp->depth);
  if (rc) return rc;
  rc = check_gather(w->rows, obs_port, w->window * w->n_feats, n_port, out_dtype, out);
  if (rc) return rc;
  if (norm_type < MDG_NORM_NONE || norm_type > MDG_NORM_EXPANDING) return set_err(MDG_E_INVALID, "bad norm_type");
  if (rows_gather_smem(*w) > 200 * 1024) return set_err(MDG_E_UNSUPPORTED, "replay rows: windows do not fit shared memory");
  return MDG_OK;
}

// Opt a rows-gather kernel in to more than 48 KB of dynamic shared memory when its windows need it.
template <class Kernel>
static inline int rows_gather_smem_attr(Kernel kernel, size_t smem, size_t* allowed) {
  if (smem <= *allowed) return MDG_OK;
  const cudaError_t ce = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (ce != cudaSuccess) return cuda_err(ce, "replay rows gather smem attr");
  *allowed = smem;
  return MDG_OK;
}

}  // namespace mdg
