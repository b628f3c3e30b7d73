// The replay gather shared by the uniform (mdg_replay.cu) and the prioritized (mdg_per.cu) samplers.
#pragma once
#include "mdg_common.cuh"

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
  for (int i = threadIdx.x; i < a.n_port; i += NT) {
    a.out.state_port[b * a.n_port + i] = a.obs_port[(ss * a.N + e) * a.n_port + i];
    a.out.next_port[b * a.n_port + i] = a.obs_port[(sn * a.N + e) * a.n_port + i];
  }
  for (int i = threadIdx.x; i < r.n_action; i += NT) a.out.action[b * r.n_action + i] = r.t_action[idx * r.n_action + i];
  for (int i = threadIdx.x; i < r.ra; i += NT) a.out.reward[b * r.ra + i] = r.t_reward[idx * r.ra + i];
  if (threadIdx.x == 0) a.out.done[b] = r.t_done[idx];
}

// The staleness test of both samplers: the observation slot of the record's state has not been overwritten (a slot
// survives `depth` steps).  t_state_step = INT64_MIN marks a slot never written (step -1 is observe_start's slot).
__device__ __forceinline__ bool replay_resident(const MdgReplay& r, long long slot, int64_t cur_step) {
  const long long sstep = r.t_state_step[slot];
  return sstep != (-9223372036854775807LL - 1) && sstep > cur_step - r.depth;
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

}  // namespace mdg
