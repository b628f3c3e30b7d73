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
  if (threadIdx.x == 0) {
    const unsigned long long cur = *r.cursor;
    const unsigned long long filled = cur < (unsigned long long)r.capacity ? cur : (unsigned long long)r.capacity;
    long long pick = -1;
    for (uint32_t attempt = 0; attempt < 64 && filled > 0; ++attempt) {
      uint64_t x0, x1;
      philox4x32_10((uint32_t)b, (uint32_t)(b >> 32) ^ (attempt << 8), (uint32_t)a.draw, (uint32_t)(a.draw >> 32),
                    (uint32_t)a.seed, (uint32_t)(a.seed >> 32), x0, x1);
      const unsigned long long j = (unsigned long long)(((x0 >> 11) * 0x1.0p-53) * (double)filled);
      const long long cand = (long long)(j < filled ? j : filled - 1);
      if (replay_resident(r, cand, a.cur_step)) { pick = cand; break; }
    }
    s_idx = pick;
  }
  __syncthreads();
  const long long idx = s_idx;
  if (threadIdx.x == 0) a.g.out.idx[b] = idx;
  replay_gather(r, a.g, b, idx);
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
