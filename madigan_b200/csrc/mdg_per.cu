// Proportional prioritized replay over the device ring (include/madigan_b200.h, "Proportional prioritized replay").
#include <stdio.h>

#include "mdg_replay.cuh"

namespace mdg {

constexpr int kSubLeaves = 1024;  // leaves of one subtree rebuilt by one block of the refresh kernel
constexpr int kRefreshThreads = kSubLeaves / 2;
constexpr int kMaxRefreshBlocks = 1024;  // grid-stride beyond this
constexpr uint32_t kPerDrawTag = 0x80000000u;  // bit 31 of the second Philox counter word (mdg_replay_sample: 0)

__device__ __forceinline__ double min2(double a, double b) { return (b < a) ? b : a; }

// list subtree s for the next refresh (once: the first marker of the subtree appends it)
__device__ __forceinline__ void mark_dirty(const MdgPrioritized& p, int64_t s) {
  if (atomicExch(p.dirty + s, 1u) == 0u) p.dirty_list[atomicAdd(p.ctl, 1u)] = (int32_t)s;
}

__device__ __forceinline__ void set_leaf(const MdgPrioritized& p, int64_t slot, double v) {
  p.sum_tree[p.tree_size + slot] = v;
  p.min_tree[p.tree_size + slot] = v;
}

struct IngestArgs {
  MdgPrioritized pr;
  const unsigned long long* cursor;
};

// grid-stride over the positions [max(seen, cursor - capacity), cursor): each record's leaf becomes
// max_priority ** alpha.  The positions are consecutive, so a subtree's first position in the range (a slot that
// starts a subtree, or the range's first) is the one that marks it.  The last block to leave records the cursor.
__global__ void __launch_bounds__(256) per_ingest_kernel(const __grid_constant__ IngestArgs a) {
  const MdgPrioritized& p = a.pr;
  const unsigned long long cap = (unsigned long long)p.capacity;
  const unsigned long long hi = *a.cursor, seen = *p.seen;
  const unsigned long long lo = (hi > cap && hi - cap > seen) ? hi - cap : seen;
  if (lo < hi) {
    const double leaf = pow(*p.max_priority, p.alpha);
    for (unsigned long long pos = lo + (unsigned long long)blockIdx.x * 256 + threadIdx.x; pos < hi;
         pos += (unsigned long long)gridDim.x * 256) {
      const int64_t slot = (int64_t)(pos % cap);
      set_leaf(p, slot, leaf);
      p.leaf_pos[slot] = (int64_t)pos;
      if (slot % kSubLeaves == 0 || pos == lo) mark_dirty(p, slot / kSubLeaves);
    }
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0 && atomicAdd(p.ctl + 2, 1u) == gridDim.x - 1) {
    *p.seen = hi;
    p.ctl[2] = 0;
  }
}

struct RefreshArgs {
  MdgPrioritized pr;
};

// One block per listed subtree (grid-stride over the list): the 1023 internal nodes of both trees from the 1024
// leaves, level by level in shared memory.  The last block to leave then rebuilds the levels above the subtree roots
// (nodes [1, S), S = tree_size / 1024) and empties the list.
__global__ void __launch_bounds__(kRefreshThreads) per_refresh_kernel(const __grid_constant__ RefreshArgs a) {
  __shared__ double s_sum[kRefreshThreads], s_min[kRefreshThreads];
  __shared__ int s_last;
  const MdgPrioritized& p = a.pr;
  const int t = threadIdx.x;
  const int64_t S = p.tree_size / kSubLeaves;
  const uint32_t count = p.ctl[0];
  for (uint32_t i = blockIdx.x; i < count; i += gridDim.x) {
    const int64_t s = p.dirty_list[i];
    const int64_t root = S + s;
    const int64_t l = (root << 10) + 2 * t;  // this thread's two leaves
    double vs = p.sum_tree[l] + p.sum_tree[l + 1];
    double vm = min2(p.min_tree[l], p.min_tree[l + 1]);
    p.sum_tree[(root << 9) + t] = vs;
    p.min_tree[(root << 9) + t] = vm;
    s_sum[t] = vs;
    s_min[t] = vm;
    __syncthreads();
    for (int n = kRefreshThreads / 2, d = 8; n >= 1; n >>= 1, --d) {
      if (t < n) {
        vs = s_sum[2 * t] + s_sum[2 * t + 1];
        vm = min2(s_min[2 * t], s_min[2 * t + 1]);
      }
      __syncthreads();
      if (t < n) {
        s_sum[t] = vs;
        s_min[t] = vm;
        p.sum_tree[(root << d) + t] = vs;
        p.min_tree[(root << d) + t] = vm;
      }
      __syncthreads();
    }
    if (t == 0) p.dirty[s] = 0u;
  }
  __threadfence();
  __syncthreads();
  if (t == 0) s_last = atomicAdd(p.ctl + 1, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (count > 0) {
    for (int64_t lo = S >> 1; lo >= 1; lo >>= 1) {  // other blocks' roots and this block's levels: read from L2
      for (int64_t j = lo + t; j < 2 * lo; j += kRefreshThreads) {
        __stcg(p.sum_tree + j, __ldcg(p.sum_tree + 2 * j) + __ldcg(p.sum_tree + 2 * j + 1));
        __stcg(p.min_tree + j, min2(__ldcg(p.min_tree + 2 * j), __ldcg(p.min_tree + 2 * j + 1)));
      }
      __threadfence_block();
      __syncthreads();
    }
  }
  if (t == 0) {
    p.ctl[0] = 0u;
    p.ctl[1] = 0u;
  }
}

struct DescentArgs {
  MdgPrioritized pr;
  MdgReplay rp;
  int64_t cur_step, batch;
  double beta;
  uint64_t seed, draw;
  int64_t* idx;
  int64_t* pos;
  double* weights;
};

// one thread per sample: the proportional descent with rejection (a leaf `resident` refuses is redrawn too), then the
// importance weight
template <class Resident>
__device__ __forceinline__ void per_descend(const DescentArgs& a, Resident resident) {
  const int64_t b = (int64_t)blockIdx.x * 128 + threadIdx.x;
  if (b >= a.batch) return;
  const MdgPrioritized& p = a.pr;
  const int64_t T = p.tree_size;
  const unsigned long long cur = *a.rp.cursor;
  const unsigned long long filled = cur < (unsigned long long)p.capacity ? cur : (unsigned long long)p.capacity;
  const double total = p.sum_tree[1];
  const double seg = total / (double)a.batch;
  long long pick = -1;
  for (uint32_t attempt = 0; attempt < 64 && filled > 0 && total > 0.; ++attempt) {
    uint64_t x0, x1;
    philox4x32_10((uint32_t)b, (uint32_t)(b >> 32) ^ (attempt << 8) ^ kPerDrawTag, (uint32_t)a.draw,
                  (uint32_t)(a.draw >> 32), (uint32_t)a.seed, (uint32_t)(a.seed >> 32), x0, x1);
    const double u = (double)(x0 >> 11) * 0x1.0p-53;
    double mass = attempt == 0 ? u * seg + (double)b * seg : u * total;
    int64_t node = 1;
    while (node < T) {
      const double left = p.sum_tree[2 * node];
      if (left > mass) {
        node = 2 * node;
      } else {
        mass = mass - left;
        node = 2 * node + 1;
      }
    }
    const int64_t leaf = node - T;
    if (leaf >= p.capacity || p.leaf_pos[leaf] < 0 || !(p.sum_tree[node] > 0.)) continue;
    if (resident(leaf)) { pick = leaf; break; }
  }
  a.idx[b] = pick;
  if (pick < 0) {
    a.pos[b] = -1;
    a.weights[b] = 0.;
    return;
  }
  a.pos[b] = p.leaf_pos[pick];
  const double n = (double)filled;
  a.weights[b] = pow(p.sum_tree[T + pick] / total * n, -a.beta) / pow(p.min_tree[1] / total * n, -a.beta);
}

__global__ void __launch_bounds__(128, 8) per_descent_kernel(const __grid_constant__ DescentArgs a) {
  per_descend(a, [&](long long leaf) { return replay_resident(a.rp, leaf, a.cur_step); });
}

struct DescentRowsArgs {
  DescentArgs d;
  MdgReplayRows rw;
  int64_t N;
};

// per_descent_kernel over the row store: a record whose state rows were overwritten is rejected too
__global__ void __launch_bounds__(128, 8) per_descent_rows_kernel(const __grid_constant__ DescentRowsArgs a) {
  per_descend(a.d, [&](long long leaf) {
    return replay_resident(a.d.rp, leaf, a.d.cur_step) && rows_resident(a.d.rp, a.rw, a.N, leaf);
  });
}

struct PerGatherArgs {
  MdgReplay rp;
  GatherArgs g;
};

// one block per sample: the gather of mdg_replay_sample for the index the descent chose
__global__ void __launch_bounds__(kGatherThreads) per_gather_kernel(const __grid_constant__ PerGatherArgs a) {
  const int64_t b = blockIdx.x;
  replay_gather(a.rp, a.g, b, a.g.out.idx[b]);
}

struct PerGatherRowsArgs {
  MdgReplay rp;
  RowsGatherArgs g;
};

// one block per sample: the rows gather of mdg_replay_sample_rows for the index the descent chose
__global__ void __launch_bounds__(kGatherThreads) per_gather_rows_kernel(const __grid_constant__ PerGatherRowsArgs a) {
  const int64_t b = blockIdx.x;
  replay_gather_rows(a.rp, a.g, b, a.g.out.idx[b]);
}

struct UpdateArgs {
  MdgPrioritized pr;
  int64_t batch;
  const int64_t* idx;
  const int64_t* pos;
  const double* prio;
};

// pass 1, one thread per batch row: drop idx = -1 and overwritten records, count and drop bad priorities; every
// applicable row raises max_priority and bids its batch position for its leaf (the highest bid wins: last wins)
__global__ void __launch_bounds__(256) per_update_bid_kernel(const __grid_constant__ UpdateArgs a) {
  const int64_t b = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (b >= a.batch) return;
  const MdgPrioritized& p = a.pr;
  const int64_t i = a.idx[b];
  if (i < 0 || i >= p.capacity || p.leaf_pos[i] != a.pos[b]) return;
  const double q = a.prio[b];
  if (!(isfinite(q) && q > 0.)) {
    atomicAdd(p.n_rejected, 1ull);
    return;
  }
  atomicMax((unsigned long long*)p.max_priority, (unsigned long long)__double_as_longlong(q));  // q > 0: bits order
  atomicMax(p.batch_pos + i, (int32_t)b);
}

// pass 2: the winning row of each leaf writes it, resets the bid and marks the leaf's subtree
__global__ void __launch_bounds__(256) per_update_apply_kernel(const __grid_constant__ UpdateArgs a) {
  const int64_t b = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (b >= a.batch) return;
  const MdgPrioritized& p = a.pr;
  const int64_t i = a.idx[b];
  if (i < 0 || i >= p.capacity || p.batch_pos[i] != (int32_t)b) return;
  set_leaf(p, i, pow(a.prio[b], p.alpha));
  p.batch_pos[i] = -1;
  mark_dirty(p, i / kSubLeaves);
}

static int check_per(const MdgPrioritized* pr) {
  if (!pr) return set_err(MDG_E_INVALID, "null prioritized replay");
  if (!pr->sum_tree || !pr->min_tree || !pr->leaf_pos || !pr->batch_pos || !pr->dirty || !pr->dirty_list ||
      !pr->ctl || !pr->seen || !pr->max_priority || !pr->n_rejected)
    return set_err(MDG_E_INVALID, "prioritized replay storage pointer is null");
  if (pr->capacity < 1 || pr->tree_size < kSubLeaves || (pr->tree_size & (pr->tree_size - 1)) ||
      pr->tree_size < pr->capacity || pr->capacity > INT32_MAX)
    return set_err(MDG_E_INVALID, "bad prioritized replay dimensions");
  if (!(pr->alpha >= 0.)) return set_err(MDG_E_INVALID, "alpha must be >= 0");
  return MDG_OK;
}

// one refresh launch sized for at most `max_marked` listed subtrees
static int launch_refresh(const MdgPrioritized* pr, int64_t max_marked, cudaStream_t st) {
  const int64_t S = pr->tree_size / kSubLeaves;
  int64_t grid = max_marked < S ? max_marked : S;
  if (grid > kMaxRefreshBlocks) grid = kMaxRefreshBlocks;
  if (grid < 1) grid = 1;
  RefreshArgs r;
  r.pr = *pr;
  per_refresh_kernel<<<(unsigned)grid, kRefreshThreads, 0, st>>>(r);
  return cuda_err(cudaGetLastError(), "per refresh launch");
}

}  // namespace mdg

using namespace mdg;

extern "C" int mdg_per_ingest(const MdgPrioritized* pr, const MdgReplay* rp, int64_t max_new, void* stream) {
  int rc = check_per(pr);
  if (!rc) rc = check_replay(rp);
  if (rc) return rc;
  if (rp->capacity != pr->capacity) return set_err(MDG_E_INVALID, "prioritized replay capacity != replay capacity");
  if (max_new < 0) return set_err(MDG_E_INVALID, "max_new < 0");
  const cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = max_new < pr->capacity ? max_new : pr->capacity;
  int64_t grid = (n + 255) / 256;
  if (grid > 4096) grid = 4096;  // grid-stride beyond
  if (grid < 1) grid = 1;
  IngestArgs a;
  a.pr = *pr;
  a.cursor = rp->cursor;
  per_ingest_kernel<<<(unsigned)grid, 256, 0, st>>>(a);
  rc = cuda_err(cudaGetLastError(), "mdg_per_ingest launch");
  if (rc) return rc;
  // consecutive slots: the range covers at most n / 1024 + 1 subtrees, + 1 where it wraps around the ring
  return launch_refresh(pr, n / kSubLeaves + 2, st);
}

extern "C" int mdg_per_sample(const MdgPrioritized* pr, const MdgReplay* rp, int64_t n_envs, int64_t cur_step,
                              const void* obs_price, const double* obs_port, int32_t window_elems, int32_t n_port,
                              int32_t obs_dtype, int64_t batch, double beta, uint64_t seed, uint64_t draw,
                              const MdgReplayBatch* out, double* weights, int64_t* pos, void* stream) {
  int rc = check_per(pr);
  if (!rc) rc = check_replay(rp);
  if (!rc) rc = check_gather(obs_price, obs_port, window_elems, n_port, obs_dtype, out);
  if (rc) return rc;
  if (rp->capacity != pr->capacity) return set_err(MDG_E_INVALID, "prioritized replay capacity != replay capacity");
  if (!weights || !pos) return set_err(MDG_E_INVALID, "null weights/pos output");
  if (!(beta >= 0.)) return set_err(MDG_E_INVALID, "beta must be >= 0");
  if (batch <= 0) return batch == 0 ? MDG_OK : set_err(MDG_E_INVALID, "batch < 0");
  const cudaStream_t st = (cudaStream_t)stream;
  DescentArgs d;
  d.pr = *pr; d.rp = *rp; d.cur_step = cur_step; d.batch = batch; d.beta = beta; d.seed = seed; d.draw = draw;
  d.idx = out->idx; d.pos = pos; d.weights = weights;
  per_descent_kernel<<<(unsigned)((batch + 127) / 128), 128, 0, st>>>(d);
  rc = cuda_err(cudaGetLastError(), "mdg_per_sample descent launch");
  if (rc) return rc;
  PerGatherArgs g;
  g.rp = *rp;
  g.g.N = n_envs; g.g.obs_price = obs_price; g.g.obs_port = obs_port; g.g.welems = window_elems; g.g.n_port = n_port;
  g.g.dtype = obs_dtype; g.g.out = *out;
  per_gather_kernel<<<(unsigned)batch, kGatherThreads, 0, st>>>(g);
  return cuda_err(cudaGetLastError(), "mdg_per_sample gather launch");
}

extern "C" int mdg_per_sample_rows(const MdgPrioritized* pr, const MdgReplay* rp, const MdgReplayRows* rows,
                                   int64_t n_envs, int64_t cur_step, const double* obs_port, int32_t n_port,
                                   int32_t norm_type, int32_t out_dtype, int64_t batch, double beta, uint64_t seed,
                                   uint64_t draw, const MdgReplayBatch* out, double* weights, int64_t* pos,
                                   void* stream) {
  int rc = check_per(pr);
  if (!rc) rc = check_replay(rp);
  if (!rc) rc = check_rows_sample(rows, rp, obs_port, n_port, norm_type, out_dtype, out);
  if (rc) return rc;
  if (rp->capacity != pr->capacity) return set_err(MDG_E_INVALID, "prioritized replay capacity != replay capacity");
  if (!weights || !pos) return set_err(MDG_E_INVALID, "null weights/pos output");
  if (!(beta >= 0.)) return set_err(MDG_E_INVALID, "beta must be >= 0");
  if (batch <= 0) return batch == 0 ? MDG_OK : set_err(MDG_E_INVALID, "batch < 0");
  const size_t smem = rows_gather_smem(*rows);
  static size_t smem_allowed = 48 * 1024;
  rc = rows_gather_smem_attr(per_gather_rows_kernel, smem, &smem_allowed);
  if (rc) return rc;
  const cudaStream_t st = (cudaStream_t)stream;
  DescentRowsArgs d;
  d.d.pr = *pr; d.d.rp = *rp; d.d.cur_step = cur_step; d.d.batch = batch; d.d.beta = beta; d.d.seed = seed;
  d.d.draw = draw; d.d.idx = out->idx; d.d.pos = pos; d.d.weights = weights;
  d.rw = *rows; d.N = n_envs;
  per_descent_rows_kernel<<<(unsigned)((batch + 127) / 128), 128, 0, st>>>(d);
  rc = cuda_err(cudaGetLastError(), "mdg_per_sample_rows descent launch");
  if (rc) return rc;
  PerGatherRowsArgs g;
  g.rp = *rp;
  g.g.N = n_envs; g.g.rw = *rows; g.g.obs_port = obs_port; g.g.n_port = n_port; g.g.dtype = out_dtype;
  g.g.norm = norm_type; g.g.out = *out;
  per_gather_rows_kernel<<<(unsigned)batch, kGatherThreads, smem, st>>>(g);
  return cuda_err(cudaGetLastError(), "mdg_per_sample_rows gather launch");
}

extern "C" int mdg_per_update(const MdgPrioritized* pr, int64_t batch, const int64_t* idx, const int64_t* pos,
                              const double* priorities, void* stream) {
  int rc = check_per(pr);
  if (rc) return rc;
  if (!idx || !pos || !priorities) return set_err(MDG_E_INVALID, "null update input");
  if (batch > INT32_MAX) return set_err(MDG_E_INVALID, "batch too large");
  if (batch <= 0) return batch == 0 ? MDG_OK : set_err(MDG_E_INVALID, "batch < 0");
  const cudaStream_t st = (cudaStream_t)stream;
  UpdateArgs a;
  a.pr = *pr; a.batch = batch; a.idx = idx; a.pos = pos; a.prio = priorities;
  const unsigned grid = (unsigned)((batch + 255) / 256);
  per_update_bid_kernel<<<grid, 256, 0, st>>>(a);
  rc = cuda_err(cudaGetLastError(), "mdg_per_update launch");
  if (rc) return rc;
  per_update_apply_kernel<<<grid, 256, 0, st>>>(a);
  rc = cuda_err(cudaGetLastError(), "mdg_per_update launch");
  if (rc) return rc;
  return launch_refresh(pr, batch, st);
}
