// Row-sharded tables over NVLink peer memory (SURVEY.md 8(e)): one process per GPU, every rank maps
// every other rank's shard / staging buffers into its own address space (CUDA IPC over NVLink P2P) and the
// exchange steps are plain loads inside the kernels -- no all-to-all, no host synchronisation, so the
// whole multi-GPU training step replays as one CUDA graph per rank.
//
//   peer_gather_rows   out[i] = shard[id % G][id / G]      (forward "fetch": P2P 128-bit row loads)
//   peer_fold_lists    owner-side gradient fold of all peers' compact (sorted unique rows, values) lists in two
//                      launches (mark + leader sum, see below): rank-ordered sums, no float atomics
//   peer_allreduce     one-shot sum of the replicated dense gradients: every rank reads all G buffers and
//                      adds them in rank order (bit-identical result on every rank)
//   peer_barrier       cross-GPU barrier on flag words in peer memory (release/acquire at system scope),
//                      with a clock64 time-out that raises a device error flag instead of hanging
#include <string.h>

#include "psb_common.cuh"
#include "adam_common.cuh"

namespace psb {

constexpr int kMaxPeers = 16;

struct PeerPtrs {
  const void* p[kMaxPeers];
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// flags.p[r] = rank r's flag block (uint32[kMaxPeers], in r's peer memory).  Thread t signals peer t by writing
// the new epoch into flags[t][rank] and waits until flags[rank][t] reaches it.
__global__ void __launch_bounds__(32) peer_barrier_kernel(PeerPtrs flags, int rank, int G, uint32_t* __restrict__ epoch,
                                                          int32_t* __restrict__ err, long long timeout_cycles,
                                                          unsigned long long* __restrict__ wait_cycles, int slot) {
  __shared__ uint32_t e_sh;
  const int t = threadIdx.x;
  const long long t_in = clock64();
  if (t == 0) {
    e_sh = *epoch + 1u;
    *epoch = e_sh;
  }
  __syncthreads();
  const uint32_t e = e_sh;
  if (t < G) {
    __threadfence_system();
    uint32_t* theirs = static_cast<uint32_t*>(const_cast<void*>(flags.p[t])) + rank;
    st_release_sys(theirs, e);
    const uint32_t* mine = static_cast<const uint32_t*>(flags.p[rank]) + t;
    const long long t0 = clock64();
    while (static_cast<int32_t>(ld_acquire_sys(mine) - e) < 0) {
      if (clock64() - t0 > timeout_cycles) {
        if (err != nullptr) *err = 1 + t;
        break;
      }
      __nanosleep(64);
    }
    __threadfence_system();
  }
  if (wait_cycles != nullptr) {   // time this rank spent in the barrier, per position of the barrier in the step
    __syncwarp();
    if (t == 0) wait_cycles[slot & 3] += static_cast<unsigned long long>(clock64() - t_in);
  }
}

// Peer rows are loaded like local gathers (ldg_row4, the non-coherent path): the plain coherent and the system-scope
// loads measured within 5 % of it on an isolated remote fetch (profiles/r02j_peer_bw_n2.jsonl, r02m_peer_bw_n2.jsonl).
template <int R>
__global__ void __launch_bounds__(256)
peer_gather_rows_kernel(PeerPtrs shards, int G, int64_t rows_total, int d4, const int64_t* __restrict__ idx, int64_t n,
                        float4* __restrict__ out, int64_t* __restrict__ remap, int64_t pad_id, int64_t pad_pos,
                        int32_t* __restrict__ err) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  const int64_t warp = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  for (int64_t base = warp * R; base < n; base += nwarps * R) {
    const float4* src[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int64_t row = base + i;
      src[i] = nullptr;
      if (row < n) {
        const int64_t v = idx[row];
        if (remap != nullptr && lane == 0) remap[row] = v == pad_id ? pad_pos : row;
        if (v < 0 || v >= rows_total) {
          if (err != nullptr && lane == 0) *err = 1;
        } else if (remap != nullptr && v == pad_id && row != pad_pos) {
          // a pad entry is read at pad_pos, never at its own position: do not fetch the pad row thousands of
          // times from its one owner (same-address peer reads serialise on that GPU's memory system)
        } else {
          // ids fit 31 bits (rows_total < 2^31 is checked on the host): 32-bit divide instead of the 64-bit routine
          const uint32_t u = static_cast<uint32_t>(v), g = static_cast<uint32_t>(G);
          const uint32_t q = u / g;
          src[i] = static_cast<const float4*>(shards.p[u - q * g]) + static_cast<int64_t>(q) * d4;
        }
      }
    }
    for (int c = lane; c < d4; c += 32) {
      float4 v[R];
#pragma unroll
      for (int i = 0; i < R; ++i) v[i] = src[i] != nullptr ? ldg_row4(src[i] + c) : zero4();
#pragma unroll
      for (int i = 0; i < R; ++i)
        if (base + i < n) stg4(out + (base + i) * d4 + c, v[i]);
    }
  }
}

// The same fetch from a table whose owners run the row-sparse Adam (psb_peer_gather_rows_lazy): a row that rests on its
// owner is handed out as it WOULD be after the dense sweep -- value + catch-up series from the row's moments -- and
// nothing is written back.  R rows per warp: their last_step words first (one remote 4-byte load each, all in flight),
// then the value rows; only the resting ones pay the two extra row loads and the series.
struct LazyShards {
  const void* p[kMaxPeers];
  const void* m[kMaxPeers];
  const void* v[kMaxPeers];
  const void* last[kMaxPeers];
};

template <int R>
__global__ void __launch_bounds__(256)
peer_gather_rows_lazy_kernel(LazyShards S, int G, int64_t rows_total, int d4, const int64_t* __restrict__ idx, int64_t n,
                             float4* __restrict__ out, int64_t* __restrict__ remap, int64_t pad_id, int64_t pad_pos,
                             int32_t* __restrict__ err, const AdamHyper h, const int64_t* __restrict__ step_dev,
                             const float2* __restrict__ hist, int64_t hist_cap, int catchup_max) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  const int64_t warp = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t cur = *step_dev;
  for (int64_t base = warp * R; base < n; base += nwarps * R) {
    int owner[R];
    int64_t local[R];
    int last[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int64_t row = base + i;
      owner[i] = -1;
      local[i] = 0;
      last[i] = 0;
      if (row < n) {
        const int64_t v = idx[row];
        if (remap != nullptr && lane == 0) remap[row] = v == pad_id ? pad_pos : row;
        if (v < 0 || v >= rows_total) {
          if (err != nullptr && lane == 0) *err = 1;
        } else if (remap != nullptr && v == pad_id && row != pad_pos) {
          // pad entries are read once, at pad_pos (see peer_gather_rows_kernel)
        } else {
          const uint32_t u = static_cast<uint32_t>(v), g = static_cast<uint32_t>(G);
          const uint32_t q = u / g;
          owner[i] = static_cast<int>(u - q * g);
          local[i] = q;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < R; ++i)
      if (owner[i] >= 0) last[i] = static_cast<const int*>(S.last[owner[i]])[local[i]];
    for (int c = lane; c < d4; c += 32) {          // d <= 128: one trip
      float4 v[R];
#pragma unroll
      for (int i = 0; i < R; ++i)
        v[i] = owner[i] >= 0 ? ldg_row4(static_cast<const float4*>(S.p[owner[i]]) + local[i] * d4 + c) : zero4();
#pragma unroll
      for (int i = 0; i < R; ++i) {
        if (owner[i] >= 0 && last[i] > 0 && last[i] < cur) {   // warp-uniform: every lane holds the same owner / last
          const float4 m = ldg_row4(static_cast<const float4*>(S.m[owner[i]]) + local[i] * d4 + c);
          const float4 vv = ldg_row4(static_cast<const float4*>(S.v[owner[i]]) + local[i] * d4 + c);
          const int64_t gap = cur - last[i];
          const float4 dl = catchup_series4(m, vv, last[i], static_cast<int>(gap < catchup_max ? gap : catchup_max), h, hist,
                                            hist_cap);
          v[i] = make_float4(v[i].x - dl.x, v[i].y - dl.y, v[i].z - dl.z, v[i].w - dl.w);
        }
      }
#pragma unroll
      for (int i = 0; i < R; ++i)
        if (base + i < n) stg4(out + (base + i) * d4 + c, v[i]);
    }
  }
}

// ---- owner-side gradient fold ---------------------------------------------------------------------------
// Every peer r publishes a compact list (rows_r[0..n_r) ascending unique GLOBAL ids, vals_r[i,:]).  The owner of
// a row must add the peers' values in rank order (reproducible) without atomics and without a launch per peer:
//   mark  posmap[r][local] = (stamp, i + 1) for every slot (r, i) this rank owns          (parallel, no conflicts)
//   sum   the slot of the LOWEST peer holding a row is its leader: it walks the later peers' posmap entries,
//         adds their value rows in rank order and OVERWRITES dense[local] once            (parallel, no RMW)
// posmap entries carry a stamp that is constant during one fold and different for the next one (the barrier
// epoch), so the map never needs clearing.
struct FoldTable {
  const int32_t* rows[kMaxPeers];
  const float4* vals[kMaxPeers];
  const int32_t* n_rows[kMaxPeers];
  int64_t cap, shard_rows;
  int d4;
  unsigned long long* posmap;  // [G][shard_rows]
  float4* dense;
  int32_t* touched;            // optional [G * cap]: local rows written (for the next step's row-wise zeroing)
  int32_t* n_touched;
};

struct FoldArgs {
  FoldTable t[2];
  int n_tables, rank, G;
  float scale;
  const uint32_t* stamp;
  int entries_per_warp;
};

template <bool SUM>
__global__ void __launch_bounds__(256) peer_fold_kernel(const FoldArgs a) {
  const FoldTable& t = a.t[blockIdx.y];
  const int r = blockIdx.z, G = a.G, rank = a.rank;
  const int lane = threadIdx.x & 31;
  const unsigned long long stamp = static_cast<unsigned long long>(*a.stamp) << 32;
  int64_t n = *t.n_rows[r];
  n = n < t.cap ? n : t.cap;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  const int64_t w0 = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (!SUM) {
    for (int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x); i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
      const int32_t g = t.rows[r][i];
      if (g < 0 || g % G != rank) continue;
      const int64_t local = g / G;
      if (local < t.shard_rows) t.posmap[r * t.shard_rows + local] = stamp | static_cast<unsigned long long>(i + 1);
    }
    return;
  }
  // SUM: a warp takes 32 consecutive entries of peer r's list with ONE coalesced peer load (the first version read
  // them one per warp iteration: a dependent NVLink round trip per entry), every lane resolves its own entry --
  // owned here? is r the lowest peer holding the row? at which slot do the later peers hold it? -- from the local
  // position map, then the warp folds the leader entries one after the other, 128-bit peer loads across the lanes.
  // E entries per warp and iteration: ~1 / G of them are owned here and are folded one after the other, so E grows
  // with G (4 G, at most 32) to keep ~4 serial folds per warp whatever the number of ranks
  const int E = a.entries_per_warp;
  for (int64_t i0 = w0 * E; i0 < n; i0 += nwarps * E) {
    const int64_t i = i0 + lane;
    const int32_t g = (lane < E && i < n) ? t.rows[r][i] : -1;
    const int64_t local = g >= 0 ? g / G : 0;
    bool leader = g >= 0 && g % G == rank && local < t.shard_rows;
    int32_t slot[kMaxPeers];
#pragma unroll
    for (int q = 0; q < kMaxPeers; ++q) slot[q] = -1;
    if (leader) {
#pragma unroll
      for (int q = 0; q < kMaxPeers; ++q) {
        if (q < G && q != r) {
          const unsigned long long e = t.posmap[q * t.shard_rows + local];
          const bool held = (e >> 32 << 32) == stamp;
          if (q < r && held) leader = false;
          if (q > r && held) slot[q] = static_cast<int32_t>(e & 0xffffffffull) - 1;
        }
        if (q == r) slot[q] = static_cast<int32_t>(i);
      }
    }
    // (measured at N = 8, profiles/r02A_bench_n8.json: folding four leaders per round in 8-lane groups -- more rows in
    // flight, but 128-byte instead of 512-byte peer requests -- is SLOWER: 86 vs 54 us; one leader per round stays)
    unsigned todo = __ballot_sync(kFull, leader);
    while (todo != 0u) {
      const int l = __ffs(todo) - 1;
      todo &= todo - 1;
      const int64_t row = __shfl_sync(kFull, local, l);
      int32_t sl[kMaxPeers];
#pragma unroll
      for (int q = 0; q < kMaxPeers; ++q) sl[q] = __shfl_sync(kFull, slot[q], l);
      for (int c = lane; c < t.d4; c += 32) {
        float4 acc = zero4();
#pragma unroll
        for (int q = 0; q < kMaxPeers; ++q) {
          if (sl[q] >= 0) {
            const float4 v = ldg_row4(t.vals[q] + static_cast<int64_t>(sl[q]) * t.d4 + c);
            acc.x += v.x;
            acc.y += v.y;
            acc.z += v.z;
            acc.w += v.w;
          }
        }
        acc.x *= a.scale;
        acc.y *= a.scale;
        acc.z *= a.scale;
        acc.w *= a.scale;
        t.dense[row * t.d4 + c] = acc;
      }
      if (t.touched != nullptr && lane == 0) t.touched[atomicAdd(t.n_touched, 1)] = static_cast<int32_t>(row);
    }
  }
}

// Loads are issued in a STAGGERED peer order (rank, rank + 1, ...: every rank starts with a different source, so
// no GPU's NVLink egress serves all readers at once) but added in rank order 0..G-1, so every rank computes the
// bit-identical sum.
__global__ void __launch_bounds__(256)
peer_allreduce_kernel(PeerPtrs bufs, int G, int rank, int64_t n, float scale, float* __restrict__ out) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t n4 = n >> 2;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v[kMaxPeers];
#pragma unroll
    for (int j = 0; j < kMaxPeers; ++j) {
      if (j < G) {
        int r = rank + j;
        r = r >= G ? r - G : r;
        const float4 x = ldg_row4(static_cast<const float4*>(bufs.p[r]) + i);
        // place by source rank without dynamic register indexing
#pragma unroll
        for (int q = 0; q < kMaxPeers; ++q)
          if (q == r) v[q] = x;
      }
    }
    float4 acc = zero4();
#pragma unroll
    for (int q = 0; q < kMaxPeers; ++q) {
      if (q < G) {
        acc.x += v[q].x;
        acc.y += v[q].y;
        acc.z += v[q].z;
        acc.w += v[q].w;
      }
    }
    acc.x *= scale;
    acc.y *= scale;
    acc.z *= scale;
    acc.w *= scale;
    reinterpret_cast<float4*>(out)[i] = acc;
  }
  for (int64_t i = (n4 << 2) + static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    float acc = 0.f;
    for (int r = 0; r < G; ++r) acc += static_cast<const float*>(bufs.p[r])[i];
    out[i] = acc * scale;
  }
}

// total squared gradient norm = sum over ranks of the published partial norms (rank order); optionally advances
// the optimizer's step counter so psb_adam_step(norm_given = 2) needs no launch of its own for it.
__global__ void peer_sum_sqnorm_kernel(PeerPtrs slots, int G, float* __restrict__ out, int64_t* __restrict__ step) {
  float acc = 0.f;
  for (int r = 0; r < G; ++r) acc += *static_cast<const float*>(slots.p[r]);
  *out = acc;
  if (step != nullptr) *step += 1;
}

// Norm exchange in ONE launch: finish this rank's partial sums (fixed order, double), publish the shard norm in this
// rank's peer-visible slot, cross-GPU barrier, sum the G slots in rank order, advance the optimizer's step counter.
// (Three launches before: sqnorm_final, peer_barrier, peer_sum_sqnorm.)
__global__ void __launch_bounds__(256)
peer_norm_exchange_kernel(const float* __restrict__ partial, int n_partial, PeerPtrs slots, PeerPtrs flags, int rank, int G,
                          uint32_t* __restrict__ epoch, int32_t* __restrict__ err, long long timeout_cycles,
                          unsigned long long* __restrict__ wait_cycles, int slot, float* __restrict__ out,
                          int64_t* __restrict__ step) {
  __shared__ double wsum[8];
  __shared__ uint32_t e_sh;
  const int t = threadIdx.x;
  double acc = 0.0;
  const int per = (n_partial + 255) / 256;
  const int lo = t * per, hi = min(n_partial, lo + per);
  for (int i = lo; i < hi; ++i) acc += static_cast<double>(partial[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
  if ((t & 31) == 0) wsum[t >> 5] = acc;
  __syncthreads();
  const long long t_in = clock64();
  if (t == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += wsum[w];
    *static_cast<float*>(const_cast<void*>(slots.p[rank])) = static_cast<float>(s);
    e_sh = *epoch + 1u;
    *epoch = e_sh;
  }
  __syncthreads();
  const uint32_t e = e_sh;
  if (t < G) {
    __threadfence_system();
    uint32_t* theirs = static_cast<uint32_t*>(const_cast<void*>(flags.p[t])) + rank;
    st_release_sys(theirs, e);
    const uint32_t* mine = static_cast<const uint32_t*>(flags.p[rank]) + t;
    const long long t0 = clock64();
    while (static_cast<int32_t>(ld_acquire_sys(mine) - e) < 0) {
      if (clock64() - t0 > timeout_cycles) {
        if (err != nullptr) *err = 1 + t;
        break;
      }
      __nanosleep(64);
    }
    __threadfence_system();
  }
  __syncthreads();
  if (t == 0) {
    float total = 0.f;
    for (int r = 0; r < G; ++r) total += *static_cast<const volatile float*>(slots.p[r]);
    *out = total;
    if (step != nullptr) *step += 1;
    if (wait_cycles != nullptr) wait_cycles[slot & 3] += static_cast<unsigned long long>(clock64() - t_in);
  }
}

}  // namespace psb

using namespace psb;

static int fill_ptrs(PeerPtrs* P, const void* const* host_ptrs, int32_t G);

extern "C" int psb_peer_norm_exchange(const psb_adam_tensor_t* dense, int32_t n_dense, const psb_adam_rows_t* tables,
                                      int32_t n_tables, const void* const* slots, const void* const* flag_blocks,
                                      int32_t rank, int32_t G, uint32_t* epoch_dev, int32_t* err_dev,
                                      int64_t timeout_cycles, uint64_t* wait_cycles_dev, int32_t wait_slot,
                                      float* sqnorm_out, int64_t* step_dev, void* workspace, int64_t workspace_bytes,
                                      psb_stream_t stream) {
  PeerPtrs S, F;
  int st;
  if ((st = fill_ptrs(&S, slots, G)) != PSB_OK || (st = fill_ptrs(&F, flag_blocks, G)) != PSB_OK) return st;
  if (rank < 0 || rank >= G || epoch_dev == nullptr || sqnorm_out == nullptr || workspace == nullptr) return PSB_E_ARG;
  if (timeout_cycles <= 0) timeout_cycles = 4000000000ll;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int n_partial = 0;
  float* partial = static_cast<float*>(workspace);
  if ((st = sqnorm_partials(dense, n_dense, tables, n_tables, partial, workspace_bytes / 4, &n_partial, s)) != PSB_OK) return st;
  PSB_PROF("peer_norm_exchange_kernel", s);
  peer_norm_exchange_kernel<<<1, 256, 0, s>>>(partial, n_partial, S, F, rank, G, epoch_dev, err_dev, timeout_cycles,
                                              reinterpret_cast<unsigned long long*>(wait_cycles_dev), wait_slot, sqnorm_out,
                                              step_dev);
  return launch_status();
}

extern "C" int psb_peer_alloc(int64_t bytes, void** out) {
  if (bytes <= 0 || out == nullptr) return PSB_E_ARG;
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, static_cast<size_t>(bytes));
  if (e != cudaSuccess) return static_cast<int>(e);
  e = cudaMemset(p, 0, static_cast<size_t>(bytes));
  if (e != cudaSuccess) return static_cast<int>(e);
  *out = p;
  return PSB_OK;
}

extern "C" int psb_peer_free(void* p) {
  if (p == nullptr) return PSB_OK;
  cudaError_t e = cudaFree(p);
  return e == cudaSuccess ? PSB_OK : static_cast<int>(e);
}

extern "C" int psb_peer_export(void* p, void* handle) {
  static_assert(sizeof(cudaIpcMemHandle_t) == PSB_PEER_HANDLE_BYTES, "handle size");
  if (p == nullptr || handle == nullptr) return PSB_E_ARG;
  cudaError_t e = cudaIpcGetMemHandle(static_cast<cudaIpcMemHandle_t*>(handle), p);
  return e == cudaSuccess ? PSB_OK : static_cast<int>(e);
}

extern "C" int psb_peer_open(const void* handle, void** out) {
  if (handle == nullptr || out == nullptr) return PSB_E_ARG;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return static_cast<int>(e);
  *out = p;
  return PSB_OK;
}

extern "C" int psb_peer_close(void* p) {
  if (p == nullptr) return PSB_OK;
  cudaError_t e = cudaIpcCloseMemHandle(p);
  return e == cudaSuccess ? PSB_OK : static_cast<int>(e);
}

static int fill_ptrs(PeerPtrs* P, const void* const* host_ptrs, int32_t G) {
  if (host_ptrs == nullptr || G <= 0 || G > kMaxPeers) return PSB_E_ARG;
  for (int i = 0; i < kMaxPeers; ++i) P->p[i] = i < G ? host_ptrs[i] : nullptr;
  for (int i = 0; i < G; ++i)
    if (P->p[i] == nullptr) return PSB_E_ARG;
  return PSB_OK;
}

extern "C" int psb_peer_barrier(const void* const* flag_blocks, int32_t rank, int32_t G, uint32_t* epoch_dev,
                                int32_t* err_dev, int64_t timeout_cycles, uint64_t* wait_cycles_dev, int32_t wait_slot,
                                psb_stream_t stream) {
  PeerPtrs F;
  int st = fill_ptrs(&F, flag_blocks, G);
  if (st != PSB_OK) return st;
  if (rank < 0 || rank >= G || epoch_dev == nullptr) return PSB_E_ARG;
  if (timeout_cycles <= 0) timeout_cycles = 4000000000ll;  // ~2 s at 1.9 GHz
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PSB_PROF("peer_barrier_kernel", s);
  peer_barrier_kernel<<<1, 32, 0, s>>>(F, rank, G, epoch_dev, err_dev, timeout_cycles,
                                       reinterpret_cast<unsigned long long*>(wait_cycles_dev), wait_slot);
  return launch_status();
}

extern "C" int psb_peer_gather_rows(const void* const* shards, int32_t G, int64_t rows_total, int64_t d,
                                    const int64_t* idx, int64_t n, float* out, int64_t* remap_out, int64_t pad_id,
                                    int64_t pad_pos, int32_t* err_flag, psb_stream_t stream) {
  PeerPtrs S;
  int st = fill_ptrs(&S, shards, G);
  if (st != PSB_OK) return st;
  if (idx == nullptr || out == nullptr || n < 0 || rows_total <= 0) return PSB_E_ARG;
  if (d <= 0 || (d & 3) != 0 || d > 512) return PSB_E_DIM;
  for (int i = 0; i < G; ++i)
    if (misaligned16(S.p[i])) return PSB_E_ALIGN;
  if (misaligned16(out)) return PSB_E_ALIGN;
  if (n == 0) return PSB_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (rows_total >= (1ll << 31)) return PSB_E_DIM;
  constexpr int R = 8;
  PSB_PROF("peer_gather_rows_kernel", s);
  peer_gather_rows_kernel<R><<<grid_for(n, 8 * R), 256, 0, s>>>(S, G, rows_total, static_cast<int>(d / 4), idx, n,
                                                                reinterpret_cast<float4*>(out), remap_out, pad_id, pad_pos,
                                                                err_flag);
  return launch_status();
}

extern "C" int32_t psb_adam_catchup_steps(double beta1, double beta2);

extern "C" int psb_peer_gather_rows_lazy(const void* const* shards_p, const void* const* shards_m,
                                         const void* const* shards_v, const void* const* shards_last, int32_t G,
                                         int64_t rows_total, int64_t d, const int64_t* idx, int64_t n, float* out,
                                         int64_t* remap_out, int64_t pad_id, int64_t pad_pos, int32_t* err_flag, double lr,
                                         double beta1, double beta2, double eps, int32_t noam, double warmup_steps,
                                         const int64_t* step_dev, const float* coef_hist, int64_t coef_cap,
                                         psb_stream_t stream) {
  PeerPtrs P, M, V, L;
  int st;
  if ((st = fill_ptrs(&P, shards_p, G)) != PSB_OK || (st = fill_ptrs(&M, shards_m, G)) != PSB_OK ||
      (st = fill_ptrs(&V, shards_v, G)) != PSB_OK || (st = fill_ptrs(&L, shards_last, G)) != PSB_OK)
    return st;
  if (idx == nullptr || out == nullptr || n < 0 || rows_total <= 0 || step_dev == nullptr) return PSB_E_ARG;
  if (d <= 0 || (d & 3) != 0 || d > 128) return PSB_E_DIM;          // the series runs on one float4 per lane
  if (rows_total >= (1ll << 31)) return PSB_E_DIM;
  for (int i = 0; i < G; ++i)
    if (misaligned16(P.p[i]) || misaligned16(M.p[i]) || misaligned16(V.p[i])) return PSB_E_ALIGN;
  if (misaligned16(out)) return PSB_E_ALIGN;
  if (n == 0) return PSB_OK;
  LazyShards S;
  for (int i = 0; i < kMaxPeers; ++i) {
    S.p[i] = P.p[i];
    S.m[i] = M.p[i];
    S.v[i] = V.p[i];
    S.last[i] = L.p[i];
  }
  const AdamHyper h = make_adam_hyper(lr, beta1, beta2, eps, 0.0, 0.0, noam, warmup_steps);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  constexpr int R = 8;
  PSB_PROF("peer_gather_rows_lazy_kernel", s);
  peer_gather_rows_lazy_kernel<R><<<grid_for(n, 8 * R), 256, 0, s>>>(
      S, G, rows_total, static_cast<int>(d / 4), idx, n, reinterpret_cast<float4*>(out), remap_out, pad_id, pad_pos,
      err_flag, h, step_dev, reinterpret_cast<const float2*>(coef_hist), coef_cap, psb_adam_catchup_steps(beta1, beta2));
  return launch_status();
}

extern "C" int psb_peer_fold_lists(const psb_fold_table_t* tables, int32_t n_tables, int32_t rank, int32_t G,
                                   float scale, const uint32_t* stamp_dev, psb_stream_t stream) {
  if (tables == nullptr || n_tables <= 0 || n_tables > 2 || G <= 0 || G > kMaxPeers || rank < 0 || rank >= G ||
      stamp_dev == nullptr)
    return PSB_E_ARG;
  FoldArgs a;
  memset(&a, 0, sizeof(a));
  a.n_tables = n_tables;
  a.rank = rank;
  a.G = G;
  a.scale = scale;
  a.stamp = stamp_dev;
  int64_t cap_max = 0;
  for (int k = 0; k < n_tables; ++k) {
    const psb_fold_table_t& in = tables[k];
    if (in.posmap == nullptr || in.dense == nullptr || in.cap <= 0 || in.shard_rows <= 0)
      return PSB_E_ARG;
    if (in.d <= 0 || (in.d & 3) != 0 || in.d > 512) return PSB_E_DIM;
    if (misaligned16(in.dense)) return PSB_E_ALIGN;
    FoldTable& t = a.t[k];
    for (int r = 0; r < G; ++r) {
      if (in.rows[r] == nullptr || in.vals[r] == nullptr || in.n_rows[r] == nullptr) return PSB_E_ARG;
      if (misaligned16(in.vals[r])) return PSB_E_ALIGN;
      t.rows[r] = in.rows[r];
      t.vals[r] = reinterpret_cast<const float4*>(in.vals[r]);
      t.n_rows[r] = in.n_rows[r];
    }
    t.cap = in.cap;
    t.shard_rows = in.shard_rows;
    t.d4 = static_cast<int>(in.d / 4);
    t.posmap = reinterpret_cast<unsigned long long*>(in.posmap);
    t.dense = reinterpret_cast<float4*>(in.dense);
    t.touched = in.touched;
    t.n_touched = in.n_touched;
    cap_max = in.cap > cap_max ? in.cap : cap_max;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int st;
  {
    dim3 grid(grid_for(cap_max, 256, 2), n_tables, G);
    PSB_PROF("peer_fold_mark_kernel", s);
    peer_fold_kernel<false><<<grid, 256, 0, s>>>(a);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  // entries per warp and iteration (~1 / G of them are folded here, one after the other), measured at N = 8
  // (profiles/r02C_bench_n8_E*.json): 32 entries 55 us / 0.502 ms per step, 16 entries 45 us / 0.484 ms, 8 entries
  // 50 us / 0.489 ms -> about two leaders per warp and iteration
  a.entries_per_warp = 2 * G < 32 ? 2 * G : 32;
  if (a.entries_per_warp < 8) a.entries_per_warp = 8;
  dim3 grid(grid_for(cap_max, 8 * a.entries_per_warp, 2), n_tables, G);
  PSB_PROF("peer_fold_sum_kernel", s);
  peer_fold_kernel<true><<<grid, 256, 0, s>>>(a);
  return launch_status();
}

extern "C" int psb_peer_allreduce(const void* const* bufs, int32_t G, int32_t rank, int64_t n, float scale, float* out,
                                  psb_stream_t stream) {
  PeerPtrs B;
  int st = fill_ptrs(&B, bufs, G);
  if (st != PSB_OK) return st;
  if (out == nullptr || n < 0 || rank < 0 || rank >= G) return PSB_E_ARG;
  for (int i = 0; i < G; ++i)
    if (misaligned16(B.p[i])) return PSB_E_ALIGN;
  if (misaligned16(out)) return PSB_E_ALIGN;
  if (n == 0) return PSB_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PSB_PROF("peer_allreduce_kernel", s);
  peer_allreduce_kernel<<<grid_for(n, 256 * 4, 4), 256, 0, s>>>(B, G, rank, n, scale, out);
  return launch_status();
}

extern "C" int psb_peer_sum_sqnorm(const void* const* slots, int32_t G, float* sqnorm_out, int64_t* step_dev,
                                   psb_stream_t stream) {
  PeerPtrs S;
  int st = fill_ptrs(&S, slots, G);
  if (st != PSB_OK) return st;
  if (sqnorm_out == nullptr) return PSB_E_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PSB_PROF("peer_sum_sqnorm_kernel", s);
  peer_sum_sqnorm_kernel<<<1, 1, 0, s>>>(S, G, sqnorm_out, step_dev);
  return launch_status();
}
