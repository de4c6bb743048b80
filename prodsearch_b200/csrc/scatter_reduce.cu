// G2: deterministic embedding backward = stable LSD radix sort of (destination row, slot)
// pairs, segment detection, then a fixed-order segmented reduction (no float atomics).
//
// Two regimes, same arithmetic:
//   * n_total <= 16384 (a TEM step: ~10k item slots, ~7k word slots): ONE single-CTA
//     kernel packs keys, sorts them in shared memory (all radix passes), finds the
//     segments and writes the sorted slot list -> 2 launches per table per step.
//   * larger batches: multi-CTA radix sort (histogram / per-digit scan / stable scatter per
//     8-bit pass) + 3-kernel segment compaction.
// The reduction kernel (one warp per destination row, 128-bit row loads, 4 source rows in
// flight) is the HBM-bound part: algorithmic bytes = n_slots * d * 4 read (when sources
// are materialised rows) + n_unique * d * 4 written + metadata; sort traffic is overhead.
#include "psb_common.cuh"

namespace psb {

struct ContribTable {
  psb_contrib_t c[PSB_MAX_CONTRIBS];
  uint32_t off[PSB_MAX_CONTRIBS + 1];
  int n;
};

__device__ __forceinline__ int locate(const ContribTable& T, uint32_t slot) {
  int c = 0;
  while (c + 1 < T.n && slot >= T.off[c + 1]) ++c;
  return c;
}

__device__ __forceinline__ uint32_t make_key(const ContribTable& T, uint32_t slot, int64_t table_rows,
                                             int64_t drop_idx) {
  const int c = locate(T, slot);
  const int64_t r = T.c[c].idx[slot - T.off[c]];
  return (r < 0 || r >= table_rows || r == drop_idx) ? static_cast<uint32_t>(table_rows)
                                                       : static_cast<uint32_t>(r);
}

// Exclusive block scan of one int per thread.  `sm` holds NT/32 ints.
template <int NT>
__device__ __forceinline__ int block_excl_scan(int v, int* sm, int* total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(kFull, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) sm[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int t = lane < NT / 32 ? sm[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(kFull, t, o);
      if (lane >= o) t += u;
    }
    if (lane < NT / 32) sm[lane] = t;
  }
  __syncthreads();
  const int base = wid > 0 ? sm[wid - 1] : 0;
  if (total != nullptr) *total = sm[NT / 32 - 1];
  __syncthreads();
  return base + incl - v;
}

// Stable rank of every key of a tile among keys with the same 8-bit digit.
// Layout: warp w, round r, lane l  <->  tile position w*32*IPT + r*32 + l.
// On return pos[r] = position of the key in the tile sorted (stably) by digit,
// dstart[256] = first sorted position of each digit.  whist: [NT/32][256] ints.
template <int NT, int IPT, bool BALLOT = false>
__device__ __forceinline__ void tile_rank(const uint32_t (&key)[IPT], const bool (&valid)[IPT], int shift,
                                          int (&pos)[IPT], int* whist, int* dstart, int* scan_sm) {
  constexpr int NW = NT / 32;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const unsigned lt = (1u << lane) - 1u;
  for (int t = threadIdx.x; t < NW * 256; t += NT) whist[t] = 0;
  __syncthreads();
  int* mine = whist + wid * 256;
#pragma unroll
  for (int r = 0; r < IPT; ++r) {
    const int dg = valid[r] ? static_cast<int>((key[r] >> shift) & 255u) : 256;
    unsigned peers;
    if (BALLOT) {  // lanes with the same 9-bit value, from 9 votes (MATCH.ANY issues far slower on sm_100)
      peers = kFull;
#pragma unroll
      for (int bit = 0; bit < 9; ++bit) {
        const unsigned vote = __ballot_sync(kFull, (dg >> bit) & 1);
        peers &= ((dg >> bit) & 1) ? vote : ~vote;
      }
    } else {
      peers = __match_any_sync(kFull, dg);
    }
    const int leader = __ffs(peers) - 1;
    int old = 0;
    if (dg < 256) old = mine[dg];
    __syncwarp();
    if (dg < 256 && lane == leader) mine[dg] = old + __popc(peers);
    __syncwarp();
    pos[r] = old + __popc(peers & lt);
  }
  __syncthreads();
  int tot = 0;
  if (threadIdx.x < 256) {
    int run = 0;
#pragma unroll 4
    for (int w2 = 0; w2 < NW; ++w2) {
      const int c = whist[w2 * 256 + threadIdx.x];
      whist[w2 * 256 + threadIdx.x] = run;
      run += c;
    }
    tot = run;
  }
  const int ex = block_excl_scan<NT>(threadIdx.x < 256 ? tot : 0, scan_sm, nullptr);
  if (threadIdx.x < 256) dstart[threadIdx.x] = ex;
  __syncthreads();
#pragma unroll
  for (int r = 0; r < IPT; ++r) {
    if (valid[r]) {
      const int dg = static_cast<int>((key[r] >> shift) & 255u);
      pos[r] += dstart[dg] + mine[dg];
    }
  }
}

// ------------------------------------------------------------------------------------
// Small regime: everything up to the segment table in one CTA.
// ------------------------------------------------------------------------------------
constexpr int kSmallNT = 1024;
constexpr int kSmallIPT = 16;
constexpr int kSmallCap = kSmallNT * kSmallIPT;  // 16384 slots

__global__ void __launch_bounds__(kSmallNT, 1)
small_sort_segments_kernel(const __grid_constant__ ContribTable T, int n_total, int64_t table_rows, int64_t drop_idx, int passes,
                           uint32_t* __restrict__ sorted_slots, uint32_t* __restrict__ sorted_keys,
                           int32_t* __restrict__ seg_start, int32_t* __restrict__ unique_rows,
                           int32_t* __restrict__ n_unique, int32_t* __restrict__ work_count) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* sk = reinterpret_cast<uint32_t*>(smem_raw);          // [cap] keys
  uint32_t* sv = sk + kSmallCap;                                 // [cap] slots
  int* whist = reinterpret_cast<int*>(sv + kSmallCap);           // [32][256]
  int* dstart = whist + (kSmallNT / 32) * 256;                   // [256]
  int* scan_sm = dstart + 256;                                   // [32]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint32_t sentinel = static_cast<uint32_t>(table_rows);

  uint32_t key[kSmallIPT], val[kSmallIPT];
  bool valid[kSmallIPT];
  int pos[kSmallIPT];
#pragma unroll
  for (int r = 0; r < kSmallIPT; ++r) {
    const int p = wid * 32 * kSmallIPT + r * 32 + lane;
    valid[r] = p < n_total;
    val[r] = static_cast<uint32_t>(p);
    key[r] = valid[r] ? make_key(T, static_cast<uint32_t>(p), table_rows, drop_idx) : 0xffffffffu;
  }
  for (int pass = 0; pass < passes; ++pass) {
    tile_rank<kSmallNT, kSmallIPT>(key, valid, pass * 8, pos, whist, dstart, scan_sm);
#pragma unroll
    for (int r = 0; r < kSmallIPT; ++r)
      if (valid[r]) {
        sk[pos[r]] = key[r];
        sv[pos[r]] = val[r];
      }
    __syncthreads();
    if (pass + 1 < passes) {
#pragma unroll
      for (int r = 0; r < kSmallIPT; ++r) {
        const int p = wid * 32 * kSmallIPT + r * 32 + lane;
        if (p < n_total) {
          key[r] = sk[p];
          val[r] = sv[p];
        }
      }
      __syncthreads();
    }
  }
  // Segment heads over the sorted keys; thread t owns positions [t*IPT, (t+1)*IPT).
  int heads = 0;
  const int p0 = threadIdx.x * kSmallIPT;
#pragma unroll
  for (int r = 0; r < kSmallIPT; ++r) {
    const int p = p0 + r;
    if (p < n_total) {
      const uint32_t kk = sk[p];
      if (kk != sentinel && (p == 0 || sk[p - 1] != kk)) ++heads;
    }
  }
  int total = 0;
  int seg = block_excl_scan<kSmallNT>(heads, scan_sm, &total);
#pragma unroll
  for (int r = 0; r < kSmallIPT; ++r) {
    const int p = p0 + r;
    if (p < n_total) {
      const uint32_t kk = sk[p];
      sorted_slots[p] = sv[p];
      sorted_keys[p] = kk;
      if (kk != sentinel && (p == 0 || sk[p - 1] != kk)) {
        seg_start[seg] = p;
        unique_rows[seg] = static_cast<int32_t>(kk);
        ++seg;
      }
      // end marker: first dropped slot, or the end of the list
      if (kk == sentinel && (p == 0 || sk[p - 1] != sentinel)) seg_start[total] = p;
      if (p == n_total - 1 && kk != sentinel) seg_start[total] = n_total;
    }
  }
  if (threadIdx.x == 0) {
    *n_unique = total;
    *work_count = 0;
    if (n_total == 0) seg_start[0] = 0;
  }
}

// ------------------------------------------------------------------------------------
// Small regime, small table (n_total <= 16384 slots AND table_rows + 1 <= 48128 bins: every table of the
// Amazon-shaped TEM step): counting sort with one shared-memory bin per destination row instead of radix passes.
//   bins   shared-memory histogram of the keys (integer atomics: order-free)
//   scan   exclusive scan of the bins, packed with the running count of non-empty bins -> segment table
//   place  every slot takes a position inside its row's run (atomic cursor: arbitrary order within the run)
//   rank   the order inside a run is made canonical again: a slot's final position is the number of slots of
//          its run with a smaller slot number, so the sorted list is exactly the stable sort's -- the
//          reduction order, and with it every bit of the gradient, is independent of the atomics' timing
// Same outputs as small_sort_segments_kernel.  Dropped slots (sentinel key) land behind the valid ones.
// ------------------------------------------------------------------------------------
constexpr int kCsMaxPer = 33;      // bins per thread (odd: conflict-free strided scan); 33 * 1024 = 33792 bins
constexpr int kCsLongMin = 33;     // runs at least this long are ordered by the bitmap path
constexpr int kCsMaxLong = kSmallCap / kCsLongMin + 1;
constexpr int kCsBitmaps = 16;     // warps 0..15 each own a 16384-bit bitmap + 512 prefix counts

__global__ void __launch_bounds__(kSmallNT, 1)
count_sort_segments_kernel(const __grid_constant__ ContribTable T, int n_total, int64_t table_rows, int64_t drop_idx, int per,
                           uint32_t* __restrict__ sorted_slots, uint32_t* __restrict__ sorted_keys,
                           int32_t* __restrict__ seg_start, int32_t* __restrict__ unique_rows,
                           int32_t* __restrict__ n_unique, int32_t* __restrict__ work_count) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int nbins = per * kSmallNT;
  uint32_t* bins = reinterpret_cast<uint32_t*>(smem_raw);                        // [nbins]
  uint32_t* bitmap = bins + nbins;                                               // [kCsBitmaps][512]
  uint32_t* long_key = bitmap + kCsBitmaps * 512;                                // [kCsMaxLong]
  unsigned short* sv = reinterpret_cast<unsigned short*>(long_key + kCsMaxLong + 3);   // [kSmallCap]
  unsigned short* pref = sv + kSmallCap;                                         // [kCsBitmaps][512]
  int* scan_sm = reinterpret_cast<int*>(pref + kCsBitmaps * 512);                // [32]
  int* n_long = scan_sm + 32;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint32_t sentinel = static_cast<uint32_t>(table_rows);
  {
    uint4* b4 = reinterpret_cast<uint4*>(bins);
    for (int i = threadIdx.x; i < nbins / 4; i += kSmallNT) b4[i] = make_uint4(0u, 0u, 0u, 0u);
    if (threadIdx.x == 0) *n_long = 0;
  }
  __syncthreads();
  uint32_t key[kSmallIPT];
#pragma unroll
  for (int r = 0; r < kSmallIPT; ++r) {
    const int p = r * kSmallNT + threadIdx.x;
    key[r] = 0xffffffffu;
    if (p < n_total) key[r] = make_key(T, static_cast<uint32_t>(p), table_rows, drop_idx);
  }
#pragma unroll
  for (int r = 0; r < kSmallIPT; ++r)
    if (key[r] != 0xffffffffu) atomicAdd(&bins[key[r]], 1u);
  __syncthreads();
  // packed exclusive scan: low 16 bits = slots before the bin, high 16 bits = non-empty bins before it
  const int b0 = threadIdx.x * per;
  uint32_t mine = 0;
  for (int j = 0; j < per; ++j) {
    const uint32_t c = bins[b0 + j];
    mine += c + ((c != 0u && static_cast<uint32_t>(b0 + j) != sentinel) ? 0x10000u : 0u);
  }
  int total = 0;
  uint32_t run = static_cast<uint32_t>(block_excl_scan<kSmallNT>(static_cast<int>(mine), scan_sm, &total));
  for (int j = 0; j < per; ++j) {
    const uint32_t b = static_cast<uint32_t>(b0 + j);
    const uint32_t c = bins[b];
    bins[b] = run;
    if (b == sentinel) seg_start[static_cast<uint32_t>(total) >> 16] = static_cast<int32_t>(run & 0xffffu);  // end marker
    if (c != 0u && b != sentinel) {
      seg_start[run >> 16] = static_cast<int32_t>(run & 0xffffu);
      unique_rows[run >> 16] = static_cast<int32_t>(b);
      if (c >= static_cast<uint32_t>(kCsLongMin)) long_key[atomicAdd(n_long, 1)] = b;
      run += 0x10000u;
    }
    run += c;
  }
  if (threadIdx.x == 0) {
    *n_unique = static_cast<int32_t>(static_cast<uint32_t>(total) >> 16);
    *work_count = 0;
  }
  __syncthreads();
  int pos[kSmallIPT];
#pragma unroll
  for (int r = 0; r < kSmallIPT; ++r) {
    pos[r] = -1;
    if (key[r] != 0xffffffffu) {
      pos[r] = static_cast<int>(atomicAdd(&bins[key[r]], 1u) & 0xffffu);
      sv[pos[r]] = static_cast<unsigned short>(r * kSmallNT + threadIdx.x);
    }
  }
  __syncthreads();
  // short runs (and the dropped slots): the owner of a slot counts the smaller slot numbers of its run
#pragma unroll
  for (int r = 0; r < kSmallIPT; ++r) {
    const int p = r * kSmallNT + threadIdx.x;
    if (p >= n_total) continue;
    const uint32_t k = key[r];
    int out = pos[r];
    if (k != sentinel) {
      const int end = static_cast<int>(bins[k] & 0xffffu);
      const int start = k == 0u ? 0 : static_cast<int>(bins[k - 1] & 0xffffu);
      if (end - start >= kCsLongMin) continue;
      int rank = 0;
      for (int q = start; q < end; ++q) rank += sv[q] < static_cast<unsigned short>(p) ? 1 : 0;
      out = start + rank;
    }
    sorted_slots[out] = static_cast<uint32_t>(p);
    sorted_keys[out] = k;
  }
  // long runs: one warp per run marks its slot numbers in a bitmap; rank = number of set bits below
  if (wid < kCsBitmaps) {
    uint32_t* bm = bitmap + wid * 512;
    unsigned short* pf = pref + wid * 512;
    const int nl = *n_long;
    for (int li = wid; li < nl; li += kCsBitmaps) {
      const uint32_t k = long_key[li];
      const int end = static_cast<int>(bins[k] & 0xffffu);
      const int start = k == 0u ? 0 : static_cast<int>(bins[k - 1] & 0xffffu);
      for (int w = lane; w < 512; w += 32) bm[w] = 0u;
      __syncwarp();
      for (int q = start + lane; q < end; q += 32) {
        const uint32_t v = sv[q];
        atomicOr(&bm[v >> 5], 1u << (v & 31u));
      }
      __syncwarp();
      int cnt = 0;
#pragma unroll
      for (int w = 0; w < 16; ++w) cnt += __popc(bm[lane * 16 + w]);
      int incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += t;
      }
      int runc = incl - cnt;
#pragma unroll
      for (int w = 0; w < 16; ++w) {
        pf[lane * 16 + w] = static_cast<unsigned short>(runc);
        runc += __popc(bm[lane * 16 + w]);
      }
      __syncwarp();
      for (int q = start + lane; q < end; q += 32) {
        const uint32_t v = sv[q];
        const int rank = pf[v >> 5] + __popc(bm[v >> 5] & ((1u << (v & 31u)) - 1u));
        sorted_slots[start + rank] = v;
        sorted_keys[start + rank] = k;
      }
      __syncwarp();
    }
  }
}

// ------------------------------------------------------------------------------------
// Large regime: multi-CTA radix sort.
// ------------------------------------------------------------------------------------
constexpr int kNT = 256;
constexpr int kIPT = 16;
constexpr int kTile = kNT * kIPT;  // 4096 keys per CTA

// hist[digit * nblocks + block].  FIRST (pass 0): the keys are formed here from the contributions' int64
// destination rows and written out (the pack pass and the first histogram pass are one kernel; the slot payload
// of pass 0 is the position itself and is never stored).  Every warp counts into its own 256 bins
// (shared-memory atomics on one CTA-wide histogram serialise on popular digits).
template <bool FIRST>
__global__ void __launch_bounds__(kNT, 8)   // 8 CTAs/SM: the ~1000 tiles of a 4M-slot sort fit in one wave
radix_hist_kernel(const __grid_constant__ ContribTable T, int64_t table_rows, int64_t drop_idx,
                  uint32_t* __restrict__ keys, int64_t n, int shift, int nblocks, int* __restrict__ hist) {
  __shared__ int h[(kNT / 32) * 256];
  for (int t = threadIdx.x; t < (kNT / 32) * 256; t += kNT) h[t] = 0;
  __syncthreads();
  int* mine = h + (threadIdx.x >> 5) * 256;
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kTile;
  constexpr int G = 4;  // keys in flight per thread (kept small: 16 int64 row ids would cost 32 registers)
#pragma unroll
  for (int r0 = 0; r0 < kIPT; r0 += G) {
    uint32_t k[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const int64_t p = base + (r0 + g) * kNT + threadIdx.x;
      k[g] = 0xffffffffu;
      if (p < n) k[g] = FIRST ? make_key(T, static_cast<uint32_t>(p), table_rows, drop_idx) : keys[p];
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const int64_t p = base + (r0 + g) * kNT + threadIdx.x;
      if (p < n) {
        if (FIRST) keys[p] = k[g];
        atomicAdd(&mine[(k[g] >> shift) & 255u], 1);  // integer counts: order-free
      }
    }
  }
  __syncthreads();
  int tot = 0;
#pragma unroll
  for (int w2 = 0; w2 < kNT / 32; ++w2) tot += h[w2 * 256 + threadIdx.x];
  hist[threadIdx.x * nblocks + blockIdx.x] = tot;
}

// One CTA per digit: exclusive scan of its row of per-block counts; totals[digit].
__global__ void __launch_bounds__(256)
radix_scan_kernel(int* __restrict__ hist, int nblocks, int* __restrict__ totals) {
  __shared__ int sm[8];
  int* row = hist + static_cast<int64_t>(blockIdx.x) * nblocks;
  int carry = 0;
  for (int b0 = 0; b0 < nblocks; b0 += 256) {
    const int b = b0 + threadIdx.x;
    const int v = b < nblocks ? row[b] : 0;
    int tot = 0;
    const int ex = block_excl_scan<256>(v, sm, &tot);
    if (b < nblocks) row[b] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) totals[blockIdx.x] = carry;
}

template <bool FIRST>
__global__ void __launch_bounds__(kNT, 3)
radix_scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, int64_t n,
                     int shift, int nblocks, const int* __restrict__ hist, const int* __restrict__ totals,
                     uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out) {
  __shared__ uint32_t sk[kTile];
  __shared__ uint32_t sv[kTile];
  __shared__ int whist[(kNT / 32) * 256];
  __shared__ int dstart[256];
  __shared__ int gbase[256];
  __shared__ int scan_sm[8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kTile;
  const int tile_valid = static_cast<int>(min(static_cast<int64_t>(kTile), n - base));
  // global base of each digit = exclusive scan of digit totals + this block's offset in the digit
  {
    const int ex = block_excl_scan<kNT>(totals[threadIdx.x], scan_sm, nullptr);
    gbase[threadIdx.x] = ex + hist[threadIdx.x * nblocks + blockIdx.x];
  }
  uint32_t key[kIPT], val[kIPT];
  bool valid[kIPT];
  int pos[kIPT];
#pragma unroll
  for (int r = 0; r < kIPT; ++r) {
    const int p = wid * 32 * kIPT + r * 32 + lane;
    valid[r] = p < tile_valid;
    key[r] = valid[r] ? keys_in[base + p] : 0xffffffffu;
    if (FIRST) val[r] = static_cast<uint32_t>(base + p);   // pass 0: the payload is the slot position
    else val[r] = valid[r] ? vals_in[base + p] : 0u;
  }
  tile_rank<kNT, kIPT, true>(key, valid, shift, pos, whist, dstart, scan_sm);
#pragma unroll
  for (int r = 0; r < kIPT; ++r)
    if (valid[r]) {
      sk[pos[r]] = key[r];
      sv[pos[r]] = val[r];
    }
  __syncthreads();
  for (int p = threadIdx.x; p < tile_valid; p += kNT) {
    const uint32_t kk = sk[p];
    const int dg = static_cast<int>((kk >> shift) & 255u);
    const int64_t o = static_cast<int64_t>(gbase[dg]) + (p - dstart[dg]);
    keys_out[o] = kk;
    vals_out[o] = sv[p];
  }
}

// Segment compaction (large regime).  Element n (virtual) is a sentinel.
__device__ __forceinline__ bool is_head(const uint32_t* keys, int64_t p, int64_t n, uint32_t sentinel) {
  if (p >= n) return false;
  const uint32_t kk = keys[p];
  return kk != sentinel && (p == 0 || keys[p - 1] != kk);
}

__global__ void __launch_bounds__(kNT)
heads_count_kernel(const uint32_t* __restrict__ keys, int64_t n, uint32_t sentinel, int* __restrict__ counts) {
  __shared__ int sm[8];
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kTile;
  int c = 0;
#pragma unroll
  for (int r = 0; r < kIPT; ++r) c += is_head(keys, base + r * kNT + threadIdx.x, n, sentinel) ? 1 : 0;  // coalesced
  int tot = 0;
  block_excl_scan<kNT>(c, sm, &tot);
  if (threadIdx.x == 0) counts[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(256)
heads_scan_kernel(int* __restrict__ counts, int nblocks, int32_t* __restrict__ n_unique,
                  int32_t* __restrict__ work_count) {
  __shared__ int sm[8];
  int carry = 0;
  for (int b0 = 0; b0 < nblocks; b0 += 256) {
    const int b = b0 + threadIdx.x;
    const int v = b < nblocks ? counts[b] : 0;
    int tot = 0;
    const int ex = block_excl_scan<256>(v, sm, &tot);
    if (b < nblocks) counts[b] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) {
    *n_unique = carry;
    *work_count = 0;
  }
}

// The tile's keys are staged in shared memory with coalesced loads (one pad word per 32 keys: the 16
// consecutive keys a thread then walks hit distinct banks), every thread numbers the segment heads among its 16
// keys, and the (start, row) pairs leave through shared memory again so the global stores are contiguous.
__global__ void __launch_bounds__(kNT)
heads_write_kernel(const uint32_t* __restrict__ keys, int64_t n, uint32_t sentinel,
                   const int* __restrict__ block_base, const int32_t* __restrict__ n_unique,
                   int32_t* __restrict__ seg_start, int32_t* __restrict__ unique_rows) {
  __shared__ uint32_t sk[kTile + kTile / 32 + 1];
  __shared__ int32_t out_pos[kTile];
  __shared__ int sm[8];
  __shared__ uint32_t s_prev;
  uint32_t* out_key = sk;  // reused once every thread holds its keys in registers (after the block scan)
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kTile;
#pragma unroll
  for (int r = 0; r < kIPT; ++r) {
    const int q = r * kNT + threadIdx.x;
    const int64_t p = base + q;
    sk[q + (q >> 5)] = p < n ? keys[p] : sentinel;
  }
  if (threadIdx.x == 0) s_prev = base > 0 ? keys[base - 1] : sentinel;
  __syncthreads();
  const int q0 = threadIdx.x * kIPT;
  uint32_t kk[kIPT];
  unsigned heads = 0;
  uint32_t prev = q0 == 0 ? s_prev : sk[(q0 - 1) + ((q0 - 1) >> 5)];
  const int total = *n_unique;
#pragma unroll
  for (int r = 0; r < kIPT; ++r) {
    const int q = q0 + r;
    const int64_t p = base + q;
    kk[r] = sk[q + (q >> 5)];
    if (p < n) {
      const bool first = p == 0;
      if (kk[r] != sentinel && (first || prev != kk[r])) heads |= 1u << r;
      if (kk[r] == sentinel && (first || prev != sentinel)) seg_start[total] = static_cast<int32_t>(p);
      if (p == n - 1 && kk[r] != sentinel) seg_start[total] = static_cast<int32_t>(n);
    }
    prev = kk[r];
  }
  int tot = 0;
  int o = block_excl_scan<kNT>(__popc(heads), sm, &tot);
#pragma unroll
  for (int r = 0; r < kIPT; ++r)
    if ((heads >> r) & 1u) {
      out_pos[o] = static_cast<int32_t>(base + q0 + r);
      out_key[o] = kk[r];
      ++o;
    }
  __syncthreads();
  const int64_t seg0 = block_base[blockIdx.x];
  for (int e = threadIdx.x; e < tot; e += kNT) {
    seg_start[seg0 + e] = out_pos[e];
    unique_rows[seg0 + e] = static_cast<int32_t>(out_key[e]);
  }
}

// ------------------------------------------------------------------------------------
// Segmented reduction.  The sorted slot list is cut into fixed units of 2^ch_shift positions; one
// warp reduces one unit, walking the destination-row segments inside it in order.  A segment that
// lies inside one unit is written directly; a segment spanning several units (a popular row:
// Zipf head, the 4-row segment table) leaves one partial per unit, and the fix-up kernel adds the
// partials in unit order.  Terms are therefore always added in ascending (contribution, slot)
// order with a bracketing that depends only on (n_total, data): bit-reproducible, no atomics.
// ------------------------------------------------------------------------------------
// Largest segment index whose start is <= pos, by a warp-wide 32-ary search: every step the 32 lanes probe 32
// evenly spaced entries of seg_start (one L2 round trip narrows the range 32x; 3 trips for a TEM step's ~10k
// segments, 5 for millions, instead of 14 / 22 dependent loads of a binary search).  seg_start[0] == 0.
__device__ __forceinline__ int warp_find_segment(const int32_t* __restrict__ seg_start, int nu, int pos, int lane) {
  int lo = 0, hi = nu;
  while (hi - lo > 1) {
    const int step = (hi - lo + 31) >> 5;
    const int probe = lo + (lane + 1) * step;
    const bool le = probe < hi && seg_start[probe] <= pos;
    const int c = __popc(__ballot_sync(kFull, le));
    lo += c * step;
    hi = min(hi, lo + step);
  }
  return lo;
}

// FULL: d4 == 32 * C (no column predicate: d = 128 with C = 1 is the reference's embedding size).
// Per 32 sorted slots the lanes fetch the slot metadata in parallel and park (source pointer, scale, key) in
// this warp's shared-memory slice; the row loop then reads them back as broadcasts, so the only warp
// collectives are the two ballots per 32 slots and every branch of the row loop is warp-uniform.
template <int C, bool FULL>
__global__ void __launch_bounds__(256)
seg_reduce_kernel(const __grid_constant__ ContribTable T, const uint32_t* __restrict__ sorted_slots,
                  const uint32_t* __restrict__ sorted_keys, const int32_t* __restrict__ seg_start,
                  const int32_t* __restrict__ n_unique, int d4, int ch_shift, float4* __restrict__ reduced,
                  float* __restrict__ reduced_bias, float4* __restrict__ dense, float* __restrict__ dense_bias,
                  float4* __restrict__ partial, float* __restrict__ partial_bias, int32_t* __restrict__ work,
                  int32_t* __restrict__ work_count) {
  __shared__ unsigned long long s_ptr[8][32];
  __shared__ float s_sc[8][32];
  __shared__ uint32_t s_key[8][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  const int warp = blockIdx.x * (blockDim.x >> 5) + wid;
  const int nu = *n_unique;
  if (nu == 0) return;
  const int n_valid = seg_start[nu];
  const int ch = 1 << ch_shift;
  const int n_units = (n_valid + ch - 1) >> ch_shift;
  constexpr int U = 8;  // source rows in flight per warp
  for (int unit = warp; unit < n_units; unit += nwarps) {
    const int u_lo = unit << ch_shift;
    const int u_hi = min(u_lo + ch, n_valid);
    int seg = warp_find_segment(seg_start, nu, u_lo, lane);
    bool started_here = seg_start[seg] == u_lo;
    float4 acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = zero4();
    float bacc = 0.f;
    bool open = false;
    for (int p = u_lo; p < u_hi; p += 32) {
      // lane-parallel metadata of the next (up to) 32 sorted slots
      const int q = p + lane;
      const bool in = q < u_hi;
      uint32_t key = 0xffffffffu;
      unsigned long long src = 0;
      float sc = 0.f;
      bool tb = false;
      if (in) {
        const uint32_t slot = sorted_slots[q];
        key = sorted_keys[q];
        const int ci = locate(T, slot);
        const psb_contrib_t& cc = T.c[ci];
        const uint32_t i = slot - T.off[ci];
        const int64_t row = cc.src_row != nullptr ? cc.src_row[i]
                                                  : static_cast<int64_t>(i / static_cast<uint32_t>(cc.src_div));
        sc = cc.scale != nullptr ? cc.scale[i] : 1.f;
        if (cc.scale2 != nullptr) sc *= cc.scale2[i / static_cast<uint32_t>(cc.scale2_div)];
        tb = cc.to_bias != 0;
        src = reinterpret_cast<unsigned long long>(reinterpret_cast<const float4*>(cc.src) + row * d4);
      }
      // a slot closes its segment when the next sorted key differs (or the valid range ends)
      uint32_t key_next = __shfl_down_sync(kFull, key, 1);
      if (lane == 31 || q + 1 >= u_hi) key_next = (q + 1 < n_valid) ? sorted_keys[min(q + 1, n_valid - 1)] : 0xfffffffeu;
      const unsigned last_mask = __ballot_sync(kFull, in && key_next != key);
      const unsigned bias_mask = __ballot_sync(kFull, tb);
      __syncwarp();  // the previous group's broadcasts have been read
      s_ptr[wid][lane] = src;
      s_sc[wid][lane] = sc;
      s_key[wid][lane] = key;
      __syncwarp();
      const int cnt = min(32, u_hi - p);
      for (int u0 = 0; u0 < cnt; u0 += U) {
        float4 v[U][C];
        float su[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int j = u0 + u;  // < 32
          const float4* ptr = reinterpret_cast<const float4*>(s_ptr[wid][j]);
          su[u] = s_sc[wid][j];
          const bool ok = j < cnt;
#pragma unroll
          for (int c = 0; c < C; ++c) {
            const int col = lane + 32 * c;
            v[u][c] = (ok && (FULL || col < d4)) ? ldg_row4(ptr + col) : zero4();
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int j = u0 + u;
          if (j < cnt) {
#pragma unroll
            for (int c = 0; c < C; ++c) fma4(acc[c], su[u], v[u][c]);
            if ((bias_mask >> j) & 1u) bacc += su[u];
            if ((last_mask >> j) & 1u) {
              // segment `seg` ends at sorted position p + j
              if (started_here) {
                const int64_t drow = s_key[wid][j];
#pragma unroll
                for (int c = 0; c < C; ++c) {
                  const int col = lane + 32 * c;
                  if (FULL || col < d4) {
                    if (reduced != nullptr) reduced[static_cast<int64_t>(seg) * d4 + col] = acc[c];
                    if (dense != nullptr) dense[drow * d4 + col] = acc[c];
                  }
                }
                if (lane == 0) {
                  if (reduced_bias != nullptr) reduced_bias[seg] = bacc;
                  if (dense_bias != nullptr) dense_bias[drow] = bacc;
                }
              } else {  // a run that began in an earlier unit: partial, combined by the fix-up kernel
                const int64_t ps = static_cast<int64_t>(unit) * 2;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                  const int col = lane + 32 * c;
                  if (FULL || col < d4) partial[ps * d4 + col] = acc[c];
                }
                if (lane == 0) partial_bias[ps] = bacc;
              }
#pragma unroll
              for (int c = 0; c < C; ++c) acc[c] = zero4();
              bacc = 0.f;
              ++seg;
              started_here = true;
            }
          }
        }
      }
      open = ((last_mask >> (cnt - 1)) & 1u) == 0u;
    }
    if (open) {  // the last run continues into the next unit
      const int64_t ps = static_cast<int64_t>(unit) * 2 + (started_here ? 1 : 0);
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const int col = lane + 32 * c;
        if (FULL || col < d4) partial[ps * d4 + col] = acc[c];
      }
      if (lane == 0) {
        partial_bias[ps] = bacc;
        // head unit of a segment that spans several units: one work item for the fix-up kernel
        // (integer atomic: the ORDER of the list is arbitrary, every item's sum is not)
        if (started_here) work[atomicAdd(work_count, 1)] = seg;
      }
    }
  }
}

// Fix-up of the segments that span several units (listed by seg_reduce_kernel): the per-unit partials are added
// in a fixed bracketing that is a pure function of the segment's unit range --
//   * U consecutive units (a "batch", U partial rows in flight) are added as a binary tree, batches in unit order;
//   * a segment of at most kFixLong units is folded by one warp;
//   * a longer one (a Zipf-head row: ~1000 units) by a whole CTA: the unit range is cut into 8 contiguous chunks,
//     one per warp, and the 8 chunk sums are added in chunk order -- the serial chain of the hottest row is 8x
//     shorter (it was the critical path of the whole kernel: 150 us).
// (The first version walked ALL segments, one per warp iteration with two dependent loads each: 184 us for 3.5M
// single-unit segments that needed no work.)
constexpr int kFixLong = 64;

template <int C, int U>
__device__ __forceinline__ void fix_range(const float4* __restrict__ partial, const float* __restrict__ partial_bias,
                                          int d4, int lane, int u_first, int u_lo, int u_hi, float4 (&acc)[C],
                                          float& bacc) {
  for (int u0 = u_lo; u0 <= u_hi; u0 += U) {
    float4 v[U][C];
    float pb[U];
#pragma unroll
    for (int t = 0; t < U; ++t) {
      const int u = min(u0 + t, u_hi);
      // the run of unit u_first starts there (slot 1); later units hold a continuing run (slot 0)
      const int64_t ps = static_cast<int64_t>(u) * 2 + (u == u_first ? 1 : 0);
      pb[t] = partial_bias[ps];
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const int col = lane + 32 * c;
        v[t][c] = col < d4 ? ldg_row4(partial + ps * d4 + col) : zero4();
      }
    }
#pragma unroll
    for (int t = 0; t < U; ++t) {
      if (u0 + t > u_hi) {  // past the end: contributes +0
        pb[t] = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) v[t][c] = zero4();
      }
    }
#pragma unroll
    for (int w2 = 1; w2 < U; w2 <<= 1) {
#pragma unroll
      for (int t = 0; t + w2 < U; t += 2 * w2) {
        pb[t] += pb[t + w2];
#pragma unroll
        for (int c = 0; c < C; ++c) {
          v[t][c].x += v[t + w2][c].x; v[t][c].y += v[t + w2][c].y;
          v[t][c].z += v[t + w2][c].z; v[t][c].w += v[t + w2][c].w;
        }
      }
    }
    bacc += pb[0];
#pragma unroll
    for (int c = 0; c < C; ++c) {
      acc[c].x += v[0][c].x; acc[c].y += v[0][c].y; acc[c].z += v[0][c].z; acc[c].w += v[0][c].w;
    }
  }
}

template <int C>
__global__ void __launch_bounds__(256)
seg_fixup_kernel(const int32_t* __restrict__ seg_start, const int32_t* __restrict__ unique_rows,
                 const int32_t* __restrict__ work, const int32_t* __restrict__ work_count, int d4, int ch_shift,
                 float4* __restrict__ reduced, float* __restrict__ reduced_bias, float4* __restrict__ dense,
                 float* __restrict__ dense_bias, const float4* __restrict__ partial,
                 const float* __restrict__ partial_bias) {
  __shared__ float4 s_acc[8][C * 32];
  __shared__ float s_b[8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  const int n_work = *work_count;
  constexpr int U = C == 1 ? 16 : 8;
  auto store = [&](int seg, const float4 (&acc)[C], float bacc) {
    const int64_t drow = unique_rows[seg];
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const int col = lane + 32 * c;
      if (col < d4) {
        if (reduced != nullptr) reduced[static_cast<int64_t>(seg) * d4 + col] = acc[c];
        if (dense != nullptr) dense[drow * d4 + col] = acc[c];
      }
    }
    if (lane == 0) {
      if (reduced_bias != nullptr) reduced_bias[seg] = bacc;
      if (dense_bias != nullptr) dense_bias[drow] = bacc;
    }
  };
  // (1) one warp per short work item
  for (int e = blockIdx.x * (blockDim.x >> 5) + wid; e < n_work; e += nwarps) {
    const int seg = work[e];
    const int s_lo = seg_start[seg], s_hi = seg_start[seg + 1];
    const int u_first = s_lo >> ch_shift, u_last = (s_hi - 1) >> ch_shift;
    if (u_last - u_first + 1 > kFixLong) continue;
    float4 acc[C];
    float bacc = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = zero4();
    fix_range<C, U>(partial, partial_bias, d4, lane, u_first, u_first, u_last, acc, bacc);
    store(seg, acc, bacc);
  }
  // (2) one CTA per long work item
  for (int e = blockIdx.x; e < n_work; e += gridDim.x) {
    const int seg = work[e];
    const int s_lo = seg_start[seg], s_hi = seg_start[seg + 1];
    const int u_first = s_lo >> ch_shift, u_last = (s_hi - 1) >> ch_shift;
    const int n_units = u_last - u_first + 1;
    if (n_units <= kFixLong) continue;      // CTA-uniform
    const int per = (n_units + 7) >> 3;
    const int lo = u_first + wid * per, hi = min(lo + per - 1, u_last);
    float4 acc[C];
    float bacc = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = zero4();
    if (lo <= hi) fix_range<C, U>(partial, partial_bias, d4, lane, u_first, lo, hi, acc, bacc);
    __syncthreads();                        // s_acc free (previous item's reads are done)
#pragma unroll
    for (int c = 0; c < C; ++c) s_acc[wid][c * 32 + lane] = acc[c];
    if (lane == 0) s_b[wid] = bacc;
    __syncthreads();
    if (wid == 0) {
#pragma unroll
      for (int w2 = 1; w2 < 8; ++w2) {
        bacc += s_b[w2];
#pragma unroll
        for (int c = 0; c < C; ++c) {
          const float4 o = s_acc[w2][c * 32 + lane];
          acc[c].x += o.x; acc[c].y += o.y; acc[c].z += o.z; acc[c].w += o.w;
        }
      }
      store(seg, acc, bacc);
    }
  }
}

__global__ void __launch_bounds__(256)
zero_rows_kernel(const int32_t* __restrict__ rows, const int32_t* __restrict__ n_rows, int d4,
                 float4* __restrict__ dense, float* __restrict__ dense_bias) {
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  const int n = *n_rows;
  for (int u = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); u < n; u += nwarps) {
    const int64_t r = rows[u];
    if (dense != nullptr)
      for (int col = lane; col < d4; col += 32) dense[r * d4 + col] = zero4();
    if (dense_bias != nullptr && lane == 0) dense_bias[r] = 0.f;
  }
}

static inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

struct WorkspaceLayout {
  int64_t keys_a, vals_a, keys_b, vals_b, hist, totals, counts, seg_start, partial, partial_bias, work, work_count, total;
};

// unit size of the segmented reduction: a pure function of n_total (~4k+ units, 8..256 slots each)
static int unit_shift_for(int64_t n_total) {
  int sh = 3;
  while (sh < 8 && (n_total >> sh) > 8192) ++sh;
  return sh;
}

static WorkspaceLayout layout_for(int64_t n_total, int64_t d = 512) {
  WorkspaceLayout L;
  const int64_t nblocks = (n_total + kTile - 1) / kTile + 1;
  int64_t o = 0;
  L.keys_a = o; o += align_up(4 * n_total, 256);
  L.vals_a = o; o += align_up(4 * n_total, 256);
  L.keys_b = o; o += align_up(4 * n_total, 256);
  L.vals_b = o; o += align_up(4 * n_total, 256);
  L.hist = o; o += align_up(4 * 256 * nblocks, 256);
  L.totals = o; o += 1024;
  L.counts = o; o += align_up(4 * (nblocks + 1), 256);
  L.seg_start = o; o += align_up(4 * (n_total + 2), 256);
  const int64_t n_units = (n_total >> unit_shift_for(n_total)) + 2;
  L.partial = o; o += align_up(2 * n_units * d * 4, 256);
  L.partial_bias = o; o += align_up(2 * n_units * 4, 256);
  L.work = o; o += align_up(n_units * 4, 256);
  L.work_count = o; o += 256;
  L.total = o + 256;
  return L;
}

}  // namespace psb

using namespace psb;

extern "C" int64_t psb_scatter_reduce_workspace_bytes(int64_t n_total, int64_t table_rows) {
  (void)table_rows;
  if (n_total < 0) return PSB_E_ARG;
  return layout_for(n_total > 0 ? n_total : 1).total;
}

// phase 0: sort + reduce (psb_scatter_reduce_rows); 1: sort only -- only idx / n of the contributions are read
// (psb_scatter_sort_rows); 2: reduce only, the workspace holds the result of a phase-1 call over the same idx / n /
// order (psb_scatter_reduce_sorted).  Which buffers hold the sorted slots is a pure function of (n_total, table_rows).
static int scatter_run(int phase, const psb_contrib_t* contribs, int32_t n_contribs, int64_t table_rows,
                       int64_t d, int64_t drop_idx, void* workspace, int64_t workspace_bytes,
                       int32_t* unique_rows, float* reduced, float* reduced_bias,
                       int32_t* n_unique, float* dense_grad, float* dense_bias_grad,
                       psb_stream_t stream) {
  if (contribs == nullptr || n_contribs <= 0 || n_contribs > PSB_MAX_CONTRIBS || workspace == nullptr ||
      unique_rows == nullptr || n_unique == nullptr || table_rows <= 0 || table_rows >= (1ll << 31))
    return PSB_E_ARG;
  if (d <= 0 || (d & 3) != 0 || d > 512) return PSB_E_DIM;
  if (misaligned16(reduced) || misaligned16(dense_grad) || misaligned16(workspace)) return PSB_E_ALIGN;
  ContribTable T;
  T.n = n_contribs;
  int64_t n_total = 0;
  for (int c = 0; c < n_contribs; ++c) {
    const psb_contrib_t& cc = contribs[c];
    if (cc.n < 0 || (cc.n > 0 && (cc.idx == nullptr || (phase != 1 && cc.src == nullptr)))) return PSB_E_ARG;
    if (phase != 1) {
      if (cc.src_row == nullptr && cc.src_div < 1) return PSB_E_ARG;
      if (cc.scale2 != nullptr && cc.scale2_div < 1) return PSB_E_ARG;
      if (misaligned16(cc.src)) return PSB_E_ALIGN;
    }
    T.c[c] = cc;
    T.off[c] = static_cast<uint32_t>(n_total);
    n_total += cc.n;
  }
  if (n_total >= (1ll << 31)) return PSB_E_ARG;
  for (int c = n_contribs; c <= PSB_MAX_CONTRIBS; ++c) T.off[c] = static_cast<uint32_t>(n_total);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const WorkspaceLayout L = layout_for(n_total > 0 ? n_total : 1);
  if (workspace_bytes < L.total) return PSB_E_WORKSPACE;
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  uint32_t* keys_a = reinterpret_cast<uint32_t*>(ws + L.keys_a);
  uint32_t* vals_a = reinterpret_cast<uint32_t*>(ws + L.vals_a);
  uint32_t* keys_b = reinterpret_cast<uint32_t*>(ws + L.keys_b);
  uint32_t* vals_b = reinterpret_cast<uint32_t*>(ws + L.vals_b);
  int* hist = reinterpret_cast<int*>(ws + L.hist);
  int* totals = reinterpret_cast<int*>(ws + L.totals);
  int* counts = reinterpret_cast<int*>(ws + L.counts);
  int32_t* seg_start = reinterpret_cast<int32_t*>(ws + L.seg_start);
  int32_t* work = reinterpret_cast<int32_t*>(ws + L.work);
  int32_t* work_count = reinterpret_cast<int32_t*>(ws + L.work_count);

  int bits = 1;
  while ((static_cast<int64_t>(1) << bits) <= table_rows) ++bits;  // sentinel == table_rows must fit
  const int passes = (bits + 7) / 8;
  const uint32_t* sorted_slots = nullptr;
  const uint32_t* sorted_keys = nullptr;
  int st;

  const int64_t cs_per = ((table_rows + 1 + kSmallNT - 1) / kSmallNT) | 1;   // odd number of bins per thread
  if (phase == 2) {                         // already sorted: where the sort phase left its result
    if (n_total <= kSmallCap || (passes & 1) == 0) {
      sorted_slots = vals_a;
      sorted_keys = keys_a;
    } else {
      sorted_slots = vals_b;
      sorted_keys = keys_b;
    }
  } else if (n_total <= kSmallCap && cs_per <= kCsMaxPer) {
    static DeviceAttr attr_smem;
    const size_t smem = static_cast<size_t>(cs_per) * kSmallNT * 4 + kCsBitmaps * 512 * 4 + (kCsMaxLong + 3) * 4 +
                        static_cast<size_t>(kSmallCap) * 2 + kCsBitmaps * 512 * 2 + 33 * 4;
    if (attr_smem.need(smem)) {
      cudaError_t e = cudaFuncSetAttribute(count_sort_segments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           static_cast<int>(smem));
      if (e != cudaSuccess) return static_cast<int>(e);
      attr_smem.done(smem);
    }
    PSB_PROF("count_sort_segments_kernel", s);
    count_sort_segments_kernel<<<1, kSmallNT, smem, s>>>(T, static_cast<int>(n_total), table_rows, drop_idx,
                                                         static_cast<int>(cs_per), vals_a, keys_a, seg_start,
                                                         unique_rows, n_unique, work_count);
    if ((st = launch_status()) != PSB_OK) return st;
    sorted_slots = vals_a;
    sorted_keys = keys_a;
  } else if (n_total <= kSmallCap) {
    static DeviceAttr attr_set;
    const size_t smem = static_cast<size_t>(kSmallCap) * 8 + (kSmallNT / 32) * 256 * 4 + 256 * 4 + 32 * 4;
    if (attr_set.need()) {
      cudaError_t e = cudaFuncSetAttribute(small_sort_segments_kernel,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
      if (e != cudaSuccess) return static_cast<int>(e);
      attr_set.done();
    }
    PSB_PROF("small_sort_segments_kernel", s);
    small_sort_segments_kernel<<<1, kSmallNT, smem, s>>>(T, static_cast<int>(n_total), table_rows, drop_idx,
                                                         passes, vals_a, keys_a, seg_start, unique_rows, n_unique, work_count);
    if ((st = launch_status()) != PSB_OK) return st;
    sorted_slots = vals_a;
    sorted_keys = keys_a;
  } else {
    const int nblocks = static_cast<int>((n_total + kTile - 1) / kTile);
    uint32_t *ki = keys_a, *vi = vals_a, *ko = keys_b, *vo = vals_b;
    for (int pass = 0; pass < passes; ++pass) {
      PSB_PROF("radix_hist_kernel", s);
      if (pass == 0) radix_hist_kernel<true><<<nblocks, kNT, 0, s>>>(T, table_rows, drop_idx, ki, n_total, 0, nblocks, hist);
      else radix_hist_kernel<false><<<nblocks, kNT, 0, s>>>(T, table_rows, drop_idx, ki, n_total, pass * 8, nblocks, hist);
      if ((st = launch_status()) != PSB_OK) return st;
      PSB_PROF("radix_scan_kernel", s);
      radix_scan_kernel<<<256, 256, 0, s>>>(hist, nblocks, totals);
      if ((st = launch_status()) != PSB_OK) return st;
      PSB_PROF("radix_scatter_kernel", s);
      if (pass == 0) radix_scatter_kernel<true><<<nblocks, kNT, 0, s>>>(ki, vi, n_total, 0, nblocks, hist, totals, ko, vo);
      else radix_scatter_kernel<false><<<nblocks, kNT, 0, s>>>(ki, vi, n_total, pass * 8, nblocks, hist, totals, ko, vo);
      if ((st = launch_status()) != PSB_OK) return st;
      uint32_t* t = ki; ki = ko; ko = t;
      t = vi; vi = vo; vo = t;
    }
    const uint32_t sentinel = static_cast<uint32_t>(table_rows);
    PSB_PROF("heads_count_kernel", s);
    heads_count_kernel<<<nblocks, kNT, 0, s>>>(ki, n_total, sentinel, counts);
    if ((st = launch_status()) != PSB_OK) return st;
    PSB_PROF("heads_scan_kernel", s);
    heads_scan_kernel<<<1, 256, 0, s>>>(counts, nblocks, n_unique, work_count);
    if ((st = launch_status()) != PSB_OK) return st;
    PSB_PROF("heads_write_kernel", s);
    heads_write_kernel<<<nblocks, kNT, 0, s>>>(ki, n_total, sentinel, counts, n_unique, seg_start, unique_rows);
    if ((st = launch_status()) != PSB_OK) return st;
    sorted_slots = vi;
    sorted_keys = ki;
  }

  if (phase != 1 && (reduced != nullptr || reduced_bias != nullptr || dense_grad != nullptr || dense_bias_grad != nullptr)) {
    const int ch_shift = unit_shift_for(n_total);
    const int grid = grid_for((n_total >> ch_shift) + 1, 8, 16);
    const int grid_fix = grid_for((n_total >> ch_shift) + 1, 8, 8);
    const int d4 = static_cast<int>(d / 4);
    float4* partial = reinterpret_cast<float4*>(ws + L.partial);
    float* partial_bias = reinterpret_cast<float*>(ws + L.partial_bias);
#define PSB_SR_LAUNCH(C)                                                                                      \
  PSB_PROF("seg_reduce_kernel", s);                                                                            \
  {                                                                                                            \
    auto kern = d4 == 32 * C ? seg_reduce_kernel<C, true> : seg_reduce_kernel<C, false>;                       \
    kern<<<grid, 256, 0, s>>>(T, sorted_slots, sorted_keys, seg_start, n_unique, d4, ch_shift,                 \
                              reinterpret_cast<float4*>(reduced), reduced_bias,                                \
                              reinterpret_cast<float4*>(dense_grad), dense_bias_grad, partial, partial_bias,   \
                              work, work_count);                                                               \
  }                                                                                                            \
  if ((st = launch_status()) != PSB_OK) return st;                                                            \
  PSB_PROF("seg_fixup_kernel", s);                                                                            \
  seg_fixup_kernel<C><<<grid_fix, 256, 0, s>>>(seg_start, unique_rows, work, work_count, d4, ch_shift,         \
                                               reinterpret_cast<float4*>(reduced), reduced_bias,              \
                                               reinterpret_cast<float4*>(dense_grad), dense_bias_grad,        \
                                               partial, partial_bias)
    if (d4 <= 32) { PSB_SR_LAUNCH(1); }
    else if (d4 <= 64) { PSB_SR_LAUNCH(2); }
    else { PSB_SR_LAUNCH(4); }
#undef PSB_SR_LAUNCH
    if ((st = launch_status()) != PSB_OK) return st;
  }
  return PSB_OK;
}

extern "C" int psb_scatter_reduce_rows(const psb_contrib_t* contribs, int32_t n_contribs, int64_t table_rows,
                                       int64_t d, int64_t drop_idx, void* workspace, int64_t workspace_bytes,
                                       int32_t* unique_rows, float* reduced, float* reduced_bias,
                                       int32_t* n_unique, float* dense_grad, float* dense_bias_grad,
                                       psb_stream_t stream) {
  return scatter_run(0, contribs, n_contribs, table_rows, d, drop_idx, workspace, workspace_bytes, unique_rows, reduced,
                     reduced_bias, n_unique, dense_grad, dense_bias_grad, stream);
}

extern "C" int psb_scatter_sort_rows(const psb_contrib_t* contribs, int32_t n_contribs, int64_t table_rows,
                                     int64_t drop_idx, void* workspace, int64_t workspace_bytes, int32_t* unique_rows,
                                     int32_t* n_unique, psb_stream_t stream) {
  return scatter_run(1, contribs, n_contribs, table_rows, 4, drop_idx, workspace, workspace_bytes, unique_rows, nullptr,
                     nullptr, n_unique, nullptr, nullptr, stream);
}

extern "C" int psb_scatter_reduce_sorted(const psb_contrib_t* contribs, int32_t n_contribs, int64_t table_rows,
                                         int64_t d, int64_t drop_idx, void* workspace, int64_t workspace_bytes,
                                         const int32_t* unique_rows, float* reduced, float* reduced_bias,
                                         const int32_t* n_unique, float* dense_grad, float* dense_bias_grad,
                                         psb_stream_t stream) {
  return scatter_run(2, contribs, n_contribs, table_rows, d, drop_idx, workspace, workspace_bytes,
                     const_cast<int32_t*>(unique_rows), reduced, reduced_bias, const_cast<int32_t*>(n_unique), dense_grad,
                     dense_bias_grad, stream);
}

extern "C" int psb_zero_rows(const int32_t* rows, const int32_t* n_rows, int64_t max_rows, int64_t d,
                             float* dense, float* dense_bias, psb_stream_t stream) {
  if (rows == nullptr || n_rows == nullptr || max_rows < 0) return PSB_E_ARG;
  if (d <= 0 || (d & 3) != 0 || d > 512) return PSB_E_DIM;
  if (misaligned16(dense)) return PSB_E_ALIGN;
  if (max_rows == 0) return PSB_OK;
  PSB_PROF("zero_rows_kernel", static_cast<cudaStream_t>(stream));
  zero_rows_kernel<<<grid_for(max_rows, 8, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      rows, n_rows, static_cast<int>(d / 4), reinterpret_cast<float4*>(dense), dense_bias);
  return launch_status();
}
