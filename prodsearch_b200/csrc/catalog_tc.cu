// G5 (tensor-core mode): full-catalog scoring as a tcgen05 / TMEM TF32 GEMM fed by TMA, with the
// top-k selection fused into the epilogue so the [M, N] score matrix is never written.
//
// TF32 products cannot give reference-exact scores (SURVEY.md 7.3.3), so the tensor cores only
// SHORTLIST: with |approx - exact| <= eps_q = 2^-8 |q| max|e| (Cauchy-Schwarz on the per-product
// truncation error, 2x headroom), every item of the exact top-k has approx >= tau - 2 eps_q for ANY
// valid lower bound tau of the k-th best approx score.  Pipeline (all on `stream`, no host sync):
//   1. pilot   : tc_score_kernel<DUMP> over a strided sample of 128-item tiles -> scores [M, S]
//   2. kth     : per query, k-th largest pilot score (radix select) -> thr = kth - 2 eps
//   3. main    : tc_score_kernel<FILTER> over the whole table; the epilogue (one thread per query
//                row reading its TMEM lane) appends (score, id) >= thr to a per-(row, CTA) list
//   4. final   : per query, k-th best of the candidates, prune by 2 eps, EXACT fp32 rescoring with
//                the canonical recurrence of catalog_topk.cu, rank-sort (score desc, id asc)
//   5. fallback: rows whose lists overflowed (degenerate ties) are redone by an exact streaming
//                scan -- always correct, only slow for pathological data.
// tc_score_kernel: grid (item slices, query tiles of 128), 192 threads = TMA producer warp, MMA
// issuer warp (one elected thread issues tcgen05.mma.kind::tf32, M=128 N=128 K=8), 4 epilogue
// warps (tcgen05.ld 32x32b.x32).  smem: Q tile resident (d/32 k-blocks of 128x32 fp32, 128B
// swizzle), 2-stage ring of item tiles, TMEM: 2 accumulators x 128 columns (double buffered).
#include <cuda.h>
#include <cuda_fp16.h>

#include "catalog_common.cuh"
#include "tc_ptx.cuh"

namespace psb {

constexpr int kTM = 128;          // queries per CTA (UMMA M, TMEM lanes)
constexpr int kTN = 128;          // items per tile (UMMA N, TMEM columns per accumulator)
constexpr int kKB = 32;           // fp32 per k-block = one 128-byte swizzle row
constexpr int kStages = 2;
constexpr int kParts = 4;          // epilogue column quarters (16 epilogue warps, 4 per SM sub-partition)
constexpr int kTcThreads = 64 + 4 * 32 * kParts;
constexpr uint32_t kKBBytes = kTM * kKB * 4;  // 16 KB per k-block of either operand
constexpr float kEpsFactor = 1.0f / 256.0f;

// cute::UMMA::InstrDescriptor: c_format F32 (1) [4,6), a/b format TF32 (2) [7,10)/[10,13), K-major A and B,
// n_dim = N>>3 [17,23), m_dim = M>>4 [24,29).
constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(kTN >> 3) << 17) |
                            (static_cast<uint32_t>(kTM >> 4) << 24);

struct TcParams {
  int m, n_items, kblocks;          // kblocks = d / 32
  int tile_begin, tile_step, n_tiles;  // tiles enumerated p = 0..n_tiles-1 -> item tile tile_begin + p*tile_step
  const float* bias;
  const float* thr;                 // [m] filter thresholds (FILTER)
  float* dump;                      // [m_pad, ld_dump] (DUMP)
  int ld_dump;
  float* cand_s;                    // [m_pad * n_slices * cap]
  int32_t* cand_i;
  int32_t* cand_n;                  // [m_pad * n_slices]
  int cap;
};

template <bool DUMP>
__global__ void __launch_bounds__(kTcThreads, 1)
tc_score_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_e,
                const TcParams P) {
  extern __shared__ unsigned char smem_dyn[];
  // 128-byte-swizzled operand tiles need a 1024-byte aligned base
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tile_bytes = static_cast<uint32_t>(P.kblocks) * kKBBytes;
  unsigned char* sA = smem;
  unsigned char* sB = smem + tile_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + tile_bytes * (1 + kStages));
  uint64_t* a_full = bars;
  uint64_t* b_full = bars + 1;
  uint64_t* b_empty = bars + 1 + kStages;
  uint64_t* t_full = bars + 1 + 2 * kStages;
  uint64_t* t_empty = bars + 3 + 2 * kStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5 + 2 * kStages);

  const int n_slices = gridDim.x, slice = blockIdx.x, mtile = blockIdx.y;
  const int per = (P.n_tiles + n_slices - 1) / n_slices;
  const int p_lo = slice * per;
  const int p_hi = min(P.n_tiles, p_lo + per);
  const int my_tiles = max(0, p_hi - p_lo);

  if (threadIdx.x == 0) {
    mbar_init(a_full, 1);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(b_full + s, 1);
      mbar_init(b_empty + s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(t_full + a, 1);
      mbar_init(t_empty + a, 4 * kParts);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // TMEM: 2 accumulators x 128 fp32 columns
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(2 * kTN));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      mbar_expect_tx(a_full, tile_bytes);
      for (int kb = 0; kb < P.kblocks; ++kb) tma_load_2d(sA + kb * kKBBytes, &map_q, kb * kKB, mtile * kTM, a_full);
      for (int it = 0; it < my_tiles; ++it) {
        const int st = it % kStages;
        const uint32_t ph = (it / kStages) & 1;
        mbar_wait(b_empty + st, ph ^ 1);
        mbar_expect_tx(b_full + st, tile_bytes);
        const int tile = P.tile_begin + (p_lo + it) * P.tile_step;
        for (int kb = 0; kb < P.kblocks; ++kb)
          tma_load_2d(sB + st * tile_bytes + kb * kKBBytes, &map_e, kb * kKB, tile * kTN, b_full + st);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      mbar_wait(a_full, 0);
      for (int it = 0; it < my_tiles; ++it) {
        const int st = it % kStages;
        const uint32_t ph = (it / kStages) & 1;
        const int acc = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        mbar_wait(t_empty + acc, aph ^ 1);
        mbar_wait(b_full + st, ph);
        tc_fence_after();
        const uint32_t d_addr = tmem_base + static_cast<uint32_t>(acc * kTN);
        const uint64_t a_base = umma_desc(smem_u32(sA));
        const uint64_t b_base = umma_desc(smem_u32(sB + st * tile_bytes));
#pragma unroll 4
        for (int kb = 0; kb < P.kblocks; ++kb) {
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4)  // 4 x (K = 8 tf32 = 32 bytes) inside one 128-byte swizzle row
            tc_mma_tf32(d_addr, a_base + static_cast<uint64_t>(kb) * (kKBBytes >> 4) + k4 * 2,
                        b_base + static_cast<uint64_t>(kb) * (kKBBytes >> 4) + k4 * 2, kIdesc, (kb | k4) != 0 ? 1u : 0u);
        }
        tc_commit(b_empty + st);   // smem stage free once these MMAs have read it
        tc_commit(t_full + acc);   // accumulator ready for the epilogue
      }
    }
  } else {
    // ===== epilogue: 8 warps; thread = (query row = TMEM lane, half of the tile's 128 columns) =====
    // A warp may only touch TMEM lanes 32*(warp%4)..+31; warps 2..9 cover each lane quarter twice,
    // the second copy taking columns 64..127.  Every thread keeps its own candidate list.
    const int quarter = warp & 3;
    const int part = (warp - 2) >> 2;
    const int row = mtile * kTM + quarter * 32 + lane;
    const bool row_ok = row < P.m;
    float thr = INFINITY;
    if (!DUMP && row_ok) thr = P.thr[row];
    int cnt = 0;
    const int n_lists = n_slices * kParts;
    const int64_t list = (static_cast<int64_t>(row) * n_lists + slice * kParts + part) * P.cap;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    for (int it = 0; it < my_tiles; ++it) {
      const int acc = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      const int p = p_lo + it;
      const int tile = P.tile_begin + p * P.tile_step;
      const bool full_tile = (tile + 1) * kTN <= P.n_items && P.bias == nullptr;
      mbar_wait(t_full + acc, aph);
      tc_fence_after();
#pragma unroll 1
      for (int c0 = part * (kTN / kParts); c0 < (part + 1) * (kTN / kParts); c0 += 32) {
        uint32_t v[32];
        __syncwarp();
        tc_ld32(lane_addr + static_cast<uint32_t>(acc * kTN + c0), v);
        const int id0 = tile * kTN + c0;
        if (DUMP) {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int id = id0 + i;
            float s = __uint_as_float(v[i]);
            if (P.bias != nullptr && id < P.n_items) s += P.bias[id];
            if (row_ok) P.dump[static_cast<int64_t>(row) * P.ld_dump + p * kTN + c0 + i] = id < P.n_items ? s : -INFINITY;
          }
        } else if (full_tile) {
          // branch once per 8 scores: almost every group is below the threshold
#pragma unroll
          for (int g8 = 0; g8 < 32; g8 += 8) {
            float mx = fmaxf(fmaxf(__uint_as_float(v[g8]), __uint_as_float(v[g8 + 1])),
                             fmaxf(__uint_as_float(v[g8 + 2]), __uint_as_float(v[g8 + 3])));
            mx = fmaxf(mx, fmaxf(fmaxf(__uint_as_float(v[g8 + 4]), __uint_as_float(v[g8 + 5])),
                                 fmaxf(__uint_as_float(v[g8 + 6]), __uint_as_float(v[g8 + 7]))));
            if (mx >= thr) {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float s = __uint_as_float(v[g8 + i]);
                if (s >= thr) {
                  if (cnt < P.cap) {
                    P.cand_s[list + cnt] = s;
                    P.cand_i[list + cnt] = id0 + g8 + i;
                  }
                  ++cnt;
                }
              }
            }
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int id = id0 + i;
            float s = __uint_as_float(v[i]);
            if (P.bias != nullptr && id < P.n_items) s += P.bias[id];
            if (s >= thr && id < P.n_items) {
              if (cnt < P.cap) {
                P.cand_s[list + cnt] = s;
                P.cand_i[list + cnt] = id;
              }
              ++cnt;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(t_empty + acc);
    }
    if (!DUMP && row_ok) P.cand_n[static_cast<int64_t>(row) * n_lists + slice * kParts + part] = cnt;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(2 * kTN));
  }
}

// ------------------------------------------------------------------ fp16 shortlist (PSB_TOPK_TC16)
// Same pipeline with the shortlist GEMM in fp16 (tcgen05 kind::f16, fp32 accumulation in TMEM) on a half-precision
// COPY of the (static) evaluation table: half the HBM bytes per pass, twice the tensor rate, and -- because a
// 128 x 128 fp16 query tile is 32 KB instead of 64 KB -- one CTA keeps up to FOUR query tiles resident and scores
// all of them against every item tile it streams: M <= 512 queries per pass over the table, 148 independent
// streams with a 5..8-stage TMA ring (the tf32 kernel re-streams the table once per 128 queries from L2 with a
// 2-stage ring and is latency-bound there).  The error bound is measured, not assumed: the conversion pass
// records max_r |e_r - half(e_r)| and max_r |e_r|, the query pass |q - half(q)| and |half(q)|, so
//   |q.e - half(q).half(e)| <= |q - hq| max|e| + |hq| max|e - he| + 2^-14 |hq| max|e|   (last term: fp32 accumulation)
// and the final stage rescored exactly in fp32 as before -> results identical to the exact mode.
constexpr int kKB16 = 64;                       // halves per k-block = one 128-byte swizzle row
constexpr uint32_t kQBlock16 = kTM * 128;       // bytes of one 128-row k-block (16 KB)

// Issue from a warp whose 32 lanes all execute the instruction stream (uniform control flow), with the instruction
// itself predicated on the elected lane: the descriptors stay in uniform registers and ptxas has no reason to wrap
// every tcgen05.mma in the per-lane "waterfall" loop it emits when the issue sits inside `if (lane == 0)`.
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t leader;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(leader));
  return leader;
}
__device__ __forceinline__ void tc_mma_f16_if(uint32_t leader, uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\tsetp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tc_commit_if(uint32_t leader, uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)),
      "r"(leader)
      : "memory");
}

struct Tc16Params {
  int m, n_items, kblocks;             // kblocks = d / 64
  int tile_begin, tile_step, n_tiles;  // item tiles of TN items
  int stages;
  int append;                          // FILTER: continue the candidate lists an earlier segment started
  const float* bias;
  const float* thr;
  float* dump;
  int ld_dump;
  float* cand_s;
  int32_t* cand_i;
  int32_t* cand_n;
  int cap;
};

// ------------------------------------------------------------------ fp16 shortlist kernel
// MT query tiles per CTA; item tile TN = 128 (MT <= 2) or 64 (MT = 3, 4): two accumulator sets of MT * TN TMEM
// columns.  grid (item slices, query groups of MT tiles), 64 + 512 threads as tc_score_kernel.  Against the tf32
// kernel's layout:
//  (1) the accumulator set is handed over per QUERY TILE (one mbarrier per (set, tile), committed right after the
//      tile's 8 MMAs): the epilogue of tile 0 runs while the MMAs of tiles 1.. are still in flight;
//  (2) every epilogue warp owns a FIXED run of 32-column chunks of ONE query tile, so threshold, count and list
//      base are scalars for the whole kernel (dealing chunks round-robin over the parts re-selects the per-tile
//      state for every chunk: ~35 of ~80 instructions per chunk in the SASS of the round-1 kernel);
//  (3) a row therefore has AP candidate lists per item slice (the parts that own chunks of its tile), not kParts;
//  (4) the MMA issuer is the whole warp 1 with elected-lane predication (see tc_mma_f16_if): 11-19 % faster end to
//      end than a lane-0 issuer (profiles/r01_summary.md).
template <int MT>
struct Tc16V2 {
  static constexpr int TN = MT <= 2 ? 128 : 64;
  static constexpr int kChunksPerTile = TN / 32;
  static constexpr int kChunks = MT * kChunksPerTile;                 // 32-column chunks per accumulator set
  static constexpr int CPP = (kChunks + kParts - 1) / kParts;         // chunks per part: a contiguous run
  static constexpr int kActiveParts = (kChunks + CPP - 1) / CPP;      // parts that own chunks (MT = 3: 3 of 4)
  static constexpr int AP = kChunksPerTile / CPP;                     // parts (= candidate lists) per query tile
  static_assert(kChunksPerTile % CPP == 0, "a part's run of chunks must stay inside one query tile");
};

template <bool DUMP, int MT>
__global__ void __launch_bounds__(kTcThreads, 1)
tc16_score_v2_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_e,
                     const Tc16Params P) {
  using V = Tc16V2<MT>;
  constexpr int TN = V::TN;
  constexpr int kAccCols = MT * TN;
  constexpr int kTmemCols = 2 * kAccCols <= 256 ? 256 : 512;
  constexpr uint32_t kIdesc16 = (1u << 4) | (static_cast<uint32_t>(TN >> 3) << 17) | (static_cast<uint32_t>(kTM >> 4) << 24);
  constexpr int kMaxStages = 8;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t q_bytes = static_cast<uint32_t>(MT * P.kblocks) * kQBlock16;
  const uint32_t e_block = static_cast<uint32_t>(TN) * 128u;
  const uint32_t stage_bytes = static_cast<uint32_t>(P.kblocks) * e_block;
  const int S = P.stages;
  unsigned char* sA = smem;
  unsigned char* sB = smem + q_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + static_cast<size_t>(S) * stage_bytes);
  uint64_t* a_full = bars;
  uint64_t* b_full = bars + 1;
  uint64_t* b_empty = bars + 1 + kMaxStages;
  uint64_t* t_full = bars + 1 + 2 * kMaxStages;          // [2 sets][MT tiles] (8 slots reserved)
  uint64_t* t_empty = bars + 9 + 2 * kMaxStages;         // [2 sets]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 11 + 2 * kMaxStages);

  const int n_slices = gridDim.x, slice = blockIdx.x, mtile0 = blockIdx.y * MT;
  const int per = (P.n_tiles + n_slices - 1) / n_slices;
  const int p_lo = slice * per;
  const int p_hi = min(P.n_tiles, p_lo + per);
  const int my_tiles = max(0, p_hi - p_lo);

  if (threadIdx.x == 0) {
    mbar_init(a_full, 1);
    for (int st = 0; st < S; ++st) {
      mbar_init(b_full + st, 1);
      mbar_init(b_empty + st, 1);
    }
    for (int a = 0; a < 2; ++a) {
      for (int mt = 0; mt < MT; ++mt) mbar_init(t_full + a * MT + mt, 1);
      mbar_init(t_empty + a, 4 * V::kActiveParts);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      mbar_expect_tx(a_full, q_bytes);
      for (int mt = 0; mt < MT; ++mt)
        for (int kb = 0; kb < P.kblocks; ++kb)
          tma_load_2d(sA + (mt * P.kblocks + kb) * kQBlock16, &map_q, kb * kKB16, (mtile0 + mt) * kTM, a_full);
      for (int it = 0; it < my_tiles; ++it) {
        const int st = it % S;
        const uint32_t ph = (it / S) & 1;
        mbar_wait(b_empty + st, ph ^ 1);
        mbar_expect_tx(b_full + st, stage_bytes);
        const int tile = P.tile_begin + (p_lo + it) * P.tile_step;
        for (int kb = 0; kb < P.kblocks; ++kb)
          tma_load_2d(sB + static_cast<size_t>(st) * stage_bytes + kb * e_block, &map_e, kb * kKB16, tile * TN, b_full + st);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: all 32 lanes run the loop, the instructions are predicated on the elected lane; one commit
    //       per query tile =====
    {
      const uint32_t leader = elect_one();
      mbar_wait(a_full, 0);
      // descriptors are the base descriptor plus an address offset (>> 4, low 14 bits), never rebuilt per MMA
      const uint64_t a_base = umma_desc(smem_u32(sA));
      const uint64_t b_base = umma_desc(smem_u32(sB));
      const uint32_t kb_a = kQBlock16 >> 4, kb_b = e_block >> 4, st_b = stage_bytes >> 4;
      for (int it = 0; it < my_tiles; ++it) {
        const int st = it % S;
        const uint32_t ph = (it / S) & 1;
        const int acc = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        mbar_wait(t_empty + acc, aph ^ 1);
        mbar_wait(b_full + st, ph);
        tc_fence_after();
        const uint64_t b_tile = b_base + static_cast<uint64_t>(st) * st_b;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          const uint32_t d_addr = tmem_base + static_cast<uint32_t>(acc * kAccCols + mt * TN);
          const uint64_t a_tile = a_base + static_cast<uint64_t>(mt * P.kblocks) * kb_a;
#pragma unroll 2
          for (int kb = 0; kb < P.kblocks; ++kb) {
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4)  // 4 x (K = 16 halves = 32 bytes) inside one 128-byte swizzle row
              tc_mma_f16_if(leader, d_addr, a_tile + static_cast<uint64_t>(kb) * kb_a + k4 * 2,
                            b_tile + static_cast<uint64_t>(kb) * kb_b + k4 * 2, kIdesc16, (kb | k4) != 0 ? 1u : 0u);
          }
          tc_commit_if(leader, t_full + acc * MT + mt);
        }
        tc_commit_if(leader, b_empty + st);
      }
    }
  } else if (((warp - 2) >> 2) < V::kActiveParts) {
    // ===== epilogue: thread = (TMEM lane = query row of ONE tile, fixed run of CPP chunks) =====
    const int quarter = warp & 3;
    const int part = (warp - 2) >> 2;
    const int chunk0 = part * V::CPP;
    const int mt = chunk0 / V::kChunksPerTile;
    const int col0 = (chunk0 % V::kChunksPerTile) * 32;     // first column inside the tile's accumulator
    const int row = (mtile0 + mt) * kTM + quarter * 32 + lane;
    const bool ok = row < P.m;
    const int n_lists = n_slices * V::AP;
    const int64_t lidx = static_cast<int64_t>(row) * n_lists + slice * V::AP + (part % V::AP);
    const int64_t li = lidx * P.cap;
    float th = INFINITY;
    int cn = 0;
    if (!DUMP && ok) {
      th = P.thr[row];
      if (P.append) cn = P.cand_n[lidx];
    }
    const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(mt * TN + col0);
    for (int it = 0; it < my_tiles; ++it) {
      const int acc = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      const int p = p_lo + it;
      const int tile = P.tile_begin + p * P.tile_step;
      const bool full_tile = (tile + 1) * TN <= P.n_items && P.bias == nullptr;
      mbar_wait(t_full + acc * MT + mt, aph);
      tc_fence_after();
#pragma unroll 1
      for (int j = 0; j < V::CPP; ++j) {
        const int c0 = col0 + j * 32;
        uint32_t v[32];
        __syncwarp();
        tc_ld32(t_addr + static_cast<uint32_t>(acc * kAccCols + j * 32), v);
        const int id0 = tile * TN + c0;
        if (DUMP) {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int id = id0 + i;
            float sc = __uint_as_float(v[i]);
            if (P.bias != nullptr && id < P.n_items) sc += P.bias[id];
            if (ok) P.dump[static_cast<int64_t>(row) * P.ld_dump + p * TN + c0 + i] = id < P.n_items ? sc : -INFINITY;
          }
        } else if (full_tile) {
          float mx8[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const int g8 = g * 8;
            const float m0 = fmaxf(fmaxf(__uint_as_float(v[g8]), __uint_as_float(v[g8 + 1])),
                                   fmaxf(__uint_as_float(v[g8 + 2]), __uint_as_float(v[g8 + 3])));
            mx8[g] = fmaxf(m0, fmaxf(fmaxf(__uint_as_float(v[g8 + 4]), __uint_as_float(v[g8 + 5])),
                                     fmaxf(__uint_as_float(v[g8 + 6]), __uint_as_float(v[g8 + 7]))));
          }
          if (!(fmaxf(fmaxf(mx8[0], mx8[1]), fmaxf(mx8[2], mx8[3])) < th)) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const int g8 = g * 8;
              if (!(mx8[g] < th)) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const float sc = __uint_as_float(v[g8 + i]);
                  if (!(sc < th)) {
                    if (cn < P.cap) {
                      P.cand_s[li + cn] = sc;
                      P.cand_i[li + cn] = id0 + g8 + i;
                    }
                    ++cn;
                  }
                }
              }
            }
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int id = id0 + i;
            float sc = __uint_as_float(v[i]);
            if (P.bias != nullptr && id < P.n_items) sc += P.bias[id];
            if (!(sc < th) && id < P.n_items) {
              if (cn < P.cap) {
                P.cand_s[li + cn] = sc;
                P.cand_i[li + cn] = id;
              }
              ++cn;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(t_empty + acc);
    }
    if (!DUMP && ok) P.cand_n[lidx] = cn;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols));
  }
}

// fp32 table -> fp16 copy (round to nearest) + stats[0] = max |e|^2, stats[1] = max |e - half(e)|^2,
// stats[2] = 1.0 if any element overflows fp16.  One warp per row; maxima via integer atomicMax (order-free).
__global__ void __launch_bounds__(256)
prep_f16_kernel(const float4* __restrict__ table, int64_t rows, int d4, uint2* __restrict__ half_out,
                float* __restrict__ stats) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * 8;
  float best = 0.f, best_err = 0.f;
  bool over = false;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5); r < rows; r += nwarps) {
    float sq = 0.f, er = 0.f;
    for (int c = lane; c < d4; c += 32) {
      const float4 v = ldg_row4(table + r * d4 + c);
      const __half2 h01 = __floats2half2_rn(v.x, v.y), h23 = __floats2half2_rn(v.z, v.w);
      const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
      over |= isinf(f01.x) || isinf(f01.y) || isinf(f23.x) || isinf(f23.y) || !(v.x == v.x) || !(v.y == v.y) ||
              !(v.z == v.z) || !(v.w == v.w);
      sq += dot4(v, v);
      const float4 e = make_float4(v.x - f01.x, v.y - f01.y, v.z - f23.x, v.w - f23.y);
      er += dot4(e, e);
      uint2 o;
      o.x = *reinterpret_cast<const uint32_t*>(&h01);
      o.y = *reinterpret_cast<const uint32_t*>(&h23);
      half_out[r * d4 + c] = o;
    }
    sq = warp_sum(sq);
    er = warp_sum(er);
    best = fmaxf(best, sq);
    best_err = fmaxf(best_err, er);
  }
  over = __any_sync(kFull, over);
  if (lane == 0) {
    atomicMax(reinterpret_cast<int*>(stats), __float_as_int(best));
    atomicMax(reinterpret_cast<int*>(stats + 1), __float_as_int(best_err));
    if (over) atomicMax(reinterpret_cast<int*>(stats + 2), __float_as_int(1.f));
  }
}

// queries -> fp16 rows (rows >= m zero) + eps[row] (see the error bound above).  One warp per row.
__global__ void __launch_bounds__(256)
q16_kernel(const float* __restrict__ Q, int m, int m_pad, int d, const float* __restrict__ stats,
           __half* __restrict__ q16, float* __restrict__ eps) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= m_pad) return;
  float qn = 0.f, dq = 0.f;
  for (int c = lane; c < d; c += 32) {
    float v = 0.f;
    if (row < m) v = Q[static_cast<int64_t>(row) * d + c];
    const __half h = __float2half_rn(v);
    const float f = __half2float(h);
    q16[static_cast<int64_t>(row) * d + c] = h;
    qn += f * f;
    dq += (v - f) * (v - f);
  }
  qn = warp_sum(qn);
  dq = warp_sum(dq);
  if (lane == 0) {
    const float E = sqrtf(stats[0]), dE = sqrtf(stats[1]);
    const float hq = sqrtf(qn);
    // 1.01: rounding of the norms themselves; 2^-14 |hq| max|e|: fp32 accumulation inside the tensor core
    float e = 1.01f * (sqrtf(dq) * E + hq * dE) + 6.1035156e-5f * hq * E + 1e-30f;
    if (stats[2] != 0.f || !(e < 3.0e38f)) e = INFINITY;   // table does not fit fp16: no pruning, rows fall back
    eps[row] = row < m ? e : 0.f;
  }
}

// ------------------------------------------------------------------ helpers
__global__ void __launch_bounds__(256)
max_row_norm_kernel(const float4* __restrict__ table, int64_t rows, int d4, float* __restrict__ out_sq) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * 8;
  float best = 0.f;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5); r < rows; r += nwarps) {
    float s = 0.f;
    for (int c = lane; c < d4; c += 32) {
      const float4 v = ldg_row4(table + r * d4 + c);
      s += dot4(v, v);
    }
    s = warp_sum(s);
    best = fmaxf(best, s);
  }
  // max over non-negative floats == max over their bit patterns; order-free, so deterministic
  if (lane == 0) atomicMax(reinterpret_cast<int*>(out_sq), __float_as_int(best));
}

__device__ __forceinline__ uint32_t order_key(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);   // ascending key order == ascending float order
}

// k-th largest of vals[0..n) by 4-pass MSB radix select; all 256 threads must call.  n >= k required.
__device__ float block_kth_largest(const float* vals, int n, int k, int* hist /*[256] smem*/, uint32_t* sh /*[2] smem*/) {
  uint32_t prefix = 0, mask = 0;
  int need = k;
  for (int shift = 24; shift >= 0; shift -= 8) {
    hist[threadIdx.x] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += 256) {
      const uint32_t key = order_key(vals[i]);
      if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1);
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      // bins are walked from 255 down until `need` entries are covered; lane l owns the 8 bins 255-8l .. 248-8l
      const int lane = threadIdx.x;
      int c[8], mine = 0;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        c[u] = hist[255 - (lane * 8 + u)];
        mine += c[u];
      }
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += t;
      }
      const int before = incl - mine;
      const unsigned hit = __ballot_sync(kFull, before < need && incl >= need);
      const int total = __shfl_sync(kFull, incl, 31);
      if (hit == 0u) {          // fewer than `need` entries above bin 0: the scalar walk stops at bin 0
        if (lane == 31) {
          sh[0] = 0u;
          sh[1] = static_cast<uint32_t>(need - (total - c[7]));
        }
      } else if (lane == __ffs(hit) - 1) {
        int run = before, u = 0;
        for (; u < 7; ++u) {
          if (run + c[u] >= need) break;
          run += c[u];
        }
        int b = 255 - (lane * 8 + u);
        if (b == 0) {           // bin 0 is never "selected by break": same arithmetic as the scalar walk
          run = total - c[7];
        }
        sh[0] = static_cast<uint32_t>(b);
        sh[1] = static_cast<uint32_t>(need - run);
      }
    }
    __syncthreads();
    prefix |= sh[0] << shift;
    mask |= 255u << shift;
    need = static_cast<int>(sh[1]);
    __syncthreads();
  }
  const uint32_t key = prefix;
  const uint32_t bits = (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
  return __uint_as_float(bits);
}

// pilot scores -> thr[row] = kth - 2 eps_row ; eps_row = 2^-8 |q_row| max|e|
__global__ void __launch_bounds__(256)
pilot_threshold_kernel(const float* __restrict__ dump, int ld, int n_pilot, int k, const float* __restrict__ Q, int d,
                       const float* __restrict__ max_sq, const float* __restrict__ eps_in, float* __restrict__ thr,
                       float* __restrict__ eps, int stage) {
  __shared__ int hist[256];
  __shared__ uint32_t sh[2];
  __shared__ float red[8];
  const int row = blockIdx.x;
  float s = 0.f;
  for (int c = threadIdx.x; c < d; c += 256) {
    const float v = Q[static_cast<int64_t>(row) * d + c];
    s += v * v;
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  float qsq = 0.f;
  for (int w = 0; w < 8; ++w) qsq += red[w];
  const float e = eps_in != nullptr ? eps_in[row] : kEpsFactor * sqrtf(qsq) * sqrtf(*max_sq) + 1e-30f;
  const float* vals = dump + static_cast<int64_t>(row) * ld;
  // count finite entries: with fewer than k valid pilot items nothing can be pruned
  int valid = 0;
  if (stage) {   // the pilot scores fit in shared memory: read them once, select there
    extern __shared__ __align__(16) unsigned char thr_raw[];
    float* sv = reinterpret_cast<float*>(thr_raw);
    for (int i = threadIdx.x * 4; i < n_pilot; i += 1024) {
      const float4 v = *reinterpret_cast<const float4*>(vals + i);   // ld and n_pilot are multiples of 128
      *reinterpret_cast<float4*>(sv + i) = v;
      valid += (v.x > -INFINITY ? 1 : 0) + (v.y > -INFINITY ? 1 : 0) + (v.z > -INFINITY ? 1 : 0) + (v.w > -INFINITY ? 1 : 0);
    }
    vals = sv;
  } else
  for (int i = threadIdx.x; i < n_pilot; i += 256) valid += vals[i] > -INFINITY ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) valid += __shfl_xor_sync(kFull, valid, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = static_cast<float>(valid);
  __syncthreads();
  float tot = 0.f;
  for (int w = 0; w < 8; ++w) tot += red[w];
  float t = -INFINITY;
  if (static_cast<int>(tot) >= k) t = block_kth_largest(vals, n_pilot, k, hist, sh) - 2.f * e;
  if (!(e < 3.0e38f)) t = -INFINITY;      // unbounded shortlist error: nothing may be pruned
  if (threadIdx.x == 0) {
    thr[row] = t;
    eps[row] = e;
  }
}

constexpr int kFinalCap = 14336;   // candidates a final-select CTA can hold in shared memory
constexpr int kKeepCap = 1024;
constexpr int kMaxLists = kNumSMs * 4;  // n_slices * kParts upper bound     // candidates that survive the 2-eps prune and get exact scores

// Candidates of one query row: n_lists per-(CTA, epilogue part) lists of at most `cap` entries -> cs / ci (ci optional)
// in shared memory.  *s_over is set when a list overflowed or the total exceeds kFinalCap (nothing is loaded then).
// All 256 threads must call; ends with a __syncthreads().
__device__ __forceinline__ void load_candidate_lists(int row, const float* __restrict__ cand_s,
                                                     const int32_t* __restrict__ cand_i,
                                                     const int32_t* __restrict__ cand_n, int n_lists, int cap,
                                                     float* cs, int32_t* ci, int* offs, int* hist, int* s_total,
                                                     int* s_over, int final_cap) {
  for (int l = threadIdx.x; l < n_lists; l += 256) offs[l + 1] = cand_n[static_cast<int64_t>(row) * n_lists + l];
  if (threadIdx.x == 0) offs[0] = 0;
  __syncthreads();
  // exclusive scan of the clamped list sizes (n_lists <= kMaxLists = 592: 3 per thread)
  {
    constexpr int kPer = (kMaxLists + 255) / 256;
    int c[kPer], mine = 0, over = 0;
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int l = threadIdx.x * kPer + u;
      c[u] = l < n_lists ? offs[l + 1] : 0;
      over |= c[u] > cap;
      c[u] = min(c[u], cap);
      mine += c[u];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(kFull, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) hist[wid] = incl;
    over = __any_sync(kFull, over) ? 1 : 0;
    if (lane == 0) hist[8 + wid] = over;
    __syncthreads();
    int base = 0, any_over = 0;
    for (int w = 0; w < 8; ++w) {
      if (w < wid) base += hist[w];
      any_over |= hist[8 + w];
    }
    int run = base + incl - mine;
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int l = threadIdx.x * kPer + u;
      if (l < n_lists) offs[l] = run;
      run += c[u];
    }
    if (threadIdx.x == 255) {
      offs[n_lists] = run;
      *s_total = run;
      *s_over = any_over | (run > final_cap);
    }
  }
  __syncthreads();
  if (*s_over) return;
  // flat gather: candidate i belongs to the list whose offset range holds i (binary search), so all loads of a
  // thread are independent (order irrelevant: the final ordering is a strict total order)
  const int tot = *s_total;
  for (int i = threadIdx.x; i < tot; i += 256) {
    int a = 0, b = n_lists;           // largest l with offs[l] <= i
    while (b - a > 1) {
      const int mid = (a + b) >> 1;
      if (offs[mid] <= i) a = mid; else b = mid;
    }
    const int64_t src = (static_cast<int64_t>(row) * n_lists + a) * cap + (i - offs[a]);
    cs[i] = cand_s[src];
    if (ci != nullptr) ci[i] = cand_i[src];
  }
  __syncthreads();
}

// Threshold refinement between segments of the main pass: with the candidates collected so far the k-th best
// approximate score is a (much) tighter lower bound than the pilot's, so thr[row] = max(thr[row], kth - 2 eps).
__global__ void __launch_bounds__(256)
refine_threshold_kernel(const float* __restrict__ cand_s, const int32_t* __restrict__ cand_n, int n_lists, int cap,
                        const float* __restrict__ eps, int k, float* __restrict__ thr, int final_cap) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  float* cs = reinterpret_cast<float*>(sm_raw);                 // [kFinalCap]
  __shared__ int hist[256];
  __shared__ uint32_t sh[2];
  __shared__ int s_total, s_over;
  __shared__ int offs[kMaxLists + 1];
  const int row = blockIdx.x;
  load_candidate_lists(row, cand_s, nullptr, cand_n, n_lists, cap, cs, nullptr, offs, hist, &s_total, &s_over, final_cap);
  if (s_over || s_total < k) return;      // keep the current threshold (an overflowed row ends in the fallback)
  const float e = eps[row];
  if (!(e < 3.0e38f)) return;
  const float t = block_kth_largest(cs, s_total, k, hist, sh) - 2.f * e;
  if (threadIdx.x == 0 && t > thr[row]) thr[row] = t;
}

// per query row: candidates -> prune -> exact rescoring -> ordered top-k.  Rows that cannot be
// finished here (overflowed lists / too many survivors) are flagged for the exact fallback.
__global__ void __launch_bounds__(256)
final_select_kernel(const float* __restrict__ cand_s, const int32_t* __restrict__ cand_i,
                    const int32_t* __restrict__ cand_n, int n_slices, int cap, const float* __restrict__ eps,
                    const float* __restrict__ Q, const float* __restrict__ E, int d, const float* __restrict__ bias,
                    int k, int64_t id_base, int64_t id_stride, int64_t* __restrict__ out_ids,
                    float* __restrict__ out_scores, int32_t* __restrict__ fallback_flag, int final_cap) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  float* cs = reinterpret_cast<float*>(sm_raw);                 // [final_cap]
  int32_t* ci = reinterpret_cast<int32_t*>(cs + final_cap);      // [final_cap]
  float* ks = reinterpret_cast<float*>(ci + final_cap);          // [kKeepCap] exact scores
  int32_t* ki = reinterpret_cast<int32_t*>(ks + kKeepCap);       // [kKeepCap]
  float* qrow = reinterpret_cast<float*>(ki + kKeepCap);         // [d]
  __shared__ int hist[256];
  __shared__ uint32_t sh[2];
  __shared__ int s_total, s_over, s_keep;
  __shared__ int offs[kMaxLists + 1];
  const int row = blockIdx.x;
  for (int c = threadIdx.x; c < d; c += 256) qrow[c] = Q[static_cast<int64_t>(row) * d + c];
  if (threadIdx.x == 0) s_keep = 0;
  load_candidate_lists(row, cand_s, cand_i, cand_n, n_slices, cap, cs, ci, offs, hist, &s_total, &s_over, final_cap);
  if (s_over) {
    if (threadIdx.x == 0) fallback_flag[row] = 1;
    return;
  }
  const int total = s_total;
  float cut = -INFINITY;
  if (total > k) cut = block_kth_largest(cs, total, k, hist, sh) - 2.f * eps[row];
  if (!(eps[row] < 3.0e38f)) cut = -INFINITY;
  for (int i = threadIdx.x; i < total; i += 256) {
    if (!(cs[i] < cut)) {
      const int slot = atomicAdd(&s_keep, 1);
      if (slot < kKeepCap) ki[slot] = ci[i];
    }
  }
  __syncthreads();
  const int keep = s_keep;
  if (keep > kKeepCap) {
    if (threadIdx.x == 0) fallback_flag[row] = 1;
    return;
  }
  // exact fp32 scores with the canonical recurrence (bit-identical to the exact mode)
  for (int i = threadIdx.x; i < keep; i += 256) {
    const int32_t id = ki[i];
    ks[i] = canonical_dot(qrow, E + static_cast<int64_t>(id) * d, d) + (bias != nullptr ? bias[id] : 0.f);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < keep; i += 256) {
    const float es = ks[i];
    const int32_t ei = ki[i];
    int rank = 0;
    for (int u = 0; u < keep; ++u) rank += beats(ks[u], ki[u], es, ei) ? 1 : 0;
    if (rank < k) {
      out_ids[static_cast<int64_t>(row) * k + rank] = id_base + static_cast<int64_t>(ei) * id_stride;
      out_scores[static_cast<int64_t>(row) * k + rank] = es;
    }
  }
  for (int r = keep + threadIdx.x; r < k; r += 256) {
    out_ids[static_cast<int64_t>(row) * k + r] = -1;
    out_scores[static_cast<int64_t>(row) * k + r] = -INFINITY;
  }
}

// exact streaming scan for flagged rows (degenerate inputs only).
__global__ void __launch_bounds__(256)
fallback_rows_kernel(const int32_t* __restrict__ flag, const float* __restrict__ Q, const float* __restrict__ E,
                     int64_t n_items, int d, const float* __restrict__ bias, int k, int64_t id_base,
                     int64_t id_stride, int64_t* __restrict__ out_ids, float* __restrict__ out_scores) {
  const int row = blockIdx.x;
  if (flag[row] == 0) return;
  extern __shared__ __align__(16) unsigned char sm_raw[];
  float* qrow = reinterpret_cast<float*>(sm_raw);   // [d]
  __shared__ float bs[kKMax], cs[256], ns[kKMax];
  __shared__ int32_t bi[kKMax], ci[256], ni[kKMax];
  __shared__ int wc[8];
  for (int c = threadIdx.x; c < d; c += 256) qrow[c] = Q[static_cast<int64_t>(row) * d + c];
  if (threadIdx.x < kKMax) {
    bs[threadIdx.x] = -INFINITY;
    bi[threadIdx.x] = 0x7fffffff;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int64_t base = 0; base < n_items; base += 256) {
    const int64_t j = base + threadIdx.x;
    float s = 0.f;
    int32_t id = 0;
    bool pass = false;
    if (j < n_items) {
      id = static_cast<int32_t>(j);
      s = canonical_dot(qrow, E + j * d, d) + (bias != nullptr ? bias[j] : 0.f);
      pass = beats(s, id, bs[k - 1], bi[k - 1]);
    }
    const unsigned bal = __ballot_sync(kFull, pass);
    if (lane == 0) wc[wid] = __popc(bal);
    __syncthreads();
    int nb = 0, total = 0;
    for (int w2 = 0; w2 < 8; ++w2) {
      if (w2 < wid) nb += wc[w2];
      total += wc[w2];
    }
    if (total > 0) {
      const int my = nb + __popc(bal & ((1u << lane) - 1u));
      if (pass) {
        cs[my] = s;
        ci[my] = id;
      }
      __syncthreads();
      // rank-merge best[kKMax] with cand[total <= 256] in two halves of the thread block
      for (int e = threadIdx.x; e < kKMax + total; e += 256) {
        const bool fb = e < kKMax;
        const float es = fb ? bs[e] : cs[e - kKMax];
        const int32_t ei = fb ? bi[e] : ci[e - kKMax];
        int rank = 0;
        for (int u = 0; u < kKMax; ++u) rank += (u != e && before(bs[u], bi[u], u, es, ei, e)) ? 1 : 0;
        for (int u = 0; u < total; ++u) rank += (kKMax + u != e && before(cs[u], ci[u], kKMax + u, es, ei, e)) ? 1 : 0;
        if (rank < kKMax) {
          ns[rank] = es;
          ni[rank] = ei;
        }
      }
      __syncthreads();
      if (threadIdx.x < kKMax) {
        bs[threadIdx.x] = ns[threadIdx.x];
        bi[threadIdx.x] = ni[threadIdx.x];
      }
    }
    __syncthreads();
  }
  for (int r = threadIdx.x; r < k; r += 256) {
    const bool empty = bi[r] == 0x7fffffff;
    out_ids[static_cast<int64_t>(row) * k + r] = empty ? -1 : id_base + static_cast<int64_t>(bi[r]) * id_stride;
    out_scores[static_cast<int64_t>(row) * k + r] = empty ? -INFINITY : bs[r];
  }
}

// ------------------------------------------------------------------ host side
// rows x d fp32 row-major -> boxes of 128 rows x 32 floats, 128-byte swizzle, OOB rows read as zero
static int make_map(CUtensorMap* map, const float* base, int64_t rows, int64_t d) {
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) return PSB_E_UNSUPPORTED;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(d), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(d) * 4};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(kKB), static_cast<cuuint32_t>(kTM)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? PSB_OK : PSB_E_ARG;
}

struct TcPlan {
  int m_tiles, m_pad, n_slices, total_tiles, pilot_tiles, pilot_step, cap;
  int64_t off_thr, off_eps, off_maxsq, off_flag, off_cand_n, off_dump, off_cand_s, off_cand_i, total;
};

static int64_t up256(int64_t x) { return (x + 255) / 256 * 256; }

static TcPlan plan_for(int64_t m, int64_t n_items, int64_t k) {
  TcPlan p;
  p.m_tiles = static_cast<int>((m + kTM - 1) / kTM);
  p.m_pad = p.m_tiles * kTM;
  p.total_tiles = static_cast<int>((n_items + kTN - 1) / kTN);
  p.n_slices = kNumSMs / p.m_tiles;
  if (p.n_slices < 1) p.n_slices = 1;
  if (p.n_slices > p.total_tiles) p.n_slices = p.total_tiles;
  p.pilot_tiles = p.total_tiles / 64 > 128 ? p.total_tiles / 64 : 128;
  if (p.pilot_tiles > p.total_tiles) p.pilot_tiles = p.total_tiles;
  p.pilot_step = p.total_tiles / p.pilot_tiles;
  const double expect = static_cast<double>(k) * p.total_tiles / p.pilot_tiles / (p.n_slices * kParts);
  p.cap = (static_cast<int>(2.0 * expect) + 96 + 31) / 32 * 32;
  int64_t o = 0;
  p.off_thr = o; o += up256(p.m_pad * 4);
  p.off_eps = o; o += up256(p.m_pad * 4);
  p.off_maxsq = o; o += 256;
  p.off_flag = o; o += up256(p.m_pad * 4);
  p.off_cand_n = o; o += up256(static_cast<int64_t>(p.m_pad) * p.n_slices * kParts * 4);
  p.off_dump = o; o += up256(static_cast<int64_t>(p.m_pad) * p.pilot_tiles * kTN * 4);
  p.off_cand_s = o; o += up256(static_cast<int64_t>(p.m_pad) * p.n_slices * kParts * p.cap * 4);
  p.off_cand_i = o; o += up256(static_cast<int64_t>(p.m_pad) * p.n_slices * kParts * p.cap * 4);
  p.total = o + 256;
  return p;
}

int64_t tc_workspace_bytes(int64_t m, int64_t n_items, int64_t d, int64_t k) {
  (void)d;
  return plan_for(m, n_items, k).total;
}

static bool tc_supported(int64_t m, int64_t n_items, int64_t d) {
  return d % kKB == 0 && d <= 128 && n_items >= 32768 && m <= kNumSMs * kTM;
}

int table_max_row_sqnorm(const float* table, int64_t rows, int64_t d, float* out, cudaStream_t s) {
  cudaMemsetAsync(out, 0, 4, s);
  PSB_PROF("max_row_norm_kernel", s);
  max_row_norm_kernel<<<kNumSMs * 8, 256, 0, s>>>(reinterpret_cast<const float4*>(table), rows,
                                                  static_cast<int>(d / 4), out);
  return launch_status();
}

int catalog_topk_tc(const float* queries, int64_t m, const float* table, int64_t n_items, int64_t d,
                    const float* bias, int64_t k, int64_t id_base, int64_t id_stride, const float* max_row_sqnorm,
                    void* workspace, int64_t workspace_bytes, int64_t* out_ids, float* out_scores, cudaStream_t s) {
  if (!tc_supported(m, n_items, d))   // shapes the tensor path does not cover run the exact kernels
    return catalog_topk_exact(queries, m, table, n_items, d, bias, k, id_base, id_stride, workspace,
                              workspace_bytes, out_ids, out_scores, s);
  const TcPlan pl = plan_for(m, n_items, k);
  const int64_t ex_bytes = (exact_workspace_bytes(m, n_items) + 255) / 256 * 256;
  if (workspace_bytes < ex_bytes + pl.total) return PSB_E_WORKSPACE;
  unsigned char* ws = static_cast<unsigned char*>(workspace) + ex_bytes;
  float* thr = reinterpret_cast<float*>(ws + pl.off_thr);
  float* eps = reinterpret_cast<float*>(ws + pl.off_eps);
  float* maxsq = reinterpret_cast<float*>(ws + pl.off_maxsq);
  int32_t* flag = reinterpret_cast<int32_t*>(ws + pl.off_flag);
  int32_t* cand_n = reinterpret_cast<int32_t*>(ws + pl.off_cand_n);
  float* dump = reinterpret_cast<float*>(ws + pl.off_dump);
  float* cand_s = reinterpret_cast<float*>(ws + pl.off_cand_s);
  int32_t* cand_i = reinterpret_cast<int32_t*>(ws + pl.off_cand_i);

  alignas(64) CUtensorMap map_q, map_e;
  int st;
  if ((st = make_map(&map_q, queries, m, d)) != PSB_OK) return st;
  if ((st = make_map(&map_e, table, n_items, d)) != PSB_OK) return st;

  const int kblocks = static_cast<int>(d / kKB);
  const size_t smem = static_cast<size_t>(kblocks) * kKBBytes * (1 + kStages) + 256 + 1024;
  static DeviceAttr attr_done;
  if (attr_done.need()) {
    cudaError_t e1 = cudaFuncSetAttribute(tc_score_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaError_t e2 = cudaFuncSetAttribute(tc_score_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaError_t e3 = cudaFuncSetAttribute(final_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    if (e3 == cudaSuccess)
      e3 = cudaFuncSetAttribute(pilot_threshold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) return static_cast<int>(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3));
    attr_done.done();
  }
  cudaMemsetAsync(flag, 0, static_cast<size_t>(pl.m_pad) * 4, s);
  if (max_row_sqnorm == nullptr) {   // one extra pass over the table; callers with a static table cache it
    if ((st = table_max_row_sqnorm(table, n_items, d, maxsq, s)) != PSB_OK) return st;
    max_row_sqnorm = maxsq;
  }

  TcParams P;
  P.m = static_cast<int>(m);
  P.n_items = static_cast<int>(n_items);
  P.kblocks = kblocks;
  P.bias = bias;
  P.thr = thr;
  P.dump = dump;
  P.ld_dump = pl.pilot_tiles * kTN;
  P.cand_s = cand_s;
  P.cand_i = cand_i;
  P.cand_n = cand_n;
  P.cap = pl.cap;
  // 1. pilot
  P.tile_begin = 0;
  P.tile_step = pl.pilot_step;
  P.n_tiles = pl.pilot_tiles;
  {
    int slices = pl.n_slices < pl.pilot_tiles ? pl.n_slices : pl.pilot_tiles;
    dim3 grid(slices, pl.m_tiles);
    PSB_PROF("tc_score_kernel", s);
    tc_score_kernel<true><<<grid, kTcThreads, smem, s>>>(map_q, map_e, P);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  // 2. thresholds
  PSB_PROF("pilot_threshold_kernel", s);
  const bool stage_pilot = static_cast<size_t>(P.ld_dump) * 4 <= 160 * 1024;
  pilot_threshold_kernel<<<static_cast<int>(m), 256, stage_pilot ? static_cast<size_t>(P.ld_dump) * 4 : 0, s>>>(
      dump, P.ld_dump, P.ld_dump, static_cast<int>(k), queries, static_cast<int>(d), max_row_sqnorm, nullptr, thr, eps,
      stage_pilot ? 1 : 0);
  if ((st = launch_status()) != PSB_OK) return st;
  // 3. main pass
  P.tile_step = 1;
  P.n_tiles = pl.total_tiles;
  {
    dim3 grid(pl.n_slices, pl.m_tiles);
    PSB_PROF("tc_score_kernel", s);
    tc_score_kernel<false><<<grid, kTcThreads, smem, s>>>(map_q, map_e, P);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  // 4. final select + exact rescoring
  const size_t fsmem = static_cast<size_t>(kFinalCap) * 8 + kKeepCap * 8 + static_cast<size_t>(d) * 4 + 64;
  PSB_PROF("final_select_kernel", s);
  final_select_kernel<<<static_cast<int>(m), 256, fsmem, s>>>(cand_s, cand_i, cand_n, pl.n_slices * kParts, pl.cap, eps, queries,
                                                              table, static_cast<int>(d), bias, static_cast<int>(k),
                                                              id_base, id_stride, out_ids, out_scores, flag, kFinalCap);
  if ((st = launch_status()) != PSB_OK) return st;
  // 5. exact fallback for flagged rows (returns immediately for unflagged ones)
  PSB_PROF("fallback_rows_kernel", s);
  fallback_rows_kernel<<<static_cast<int>(m), 256, static_cast<size_t>(d) * 4, s>>>(
      flag, queries, table, n_items, static_cast<int>(d), bias, static_cast<int>(k), id_base, id_stride, out_ids,
      out_scores);
  return launch_status();
}

// ------------------------------------------------------------------ fp16 shortlist: host side
static int make_map16(CUtensorMap* map, const void* base, int64_t rows, int64_t d, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) return PSB_E_UNSUPPORTED;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(d), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(d) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(kKB16), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? PSB_OK : PSB_E_ARG;
}

// Query tiles resident per CTA: 4 = 512 queries per pass over the table at 64 items per MMA; 2 = 256 queries per pass
// at 128 items per MMA -- half the tcgen05.mma instructions for the same flops (the issuing thread, not the tensor pipe,
// paces the MT = 4 kernel: DESIGN.md section 8) against twice the table passes.  Measured on B200
// (profiles/r02a_tc16_variants.jsonl, 1M items): 4 tiles per CTA win up to a few hundred queries (M = 384: 0.305 vs
// 0.314 ms), 2 tiles x 128 items per MMA from a few thousand on (M = 4096: 2.01 vs 2.06 ms).
static int tc16_max_tiles_per_cta(int m_tiles) { return m_tiles >= 16 ? 2 : 4; }

// candidate lists per (query row, item slice): one per epilogue part that scores columns of the row's query tile
static int tc16_lists_per_slice(int MT) {
  switch (MT) {
    case 1: return Tc16V2<1>::AP;
    case 2: return Tc16V2<2>::AP;
    case 3: return Tc16V2<3>::AP;
    default: return Tc16V2<4>::AP;
  }
}

constexpr int kMaxSegs = 8;
struct Tc16Plan {
  int m_tiles, groups, MT, TN, m_pad, n_slices, total_tiles, pilot_tiles, pilot_step, cap, stages;
  int lists;    // candidate lists per (row, slice)
  int seg[kMaxSegs];   // main-pass segment ends in tiles: [0, seg0) | [seg0, seg1) | ... | [seg(nseg-2), total)
  int nseg;
  int final_cap; // candidates per row the select kernels hold in shared memory (4x the expectation: several CTAs / SM)
  size_t smem;
  int64_t off_thr, off_eps, off_epsin, off_flag, off_cand_n, off_q16, off_dump, off_cand_s, off_cand_i, total;
};

static Tc16Plan plan16_for(int64_t m, int64_t n_items, int64_t d, int64_t k) {
  Tc16Plan p;
  p.m_tiles = static_cast<int>((m + kTM - 1) / kTM);
  const int max_mt = tc16_max_tiles_per_cta(p.m_tiles);
  p.groups = (p.m_tiles + max_mt - 1) / max_mt;
  p.MT = (p.m_tiles + p.groups - 1) / p.groups;
  p.TN = p.MT <= 2 ? 128 : 64;
  p.m_pad = p.groups * p.MT * kTM;
  p.total_tiles = static_cast<int>((n_items + p.TN - 1) / p.TN);
  p.n_slices = kNumSMs / p.groups;
  if (p.n_slices < 1) p.n_slices = 1;
  if (p.n_slices > p.total_tiles) p.n_slices = p.total_tiles;
  // pilot: 8192 items spread over the table.  Its k-th best score only has to carry the first segment of the
  // main pass: the threshold is then refined from the candidates found so far (see catalog_topk_tc16)
  p.pilot_tiles = 8192 / p.TN;
  if (p.pilot_tiles > p.total_tiles) p.pilot_tiles = p.total_tiles;
  p.pilot_step = p.total_tiles / p.pilot_tiles;
  // Main-pass segments: the threshold of segment j is the k-th best of everything seen before it, so a segment that
  // is `ratio` times what has been seen yields ~k * ratio candidates per row -- and every candidate costs epilogue
  // slow-path work that grows with the number of queries, while every extra segment costs a refine launch (~25-55 us).
  // Measured at 1M / 2M items (profiles/tc16_segs.py): dropping the middle segment (2150 instead of 1550 candidates
  // per row) costs +33 us at 384 queries and +0.32 ms at 4096, but saves 17 us at 24.  Hence: few queries -> one
  // refinement; a few hundred -> first segment 10x the pilot, then 5x steps; thousands -> 3x steps from the start.
  // (r = 0: no further refinement; profiles/r02D_tc16_sched.jsonl: 1M items, 4096 queries 2.02 -> 1.90 ms with 3x steps; 24 queries 0.163 -> 0.143 ms
  // with one refinement -- but only on small tables: at 16M one refinement leaves 18k candidates per row, the lists
  // overflow and the exact fallback answers, 341 ms)
  const bool small_table = n_items <= 2500000;
  const int r0 = m <= 1024 ? 10 : 3, r = m <= 64 ? (small_table ? 0 : 5) : (m <= 1024 ? 5 : 3);
  p.nseg = 0;
  {
    int64_t end = static_cast<int64_t>(r0) * 8192 / p.TN;
    while (p.nseg < kMaxSegs - 1 && end < p.total_tiles) {
      p.seg[p.nseg++] = static_cast<int>(end);
      if (r < 2) break;
      // the last refinement must still pay for itself: stop when what is left is less than twice what has been seen
      if (p.total_tiles - end < 2 * end && p.nseg >= 2) break;
      end *= r;
    }
    p.seg[p.nseg++] = p.total_tiles;
  }
  // expected candidates per row: k * sum_j (segment j) / (items seen before segment j)
  const double pil = static_cast<double>(p.pilot_tiles);
  double cands = 0.0;
  {
    double seen = pil;
    int lo = 0;
    for (int j = 0; j < p.nseg; ++j) {
      cands += static_cast<double>(k) * (p.seg[j] - lo) / seen;
      seen = p.seg[j];      // (the pilot tiles are part of the table: seen = segment end)
      lo = p.seg[j];
    }
  }
  p.lists = tc16_lists_per_slice(p.MT);
  const double expect = cands / (p.n_slices * p.lists);
  p.cap = (static_cast<int>(2.0 * expect) + 96 + 31) / 32 * 32;
  p.final_cap = (static_cast<int>(4.0 * cands) + 1024 + 255) / 256 * 256;
  if (p.final_cap > kFinalCap) p.final_cap = kFinalCap;
  const int kblocks = static_cast<int>(d / kKB16);
  const size_t q_bytes = static_cast<size_t>(p.MT) * kblocks * kQBlock16;
  const size_t stage_bytes = static_cast<size_t>(kblocks) * p.TN * 128;
  size_t st = (220 * 1024 - q_bytes) / stage_bytes;
  p.stages = static_cast<int>(st > 8 ? 8 : st);
  p.smem = q_bytes + p.stages * stage_bytes + 512 + 1024;
  int64_t o = 0;
  p.off_thr = o; o += up256(p.m_pad * 4);
  p.off_eps = o; o += up256(p.m_pad * 4);
  p.off_epsin = o; o += up256(p.m_pad * 4);
  p.off_flag = o; o += up256(p.m_pad * 4);
  p.off_cand_n = o; o += up256(static_cast<int64_t>(p.m_pad) * p.n_slices * p.lists * 4);
  p.off_q16 = o; o += up256(static_cast<int64_t>(p.m_pad) * d * 2);
  p.off_dump = o; o += up256(static_cast<int64_t>(p.m_pad) * p.pilot_tiles * p.TN * 4);
  p.off_cand_s = o; o += up256(static_cast<int64_t>(p.m_pad) * p.n_slices * p.lists * p.cap * 4);
  p.off_cand_i = o; o += up256(static_cast<int64_t>(p.m_pad) * p.n_slices * p.lists * p.cap * 4);
  p.total = o + 256;
  return p;
}

static bool tc16_supported(int64_t m, int64_t n_items, int64_t d) {
  return d % kKB16 == 0 && d <= 128 && n_items >= 32768 && m <= static_cast<int64_t>(kNumSMs) * 4 * kTM;
}

int64_t tc16_workspace_bytes(int64_t m, int64_t n_items, int64_t d, int64_t k) {
  if (!tc16_supported(m, n_items, d)) return 0;
  return plan16_for(m, n_items, d, k).total;
}

int catalog_prepare_f16(const float* table, int64_t n_items, int64_t d, void* table_f16, float* stats, cudaStream_t s) {
  cudaMemsetAsync(stats, 0, 16, s);
  PSB_PROF("prep_f16_kernel", s);
  prep_f16_kernel<<<kNumSMs * 8, 256, 0, s>>>(reinterpret_cast<const float4*>(table), n_items, static_cast<int>(d / 4),
                                              static_cast<uint2*>(table_f16), stats);
  return launch_status();
}

template <bool DUMP>
static int launch_tc16(int MT, dim3 grid, size_t smem, cudaStream_t s, const CUtensorMap& mq, const CUtensorMap& me,
                       const Tc16Params& P) {
  static DeviceAttr attr_done;
  if (attr_done.need()) {
    const int lim = 227 * 1024;
    cudaError_t e = cudaFuncSetAttribute(tc16_score_v2_kernel<DUMP, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tc16_score_v2_kernel<DUMP, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tc16_score_v2_kernel<DUMP, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tc16_score_v2_kernel<DUMP, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_done.done();
  }
  PSB_PROF("tc16_score_v3_kernel", s);   // the profiler label the benchmark output has always used for this kernel
  switch (MT) {
    case 1: tc16_score_v2_kernel<DUMP, 1><<<grid, kTcThreads, smem, s>>>(mq, me, P); break;
    case 2: tc16_score_v2_kernel<DUMP, 2><<<grid, kTcThreads, smem, s>>>(mq, me, P); break;
    case 3: tc16_score_v2_kernel<DUMP, 3><<<grid, kTcThreads, smem, s>>>(mq, me, P); break;
    default: tc16_score_v2_kernel<DUMP, 4><<<grid, kTcThreads, smem, s>>>(mq, me, P); break;
  }
  return launch_status();
}

int catalog_topk_tc16(const float* queries, int64_t m, const float* table, const void* table_f16, const float* stats,
                      int64_t n_items, int64_t d, const float* bias, int64_t k, int64_t id_base, int64_t id_stride,
                      void* workspace, int64_t workspace_bytes, int64_t* out_ids, float* out_scores, cudaStream_t s) {
  if (!tc16_supported(m, n_items, d))
    return catalog_topk_exact(queries, m, table, n_items, d, bias, k, id_base, id_stride, workspace,
                              workspace_bytes, out_ids, out_scores, s);
  const Tc16Plan pl = plan16_for(m, n_items, d, k);
  const int64_t ex_bytes = (exact_workspace_bytes(m, n_items) + 255) / 256 * 256;
  if (workspace_bytes < ex_bytes + pl.total) return PSB_E_WORKSPACE;
  unsigned char* ws = static_cast<unsigned char*>(workspace) + ex_bytes;
  float* thr = reinterpret_cast<float*>(ws + pl.off_thr);
  float* eps = reinterpret_cast<float*>(ws + pl.off_eps);
  float* eps_in = reinterpret_cast<float*>(ws + pl.off_epsin);
  int32_t* flag = reinterpret_cast<int32_t*>(ws + pl.off_flag);
  int32_t* cand_n = reinterpret_cast<int32_t*>(ws + pl.off_cand_n);
  __half* q16 = reinterpret_cast<__half*>(ws + pl.off_q16);
  float* dump = reinterpret_cast<float*>(ws + pl.off_dump);
  float* cand_s = reinterpret_cast<float*>(ws + pl.off_cand_s);
  int32_t* cand_i = reinterpret_cast<int32_t*>(ws + pl.off_cand_i);

  alignas(64) CUtensorMap map_q, map_e;
  int st;
  if ((st = make_map16(&map_q, q16, pl.m_pad, d, kTM)) != PSB_OK) return st;
  if ((st = make_map16(&map_e, table_f16, n_items, d, pl.TN)) != PSB_OK) return st;
  static DeviceAttr attr_done;
  if (attr_done.need()) {
    cudaError_t e1 = cudaFuncSetAttribute(final_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    cudaError_t e2 = cudaFuncSetAttribute(pilot_threshold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    if (e2 == cudaSuccess)
      e2 = cudaFuncSetAttribute(refine_threshold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    if (e1 != cudaSuccess || e2 != cudaSuccess) return static_cast<int>(e1 != cudaSuccess ? e1 : e2);
    attr_done.done();
  }
  cudaMemsetAsync(flag, 0, static_cast<size_t>(pl.m_pad) * 4, s);
  PSB_PROF("q16_kernel", s);
  q16_kernel<<<(pl.m_pad + 7) / 8, 256, 0, s>>>(queries, static_cast<int>(m), pl.m_pad, static_cast<int>(d), stats, q16, eps_in);
  if ((st = launch_status()) != PSB_OK) return st;

  Tc16Params P;
  P.m = static_cast<int>(m);
  P.n_items = static_cast<int>(n_items);
  P.kblocks = static_cast<int>(d / kKB16);
  P.stages = pl.stages;
  P.bias = bias;
  P.thr = thr;
  P.dump = dump;
  P.ld_dump = pl.pilot_tiles * pl.TN;
  P.cand_s = cand_s;
  P.cand_i = cand_i;
  P.cand_n = cand_n;
  P.cap = pl.cap;
  P.append = 0;
  // 1. pilot
  P.tile_begin = 0;
  P.tile_step = pl.pilot_step;
  P.n_tiles = pl.pilot_tiles;
  {
    const int slices = pl.n_slices < pl.pilot_tiles ? pl.n_slices : pl.pilot_tiles;
    if ((st = launch_tc16<true>(pl.MT, dim3(slices, pl.groups), pl.smem, s, map_q, map_e, P)) != PSB_OK) return st;
  }
  // 2. thresholds (eps from the measured quantisation errors)
  const bool stage_pilot = static_cast<size_t>(P.ld_dump) * 4 <= 160 * 1024;
  PSB_PROF("pilot_threshold_kernel", s);
  pilot_threshold_kernel<<<static_cast<int>(m), 256, stage_pilot ? static_cast<size_t>(P.ld_dump) * 4 : 0, s>>>(
      dump, P.ld_dump, P.ld_dump, static_cast<int>(k), queries, static_cast<int>(d), stats, eps_in, thr, eps,
      stage_pilot ? 1 : 0);
  if ((st = launch_status()) != PSB_OK) return st;
  // 3. main pass in three growing segments; after each of the first two the threshold is refined from the
  //    candidates found so far (the k-th best of 80k / 400k items prunes 10x / 40x harder than the pilot's), which
  //    keeps the epilogue's slow path -- appending a candidate -- rare for most of the table
  P.tile_step = 1;
  P.append = 0;
  int seg_lo = 0;
  for (int sgi = 0; sgi < pl.nseg; ++sgi) {
    const int seg_hi = pl.seg[sgi];
    if (seg_hi > seg_lo) {
      P.tile_begin = seg_lo;
      P.n_tiles = seg_hi - seg_lo;
      const int slices = pl.n_slices;   // the bucket index of a candidate list must not depend on the segment
      if ((st = launch_tc16<false>(pl.MT, dim3(slices, pl.groups), pl.smem, s, map_q, map_e, P)) != PSB_OK) return st;
      P.append = 1;
      if (sgi < pl.nseg - 1 && seg_hi < pl.total_tiles) {
        PSB_PROF("refine_threshold_kernel", s);
        refine_threshold_kernel<<<static_cast<int>(m), 256, static_cast<size_t>(pl.final_cap) * 4, s>>>(
            cand_s, cand_n, pl.n_slices * pl.lists, pl.cap, eps, static_cast<int>(k), thr, pl.final_cap);
        if ((st = launch_status()) != PSB_OK) return st;
      }
    }
    seg_lo = seg_hi > seg_lo ? seg_hi : seg_lo;
  }
  // 4. final select + exact fp32 rescoring, 5. exact fallback for flagged rows
  const size_t fsmem = static_cast<size_t>(pl.final_cap) * 8 + kKeepCap * 8 + static_cast<size_t>(d) * 4 + 64;
  PSB_PROF("final_select_kernel", s);
  final_select_kernel<<<static_cast<int>(m), 256, fsmem, s>>>(cand_s, cand_i, cand_n, pl.n_slices * pl.lists, pl.cap, eps, queries,
                                                              table, static_cast<int>(d), bias, static_cast<int>(k),
                                                              id_base, id_stride, out_ids, out_scores, flag, pl.final_cap);
  if ((st = launch_status()) != PSB_OK) return st;
  PSB_PROF("fallback_rows_kernel", s);
  fallback_rows_kernel<<<static_cast<int>(m), 256, static_cast<size_t>(d) * 4, s>>>(
      flag, queries, table, n_items, static_cast<int>(d), bias, static_cast<int>(k), id_base, id_stride, out_ids,
      out_scores);
  return launch_status();
}

}  // namespace psb

// ------------------------------------------------------------------ TMEM read bandwidth probe (debug aid)
// The catalog contraction has K = d = 128: every fp32 accumulator element is read back (tcgen05.ld) after only 8
// MMAs, i.e. 4 B of TMEM read per 256 flop, so the TMEM read rate bounds the tensor-pipe utilisation this design
// can reach (128 B/clk/SM are needed to keep kind::f16 at peak, 77 B/clk for 60 %).  The B300 notes quote "64 B/clk"
// without saying per SM or per sub-partition; this probe measures it on the part at hand: `warps` warps (4 per SM
// sub-partition at 16) each issue `iters` x tcgen05.ld.32x32b.x32 (4 KB) back to back.
namespace psb {
__global__ void __launch_bounds__(512, 1) tmem_read_probe_kernel(int iters, unsigned long long* __restrict__ cycles,
                                                                 uint32_t* __restrict__ sink) {
  __shared__ uint32_t slot;
  const int warp = threadIdx.x >> 5;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t base = slot + (static_cast<uint32_t>((warp & 3) * 32) << 16);
  uint32_t acc = 0;
  uint32_t v[32];
  const long long t0 = clock64();
#pragma unroll 4
  for (int i = 0; i < iters; ++i) {
    tc_ld32(base + static_cast<uint32_t>(((i + warp) & 15) * 32), v);      // walks the 512 columns; ld + wait::ld
    acc ^= v[0] ^ v[13] ^ v[31];
  }
  const long long t1 = clock64();
  if ((threadIdx.x & 31) == 0) cycles[blockIdx.x * 16 + warp] = static_cast<unsigned long long>(t1 - t0);
  if (acc == 0x9e3779b9u) sink[0] = acc;                                    // keeps the loads alive
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(slot), "n"(512));
  }
}
}  // namespace psb

// bytes_per_clk[0] = TMEM bytes read per SM clock by ONE CTA with `warps` warps (4, 8, 12 or 16), slowest warp's
// clock; bytes_per_clk[1] = the same with one such CTA on every SM at once.  Allocates 20 KB of scratch for the call.
extern "C" int psb_debug_tmem_read_bw(int32_t warps, int32_t iters, double* bytes_per_clk) {
  if (bytes_per_clk == nullptr || warps < 1 || warps > 16 || iters < 1) return PSB_E_ARG;
  unsigned long long* cyc = nullptr;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&cyc), (psb::kNumSMs * 16 + 1) * sizeof(unsigned long long));
  if (e != cudaSuccess) return static_cast<int>(e);
  uint32_t* sink = reinterpret_cast<uint32_t*>(cyc + psb::kNumSMs * 16);
  static unsigned long long h[psb::kNumSMs * 16];
  for (int pass = 0; pass < 2 && e == cudaSuccess; ++pass) {
    const int ctas = pass == 0 ? 1 : psb::kNumSMs;
    e = cudaMemset(cyc, 0, psb::kNumSMs * 16 * sizeof(unsigned long long));
    for (int rep = 0; rep < 2 && e == cudaSuccess; ++rep) {               // first launch warms the instruction cache
      psb::tmem_read_probe_kernel<<<ctas, warps * 32>>>(iters, cyc, sink);
      e = cudaDeviceSynchronize();
    }
    if (e == cudaSuccess) e = cudaMemcpy(h, cyc, sizeof(h), cudaMemcpyDeviceToHost);
    unsigned long long worst = 1;
    for (int i = 0; i < ctas * 16; ++i) worst = h[i] > worst ? h[i] : worst;
    bytes_per_clk[pass] = static_cast<double>(warps) * iters * 4096.0 / static_cast<double>(worst);
  }
  cudaFree(cyc);
  return e == cudaSuccess ? PSB_OK : static_cast<int>(e);
}
