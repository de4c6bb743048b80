// out[M, J] = A[M, K] . Bt[J, K]^T (+ bias) on tcgen05 with fp32-grade accuracy: the "3xTF32" split.
//
// Why: the encoder's projections (models/neural.py:98-231 MultiHeadedAttention linear_keys / linear_values /
// linear_query, models/transformer.py:37-88) are GEMM-shaped but run as fp32 FFMA tiles (encoder_fwd.cu rows_gemm_kernel,
// 18.6 us per launch at batch 384) because plain TF32 misses the 1e-5 parity bar by two orders of magnitude
// (tools/tf32x3_numerics.py: 8.6e-4).  kind::tf32 reads fp32 words and uses 19 of their bits, so
//     a = a_hi + a_lo,   a_hi = a with the low 13 mantissa bits cleared,   a_lo = a - a_hi   (exact in fp32)
//     a.b = a_hi.b_hi + a_lo.b_hi + a_hi.b_lo + O(2^-22 |a||b|)
// is three MMAs per k-step with fp32 accumulation in TMEM.  The two correction products go to an accumulator of their
// own (64 extra TMEM columns): whatever rounding the accumulate step uses, its error there is relative to a sum 2^-11
// times smaller (same study: <= 3e-6 of max|out| even if every accumulate truncates; 8e-7 with round-to-nearest).
//
// One CTA = 128 rows x N output columns (N = 64, K chunks of 64, 2 stages; or N = 128, K chunks of 32, 3 stages):
//   warp 0      TMA producer: A chunk (boxes of 128 rows x 32 fp32) and Bt chunk (boxes of N rows x 32 fp32),
//               128-byte swizzle, straight from the row-major operands (K contiguous = K-major, no transposes)
//   warps 2..5  split: every fp32 word of the landed tiles is rewritten in place as its hi part (so the tensor core sees
//               the same value whether it truncates or rounds) and its lo part goes to the twin tile at the SAME offset --
//               an elementwise map, so the swizzled layout carries over; fence.proxy.async, then one arrive per warp
//   warp 1      MMA issuer (converged warp, elected-lane predicate: see catalog_tc.cu tc_mma_f16_if for why):
//               per k-step of 8: main += hi.hi, corr += lo.hi, corr += hi.lo   (M 128, N, K 8)
//   warps 2..5  epilogue: thread = output row (TMEM lane) holding its N sums (main + corr) in registers, handed to an
//               epilogue functor (EpiBias: out = acc + bias) -- a row never leaves its thread
// Rows >= M (M may live on the device: the number of active tokens) are computed on whatever the buffer holds and not
// stored; a GEMM row depends on its own A row only.  CTAs whose first row is >= M exit at once.
//
// This file holds the encoder's tensor-core path (the default; PSB_ENC_TC=0 selects the FFMA path, see enc_tc_enabled):
//   gemm3_tf32_kernel          one product with a fused epilogue: the q / K|V projections, the backward's grad-xn product
//   tail_ctx_kernel + tail_fused_tc_kernel      the forward tail as ONE cluster kernel (three chained products)
//   tail_bwd_fused_tc_kernel   the backward tail's product chain as one cluster kernel, transposed form
//                              (+ encoder_bwd.cu tail_attn_bwd_kernel for the attention backward)
// All of them have run on B200s: profiles/r02a_gemm3.jsonl (accuracy against fp64), profiles/r02W_diff_enc_*.jsonl (stage by
// stage against the FFMA kernels), tests/test_gpu_enc_tc_levels.py (forward and backward, every round).
#include <stdlib.h>
#include <string.h>

#include "encoder_common.cuh"
#include "tc_ptx.cuh"

namespace psb {
namespace enc {

constexpr int kG3M = 128;                                   // rows per CTA (UMMA M = TMEM lanes)
constexpr int kG3Threads = 64 + 128;                        // TMA warp, MMA warp, 4 split / epilogue warps

// Tile shapes: N output columns per CTA (UMMA N), KC floats of K per stage.  <64, 64>: projections and the FFN's first
// layer (many column tiles); <128, 32>: products whose epilogue needs the whole d = 128 row (LayerNorm).
template <int N, int KC>
struct G3Cfg {
  static_assert((N == 64 || N == 128) && (KC == 32 || KC == 64), "tile shapes");
  static constexpr int kKB = KC / 32;                                   // 128-byte swizzle rows per stage
  static constexpr uint32_t kABlock = kG3M * 128;                       // 128 rows x 128 B = 16 KB
  static constexpr uint32_t kBBlock = N * 128;                          // N rows x 128 B
  static constexpr uint32_t kAStage = kKB * kABlock;                    // hi (or lo) A tile of one stage
  static constexpr uint32_t kBStage = kKB * kBBlock;
  static constexpr uint32_t kStageBytes = 2 * (kAStage + kBStage);      // [A hi][A lo][B hi][B lo]
  static constexpr int kStages = kStageBytes <= 64 * 1024 ? 3 : 2;      // 64 KB x 3 or 96 KB x 2
  static constexpr size_t kSmem = static_cast<size_t>(kStages) * kStageBytes + 1024 /* alignment slack */ + 128 /* barriers */;
  static constexpr int kTmemCols = 2 * N;                               // main accumulator: columns 0..N-1, corrections: N..2N-1
  // cute::UMMA::InstrDescriptor (see catalog_tc.cu kIdesc): F32 accumulate, TF32 x TF32, K-major A and B, N, M = 128
  static constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
                                     (static_cast<uint32_t>(kG3M >> 4) << 24);
};

struct G3Params {
  const int32_t* m_dev;   // rows on the device (active tokens) or NULL
  int m_host;
  int K;
  int split;              // Bt rows [0, split) come from map_b0, the rest from map_b1 (K | V: two weight tensors)
};

__device__ __forceinline__ uint32_t g3_elect_one() {
  uint32_t leader;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(leader));
  return leader;
}
__device__ __forceinline__ void g3_mma_tf32_if(uint32_t leader, uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\tsetp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void g3_commit_if(uint32_t leader, uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)),
      "r"(leader)
      : "memory");
}

// hi = the 19 bits kind::tf32 uses (sign, exponent, 10 mantissa bits); lo = the rest, exact
__device__ __forceinline__ void g3_split(float4 v, float4& hi, float4& lo) {
  hi.x = __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
  hi.y = __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
  hi.z = __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
  hi.w = __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
  lo.x = v.x - hi.x;
  lo.y = v.y - hi.y;
  lo.z = v.z - hi.z;
  lo.w = v.w - hi.w;
}

// ------------------------------------------------------------------ epilogues: thread = one output row, N columns
// out = acc + bias
template <int N>
struct EpiBias {
  const float* bias;      // [J] or NULL
  float* out;
  int ldo;
  __device__ __forceinline__ void operator()(int row, int n0, float (&acc)[N]) const {
    float* o = out + static_cast<size_t>(row) * ldo + n0;
#pragma unroll
    for (int i = 0; i < N; i += 4) {
      float4 r = make_float4(acc[i], acc[i + 1], acc[i + 2], acc[i + 3]);
      if (bias != nullptr) {
        const float4 b = *reinterpret_cast<const float4*>(bias + n0 + i);
        r.x += b.x; r.y += b.y; r.z += b.z; r.w += b.w;
      }
      *reinterpret_cast<float4*>(o + i) = r;
    }
  }
};

// ------------------------------------------------------------------ the kernel
template <int N, int KC, class Epi>
__global__ void __launch_bounds__(kG3Threads, 1)
gemm3_tf32_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b0,
                  const __grid_constant__ CUtensorMap map_b1, const G3Params P, const Epi epi) {
  using C = G3Cfg<N, KC>;
  const int M = P.m_dev != nullptr ? *P.m_dev : P.m_host;
  const int r0 = blockIdx.x * kG3M;
  if (r0 >= M) {                                            // uniform: before any barrier / TMEM allocation
    pdl_wait();                                             // (a grid that completes has waited for its predecessor)
    return;
  }
  extern __shared__ unsigned char smem_dyn[];
  // 128-byte-swizzled operand tiles need a 1024-byte aligned base
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(C::kStages) * C::kStageBytes);
  uint64_t* full = bars;                                    // [stage] TMA bytes landed
  uint64_t* split_done = bars + C::kStages;                 // [stage] hi / lo tiles written, visible to the async proxy
  uint64_t* empty = bars + 2 * C::kStages;                  // [stage] the stage's MMAs have read it
  uint64_t* acc_full = bars + 3 * C::kStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * C::kStages + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.y * N;
  const int chunks = P.K / KC;

  if (threadIdx.x == 0) {
    for (int st = 0; st < C::kStages; ++st) {
      mbar_init(full + st, 1);
      mbar_init(split_done + st, 4);
      mbar_init(empty + st, 1);
    }
    mbar_init(acc_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(C::kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      pdl_wait();                                           // A rows come from the kernel before this one in the stream
      const bool first = n0 < P.split;
      const CUtensorMap* mb = first ? &map_b0 : &map_b1;
      const int brow = first ? n0 : n0 - P.split;
      for (int c = 0; c < chunks; ++c) {
        const int st = c % C::kStages;
        const uint32_t ph = (c / C::kStages) & 1;
        mbar_wait(empty + st, ph ^ 1);
        mbar_expect_tx(full + st, C::kAStage + C::kBStage);
        unsigned char* base = smem + static_cast<size_t>(st) * C::kStageBytes;
        for (int kb = 0; kb < C::kKB; ++kb) tma_load_2d(base + kb * C::kABlock, &map_a, c * KC + kb * 32, r0, full + st);
        for (int kb = 0; kb < C::kKB; ++kb)
          tma_load_2d(base + 2 * C::kAStage + kb * C::kBBlock, mb, c * KC + kb * 32, brow, full + st);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: all 32 lanes run the loop, the instructions are predicated on the elected lane =====
    const uint32_t leader = g3_elect_one();
    for (int c = 0; c < chunks; ++c) {
      const int st = c % C::kStages;
      const uint32_t ph = (c / C::kStages) & 1;
      mbar_wait(split_done + st, ph);
      tc_fence_after();
      const uint32_t base = smem_u32(smem + static_cast<size_t>(st) * C::kStageBytes);
      const uint64_t a_hi = umma_desc(base);
      const uint64_t a_lo = umma_desc(base + C::kAStage);
      const uint64_t b_hi = umma_desc(base + 2 * C::kAStage);
      const uint64_t b_lo = umma_desc(base + 2 * C::kAStage + C::kBStage);
#pragma unroll
      for (int kb = 0; kb < C::kKB; ++kb) {
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {                    // 4 x (K = 8 tf32 = 32 bytes) inside one swizzle row
          const uint64_t oa = static_cast<uint64_t>(kb) * (C::kABlock >> 4) + k4 * 2;
          const uint64_t ob = static_cast<uint64_t>(kb) * (C::kBBlock >> 4) + k4 * 2;
          const uint32_t acc = (c | kb | k4) != 0 ? 1u : 0u;
          g3_mma_tf32_if(leader, tmem_base, a_hi + oa, b_hi + ob, C::kIdesc, acc);
          g3_mma_tf32_if(leader, tmem_base + N, a_lo + oa, b_hi + ob, C::kIdesc, acc);
          g3_mma_tf32_if(leader, tmem_base + N, a_hi + oa, b_lo + ob, C::kIdesc, 1u);
        }
      }
      g3_commit_if(leader, empty + st);                     // the stage may be refilled once these MMAs have read it
    }
    g3_commit_if(leader, acc_full);
  } else {
    // ===== split (per stage), then epilogue =====
    const int t = threadIdx.x - 64;                         // 0..127
    for (int c = 0; c < chunks; ++c) {
      const int st = c % C::kStages;
      const uint32_t ph = (c / C::kStages) & 1;
      mbar_wait(full + st, ph);
      unsigned char* base = smem + static_cast<size_t>(st) * C::kStageBytes;
      float4* a_hi = reinterpret_cast<float4*>(base);
      float4* a_lo = reinterpret_cast<float4*>(base + C::kAStage);
      float4* b_hi = reinterpret_cast<float4*>(base + 2 * C::kAStage);
      float4* b_lo = reinterpret_cast<float4*>(base + 2 * C::kAStage + C::kBStage);
#pragma unroll 4
      for (int i = t; i < static_cast<int>(C::kAStage / 16); i += 128) {
        float4 hi, lo;
        g3_split(a_hi[i], hi, lo);
        a_hi[i] = hi;
        a_lo[i] = lo;
      }
#pragma unroll 4
      for (int i = t; i < static_cast<int>(C::kBStage / 16); i += 128) {
        float4 hi, lo;
        g3_split(b_hi[i], hi, lo);
        b_hi[i] = hi;
        b_lo[i] = lo;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core reads
      __syncwarp();
      if (lane == 0) mbar_arrive(split_done + st);
    }
    const int quarter = warp & 3;                           // a warp may only touch TMEM lanes 32 * (warp % 4) .. + 31
    const int row = r0 + quarter * 32 + lane;
    const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    mbar_wait(acc_full, 0);
    tc_fence_after();
    float acc[N];
#pragma unroll
    for (int cc = 0; cc < N / 32; ++cc) {
      uint32_t vm[32], vc[32];
      __syncwarp();
      tc_ld32x2(t_addr + static_cast<uint32_t>(cc * 32), vm, vc, static_cast<uint32_t>(N));
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[cc * 32 + i] = __uint_as_float(vm[i]) + __uint_as_float(vc[i]);
    }
    if (row < M) epi(row, n0, acc);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(C::kTmemCols));
  }
}

// ------------------------------------------------------------------ host side
// rows x cols fp32, row stride ld floats -> boxes of box_rows rows x 32 floats, 128-byte swizzle, OOB reads as zero
static int g3_make_map(CUtensorMap* map, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) return PSB_E_UNSUPPORTED;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 4};
  cuuint32_t box[2] = {32u, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? PSB_OK : PSB_E_ARG;
}

// PSB_ENC_TC=0 selects the fp32 FFMA kernels everywhere (encoder_fwd.cu / encoder_bwd.cu): the reference the tests compare
// the tensor-core path against.  Unset, or any other value: every encoder product that has a tensor-core form runs on
// tcgen05 (the projections, the forward tail, the backward tail).  The FFMA kernels also remain the fallback for the shapes
// the tensor-core kernels do not take (d != 128, ff != 512, misaligned operands).  Read once per process.
bool enc_tc_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("PSB_ENC_TC");
    v = (e != nullptr && strcmp(e, "0") == 0) ? 0 : 1;
  }
  return v == 1;
}

// One launch: out-tile epilogue `epi` over A [m rows, K] (row stride lda) and Bt rows [0, split) from Bt0, the rest from Bt1
template <int N, int KC, class Epi>
static int g3_launch(const char* name, const float* A, int lda, const int32_t* m_dev, int m_host, int m_max, int K,
                     const float* Bt0, const float* Bt1, int split, int J, const Epi& epi, cudaStream_t s) {
  using C = G3Cfg<N, KC>;
  if (m_max <= 0) return PSB_OK;
  static DeviceAttr attr_done;                            // one flag per instantiation
  if (attr_done.need()) {
    cudaError_t e = cudaFuncSetAttribute(gemm3_tf32_kernel<N, KC, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(C::kSmem));
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_done.done();
  }
  alignas(64) CUtensorMap map_a, map_b0, map_b1;
  const int rows0 = Bt1 != nullptr ? split : J;
  int st;
  if ((st = g3_make_map(&map_a, A, m_max, K, lda, kG3M)) != PSB_OK) return st;
  if ((st = g3_make_map(&map_b0, Bt0, rows0, K, K, N)) != PSB_OK) return st;
  if (Bt1 != nullptr) {
    if ((st = g3_make_map(&map_b1, Bt1, J - split, K, K, N)) != PSB_OK) return st;
  } else {
    map_b1 = map_b0;
  }
  G3Params P;
  P.m_dev = m_dev;
  P.m_host = m_host;
  P.K = K;
  P.split = rows0;
  const dim3 grid(static_cast<unsigned>((m_max + kG3M - 1) / kG3M), static_cast<unsigned>(J / N));
  PSB_PROF(name, s);
  {
    const cudaError_t le = launch_pdl(gemm3_tf32_kernel<N, KC, Epi>, grid, dim3(kG3Threads), C::kSmem, s, map_a, map_b0, map_b1,
                                      P, epi);
    if (le != cudaSuccess) return static_cast<int>(le);
  }
  return launch_status();
}

bool rows_gemm_tc_supported(const float* A, int lda, int K, const float* Bt0, const float* Bt1, int split, int J,
                            const float* bias, const float* out, int ldo) {
  if (K <= 0 || K % 64 != 0 || J <= 0 || J % 64 != 0 || (lda & 3) != 0 || (ldo & 3) != 0) return false;
  if (Bt1 != nullptr && (split <= 0 || split >= J || split % 64 != 0)) return false;
  return A != nullptr && Bt0 != nullptr && out != nullptr && !misaligned16(A) && !misaligned16(Bt0) &&
         !misaligned16(Bt1) && !misaligned16(bias) && !misaligned16(out);
}

int launch_rows_gemm_tc(const float* A, int lda, const int32_t* m_dev, int m_host, int m_max, int K, const float* Bt0,
                        const float* Bt1, int split, int J, const float* bias, float* out, int ldo, cudaStream_t s) {
  if (!rows_gemm_tc_supported(A, lda, K, Bt0, Bt1, split, J, bias, out, ldo)) return PSB_E_UNSUPPORTED;
  EpiBias<64> epi;
  epi.bias = bias;
  epi.out = out;
  epi.ldo = ldo;
  return g3_launch<64, 64>("gemm3_tf32_kernel", A, lda, m_dev, m_host, m_max, K, Bt0, Bt1, split, J, epi, s);
}

// ------------------------------------------------------------------ forward tail: attention context
// Steps 1 + 2 of tail_fwd_kernel on their own: ctx[row] = sum_al dropout_1(P)[h, al] * V[al], one warp per copy row,
// lane = 4 columns (d = 128), the same sequential fmaf chain over the active tokens -> the same bits.
__global__ void __launch_bounds__(256) tail_ctx_kernel(Dims D, const int32_t* __restrict__ nact, const int32_t* __restrict__ off,
                                                       const int32_t* __restrict__ tok, const float* __restrict__ Pw,
                                                       const float* __restrict__ kv, float* __restrict__ ctx,
                                                       const uint64_t* __restrict__ seed_dev, float* __restrict__ ctx_hl = nullptr) {
  pdl_trigger();                            // tail_fused_tc_kernel may set itself up and prefetch its weights
  pdl_wait();                               // P comes from attn_fwd_kernel, the kernel before this one
  const int lane = threadIdx.x & 31;
  const int grow = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (grow >= D.S * D.C) return;
  const int s = grow / D.C, d = D.d, H = D.H, T = D.T, dh = D.dh;
  const int j = lane * 4;
  const Drop drop = make_drop(seed_dev, D.thr, D.keep);
  const int na = nact[s], base = off[s];
  const int h0 = j / dh, h1 = (j + 1) / dh, h2 = (j + 2) / dh, h3 = (j + 3) / dh;
  float4 acc = zero4();
  // four tokens per trip: their loads and Philox draws are independent, only the fmaf chain is sequential (and keeps the
  // token order of tail_fwd_kernel, so the sums are the same bits)
  // dh % 16 == 0: the four lanes lane & ~3 .. + 3 hold columns of ONE head, so each of them draws the multiplier of one of
  // the trip's four tokens and the four are swapped by shuffle -- a quarter of the Philox calls
  const bool share = (dh & 15) == 0;
  for (int a0 = 0; a0 < na; a0 += 4) {
    float w[4][4];
    float4 v[4];
    float msh = 1.f;
    if (drop.on() && share) {
      const int al = a0 + (lane & 3) < na ? a0 + (lane & 3) : na - 1;
      msh = drop.mul1(1u, (static_cast<uint64_t>(grow) * H + h0) * T + static_cast<uint64_t>(tok[base + al]));
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int al = a0 + u < na ? a0 + u : na - 1;
      const float* pw = Pw + static_cast<size_t>(base + al) * H;
      w[u][0] = pw[h0]; w[u][1] = pw[h1]; w[u][2] = pw[h2]; w[u][3] = pw[h3];
      v[u] = *reinterpret_cast<const float4*>(kv + static_cast<size_t>(base + al) * 2 * d + d + j);
      if (drop.on()) {
        if (share) {
          const float m0 = __shfl_sync(kFull, msh, (lane & ~3) | u);
          w[u][0] *= m0; w[u][1] *= m0; w[u][2] *= m0; w[u][3] *= m0;
          continue;
        }
        const uint64_t t = static_cast<uint64_t>(tok[base + al]);
        const float m0 = drop.mul1(1u, (static_cast<uint64_t>(grow) * H + h0) * T + t);
        if (h0 == h3) {                     // dh % 4 == 0: the lane's four columns belong to one head -> one draw
          w[u][0] *= m0; w[u][1] *= m0; w[u][2] *= m0; w[u][3] *= m0;
        } else {
          w[u][0] *= m0;
          w[u][1] *= drop.mul1(1u, (static_cast<uint64_t>(grow) * H + h1) * T + t);
          w[u][2] *= drop.mul1(1u, (static_cast<uint64_t>(grow) * H + h2) * T + t);
          w[u][3] *= drop.mul1(1u, (static_cast<uint64_t>(grow) * H + h3) * T + t);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (a0 + u < na) {
        acc.x = fmaf(w[u][0], v[u].x, acc.x);
        acc.y = fmaf(w[u][1], v[u].y, acc.y);
        acc.z = fmaf(w[u][2], v[u].z, acc.z);
        acc.w = fmaf(w[u][3], v[u].w, acc.w);
      }
    }
  }
  *reinterpret_cast<float4*>(ctx + static_cast<size_t>(grow) * d + j) = acc;
  if (ctx_hl != nullptr) {                  // operand of tail_fused_tc_kernel: tf32 hi part, exact remainder S*C rows further
    float4 hi, lo;
    g3_split(acc, hi, lo);
    *reinterpret_cast<float4*>(ctx_hl + static_cast<size_t>(grow) * d + j) = hi;
    *reinterpret_cast<float4*>(ctx_hl + (static_cast<size_t>(D.S) * D.C + grow) * d + j) = lo;
  }
}

// ------------------------------------------------------------------ forward tail as ONE cluster kernel
// tail_ctx_kernel, then tail_fused_tc_kernel: the three products of the tail (out-projection, FFN up, FFN down) chained
// inside one launch, the FFN's hidden dimension split over a cluster of 4 CTAs.
//
//   cluster = one tile of 128 copy rows; CTA q of the cluster owns hidden columns [128 q, 128 q + 128)
//   phase 1  acc1 = ctx . Wo^T           (every CTA of the cluster: 128 x 128 x 128, replicated -- it is 1/9 of the flops
//            and replicating it is cheaper than a broadcast)      epilogue: y, n = LN_ff(y) -> A operand of phase 2
//   phase 2  acc2 = n . W1[q]^T          epilogue: pre1, h1 = dropout(gelu(pre1)) (saved) -> A operand of phase 3
//   phase 3  acc3 = h1[:, q] . W2[:, q]^T   (partial sums over this CTA's 128 hidden columns)
//   reduce   the four partial tiles are summed through distributed shared memory in CTA order 0..3 (deterministic);
//            CTA q finishes rows [32 q, 32 q + 32): z, out = LN_out(z)
// One A buffer (128 rows x 128 K as hi + lo tiles, 128 KB) is rewritten by each epilogue in the swizzled K-major layout
// the next phase's MMAs read -- activations never leave the SM between the products; the 12 weight chunks (128 x 32
// fp32 each) stream through 3 stages, prefetched across the phases by the TMA warp and split by warps of their own.
// Every operand is split hi / lo as in gemm3_tf32_kernel (3 MMAs per k-step, corrections in their own accumulator).
constexpr int kFtThreads = 576;            // warp 0 TMA, warp 1 MMA, warps 2-17 epilogue
constexpr int kFtEpiWarps = 16;            // epilogue warp e = warp - 2: TMEM lane quarter warp % 4, columns [32 (e / 4), + 32)
constexpr int kFtCluster = 4;
constexpr uint32_t kFtABytes = 128 * 128 * 4;             // one A tile (hi or lo): 4 swizzle blocks of 16 KB
constexpr uint32_t kFtBBytes = 128 * 32 * 4;              // one weight chunk (hi or lo)
constexpr int kFtStages = 3;
constexpr uint32_t kFtStage = 2 * kFtBBytes;
constexpr size_t kFtSmem = 2 * kFtABytes + kFtStages * kFtStage + 1024 /* alignment slack */ + 256 /* barriers */;
constexpr uint32_t kFtIdesc = G3Cfg<128, 32>::kIdesc;

struct FtParams {
  Dims D;
  int SC;
  const float *xo, *bo, *b1, *b2, *ln_ff_g, *ln_ff_b, *ln_out_g, *ln_out_b;
  float *y, *n, *z, *pre1, *h1, *out;
  const uint64_t* seed_dev;
  int save_dact;               // the pre1 slot receives dropout_3 . gelu'(pre1) (what the tensor-core backward multiplies by)
  unsigned long long* trace;   // PSB_FT_TRACE=1: %globaltimer at the phase boundaries of CTA 0 (psb_debug_tail_trace)
};

__device__ __forceinline__ void ft_mark(const FtParams& P, int slot) {
  if (P.trace != nullptr && blockIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    P.trace[slot] = t;
  }
}

__device__ __forceinline__ uint32_t ft_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void ft_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void ft_epi_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }   // the 16 epilogue warps
__device__ __forceinline__ float4 ft_ld_peer4(uint32_t local_addr, uint32_t cta) {
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(local_addr), "r"(cta));
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(ra) : "memory");
  return v;
}
// float4 chunk c4 (columns 4 c4 .. 4 c4 + 3 of K = 128) of row r inside a K-major 128-byte-swizzled A tile
__device__ __forceinline__ uint32_t ft_a_off(int r, int c4) {
  return static_cast<uint32_t>((c4 >> 3) * 16384 + r * 128 + (((c4 & 7) ^ (r & 7)) << 4));
}
__device__ __forceinline__ void ft_store_a(unsigned char* a_hi, unsigned char* a_lo, int r, int c4, const float4& v) {
  float4 hi, lo;
  g3_split(v, hi, lo);
  const uint32_t o = ft_a_off(r, c4);
  *reinterpret_cast<float4*>(a_hi + o) = hi;
  *reinterpret_cast<float4*>(a_lo + o) = lo;
}
// accumulator columns [col, col + 32) of this thread's TMEM lane: main + corrections
// (two 16-column halves: 18 warps leave 96 registers per thread, and 64 transient ones on top of the 32 sums do not fit)
__device__ __forceinline__ void ft_ld16x2(uint32_t taddr, uint32_t (&v)[16], uint32_t (&w)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]), "=r"(w[8]),
        "=r"(w[9]), "=r"(w[10]), "=r"(w[11]), "=r"(w[12]), "=r"(w[13]), "=r"(w[14]), "=r"(w[15])
      : "r"(taddr + 128u));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 32 values of this thread's TMEM lane written back to columns [taddr, taddr + 32): the forward kernel parks
// dropout_3 . gelu'(pre1) over the main accumulator of product 2 until the end of the kernel
__device__ __forceinline__ void ft_st32(uint32_t taddr, const float (&v)[32]) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(
            taddr + static_cast<uint32_t>(h * 16)),
        "r"(__float_as_uint(v[h * 16 + 0])), "r"(__float_as_uint(v[h * 16 + 1])), "r"(__float_as_uint(v[h * 16 + 2])),
        "r"(__float_as_uint(v[h * 16 + 3])), "r"(__float_as_uint(v[h * 16 + 4])), "r"(__float_as_uint(v[h * 16 + 5])),
        "r"(__float_as_uint(v[h * 16 + 6])), "r"(__float_as_uint(v[h * 16 + 7])), "r"(__float_as_uint(v[h * 16 + 8])),
        "r"(__float_as_uint(v[h * 16 + 9])), "r"(__float_as_uint(v[h * 16 + 10])), "r"(__float_as_uint(v[h * 16 + 11])),
        "r"(__float_as_uint(v[h * 16 + 12])), "r"(__float_as_uint(v[h * 16 + 13])), "r"(__float_as_uint(v[h * 16 + 14])),
        "r"(__float_as_uint(v[h * 16 + 15]))
        : "memory");
  }
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void ft_ld_main(uint32_t taddr, float (&v)[32]) {
  uint32_t w[32];
  __syncwarp();
  tc_ld32(taddr, w);
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(w[i]);
}
__device__ __forceinline__ void ft_ld_acc(uint32_t taddr, float (&v)[32]) {
  __syncwarp();
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    uint32_t vm[16], vc[16];
    ft_ld16x2(taddr + static_cast<uint32_t>(h * 16), vm, vc);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[h * 16 + i] = __uint_as_float(vm[i]) + __uint_as_float(vc[i]);
  }
}
// out[row0 + r][c0 + ..] = hi + lo (or the hi tile alone) for rows [4 it0, 4 it1) of the 32 rows x 32 columns block one
// epilogue warp wrote into the A tiles (rows 32 quarter .., swizzle block kb): 8 lanes read one row's 128 bytes, so every
// store instruction writes 4 full lines -- the thread = row layout of the accumulators touches 32 lines per instruction
template <bool kAddLo>
__device__ __forceinline__ void ft_store_block(const unsigned char* a_hi, const unsigned char* a_lo, int quarter, int kb,
                                               float* out, int ld, int row0, int c0, int rows_valid, int it0, int it1) {
  const int lane = threadIdx.x & 31;
  const int j = lane & 7;
  for (int it = it0; it < it1; ++it) {
    const int r = quarter * 32 + it * 4 + (lane >> 3);
    const uint32_t o = static_cast<uint32_t>(kb * 16384 + r * 128 + j * 16);
    float4 h = *reinterpret_cast<const float4*>(a_hi + o);
    if (kAddLo) {
      const float4 l = *reinterpret_cast<const float4*>(a_lo + o);
      h.x += l.x; h.y += l.y; h.z += l.z; h.w += l.w;
    }
    if (row0 + r < rows_valid) *reinterpret_cast<float4*>(out + static_cast<size_t>(row0 + r) * ld + c0 + 4 * (j ^ (r & 7))) = h;
  }
}
// d gelu_tanh(x) / dx through the sigmoid form (encoder_common.cuh gelu_tanh_fast): s = sigmoid(2u), g' = s + x s (1 - s) 2u'
__device__ __forceinline__ float gelu_tanh_grad_fast(float x) {
  const float c = 0.7978845608028654f;
  const float x2 = x * x;
  const float t = -2.f * c * 1.4426950408889634f * (x + 0.044715f * x * x2);
  const float sg = __fdividef(1.f, 1.f + exp2f(t));
  return fmaf(x * sg * (1.f - sg), 2.f * c * fmaf(3.f * 0.044715f, x2, 1.f), sg);
}

// keep bits of elements e .. e + 31 (e % 4 == 0) of dropout stream sid: bit i set = element e + i is kept
__device__ __forceinline__ uint32_t ft_keep32(const Drop& drop, uint32_t sid, uint64_t e) {
  uint32_t bits = 0xffffffffu;
  if (drop.on()) {
    bits = 0u;
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      const float4 m = drop.mul4(sid, e + i);
      bits |= (m.x != 0.f ? 1u : 0u) << i | (m.y != 0.f ? 2u : 0u) << i | (m.z != 0.f ? 4u : 0u) << i | (m.w != 0.f ? 8u : 0u) << i;
    }
  }
  return bits;
}

__global__ void __cluster_dims__(kFtCluster, 1, 1) __launch_bounds__(kFtThreads, 1)
tail_fused_tc_kernel(const __grid_constant__ CUtensorMap map_ctx, const __grid_constant__ CUtensorMap map_wo,
                     const __grid_constant__ CUtensorMap map_w1, const __grid_constant__ CUtensorMap map_w2,
                     const FtParams P) {
  pdl_trigger();                                    // the loss kernel behind this one may be scheduled
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* a_hi = smem;
  unsigned char* a_lo = smem + kFtABytes;
  unsigned char* bst = smem + 2 * kFtABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(bst + kFtStages * kFtStage);
  uint64_t* full = bars;                   // [3] weight chunk (hi + lo) landed
  uint64_t* empty = bars + 3;              // [3] its MMAs have read it
  uint64_t* a_ready = bars + 6;            // [3] the A operand of phase p is in place (hi / lo): TMA for p = 0, epilogues after
  uint64_t* acc_full = bars + 9;           // [3] phase p's accumulators are complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);
  // LayerNorm partial sums are exchanged through the head of the lo tile while no MMA reads it: [2][512] floats
  float* lnsc = reinterpret_cast<float*>(a_lo);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = static_cast<int>(ft_cluster_rank());
  const int r0 = (blockIdx.x / kFtCluster) * 128;
  const int d = 128, F = P.D.F;

  if (threadIdx.x == 0) {
    ft_mark(P, 0);
    for (int st = 0; st < kFtStages; ++st) {
      mbar_init(full + st, 1);
      mbar_init(empty + st, 1);
    }
    mbar_init(a_ready + 0, 1);
    mbar_init(a_ready + 1, kFtEpiWarps);
    mbar_init(a_ready + 2, kFtEpiWarps);
    for (int p = 0; p < 3; ++p) mbar_init(acc_full + p, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) ft_mark(P, 1);

  if (warp == 0) {
    // ===== TMA producer: the ctx tile, then the 12 weight chunks of the three phases; hi rows, lo rows `rows` further =====
    if (lane == 0) {
      for (int c = 0; c < 12; ++c) {
        if (c == kFtStages) {
          // the first weight chunks are in flight; the ctx rows come from the kernel before this one in the stream
          // (programmatic dependent launch: wait for it to have finished only now)
          pdl_wait();
          mbar_expect_tx(a_ready + 0, 2 * kFtABytes);
          for (int kb = 0; kb < 4; ++kb) {
            tma_load_2d(a_hi + kb * 16384, &map_ctx, kb * 32, r0, a_ready + 0);
            tma_load_2d(a_lo + kb * 16384, &map_ctx, kb * 32, P.SC + r0, a_ready + 0);
          }
        }
        const int st = c % kFtStages;
        const uint32_t ph = (c / kFtStages) & 1;
        mbar_wait(empty + st, ph ^ 1);
        mbar_expect_tx(full + st, 2 * kFtBBytes);
        unsigned char* dst = bst + st * kFtStage;
        const int p = c >> 2, kc = c & 3;
        if (p == 0) {
          tma_load_2d(dst, &map_wo, kc * 32, 0, full + st);
          tma_load_2d(dst + kFtBBytes, &map_wo, kc * 32, d, full + st);
        } else if (p == 1) {
          tma_load_2d(dst, &map_w1, kc * 32, q * 128, full + st);
          tma_load_2d(dst + kFtBBytes, &map_w1, kc * 32, F + q * 128, full + st);
        } else {
          tma_load_2d(dst, &map_w2, q * 128 + kc * 32, 0, full + st);
          tma_load_2d(dst + kFtBBytes, &map_w2, q * 128 + kc * 32, d, full + st);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    const uint32_t leader = g3_elect_one();
    const uint32_t a_hi_u = smem_u32(a_hi), a_lo_u = smem_u32(a_lo);
    for (int p = 0; p < 3; ++p) {
      mbar_wait(a_ready + p, 0);
      tc_fence_after();
      if (lane == 0) ft_mark(P, 3 + 4 * p);
      const uint32_t t_main = tmem_base + (p == 1 ? 256u : 0u), t_corr = t_main + 128u;
      for (int kc = 0; kc < 4; ++kc) {
        const int c = p * 4 + kc;
        const int st = c % kFtStages;
        const uint32_t ph = (c / kFtStages) & 1;
        mbar_wait(full + st, ph);
        tc_fence_after();
        if (lane == 0 && kc == 0) ft_mark(P, 4 + 4 * p);
        const uint32_t bbase = smem_u32(bst + st * kFtStage);
        const uint64_t ah = umma_desc(a_hi_u + kc * 16384), al = umma_desc(a_lo_u + kc * 16384);
        const uint64_t bh = umma_desc(bbase), bl = umma_desc(bbase + kFtBBytes);
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
          const uint64_t o = static_cast<uint64_t>(k4 * 2);
          const uint32_t acc = (kc | k4) != 0 ? 1u : 0u;
          g3_mma_tf32_if(leader, t_main, ah + o, bh + o, kFtIdesc, acc);
          g3_mma_tf32_if(leader, t_corr, al + o, bh + o, kFtIdesc, acc);
          g3_mma_tf32_if(leader, t_corr, ah + o, bl + o, kFtIdesc, 1u);
        }
        g3_commit_if(leader, empty + st);
      }
      g3_commit_if(leader, acc_full + p);
      if (lane == 0) ft_mark(P, 5 + 4 * p);
    }
  } else {
    // ===== epilogue warps: thread = (row of the tile, 32 columns) =====
    const int e = warp - 2;
    const int quarter = warp & 3;                           // TMEM lanes 32 * (warp % 4) .. + 31
    const int cg = e >> 2;
    const int c0 = cg * 32;                                 // first column
    const int rl = quarter * 32 + lane;                     // row inside the tile
    const int row = r0 + rl;
    const bool live = row < P.SC;
    const bool mine = (lane >> 3) == q && live;             // this CTA stores y / n for rows 8 q .. 8 q + 7 of every quarter
    const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(c0);
    const Drop drop = make_drop(P.seed_dev, P.D.thr, P.D.keep);
    const size_t base = static_cast<size_t>(row) * d + c0;
    const size_t fbase = static_cast<size_t>(row) * F + q * 128 + c0;
    // ---- before the first accumulator exists: everything epilogue 1 needs that does not depend on it
    //      y = m (acc + bo) + x = m acc + (m bo + x)
    float cst[32];
    const uint32_t keep2 = ft_keep32(drop, 2u, base);
    {
      const int rs = live ? row : P.SC - 1;                 // rows past the end compute on a valid row, store nothing
      const float* xr = P.xo + static_cast<size_t>(rs / P.D.C) * d + c0;
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        const float4 b = *reinterpret_cast<const float4*>(P.bo + c0 + i);
        const float4 x = *reinterpret_cast<const float4*>(xr + i);
        cst[i] = fmaf((keep2 >> i) & 1u ? drop.scale : 0.f, b.x, x.x);
        cst[i + 1] = fmaf((keep2 >> (i + 1)) & 1u ? drop.scale : 0.f, b.y, x.y);
        cst[i + 2] = fmaf((keep2 >> (i + 2)) & 1u ? drop.scale : 0.f, b.z, x.z);
        cst[i + 3] = fmaf((keep2 >> (i + 3)) & 1u ? drop.scale : 0.f, b.w, x.w);
      }
    }
    // ---- epilogue 1: y = dropout_2(acc + bo) + x[o];  n = LN_ff(y)
    mbar_wait(acc_full + 0, 0);
    tc_fence_after();
    if (threadIdx.x == 64) ft_mark(P, 6);
    {
      float v[32];
      ft_ld_acc(t_addr, v);
      float s1 = 0.f;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        v[i] = fmaf((keep2 >> i) & 1u ? drop.scale : 0.f, v[i], cst[i]);
        s1 += v[i];
      }
      lnsc[cg * 128 + rl] = s1;
      if (mine) {                                           // (the final step of this CTA re-reads these rows)
#pragma unroll
        for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(P.y + base + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
      }
      ft_epi_sync();
      const float mean = ((lnsc[rl] + lnsc[128 + rl]) + (lnsc[256 + rl] + lnsc[384 + rl])) / 128.f;
      float s2 = 0.f;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float a = v[i] - mean;
        s2 = fmaf(a, a, s2);
      }
      lnsc[512 + cg * 128 + rl] = s2;
      ft_epi_sync();
      const float var = ((lnsc[512 + rl] + lnsc[640 + rl]) + (lnsc[768 + rl] + lnsc[896 + rl])) / 128.f;
      const RowStats st{mean, 1.f / sqrtf(var + P.D.eps)};
      ft_epi_sync();                                        // the scratch lives inside the tile written next
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        const float4 nv = ln_apply(make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]), st,
                                   *reinterpret_cast<const float4*>(P.ln_ff_g + c0 + i),
                                   *reinterpret_cast<const float4*>(P.ln_ff_b + c0 + i));
        ft_store_a(a_hi, a_lo, rl, (c0 + i) >> 2, nv);
      }
    }
    tc_fence_before();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) mbar_arrive(a_ready + 1);
    // off the critical path (the phase-2 MMAs only read the tiles): n = hi + lo, row-contiguous
    ft_store_block<true>(a_hi, a_lo, quarter, cg, P.n, d, r0, c0, P.SC, 2 * q, 2 * q + 2);
    // ---- epilogue 2: pre1 = acc + b1;  h1 = dropout_3(gelu(pre1)) for this CTA's 128 hidden columns
    const uint32_t keep3 = ft_keep32(drop, 3u, fbase);
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      const float4 b = *reinterpret_cast<const float4*>(P.b1 + q * 128 + c0 + i);
      cst[i] = b.x; cst[i + 1] = b.y; cst[i + 2] = b.z; cst[i + 3] = b.w;
    }
    mbar_wait(acc_full + 1, 0);
    tc_fence_after();
    if (threadIdx.x == 64) ft_mark(P, 10);
    {
      float v[32];
      ft_ld_acc(t_addr + 256u, v);
      const float sc = drop.on() ? drop.scale : 1.f;
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        float hv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float x = v[i + u] + cst[i + u];
          const float m = (keep3 >> (i + u)) & 1u ? sc : 0.f;
          float dg;
          hv[u] = gelu_tanh_fast_both(x, &dg) * m;
          v[i + u] = P.save_dact ? dg * m : x;
        }
        ft_store_a(a_hi, a_lo, rl, (c0 + i) >> 2, make_float4(hv[0], hv[1], hv[2], hv[3]));
      }
      // with the tensor-core backward the pre1 slot gets dropout_3 . gelu'(pre1): parked over the main accumulator
      if (P.save_dact) ft_st32(t_addr + 256u, v);
      tc_fence_before();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(a_ready + 2);
      // off the critical path, next to the phase-3 MMAs: h1 = hi + lo row-contiguous (pre1 follows at the very end)
      ft_store_block<true>(a_hi, a_lo, quarter, cg, P.h1, F, r0, q * 128 + c0, P.SC, 0, 8);
    }
    // ---- epilogue 3: this CTA's partial sums of the FFN's second product -> shared memory, [chunk][row] float4
    mbar_wait(acc_full + 2, 0);
    tc_fence_after();
    if (threadIdx.x == 64) ft_mark(P, 14);
    {
      float v[32];
      ft_ld_acc(t_addr, v);
      ft_epi_sync();                                        // every warp has stored its h1 block from the tiles
      float4* redbuf = reinterpret_cast<float4*>(a_hi);     // the phase-3 MMAs have read the A tiles: reuse
#pragma unroll
      for (int i = 0; i < 32; i += 4)                        // [row][32 chunks], chunk ^ row: rows and chunks both conflict-free
        redbuf[rl * 32 + ((((c0 + i) >> 2) ^ rl) & 31)] = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
    }
    tc_fence_before();
  }
  // ---- CTA q finishes rows [32 q, 32 q + 32): epilogue warp e takes rows 2 e and 2 e + 1, lane = 4 columns (row-contiguous
  //      loads and stores, LayerNorm sums by warp shuffle); what does not depend on the partial tiles is fetched first.
  //      Rows 8 q .. 8 q + 7 of every quarter: the rows whose y this CTA stored itself
  const int fe = warp - 2;
  float4 yv[2], b2v, gv, bv, fm[2];
  bool fok[2];
  if (warp >= 2) {
    const Drop drop = make_drop(P.seed_dev, P.D.thr, P.D.keep);
    b2v = *reinterpret_cast<const float4*>(P.b2 + lane * 4);
    gv = *reinterpret_cast<const float4*>(P.ln_out_g + lane * 4);
    bv = *reinterpret_cast<const float4*>(P.ln_out_b + lane * 4);
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int fk = fe * 2 + i;
      const int frow = r0 + (fk >> 3) * 32 + q * 8 + (fk & 7);
      fok[i] = frow < P.SC;
      const size_t fb = static_cast<size_t>(frow) * d + lane * 4;
      yv[i] = fok[i] ? *reinterpret_cast<const float4*>(P.y + fb) : zero4();   // written by this CTA in epilogue 1
      fm[i] = drop.on() ? drop.mul4(4u, fb) : make_float4(1.f, 1.f, 1.f, 1.f);
    }
  }
  // every CTA's partial tile is in its shared memory
  ft_cluster_sync();
  if (threadIdx.x == 64) ft_mark(P, 15);
  if (warp >= 2) {
    const uint32_t red_u = smem_u32(a_hi);
    float4 pz[2][kFtCluster];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int fk = fe * 2 + i;
      const int frl = (fk >> 3) * 32 + q * 8 + (fk & 7);
      const uint32_t addr = red_u + static_cast<uint32_t>((frl * 32 + ((lane ^ frl) & 31)) * 16);
#pragma unroll
      for (uint32_t src = 0; src < kFtCluster; ++src) pz[i][src] = ft_ld_peer4(addr, src);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int fk = fe * 2 + i;
      const size_t fb = static_cast<size_t>(r0 + (fk >> 3) * 32 + q * 8 + (fk & 7)) * d + lane * 4;
      float4 a = pz[i][0];
#pragma unroll
      for (uint32_t src = 1; src < kFtCluster; ++src) {
        a.x += pz[i][src].x; a.y += pz[i][src].y; a.z += pz[i][src].z; a.w += pz[i][src].w;
      }
      a.x = fmaf(a.x + b2v.x, fm[i].x, yv[i].x);
      a.y = fmaf(a.y + b2v.y, fm[i].y, yv[i].y);
      a.z = fmaf(a.z + b2v.z, fm[i].z, yv[i].z);
      a.w = fmaf(a.w + b2v.w, fm[i].w, yv[i].w);
      if (fok[i]) *reinterpret_cast<float4*>(P.z + fb) = a;
      const RowStats st = row_stats(a, true, d, P.D.eps);
      if (fok[i]) *reinterpret_cast<float4*>(P.out + fb) = ln_apply(a, st, gv, bv);
    }
  }
  // ---- pre1 = acc2 + b1, the last saved tensor: the phase-2 accumulators are still in TMEM; staged through the (dead) lo
  //      tile in the A layout so that the stores are row-contiguous like h1's.  With the tensor-core backward
  //      (save_dact) the slot holds dropout_3 . gelu'(pre1) instead: all the backward pass ever forms from pre1.
  if (warp >= 2) {
    const int e = warp - 2, quarter = warp & 3, cg = e >> 2, c0 = cg * 32;
    const int rl = quarter * 32 + lane;
    float v[32];
    tc_fence_after();
    const uint32_t ta = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + 256u + static_cast<uint32_t>(c0);
    if (P.save_dact) ft_ld_main(ta, v);
    else ft_ld_acc(ta, v);
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      float4 w = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
      if (!P.save_dact) {
        const float4 b = *reinterpret_cast<const float4*>(P.b1 + q * 128 + c0 + i);
        w.x += b.x; w.y += b.y; w.z += b.z; w.w += b.w;
      }
      *reinterpret_cast<float4*>(a_lo + ft_a_off(rl, (c0 + i) >> 2)) = w;
    }
    __syncwarp();
    ft_store_block<false>(a_lo, a_lo, quarter, cg, P.pre1, F, r0, q * 128 + c0, P.SC, 0, 8);
    tc_fence_before();
  }
  // nobody leaves while a peer may still read its partial tile
  if (threadIdx.x == 64) ft_mark(P, 16);
  ft_cluster_sync();
  if (threadIdx.x == 64) ft_mark(P, 17);
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512));
  }
}

// PSB_FT_TRACE=1: a 64-slot device buffer CTA 0 of the fused tail kernels stamps with %globaltimer (forward: slots 0..31,
// backward: 32..63; read back by psb_debug_tail_trace)
unsigned long long* ft_trace_buffer() {
  static unsigned long long* buf = nullptr;
  static int state = -1;
  if (state < 0) {
    const char* e = getenv("PSB_FT_TRACE");
    state = (e != nullptr && atoi(e) != 0) ? 1 : 0;
    if (state == 1 && (cudaMalloc(&buf, 64 * sizeof(unsigned long long)) != cudaSuccess ||
                       cudaMemset(buf, 0, 64 * sizeof(unsigned long long)) != cudaSuccess)) {
      buf = nullptr;
    }
  }
  return buf;
}

bool tail_fused_supported(const TailTcArgs& a) {
  const Dims& D = a.D;
  if (D.d != 128 || D.F != 128 * kFtCluster || D.S * D.C <= 0) return false;
  if (a.P == nullptr || a.nact == nullptr || a.off == nullptr || a.tok == nullptr) return false;
  const float* ptrs[] = {a.kv, a.xo, a.wo, a.bo, a.w1, a.b1, a.w2, a.b2, a.ln_ff_g, a.ln_ff_b, a.ln_out_g, a.ln_out_b,
                         a.ctx, a.y, a.n, a.z, a.pre1, a.h1, a.out, a.wo_hl, a.w1_hl, a.w2_hl, a.ctx_hl};
  for (const float* q : ptrs)
    if (q == nullptr || misaligned16(q)) return false;
  return true;
}

int launch_tail_fwd_fused(const TailTcArgs& a, cudaStream_t s) {
  if (!tail_fused_supported(a)) return PSB_E_UNSUPPORTED;
  const Dims& D = a.D;
  const int SC = D.S * D.C, d = D.d, F = D.F;
  int st;
  static DeviceAttr attr_done;
  if (attr_done.need()) {
    cudaError_t e = cudaFuncSetAttribute(tail_fused_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(kFtSmem));
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_done.done();
  }
  PSB_PROF("tail_ctx_kernel", s);
  {
    const cudaError_t le = launch_pdl(tail_ctx_kernel, dim3((SC + 7) / 8), dim3(256), 0, s, D, a.nact, a.off, a.tok, a.P, a.kv,
                                      a.ctx, a.seed_dev, a.ctx_hl);
    if (le != cudaSuccess) return static_cast<int>(le);
  }
  if ((st = launch_status()) != PSB_OK) return st;
  // hi rows stacked on lo rows: one map per operand, the lo tile `rows` further down
  alignas(64) CUtensorMap map_ctx, map_wo, map_w1, map_w2;
  if ((st = g3_make_map(&map_ctx, a.ctx_hl, 2 * static_cast<int64_t>(SC), d, d, 128)) != PSB_OK) return st;
  if ((st = g3_make_map(&map_wo, a.wo_hl, 2 * d, d, d, 128)) != PSB_OK) return st;
  if ((st = g3_make_map(&map_w1, a.w1_hl, 2 * F, d, d, 128)) != PSB_OK) return st;
  if ((st = g3_make_map(&map_w2, a.w2_hl, 2 * d, F, F, 128)) != PSB_OK) return st;
  FtParams P;
  P.D = D;
  P.SC = SC;
  P.xo = a.xo; P.bo = a.bo; P.b1 = a.b1; P.b2 = a.b2;
  P.ln_ff_g = a.ln_ff_g; P.ln_ff_b = a.ln_ff_b; P.ln_out_g = a.ln_out_g; P.ln_out_b = a.ln_out_b;
  P.y = a.y; P.n = a.n; P.z = a.z; P.pre1 = a.pre1; P.h1 = a.h1; P.out = a.out;
  P.seed_dev = a.seed_dev;
  P.trace = ft_trace_buffer();
  P.save_dact = a.save_dact;
  const unsigned tiles = static_cast<unsigned>((SC + 127) / 128);
  PSB_PROF("tail_fused_tc_kernel", s);
  {
    const cudaError_t le = launch_pdl(tail_fused_tc_kernel, dim3(tiles * kFtCluster), dim3(kFtThreads), kFtSmem, s, map_ctx,
                                      map_wo, map_w1, map_w2, P);
    if (le != cudaSuccess) return static_cast<int>(le);
  }
  return launch_status();
}


// ------------------------------------------------------------------ backward tail as ONE cluster kernel
// encoder_bwd.cu tail_bwd_kernel steps (1)..(6) on tcgen05, TRANSPOSED: the weights are the M operand (128 output
// features = TMEM lanes) and the tile's 128 copy rows the N operand (TMEM columns), so a thread of the epilogue owns one
// feature for 32 rows and every global load / store of the epilogues runs along a row (coalesced), and the activation
// tiles it writes for the next product are conflict-free 4-byte stores.
//
//   cluster = one tile of 128 copy rows; CTA q owns hidden columns [128 q, 128 q + 128) and finishes rows 8 e + 2 q + {0, 1}
//   prologue  gz = LN_out'(gout; z), g_h2 = dropout_4 gz (saved for dW2)                         -> N operand of product 1
//   product 1 g_h1^T[f, m] = W2^T[f, :] . g_h2[m, :]   (this CTA's 128 hidden columns f)
//   epilogue  g_pre = g_h1 * gelu'(pre1) * dropout_3 (saved for dW1)                             -> N operand of product 2
//   product 2 gn^T[i, m] (partial) = W1^T[i, 128 q ..] . g_pre[m, :]
//   reduce    the four partial tiles through distributed shared memory, CTA order 0..3; for its 32 rows the CTA forms
//             gy = gz + LN_ff'(gn; y) (-> global, for the attention backward), g_o1 = dropout_2 gy (saved for dWo)
//   product 3 g_ctx^T[k, m] = Wo^T[k, :] . g_o1[m, :] for those 32 rows only (N = 32: no gather of the rows needed)
//   LayerNorm parameter partials: one row of lnp per CTA, summed by the backward's reduce kernel.
struct FbParams {
  Dims D;
  int SC;
  const float *z, *gout, *y, *pre1, *ln_out_g, *ln_ff_g;
  float *g_h2, *g_pre, *g_o1, *gy, *g_ctx, *lnp;
  const uint64_t* seed_dev;
  unsigned long long* trace;   // PSB_FT_TRACE=1 (slots 32..63 of the trace buffer)
};
__device__ __forceinline__ void fb_mark(const FbParams& P, int slot) {
  if (P.trace != nullptr && blockIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    P.trace[32 + slot] = t;
  }
}
constexpr uint32_t kFbIdesc32 = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(32 >> 3) << 17) |
                                (static_cast<uint32_t>(128 >> 4) << 24);          // as kFtIdesc with N = 32

// one element (row m of the tile, K index k) of a K-major 128-byte-swizzled tile of `rows_per_block` rows per 32-float block
__device__ __forceinline__ uint32_t fb_elem_off(int m, int k, int block_bytes) {
  return static_cast<uint32_t>((k >> 5) * block_bytes + m * 128 + ((((k & 31) >> 2) ^ (m & 7)) << 4) + (k & 3) * 4);
}
__device__ __forceinline__ void fb_ld8x2(uint32_t taddr, uint32_t (&v)[8], uint32_t (&w)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
               : "r"(taddr + 128u));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__global__ void __cluster_dims__(kFtCluster, 1, 1) __launch_bounds__(kFtThreads, 1)
tail_bwd_fused_tc_kernel(const __grid_constant__ CUtensorMap map_w2t, const __grid_constant__ CUtensorMap map_w1t,
                         const __grid_constant__ CUtensorMap map_wot, const FbParams P) {
  pdl_trigger();                                    // tail_attn_bwd_kernel may start staging its K | V rows
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* t_hi = smem;                       // activation tile (N operand), hi / lo
  unsigned char* t_lo = smem + kFtABytes;
  unsigned char* wst = smem + 2 * kFtABytes;        // weight chunk stages (M operand), hi + lo each
  uint64_t* bars = reinterpret_cast<uint64_t*>(wst + kFtStages * kFtStage);
  uint64_t* full = bars;
  uint64_t* empty = bars + 3;
  uint64_t* a_ready = bars + 6;                     // [3] the activation tile of product p is in place
  uint64_t* acc_full = bars + 9;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = static_cast<int>(ft_cluster_rank());
  const int tile = blockIdx.x / kFtCluster;
  const int r0 = tile * 128;
  const int d = 128, F = P.D.F;

  if (threadIdx.x == 0) {
    fb_mark(P, 0);
    for (int st = 0; st < kFtStages; ++st) {
      mbar_init(full + st, 1);
      mbar_init(empty + st, 1);
    }
    for (int p = 0; p < 3; ++p) {
      mbar_init(a_ready + p, kFtEpiWarps);
      mbar_init(acc_full + p, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // LayerNorm parameter partials of this CTA's rows, per lane (4 columns): ln_out gamma / beta, ln_ff gamma / beta
  float4 pg_out = zero4(), pb_out = zero4(), pg_ff = zero4(), pb_ff = zero4();

  // Product 3 runs AFTER the reduce, so the TMA and MMA warps cannot wait at the cluster barrier in between: they arrive
  // for it at once (they never touch a peer's memory) and collect the phase when their loops are done.
  if (warp < 2) asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  if (warp == 0) {
    // ===== TMA producer: the 12 weight chunks of the three products; hi rows, lo rows `rows` further =====
    if (lane == 0) {
      for (int c = 0; c < 12; ++c) {
        const int st = c % kFtStages;
        const uint32_t ph = (c / kFtStages) & 1;
        mbar_wait(empty + st, ph ^ 1);
        mbar_expect_tx(full + st, 2 * kFtBBytes);
        unsigned char* dst = wst + st * kFtStage;
        const int p = c >> 2, kc = c & 3;
        if (p == 0) {                                       // W2^T [F][d]: rows 128 q .., K = j
          tma_load_2d(dst, &map_w2t, kc * 32, q * 128, full + st);
          tma_load_2d(dst + kFtBBytes, &map_w2t, kc * 32, F + q * 128, full + st);
        } else if (p == 1) {                                // W1^T [d][F]: all rows, K = hidden columns 128 q ..
          tma_load_2d(dst, &map_w1t, q * 128 + kc * 32, 0, full + st);
          tma_load_2d(dst + kFtBBytes, &map_w1t, q * 128 + kc * 32, d, full + st);
        } else {                                            // Wo^T [d][d]
          tma_load_2d(dst, &map_wot, kc * 32, 0, full + st);
          tma_load_2d(dst + kFtBBytes, &map_wot, kc * 32, d, full + st);
        }
      }
    }
    __syncwarp();
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  } else if (warp == 1) {
    // ===== MMA issuer: D[feature, row] += W chunk (M operand) . tile chunk (N operand) =====
    const uint32_t leader = g3_elect_one();
    const uint32_t t_hi_u = smem_u32(t_hi), t_lo_u = smem_u32(t_lo);
    for (int p = 0; p < 3; ++p) {
      mbar_wait(a_ready + p, 0);
      tc_fence_after();
      const uint32_t t_main = tmem_base + (p == 1 ? 256u : 0u), t_corr = t_main + 128u;
      const uint32_t idesc = p == 2 ? kFbIdesc32 : kFtIdesc;
      // product 3: the 32-row tile sits in the lo tile's memory, 4 KB per K block, hi then lo
      const uint32_t nb_hi = p == 2 ? t_lo_u : t_hi_u, nb_lo = p == 2 ? t_lo_u + 16384u : t_lo_u;
      const uint32_t nblk = p == 2 ? 4096u : 16384u;
      for (int kc = 0; kc < 4; ++kc) {
        const int c = p * 4 + kc;
        const int st = c % kFtStages;
        const uint32_t ph = (c / kFtStages) & 1;
        mbar_wait(full + st, ph);
        tc_fence_after();
        const uint32_t wbase = smem_u32(wst + st * kFtStage);
        const uint64_t wh = umma_desc(wbase), wl = umma_desc(wbase + kFtBBytes);
        const uint64_t nh = umma_desc(nb_hi + kc * nblk), nl = umma_desc(nb_lo + kc * nblk);
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
          const uint64_t o = static_cast<uint64_t>(k4 * 2);
          const uint32_t acc = (kc | k4) != 0 ? 1u : 0u;
          g3_mma_tf32_if(leader, t_main, wh + o, nh + o, idesc, acc);
          g3_mma_tf32_if(leader, t_corr, wl + o, nh + o, idesc, acc);
          g3_mma_tf32_if(leader, t_corr, wh + o, nl + o, idesc, 1u);
        }
        g3_commit_if(leader, empty + st);
      }
      g3_commit_if(leader, acc_full + p);
    }
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  } else {
    // ===== the 16 epilogue warps =====
    const int e = warp - 2;
    const int quarter = warp & 3;                           // TMEM lanes 32 * (warp % 4) .. + 31
    const int cg = e >> 2;
    const int f = quarter * 32 + lane;                      // the feature (TMEM lane) of this thread in the epilogues
    const Drop drop = make_drop(P.seed_dev, P.D.thr, P.D.keep);
    const float dscale = drop.on() ? drop.scale : 1.f;
    // ---- prologue, warp per row (lane = 4 columns): rows 8 e .. 8 e + 7 of the tile, four at a time
    {
      const float4 g = *reinterpret_cast<const float4*>(P.ln_out_g + lane * 4);
#pragma unroll
      for (int b4 = 0; b4 < 2; ++b4) {
        float4 z[4], go[4], gz[4], zh[4], mk[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = r0 + e * 8 + b4 * 4 + i;
          const size_t base = static_cast<size_t>(row) * d + lane * 4;
          z[i] = row < P.SC ? *reinterpret_cast<const float4*>(P.z + base) : zero4();
          go[i] = row < P.SC ? *reinterpret_cast<const float4*>(P.gout + base) : zero4();
          mk[i] = drop.on() ? drop.mul4(4u, base) : make_float4(1.f, 1.f, 1.f, 1.f);
        }
        ln_bwd_rows<4>(z, go, g, d, P.D.eps, gz, zh);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int rr = b4 * 4 + i, r = e * 8 + rr, row = r0 + r;
          const size_t base = static_cast<size_t>(row) * d + lane * 4;
          const float4 gh2 = make_float4(gz[i].x * mk[i].x, gz[i].y * mk[i].y, gz[i].z * mk[i].z, gz[i].w * mk[i].w);
          ft_store_a(t_hi, t_lo, r, lane, gh2);
          if ((rr >> 1) == q && row < P.SC) {               // this CTA's rows: saved operand, gz parked in gy, LN partials
            *reinterpret_cast<float4*>(P.g_h2 + base) = gh2;
            *reinterpret_cast<float4*>(P.gy + base) = gz[i];
            pg_out.x += go[i].x * zh[i].x; pg_out.y += go[i].y * zh[i].y; pg_out.z += go[i].z * zh[i].z; pg_out.w += go[i].w * zh[i].w;
            pb_out.x += go[i].x; pb_out.y += go[i].y; pb_out.z += go[i].z; pb_out.w += go[i].w;
          }
        }
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) mbar_arrive(a_ready + 0);
    if (threadIdx.x == 64) fb_mark(P, 1);
    // ---- epilogue 1: thread = hidden column f (of this CTA's 128), rows m = 32 cg .. + 31
    {
      float pre[32];                                        // dropout_3 . gelu'(pre1), saved by the forward kernel
      const size_t col = static_cast<size_t>(q) * 128 + f;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int row = r0 + cg * 32 + i;
        pre[i] = row < P.SC ? P.pre1[static_cast<size_t>(row) * F + col] : 0.f;
      }
      if (threadIdx.x == 64) fb_mark(P, 2);
      mbar_wait(acc_full + 0, 0);
      tc_fence_after();
      if (threadIdx.x == 64) fb_mark(P, 3);
      float v[32];
      ft_ld_acc(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(cg * 32), v);
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int m = cg * 32 + i;
        const float gp = v[i] * pre[i];
        const float hi = __uint_as_float(__float_as_uint(gp) & 0xFFFFE000u);
        const uint32_t o = fb_elem_off(m, f, 16384);
        *reinterpret_cast<float*>(t_hi + o) = hi;
        *reinterpret_cast<float*>(t_lo + o) = gp - hi;
        v[i] = gp;
      }
      tc_fence_before();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(a_ready + 1);
      if (threadIdx.x == 64) fb_mark(P, 4);
#pragma unroll
      for (int i = 0; i < 32; ++i) {                        // off the critical path: the saved operand of dW1
        const int row = r0 + cg * 32 + i;
        if (row < P.SC) P.g_pre[static_cast<size_t>(row) * F + col] = v[i];
      }
    }
    // ---- epilogue 2: partial gn^T[i = f, m] -> shared memory as [m][i] (row-contiguous for the reduce)
    if (threadIdx.x == 64) fb_mark(P, 5);
    mbar_wait(acc_full + 1, 0);
    tc_fence_after();
    if (threadIdx.x == 64) fb_mark(P, 6);
    {
      float v[32];
      ft_ld_acc(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + 256u + static_cast<uint32_t>(cg * 32), v);
      float* redbuf = reinterpret_cast<float*>(t_hi);       // the product-2 MMAs have read the tiles
#pragma unroll
      for (int i = 0; i < 32; ++i) redbuf[(cg * 32 + i) * 128 + f] = v[i];
    }
    tc_fence_before();
  }
  // ---- this CTA's rows: r = 8 e + 2 q + i; what does not depend on the partial tiles first
  const int fe = warp - 2;
  float4 yv[2], gzv[2], m2[2], gff;
  bool fok[2];
  if (warp >= 2) {
    const Drop drop = make_drop(P.seed_dev, P.D.thr, P.D.keep);
    gff = *reinterpret_cast<const float4*>(P.ln_ff_g + lane * 4);
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int row = r0 + fe * 8 + 2 * q + i;
      fok[i] = row < P.SC;
      const size_t base = static_cast<size_t>(row) * d + lane * 4;
      yv[i] = fok[i] ? *reinterpret_cast<const float4*>(P.y + base) : zero4();
      gzv[i] = fok[i] ? *reinterpret_cast<const float4*>(P.gy + base) : zero4();    // parked by this warp in the prologue
      m2[i] = drop.on() ? drop.mul4(2u, base) : make_float4(1.f, 1.f, 1.f, 1.f);
    }
    if (threadIdx.x == 64) fb_mark(P, 7);
    ft_cluster_sync();                                      // every CTA's partial tile is in its shared memory
    if (threadIdx.x == 64) fb_mark(P, 8);
  }
  if (warp >= 2) {
    const uint32_t red_u = smem_u32(t_hi);
    float4 pz[2][kFtCluster];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const uint32_t addr = red_u + static_cast<uint32_t>(((fe * 8 + 2 * q + i) * 128 + lane * 4) * 4);
#pragma unroll
      for (uint32_t src = 0; src < kFtCluster; ++src) pz[i][src] = ft_ld_peer4(addr, src);
    }
    float4 gn[2], gl[2], yh[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      gn[i] = pz[i][0];
#pragma unroll
      for (uint32_t src = 1; src < kFtCluster; ++src) {
        gn[i].x += pz[i][src].x; gn[i].y += pz[i][src].y; gn[i].z += pz[i][src].z; gn[i].w += pz[i][src].w;
      }
    }
    ln_bwd_rows<2>(yv, gn, gff, d, P.D.eps, gl, yh);
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int li = fe * 2 + i;                            // row of the 32-row tile of product 3
      const size_t base = static_cast<size_t>(r0 + fe * 8 + 2 * q + i) * d + lane * 4;
      float4 go1 = zero4();
      if (fok[i]) {
        pg_ff.x += gn[i].x * yh[i].x; pg_ff.y += gn[i].y * yh[i].y; pg_ff.z += gn[i].z * yh[i].z; pg_ff.w += gn[i].w * yh[i].w;
        pb_ff.x += gn[i].x; pb_ff.y += gn[i].y; pb_ff.z += gn[i].z; pb_ff.w += gn[i].w;
        const float4 gy = make_float4(gzv[i].x + gl[i].x, gzv[i].y + gl[i].y, gzv[i].z + gl[i].z, gzv[i].w + gl[i].w);
        go1 = make_float4(gy.x * m2[i].x, gy.y * m2[i].y, gy.z * m2[i].z, gy.w * m2[i].w);
        *reinterpret_cast<float4*>(P.gy + base) = gy;
        *reinterpret_cast<float4*>(P.g_o1 + base) = go1;
      }
      float4 hi, lo;
      g3_split(go1, hi, lo);
      const uint32_t o = static_cast<uint32_t>((lane >> 3) * 4096 + li * 128 + (((lane & 7) ^ (li & 7)) << 4));
      *reinterpret_cast<float4*>(t_lo + o) = hi;            // 32-row tile: 4 KB per K block, hi then lo (the lo tile is dead)
      *reinterpret_cast<float4*>(t_lo + 16384 + o) = lo;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) mbar_arrive(a_ready + 2);
    if (threadIdx.x == 64) fb_mark(P, 9);
    // LayerNorm parameter partials: per-warp sums -> [16][4][128] floats in the upper half of the lo tile
    float* sc = reinterpret_cast<float*>(t_lo + 32768);
    *reinterpret_cast<float4*>(sc + (fe * 4 + 0) * 128 + lane * 4) = pg_out;
    *reinterpret_cast<float4*>(sc + (fe * 4 + 1) * 128 + lane * 4) = pb_out;
    *reinterpret_cast<float4*>(sc + (fe * 4 + 2) * 128 + lane * 4) = pg_ff;
    *reinterpret_cast<float4*>(sc + (fe * 4 + 3) * 128 + lane * 4) = pb_ff;
    ft_epi_sync();
    {
      const int t = threadIdx.x - 64;                       // 0..511 = (parameter, column)
      float acc = 0.f;
#pragma unroll
      for (int w = 0; w < kFtEpiWarps; ++w) acc += sc[w * 512 + t];
      P.lnp[(static_cast<size_t>(tile) * kFtCluster + q) * 4 * d + t] = acc;
    }
    // ---- epilogue 3: g_ctx^T[k, li]: thread = feature k, 8 of the 32 rows
    const int quarter = warp & 3, cg = fe >> 2;
    const int k = quarter * 32 + lane;
    if (threadIdx.x == 64) fb_mark(P, 10);
    mbar_wait(acc_full + 2, 0);
    tc_fence_after();
    if (threadIdx.x == 64) fb_mark(P, 11);
    uint32_t vm[8], vc[8];
    __syncwarp();
    fb_ld8x2(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(cg * 8), vm, vc);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int li = cg * 8 + i;
      const int row = r0 + (li >> 1) * 8 + 2 * q + (li & 1);
      if (row < P.SC) P.g_ctx[static_cast<size_t>(row) * d + k] = __uint_as_float(vm[i]) + __uint_as_float(vc[i]);
    }
    tc_fence_before();
  }
  // nobody leaves while a peer may still read its partial tile
  if (threadIdx.x == 64) fb_mark(P, 12);
  ft_cluster_sync();
  if (threadIdx.x == 64) fb_mark(P, 13);
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512));
  }
}

int tail_bwd_fused_parts(const Dims& D) { return ((D.S * D.C + 127) / 128) * kFtCluster; }

bool tail_bwd_fused_supported(const TailBwdTcArgs& a) {
  const Dims& D = a.D;
  if (D.d != 128 || D.F != 128 * kFtCluster || D.S * D.C <= 0) return false;
  const float* ptrs[] = {a.z, a.gout, a.y, a.pre1, a.ln_out_g, a.ln_ff_g, a.wot_hl, a.w1t_hl, a.w2t_hl,
                         a.g_h2, a.g_pre, a.g_o1, a.gy, a.g_ctx, a.lnp};
  for (const float* p : ptrs)
    if (p == nullptr || misaligned16(p)) return false;
  return true;
}

int launch_tail_bwd_fused(const TailBwdTcArgs& a, cudaStream_t s) {
  if (!tail_bwd_fused_supported(a)) return PSB_E_UNSUPPORTED;
  const Dims& D = a.D;
  const int SC = D.S * D.C, d = D.d, F = D.F;
  int st;
  static DeviceAttr attr_done;
  if (attr_done.need()) {
    cudaError_t e = cudaFuncSetAttribute(tail_bwd_fused_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(kFtSmem));
    if (e != cudaSuccess) return static_cast<int>(e);
    attr_done.done();
  }
  alignas(64) CUtensorMap map_w2t, map_w1t, map_wot;
  if ((st = g3_make_map(&map_w2t, a.w2t_hl, 2 * F, d, d, 128)) != PSB_OK) return st;
  if ((st = g3_make_map(&map_w1t, a.w1t_hl, 2 * d, F, F, 128)) != PSB_OK) return st;
  if ((st = g3_make_map(&map_wot, a.wot_hl, 2 * d, d, d, 128)) != PSB_OK) return st;
  FbParams P;
  P.D = D;
  P.SC = SC;
  P.z = a.z; P.gout = a.gout; P.y = a.y; P.pre1 = a.pre1; P.ln_out_g = a.ln_out_g; P.ln_ff_g = a.ln_ff_g;
  P.g_h2 = a.g_h2; P.g_pre = a.g_pre; P.g_o1 = a.g_o1; P.gy = a.gy; P.g_ctx = a.g_ctx; P.lnp = a.lnp;
  P.seed_dev = a.seed_dev;
  P.trace = ft_trace_buffer();
  const unsigned tiles = static_cast<unsigned>((SC + 127) / 128);
  PSB_PROF("tail_bwd_fused_tc_kernel", s);
  tail_bwd_fused_tc_kernel<<<tiles * kFtCluster, kFtThreads, kFtSmem, s>>>(map_w2t, map_w1t, map_wot, P);
  return launch_status();
}

}  // namespace enc
}  // namespace psb

extern "C" int psb_debug_tail_trace(uint64_t* out64) {
  unsigned long long* buf = psb::enc::ft_trace_buffer();
  if (out64 == nullptr) return PSB_E_ARG;
  if (buf == nullptr) return PSB_E_UNSUPPORTED;
  const cudaError_t e = cudaMemcpy(out64, buf, 64 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? PSB_OK : static_cast<int>(e);
}

extern "C" int psb_debug_gemm3_tf32(const float* a, int64_t lda, int64_t m, int64_t k, const float* bt, int64_t j,
                                    const float* bias, float* out, int64_t ldo, psb_stream_t stream) {
  if (m < 0 || m > (1 << 24) || lda < k || ldo < j) return PSB_E_ARG;
  return psb::enc::launch_rows_gemm_tc(a, static_cast<int>(lda), nullptr, static_cast<int>(m), static_cast<int>(m),
                                       static_cast<int>(k), bt, nullptr, 0, static_cast<int>(j), bias, out,
                                       static_cast<int>(ldo), static_cast<cudaStream_t>(stream));
}
