// Fused single-position sequence encoder, forward (psb_encoder_fwd; include/psb.h "N1").
//
// Launch sequence (all on the caller's stream, no host sync):
//   plan       active-token lists + compact row offsets per sequence (one CTA, block scan)
//   transpose  W^T copies of the projection weights so every product streams B row-major
//   embed      x = valid * in + pe (+ pre-LN) for the active tokens, gathered straight from the
//              item table (TEM) or a dense tensor -> compact rows
//   rows_gemm  [K | V] = xn . [Wk | Wv]^T   and   q = xn[o] . Wq^T     (FFMA CTA tiles)
//   attn       per sequence: scores of the ONE query position, softmax -> P
//   tail       per tile of R copy-rows: dropout(P) V -> Wo -> +x[o] -> LN -> W1 -> gelu -> W2 ->
//              +y -> LN, everything between the two HBM touches kept in shared memory
// On the tensor-core path (the default) the projections run on tcgen05 (gemm3_tf32_kernel) and the tail is
// tail_ctx_kernel + tail_fused_tc_kernel (gemm3_tf32.cu); the FFMA kernels below are the FFMA path (PSB_ENC_TC=0) and
// the fallback for the shapes the tensor-core kernels do not take.
#include "encoder_common.cuh"

namespace psb {
namespace enc {

// ------------------------------------------------------------------ cfg -> Dims
int dims_from_cfg(const psb_encoder_cfg_t* c, Dims* D) {
  if (c == nullptr) return PSB_E_ARG;
  if (c->S <= 0 || c->T <= 0 || c->copies <= 0 || c->heads <= 0) return PSB_E_ARG;
  if (c->d <= 0 || (c->d & 3) != 0 || c->d > 128 || c->ff <= 0 || (c->ff & 3) != 0 || c->ff > 1024) return PSB_E_DIM;
  if (c->T > 64 || c->d % c->heads != 0 || c->copies > 24 || c->out_pos < 0 || c->out_pos >= c->T) return PSB_E_DIM;
  if (c->S * c->T > (1ll << 30) / 256 * 64) return PSB_E_DIM;
  if (c->p_drop < 0.f || c->p_drop >= 1.f) return PSB_E_ARG;
  if (c->p_drop > 0.f && c->seed_dev == nullptr) return PSB_E_ARG;
  const bool tem = c->first != nullptr;
  if (tem) {
    if (c->T > 1 && (c->table == nullptr || c->idx == nullptr || c->table_rows <= 0)) return PSB_E_ARG;
  } else if (c->dense == nullptr) {
    return PSB_E_ARG;
  }
  if (misaligned16(c->first) || misaligned16(c->table) || misaligned16(c->dense) || misaligned16(c->pe))
    return PSB_E_ALIGN;
  D->S = static_cast<int>(c->S);
  D->T = static_cast<int>(c->T);
  D->d = static_cast<int>(c->d);
  D->H = static_cast<int>(c->heads);
  D->dh = D->d / D->H;
  D->F = static_cast<int>(c->ff);
  D->C = static_cast<int>(c->copies);
  D->o = static_cast<int>(c->out_pos);
  D->pre_ln = c->pre_ln != 0;
  // tile rows R (whole sequences per tile, spt = R / copies): the tail kernels run one CTA per SM whose time is
  // ~ (fixed latency + R), so pick the R in {16, 20, 24} with the least waves * (R + 10).  At the reference's
  // 1 + 5 copies and batch 384: R = 20 -> 128 tiles in one wave (R = 24: 96 tiles on 148 SMs; R = 16: two waves).
  const size_t smem_cap = 227 * 1024;
  int best_R = 0;
  long best_cost = 0;
  for (int R = 16; R <= 24; R += 4) {
    const int spt = R / D->C;
    if (spt == 0) continue;
    if (tail_bwd_smem_floats(R, D->d, D->F, D->H, D->T, spt) * sizeof(float) > smem_cap) continue;
    const long tiles = (D->S + spt - 1) / spt;
    const long cost = ((tiles + kNumSMs - 1) / kNumSMs) * (R + 10);
    if (best_R == 0 || cost < best_cost) {
      best_R = R;
      best_cost = cost;
    }
  }
  if (best_R == 0) return PSB_E_UNSUPPORTED;
  D->R = best_R;
  D->spt = best_R / D->C;
  D->ntile = (D->S + D->spt - 1) / D->spt;
  D->eps = c->ln_eps;
  D->qscale = 1.f / sqrtf(static_cast<float>(D->dh));
  D->thr = 0;
  D->keep = 1.f;
  if (c->p_drop > 0.f) {
    D->thr = static_cast<uint32_t>(static_cast<double>(c->p_drop) * 16777216.0 + 0.5);
    if (D->thr == 0) D->thr = 1;
    D->keep = 1.f / (1.f - c->p_drop);
  }
  return PSB_OK;
}

// ------------------------------------------------------------------ plan
__global__ void __launch_bounds__(1024) plan_kernel(TokSrc ts, int S, int T, int32_t* __restrict__ nact,
                                                    int32_t* __restrict__ off, int32_t* __restrict__ tok) {
  __shared__ int wsum[32];
  __shared__ int base_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) base_s = 0;
  __syncthreads();
  for (int s0 = 0; s0 < S; s0 += 1024) {
    const int s = s0 + threadIdx.x;
    int cnt = 0;
    uint64_t bits = 0;
    if (s < S) {
      for (int t = 0; t < T; ++t)
        if (tok_valid(ts, s, t, T)) {
          bits |= 1ull << t;
          ++cnt;
        }
      if (cnt == 0) {  // no valid token: the reference's softmax is uniform over all T
        cnt = T;
        bits = T >= 64 ? ~0ull : ((1ull << T) - 1);
      }
    }
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(kFull, inc, o);
      if (lane >= o) inc += v;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      int w = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(kFull, w, o);
        if (lane >= o) w += v;
      }
      wsum[lane] = w;
    }
    __syncthreads();
    const int base = base_s;
    const int excl = base + (warp > 0 ? wsum[warp - 1] : 0) + inc - cnt;
    if (s < S) {
      nact[s] = cnt;
      off[s] = excl;
      int a = 0;
      for (int t = 0; t < T; ++t)
        if ((bits >> t) & 1ull) tok[excl + a++] = t;
    }
    __syncthreads();
    if (threadIdx.x == 1023) base_s = excl + cnt;
    if (s0 + 1024 >= S && s == S - 1) off[S] = excl + cnt;
    __syncthreads();
  }
}

// ------------------------------------------------------------------ transposes
__global__ void __launch_bounds__(256) transpose_kernel(TrJobs jobs) {
  __shared__ float tile[32][33];
  int b = blockIdx.x;
  for (int q = 0; q < jobs.n; ++q) {
    const TrJob J = jobs.j[q];
    if (J.src == nullptr) {  // plain copy job: dst[i] = src2 rows (used for bias concat) -- not used
      continue;
    }
    if (J.ldd < 0) {         // split job: 1024 elements per block
      const int n = J.rows * J.cols, nb = (n + 1023) / 1024;
      if (b >= nb) {
        b -= nb;
        continue;
      }
      const int i = b * 1024 + threadIdx.x * 4;
      if (i < n) {
        const float4 v = *reinterpret_cast<const float4*>(J.src + i);
        const float4 hi = make_float4(__uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u), __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u),
                                      __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u), __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u));
        *reinterpret_cast<float4*>(J.dst + i) = hi;
        *reinterpret_cast<float4*>(J.dst + n + i) = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
      }
      return;
    }
    const int tr = (J.rows + 31) / 32, tc = (J.cols + 31) / 32;
    if (b >= tr * tc) {
      b -= tr * tc;
      continue;
    }
    const int r0 = (b / tc) * 32, c0 = (b % tc) * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int i = ty; i < 32; i += 8) {
      const int r = r0 + i, c = c0 + tx;
      tile[i][tx] = (r < J.rows && c < J.cols) ? J.src[static_cast<size_t>(r) * J.cols + c] : 0.f;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
      const int c = c0 + i, r = r0 + tx;
      if (r < J.rows && c < J.cols) {
        const float v = tile[tx][i];
        float* o = J.dst + static_cast<size_t>(c) * J.ldd + J.col0 + r;
        if (J.split) {
          const float hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
          o[0] = hi;
          o[static_cast<size_t>(J.rows) * J.cols] = v - hi;
        } else {
          o[0] = v;
        }
      }
    }
    return;
  }
}
inline int tr_blocks(const TrJobs& J) {
  int n = 0;
  for (int q = 0; q < J.n; ++q)
    n += J.j[q].ldd < 0 ? (J.j[q].rows * J.j[q].cols + 1023) / 1024 : ((J.j[q].rows + 31) / 32) * ((J.j[q].cols + 31) / 32);
  return n;
}
int launch_transposes(const TrJobs& jobs, cudaStream_t s) {
  PSB_PROF("transpose_kernel", s);
  transpose_kernel<<<tr_blocks(jobs), 256, 0, s>>>(jobs);
  return launch_status();
}

// ------------------------------------------------------------------ embed
// 4 warps per sequence; warp per active token.  Slot a == nact is the output position o when it
// is not itself active (masked): its x row (= pe[o]) still feeds q and the residual.
__global__ void __launch_bounds__(128) embed_kernel(TokSrc ts, Dims D, const float* __restrict__ ln_g,
                                                    const float* __restrict__ ln_b,
                                                    const int32_t* __restrict__ nact, const int32_t* __restrict__ off,
                                                    const int32_t* __restrict__ tok, float* __restrict__ xn,
                                                    float* __restrict__ xo, float* __restrict__ xno) {
  pdl_trigger();   // the K | V projection (gemm3_tf32_kernel) may set itself up
  const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int na = nact[s], base = off[s], d = D.d, T = D.T;
  const int j = lane * 4;
  const bool act = j < d;
  for (int a = warp; a <= na; a += 4) {
    int t;
    if (a < na) {
      t = tok[base + a];
    } else {
      t = D.o;
      bool found = false;
      for (int q = 0; q < na; ++q) found |= tok[base + q] == t;
      if (found) continue;
    }
    float4 v = zero4();
    if (act) {
      const bool valid = ts.raw || tok_valid(ts, s, t, T);
      if (valid) {
        const float* src;
        if (ts.first != nullptr)
          src = t == 0 ? ts.first + static_cast<size_t>(s) * d
                       : ts.table + static_cast<size_t>(ts.idx[static_cast<int64_t>(s) * (T - 1) + (t - 1)]) * d;
        else
          src = ts.dense + (static_cast<size_t>(s) * T + t) * d;
        v = ldg_row4(reinterpret_cast<const float4*>(src + j));
      }
      if (ts.pe != nullptr) {
        const float4 p = *reinterpret_cast<const float4*>(ts.pe + static_cast<size_t>(t) * d + j);
        v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
      }
    }
    float4 n = v;
    if (D.pre_ln) {
      const RowStats st = row_stats(v, act, d, D.eps);
      if (act)
        n = ln_apply(v, st, *reinterpret_cast<const float4*>(ln_g + j), *reinterpret_cast<const float4*>(ln_b + j));
    }
    if (act) {
      if (a < na) *reinterpret_cast<float4*>(xn + static_cast<size_t>(base + a) * d + j) = n;
      if (t == D.o) {
        *reinterpret_cast<float4*>(xo + static_cast<size_t>(s) * d + j) = v;
        *reinterpret_cast<float4*>(xno + static_cast<size_t>(s) * d + j) = n;
      }
    }
  }
}

// ------------------------------------------------------------------ rows GEMM: out = A . B (+ bias)
// A [M][lda] row-major (M on the device when m_dev != NULL), B [I][J] row-major, tiles of R rows.
template <int R>
__global__ void __launch_bounds__(kThreads) rows_gemm_kernel(const float* __restrict__ A, int lda,
                                                             const int32_t* __restrict__ m_dev, int m_host, int I,
                                                             const float* __restrict__ B, int J,
                                                             const float* __restrict__ bias, float* __restrict__ out,
                                                             int ldo) {
  extern __shared__ float4 smem4[];
  float4* A4 = smem4;
  float* red = reinterpret_cast<float*>(smem4 + (I >> 2) * R);
  const int M = m_dev != nullptr ? *m_dev : m_host;
  const int r0 = blockIdx.x * R;
  if (r0 >= M) return;
  const int n4 = I >> 2;
  for (int e = threadIdx.x; e < R * n4; e += kThreads) {
    const int r = e / n4, i4 = e - r * n4;
    float4 v = zero4();
    if (r0 + r < M) v = *reinterpret_cast<const float4*>(A + static_cast<size_t>(r0 + r) * lda + i4 * 4);
    A4[i4 * R + r] = v;
  }
  __syncthreads();
  tile_gemm<R>(A4, I, B, J, red);
  __syncthreads();
  tile_epilogue<R>(red, J, [&](int r, int j, float4 v) {
    if (r0 + r >= M) return;
    if (bias != nullptr) {
      const float4 b = *reinterpret_cast<const float4*>(bias + j);
      v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
    }
    *reinterpret_cast<float4*>(out + static_cast<size_t>(r0 + r) * ldo + j) = v;
  });
}

int launch_rows_gemm(const float* A, int lda, const int32_t* m_dev, int m_host, int m_max, int I, const float* B,
                     int J, const float* bias, float* out, int ldo, cudaStream_t s) {
  constexpr int R = 16;
  const size_t smem = (static_cast<size_t>(a4_floats(R, I)) + red_floats(R, J)) * sizeof(float);
  static DeviceAttr configured;
  if (configured.need(smem)) {
    cudaError_t e = cudaFuncSetAttribute(rows_gemm_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem));
    if (e != cudaSuccess) return static_cast<int>(e);
    configured.done(smem);
  }
  const int grid = (m_max + R - 1) / R;
  if (grid <= 0) return PSB_OK;
  PSB_PROF("rows_gemm_kernel", s);
  rows_gemm_kernel<R><<<grid, kThreads, smem, s>>>(A, lda, m_dev, m_host, I, B, J, bias, out, ldo);
  return launch_status();
}

// ------------------------------------------------------------------ attention of the one query position
__global__ void __launch_bounds__(128) attn_fwd_kernel(Dims D, const int32_t* __restrict__ nact,
                                                       const int32_t* __restrict__ off,
                                                       const int32_t* __restrict__ tok, TokSrc ts,
                                                       float* __restrict__ qv /* in: q + bq, out: scaled */,
                                                       const float* __restrict__ kv, float* __restrict__ P) {
  pdl_trigger();   // tail_ctx_kernel may be scheduled
  __shared__ float q_s[128];
  extern __shared__ float dyn[];
  float* scd = dyn;  // [H][T] scores
  const int s = blockIdx.x, d = D.d, H = D.H, dh = D.dh, T = D.T;
  const int na = nact[s], base = off[s];
  for (int j = threadIdx.x; j < d; j += blockDim.x) {
    const float v = qv[static_cast<size_t>(s) * d + j] * D.qscale;
    q_s[j] = v;
    qv[static_cast<size_t>(s) * d + j] = v;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < H * na; e += blockDim.x) {
    const int a = e / H, h = e - a * H;
    const float* kr = kv + static_cast<size_t>(base + a) * 2 * d + h * dh;
    float acc = 0.f;
    for (int j = 0; j < dh; ++j) acc = fmaf(q_s[h * dh + j], kr[j], acc);
    // masked keys (only present when NO token is valid) all carry the fill value
    if (!tok_valid(ts, s, tok[base + a], T)) acc = -1e18f;
    scd[h * T + a] = acc;
  }
  __syncthreads();
  for (int h = threadIdx.x; h < H; h += blockDim.x) {
    float m = -INFINITY;
    for (int a = 0; a < na; ++a) m = fmaxf(m, scd[h * T + a]);
    float sum = 0.f;
    for (int a = 0; a < na; ++a) {
      const float e = expf(scd[h * T + a] - m);
      scd[h * T + a] = e;
      sum += e;
    }
    for (int a = 0; a < na; ++a) P[static_cast<size_t>(base + a) * H + h] = scd[h * T + a] / sum;
  }
}

// ------------------------------------------------------------------ per-copy tail
struct TailFwdArgs {
  Dims D;
  const int32_t *nact, *off, *tok;
  const float *P, *kv, *xo;
  const float *wo_t, *bo, *w1_t, *b1, *w2_t, *b2;
  const float *ln_ff_g, *ln_ff_b, *ln_out_g, *ln_out_b;
  float *ctx, *y, *n, *z, *pre1, *h1;  // saved
  float* out;
  const uint64_t* seed_dev;
};

__host__ __device__ inline size_t tail_smem_floats(int R, int d, int F, int H, int T) {
  const int imax = d > F ? d : F;
  const int r1 = red_floats(R, d), r2 = red_floats(R, F);
  return static_cast<size_t>(a4_floats(R, imax)) + (r1 > r2 ? r1 : r2) + 2 * static_cast<size_t>(R) * (d + 4) +
         static_cast<size_t>(R) * H * T;
}

template <int R>
__global__ void __launch_bounds__(kTailThreads, 1) tail_fwd_kernel(const TailFwdArgs a) {
  extern __shared__ float4 smem4[];
  const Dims& D = a.D;
  const int d = D.d, F = D.F, H = D.H, T = D.T, C = D.C, dh = D.dh;
  const int imax = d > F ? d : F;
  float4* A4 = smem4;
  float* red = reinterpret_cast<float*>(smem4) + a4_floats(R, imax);
  const int rmax = red_floats(R, d) > red_floats(R, F) ? red_floats(R, d) : red_floats(R, F);
  float* rowsY = red + rmax;
  float* rowsZ = rowsY + R * (d + 4);
  float* Ad = rowsZ + R * (d + 4);
  const int DP = d + 4, HT = H * T;
  const int s0 = blockIdx.x * D.spt;
  const int rused = D.spt * C;
  const Drop drop = make_drop(a.seed_dev, D.thr, D.keep);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  auto row_seq = [&](int r, int* s, int* grow) -> bool {
    if (r >= rused) return false;
    const int sl = r / C;
    *s = s0 + sl;
    *grow = *s * C + (r - sl * C);
    return *s < D.S;
  };

  // (1) dropped attention weights of every copy row
  for (int e = threadIdx.x; e < R * HT; e += kTailThreads) {
    const int r = e / HT, rem = e - r * HT, h = rem / T, al = rem - h * T;
    int s, grow;
    float v = 0.f;
    if (row_seq(r, &s, &grow) && al < a.nact[s]) {
      const int base = a.off[s];
      v = a.P[static_cast<size_t>(base + al) * H + h];
      if (drop.on()) v *= drop.mul1(1u, (static_cast<uint64_t>(grow) * H + h) * T + a.tok[base + al]);
    }
    Ad[e] = v;
  }
  __syncthreads();
  // (2) context rows
  const int nd4 = d >> 2;
  for (int e = threadIdx.x; e < R * nd4; e += kTailThreads) {
    const int r = e / nd4, j = (e - r * nd4) * 4;
    int s, grow;
    float4 acc = zero4();
    if (row_seq(r, &s, &grow)) {
      const int na = a.nact[s], base = a.off[s];
      const float* ad = Ad + r * HT;
      const int h0 = j / dh, h1 = (j + 1) / dh, h2 = (j + 2) / dh, h3 = (j + 3) / dh;
      for (int al = 0; al < na; ++al) {
        const float4 v = *reinterpret_cast<const float4*>(a.kv + static_cast<size_t>(base + al) * 2 * d + d + j);
        acc.x = fmaf(ad[h0 * T + al], v.x, acc.x);
        acc.y = fmaf(ad[h1 * T + al], v.y, acc.y);
        acc.z = fmaf(ad[h2 * T + al], v.z, acc.z);
        acc.w = fmaf(ad[h3 * T + al], v.w, acc.w);
      }
      *reinterpret_cast<float4*>(a.ctx + static_cast<size_t>(grow) * d + j) = acc;
    }
    a4_store<R>(A4, r, j, acc);
  }
  __syncthreads();
  // (3) output projection + dropout + residual
  tile_gemm<R, kTailWarps>(A4, d, a.wo_t, d, red);
  __syncthreads();
  tile_epilogue<R, kTailThreads>(red, d, [&](int r, int j, float4 v) {
    int s, grow;
    if (row_seq(r, &s, &grow)) {
      const float4 b = *reinterpret_cast<const float4*>(a.bo + j);
      v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
      if (drop.on()) {
        const float4 m = drop.mul4(2u, static_cast<uint64_t>(grow) * d + j);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
      }
      const float4 x = *reinterpret_cast<const float4*>(a.xo + static_cast<size_t>(s) * d + j);
      v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
      *reinterpret_cast<float4*>(a.y + static_cast<size_t>(grow) * d + j) = v;
    } else {
      v = zero4();
    }
    *reinterpret_cast<float4*>(rowsY + r * DP + j) = v;
  });
  __syncthreads();
  // (4) feed-forward LayerNorm
  for (int r = warp; r < R; r += kTailWarps) {
    const int j = lane * 4;
    const bool act = j < d;
    int s, grow;
    const bool rv = row_seq(r, &s, &grow);
    float4 v = act ? *reinterpret_cast<const float4*>(rowsY + r * DP + j) : zero4();
    const RowStats st = row_stats(v, act, d, D.eps);
    if (act) {
      float4 n = zero4();
      if (rv) {
        n = ln_apply(v, st, *reinterpret_cast<const float4*>(a.ln_ff_g + j),
                     *reinterpret_cast<const float4*>(a.ln_ff_b + j));
        *reinterpret_cast<float4*>(a.n + static_cast<size_t>(grow) * d + j) = n;
      }
      a4_store<R>(A4, r, j, n);
    }
  }
  __syncthreads();
  // (5) W1 + gelu + dropout
  tile_gemm<R, kTailWarps>(A4, d, a.w1_t, F, red);
  __syncthreads();
  tile_epilogue<R, kTailThreads>(red, F, [&](int r, int j, float4 v) {
    int s, grow;
    float4 h = zero4();
    if (row_seq(r, &s, &grow)) {
      const float4 b = *reinterpret_cast<const float4*>(a.b1 + j);
      v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
      *reinterpret_cast<float4*>(a.pre1 + static_cast<size_t>(grow) * F + j) = v;
      h = make_float4(gelu_tanh(v.x), gelu_tanh(v.y), gelu_tanh(v.z), gelu_tanh(v.w));
      if (drop.on()) {
        const float4 m = drop.mul4(3u, static_cast<uint64_t>(grow) * F + j);
        h.x *= m.x; h.y *= m.y; h.z *= m.z; h.w *= m.w;
      }
      *reinterpret_cast<float4*>(a.h1 + static_cast<size_t>(grow) * F + j) = h;
    }
    a4_store<R>(A4, r, j, h);
  });
  __syncthreads();
  // (6) W2 + dropout + residual
  tile_gemm<R, kTailWarps>(A4, F, a.w2_t, d, red);
  __syncthreads();
  tile_epilogue<R, kTailThreads>(red, d, [&](int r, int j, float4 v) {
    int s, grow;
    if (row_seq(r, &s, &grow)) {
      const float4 b = *reinterpret_cast<const float4*>(a.b2 + j);
      v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
      if (drop.on()) {
        const float4 m = drop.mul4(4u, static_cast<uint64_t>(grow) * d + j);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
      }
      const float4 y = *reinterpret_cast<const float4*>(rowsY + r * DP + j);
      v.x += y.x; v.y += y.y; v.z += y.z; v.w += y.w;
      *reinterpret_cast<float4*>(a.z + static_cast<size_t>(grow) * d + j) = v;
    } else {
      v = zero4();
    }
    *reinterpret_cast<float4*>(rowsZ + r * DP + j) = v;
  });
  __syncthreads();
  // (7) final LayerNorm
  for (int r = warp; r < R; r += kTailWarps) {
    const int j = lane * 4;
    const bool act = j < d;
    int s, grow;
    const bool rv = row_seq(r, &s, &grow);
    float4 v = act ? *reinterpret_cast<const float4*>(rowsZ + r * DP + j) : zero4();
    const RowStats st = row_stats(v, act, d, D.eps);
    if (act && rv)
      *reinterpret_cast<float4*>(a.out + static_cast<size_t>(grow) * d + j) =
          ln_apply(v, st, *reinterpret_cast<const float4*>(a.ln_out_g + j),
                   *reinterpret_cast<const float4*>(a.ln_out_b + j));
  }
}

template <int R>
static int launch_tail_fwd(const TailFwdArgs& a, cudaStream_t s) {
  const Dims& D = a.D;
  const size_t smem = tail_smem_floats(R, D.d, D.F, D.H, D.T) * sizeof(float);
  static DeviceAttr configured;
  if (configured.need(smem)) {
    cudaError_t e = cudaFuncSetAttribute(tail_fwd_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem));
    if (e != cudaSuccess) return static_cast<int>(e);
    configured.done(smem);
  }
  PSB_PROF("tail_fwd_kernel", s);
  tail_fwd_kernel<R><<<D.ntile, kTailThreads, smem, s>>>(a);
  return launch_status();
}

}  // namespace enc
}  // namespace psb

using namespace psb;
using namespace psb::enc;

extern "C" int64_t psb_encoder_saved_bytes(const psb_encoder_cfg_t* cfg) {
  Dims D;
  const int st = dims_from_cfg(cfg, &D);
  if (st != PSB_OK) return st;
  return static_cast<int64_t>(saved_layout(D).total * sizeof(float));
}

extern "C" int psb_encoder_fwd(const psb_encoder_cfg_t* cfg, const psb_encoder_params_t* p, void* saved,
                               int64_t saved_bytes, void* workspace, int64_t workspace_bytes, float* out,
                               psb_stream_t stream) {
  Dims D;
  int st = dims_from_cfg(cfg, &D);
  if (st != PSB_OK) return st;
  if (p == nullptr || saved == nullptr || workspace == nullptr || out == nullptr) return PSB_E_ARG;
  if (p->wq == nullptr || p->wk == nullptr || p->wv == nullptr || p->wo == nullptr || p->w1 == nullptr ||
      p->w2 == nullptr || p->bq == nullptr || p->bk == nullptr || p->bv == nullptr || p->bo == nullptr ||
      p->b1 == nullptr || p->b2 == nullptr || p->ln_ff_g == nullptr || p->ln_ff_b == nullptr ||
      p->ln_out_g == nullptr || p->ln_out_b == nullptr)
    return PSB_E_ARG;
  if (D.pre_ln && (p->ln_attn_g == nullptr || p->ln_attn_b == nullptr)) return PSB_E_ARG;
  const Saved L = saved_layout(D);
  const FwdWs W = fwd_ws_layout(D);
  if (saved_bytes < static_cast<int64_t>(L.total * sizeof(float))) return PSB_E_WORKSPACE;
  if (workspace_bytes < static_cast<int64_t>(W.total * sizeof(float))) return PSB_E_WORKSPACE;
  if (misaligned16(saved) || misaligned16(workspace) || misaligned16(out)) return PSB_E_ALIGN;
  if (D.H > 32) return PSB_E_DIM;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* sv = static_cast<float*>(saved);
  float* ws = static_cast<float*>(workspace);
  int32_t* nact = reinterpret_cast<int32_t*>(sv + L.nact);
  int32_t* off = reinterpret_cast<int32_t*>(sv + L.off);
  int32_t* tok = reinterpret_cast<int32_t*>(sv + L.tok);
  const TokSrc ts{cfg->first, cfg->table, cfg->table_rows, cfg->idx, cfg->pad_idx, cfg->dense, cfg->mask, cfg->pe, cfg->raw_input != 0 && cfg->first == nullptr};
  const int d = D.d, F = D.F;

  TrJobs jobs;
  jobs.n = 0;
  auto add = [&](const float* src, float* dst, int rows, int cols, int ldd, int col0) {
    jobs.j[jobs.n++] = TrJob{src, dst, rows, cols, ldd, col0, 0};
  };
  add(p->wq, ws + W.wq_t, d, d, d, 0);           // Wq [n][k] -> Wq_t [k][n]
  add(p->wk, ws + W.wkv_t, d, d, 2 * d, 0);      // [Wk^T | Wv^T] : [k][2d]
  add(p->wv, ws + W.wkv_t, d, d, 2 * d, d);
  add(p->wo, ws + W.wo_t, d, d, d, 0);
  add(p->w1, ws + W.w1_t, F, d, F, 0);           // W1 [F][d] -> [d][F]
  add(p->w2, ws + W.w2_t, d, F, d, 0);           // W2 [d][F] -> [F][d]
  add(p->bk, ws + W.bkv, d, 1, 2 * d, 0);        // bias concat as 1-column "transposes"
  add(p->bv, ws + W.bkv, d, 1, 2 * d, d);
  const bool tc = enc_tc_enabled();
  if (tc) {                                        // the backward's grad-xn product reads [Wk^T | Wv^T] from the saved state
    add(p->wk, sv + L.wkv_t, d, d, 2 * d, 0);
    add(p->wv, sv + L.wkv_t, d, d, 2 * d, d);
  }
  const bool fused_tail = tc && d == 128 && F == 512;
  if (fused_tail) {                                // hi / lo parts of the tail's weights for tail_fused_tc_kernel
    add(p->wo, ws + W.wo_hl, d, d, -1, 0);
    add(p->w1, ws + W.w1_hl, F, d, -1, 0);
    add(p->w2, ws + W.w2_hl, d, F, -1, 0);
    // ... and, for the backward pass, of their transposes (kept with the saved activations)
    jobs.j[jobs.n++] = TrJob{p->wo, sv + L.wot_hl, d, d, d, 0, 1};
    jobs.j[jobs.n++] = TrJob{p->w1, sv + L.w1t_hl, F, d, F, 0, 1};
    jobs.j[jobs.n++] = TrJob{p->w2, sv + L.w2t_hl, d, F, d, 0, 1};
  }
  // the token plan (one CTA) and the weight transposes are independent: side by side
  st = fork_join(
      s, 0,
      [&](cudaStream_t s2) {
        PSB_PROF("transpose_kernel", s2);
        transpose_kernel<<<tr_blocks(jobs), 256, 0, s2>>>(jobs);
        return launch_status();
      },
      [&]() {
        PSB_PROF("plan_kernel", s);
        plan_kernel<<<1, 1024, 0, s>>>(ts, D.S, D.T, nact, off, tok);
        return launch_status();
      });
  if (st != PSB_OK) return st;

  if (cfg->first_ready != nullptr) {  // `first` comes from another stream: wait for it only now
    const cudaError_t we = cudaStreamWaitEvent(s, static_cast<cudaEvent_t>(cfg->first_ready), 0);
    if (we != cudaSuccess) return static_cast<int>(we);
  }
  PSB_PROF("embed_kernel", s);
  embed_kernel<<<D.S, 128, 0, s>>>(ts, D, p->ln_attn_g, p->ln_attn_b, nact, off, tok, sv + L.xn, sv + L.xo,
                                   sv + L.xno);
  if ((st = launch_status()) != PSB_OK) return st;

  // [K | V] rows of the active tokens, q of the output position
  // (independent products: the small q projection runs on the library's side stream next to the K|V one)
  // tensor-core path: both products on tcgen05 (gemm3_tf32.cu) straight from the K-major weights Wq / Wk / Wv
  const bool tc_q = tc && rows_gemm_tc_supported(sv + L.xno, d, d, p->wq, nullptr, 0, d, p->bq, sv + L.qv, d);
  const bool tc_kv = tc && rows_gemm_tc_supported(sv + L.xn, d, d, p->wk, p->wv, d, 2 * d, ws + W.bkv, sv + L.kv, 2 * d);
  st = fork_join(
      s, 1,
      [&](cudaStream_t s2) {
        if (tc_q)
          return launch_rows_gemm_tc(sv + L.xno, d, nullptr, D.S, D.S, d, p->wq, nullptr, 0, d, p->bq, sv + L.qv, d, s2);
        return launch_rows_gemm(sv + L.xno, d, nullptr, D.S, D.S, d, ws + W.wq_t, d, p->bq, sv + L.qv, d, s2);
      },
      [&]() {
        if (tc_kv)
          return launch_rows_gemm_tc(sv + L.xn, d, off + D.S, 0, D.S * D.T, d, p->wk, p->wv, d, 2 * d, ws + W.bkv,
                                     sv + L.kv, 2 * d, s);
        return launch_rows_gemm(sv + L.xn, d, off + D.S, 0, D.S * D.T, d, ws + W.wkv_t, 2 * d, ws + W.bkv, sv + L.kv,
                                2 * d, s);
      });
  if (st != PSB_OK) return st;

  PSB_PROF("attn_fwd_kernel", s);
  attn_fwd_kernel<<<D.S, 128, static_cast<size_t>(D.H) * D.T * sizeof(float), s>>>(D, nact, off, tok, ts, sv + L.qv,
                                                                                   sv + L.kv, sv + L.p);
  if ((st = launch_status()) != PSB_OK) return st;

  if (fused_tail) {
    // tensor-core path: ctx kernel + one cluster kernel chaining the tail's three products (gemm3_tf32.cu)
    TailTcArgs t;
    t.D = D;
    t.nact = nact; t.off = off; t.tok = tok;
    t.P = sv + L.p; t.kv = sv + L.kv; t.xo = sv + L.xo;
    t.wo = p->wo; t.bo = p->bo; t.w1 = p->w1; t.b1 = p->b1; t.w2 = p->w2; t.b2 = p->b2;
    t.ln_ff_g = p->ln_ff_g; t.ln_ff_b = p->ln_ff_b; t.ln_out_g = p->ln_out_g; t.ln_out_b = p->ln_out_b;
    t.ctx = sv + L.ctx; t.y = sv + L.y; t.n = sv + L.n; t.z = sv + L.z; t.pre1 = sv + L.pre1; t.h1 = sv + L.h1;
    t.out = out;
    t.seed_dev = cfg->seed_dev;
    t.wo_hl = ws + W.wo_hl; t.w1_hl = ws + W.w1_hl; t.w2_hl = ws + W.w2_hl; t.ctx_hl = ws + W.ctx_hl;
    t.save_dact = tail_bwd_fused_for(D) ? 1 : 0;
    return tail_fused_supported(t) ? launch_tail_fwd_fused(t, s) : PSB_E_ALIGN;
  }
  TailFwdArgs a;
  a.D = D;
  a.nact = nact; a.off = off; a.tok = tok;
  a.P = sv + L.p; a.kv = sv + L.kv; a.xo = sv + L.xo;
  a.wo_t = ws + W.wo_t; a.bo = p->bo; a.w1_t = ws + W.w1_t; a.b1 = p->b1; a.w2_t = ws + W.w2_t; a.b2 = p->b2;
  a.ln_ff_g = p->ln_ff_g; a.ln_ff_b = p->ln_ff_b; a.ln_out_g = p->ln_out_g; a.ln_out_b = p->ln_out_b;
  a.ctx = sv + L.ctx; a.y = sv + L.y; a.n = sv + L.n; a.z = sv + L.z; a.pre1 = sv + L.pre1; a.h1 = sv + L.h1;
  a.out = out;
  a.seed_dev = cfg->seed_dev;
  return D.R == 24 ? launch_tail_fwd<24>(a, s) : D.R == 20 ? launch_tail_fwd<20>(a, s) : launch_tail_fwd<16>(a, s);
}
