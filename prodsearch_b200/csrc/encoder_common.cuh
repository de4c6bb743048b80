// Building blocks of the fused sequence encoder (encoder_fwd.cu / encoder_bwd.cu): Philox dropout,
// the CTA-tile FFMA product every projection runs through, LayerNorm rows, saved-state layout.
//
// Work shape (SURVEY.md 8(f) N1): after restricting the last layer to the one output position the
// model reads, a TEM step has S*copies = 2304 rows of 128..512-wide projections and ~3.3k token
// rows of K/V projections -- ~1.2 GFLOP forward: latency-bound whatever computes it.  Two forms of
// every product exist: fp32 FFMA CTA tiles of R = 16/24 rows (this header's tile_gemm; ~100-200
// CTAs, weights streamed from L2 once per CTA, activations broadcast from shared memory) -- the
// fallback for any d <= 128 / ff <= 1024 -- and, for d = 128 / ff = 512, 3xTF32 products on tcgen05
// chained inside cluster kernels (gemm3_tf32.cu), the default since round 2 (PSB_ENC_TC=0 selects the FFMA path).
#pragma once
#include "psb_common.cuh"

namespace psb {
namespace enc {

constexpr int kThreads = 256;
constexpr int kWarps = 8;
// The per-copy tail kernels run ONE CTA per SM (their tiles fill shared memory); 16 warps instead of 8 double the
// warps the scheduler can pick from (ncu: IPC 1.3-1.7 at 8 warps, no single hot line -- issue-limited).
constexpr int kTailThreads = 512;
constexpr int kTailWarps = 16;

// ------------------------------------------------------------------ Philox4x32-10
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

struct Drop {
  uint2 key;
  uint32_t thr;  // keep iff (bits >> 8) >= thr, thr = round(p * 2^24); 0 = dropout off
  float scale;   // 1 / (1 - p)
  __device__ __forceinline__ bool on() const { return thr != 0u; }
  // multipliers of elements e .. e+3 (e % 4 == 0) of dropout stream `sid`
  __device__ __forceinline__ float4 mul4(uint32_t sid, uint64_t e) const {
    const uint64_t c = e >> 2;
    const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(c), static_cast<uint32_t>(c >> 32), sid, 0u), key);
    return make_float4((r.x >> 8) >= thr ? scale : 0.f, (r.y >> 8) >= thr ? scale : 0.f,
                       (r.z >> 8) >= thr ? scale : 0.f, (r.w >> 8) >= thr ? scale : 0.f);
  }
  __device__ __forceinline__ float mul1(uint32_t sid, uint64_t e) const {
    const uint64_t c = e >> 2;
    const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(c), static_cast<uint32_t>(c >> 32), sid, 0u), key);
    const uint32_t q = static_cast<uint32_t>(e & 3);
    const uint32_t b = q == 0 ? r.x : q == 1 ? r.y : q == 2 ? r.z : r.w;
    return (b >> 8) >= thr ? scale : 0.f;
  }
};

__device__ __forceinline__ Drop make_drop(const uint64_t* seed_dev, uint32_t thr, float scale) {
  Drop d;
  d.thr = thr;
  d.scale = scale;
  d.key = make_uint2(0u, 0u);
  if (thr != 0u) {
    const uint64_t s = *seed_dev;
    d.key = make_uint2(static_cast<uint32_t>(s), static_cast<uint32_t>(s >> 32));
  }
  return d;
}

// ------------------------------------------------------------------ CTA-tile product
// Y[R x J] = A[R x I] . B[I x J]: A lives in shared memory as float4 A4[i/4][r] (four consecutive
// i of row r), B row-major in global memory (read once per CTA, 128-bit coalesced, prefetched one
// 4-row block ahead).  The 8 warps split the J columns into cg groups of 128 (lane = 4 columns)
// and the I range into ks = 8 / cg slices; each warp writes its partial tile to `red`
// ([ks][R][J + 4] floats) and the caller combines the slices in fixed order (deterministic).
struct Split {
  int cg, ks;
};
__host__ __device__ inline Split split_for(int J) {
  int cg = (J + 127) / 128;
  cg = cg <= 1 ? 1 : cg <= 2 ? 2 : cg <= 4 ? 4 : 8;
  return Split{cg, 8 / cg};
}
__host__ __device__ inline int red_floats(int R, int J) { return split_for(J).ks * R * (J + 4); }
__host__ __device__ inline int a4_floats(int R, int I) { return I * R; }

template <int R, int NW = kWarps>
__device__ __forceinline__ void tile_gemm(const float4* __restrict__ A4, int I, const float* __restrict__ B, int J,
                                          float* __restrict__ red) {
  static_assert(R % 4 == 0, "tile rows");
  static_assert(NW % 8 == 0 && R % (NW / 8) == 0, "warps come in groups of 8, each group owns R / groups rows");
  constexpr int RH = R / (NW / 8);             // rows of this warp group (16 warps: two groups, each re-reads B)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w8 = warp & 7, r0 = (warp >> 3) * RH;
  const Split sp = split_for(J);
  const int cgi = w8 % sp.cg, ksi = w8 / sp.cg;
  const int col = cgi * 128 + lane * 4;
  const int n4 = I >> 2;                       // blocks of 4 rows of B
  const int per = (n4 + sp.ks - 1) / sp.ks;
  const int b0 = min(n4, ksi * per), b1 = min(n4, b0 + per);
  if (col >= J) return;
  float4 acc[RH];
#pragma unroll
  for (int r = 0; r < RH; ++r) acc[r] = zero4();
  if (b0 < b1) {
    const float* bp = B + static_cast<size_t>(b0) * 4 * J + col;
    float4 b[4], bn[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) b[u] = ldg_row4(reinterpret_cast<const float4*>(bp + static_cast<size_t>(u) * J));
    for (int blk = b0; blk < b1; ++blk) {
      const bool more = blk + 1 < b1;
      bp += static_cast<size_t>(4) * J;
#pragma unroll
      for (int u = 0; u < 4; ++u)
        bn[u] = more ? ldg_row4(reinterpret_cast<const float4*>(bp + static_cast<size_t>(u) * J)) : zero4();
      const float4* a = A4 + static_cast<size_t>(blk) * R + r0;
#pragma unroll
      for (int r = 0; r < RH; ++r) {
        const float4 av = a[r];
        fma4(acc[r], av.x, b[0]);
        fma4(acc[r], av.y, b[1]);
        fma4(acc[r], av.z, b[2]);
        fma4(acc[r], av.w, b[3]);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) b[u] = bn[u];
    }
  }
  float* rp = red + (static_cast<size_t>(ksi) * R + r0) * (J + 4) + col;
#pragma unroll
  for (int r = 0; r < RH; ++r) *reinterpret_cast<float4*>(rp + static_cast<size_t>(r) * (J + 4)) = acc[r];
}

// Combine the ks slices of `red` and hand each (row, 4 columns) to f(r, j, v).  Lanes run along
// the rows, so transposed (A4) and padded row-major stores from f are bank-conflict free.
template <int R, int NT = kThreads, typename F>
__device__ __forceinline__ void tile_epilogue(const float* __restrict__ red, int J, F&& f) {
  const int ks = split_for(J).ks;
  const int nj4 = J >> 2;
  const int JP = J + 4;
  for (int e = threadIdx.x; e < R * nj4; e += NT) {
    const int r = e % R, j = (e / R) * 4;
    float4 v = *reinterpret_cast<const float4*>(red + static_cast<size_t>(r) * JP + j);
    for (int k = 1; k < ks; ++k) {
      const float4 w = *reinterpret_cast<const float4*>(red + (static_cast<size_t>(k) * R + r) * JP + j);
      v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
    }
    f(r, j, v);
  }
}

// store 4 consecutive i (columns j..j+3 of a row-major activation) of row r into an A4 operand
template <int R>
__device__ __forceinline__ void a4_store(float4* A4, int r, int j, const float4& v) { A4[(j >> 2) * R + r] = v; }

// ------------------------------------------------------------------ LayerNorm on one row per warp
// lane holds columns lane*4 .. lane*4+3 (d <= 128); lanes beyond d hold zeros and `act` = false.
struct RowStats {
  float mean, rstd;
};
__device__ __forceinline__ RowStats row_stats(const float4& v, bool act, int d, float eps) {
  float s = act ? (v.x + v.y) + (v.z + v.w) : 0.f;
  const float mean = warp_sum(s) / static_cast<float>(d);
  float q = 0.f;
  if (act) {
    const float a = v.x - mean, b = v.y - mean, c = v.z - mean, e = v.w - mean;
    q = (a * a + b * b) + (c * c + e * e);
  }
  const float var = warp_sum(q) / static_cast<float>(d);
  return RowStats{mean, 1.f / sqrtf(var + eps)};
}
__device__ __forceinline__ float4 ln_apply(const float4& v, const RowStats& st, const float4& g, const float4& b) {
  return make_float4((v.x - st.mean) * st.rstd * g.x + b.x, (v.y - st.mean) * st.rstd * g.y + b.y,
                     (v.z - st.mean) * st.rstd * g.z + b.z, (v.w - st.mean) * st.rstd * g.w + b.w);
}
// dx of y = LN(x) given dy (per row): rstd * (gy*g - mean(gy*g) - xhat * mean(gy*g*xhat)); also
// returns xhat so the caller can accumulate the gamma gradient.
__device__ __forceinline__ float4 ln_bwd_row(const float4& x, const float4& gy, const float4& g, bool act, int d,
                                             float eps, float4* xhat_out) {
  const RowStats st = row_stats(x, act, d, eps);
  float4 xh = make_float4((x.x - st.mean) * st.rstd, (x.y - st.mean) * st.rstd, (x.z - st.mean) * st.rstd,
                          (x.w - st.mean) * st.rstd);
  float4 gg = make_float4(gy.x * g.x, gy.y * g.y, gy.z * g.z, gy.w * g.w);
  if (!act) {
    xh = zero4();
    gg = zero4();
  }
  const float m1 = warp_sum((gg.x + gg.y) + (gg.z + gg.w)) / static_cast<float>(d);
  const float m2 = warp_sum((gg.x * xh.x + gg.y * xh.y) + (gg.z * xh.z + gg.w * xh.w)) / static_cast<float>(d);
  *xhat_out = xh;
  return make_float4(st.rstd * (gg.x - m1 - xh.x * m2), st.rstd * (gg.y - m1 - xh.y * m2),
                     st.rstd * (gg.z - m1 - xh.z * m2), st.rstd * (gg.w - m1 - xh.w * m2));
}

// ln_bwd_row for N rows at once (one warp, lane = 4 columns, d = 128): the N reductions of each stage share their
// shuffle rounds, so the dependent-shuffle latency is paid three times per batch instead of four times per row.
template <int N>
__device__ __forceinline__ void warp_sum_n(float (&v)[N]) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] += __shfl_xor_sync(kFull, v[i], o);
  }
}
template <int N>
__device__ __forceinline__ void ln_bwd_rows(const float4 (&x)[N], const float4 (&gy)[N], const float4& g, int d, float eps,
                                            float4 (&dx)[N], float4 (&xhat)[N]) {
  const float inv_d = 1.f / static_cast<float>(d);
  float s[N];
#pragma unroll
  for (int i = 0; i < N; ++i) s[i] = (x[i].x + x[i].y) + (x[i].z + x[i].w);
  warp_sum_n<N>(s);
  float mean[N], q[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    mean[i] = s[i] * inv_d;
    const float a = x[i].x - mean[i], b = x[i].y - mean[i], c = x[i].z - mean[i], e = x[i].w - mean[i];
    q[i] = (a * a + b * b) + (c * c + e * e);
  }
  warp_sum_n<N>(q);
  float m[2 * N];
  float4 gg[N];
  float rstd[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    rstd[i] = 1.f / sqrtf(q[i] * inv_d + eps);
    xhat[i] = make_float4((x[i].x - mean[i]) * rstd[i], (x[i].y - mean[i]) * rstd[i], (x[i].z - mean[i]) * rstd[i],
                          (x[i].w - mean[i]) * rstd[i]);
    gg[i] = make_float4(gy[i].x * g.x, gy[i].y * g.y, gy[i].z * g.z, gy[i].w * g.w);
    m[2 * i] = (gg[i].x + gg[i].y) + (gg[i].z + gg[i].w);
    m[2 * i + 1] = (gg[i].x * xhat[i].x + gg[i].y * xhat[i].y) + (gg[i].z * xhat[i].z + gg[i].w * xhat[i].w);
  }
  warp_sum_n<2 * N>(m);
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const float m1 = m[2 * i] * inv_d, m2 = m[2 * i + 1] * inv_d;
    dx[i] = make_float4(rstd[i] * (gg[i].x - m1 - xhat[i].x * m2), rstd[i] * (gg[i].y - m1 - xhat[i].y * m2),
                        rstd[i] * (gg[i].z - m1 - xhat[i].z * m2), rstd[i] * (gg[i].w - m1 - xhat[i].w * m2));
  }
}

__device__ __forceinline__ float gelu_tanh(float x) {
  // 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3)))   models/neural.py:7-8
  const float c = 0.7978845608028654f;
  return 0.5f * x * (1.f + tanhf(c * (x + 0.044715f * x * x * x)));
}
// The same function as x * sigmoid(2 u), u = sqrt(2/pi) (x + 0.044715 x^3)  [0.5 (1 + tanh u) = 1 / (1 + e^(-2u))] on the
// special-function unit: ex2.approx + rcp.approx, relative error ~4e-7 (tanhf form: ~1e-7), a third of the instructions.
// Used where the epilogue of a tensor-core product is the critical path (gemm3_tf32.cu tail_fused_tc_kernel).
__device__ __forceinline__ float gelu_tanh_fast(float x) {
  const float c2 = -2.f * 0.7978845608028654f * 1.4426950408889634f;      // -2 sqrt(2/pi) log2(e)
  const float t = c2 * (x + 0.044715f * x * x * x);
  return __fdividef(x, 1.f + exp2f(t));
}
// value and derivative from one sigmoid: g = x s, g' = s + x s (1 - s) 2 u'
__device__ __forceinline__ float gelu_tanh_fast_both(float x, float* grad) {
  const float c = 0.7978845608028654f;
  const float x2 = x * x;
  const float t = -2.f * c * 1.4426950408889634f * (x + 0.044715f * x * x2);
  const float sg = __fdividef(1.f, 1.f + exp2f(t));
  const float xs = x * sg;
  *grad = fmaf(xs * (1.f - sg), 2.f * c * fmaf(3.f * 0.044715f, x2, 1.f), sg);
  return xs;
}
__device__ __forceinline__ float gelu_tanh_grad(float x) {
  const float c = 0.7978845608028654f;
  const float t = tanhf(c * (x + 0.044715f * x * x * x));
  return 0.5f * (1.f + t) + 0.5f * x * (1.f - t * t) * c * (1.f + 3.f * 0.044715f * x * x);
}

// ------------------------------------------------------------------ problem dimensions + saved state
struct Dims {
  int S, T, d, H, dh, F, C, o, pre_ln;
  int R;     // tile rows of the per-copy kernels (16 or 24)
  int spt;   // sequences per tile = R / C (>= 1)
  int ntile; // ceil(S / spt)
  float eps, qscale;
  uint32_t thr;
  float keep;
};

// float offsets inside the `saved` buffer (all sections 16-byte aligned)
struct Saved {
  size_t nact, off, tok;            // int32 [S], [S+1 (+pad)], [S*T]
  size_t xo, xno, qv;               // [S,d]
  size_t xn, kv, p;                 // compact token rows: [S*T,d], [S*T,2d], [S*T,H]
  size_t ctx, y, n, z, pre1, h1;    // [S*C,d] x4, [S*C,F] x2
  // transposed tail weights for the tensor-core backward tail (gemm3_tf32.cu tail_bwd_fused_tc_kernel), split into tf32
  // hi part and exact remainder, hi rows stacked on lo rows: Wo^T [2][d][d], W1^T [2][d][F], W2^T [2][F][d].  Written by
  // the forward pass's transpose launch (they are this step's weights) on the tensor-core path.
  size_t wot_hl, w1t_hl, w2t_hl;
  size_t wkv_t;                     // [Wk^T | Wv^T] : [d][2d], the K-major operand of the backward's grad-xn product on tcgen05
  size_t total;                     // floats
};
__host__ inline size_t align4(size_t x) { return (x + 3) & ~static_cast<size_t>(3); }
__host__ inline Saved saved_layout(const Dims& D) {
  Saved L;
  size_t p = 0;
  const size_t S = D.S, T = D.T, d = D.d, F = D.F, SC = static_cast<size_t>(D.S) * D.C, H = D.H;
  L.nact = p; p += align4(S);
  L.off = p; p += align4(S + 1);
  L.tok = p; p += align4(S * T);
  L.xo = p; p += S * d;
  L.xno = p; p += S * d;
  L.qv = p; p += S * d;
  L.xn = p; p += S * T * d;
  L.kv = p; p += S * T * 2 * d;
  L.p = p; p += align4(S * T * H);
  L.ctx = p; p += SC * d;
  L.y = p; p += SC * d;
  L.n = p; p += SC * d;
  L.z = p; p += SC * d;
  L.pre1 = p; p += SC * F;
  L.h1 = p; p += SC * F;
  L.wot_hl = p; p += 2 * d * d;
  L.w1t_hl = p; p += 2 * d * F;
  L.w2t_hl = p; p += 2 * F * d;
  L.wkv_t = p; p += 2 * d * d;
  L.total = p;
  return L;
}

// forward workspace: transposed weights (float offsets)
struct FwdWs {
  size_t wq_t, wkv_t, wo_t, w1_t, w2_t, bkv;
  // operands of the fused tensor-core tail (gemm3_tf32.cu tail_fused_tc_kernel), pre-split into their tf32 hi part and
  // the exact remainder, hi rows stacked on lo rows: [2][d][d], [2][F][d], [2][d][F] (original layouts), [2][S*C][d]
  size_t wo_hl, w1_hl, w2_hl, ctx_hl;
  size_t total;
};
__host__ inline FwdWs fwd_ws_layout(const Dims& D) {
  FwdWs W;
  size_t p = 0;
  const size_t d = D.d, F = D.F;
  W.wq_t = p; p += d * d;
  W.wkv_t = p; p += d * 2 * d;
  W.wo_t = p; p += d * d;
  W.w1_t = p; p += d * F;
  W.w2_t = p; p += F * d;
  W.bkv = p; p += 2 * d;
  W.wo_hl = p; p += 2 * d * d;
  W.w1_hl = p; p += 2 * F * d;
  W.w2_hl = p; p += 2 * d * F;
  W.ctx_hl = p; p += 2 * static_cast<size_t>(D.S) * D.C * d;
  W.total = p;
  return W;
}

struct TokSrc {
  const float* first;
  const float* table;
  int64_t table_rows;
  const int64_t* idx;
  int64_t pad_idx;
  const float* dense;
  const uint8_t* mask;
  const float* pe;
  int raw;  // dense rows are raw layer inputs: never zeroed by the mask
};

__device__ __forceinline__ bool tok_valid(const TokSrc& ts, int s, int t, int T) {
  if (ts.first != nullptr) {
    if (t == 0) return true;
    const int64_t v = ts.idx[static_cast<int64_t>(s) * (T - 1) + (t - 1)];
    return v != ts.pad_idx && v >= 0 && v < ts.table_rows;
  }
  return ts.mask == nullptr || ts.mask[static_cast<int64_t>(s) * T + t] != 0;
}

int dims_from_cfg(const psb_encoder_cfg_t* cfg, Dims* D);
size_t tail_bwd_smem_floats(int R, int d, int F, int H, int T, int spt);
struct TrJob {
  const float* src;  // [rows][cols]
  float* dst;        // dst[c * ldd + col0 + r]; split job (ldd < 0): dst[i] = hi(src[i]), dst[rows * cols + i] = src[i] - hi
  int rows, cols, ldd, col0;
  int split;         // transpose job only: 1 = dst gets the tf32 hi part, dst + rows * cols the exact remainder
};
struct TrJobs {
  TrJob j[16];
  int n;
};
int launch_transposes(const TrJobs& jobs, cudaStream_t s);   // encoder_fwd.cu: weight transposes, one launch
int launch_rows_gemm(const float* A, int lda, const int32_t* m_dev, int m_host, int m_max, int I, const float* B,
                     int J, const float* bias, float* out, int ldo, cudaStream_t s);
// gemm3_tf32.cu: true = the tensor-core path (default), false = the FFMA path for every encoder product (PSB_ENC_TC=0)
bool enc_tc_enabled();
// launch_rows_gemm's product on tcgen05 (3xTF32 split) from the K-major operand Bt [J][K] (rows [split, J) from Bt1 when
// given)
bool rows_gemm_tc_supported(const float* A, int lda, int K, const float* Bt0, const float* Bt1, int split, int J,
                            const float* bias, const float* out, int ldo);
int launch_rows_gemm_tc(const float* A, int lda, const int32_t* m_dev, int m_host, int m_max, int K, const float* Bt0,
                        const float* Bt1, int split, int J, const float* bias, float* out, int ldo, cudaStream_t s);
// The forward tail (encoder_fwd.cu tail_fwd_kernel) on tcgen05: ctx kernel + ONE cluster kernel chaining the three
// products (FFN hidden dimension split over 4 CTAs); same saved tensors, same dropout streams
struct TailTcArgs {
  Dims D;
  const int32_t *nact, *off, *tok;
  const float *P, *kv, *xo;
  const float *wo, *bo, *w1, *b1, *w2, *b2;      // wo [d][d], w1 [F][d], w2 [d][F] as the modules hold them
  const float *ln_ff_g, *ln_ff_b, *ln_out_g, *ln_out_b;
  float *ctx, *y, *n, *z, *pre1, *h1;            // saved for the backward pass
  float* out;
  const uint64_t* seed_dev;
  const float *wo_hl, *w1_hl, *w2_hl;            // pre-split weights (FwdWs), written by the transpose launch
  float* ctx_hl;                                 // pre-split ctx rows
  int save_dact;                                 // the pre1 slot receives dropout_3 . gelu'(pre1)
};
bool tail_fused_supported(const TailTcArgs& a);
int launch_tail_fwd_fused(const TailTcArgs& a, cudaStream_t s);
// The backward tail's product chain (LN_out' -> W2' -> gelu' -> W1' -> LN_ff' -> Wo') as ONE cluster kernel
// in the transposed form (weights are the M operand, the 128 copy rows the N operand: every global access of the
// epilogues runs along a row); the attention backward then reads gy / g_ctx from global memory (tail_bwd_kernel<R, true>)
struct TailBwdTcArgs {
  Dims D;
  const float *z, *gout, *y, *pre1, *ln_out_g, *ln_ff_g;
  const float *wot_hl, *w1t_hl, *w2t_hl;
  float *g_h2, *g_pre, *g_o1, *gy, *g_ctx;
  float* lnp;                                    // [4 * tiles][4][d]
  const uint64_t* seed_dev;
};
unsigned long long* ft_trace_buffer();           // PSB_FT_TRACE=1: 64 %globaltimer slots (psb_debug_tail_trace), else NULL
// Shared-memory floats of tail_attn_bwd_kernel (encoder_bwd.cu) for a tile of spt sequences, R = spt * C copy rows
__host__ __device__ inline size_t attn_bwd_smem_floats(int R, int d, int H, int T, int spt) {
  return 2 * static_cast<size_t>(R) * (d + 4) + 2 * static_cast<size_t>(R) * H * T + 2 * static_cast<size_t>(spt) * H * T +
         2 * static_cast<size_t>(spt) * T * (d + 4);
}
// Does the backward pass of a call with these dimensions take the tensor-core tail?  Decided from the dimensions alone,
// because the forward pass must know: it then saves dropout_3 . gelu'(pre1) in the pre1 slot and the transposed weights.
// sequences per CTA of tail_attn_bwd_kernel: as many of the tail kernels' spt as fit in shared memory (0: none does)
inline int attn_bwd_spt(const Dims& D) {
  int spt = D.spt;
  while (spt > 0 && attn_bwd_smem_floats(spt * D.C, D.d, D.H, D.T, spt) * sizeof(float) > 227 * 1024) --spt;
  return spt;
}
inline bool tail_bwd_fused_for(const Dims& D) {
  return enc_tc_enabled() && D.d == 128 && D.F == 512 && D.S * D.C > 0 && attn_bwd_spt(D) > 0;
}
int tail_bwd_fused_parts(const Dims& D);         // LayerNorm partial rows the kernel writes (4 per 128-row tile)
bool tail_bwd_fused_supported(const TailBwdTcArgs& a);
int launch_tail_bwd_fused(const TailBwdTcArgs& a, cudaStream_t s);

}  // namespace enc
}  // namespace psb
