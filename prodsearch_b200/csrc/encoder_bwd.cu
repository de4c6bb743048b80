// Fused single-position sequence encoder, backward (psb_encoder_bwd; include/psb.h "N1").
//
//   tail_bwd   per tile of R copy-rows, all in shared memory: LN_out' -> W2' -> gelu' -> W1' -> LN_ff'
//              -> Wo' -> attention' (sum over the copies of a sequence) -> softmax' ;
//              writes the operands the weight-gradient products need and grad K | V, grad q
//   rows_gemm  grad xn = [gK | gV] . [Wk ; Wv]   and   grad xn[o] += gq . Wq
//   embed_bwd  (+ pre-LN') + residual, masked -> grad of the token inputs
//   wgrad      every dW = G^T A as split-M 128x128 FFMA tiles with per-chunk partials
//   reduce     partials summed in chunk order (deterministic; no float atomics anywhere)
// On the tensor-core path (the default) tail_bwd becomes tail_bwd_fused_tc_kernel (gemm3_tf32.cu: the product chain on
// tcgen05) + tail_attn_bwd_kernel (below), the grad-xn product runs on gemm3_tf32_kernel, and wgrad / reduce are
// launched in two halves on streams of their own (see psb_encoder_bwd).
#include "encoder_common.cuh"

namespace psb {
namespace enc {

size_t tail_bwd_smem_floats(int R, int d, int F, int H, int T, int spt) {
  const int imax = d > F ? d : F;
  const int r1 = red_floats(R, d), r2 = red_floats(R, F);
  return static_cast<size_t>(a4_floats(R, imax)) + (r1 > r2 ? r1 : r2) + 2 * static_cast<size_t>(R) * (d + 4) +
         2 * static_cast<size_t>(R) * H * T + 2 * static_cast<size_t>(spt) * H * T;
}

struct TailBwdArgs {
  Dims D;
  TokSrc ts;
  const int32_t *nact, *off, *tok;
  const float *P, *kv, *qv;
  const float *wo, *w1, *w2;  // original [out,in] layouts: the transposed products read them row-major
  const float *ln_ff_g, *ln_out_g;
  const float *y, *z, *pre1;  // saved
  const float* gout;
  float *g_h2, *g_pre, *g_o1, *gxo, *g_qlin, *gkv;
  float* lnp;  // [ntile][4][d] : d ln_out_g, d ln_out_b, d ln_ff_g, d ln_ff_b
  const uint64_t* seed_dev;
  unsigned long long* trace;     // tail_attn_bwd_kernel: phase stamps of CTA 0 (slots 48..55 of the trace buffer) or NULL
  const float *gy_in, *gctx_in;  // tail_attn_bwd_kernel: the product chain ran on tcgen05 (gemm3_tf32.cu), [S*C][d] each
};

template <int R>
__global__ void __launch_bounds__(kTailThreads, 1) tail_bwd_kernel(const TailBwdArgs a) {
  extern __shared__ float4 smem4[];
  const Dims& D = a.D;
  const int d = D.d, F = D.F, H = D.H, T = D.T, C = D.C, dh = D.dh;
  const int imax = d > F ? d : F;
  const int DP = d + 4, HT = H * T;
  float4* A4 = smem4;
  float* red = reinterpret_cast<float*>(smem4) + a4_floats(R, imax);
  const int rmax = red_floats(R, d) > red_floats(R, F) ? red_floats(R, d) : red_floats(R, F);
  float* rowA = red + rmax;        // gz, then gy
  float* rowB = rowA + R * DP;     // gn, then g_ctx
  float* M1 = rowB + R * DP;       // [R][HT] attention dropout multipliers
  float* gA = M1 + R * HT;         // [R][HT]
  float* Ps = gA + R * HT;         // [spt][HT]
  float* gsc = Ps + D.spt * HT;    // [spt][HT]
  const int s0 = blockIdx.x * D.spt;
  const int rused = D.spt * C;
  const Drop drop = make_drop(a.seed_dev, D.thr, D.keep);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j4 = lane * 4;
  const bool act = j4 < d;

  auto row_seq = [&](int r, int* s, int* grow) -> bool {
    if (r >= rused) return false;
    const int sl = r / C;
    *s = s0 + sl;
    *grow = *s * C + (r - sl * C);
    return *s < D.S;
  };

  // (0) attention dropout multipliers + P of the tile's sequences
  for (int e = threadIdx.x; e < R * HT; e += kTailThreads) {
    const int r = e / HT, rem = e - r * HT, h = rem / T, al = rem - h * T;
    int s, grow;
    float v = 0.f;
    if (row_seq(r, &s, &grow) && al < a.nact[s])
      v = drop.on() ? drop.mul1(1u, (static_cast<uint64_t>(grow) * H + h) * T + a.tok[a.off[s] + al]) : 1.f;
    M1[e] = v;
  }
  for (int e = threadIdx.x; e < D.spt * HT; e += kTailThreads) {
    const int sl = e / HT, rem = e - sl * HT, h = rem / T, al = rem - h * T;
    const int s = s0 + sl;
    Ps[e] = (s < D.S && al < a.nact[s]) ? a.P[static_cast<size_t>(a.off[s] + al) * H + h] : 0.f;
  }
  // (1) LN_out backward, (2) g_h2 = gz * drop4
  float4 pg = zero4(), pb = zero4();
  for (int r = warp; r < R; r += kTailWarps) {
    int s, grow;
    const bool rv = row_seq(r, &s, &grow);
    float4 gz = zero4(), gh2 = zero4();
    if (rv) {  // warp-uniform
      const float4 z = act ? *reinterpret_cast<const float4*>(a.z + static_cast<size_t>(grow) * d + j4) : zero4();
      const float4 go = act ? *reinterpret_cast<const float4*>(a.gout + static_cast<size_t>(grow) * d + j4) : zero4();
      const float4 g = act ? *reinterpret_cast<const float4*>(a.ln_out_g + j4) : zero4();
      float4 zh;
      gz = ln_bwd_row(z, go, g, act, d, D.eps, &zh);
      pg.x += go.x * zh.x; pg.y += go.y * zh.y; pg.z += go.z * zh.z; pg.w += go.w * zh.w;
      pb.x += go.x; pb.y += go.y; pb.z += go.z; pb.w += go.w;
      gh2 = gz;
      if (act && drop.on()) {
        const float4 m = drop.mul4(4u, static_cast<uint64_t>(grow) * d + j4);
        gh2.x *= m.x; gh2.y *= m.y; gh2.z *= m.z; gh2.w *= m.w;
      }
      if (act) *reinterpret_cast<float4*>(a.g_h2 + static_cast<size_t>(grow) * d + j4) = gh2;
    }
    if (act) {
      *reinterpret_cast<float4*>(rowA + r * DP + j4) = gz;
      a4_store<R>(A4, r, j4, gh2);
    }
  }
  if (act) {  // per-warp LayerNorm parameter partials -> red (free until the first product)
    *reinterpret_cast<float4*>(red + (warp * 2 + 0) * d + j4) = pg;
    *reinterpret_cast<float4*>(red + (warp * 2 + 1) * d + j4) = pb;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 2 * d; e += kTailThreads) {
    float sacc = 0.f;
    for (int w = 0; w < kTailWarps; ++w) sacc += red[w * 2 * d + e];
    a.lnp[(static_cast<size_t>(blockIdx.x) * 4) * d + e] = sacc;
  }
  __syncthreads();
  // (3) g_h1 = g_h2 . W2  ->  g_pre = g_h1 * drop3 * gelu'(pre1)
  tile_gemm<R, kTailWarps>(A4, d, a.w2, F, red);
  __syncthreads();
  tile_epilogue<R, kTailThreads>(red, F, [&](int r, int j, float4 v) {
    int s, grow;
    float4 g = zero4();
    if (row_seq(r, &s, &grow)) {
      const float4 p = *reinterpret_cast<const float4*>(a.pre1 + static_cast<size_t>(grow) * F + j);
      g = make_float4(v.x * gelu_tanh_grad(p.x), v.y * gelu_tanh_grad(p.y), v.z * gelu_tanh_grad(p.z),
                      v.w * gelu_tanh_grad(p.w));
      if (drop.on()) {
        const float4 m = drop.mul4(3u, static_cast<uint64_t>(grow) * F + j);
        g.x *= m.x; g.y *= m.y; g.z *= m.z; g.w *= m.w;
      }
      *reinterpret_cast<float4*>(a.g_pre + static_cast<size_t>(grow) * F + j) = g;
    }
    a4_store<R>(A4, r, j, g);
  });
  __syncthreads();
  // (4) gn = g_pre . W1
  tile_gemm<R, kTailWarps>(A4, F, a.w1, d, red);
  __syncthreads();
  tile_epilogue<R, kTailThreads>(red, d, [&](int r, int j, float4 v) { *reinterpret_cast<float4*>(rowB + r * DP + j) = v; });
  __syncthreads();
  // (5) LN_ff backward + residual -> gy ; g_o1 = gy * drop2
  pg = zero4();
  pb = zero4();
  for (int r = warp; r < R; r += kTailWarps) {
    int s, grow;
    const bool rv = row_seq(r, &s, &grow);
    float4 gy = zero4(), go1 = zero4();
    if (rv) {
      const float4 y = act ? *reinterpret_cast<const float4*>(a.y + static_cast<size_t>(grow) * d + j4) : zero4();
      const float4 gn = act ? *reinterpret_cast<const float4*>(rowB + r * DP + j4) : zero4();
      const float4 g = act ? *reinterpret_cast<const float4*>(a.ln_ff_g + j4) : zero4();
      float4 yh;
      const float4 gl = ln_bwd_row(y, gn, g, act, d, D.eps, &yh);
      pg.x += gn.x * yh.x; pg.y += gn.y * yh.y; pg.z += gn.z * yh.z; pg.w += gn.w * yh.w;
      pb.x += gn.x; pb.y += gn.y; pb.z += gn.z; pb.w += gn.w;
      if (act) {
        const float4 gz = *reinterpret_cast<const float4*>(rowA + r * DP + j4);
        gy = make_float4(gz.x + gl.x, gz.y + gl.y, gz.z + gl.z, gz.w + gl.w);
        go1 = gy;
        if (drop.on()) {
          const float4 m = drop.mul4(2u, static_cast<uint64_t>(grow) * d + j4);
          go1.x *= m.x; go1.y *= m.y; go1.z *= m.z; go1.w *= m.w;
        }
        *reinterpret_cast<float4*>(a.g_o1 + static_cast<size_t>(grow) * d + j4) = go1;
      }
    }
    if (act) {
      *reinterpret_cast<float4*>(rowA + r * DP + j4) = gy;
      a4_store<R>(A4, r, j4, go1);
    }
  }
  if (act) {
    *reinterpret_cast<float4*>(red + (warp * 2 + 0) * d + j4) = pg;
    *reinterpret_cast<float4*>(red + (warp * 2 + 1) * d + j4) = pb;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 2 * d; e += kTailThreads) {
    float sacc = 0.f;
    for (int w = 0; w < kTailWarps; ++w) sacc += red[w * 2 * d + e];
    a.lnp[(static_cast<size_t>(blockIdx.x) * 4 + 2) * d + e] = sacc;
  }
  // residual gradient of x[o]: sum of gy over the copies of each sequence (copy order)
  for (int e = threadIdx.x; e < D.spt * d; e += kTailThreads) {
    const int sl = e / d, j = e - sl * d;
    const int s = s0 + sl;
    if (s < D.S) {
      float sacc = 0.f;
      for (int c = 0; c < C; ++c) sacc += rowA[(sl * C + c) * DP + j];
      a.gxo[static_cast<size_t>(s) * d + j] = sacc;
    }
  }
  __syncthreads();
  // (6) g_ctx = g_o1 . Wo
  tile_gemm<R, kTailWarps>(A4, d, a.wo, d, red);
  __syncthreads();
  tile_epilogue<R, kTailThreads>(red, d, [&](int r, int j, float4 v) { *reinterpret_cast<float4*>(rowB + r * DP + j) = v; });
  __syncthreads();
  // (7a) gA[r][h][al] = <g_ctx[r, head h], V[al, head h]>
  for (int e = threadIdx.x; e < R * HT; e += kTailThreads) {
    const int r = e / HT, rem = e - r * HT, h = rem / T, al = rem - h * T;
    int s, grow;
    float acc = 0.f;
    if (row_seq(r, &s, &grow) && al < a.nact[s]) {
      const float* v = a.kv + static_cast<size_t>(a.off[s] + al) * 2 * d + d + h * dh;
      const float* g = rowB + r * DP + h * dh;
      for (int j = 0; j < dh; ++j) acc = fmaf(g[j], v[j], acc);
    }
    gA[e] = acc;
  }
  __syncthreads();
  // (7b) softmax backward per (sequence, head)
  for (int e = threadIdx.x; e < D.spt * H; e += kTailThreads) {
    const int sl = e / H, h = e - sl * H;
    const int s = s0 + sl;
    if (s >= D.S) continue;
    const int na = a.nact[s], base = a.off[s];
    float* gs = gsc + sl * HT + h * T;
    const float* p = Ps + sl * HT + h * T;
    float dot = 0.f;
    for (int al = 0; al < na; ++al) {
      float gp = 0.f;
      for (int c = 0; c < C; ++c) {
        const int r = sl * C + c;
        gp += gA[r * HT + h * T + al] * M1[r * HT + h * T + al];
      }
      gs[al] = gp;
      dot = fmaf(p[al], gp, dot);
    }
    for (int al = 0; al < na; ++al) {
      const bool valid = tok_valid(a.ts, s, a.tok[base + al], T);  // masked scores were constants
      gs[al] = valid ? p[al] * (gs[al] - dot) : 0.f;
    }
  }
  __syncthreads();
  // (7c) grad K | V rows of the tile's sequences, grad q
  const int nd4 = d >> 2;
  for (int e = threadIdx.x; e < D.spt * T * nd4; e += kTailThreads) {
    const int sl = e / (T * nd4), rem = e - sl * (T * nd4), al = rem / nd4, j = (rem - al * nd4) * 4;
    const int s = s0 + sl;
    if (s >= D.S || al >= a.nact[s]) continue;
    const int hh[4] = {j / dh, (j + 1) / dh, (j + 2) / dh, (j + 3) / dh};
    const float4 q = *reinterpret_cast<const float4*>(a.qv + static_cast<size_t>(s) * d + j);
    const float* gs = gsc + sl * HT;
    const float4 gk = make_float4(gs[hh[0] * T + al] * q.x, gs[hh[1] * T + al] * q.y, gs[hh[2] * T + al] * q.z,
                                  gs[hh[3] * T + al] * q.w);
    float4 gv = zero4();
    const float* p = Ps + sl * HT;
    for (int c = 0; c < C; ++c) {
      const int r = sl * C + c;
      const float4 g = *reinterpret_cast<const float4*>(rowB + r * DP + j);
      const float* m = M1 + r * HT;
      gv.x = fmaf(p[hh[0] * T + al] * m[hh[0] * T + al], g.x, gv.x);
      gv.y = fmaf(p[hh[1] * T + al] * m[hh[1] * T + al], g.y, gv.y);
      gv.z = fmaf(p[hh[2] * T + al] * m[hh[2] * T + al], g.z, gv.z);
      gv.w = fmaf(p[hh[3] * T + al] * m[hh[3] * T + al], g.w, gv.w);
    }
    float* dst = a.gkv + static_cast<size_t>(a.off[s] + al) * 2 * d + j;
    *reinterpret_cast<float4*>(dst) = gk;
    *reinterpret_cast<float4*>(dst + d) = gv;
  }
  for (int e = threadIdx.x; e < D.spt * nd4; e += kTailThreads) {
    const int sl = e / nd4, j = (e - sl * nd4) * 4;
    const int s = s0 + sl;
    if (s >= D.S) continue;
    const int na = a.nact[s], base = a.off[s];
    const int hh[4] = {j / dh, (j + 1) / dh, (j + 2) / dh, (j + 3) / dh};
    const float* gs = gsc + sl * HT;
    float4 acc = zero4();
    for (int al = 0; al < na; ++al) {
      const float4 k = *reinterpret_cast<const float4*>(a.kv + static_cast<size_t>(base + al) * 2 * d + j);
      acc.x = fmaf(gs[hh[0] * T + al], k.x, acc.x);
      acc.y = fmaf(gs[hh[1] * T + al], k.y, acc.y);
      acc.z = fmaf(gs[hh[2] * T + al], k.z, acc.z);
      acc.w = fmaf(gs[hh[3] * T + al], k.w, acc.w);
    }
    acc.x *= D.qscale; acc.y *= D.qscale; acc.z *= D.qscale; acc.w *= D.qscale;
    *reinterpret_cast<float4*>(a.g_qlin + static_cast<size_t>(s) * d + j) = acc;
  }
}

template <int R>
static int launch_tail_bwd(const TailBwdArgs& a, cudaStream_t s) {
  const Dims& D = a.D;
  const size_t smem = tail_bwd_smem_floats(R, D.d, D.F, D.H, D.T, D.spt) * sizeof(float);
  static DeviceAttr configured;
  if (configured.need(smem)) {
    cudaError_t e = cudaFuncSetAttribute(tail_bwd_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem));
    if (e != cudaSuccess) return static_cast<int>(e);
    configured.done(smem);
  }
  PSB_PROF("tail_bwd_kernel", s);
  tail_bwd_kernel<R><<<D.ntile, kTailThreads, smem, s>>>(a);
  return launch_status();
}

// ------------------------------------------------------------------ attention backward on its own (tensor-core path)
// Steps (7a-c) of tail_bwd_kernel + the residual sum for a tile of spt sequences (R = spt * C copy rows) when the product
// chain ran on tcgen05 (gemm3_tf32.cu tail_bwd_fused_tc_kernel): gy and g_ctx come from global memory.  Everything the
// tile reads more than once -- its K | V rows included -- is staged in shared memory with one wave of coalesced loads,
// the softmax backward runs one warp per (sequence, head) and the grad-q sum four threads per column group, so no
// phase is a chain of dependent global loads.
__global__ void __launch_bounds__(kTailThreads, 1) tail_attn_bwd_kernel(const TailBwdArgs a, const int R) {
  pdl_trigger();                                   // the grad-xn product may set itself up
  extern __shared__ float4 smem4[];
  const Dims& D = a.D;
  const int d = D.d, H = D.H, T = D.T, C = D.C, dh = D.dh;
  const int DP = d + 4, HT = H * T, nd4 = d >> 2;
  float* rowA = reinterpret_cast<float*>(smem4);   // gy
  float* rowB = rowA + R * DP;                     // g_ctx
  float* M1 = rowB + R * DP;                       // [R][HT] attention dropout multipliers
  float* gA = M1 + R * HT;                         // [R][HT]
  float* Ps = gA + R * HT;                         // [spt][HT]
  float* gsc = Ps + D.spt * HT;                    // [spt][HT]
  float* Ks = gsc + D.spt * HT;                    // [spt][T][DP]
  float* Vs = Ks + D.spt * T * DP;                 // [spt][T][DP]
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

  if (a.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); a.trace[48 + 0] = t_; }
  // (0) one wave of loads: gy / g_ctx rows, K | V rows and P of the tile's sequences, the dropout multipliers
  for (int e = threadIdx.x; e < D.spt * T * 2 * nd4; e += kTailThreads) {
    const int sl = e / (T * 2 * nd4), rem = e - sl * (T * 2 * nd4), al = rem / (2 * nd4), c = rem - al * 2 * nd4;
    const int s = s0 + sl;
    float4 v = zero4();
    if (s < D.S && al < a.nact[s]) v = *reinterpret_cast<const float4*>(a.kv + static_cast<size_t>(a.off[s] + al) * 2 * d + c * 4);
    float* dst = (c < nd4 ? Ks : Vs) + (sl * T + al) * DP + (c < nd4 ? c : c - nd4) * 4;
    *reinterpret_cast<float4*>(dst) = v;
  }
  for (int e = threadIdx.x; e < R * HT; e += kTailThreads) {
    const int r = e / HT, rem = e - r * HT, h = rem / T, al = rem - h * T;
    int s, grow;
    float v = 0.f;
    if (row_seq(r, &s, &grow) && al < a.nact[s])
      v = drop.on() ? drop.mul1(1u, (static_cast<uint64_t>(grow) * H + h) * T + a.tok[a.off[s] + al]) : 1.f;
    M1[e] = v;
  }
  for (int e = threadIdx.x; e < D.spt * HT; e += kTailThreads) {
    const int sl = e / HT, rem = e - sl * HT, h = rem / T, al = rem - h * T;
    const int s = s0 + sl;
    Ps[e] = (s < D.S && al < a.nact[s]) ? a.P[static_cast<size_t>(a.off[s] + al) * H + h] : 0.f;
  }
  // everything above reads the forward pass's saved state only; gy / g_ctx come from the kernel before this one in the
  // stream (tail_bwd_fused_tc_kernel; programmatic dependent launch: this kernel may have started before it finished)
  pdl_wait();
  for (int e = threadIdx.x; e < R * nd4; e += kTailThreads) {
    const int r = e / nd4, j = (e - r * nd4) * 4;
    int s, grow;
    float4 gy = zero4(), gc = zero4();
    if (row_seq(r, &s, &grow)) {
      gy = *reinterpret_cast<const float4*>(a.gy_in + static_cast<size_t>(grow) * d + j);
      gc = *reinterpret_cast<const float4*>(a.gctx_in + static_cast<size_t>(grow) * d + j);
    }
    *reinterpret_cast<float4*>(rowA + r * DP + j) = gy;
    *reinterpret_cast<float4*>(rowB + r * DP + j) = gc;
  }
  __syncthreads();
  if (a.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); a.trace[48 + 1] = t_; }
  // residual gradient of x[o]: sum of gy over the copies of each sequence (copy order)
  for (int e = threadIdx.x; e < D.spt * d; e += kTailThreads) {
    const int sl = e / d, j = e - sl * d;
    const int s = s0 + sl;
    if (s < D.S) {
      float sacc = 0.f;
      for (int c = 0; c < C; ++c) sacc += rowA[(sl * C + c) * DP + j];
      a.gxo[static_cast<size_t>(s) * d + j] = sacc;
    }
  }
  // (7a) gA[r][h][al] = <g_ctx[r, head h], V[al, head h]>
  for (int e = threadIdx.x; e < R * HT; e += kTailThreads) {
    const int r = e / HT, rem = e - r * HT, h = rem / T, al = rem - h * T;
    int s, grow;
    float acc = 0.f;
    if (row_seq(r, &s, &grow) && al < a.nact[s]) {
      const float* v = Vs + ((r / C) * T + al) * DP + h * dh;
      const float* g = rowB + r * DP + h * dh;
      if ((dh & 3) == 0) {                                   // 128-bit shared-memory reads (rows are 16-byte aligned)
        for (int j = 0; j < dh; j += 4) {
          const float4 gv = *reinterpret_cast<const float4*>(g + j);
          const float4 vv = *reinterpret_cast<const float4*>(v + j);
          acc = fmaf(gv.x, vv.x, acc);
          acc = fmaf(gv.y, vv.y, acc);
          acc = fmaf(gv.z, vv.z, acc);
          acc = fmaf(gv.w, vv.w, acc);
        }
      } else {
        for (int j = 0; j < dh; ++j) acc = fmaf(g[j], v[j], acc);
      }
    }
    gA[e] = acc;
  }
  __syncthreads();
  if (a.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); a.trace[48 + 2] = t_; }
  // (7b) softmax backward, one warp per (sequence, head), lanes along the tokens
  for (int e = warp; e < D.spt * H; e += kTailWarps) {
    const int sl = e / H, h = e - sl * H;
    const int s = s0 + sl;
    if (s >= D.S) continue;                                  // warp-uniform
    const int na = a.nact[s], base = a.off[s];
    float* gs = gsc + sl * HT + h * T;
    const float* p = Ps + sl * HT + h * T;
    float dot = 0.f;
    for (int al = lane; al < na; al += 32) {
      float gp = 0.f;
      for (int c = 0; c < C; ++c) {
        const int r = sl * C + c;
        gp += gA[r * HT + h * T + al] * M1[r * HT + h * T + al];
      }
      gs[al] = gp;
      dot = fmaf(p[al], gp, dot);
    }
    dot = warp_sum(dot);
    for (int al = lane; al < na; al += 32) {
      const bool valid = tok_valid(a.ts, s, a.tok[base + al], T);  // masked scores were constants
      gs[al] = valid ? p[al] * (gs[al] - dot) : 0.f;
    }
  }
  __syncthreads();
  if (a.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); a.trace[48 + 3] = t_; }
  // (7c) grad K | V rows of the tile's sequences
  for (int e = threadIdx.x; e < D.spt * T * nd4; e += kTailThreads) {
    const int sl = e / (T * nd4), rem = e - sl * (T * nd4), al = rem / nd4, j = (rem - al * nd4) * 4;
    const int s = s0 + sl;
    if (s >= D.S || al >= a.nact[s]) continue;
    const int hh[4] = {j / dh, (j + 1) / dh, (j + 2) / dh, (j + 3) / dh};
    const float4 q = *reinterpret_cast<const float4*>(a.qv + static_cast<size_t>(s) * d + j);
    const float* gs = gsc + sl * HT;
    const float4 gk = make_float4(gs[hh[0] * T + al] * q.x, gs[hh[1] * T + al] * q.y, gs[hh[2] * T + al] * q.z,
                                  gs[hh[3] * T + al] * q.w);
    float4 gv = zero4();
    const float* p = Ps + sl * HT;
    for (int c = 0; c < C; ++c) {
      const int r = sl * C + c;
      const float4 g = *reinterpret_cast<const float4*>(rowB + r * DP + j);
      const float* m = M1 + r * HT;
      gv.x = fmaf(p[hh[0] * T + al] * m[hh[0] * T + al], g.x, gv.x);
      gv.y = fmaf(p[hh[1] * T + al] * m[hh[1] * T + al], g.y, gv.y);
      gv.z = fmaf(p[hh[2] * T + al] * m[hh[2] * T + al], g.z, gv.z);
      gv.w = fmaf(p[hh[3] * T + al] * m[hh[3] * T + al], g.w, gv.w);
    }
    float* dst = a.gkv + static_cast<size_t>(a.off[s] + al) * 2 * d + j;
    *reinterpret_cast<float4*>(dst) = gk;
    *reinterpret_cast<float4*>(dst + d) = gv;
  }
  if (a.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); a.trace[48 + 4] = t_; }
  // grad q: four threads per (sequence, 4 columns), each every fourth token, combined in fixed order
  for (int e = threadIdx.x; e < D.spt * nd4 * 4; e += kTailThreads) {
    const int part = e & 3, sl = (e >> 2) / nd4, j = ((e >> 2) - sl * nd4) * 4;
    const int s = s0 + sl;
    const int na = s < D.S ? a.nact[s] : 0;
    const int hh[4] = {j / dh, (j + 1) / dh, (j + 2) / dh, (j + 3) / dh};
    const float* gs = gsc + sl * HT;
    float4 acc = zero4();
    for (int al = part; al < na; al += 4) {
      const float4 k = *reinterpret_cast<const float4*>(Ks + (sl * T + al) * DP + j);
      acc.x = fmaf(gs[hh[0] * T + al], k.x, acc.x);
      acc.y = fmaf(gs[hh[1] * T + al], k.y, acc.y);
      acc.z = fmaf(gs[hh[2] * T + al], k.z, acc.z);
      acc.w = fmaf(gs[hh[3] * T + al], k.w, acc.w);
    }
    // (e & 3) are adjacent lanes: parts 0 + 1, 2 + 3, then the pairs
    acc.x += __shfl_xor_sync(kFull, acc.x, 1); acc.y += __shfl_xor_sync(kFull, acc.y, 1);
    acc.z += __shfl_xor_sync(kFull, acc.z, 1); acc.w += __shfl_xor_sync(kFull, acc.w, 1);
    acc.x += __shfl_xor_sync(kFull, acc.x, 2); acc.y += __shfl_xor_sync(kFull, acc.y, 2);
    acc.z += __shfl_xor_sync(kFull, acc.z, 2); acc.w += __shfl_xor_sync(kFull, acc.w, 2);
    if (part == 0 && s < D.S) {
      acc.x *= D.qscale; acc.y *= D.qscale; acc.z *= D.qscale; acc.w *= D.qscale;
      *reinterpret_cast<float4*>(a.g_qlin + static_cast<size_t>(s) * d + j) = acc;
    }
  }
  if (a.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); a.trace[48 + 5] = t_; }
}

static int launch_tail_attn_bwd(const TailBwdArgs& a_in, cudaStream_t s) {
  TailBwdArgs a = a_in;                             // its own tiling: as many sequences per CTA as shared memory holds
  a.D.spt = attn_bwd_spt(a_in.D);
  if (a.D.spt <= 0) return PSB_E_UNSUPPORTED;
  a.D.ntile = (a.D.S + a.D.spt - 1) / a.D.spt;
  const Dims& D = a.D;
  const int R = D.spt * D.C;
  const size_t smem = attn_bwd_smem_floats(R, D.d, D.H, D.T, D.spt) * sizeof(float);
  static DeviceAttr configured;
  if (configured.need(smem)) {
    cudaError_t e = cudaFuncSetAttribute(tail_attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem));
    if (e != cudaSuccess) return static_cast<int>(e);
    configured.done(smem);
  }
  PSB_PROF("tail_attn_bwd_kernel", s);
  {
    const cudaError_t le = launch_pdl(tail_attn_bwd_kernel, dim3(D.ntile), dim3(kTailThreads), smem, s, a, R);
    if (le != cudaSuccess) return static_cast<int>(le);
  }
  return launch_status();
}

// ------------------------------------------------------------------ embed backward
struct EmbedBwdArgs {
  Dims D;
  TokSrc ts;
  const int32_t *nact, *off, *tok;
  const float *gxn, *gxno, *gxo;
  const float* ln_g;
  float *g_first, *g_rest, *g_dense;
  float* lnp;  // [S][2][d] (pre_ln only)
};

__global__ void __launch_bounds__(128) embed_bwd_kernel(const EmbedBwdArgs a) {
  __shared__ float part[4 * 2 * 128];
  const Dims& D = a.D;
  const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int na = a.nact[s], base = a.off[s], d = D.d, T = D.T;
  const int j = lane * 4;
  const bool act = j < d;
  float4 pg = zero4(), pb = zero4();
  // every token gets a gradient row: zero unless the token is active (a key) or the output position
  for (int t = warp; t < T; t += 4) {
    int al = -1;
    for (int q = 0; q < na; ++q)
      if (a.tok[base + q] == t) al = q;
    const bool is_o = t == D.o;
    const bool live = al >= 0 || is_o;
    const bool valid = a.ts.raw || tok_valid(a.ts, s, t, T);  // does the input row reach x[t]?
    float4 g = zero4();
    if (live && act) {
      if (al >= 0) g = *reinterpret_cast<const float4*>(a.gxn + static_cast<size_t>(base + al) * d + j);
      if (is_o) {
        const float4 q = *reinterpret_cast<const float4*>(a.gxno + static_cast<size_t>(s) * d + j);
        g.x += q.x; g.y += q.y; g.z += q.z; g.w += q.w;
      }
    }
    if (live && D.pre_ln) {  // warp-uniform
      float4 x = zero4();
      if (act) {
        if (valid) {
          const float* src;
          if (a.ts.first != nullptr)
            src = t == 0 ? a.ts.first + static_cast<size_t>(s) * d
                         : a.ts.table + static_cast<size_t>(a.ts.idx[static_cast<int64_t>(s) * (T - 1) + (t - 1)]) * d;
          else
            src = a.ts.dense + (static_cast<size_t>(s) * T + t) * d;
          x = ldg_row4(reinterpret_cast<const float4*>(src + j));
        }
        if (a.ts.pe != nullptr) {
          const float4 p = *reinterpret_cast<const float4*>(a.ts.pe + static_cast<size_t>(t) * d + j);
          x.x += p.x; x.y += p.y; x.z += p.z; x.w += p.w;
        }
      }
      const float4 lg = act ? *reinterpret_cast<const float4*>(a.ln_g + j) : zero4();
      float4 xh;
      const float4 gx = ln_bwd_row(x, g, lg, act, d, D.eps, &xh);
      pg.x += g.x * xh.x; pg.y += g.y * xh.y; pg.z += g.z * xh.z; pg.w += g.w * xh.w;
      pb.x += g.x; pb.y += g.y; pb.z += g.z; pb.w += g.w;
      g = gx;
    }
    if (live && act && is_o) {
      const float4 r = *reinterpret_cast<const float4*>(a.gxo + static_cast<size_t>(s) * d + j);
      g.x += r.x; g.y += r.y; g.z += r.z; g.w += r.w;
    }
    if (!valid || !live) g = zero4();
    if (act) {
      float* dst;
      if (a.ts.first != nullptr)
        dst = t == 0 ? a.g_first + static_cast<size_t>(s) * d : a.g_rest + (static_cast<size_t>(s) * (T - 1) + (t - 1)) * d;
      else
        dst = a.g_dense + (static_cast<size_t>(s) * T + t) * d;
      *reinterpret_cast<float4*>(dst + j) = g;
    }
  }
  if (D.pre_ln) {
    if (act) {
      *reinterpret_cast<float4*>(part + (warp * 2 + 0) * d + j) = pg;
      *reinterpret_cast<float4*>(part + (warp * 2 + 1) * d + j) = pb;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 2 * d; e += blockDim.x) {
      float sacc = 0.f;
      for (int w = 0; w < 4; ++w) sacc += part[w * 2 * d + e];
      a.lnp[static_cast<size_t>(s) * 2 * d + e] = sacc;
    }
  }
}

// ------------------------------------------------------------------ weight gradients dW = G^T A
// rows of M per CTA (a multiple of kSub; 96 / 128 / 160 / 192 measured within 1 % of each other on the batch-384 step:
// profiles/r02_summary.md)
constexpr int kChunk = 128;
constexpr int kSub = 32;      // rows staged in shared memory at a time
struct WgProb {
  const float* G;  // [M][ldg], columns n0.. of the gradient operand
  const float* A;  // [M][lda]
  int ldg, lda;
  const int32_t* m_dev;
  int m_host, m_max;
  int N, K;
  float* part_w;  // [nch][N][K]
  float* part_b;  // [nch][N]
  int ntn, ntk, nch, tiles;  // tiles = ntn * ntk * nch
};
struct WgProbs {
  WgProb p[6];
  int n;
};

__global__ void __launch_bounds__(256) wgrad_kernel(const WgProbs probs) {
  __shared__ float4 Gs[kSub][32];  // [row][128 cols]
  __shared__ float4 As[kSub][32];
  int b = blockIdx.x, q = 0;
  while (q < probs.n && b >= probs.p[q].tiles) b -= probs.p[q++].tiles;
  if (q >= probs.n) return;
  const WgProb& P = probs.p[q];
  const int ch = b / (P.ntn * P.ntk), t2 = b - ch * (P.ntn * P.ntk), tn = t2 / P.ntk, tk = t2 - tn * P.ntk;
  const int M = P.m_dev != nullptr ? *P.m_dev : P.m_host;
  const int m0 = ch * kChunk;
  if (m0 >= M) return;
  const int m1 = min(M, m0 + kChunk);
  const int n0 = tn * 128, k0 = tk * 128;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  float bsum = 0.f;
  for (int r0 = m0; r0 < m1; r0 += kSub) {
    for (int e = threadIdx.x; e < kSub * 32; e += 256) {
      const int r = e >> 5, c4 = e & 31;
      const int row = r0 + r;
      float4 g = zero4(), av = zero4();
      if (row < m1) {
        if (n0 + c4 * 4 < P.N) g = *reinterpret_cast<const float4*>(P.G + static_cast<size_t>(row) * P.ldg + n0 + c4 * 4);
        if (k0 + c4 * 4 < P.K) av = *reinterpret_cast<const float4*>(P.A + static_cast<size_t>(row) * P.lda + k0 + c4 * 4);
      }
      Gs[r][c4] = g;
      As[r][c4] = av;
    }
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < kSub; ++r) {
      const float4 g0 = Gs[r][ty], g1 = Gs[r][16 + ty];
      const float4 a0 = As[r][tx], a1 = As[r][16 + tx];
      const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(g[i], av[j], acc[i][j]);
    }
    if (tk == 0 && threadIdx.x < 128) {
      const float* gcol = reinterpret_cast<const float*>(&Gs[0][0]) + threadIdx.x;
      for (int r = 0; r < kSub; ++r) bsum += gcol[r * 128];
    }
    __syncthreads();
  }
  float* pw = P.part_w + static_cast<size_t>(ch) * P.N * P.K;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int n = n0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (n >= P.N) continue;
    const int ka = k0 + tx * 4, kb = k0 + 64 + tx * 4;
    if (ka < P.K) *reinterpret_cast<float4*>(pw + static_cast<size_t>(n) * P.K + ka) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    if (kb < P.K) *reinterpret_cast<float4*>(pw + static_cast<size_t>(n) * P.K + kb) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
  }
  if (tk == 0 && threadIdx.x < 128 && n0 + static_cast<int>(threadIdx.x) < P.N && P.part_b != nullptr)
    P.part_b[static_cast<size_t>(ch) * P.N + n0 + threadIdx.x] = bsum;
}

struct RedJob {
  const float* part;
  float* out;
  int count, stride;  // elements per chunk, distance between chunks
  const int32_t* m_dev;
  int m_host, chunk;  // live chunks = ceil(M / chunk)
  int blocks;
};
struct RedJobs {
  RedJob j[24];
  int n;
};
__global__ void __launch_bounds__(256) reduce_kernel(const RedJobs jobs) {
  int b = blockIdx.x, q = 0;
  while (q < jobs.n && b >= jobs.j[q].blocks) b -= jobs.j[q++].blocks;
  if (q >= jobs.n) return;
  const RedJob& J = jobs.j[q];
  const int M = J.m_dev != nullptr ? *J.m_dev : J.m_host;
  const int live = (M + J.chunk - 1) / J.chunk;
  const int i = (b * 256 + threadIdx.x) * 4;
  if (i >= J.count) return;
  float4 acc = zero4();
  for (int c = 0; c < live; ++c) {
    const float4 v = *reinterpret_cast<const float4*>(J.part + static_cast<size_t>(c) * J.stride + i);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  *reinterpret_cast<float4*>(J.out + i) = acc;
}

// backward workspace (float offsets)
struct BwdWs {
  size_t wkv, g_h2, g_pre, g_o1, gxo, g_qlin, gxno, gkv, gxn, lnp_t, lnp_e, gy, g_ctx;
  size_t pw[6], pb[6];
  size_t total;
};
static BwdWs bwd_ws_layout(const Dims& D) {
  BwdWs W;
  size_t p = 0;
  const size_t S = D.S, T = D.T, d = D.d, F = D.F, SC = static_cast<size_t>(D.S) * D.C;
  W.wkv = p; p += 2 * d * d;
  W.g_h2 = p; p += SC * d;
  W.g_pre = p; p += SC * F;
  W.g_o1 = p; p += SC * d;
  W.gxo = p; p += S * d;
  W.g_qlin = p; p += S * d;
  W.gxno = p; p += S * d;
  W.gkv = p; p += S * T * 2 * d;
  W.gxn = p; p += S * T * d;
  const size_t nparts = static_cast<size_t>(D.ntile) > ((SC + 127) / 128) * 4 ? static_cast<size_t>(D.ntile) : ((SC + 127) / 128) * 4;
  W.lnp_t = p; p += nparts * 4 * d;   // tail_bwd_kernel: one row per tile; tail_bwd_fused_tc_kernel: 4 per 128 rows
  W.gy = p; p += SC * d;
  W.g_ctx = p; p += SC * d;
  W.lnp_e = p; p += S * 2 * d;
  const size_t nch_c = (SC + kChunk - 1) / kChunk, nch_t = (S * T + kChunk - 1) / kChunk, nch_s = (S + kChunk - 1) / kChunk;
  const size_t N[6] = {d, F, d, d, d, d}, K[6] = {F, d, d, d, d, d}, nch[6] = {nch_c, nch_c, nch_c, nch_t, nch_t, nch_s};
  for (int i = 0; i < 6; ++i) {
    W.pw[i] = p; p += nch[i] * N[i] * K[i];
    W.pb[i] = p; p += nch[i] * N[i];
  }
  W.total = p;
  return W;
}

}  // namespace enc
}  // namespace psb

using namespace psb;
using namespace psb::enc;

extern "C" int64_t psb_encoder_workspace_bytes(const psb_encoder_cfg_t* cfg, int32_t backward) {
  Dims D;
  const int st = dims_from_cfg(cfg, &D);
  if (st != PSB_OK) return st;
  const size_t f = backward ? bwd_ws_layout(D).total : fwd_ws_layout(D).total;
  return static_cast<int64_t>(f * sizeof(float));
}

extern "C" int psb_encoder_bwd(const psb_encoder_cfg_t* cfg, const psb_encoder_params_t* p, const void* saved,
                               int64_t saved_bytes, void* workspace, int64_t workspace_bytes, const float* grad_out,
                               float* grad_first, float* grad_rest, float* grad_dense,
                               const psb_encoder_grads_t* gr, psb_stream_t stream) {
  Dims D;
  int st = dims_from_cfg(cfg, &D);
  if (st != PSB_OK) return st;
  if (p == nullptr || saved == nullptr || workspace == nullptr || grad_out == nullptr || gr == nullptr) return PSB_E_ARG;
  const bool tem = cfg->first != nullptr;
  if (tem ? (grad_first == nullptr || (D.T > 1 && grad_rest == nullptr)) : grad_dense == nullptr) return PSB_E_ARG;
  const Saved L = saved_layout(D);
  const BwdWs W = bwd_ws_layout(D);
  if (saved_bytes < static_cast<int64_t>(L.total * sizeof(float))) return PSB_E_WORKSPACE;
  if (workspace_bytes < static_cast<int64_t>(W.total * sizeof(float))) return PSB_E_WORKSPACE;
  if (misaligned16(saved) || misaligned16(workspace) || misaligned16(grad_out) || misaligned16(grad_first) ||
      misaligned16(grad_rest) || misaligned16(grad_dense))
    return PSB_E_ALIGN;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const float* sv = static_cast<const float*>(saved);
  float* ws = static_cast<float*>(workspace);
  const int32_t* nact = reinterpret_cast<const int32_t*>(sv + L.nact);
  const int32_t* off = reinterpret_cast<const int32_t*>(sv + L.off);
  const int32_t* tok = reinterpret_cast<const int32_t*>(sv + L.tok);
  const TokSrc ts{cfg->first, cfg->table, cfg->table_rows, cfg->idx, cfg->pad_idx, cfg->dense, cfg->mask, cfg->pe, cfg->raw_input != 0 && cfg->first == nullptr};
  const int d = D.d, F = D.F, SC = D.S * D.C;

  // [Wk ; Wv] stacked so grad xn is ONE product over the 2d-wide [gK | gV] rows.  On the tensor-core path that product
  // runs on tcgen05 (gemm3_tf32.cu), which wants the K-major operand [Wk^T | Wv^T] : [d][2d] instead: the forward pass
  // left it in the saved state.
  const bool tc_gxn = enc_tc_enabled() &&
                      rows_gemm_tc_supported(ws + W.gkv, 2 * d, 2 * d, sv + L.wkv_t, nullptr, 0, d, nullptr, ws + W.gxn, d);
  cudaError_t ce = cudaSuccess;
  if (!tc_gxn) {
    ce = cudaMemcpyAsync(ws + W.wkv, p->wk, sizeof(float) * d * d, cudaMemcpyDeviceToDevice, s);
    if (ce == cudaSuccess)
      ce = cudaMemcpyAsync(ws + W.wkv + static_cast<size_t>(d) * d, p->wv, sizeof(float) * d * d, cudaMemcpyDeviceToDevice, s);
    if (ce != cudaSuccess) return static_cast<int>(ce);
  }

  TailBwdArgs a;
  a.D = D;
  a.ts = ts;
  a.nact = nact; a.off = off; a.tok = tok;
  a.P = sv + L.p; a.kv = sv + L.kv; a.qv = sv + L.qv;
  a.wo = p->wo; a.w1 = p->w1; a.w2 = p->w2;
  a.ln_ff_g = p->ln_ff_g; a.ln_out_g = p->ln_out_g;
  a.y = sv + L.y; a.z = sv + L.z; a.pre1 = sv + L.pre1;
  a.gout = grad_out;
  a.g_h2 = ws + W.g_h2; a.g_pre = ws + W.g_pre; a.g_o1 = ws + W.g_o1; a.gxo = ws + W.gxo; a.g_qlin = ws + W.g_qlin;
  a.gkv = ws + W.gkv;
  a.lnp = ws + W.lnp_t;
  a.seed_dev = cfg->seed_dev;
  a.gy_in = nullptr; a.gctx_in = nullptr;
  a.trace = ft_trace_buffer();
  // weight gradients
  WgProbs probs;
  probs.n = 0;
  int total_tiles = 0;
  auto add = [&](int i, const float* G, int ldg, const float* A, int lda, const int32_t* m_dev, int m_host, int m_max,
                 int N, int K) {
    WgProb& P = probs.p[probs.n++];
    P.G = G; P.ldg = ldg; P.A = A; P.lda = lda; P.m_dev = m_dev; P.m_host = m_host; P.m_max = m_max; P.N = N; P.K = K;
    P.part_w = ws + W.pw[i]; P.part_b = ws + W.pb[i];
    P.ntn = (N + 127) / 128; P.ntk = (K + 127) / 128; P.nch = (m_max + kChunk - 1) / kChunk;
    P.tiles = P.ntn * P.ntk * P.nch;
    total_tiles += P.tiles;
  };
  add(0, ws + W.g_h2, d, sv + L.h1, F, nullptr, SC, SC, d, F);             // dW2, db2
  add(1, ws + W.g_pre, F, sv + L.n, d, nullptr, SC, SC, F, d);             // dW1, db1
  add(2, ws + W.g_o1, d, sv + L.ctx, d, nullptr, SC, SC, d, d);            // dWo, dbo
  add(3, ws + W.gkv, 2 * d, sv + L.xn, d, off + D.S, 0, D.S * D.T, d, d);  // dWk, dbk
  add(4, ws + W.gkv + d, 2 * d, sv + L.xn, d, off + D.S, 0, D.S * D.T, d, d);  // dWv, dbv
  add(5, ws + W.g_qlin, d, sv + L.xno, d, nullptr, D.S, D.S, d, d);        // dWq, dbq
  int ln_parts = D.ntile;
  int wgrad_from = 0;          // problems [wgrad_from, 6) are still to be launched after the tail
  cudaEvent_t first_done = nullptr;   // recorded behind the first part (its stream) when the weight gradients are split
  float* gw[6] = {gr->w2, gr->w1, gr->wo, gr->wk, gr->wv, gr->wq};
  float* gb[6] = {gr->b2, gr->b1, gr->bo, gr->bk, gr->bv, gr->bq};
  auto red_into = [&](RedJobs& J, int& blocks, const float* part, float* out, int count, int stride, const int32_t* m_dev,
                      int m_host, int chunk) {
    if (out == nullptr) return;
    RedJob& R = J.j[J.n++];
    R.part = part; R.out = out; R.count = count; R.stride = stride; R.m_dev = m_dev; R.m_host = m_host; R.chunk = chunk;
    R.blocks = (count / 4 + 255) / 256;
    blocks += R.blocks;
  };
  TailBwdTcArgs tb;
  tb.D = D;
  tb.z = sv + L.z; tb.gout = grad_out; tb.y = sv + L.y; tb.pre1 = sv + L.pre1;
  tb.ln_out_g = p->ln_out_g; tb.ln_ff_g = p->ln_ff_g;
  tb.wot_hl = sv + L.wot_hl; tb.w1t_hl = sv + L.w1t_hl; tb.w2t_hl = sv + L.w2t_hl;
  tb.g_h2 = a.g_h2; tb.g_pre = a.g_pre; tb.g_o1 = a.g_o1; tb.gy = ws + W.gy; tb.g_ctx = ws + W.g_ctx;
  tb.lnp = a.lnp;
  tb.seed_dev = cfg->seed_dev;
  if (tail_bwd_fused_for(D)) {
    // (the forward pass took the same decision and saved what this path reads: no falling back from here)
    if (!tail_bwd_fused_supported(tb)) return PSB_E_ALIGN;
    // tensor-core path: the product chain on tcgen05 (gemm3_tf32.cu), then the attention backward from gy / g_ctx
    if ((st = launch_tail_bwd_fused(tb, s)) != PSB_OK) return st;
    a.gy_in = tb.gy;
    a.gctx_in = tb.g_ctx;
    ln_parts = tail_bwd_fused_parts(D);
    if (cfg->wgrad_done != nullptr && !D.pre_ln) {
      // dW2 / dW1 / dWo (90 % of the weight-gradient flops) need the product chain's outputs only: on the side stream
      // next to the attention backward
      cudaStream_t sw0 = nullptr;
      cudaEvent_t ev0 = nullptr;
      if ((st = side_stream(&sw0, &ev0, 0, &first_done)) != PSB_OK) return st;
      cudaError_t e0 = cudaEventRecord(ev0, s);
      if (e0 == cudaSuccess) e0 = cudaStreamWaitEvent(sw0, ev0, 0);
      if (e0 != cudaSuccess) return static_cast<int>(e0);
      WgProbs first;
      first.n = 3;
      int tiles = 0;
      for (int i = 0; i < 3; ++i) {
        first.p[i] = probs.p[i];
        tiles += probs.p[i].tiles;
      }
      PSB_PROF("wgrad_kernel", sw0);
      wgrad_kernel<<<tiles, 256, 0, sw0>>>(first);
      if ((st = launch_status()) != PSB_OK) return st;
      // ... and their partial sums are reduced right behind them, on the same stream; the rest of the weight gradients
      // (dWk / dWv / dWq, which wait for the attention backward) get a stream of their own
      RedJobs ja;
      ja.n = 0;
      int blocks_a = 0;
      for (int i = 0; i < 3; ++i) {
        const WgProb& P = probs.p[i];
        red_into(ja, blocks_a, P.part_w, gw[i], P.N * P.K, P.N * P.K, P.m_dev, P.m_host, kChunk);
        red_into(ja, blocks_a, P.part_b, gb[i], P.N, P.N, P.m_dev, P.m_host, kChunk);
      }
      if (blocks_a > 0) {
        PSB_PROF("reduce_kernel", sw0);
        reduce_kernel<<<blocks_a, 256, 0, sw0>>>(ja);
        if ((st = launch_status()) != PSB_OK) return st;
      }
      if ((e0 = cudaEventRecord(first_done, sw0)) != cudaSuccess) return static_cast<int>(e0);
      wgrad_from = 3;
    }
    st = launch_tail_attn_bwd(a, s);
  } else {
    st = D.R == 24 ? launch_tail_bwd<24>(a, s) : D.R == 20 ? launch_tail_bwd<20>(a, s) : launch_tail_bwd<16>(a, s);
  }
  if (st != PSB_OK) return st;

  // The weight gradients depend on the tail kernel's outputs only (and, with pre_ln, on embed_bwd's LayerNorm
  // partials): with cfg->wgrad_done they run on the library's side stream next to the data-gradient chain below.
  const bool fork_wgrad = cfg->wgrad_done != nullptr && !D.pre_ln;
  cudaStream_t sw = s;
  if (fork_wgrad) {
    cudaEvent_t fork_ev = nullptr;
    if ((st = side_stream(&sw, &fork_ev, wgrad_from > 0 ? 2 : 0)) != PSB_OK) return st;   // slot 0 runs the first part
    ce = cudaEventRecord(fork_ev, s);
    if (ce == cudaSuccess) ce = cudaStreamWaitEvent(sw, fork_ev, 0);
    if (ce != cudaSuccess) return static_cast<int>(ce);
  }
  auto data_grads = [&]() -> int {
    st = fork_join(
        s, 1,
        [&](cudaStream_t s2) {
          return launch_rows_gemm(ws + W.g_qlin, d, nullptr, D.S, D.S, d, p->wq, d, nullptr, ws + W.gxno, d, s2);
        },
        [&]() {
          if (tc_gxn)
            return launch_rows_gemm_tc(ws + W.gkv, 2 * d, off + D.S, 0, D.S * D.T, 2 * d, sv + L.wkv_t, nullptr, 0, d,
                                       nullptr, ws + W.gxn, d, s);
          return launch_rows_gemm(ws + W.gkv, 2 * d, off + D.S, 0, D.S * D.T, 2 * d, ws + W.wkv, d, nullptr,
                                  ws + W.gxn, d, s);
        });
    if (st != PSB_OK) return st;

    EmbedBwdArgs eb;
    eb.D = D;
    eb.ts = ts;
    eb.nact = nact; eb.off = off; eb.tok = tok;
    eb.gxn = ws + W.gxn; eb.gxno = ws + W.gxno; eb.gxo = ws + W.gxo;
    eb.ln_g = p->ln_attn_g;
    eb.g_first = grad_first; eb.g_rest = grad_rest; eb.g_dense = grad_dense;
    eb.lnp = ws + W.lnp_e;
    PSB_PROF("embed_bwd_kernel", s);
    embed_bwd_kernel<<<D.S, 128, 0, s>>>(eb);
    if ((st = launch_status()) != PSB_OK) return st;
    return PSB_OK;
  };
  if (!fork_wgrad && (st = data_grads()) != PSB_OK) return st;   // pre_ln: the reduce below reads embed_bwd's partials

  {
    WgProbs rest;
    rest.n = 0;
    int tiles = 0;
    for (int i = wgrad_from; i < 6; ++i) {
      rest.p[rest.n++] = probs.p[i];
      tiles += probs.p[i].tiles;
    }
    PSB_PROF("wgrad_kernel", sw);
    wgrad_kernel<<<tiles, 256, 0, sw>>>(rest);
    if ((st = launch_status()) != PSB_OK) return st;
  }

  RedJobs jobs;
  jobs.n = 0;
  int total_blocks = 0;
  auto red = [&](const float* part, float* out, int count, int stride, const int32_t* m_dev, int m_host, int chunk) {
    red_into(jobs, total_blocks, part, out, count, stride, m_dev, m_host, chunk);
  };
  for (int i = wgrad_from; i < 6; ++i) {
    const WgProb& P = probs.p[i];
    red(P.part_w, gw[i], P.N * P.K, P.N * P.K, P.m_dev, P.m_host, kChunk);
    red(P.part_b, gb[i], P.N, P.N, P.m_dev, P.m_host, kChunk);
  }
  float* lnt[4] = {gr->ln_out_g, gr->ln_out_b, gr->ln_ff_g, gr->ln_ff_b};
  for (int i = 0; i < 4; ++i) red(ws + W.lnp_t + static_cast<size_t>(i) * d, lnt[i], d, 4 * d, nullptr, ln_parts, 1);
  if (D.pre_ln) {
    red(ws + W.lnp_e, gr->ln_attn_g, d, 2 * d, nullptr, D.S, 1);
    red(ws + W.lnp_e + d, gr->ln_attn_b, d, 2 * d, nullptr, D.S, 1);
  }
  if (total_blocks > 0) {
    PSB_PROF("reduce_kernel", sw);
    reduce_kernel<<<total_blocks, 256, 0, sw>>>(jobs);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  if (fork_wgrad) {
    if (first_done != nullptr && (ce = cudaStreamWaitEvent(sw, first_done, 0)) != cudaSuccess) return static_cast<int>(ce);
    ce = cudaEventRecord(static_cast<cudaEvent_t>(cfg->wgrad_done), sw);
    if (ce != cudaSuccess) return static_cast<int>(ce);
    if ((st = data_grads()) != PSB_OK) return st;
  } else if (cfg->wgrad_done != nullptr) {
    ce = cudaEventRecord(static_cast<cudaEvent_t>(cfg->wgrad_done), s);
    if (ce != cudaSuccess) return static_cast<int>(ce);
  }
  return PSB_OK;
}
