// Fused clipped Adam over ALL parameter tensors of the model in three launches
// (psb_adam_step; SURVEY.md 8(f) N2; reference models/optimizers.py:205-243 + torch.optim.Adam):
//   sqnorm partials -> final (global L2 norm, step counter += 1) -> update.
// HBM-bound: per element 4 loads (p, g, m, v) + 3 stores = 28 B; the dense embedding tables dominate.
// No host synchronisation: the step counter, the norm and the clip factor live in device memory, so
// the whole optimizer step replays inside a CUDA graph.  Deterministic (fixed-order partial sums).
#include "psb_common.cuh"
#include "adam_common.cuh"

namespace psb {

constexpr int kAdamChunk = 4096;  // floats per CTA (256 threads x 4 float4)

struct AdamTensors {
  psb_adam_tensor_t t[PSB_ADAM_MAX_TENSORS];
  int n;
};

__device__ __forceinline__ bool locate(const AdamTensors& T, int b, int* ti, int64_t* start) {
  for (int q = 0; q < T.n; ++q) {
    const int64_t chunks = (T.t[q].n + kAdamChunk - 1) / kAdamChunk;
    if (b < chunks) {
      *ti = q;
      *start = static_cast<int64_t>(b) * kAdamChunk;
      return true;
    }
    b -= static_cast<int>(chunks);
  }
  return false;
}

__global__ void __launch_bounds__(256) sqnorm_partial_kernel(const AdamTensors T, float* __restrict__ partial) {
  __shared__ float wsum[8];
  int ti;
  int64_t start;
  float acc = 0.f;
  if (locate(T, blockIdx.x, &ti, &start)) {
    const float* g = T.t[ti].g;
    const int64_t n = T.t[ti].n;
    const int64_t end = min(n, start + kAdamChunk);
    if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
      for (int64_t i = start + threadIdx.x * 4; i < end; i += 1024) {
        if (i + 4 <= end) {
          const float4 v = *reinterpret_cast<const float4*>(g + i);
          acc += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
        } else {
          for (int64_t j = i; j < end; ++j) acc = fmaf(g[j], g[j], acc);
        }
      }
    } else {
      for (int64_t i = start + threadIdx.x; i < end; i += 256) acc = fmaf(g[i], g[i], acc);
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += wsum[w];
    partial[blockIdx.x] = s;
  }
}

// state[0] = step (as float-exact int64 in state_i), out: sqnorm
__global__ void __launch_bounds__(256) sqnorm_final_kernel(const float* __restrict__ partial, int n,
                                                           float* __restrict__ sqnorm, int64_t* __restrict__ step) {
  __shared__ double wsum[8];
  double acc = 0.0;
  const int per = (n + 255) / 256;
  const int lo = threadIdx.x * per, hi = min(n, lo + per);
  for (int i = lo; i < hi; ++i) acc += static_cast<double>(partial[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += wsum[w];
    *sqnorm = static_cast<float>(s);
    if (step != nullptr) *step += 1;
  }
}

__global__ void bump_step_kernel(int64_t* __restrict__ step) { *step += 1; }

struct AdamCoef {
  float clip, wd, omb1, b2, omb2, step_size, inv_bc2_sqrt, eps;
};

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, const AdamCoef& c) {
  const float wd = c.wd, step_size = c.step_size, inv_bc2_sqrt = c.inv_bc2_sqrt, eps = c.eps;
  g *= c.clip;
  if (wd != 0.f) g = fmaf(wd, p, g);
  m = fmaf(c.omb1, g - m, m);                 // exp_avg.lerp_(grad, 1 - beta1)
  v = fmaf(c.omb2, g * g, v * c.b2);          // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
  const float denom = sqrtf(v) * inv_bc2_sqrt + eps;
  p = fmaf(-step_size, m / denom, p);         // param.addcdiv_(exp_avg, denom, value=-step_size)
}

__global__ void __launch_bounds__(256) adam_kernel(const AdamTensors T, const AdamHyper h,
                                                   const float* __restrict__ sqnorm,
                                                   const int64_t* __restrict__ step_dev) {
  int ti;
  int64_t start;
  if (!locate(T, blockIdx.x, &ti, &start)) return;      // uniform per CTA
  // The step's coefficients are the same for every element: ONE thread per CTA forms them (double-precision pow /
  // sqrt: a few hundred FP64 instructions) and the CTA reads them from shared memory -- evaluated by all 256
  // threads they kept the SM's FP64 pipe busy for longer than the CTA's memory traffic takes.
  __shared__ AdamCoef coef;
  if (threadIdx.x == 0) {
    const float step = static_cast<float>(*step_dev);
    float clip = 1.f;
    if (h.max_norm > 0.f) {
      const float total = sqrtf(*sqnorm);
      clip = fminf(h.max_norm / (total + 1e-6f), 1.f);   // torch.nn.utils.clip_grad_norm_
    }
    double lr = h.lr;
    if (h.noam) {  // optimizers.py:214-219
      const double sd = static_cast<double>(step);
      lr = h.lr * fmin(1.0 / sqrt(sd), sd * pow(static_cast<double>(h.warmup), -1.5));
    }
    const double bc1 = 1.0 - pow(h.beta1, static_cast<double>(step));
    const double bc2 = 1.0 - pow(h.beta2, static_cast<double>(step));
    AdamCoef c0;
    c0.clip = clip;
    c0.wd = h.weight_decay;
    c0.omb1 = h.omb1;
    c0.b2 = h.b2;
    c0.omb2 = h.omb2;
    c0.step_size = static_cast<float>(lr / bc1);
    c0.inv_bc2_sqrt = static_cast<float>(1.0 / sqrt(bc2));
    c0.eps = h.eps;
    coef = c0;
  }
  __syncthreads();
  const AdamCoef c = coef;
  const psb_adam_tensor_t t = T.t[ti];
  const int64_t end = min(t.n, start + kAdamChunk);
  const bool al = ((reinterpret_cast<uintptr_t>(t.p) | reinterpret_cast<uintptr_t>(t.g) |
                    reinterpret_cast<uintptr_t>(t.m) | reinterpret_cast<uintptr_t>(t.v)) & 15) == 0;
  if (al) {
    for (int64_t i = start + threadIdx.x * 4; i < end; i += 1024) {
      if (i + 4 <= end) {
        float4 p = *reinterpret_cast<float4*>(t.p + i);
        const float4 g = *reinterpret_cast<const float4*>(t.g + i);
        float4 m = *reinterpret_cast<float4*>(t.m + i);
        float4 v = *reinterpret_cast<float4*>(t.v + i);
        adam_one(p.x, g.x, m.x, v.x, c);
        adam_one(p.y, g.y, m.y, v.y, c);
        adam_one(p.z, g.z, m.z, v.z, c);
        adam_one(p.w, g.w, m.w, v.w, c);
        *reinterpret_cast<float4*>(t.p + i) = p;
        *reinterpret_cast<float4*>(t.m + i) = m;
        *reinterpret_cast<float4*>(t.v + i) = v;
      } else {
        for (int64_t j = i; j < end; ++j)
          adam_one(t.p[j], t.g[j], t.m[j], t.v[j], c);
      }
    }
  } else {
    for (int64_t i = start + threadIdx.x; i < end; i += 256)
      adam_one(t.p[i], t.g[i], t.m[i], t.v[i], c);
  }
}


// ---------------------------------------------------------------------------------------------------------------
// Row-sparse, lazily caught-up Adam for embedding tables (psb_adam_sparse_step / psb_adam_rows_catchup).
//
// Dense Adam updates EVERY row every step, also rows whose gradient is zero: their moments decay (m *= b1, v *= b2)
// and the parameter keeps moving by -lr_t m_hat / (sqrt(v_hat) + eps).  At 16M rows that sweep is 57 GB per step for
// ~10k rows with a gradient.  Here a row carries `last_step` (the optimizer step up to which it is current) and is
// brought up to date only when somebody is about to read or update it.  A resting row's moments decay geometrically,
// so its skipped updates form a series with independent terms (catchup_row): the first min(rest, catchup_max) terms
// are summed with the per-step coefficients of the history table (they fall like (b1 / sqrt(b2))^j: 1e-9 of the first
// one after catchup_max = 198 steps at the reference's betas, far below fp32 resolution of the parameter), the
// moments decay in closed form over the whole rest.  The result equals the dense sweep within fp32 rounding
// (tests/test_gpu_adam_fp64.py holds it to a float64 replay of the dense steps).
// weight_decay must be 0 (a decayed row never rests).
struct RowTables {
  psb_adam_rows_t t[PSB_ADAM_MAX_ROW_TABLES];
  int n;
};

// One resting element over steps from+1 .. from+n: with a zero gradient the moments decay geometrically,
// m_j = m0 b1^j, v_j = v0 b2^j, so the skipped parameter updates are a series whose terms do not depend on each other:
//   p -= sum_j  a_j m0 / (b_j sqrt(v0) + eps),   a_j = step_size(from + j) b1^j,   b_j = b2^(j/2) inv_bc2_sqrt(from + j)
// (a_j, b_j are the same for every element of every row that rests from the same step: one lane forms each).
// Warp-cooperative: bring row r (and its bias element) from step `from` to step `to` (both counted in completed
// optimizer steps; from < to), all lanes of the warp active.  The series is summed over the first
// min(to - from, catchup_max) steps -- its terms fall like (b1 / sqrt(b2))^j --, the moments take their closed-form
// decay over the whole rest.
__device__ void catchup_row(const psb_adam_rows_t& t, int64_t r, int64_t from, int64_t to, const AdamHyper& h,
                            const float2* __restrict__ hist, int64_t hist_cap, int catchup_max) {
  const int lane = threadIdx.x & 31;
  const int d4 = static_cast<int>(t.d >> 2);
  const int64_t gap = to - from;
  const int nterm = static_cast<int>(gap < catchup_max ? gap : catchup_max);
  // the bases the dense step applies: m *= 1 - fl(1 - beta1) (lerp), v *= fl(beta2)
  const float m_dec = static_cast<float>(pow(1.0 - static_cast<double>(h.omb1), static_cast<double>(gap)));
  const float v_dec = static_cast<float>(pow(static_cast<double>(h.b2), static_cast<double>(gap)));
  const float l2b1 = h.l2b1, hl2b2 = 0.5f * log2f(h.b2);
  float4* p4 = reinterpret_cast<float4*>(t.p + r * t.d);
  float4* m4 = reinterpret_cast<float4*>(t.m + r * t.d);
  float4* v4 = reinterpret_cast<float4*>(t.v + r * t.d);
  const bool has_bias = t.bias_p != nullptr && lane == 0;
  float bp = 0.f, bm = 0.f, bs = 0.f, bacc = 0.f;
  if (has_bias) {
    bp = t.bias_p[r];
    bm = t.bias_m[r];
    bs = sqrtf(t.bias_v[r]);
  }
  for (int c0 = 0; c0 < d4; c0 += 32) {
    const int c = c0 + lane;
    const bool on = c < d4;
    float4 p = zero4(), m = zero4(), v = zero4();
    if (on) {
      p = p4[c];
      m = m4[c];
      v = v4[c];
    }
    const float4 s = make_float4(sqrtf(v.x), sqrtf(v.y), sqrtf(v.z), sqrtf(v.w));
    float4 acc = zero4();
    for (int j0 = 0; j0 < nterm; j0 += 32) {        // 32 terms' coefficients per trip: one per lane, then shuffled
      const int nj = min(32, nterm - j0);
      float a_mine = 0.f, b_mine = 1.f;
      if (lane < nj) {
        const float j = static_cast<float>(j0 + lane + 1);
        const StepCoef sc = load_coef(h, hist, hist_cap, from + j0 + lane + 1);
        a_mine = sc.step_size * exp2f(j * l2b1);
        b_mine = sc.inv_bc2_sqrt * exp2f(j * hl2b2);
      }
#pragma unroll 4
      for (int j = 0; j < nj; ++j) {
        const float a = __shfl_sync(kFull, a_mine, j);
        const float b = __shfl_sync(kFull, b_mine, j);
        acc.x = fmaf(a, __fdividef(m.x, fmaf(b, s.x, h.eps)), acc.x);
        acc.y = fmaf(a, __fdividef(m.y, fmaf(b, s.y, h.eps)), acc.y);
        acc.z = fmaf(a, __fdividef(m.z, fmaf(b, s.z, h.eps)), acc.z);
        acc.w = fmaf(a, __fdividef(m.w, fmaf(b, s.w, h.eps)), acc.w);
        if (c0 == 0 && has_bias) bacc = fmaf(a, __fdividef(bm, fmaf(b, bs, h.eps)), bacc);
      }
    }
    if (on) {
      p4[c] = make_float4(p.x - acc.x, p.y - acc.y, p.z - acc.z, p.w - acc.w);
      m4[c] = make_float4(m.x * m_dec, m.y * m_dec, m.z * m_dec, m.w * m_dec);
      v4[c] = make_float4(v.x * v_dec, v.y * v_dec, v.z * v_dec, v.w * v_dec);
    }
  }
  if (has_bias) {
    t.bias_p[r] = bp - bacc;
    t.bias_m[r] = bm * m_dec;
    t.bias_v[r] = t.bias_v[r] * v_dec;
  }
}

struct IdxLists {
  const int64_t* idx[PSB_ADAM_MAX_IDX_LISTS];
  int64_t start[PSB_ADAM_MAX_IDX_LISTS + 1];   // prefix sums of the list lengths
  int n;
};

// One warp per index occurrence (or per table row when L.n == 0: flush).  Duplicates -- within the launch or from an
// earlier launch of the same step -- are resolved by an atomicMax claim on last_step: exactly one warp replays the
// row, the others see it claimed and leave.  Readers of the rows run in LATER kernels (stream order), so nobody
// observes a half-updated row.
__global__ void __launch_bounds__(256) adam_rows_catchup_kernel(const psb_adam_rows_t t, const IdxLists L,
                                                                int64_t total, int64_t skip_row, const AdamHyper h,
                                                                const int64_t* __restrict__ step_dev,
                                                                const float2* __restrict__ hist, int64_t hist_cap,
                                                                int catchup_max) {
  const int lane = threadIdx.x & 31;
  const int64_t cur = *step_dev;
  if (cur <= 0) return;
  const int64_t warp0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  for (int64_t i = warp0; i < total; i += nwarp) {
    int64_t r = i;
    if (L.n > 0) {
      int q = 0;
      while (q + 1 < L.n && i >= L.start[q + 1]) ++q;
      r = L.idx[q][i - L.start[q]];
    }
    if (r < 0 || r >= t.table_rows || r == skip_row) continue;
    int prev = 0;
    if (lane == 0) {
      prev = t.last_step[r];
      if (prev < cur) prev = atomicMax(t.last_step + r, static_cast<int>(cur));
    }
    prev = __shfl_sync(kFull, prev, 0);
    if (prev >= cur || prev == 0) continue;      // current, or never updated: moments are zero, nothing to replay
    catchup_row(t, r, prev, cur, h, hist, hist_cap, catchup_max);
  }
}

// |g|^2 partials of the compact row gradients (and bias gradients) of the row-sparse tables, appended to the dense
// tensors' partials: block b covers rows [32 b, 32 b + 32) of one table's list; rows past *n_rows count 0.
__global__ void __launch_bounds__(256) sqnorm_rows_partial_kernel(const RowTables R, float* __restrict__ partial) {
  __shared__ float wsum[8];
  int b = blockIdx.x, ti = -1;
  for (int q = 0; q < R.n; ++q) {
    const int blocks = static_cast<int>((R.t[q].cap + 31) / 32);
    if (b < blocks) {
      ti = q;
      break;
    }
    b -= blocks;
  }
  float acc = 0.f;
  if (ti >= 0) {
    const psb_adam_rows_t& t = R.t[ti];
    const int64_t n = *t.n_rows;
    const int64_t lo = static_cast<int64_t>(b) * 32, hi = min(n, lo + 32);
    if (lo < hi && !t.grad_by_row) {
      const float4* g4 = reinterpret_cast<const float4*>(t.grad + lo * t.d);
      const int64_t n4 = (hi - lo) * (t.d >> 2);
      for (int64_t i = threadIdx.x; i < n4; i += 256) {
        const float4 v = g4[i];
        acc += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
      }
      if (t.bias_grad != nullptr && threadIdx.x < hi - lo) {
        const float gb = t.bias_grad[lo + threadIdx.x];
        acc = fmaf(gb, gb, acc);
      }
    } else if (lo < hi) {              // dense gradient buffer, only the listed rows are valid: one warp per entry
      const int d4 = static_cast<int>(t.d >> 2);
      for (int64_t e = lo + (threadIdx.x >> 5); e < hi; e += 8) {
        const int64_t r = t.rows[e];
        if (r < 0 || r >= t.table_rows) continue;
        const float4* g4 = reinterpret_cast<const float4*>(t.grad + r * t.d);
        for (int c = threadIdx.x & 31; c < d4; c += 32) {
          const float4 v = g4[c];
          acc += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
        }
        if (t.bias_grad != nullptr && (threadIdx.x & 31) == 0) acc = fmaf(t.bias_grad[r], t.bias_grad[r], acc);
      }
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += wsum[w];
    partial[blockIdx.x] = s;
  }
}

__device__ __forceinline__ AdamCoef make_coef(const AdamHyper& h, const float* sqnorm, int64_t step) {
  float clip = 1.f;
  if (h.max_norm > 0.f) {
    const float total = sqrtf(*sqnorm);
    clip = fminf(h.max_norm / (total + 1e-6f), 1.f);   // torch.nn.utils.clip_grad_norm_
  }
  const StepCoef sc = step_coef(h, step);
  AdamCoef c0;
  c0.clip = clip;
  c0.wd = h.weight_decay;
  c0.omb1 = h.omb1;
  c0.b2 = h.b2;
  c0.omb2 = h.omb2;
  c0.step_size = sc.step_size;
  c0.inv_bc2_sqrt = sc.inv_bc2_sqrt;
  c0.eps = h.eps;
  return c0;
}

// The update of the step's touched rows: one warp per list entry.  The row is first caught up to step - 1 (normally
// a no-op: the forward pass read the row, so psb_adam_rows_catchup has already run for it), then takes the ordinary
// Adam update with its reduced gradient and is stamped with the new step.  Block 0 also appends the step's
// coefficients to the history table (also when no table has a list this step: the launch then has one block).
__global__ void __launch_bounds__(256) adam_rows_kernel(const RowTables R, const AdamHyper h,
                                                        const float* __restrict__ sqnorm,
                                                        const int64_t* __restrict__ step_dev, float2* __restrict__ hist,
                                                        int64_t hist_cap, int catchup_max) {
  __shared__ AdamCoef coef;
  const int64_t step = *step_dev;
  if (threadIdx.x == 0) {
    coef = make_coef(h, sqnorm, step);
    if (blockIdx.x == 0 && hist != nullptr && step < hist_cap) hist[step] = make_float2(coef.step_size, coef.inv_bc2_sqrt);
  }
  __syncthreads();
  const AdamCoef c = coef;
  int b = blockIdx.x, ti = -1;
  for (int q = 0; q < R.n; ++q) {
    const int blocks = static_cast<int>((R.t[q].cap + 7) / 8);
    if (b < blocks) {
      ti = q;
      break;
    }
    b -= blocks;
  }
  if (ti < 0) return;
  const psb_adam_rows_t& t = R.t[ti];
  const int lane = threadIdx.x & 31;
  const int64_t i = static_cast<int64_t>(b) * 8 + (threadIdx.x >> 5);
  if (i >= *t.n_rows) return;
  const int64_t r = t.rows[i];
  if (r < 0 || r >= t.table_rows) return;
  const int prev = t.last_step[r];
  if (prev > 0 && prev < step - 1) catchup_row(t, r, prev, step - 1, h, hist, hist_cap, catchup_max);
  __syncwarp();
  const int d4 = static_cast<int>(t.d >> 2);
  float4* p4 = reinterpret_cast<float4*>(t.p + r * t.d);
  float4* m4 = reinterpret_cast<float4*>(t.m + r * t.d);
  float4* v4 = reinterpret_cast<float4*>(t.v + r * t.d);
  const float4* g4 = reinterpret_cast<const float4*>(t.grad + (t.grad_by_row ? r : i) * t.d);
  for (int k = lane; k < d4; k += 32) {
    float4 p = p4[k], m = m4[k], v = v4[k];
    const float4 g = g4[k];
    adam_one(p.x, g.x, m.x, v.x, c);
    adam_one(p.y, g.y, m.y, v.y, c);
    adam_one(p.z, g.z, m.z, v.z, c);
    adam_one(p.w, g.w, m.w, v.w, c);
    p4[k] = p;
    m4[k] = m;
    v4[k] = v;
  }
  if (lane == 0) {
    if (t.bias_p != nullptr) {
      const float g = t.bias_grad != nullptr ? t.bias_grad[t.grad_by_row ? r : i] : 0.f;
      adam_one(t.bias_p[r], g, t.bias_m[r], t.bias_v[r], c);
    }
    t.last_step[r] = static_cast<int>(step);
  }
}

}  // namespace psb

using namespace psb;

static int64_t adam_chunks(const psb_adam_tensor_t* t, int32_t n) {
  int64_t c = 0;
  for (int i = 0; i < n; ++i) c += (t[i].n + kAdamChunk - 1) / kAdamChunk;
  return c;
}

extern "C" int64_t psb_adam_workspace_bytes(const psb_adam_tensor_t* tensors, int32_t n_tensors) {
  if (tensors == nullptr || n_tensors <= 0 || n_tensors > PSB_ADAM_MAX_TENSORS) return PSB_E_ARG;
  return (adam_chunks(tensors, n_tensors) + 4) * static_cast<int64_t>(sizeof(float));
}

extern "C" int psb_adam_step(const psb_adam_tensor_t* tensors, int32_t n_tensors, double lr, double beta1, double beta2,
                             double eps, double weight_decay, double max_grad_norm, int32_t noam, double warmup_steps,
                             int32_t norm_given, int64_t* step_dev, float* sqnorm_dev, void* workspace, int64_t workspace_bytes,
                             psb_stream_t stream) {
  if (tensors == nullptr || n_tensors <= 0 || n_tensors > PSB_ADAM_MAX_TENSORS || step_dev == nullptr ||
      sqnorm_dev == nullptr || workspace == nullptr)
    return PSB_E_ARG;
  AdamTensors T;
  T.n = n_tensors;
  for (int i = 0; i < n_tensors; ++i) {
    if (tensors[i].p == nullptr || tensors[i].g == nullptr || tensors[i].m == nullptr || tensors[i].v == nullptr ||
        tensors[i].n <= 0)
      return PSB_E_ARG;
    T.t[i] = tensors[i];
  }
  const int64_t chunks = adam_chunks(tensors, n_tensors);
  if (chunks > (1ll << 30)) return PSB_E_DIM;
  if (workspace_bytes < (chunks + 4) * static_cast<int64_t>(sizeof(float))) return PSB_E_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(workspace);
  int st;
  if (norm_given == 2) {
    // norm and step counter were both written by the caller
  } else if (norm_given) {
    PSB_PROF("bump_step_kernel", s);
    bump_step_kernel<<<1, 1, 0, s>>>(step_dev);
    if ((st = launch_status()) != PSB_OK) return st;
  } else {
    PSB_PROF("sqnorm_partial_kernel", s);
    sqnorm_partial_kernel<<<static_cast<int>(chunks), 256, 0, s>>>(T, partial);
    if ((st = launch_status()) != PSB_OK) return st;
    PSB_PROF("sqnorm_final_kernel", s);
    sqnorm_final_kernel<<<1, 256, 0, s>>>(partial, static_cast<int>(chunks), sqnorm_dev, step_dev);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  const AdamHyper h = make_adam_hyper(lr, beta1, beta2, eps, weight_decay, max_grad_norm, noam, warmup_steps);
  PSB_PROF("adam_kernel", s);
  adam_kernel<<<static_cast<int>(chunks), 256, 0, s>>>(T, h, sqnorm_dev, step_dev);
  return launch_status();
}


extern "C" int psb_grad_sqnorm(const psb_adam_tensor_t* tensors, int32_t n_tensors, float* sqnorm_out, void* workspace,
                               int64_t workspace_bytes, psb_stream_t stream) {
  if (tensors == nullptr || n_tensors <= 0 || n_tensors > PSB_ADAM_MAX_TENSORS || sqnorm_out == nullptr ||
      workspace == nullptr)
    return PSB_E_ARG;
  AdamTensors T;
  T.n = n_tensors;
  for (int i = 0; i < n_tensors; ++i) {
    if (tensors[i].g == nullptr || tensors[i].n <= 0) return PSB_E_ARG;
    T.t[i] = tensors[i];
  }
  const int64_t chunks = adam_chunks(tensors, n_tensors);
  if (chunks > (1ll << 30)) return PSB_E_DIM;
  if (workspace_bytes < (chunks + 4) * static_cast<int64_t>(sizeof(float))) return PSB_E_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(workspace);
  int st;
  PSB_PROF("sqnorm_partial_kernel", s);
  sqnorm_partial_kernel<<<static_cast<int>(chunks), 256, 0, s>>>(T, partial);
  if ((st = launch_status()) != PSB_OK) return st;
  PSB_PROF("sqnorm_final_kernel", s);
  sqnorm_final_kernel<<<1, 256, 0, s>>>(partial, static_cast<int>(chunks), sqnorm_out, nullptr);
  return launch_status();
}


// ---- row-sparse Adam (see the kernels above) ------------------------------------------------------------------
static int check_row_table(const psb_adam_rows_t& t, bool need_list) {
  if (t.p == nullptr || t.m == nullptr || t.v == nullptr || t.last_step == nullptr || t.table_rows <= 0) return PSB_E_ARG;
  if (t.d <= 0 || (t.d & 3) != 0 || t.d > 512) return PSB_E_DIM;
  if (misaligned16(t.p) || misaligned16(t.m) || misaligned16(t.v) || misaligned16(t.grad)) return PSB_E_ALIGN;
  if (need_list && (t.rows == nullptr || t.grad == nullptr || t.n_rows == nullptr || t.cap <= 0)) return PSB_E_ARG;
  if (t.bias_p != nullptr && (t.bias_m == nullptr || t.bias_v == nullptr)) return PSB_E_ARG;
  return PSB_OK;
}

static AdamHyper make_hyper(double lr, double beta1, double beta2, double eps, double weight_decay, double max_grad_norm,
                            int32_t noam, double warmup_steps) {
  return make_adam_hyper(lr, beta1, beta2, eps, weight_decay, max_grad_norm, noam, warmup_steps);
}

static int64_t row_norm_blocks(const psb_adam_rows_t* t, int32_t n) {
  int64_t b = 0;
  for (int i = 0; i < n; ++i) b += (t[i].cap + 31) / 32;
  return b;
}

extern "C" int32_t psb_adam_catchup_steps(double beta1, double beta2) {
  // skipped updates shrink like (b1 / sqrt(b2))^k: sum them until they are 1e-9 of the first one (what is cut off is
  // < 1e-8 of ONE update, i.e. ~1e-11 absolute at the reference's learning rate)
  const double r = beta1 / sqrt(beta2);
  if (!(r > 0.0) || r >= 1.0) return 4096;
  const double k = ceil(log(1e-9) / log(r));
  return static_cast<int32_t>(k < 1.0 ? 1.0 : (k > 4096.0 ? 4096.0 : k));
}

extern "C" int64_t psb_adam_sparse_workspace_bytes(const psb_adam_tensor_t* dense, int32_t n_dense,
                                                   const psb_adam_rows_t* tables, int32_t n_tables) {
  if (n_dense < 0 || n_dense > PSB_ADAM_MAX_TENSORS || n_tables < 0 || n_tables > PSB_ADAM_MAX_ROW_TABLES ||
      (n_dense > 0 && dense == nullptr) || (n_tables > 0 && tables == nullptr))
    return PSB_E_ARG;
  return (adam_chunks(dense, n_dense) + row_norm_blocks(tables, n_tables) + 4) * static_cast<int64_t>(sizeof(float));
}

extern "C" int psb_adam_sparse_step(const psb_adam_tensor_t* dense, int32_t n_dense, const psb_adam_rows_t* tables,
                                    int32_t n_tables, double lr, double beta1, double beta2, double eps,
                                    double max_grad_norm, int32_t noam, double warmup_steps, int32_t norm_given,
                                    int64_t* step_dev, float* sqnorm_dev, float* coef_hist, int64_t coef_cap,
                                    void* workspace, int64_t workspace_bytes, psb_stream_t stream) {
  if (n_dense < 0 || n_dense > PSB_ADAM_MAX_TENSORS || n_tables < 0 || n_tables > PSB_ADAM_MAX_ROW_TABLES ||
      n_dense + n_tables == 0 || step_dev == nullptr || sqnorm_dev == nullptr || workspace == nullptr ||
      (n_dense > 0 && dense == nullptr) || (n_tables > 0 && tables == nullptr))
    return PSB_E_ARG;
  if (coef_hist != nullptr && ((reinterpret_cast<uintptr_t>(coef_hist) & 7) != 0 || coef_cap <= 0)) return PSB_E_ALIGN;
  AdamTensors T;
  T.n = n_dense;
  for (int i = 0; i < n_dense; ++i) {
    if (dense[i].p == nullptr || dense[i].g == nullptr || dense[i].m == nullptr || dense[i].v == nullptr || dense[i].n <= 0)
      return PSB_E_ARG;
    T.t[i] = dense[i];
  }
  RowTables R;
  R.n = n_tables;
  int st;
  for (int i = 0; i < n_tables; ++i) {
    if ((st = check_row_table(tables[i], true)) != PSB_OK) return st;
    R.t[i] = tables[i];
  }
  const int64_t chunks = adam_chunks(dense, n_dense);
  const int64_t nblocks = row_norm_blocks(tables, n_tables);
  int64_t ublocks = 0;
  for (int i = 0; i < n_tables; ++i) ublocks += (tables[i].cap + 7) / 8;
  if (chunks + nblocks > (1ll << 30) || ublocks > (1ll << 30)) return PSB_E_DIM;
  if (workspace_bytes < (chunks + nblocks + 4) * static_cast<int64_t>(sizeof(float))) return PSB_E_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(workspace);
  if (norm_given == 2) {
    // norm and step counter were both written by the caller
  } else if (norm_given) {
    PSB_PROF("bump_step_kernel", s);
    bump_step_kernel<<<1, 1, 0, s>>>(step_dev);
    if ((st = launch_status()) != PSB_OK) return st;
  } else {
    if (chunks > 0) {
      PSB_PROF("sqnorm_partial_kernel", s);
      sqnorm_partial_kernel<<<static_cast<int>(chunks), 256, 0, s>>>(T, partial);
      if ((st = launch_status()) != PSB_OK) return st;
    }
    if (nblocks > 0) {
      PSB_PROF("sqnorm_rows_partial_kernel", s);
      sqnorm_rows_partial_kernel<<<static_cast<int>(nblocks), 256, 0, s>>>(R, partial + chunks);
      if ((st = launch_status()) != PSB_OK) return st;
    }
    PSB_PROF("sqnorm_final_kernel", s);
    sqnorm_final_kernel<<<1, 256, 0, s>>>(partial, static_cast<int>(chunks + nblocks), sqnorm_dev, step_dev);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  const AdamHyper h = make_hyper(lr, beta1, beta2, eps, 0.0, max_grad_norm, noam, warmup_steps);
  if (chunks > 0) {
    PSB_PROF("adam_kernel", s);
    adam_kernel<<<static_cast<int>(chunks), 256, 0, s>>>(T, h, sqnorm_dev, step_dev);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  // A step in which a table has no row list is a zero-gradient step for all its rows: its coefficients still go into
  // the history (block 0 writes them; a block without a table returns), or a later catch-up would skip that step.
  if (ublocks == 0 && coef_hist != nullptr) ublocks = 1;
  if (ublocks > 0) {
    PSB_PROF("adam_rows_kernel", s);
    adam_rows_kernel<<<static_cast<int>(ublocks), 256, 0, s>>>(R, h, sqnorm_dev, step_dev,
                                                              reinterpret_cast<float2*>(coef_hist), coef_cap,
                                                              psb_adam_catchup_steps(beta1, beta2));
    if ((st = launch_status()) != PSB_OK) return st;
  }
  return PSB_OK;
}

// The partial sums only (for psb_peer_norm_exchange in peer.cu, which finishes them inside its fused kernel)
namespace psb {
int sqnorm_partials(const psb_adam_tensor_t* dense, int32_t n_dense, const psb_adam_rows_t* tables, int32_t n_tables,
                    float* partial, int64_t partial_cap, int* n_partials, cudaStream_t s) {
  if (n_dense < 0 || n_dense > PSB_ADAM_MAX_TENSORS || n_tables < 0 || n_tables > PSB_ADAM_MAX_ROW_TABLES ||
      n_dense + n_tables == 0 || partial == nullptr || (n_dense > 0 && dense == nullptr) ||
      (n_tables > 0 && tables == nullptr))
    return PSB_E_ARG;
  AdamTensors T;
  T.n = n_dense;
  for (int i = 0; i < n_dense; ++i) {
    if (dense[i].g == nullptr || dense[i].n <= 0) return PSB_E_ARG;
    T.t[i] = dense[i];
  }
  RowTables R;
  R.n = n_tables;
  for (int i = 0; i < n_tables; ++i) {
    if (tables[i].rows == nullptr || tables[i].grad == nullptr || tables[i].n_rows == nullptr || tables[i].cap <= 0 ||
        tables[i].d <= 0 || (tables[i].d & 3) != 0)
      return PSB_E_ARG;
    R.t[i] = tables[i];
  }
  const int64_t chunks = adam_chunks(dense, n_dense);
  const int64_t nblocks = row_norm_blocks(tables, n_tables);
  if (chunks + nblocks > (1ll << 30)) return PSB_E_DIM;
  if (partial_cap < chunks + nblocks) return PSB_E_WORKSPACE;
  int st;
  if (chunks > 0) {
    PSB_PROF("sqnorm_partial_kernel", s);
    sqnorm_partial_kernel<<<static_cast<int>(chunks), 256, 0, s>>>(T, partial);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  if (nblocks > 0) {
    PSB_PROF("sqnorm_rows_partial_kernel", s);
    sqnorm_rows_partial_kernel<<<static_cast<int>(nblocks), 256, 0, s>>>(R, partial + chunks);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  *n_partials = static_cast<int>(chunks + nblocks);
  return PSB_OK;
}
}  // namespace psb

extern "C" int psb_grad_sqnorm_sparse(const psb_adam_tensor_t* dense, int32_t n_dense, const psb_adam_rows_t* tables,
                                      int32_t n_tables, float* sqnorm_out, void* workspace, int64_t workspace_bytes,
                                      psb_stream_t stream) {
  if (n_dense < 0 || n_dense > PSB_ADAM_MAX_TENSORS || n_tables < 0 || n_tables > PSB_ADAM_MAX_ROW_TABLES ||
      n_dense + n_tables == 0 || sqnorm_out == nullptr || workspace == nullptr || (n_dense > 0 && dense == nullptr) ||
      (n_tables > 0 && tables == nullptr))
    return PSB_E_ARG;
  AdamTensors T;
  T.n = n_dense;
  for (int i = 0; i < n_dense; ++i) {
    if (dense[i].g == nullptr || dense[i].n <= 0) return PSB_E_ARG;
    T.t[i] = dense[i];
  }
  RowTables R;
  R.n = n_tables;
  for (int i = 0; i < n_tables; ++i) {
    if (tables[i].rows == nullptr || tables[i].grad == nullptr || tables[i].n_rows == nullptr || tables[i].cap <= 0 ||
        tables[i].d <= 0 || (tables[i].d & 3) != 0)
      return PSB_E_ARG;
    R.t[i] = tables[i];
  }
  const int64_t chunks = adam_chunks(dense, n_dense);
  const int64_t nblocks = row_norm_blocks(tables, n_tables);
  if (chunks + nblocks > (1ll << 30)) return PSB_E_DIM;
  if (workspace_bytes < (chunks + nblocks + 4) * static_cast<int64_t>(sizeof(float))) return PSB_E_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(workspace);
  int st;
  if (chunks > 0) {
    PSB_PROF("sqnorm_partial_kernel", s);
    sqnorm_partial_kernel<<<static_cast<int>(chunks), 256, 0, s>>>(T, partial);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  if (nblocks > 0) {
    PSB_PROF("sqnorm_rows_partial_kernel", s);
    sqnorm_rows_partial_kernel<<<static_cast<int>(nblocks), 256, 0, s>>>(R, partial + chunks);
    if ((st = launch_status()) != PSB_OK) return st;
  }
  PSB_PROF("sqnorm_final_kernel", s);
  sqnorm_final_kernel<<<1, 256, 0, s>>>(partial, static_cast<int>(chunks + nblocks), sqnorm_out, nullptr);
  return launch_status();
}

extern "C" int psb_adam_rows_catchup(const psb_adam_rows_t* table, const int64_t* const* idx_lists,
                                     const int64_t* idx_counts, int32_t n_lists, int64_t skip_row, double lr,
                                     double beta1, double beta2, double eps, int32_t noam, double warmup_steps,
                                     const int64_t* step_dev, const float* coef_hist, int64_t coef_cap,
                                     psb_stream_t stream) {
  if (table == nullptr || step_dev == nullptr || n_lists < 0 || n_lists > PSB_ADAM_MAX_IDX_LISTS ||
      (n_lists > 0 && (idx_lists == nullptr || idx_counts == nullptr)))
    return PSB_E_ARG;
  int st = check_row_table(*table, false);
  if (st != PSB_OK) return st;
  IdxLists L;
  L.n = n_lists;
  L.start[0] = 0;
  for (int i = 0; i < n_lists; ++i) {
    if (idx_counts[i] < 0 || (idx_counts[i] > 0 && idx_lists[i] == nullptr)) return PSB_E_ARG;
    L.idx[i] = idx_lists[i];
    L.start[i + 1] = L.start[i] + idx_counts[i];
  }
  const int64_t total = n_lists > 0 ? L.start[n_lists] : table->table_rows;      // no lists: every row (flush)
  if (total == 0) return PSB_OK;
  const AdamHyper h = make_hyper(lr, beta1, beta2, eps, 0.0, 0.0, noam, warmup_steps);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PSB_PROF("adam_rows_catchup_kernel", s);
  adam_rows_catchup_kernel<<<grid_for(total, 8, 32), 256, 0, s>>>(*table, L, total, skip_row, h, step_dev,
                                                                 reinterpret_cast<const float2*>(coef_hist), coef_cap,
                                                                 psb_adam_catchup_steps(beta1, beta2));
  return launch_status();
}
