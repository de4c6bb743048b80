// Adam arithmetic shared by the optimizer kernels (optimizer.cu) and the peer-memory row fetch that brings resting
// rows up to date on the fly (peer.cu): hyper-parameters, per-step coefficients and the catch-up series of a row
// whose gradient was zero for a number of steps.
#pragma once
#include "psb_common.cuh"

namespace psb {

struct AdamHyper {  // the reference's hyper-parameters are Python doubles: 1 - beta is formed in double, then rounded
  double lr, beta1, beta2;
  float b1, b2, omb1, omb2, eps, max_norm, weight_decay;
  float l2b1;        // log2(1 - omb1) of the exact double: m decays by 1 - omb1 per zero-gradient step (lerp), not b1
  int noam;
  float warmup;
};

struct StepCoef {
  float step_size, inv_bc2_sqrt;
};

__device__ __forceinline__ StepCoef step_coef(const AdamHyper& h, int64_t step) {
  const double sd = static_cast<double>(step);
  double lr = h.lr;
  if (h.noam) lr = h.lr * fmin(1.0 / sqrt(sd), sd * pow(static_cast<double>(h.warmup), -1.5));
  const double bc1 = 1.0 - pow(h.beta1, sd);
  const double bc2 = 1.0 - pow(h.beta2, sd);
  StepCoef c;
  c.step_size = static_cast<float>(lr / bc1);
  c.inv_bc2_sqrt = static_cast<float>(1.0 / sqrt(bc2));
  return c;
}

// coefficients of step tau: from the history table when it holds them (written by the optimizer step itself),
// else recomputed (steps beyond the table's capacity)
__device__ __forceinline__ StepCoef load_coef(const AdamHyper& h, const float2* __restrict__ hist, int64_t cap,
                                              int64_t tau) {
  if (hist != nullptr && tau < cap) {
    const float2 c = hist[tau];
    StepCoef r;
    r.step_size = c.x;
    r.inv_bc2_sqrt = c.y;
    return r;
  }
  return step_coef(h, tau);
}

// Catch-up series of ONE float4 of a resting row over steps from+1 .. from+nterm (see catchup_row in optimizer.cu):
//   delta = sum_j a_j m / (b_j sqrt(v) + eps),  a_j = step_size(from + j) b1^j,  b_j = b2^(j/2) inv_bc2_sqrt(from + j)
// Warp-cooperative (all 32 lanes call it; each lane forms 32 terms' coefficients at a time and they are shuffled).
__device__ __forceinline__ float4 catchup_series4(const float4& m, const float4& v, int64_t from, int nterm,
                                                  const AdamHyper& h, const float2* __restrict__ hist, int64_t hist_cap) {
  const int lane = threadIdx.x & 31;
  const float l2b1 = h.l2b1, hl2b2 = 0.5f * log2f(h.b2);
  const float4 s = make_float4(sqrtf(v.x), sqrtf(v.y), sqrtf(v.z), sqrtf(v.w));
  float4 acc = zero4();
  for (int j0 = 0; j0 < nterm; j0 += 32) {
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
    }
  }
  return acc;
}

inline AdamHyper make_adam_hyper(double lr, double beta1, double beta2, double eps, double weight_decay,
                                 double max_grad_norm, int32_t noam, double warmup_steps) {
  AdamHyper h;
  h.lr = lr;
  h.beta1 = beta1;
  h.beta2 = beta2;
  h.b1 = static_cast<float>(beta1);
  h.b2 = static_cast<float>(beta2);
  h.omb1 = static_cast<float>(1.0 - beta1);
  h.omb2 = static_cast<float>(1.0 - beta2);
  h.l2b1 = static_cast<float>(log2(1.0 - static_cast<double>(h.omb1)));
  h.eps = static_cast<float>(eps);
  h.max_norm = static_cast<float>(max_grad_norm);
  h.weight_decay = static_cast<float>(weight_decay);
  h.noam = noam;
  h.warmup = static_cast<float>(warmup_steps);
  return h;
}

// optimizer.cu: |g|^2 partial sums of dense tensors + row lists into partial[0 .. *n_partials) (fixed order)
int sqnorm_partials(const psb_adam_tensor_t* dense, int32_t n_dense, const psb_adam_rows_t* tables, int32_t n_tables,
                    float* partial, int64_t partial_cap, int* n_partials, cudaStream_t s);

}  // namespace psb
