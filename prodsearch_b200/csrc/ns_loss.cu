// G3 / A4: fused gather + dot + bias + BCE-with-logits negative-sampling loss.
//
// One warp owns one anchor i.  For every target position j it loads the positive row
// and the k sampled-negative rows (1 + k independent LDG.128 per lane in flight), scores
// them against the anchor with warp-shuffle reductions, evaluates the loss and its
// analytic derivative, and accumulates d loss / d anchor on the fly -- every table row is
// read from HBM exactly once per use and no [n, w, 1+k, d] tensor is ever materialised.
// HBM-bound: algorithmic bytes per anchor = w * (1 + k) * d * 4 (rows) + d * 4 (anchor)
// + d * 4 (grad_anchor) (+ k * d * 8 when per-negative anchors are used).
#include "psb_common.cuh"

namespace psb {

constexpr int kMaxNeg = 16;

__device__ __forceinline__ float bce_value(float x, float t) {
  // max(x,0) - x t + log1p(exp(-|x|))     (SURVEY.md 8(a) A4)
  return fmaxf(x, 0.f) - x * t + log1pf(expf(-fabsf(x)));
}

__device__ __forceinline__ float sigmoidf_(float x) {
  // stable for both signs
  const float e = expf(-fabsf(x));
  return x >= 0.f ? 1.f / (1.f + e) : e / (1.f + e);
}

template <int C>
__global__ void __launch_bounds__(256)
ns_loss_kernel(const float4* __restrict__ anchor_a, const float4* __restrict__ anchor_b,
               const float4* __restrict__ table, int64_t table_rows, int d4,
               const float* __restrict__ bias, const int64_t* __restrict__ pos_idx,
               const int64_t* __restrict__ neg_idx, const uint8_t* __restrict__ mask, int64_t pad_idx,
               const float* __restrict__ neg_weight, float pos_weight, int64_t n, int w, int k,
               float* __restrict__ loss, float* __restrict__ coef_pos, float* __restrict__ coef_neg,
               float4* __restrict__ grad_a, float4* __restrict__ grad_b) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  const int64_t warp = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  for (int64_t i = warp; i < n; i += nwarps) {
    // number of valid target positions (the masked-mean denominator)
    int cnt = 0;
    for (int j0 = 0; j0 < w; j0 += 32) {
      const int j = j0 + lane;
      bool valid = false;
      if (j < w) valid = mask != nullptr ? mask[i * w + j] != 0 : (pad_idx < 0 || pos_idx[i * w + j] != pad_idx);
      cnt += __popc(__ballot_sync(kFull, valid));
    }
    const float denom = static_cast<float>(cnt > 0 ? cnt : 1);

    float4 a[C], ga[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const int col = lane + 32 * c;
      a[c] = col < d4 ? anchor_a[i * d4 + col] : zero4();
      ga[c] = zero4();
    }
    float loss_acc = 0.f;
    for (int j = 0; j < w; ++j) {
      const int64_t pj = pos_idx[i * w + j];
      const bool valid = mask != nullptr ? mask[i * w + j] != 0 : (pad_idx < 0 || pj != pad_idx);
      const float m = valid ? 1.f : 0.f;
      // positive (slot 0) and negatives (slots 1..k), processed in groups of 4 rows in flight
      float lsum = 0.f;
      for (int s0 = 0; s0 <= k; s0 += 4) {
        int64_t r[4];
        float4 row[4][C];
        float4 anc[4][C];
        float part[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int s = s0 + u;
          r[u] = -1;
          if (s <= k) r[u] = s == 0 ? pj : neg_idx[(i * w + j) * k + (s - 1)];
          if (r[u] < 0 || r[u] >= table_rows) r[u] = -1;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int s = s0 + u;
#pragma unroll
          for (int c = 0; c < C; ++c) {
            const int col = lane + 32 * c;
            row[u][c] = (r[u] >= 0 && col < d4) ? ldg_row4(table + r[u] * d4 + col) : zero4();
            if (anchor_b != nullptr && s >= 1 && s <= k)
              anc[u][c] = col < d4 ? anchor_b[(i * k + (s - 1)) * d4 + col] : zero4();
            else
              anc[u][c] = a[c];
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          float t = 0.f;
#pragma unroll
          for (int c = 0; c < C; ++c) t += dot4(anc[u][c], row[u][c]);
          part[u] = t;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) part[u] = warp_sum(part[u]);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int s = s0 + u;
          if (s > k) continue;
          float x = part[u];
          if (bias != nullptr && r[u] >= 0) x += bias[r[u]];
          const float t = s == 0 ? 1.f : 0.f;
          const float wt = s == 0 ? pos_weight : (neg_weight != nullptr ? neg_weight[i * k + (s - 1)] : 1.f);
          lsum += wt * bce_value(x, t);
          const float g = m * wt * (sigmoidf_(x) - t) / denom;
          if (lane == 0) {
            if (s == 0) coef_pos[i * w + j] = g;
            else coef_neg[(i * w + j) * k + (s - 1)] = g;
          }
          if (anchor_b != nullptr && s >= 1) {
#pragma unroll
            for (int c = 0; c < C; ++c) {
              const int col = lane + 32 * c;
              if (col < d4) {
                float4 o = zero4();
                fma4(o, g, row[u][c]);
                grad_b[(i * k + (s - 1)) * d4 + col] = o;
              }
            }
          } else {
#pragma unroll
            for (int c = 0; c < C; ++c) fma4(ga[c], g, row[u][c]);
          }
        }
      }
      loss_acc += m * lsum;
    }
    if (lane == 0) loss[i] = loss_acc / denom;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const int col = lane + 32 * c;
      if (col < d4) grad_a[i * d4 + col] = ga[c];
    }
  }
}

// Fast path for d <= 128 and 1 + k <= 8: all rows of one target position are loaded before any
// arithmetic (up to 8 independent 512 B row reads per warp), the 8 partial dot products are reduced
// together with a halving butterfly (9 shuffles instead of 40), and each score's loss / gradient is
// evaluated by the lanes that hold its sum instead of redundantly by all 32.
template <bool HAS_B>
__global__ void __launch_bounds__(256, HAS_B ? 2 : 3)
ns_loss_fast_kernel(const float4* __restrict__ anchor_a, const float4* __restrict__ anchor_b,
                    const float4* __restrict__ table, int64_t table_rows, int d4,
                    const float* __restrict__ bias, const int64_t* __restrict__ pos_idx,
                    const int64_t* __restrict__ neg_idx, const uint8_t* __restrict__ mask, int64_t pad_idx,
                    const float* __restrict__ neg_weight, float pos_weight, int64_t n, int w, int k,
                    float* __restrict__ loss, float* __restrict__ coef_pos, float* __restrict__ coef_neg,
                    float4* __restrict__ grad_a, float4* __restrict__ grad_b) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  const int64_t warp = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const bool col_ok = lane < d4;
  // which score this lane owns after the butterfly, and the lane that is its designated writer
  const int my_s = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
  const bool writer = (lane & 3) == 0;
  // Software pipeline over (anchor, position): the index / weight / mask words of the NEXT position (and the
  // anchor row + valid-count predicate of the next anchor) are requested right after the current position's row
  // loads, so one anchor costs one dependent HBM round trip (its rows) instead of three (count, indices, rows).
  auto fetch_meta = [&](int64_t i, int j, int64_t& idx_o, float& wt_o, uint8_t& mk_o) {
    idx_o = -1;
    wt_o = 0.f;
    if (lane <= k) {
      idx_o = lane == 0 ? pos_idx[i * w + j] : neg_idx[(i * w + j) * k + (lane - 1)];
      wt_o = lane == 0 ? pos_weight : (neg_weight != nullptr ? neg_weight[i * k + (lane - 1)] : 1.f);
    }
    mk_o = mask != nullptr ? mask[i * w + j] : static_cast<uint8_t>(1);
  };
  auto count_pred = [&](int64_t i) {  // lane j < w: is position j of anchor i a valid target (w <= 32)
    bool valid = false;
    if (lane < w) valid = mask != nullptr ? mask[i * w + lane] != 0 : (pad_idx < 0 || pos_idx[i * w + lane] != pad_idx);
    return valid;
  };
  if (warp >= n) return;
  float4 a_n = col_ok ? anchor_a[warp * d4 + lane] : zero4();
  bool cv_n = w <= 32 ? count_pred(warp) : false;
  int64_t idx_n;
  float wt_n;
  uint8_t mk_n;
  fetch_meta(warp, 0, idx_n, wt_n, mk_n);
  for (int64_t i = warp; i < n; i += nwarps) {
    int cnt = 0;
    if (w <= 32) {
      cnt = __popc(__ballot_sync(kFull, cv_n));
    } else {
      for (int j0 = 0; j0 < w; j0 += 32) {
        const int j = j0 + lane;
        bool valid = false;
        if (j < w) valid = mask != nullptr ? mask[i * w + j] != 0 : (pad_idx < 0 || pos_idx[i * w + j] != pad_idx);
        cnt += __popc(__ballot_sync(kFull, valid));
      }
    }
    const float denom = static_cast<float>(cnt > 0 ? cnt : 1);
    const float4 a = a_n;
    const int64_t i_next = i + nwarps;
    float4 ga = zero4();
    float loss_acc = 0.f;
    for (int j = 0; j < w; ++j) {
      // lane s <= k holds the index / weight of score s (fetched one position ahead)
      int64_t myidx = idx_n;
      float mybias = 0.f;
      const float mywt = wt_n;
      const uint8_t mk = mk_n;
      const int64_t pj = __shfl_sync(kFull, myidx, 0);
      const bool valid = mask != nullptr ? mk != 0 : (pad_idx < 0 || pj != pad_idx);
      if (myidx < 0 || myidx >= table_rows) myidx = -1;
      if (bias != nullptr && myidx >= 0) mybias = bias[myidx];
      float4 row[8];
#pragma unroll
      for (int s = 0; s < 8; ++s) {
        const int64_t r = __shfl_sync(kFull, myidx, s);
        row[s] = (r >= 0 && col_ok) ? ldg_row4(table + r * d4 + lane) : zero4();
      }
      if (j + 1 < w) {
        fetch_meta(i, j + 1, idx_n, wt_n, mk_n);
      } else if (i_next < n) {
        fetch_meta(i_next, 0, idx_n, wt_n, mk_n);
        a_n = col_ok ? anchor_a[i_next * d4 + lane] : zero4();
        if (w <= 32) cv_n = count_pred(i_next);
      }
      float v[8];
#pragma unroll
      for (int s = 0; s < 8; ++s) {
        float4 anc = a;
        if (HAS_B && s >= 1 && s <= k && col_ok) anc = anchor_b[(i * k + (s - 1)) * d4 + lane];
        v[s] = dot4(anc, row[s]);
      }
      // halving butterfly: 8 values x 32 lanes -> lane L holds the full sum of value my_s
      float u[4], t2[2];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float mine = (lane & 16) ? v[t + 4] : v[t];
        const float other = (lane & 16) ? v[t] : v[t + 4];
        u[t] = mine + __shfl_xor_sync(kFull, other, 16);
      }
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const float mine = (lane & 8) ? u[t + 2] : u[t];
        const float other = (lane & 8) ? u[t] : u[t + 2];
        t2[t] = mine + __shfl_xor_sync(kFull, other, 8);
      }
      float z;
      {
        const float mine = (lane & 4) ? t2[1] : t2[0];
        const float other = (lane & 4) ? t2[0] : t2[1];
        z = mine + __shfl_xor_sync(kFull, other, 4);
      }
      z += __shfl_xor_sync(kFull, z, 2);
      z += __shfl_xor_sync(kFull, z, 1);
      const float b_s = __shfl_sync(kFull, mybias, my_s);
      const float wt = __shfl_sync(kFull, mywt, my_s);
      const float x = z + b_s;
      const float tgt = my_s == 0 ? 1.f : 0.f;
      const float m = valid ? 1.f : 0.f;
      float g = 0.f, lterm = 0.f;
      if (my_s <= k) {
        g = m * wt * (sigmoidf_(x) - tgt) / denom;
        if (writer) {
          lterm = wt * bce_value(x, tgt);
          if (my_s == 0) coef_pos[i * w + j] = g;
          else coef_neg[(i * w + j) * k + (my_s - 1)] = g;
        }
      }
      loss_acc += m * warp_sum(lterm);
#pragma unroll
      for (int s = 0; s < 8; ++s) {
        const int holder = ((s >> 2) & 1) * 16 + ((s >> 1) & 1) * 8 + (s & 1) * 4;
        const float gs = __shfl_sync(kFull, g, holder);
        if (HAS_B && s >= 1) {
          if (s <= k && col_ok) {
            float4 o = zero4();
            fma4(o, gs, row[s]);
            grad_b[(i * k + (s - 1)) * d4 + lane] = o;
          }
        } else {
          fma4(ga, gs, row[s]);   // gs == 0 for s > k
        }
      }
    }
    if (lane == 0) loss[i] = loss_acc / denom;
    if (col_ok) grad_a[i * d4 + lane] = ga;
  }
}

// w == 1 (one target position per anchor: the TEM score/loss tail, item_to_words and PV with pv_window_size 1):
// every position is its own anchor, the masked-mean denominator is 1, and the kernel is a pure stream of
// (anchor row, 1 + k table rows) reads.  NR = rows handled per anchor (1 + k <= NR; 6 for the reference's 5
// negatives); row ids travel through the shuffles as int32.  One row buffer: requesting the next anchor's rows
// into a second buffer before evaluating the current one measured 0.69 of HBM peak against 0.85 for this form on
// the 16M-row table (profiles/r01i_ab.jsonl), because its 103 registers drop it to 2 CTAs/SM.
template <bool HAS_B, int NR>
__global__ void __launch_bounds__(256, HAS_B ? 2 : 3)
ns_loss_w1_kernel(const float4* __restrict__ anchor_a, const float4* __restrict__ anchor_b,
                  const float4* __restrict__ table, int64_t table_rows, int d4,
                  const float* __restrict__ bias, const int64_t* __restrict__ pos_idx,
                  const int64_t* __restrict__ neg_idx, const uint8_t* __restrict__ mask, int64_t pad_idx,
                  const float* __restrict__ neg_weight, float pos_weight, int64_t n, int k,
                  float* __restrict__ loss, float* __restrict__ coef_pos, float* __restrict__ coef_neg,
                  float4* __restrict__ grad_a, float4* __restrict__ grad_b, int a_stride = 1, int b_stride = -1,
                  float grad_scale = 1.f) {
  // Anchor layout: anchor_a row of anchor i at row i * a_stride, anchor_b row of (i, c) at row i * b_stride + c (the
  // gradient outputs use the same layout).  Defaults (1, k): two packed matrices [n, d] and [n * k, d].  The TEM tail
  // reads / writes the encoder's [n, 1 + k, d] block in place: a_stride = b_stride = 1 + k, anchor_b = block + d.
  // grad_scale multiplies coefficients and anchor gradients (the 1 / n of the batch mean).
  if (b_stride < 0) b_stride = k;
  pdl_trigger();   // (TEM tail: launched programmatically behind the encoder's tail kernel, and the loss combination behind it)
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int64_t nw = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  int64_t i = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= n) return;
  const bool col_ok = lane < d4;
  // which score this lane owns after the butterfly, and the lane that is its designated writer
  const int my_s = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
  const bool writer = (lane & 3) == 0;
  const float tgt = my_s == 0 ? 1.f : 0.f;
  struct Meta {
    int idx;      // lane s <= k: table row of score s (-1: out of range / no such score)
    float wt;     // lane s <= k: loss weight of score s
    bool valid;   // lane 0: the target position counts (mask / pad)
  };
  auto fetch = [&](int64_t a_i, Meta& m) {
    int64_t r = -1;
    m.wt = 0.f;
    if (lane <= k) {
      r = lane == 0 ? pos_idx[a_i] : neg_idx[a_i * k + (lane - 1)];
      m.wt = lane == 0 ? pos_weight : (neg_weight != nullptr ? neg_weight[a_i * k + (lane - 1)] : 1.f);
    }
    m.valid = mask != nullptr ? mask[a_i] != 0 : (pad_idx < 0 || r != pad_idx);
    m.idx = (r < 0 || r >= table_rows) ? -1 : static_cast<int>(r);
  };
  auto issue = [&](const Meta& m, int64_t a_i, float4 (&row)[NR], float4& a, float& bias_v) {
    a = col_ok ? anchor_a[a_i * a_stride * d4 + lane] : zero4();
    bias_v = (bias != nullptr && m.idx >= 0) ? bias[m.idx] : 0.f;
#pragma unroll
    for (int s = 0; s < NR; ++s) {
      const int r = __shfl_sync(kFull, m.idx, s);
      row[s] = (r >= 0 && col_ok) ? ldg_row4(table + static_cast<int64_t>(r) * d4 + lane) : zero4();
    }
  };
  auto compute = [&](const Meta& m, int64_t a_i, const float4 (&row)[NR], const float4& a, float bias_v) {
    float v[8];
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      if (s < NR) {
        float4 anc = a;
        if (HAS_B && s >= 1 && s <= k && col_ok) anc = anchor_b[(a_i * b_stride + (s - 1)) * d4 + lane];
        v[s] = dot4(anc, row[s]);
      } else {
        v[s] = 0.f;
      }
    }
    // halving butterfly: 8 values x 32 lanes -> lane L holds the full sum of value my_s
    float u[4], t2[2];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float mine = (lane & 16) ? v[t + 4] : v[t];
      const float other = (lane & 16) ? v[t] : v[t + 4];
      u[t] = mine + __shfl_xor_sync(kFull, other, 16);
    }
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const float mine = (lane & 8) ? u[t + 2] : u[t];
      const float other = (lane & 8) ? u[t] : u[t + 2];
      t2[t] = mine + __shfl_xor_sync(kFull, other, 8);
    }
    float z;
    {
      const float mine = (lane & 4) ? t2[1] : t2[0];
      const float other = (lane & 4) ? t2[0] : t2[1];
      z = mine + __shfl_xor_sync(kFull, other, 4);
    }
    z += __shfl_xor_sync(kFull, z, 2);
    z += __shfl_xor_sync(kFull, z, 1);
    const float x = z + __shfl_sync(kFull, bias_v, my_s);
    const float wt = __shfl_sync(kFull, m.wt, my_s);
    const float mv = __shfl_sync(kFull, m.valid ? 1.f : 0.f, 0);
    float g = 0.f, lterm = 0.f;
    if (my_s <= k) {
      g = grad_scale * (mv * wt * (sigmoidf_(x) - tgt));   // masked-mean denominator is 1 when w == 1
      if (writer) {
        lterm = wt * bce_value(x, tgt);
        if (my_s == 0) coef_pos[a_i] = g;
        else coef_neg[a_i * k + (my_s - 1)] = g;
      }
    }
    const float lsum = mv * warp_sum(lterm);
    float4 ga = zero4();
#pragma unroll
    for (int s = 0; s < NR; ++s) {
      const int holder = ((s >> 2) & 1) * 16 + ((s >> 1) & 1) * 8 + (s & 1) * 4;
      const float gs = __shfl_sync(kFull, g, holder);
      if (HAS_B && s >= 1) {
        if (s <= k && col_ok) {
          float4 o = zero4();
          fma4(o, gs, row[s]);
          grad_b[(a_i * b_stride + (s - 1)) * d4 + lane] = o;
        }
      } else {
        fma4(ga, gs, row[s]);   // gs == 0 for s > k
      }
    }
    if (lane == 0) loss[a_i] = lsum;
    if (col_ok) grad_a[a_i * a_stride * d4 + lane] = ga;
  };

  Meta mn;
  fetch(i, mn);
  for (; i < n; i += nw) {
    const Meta m = mn;
    float4 row[NR], a;
    float bv;
    issue(m, i, row, a, bv);
    if (i + nw < n) fetch(i + nw, mn);
    compute(m, i, row, a, bv);
  }
}

// scores[i, c] = <anchor[i], table[idx[i, c]]> (+ bias[idx[i, c]]): the candidate scoring of
// test_dotproduct (item_transformer.py:141-145).  One warp per query, 4 candidate rows in flight.
template <int C>
__global__ void __launch_bounds__(256)
score_rows_kernel(const float4* __restrict__ anchor, const float4* __restrict__ table, int64_t table_rows, int d4,
                  const float* __restrict__ bias, const int64_t* __restrict__ idx, int64_t n, int c_per,
                  float* __restrict__ scores) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  const int64_t warp = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int groups = (c_per + 31) / 32;   // a warp handles 32 candidates of one query at a time
  for (int64_t item = warp; item < n * groups; item += nwarps) {
    const int64_t i = item / groups;
    const int c0 = static_cast<int>(item % groups) * 32;
    float4 a[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const int col = lane + 32 * c;
      a[c] = col < d4 ? anchor[i * d4 + col] : zero4();
    }
    const int cn = min(32, c_per - c0);
    int64_t my = -1;
    if (lane < cn) {
      my = idx[i * c_per + c0 + lane];
      if (my < 0 || my >= table_rows) my = -1;
    }
    float mine = 0.f;
    for (int j = 0; j < cn; j += 4) {
      int64_t r[4];
      float part[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) r[u] = __shfl_sync(kFull, my, min(j + u, 31));
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float t = 0.f;
        if (j + u < cn && r[u] >= 0) {
#pragma unroll
          for (int c = 0; c < C; ++c) {
            const int col = lane + 32 * c;
            if (col < d4) t += dot4(a[c], ldg_row4(table + r[u] * d4 + col));
          }
        }
        part[u] = t;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float t = warp_sum(part[u]);
        if (lane == j + u) mine = t;
      }
    }
    if (lane < cn) scores[i * c_per + c0 + lane] = mine + ((bias != nullptr && my >= 0) ? bias[my] : 0.f);
  }
}

// loss = mean(ps_rows) + mean(il_rows) with fixed-order sums (one CTA); the running sums the trainer reads
// (model.ps_loss / item_loss, trainer.py:88-98) are advanced in the same launch.
__global__ void __launch_bounds__(256) tem_loss_finish_kernel(const float* __restrict__ ps_rows,
                                                              const float* __restrict__ il_rows, int n_ps, int n_il,
                                                              float* __restrict__ loss_out, float* __restrict__ acc_ps,
                                                              float* __restrict__ acc_il) {
  __shared__ float wa[8], wb[8];
  pdl_wait();
  float a = 0.f, b = 0.f;
  for (int i = threadIdx.x; i < n_ps; i += 256) a += ps_rows[i];
  for (int i = threadIdx.x; i < n_il; i += 256) b += il_rows[i];
  a = warp_sum(a);
  b = warp_sum(b);
  if ((threadIdx.x & 31) == 0) {
    wa[threadIdx.x >> 5] = a;
    wb[threadIdx.x >> 5] = b;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float sa = 0.f, sb = 0.f;
    for (int w = 0; w < 8; ++w) {
      sa += wa[w];
      sb += wb[w];
    }
    const float ps = sa / static_cast<float>(n_ps > 0 ? n_ps : 1);
    const float il = n_il > 0 ? sb / static_cast<float>(n_il) : 0.f;
    *loss_out = ps + il;
    if (acc_ps != nullptr) *acc_ps += ps;
    if (acc_il != nullptr) *acc_il += il;
  }
}

}  // namespace psb

using namespace psb;

extern "C" int psb_tem_loss_fwd(const float* enc_out, const float* table, int64_t table_rows, int64_t d,
                                const float* bias, const int64_t* pos_idx, const int64_t* neg_idx, float pos_weight,
                                int64_t n, int64_t k, float grad_scale, float* loss_rows, float* coef_pos,
                                float* coef_neg, float* grad_enc_out, psb_stream_t stream) {
  int st = check_table_args(table, table_rows, d);
  if (st != PSB_OK) return st;
  if (n < 0 || k < 1 || k > 7 || d > 128) return PSB_E_DIM;
  if (n == 0) return PSB_OK;
  if (enc_out == nullptr || pos_idx == nullptr || neg_idx == nullptr || loss_rows == nullptr || coef_pos == nullptr ||
      coef_neg == nullptr || grad_enc_out == nullptr)
    return PSB_E_ARG;
  if (misaligned16(enc_out) || misaligned16(grad_enc_out)) return PSB_E_ALIGN;
  if (table_rows >= (1ll << 31)) return PSB_E_DIM;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int d4 = static_cast<int>(d / 4);
  const int C = static_cast<int>(k) + 1;
  const int gridf = grid_for(n, 8, 32);
  const float4* a4 = reinterpret_cast<const float4*>(enc_out);
  float4* g4 = reinterpret_cast<float4*>(grad_enc_out);
  PSB_PROF("ns_loss_w1_kernel", s);
#define PSB_TEM_LAUNCH(NR)                                                                                          \
  {                                                                                                                 \
    const cudaError_t le = launch_pdl(ns_loss_w1_kernel<true, NR>, dim3(gridf), dim3(256), 0, s, a4, a4 + d4,         \
                                      reinterpret_cast<const float4*>(table), table_rows, d4, bias, pos_idx, neg_idx, \
                                      nullptr, -1, nullptr, pos_weight, n, static_cast<int>(k), loss_rows, coef_pos,  \
                                      coef_neg, g4, g4 + d4, C, C, grad_scale);                                       \
    if (le != cudaSuccess) return static_cast<int>(le);                                                               \
  }
  if (k <= 5) PSB_TEM_LAUNCH(6) else PSB_TEM_LAUNCH(8)
#undef PSB_TEM_LAUNCH
  return launch_status();
}

extern "C" int psb_tem_loss_finish(const float* ps_rows, const float* il_rows, int64_t n_ps, int64_t n_il,
                                   float* loss_out, float* acc_ps, float* acc_il, psb_stream_t stream) {
  if (ps_rows == nullptr || loss_out == nullptr || n_ps <= 0 || n_il < 0 || (n_il > 0 && il_rows == nullptr) ||
      n_ps > (1 << 30) || n_il > (1 << 30))
    return PSB_E_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PSB_PROF("tem_loss_finish_kernel", s);
  {
    const cudaError_t le = launch_pdl(tem_loss_finish_kernel, dim3(1), dim3(256), 0, s, ps_rows, il_rows, static_cast<int>(n_ps),
                                      static_cast<int>(n_il), loss_out, acc_ps, acc_il);
    if (le != cudaSuccess) return static_cast<int>(le);
  }
  return launch_status();
}

extern "C" int psb_score_rows(const float* anchor, const float* table, int64_t table_rows, int64_t d,
                              const float* bias, const int64_t* idx, int64_t n, int64_t c_per, float* scores,
                              psb_stream_t stream) {
  int st = check_table_args(table, table_rows, d);
  if (st != PSB_OK) return st;
  if (n < 0 || c_per <= 0) return PSB_E_ARG;
  if (n == 0) return PSB_OK;
  if (anchor == nullptr || idx == nullptr || scores == nullptr) return PSB_E_ARG;
  if (misaligned16(anchor)) return PSB_E_ALIGN;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int d4 = static_cast<int>(d / 4);
  const int grid = grid_for(n * ((c_per + 31) / 32), 8);
#define PSB_SC_LAUNCH(C)                                                                                     \
  score_rows_kernel<C><<<grid, 256, 0, s>>>(reinterpret_cast<const float4*>(anchor),                         \
                                            reinterpret_cast<const float4*>(table), table_rows, d4, bias, idx, n, \
                                            static_cast<int>(c_per), scores)
  PSB_PROF("score_rows_kernel", s);
  if (d4 <= 32) PSB_SC_LAUNCH(1);
  else if (d4 <= 64) PSB_SC_LAUNCH(2);
  else PSB_SC_LAUNCH(4);
#undef PSB_SC_LAUNCH
  return launch_status();
}

extern "C" int psb_ns_loss_fwd(const float* anchor_a, const float* anchor_b, const float* table,
                               int64_t table_rows, int64_t d, const float* bias, const int64_t* pos_idx,
                               const int64_t* neg_idx, const uint8_t* mask, int64_t pad_idx,
                               const float* neg_weight, float pos_weight, int64_t n, int64_t w, int64_t k,
                               float* loss, float* coef_pos, float* coef_neg, float* grad_anchor_a,
                               float* grad_anchor_b, psb_stream_t stream) {
  int st = check_table_args(table, table_rows, d);
  if (st != PSB_OK) return st;
  if (n < 0 || w <= 0 || k < 0 || k > kMaxNeg) return k > kMaxNeg ? PSB_E_DIM : PSB_E_ARG;
  if (n == 0) return PSB_OK;
  if (anchor_a == nullptr || pos_idx == nullptr || (k > 0 && neg_idx == nullptr) || loss == nullptr ||
      coef_pos == nullptr || (k > 0 && coef_neg == nullptr) || grad_anchor_a == nullptr)
    return PSB_E_ARG;
  if (anchor_b != nullptr && (w != 1 || grad_anchor_b == nullptr)) return PSB_E_ARG;
  if (misaligned16(anchor_a) || misaligned16(anchor_b) || misaligned16(grad_anchor_a) ||
      misaligned16(grad_anchor_b))
    return PSB_E_ALIGN;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int grid = grid_for(n, 8);
  const int d4 = static_cast<int>(d / 4);
#define PSB_NS_LAUNCH(C)                                                                                   \
  ns_loss_kernel<C><<<grid, 256, 0, s>>>(                                                                  \
      reinterpret_cast<const float4*>(anchor_a), reinterpret_cast<const float4*>(anchor_b),                \
      reinterpret_cast<const float4*>(table), table_rows, d4, bias, pos_idx, neg_idx, mask, pad_idx,       \
      neg_weight, pos_weight, n, static_cast<int>(w), static_cast<int>(k), loss, coef_pos, coef_neg,       \
      reinterpret_cast<float4*>(grad_anchor_a), reinterpret_cast<float4*>(grad_anchor_b))
  if (w == 1 && d4 <= 32 && k <= 7 && table_rows < (1ll << 31)) {
    const int gridf = grid_for(n, 8, 32);
    PSB_PROF("ns_loss_w1_kernel", s);
#define PSB_W1_LAUNCH(HASB, NR)                                                                              \
  ns_loss_w1_kernel<HASB, NR><<<gridf, 256, 0, s>>>(                                                          \
      reinterpret_cast<const float4*>(anchor_a), reinterpret_cast<const float4*>(anchor_b),                  \
      reinterpret_cast<const float4*>(table), table_rows, d4, bias, pos_idx, neg_idx, mask, pad_idx, neg_weight, \
      pos_weight, n, static_cast<int>(k), loss, coef_pos, coef_neg, reinterpret_cast<float4*>(grad_anchor_a),  \
      reinterpret_cast<float4*>(grad_anchor_b))
    if (anchor_b != nullptr) {
      if (k <= 5) PSB_W1_LAUNCH(true, 6); else PSB_W1_LAUNCH(true, 8);
    } else {
      if (k <= 5) PSB_W1_LAUNCH(false, 6); else PSB_W1_LAUNCH(false, 8);
    }
#undef PSB_W1_LAUNCH
  } else if (d4 <= 32 && k <= 7) {
    const int gridf = grid_for(n, 8, 32);
    PSB_PROF("ns_loss_fast_kernel", s);
    if (anchor_b != nullptr)
      ns_loss_fast_kernel<true><<<gridf, 256, 0, s>>>(
          reinterpret_cast<const float4*>(anchor_a), reinterpret_cast<const float4*>(anchor_b),
          reinterpret_cast<const float4*>(table), table_rows, d4, bias, pos_idx, neg_idx, mask, pad_idx, neg_weight,
          pos_weight, n, static_cast<int>(w), static_cast<int>(k), loss, coef_pos, coef_neg,
          reinterpret_cast<float4*>(grad_anchor_a), reinterpret_cast<float4*>(grad_anchor_b));
    else
      ns_loss_fast_kernel<false><<<gridf, 256, 0, s>>>(
          reinterpret_cast<const float4*>(anchor_a), reinterpret_cast<const float4*>(anchor_b),
          reinterpret_cast<const float4*>(table), table_rows, d4, bias, pos_idx, neg_idx, mask, pad_idx, neg_weight,
          pos_weight, n, static_cast<int>(w), static_cast<int>(k), loss, coef_pos, coef_neg,
          reinterpret_cast<float4*>(grad_anchor_a), reinterpret_cast<float4*>(grad_anchor_b));
  }
  else if (d4 <= 32) { PSB_PROF("ns_loss_kernel", s); PSB_NS_LAUNCH(1); }
  else if (d4 <= 64) { PSB_PROF("ns_loss_kernel", s); PSB_NS_LAUNCH(2); }
  else { PSB_PROF("ns_loss_kernel", s); PSB_NS_LAUNCH(4); }
#undef PSB_NS_LAUNCH
  return launch_status();
}
