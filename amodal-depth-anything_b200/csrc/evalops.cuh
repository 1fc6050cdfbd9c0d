// Per-sample evaluation post-ops of the reference's validation loop on the device (discriminative_trainer.py:542-613;
// SURVEY.md section 8 row f3): nearest resize of the prediction to the ground-truth size (:542), least-squares scale/shift
// alignment against the observation over the visible mask (src/util/alignment.py:7-54, solved as 2x2 normal equations
// instead of np.linalg.lstsq) and the ten masked metrics of src/util/metric.py:37-161 for the raw and the aligned
// prediction (:584-613). The reference does this on the host with a .cpu().numpy() round trip per sample.
// Per-pixel terms are evaluated in fp32 like the torch expressions; sums are accumulated in fp64.
//
// One kernel runs a batch of samples of any sizes: sample b is one cluster of kEvalCluster CTAs (blockIdx.y = b). The
// pixels a thread visits and the order in which the partial sums are combined depend only on the sample's own geometry,
// never on B or b, and there are no atomics: a sample's row is the same bits in any batch and on every run.
// eval_accumulate_kernel then folds rows into per-bucket dataset sums in row order.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/amodal_b200.h"
#include "ptx.cuh"

namespace ada {

constexpr int kEvalCluster = 8;      // CTAs per sample: the largest portable cluster size
constexpr int kEvalThreads = 512;
constexpr int kEvalWarps = kEvalThreads / 32;
constexpr int kEvalAlignSums = 5;    // n, sum p, sum p^2, sum g, sum p g          (visible mask)
constexpr int kEvalMetricSums = 10;  // absrel, sqrel, se, sle, sl, l10, d1, d2, d3, inv-se (object mask), x2 variants
constexpr int kEvalObjectSums = 1 + 2 * kEvalMetricSums;  // object pixels, then the metric sums of pred and aligned
constexpr int kEvalOut = 24;  // scale, shift, 10 metrics (pred), 10 metrics (aligned), n_visible, n_object
constexpr int kEvalAccSlots = 2 + 2 * kEvalMetricSums;  // per group: n_used, n_skipped, 20 metric sums

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  return v;
}

struct EvalSample {
  const float* pred;  // [h, w] network output
  int h, w;
  const float* gt;    // [H, W] depth_raw_ts
  const float* obs;   // [H, W] depth_observation
  const uint8_t* visible;  // [H, W]
  const uint8_t* object;   // [H, W]
  int H, W;
};

// Sample blockIdx.y: its row of the descriptor table, or, without a table (ada_eval_sample), `one`.
__device__ __forceinline__ EvalSample eval_sample_at(const float* pred, const uint8_t* src,
                                                     const ada_eval_desc* __restrict__ table, const EvalSample& one) {
  if (!table) return one;
  const ada_eval_desc d = table[blockIdx.y];
  return EvalSample{pred + d.pred, static_cast<int>(d.h), static_cast<int>(d.w),
                    reinterpret_cast<const float*>(src + d.gt), reinterpret_cast<const float*>(src + d.obs),
                    src + d.visible, src + d.object, static_cast<int>(d.H), static_cast<int>(d.W)};
}

__device__ __forceinline__ float eval_pred_at(const EvalSample& a, int i) {
  const int y = i / a.W, x = i - y * a.W;
  const int sy = min(static_cast<int>(floorf(static_cast<float>(y) * (static_cast<float>(a.h) / static_cast<float>(a.H)))), a.h - 1);
  const int sx = min(static_cast<int>(floorf(static_cast<float>(x) * (static_cast<float>(a.w) / static_cast<float>(a.W)))), a.w - 1);
  return a.pred[sy * a.w + sx];
}

__device__ __forceinline__ void eval_scale_shift(const double* s, float& scale, float& shift) {
  const double n = s[0], sp = s[1], spp = s[2], sg = s[3], spg = s[4];
  const double det = n * spp - sp * sp;
  const double sc = (n * spg - sp * sg) / det;
  scale = static_cast<float>(sc);
  shift = static_cast<float>((sg - sc * sp) / n);
}

// The metric terms of one object pixel: prediction p (already resized), ground truth g. s[v * kEvalMetricSums + k] for
// v = 0 the prediction, v = 1 the aligned prediction p * scale + shift.
__device__ __forceinline__ void eval_metric_terms(float p, float g, float scale, float shift, double* s) {
  const float t = __fadd_rn(g, 1e-5f);                                         // depth_raw_ts + 1e-5 (:587)
  const float o2[2] = {__fadd_rn(p, 1e-5f), __fadd_rn(__fadd_rn(__fmul_rn(p, scale), shift), 1e-5f)};  // pred / aligned
  const float lt = logf(t), l10t = log10f(t), it = 1.0f / t;
#pragma unroll
  for (int v = 0; v < 2; ++v) {
    double* sv = s + v * kEvalMetricSums;
    const float o = o2[v];
    const float d = o - t, ad = fabsf(d);
    const float ld = logf(o) - lt;
    const float r = fmaxf(o / t, t / o);
    const float id = 1.0f / o - it;
    sv[0] += ad / t;                     // abs_relative_difference  metric.py:37-47
    sv[1] += (ad * ad) / t;              // squared_relative_difference :50-62
    sv[2] += static_cast<double>(d) * d;        // rmse_linear :65-77
    sv[3] += static_cast<double>(ld) * ld;      // rmse_log :80-90, silog first term :149-158
    sv[4] += ld;                         // silog second term
    sv[5] += fabsf(log10f(o) - l10t);    // log10 :93-101
    sv[6] += (r < 1.25f) ? 1.0 : 0.0;    // delta1_acc :105-121 (1.25, 1.25**2, 1.25**3 as Python floats)
    sv[7] += (r < 1.5625f) ? 1.0 : 0.0;
    sv[8] += (r < 1.953125f) ? 1.0 : 0.0;
    sv[9] += static_cast<double>(id) * id;      // i_rmse :132-145
  }
}

// The 24 output doubles from the visible-mask sums a[kEvalAlignSums] and the object-mask sums m[kEvalObjectSums].
__device__ __forceinline__ void eval_finalize(const double* a, const double* m, double* out) {
  float scale, shift;
  eval_scale_shift(a, scale, shift);
  out[0] = scale;
  out[1] = shift;
  const double n = m[0];
  for (int v = 0; v < 2; ++v) {
    const double* s = m + 1 + v * kEvalMetricSums;
    double* o = out + 2 + v * kEvalMetricSums;
    o[0] = s[0] / n;
    o[1] = s[1] / n;
    o[2] = sqrt(s[2] / n);
    o[3] = sqrt(s[3] / n);
    o[4] = s[5] / n;
    o[5] = s[6] / n;
    o[6] = s[7] / n;
    o[7] = s[8] / n;
    o[8] = sqrt(s[9] / n);
    o[9] = sqrt(s[3] / n - (s[4] * s[4]) / (n * n)) * 100.0;  // silog_rmse
  }
  out[22] = a[0];
  out[23] = n;
}

// Sums v[0..K) over the cluster in a fixed order: warp butterfly, the CTA's warps in index order, then the CTAs in rank
// order 0..kEvalCluster-1, read from each one's `part` in shared memory. Every thread of the cluster returns with the same
// K sums in v. A peer may read `part` until the next cluster barrier after this call returns, so each call needs its own.
template <int K>
__device__ __forceinline__ void eval_cluster_sum(double (&v)[K], double* warp_part, double* part, double* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) v[k] = warp_sum_d(v[k]);
  if (lane == 0)
#pragma unroll
    for (int k = 0; k < K; ++k) warp_part[warp * K + k] = v[k];
  __syncthreads();
  if (threadIdx.x < K) {
    double s = 0.0;
    for (int w = 0; w < kEvalWarps; ++w) s += warp_part[w * K + threadIdx.x];
    part[threadIdx.x] = s;
  }
  cluster_sync_all();  // every CTA's part is written and visible to the cluster
  if (threadIdx.x < K) {
    const uint32_t addr = smem_u32(part + threadIdx.x);
    double s = 0.0;
    for (int r = 0; r < kEvalCluster; ++r) s += ld_shared_cluster_f64(mapa_shared(addr, r));
    total[threadIdx.x] = s;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) v[k] = total[k];
}

// grid (kEvalCluster, B): sample b = blockIdx.y is one cluster. Pass 1 sums over the visible mask, pass 2 over the object
// mask; rank 0 writes out[b * kEvalOut ..].
__global__ void __cluster_dims__(kEvalCluster, 1, 1) __launch_bounds__(kEvalThreads)
eval_batch_kernel(const float* pred, const uint8_t* src, const ada_eval_desc* __restrict__ table, const EvalSample one,
                  double* __restrict__ out) {
  __shared__ double warp_part[kEvalWarps * kEvalObjectSums];
  __shared__ double total[kEvalObjectSums];
  __shared__ double part_align[kEvalAlignSums], part_object[kEvalObjectSums];
  const EvalSample a = eval_sample_at(pred, src, table, one);
  const int rank = static_cast<int>(cluster_ctarank());
  const int n = a.H * a.W;
  const int first = rank * kEvalThreads + threadIdx.x, step = kEvalCluster * kEvalThreads;

  double s1[kEvalAlignSums] = {0, 0, 0, 0, 0};
  for (int i = first; i < n; i += step) {
    if (a.visible[i]) {
      const double p = eval_pred_at(a, i), g = a.obs[i];
      s1[0] += 1.0; s1[1] += p; s1[2] += p * p; s1[3] += g; s1[4] += p * g;
    }
  }
  eval_cluster_sum(s1, warp_part, part_align, total);
  float scale, shift;
  eval_scale_shift(s1, scale, shift);

  double s2[kEvalObjectSums];
#pragma unroll
  for (int k = 0; k < kEvalObjectSums; ++k) s2[k] = 0.0;
  for (int i = first; i < n; i += step) {
    if (!a.object[i]) continue;
    s2[0] += 1.0;
    eval_metric_terms(eval_pred_at(a, i), a.gt[i], scale, shift, s2 + 1);
  }
  eval_cluster_sum(s2, warp_part, part_object, total);
  if (rank == 0 && threadIdx.x == 0) eval_finalize(s1, s2, out + static_cast<long long>(blockIdx.y) * kEvalOut);
  cluster_sync_all();  // no CTA leaves while a peer may still read its part_object
}

// The skip rule of the validation loop (discriminative_trainer.py:596-597, the reading tests/test_eval_gpu.py records):
// a sample with a NaN among its 20 metric values is left out of every mean. This covers non-positive aligned depth
// (log of a negative), an empty object mask (0/0) and a degenerate visible mask (NaN scale).
__device__ __forceinline__ bool eval_row_skipped(const double* row) {
  bool nan = false;
#pragma unroll
  for (int k = 2; k < 2 + 2 * kEvalMetricSums; ++k) nan |= row[k] != row[k];
  return nan;
}

// acc [(n_buckets + 1), kEvalAccSlots] += rows [B, kEvalOut]. Group 0 is "overall", group 1 + k is bucket k; slots are
// n_used, n_skipped and the sums of row[2..21]. One thread owns each (group, slot) and adds the rows in order b = 0..B-1,
// so the additions into a slot are the same sequence however the samples are split into calls. A row whose label is
// outside [0, n_buckets) (or bucket == nullptr) counts in "overall" only.
__global__ void __launch_bounds__(256)
eval_accumulate_kernel(const double* __restrict__ rows, int B, const int32_t* __restrict__ bucket, int n_buckets,
                       double* __restrict__ acc) {
  const int slots = (n_buckets + 1) * kEvalAccSlots;
  for (int j = threadIdx.x; j < slots; j += blockDim.x) {
    const int g = j / kEvalAccSlots, slot = j - g * kEvalAccSlots;
    double s = acc[j];
    for (int b = 0; b < B; ++b) {
      if (g > 0 && (!bucket || bucket[b] != g - 1)) continue;
      const double* row = rows + static_cast<long long>(b) * kEvalOut;
      const bool skip = eval_row_skipped(row);
      if (slot == 0) {
        if (!skip) s += 1.0;
      } else if (slot == 1) {
        if (skip) s += 1.0;
      } else if (!skip) {
        s += row[slot];
      }
    }
    acc[j] = s;
  }
}

}  // namespace ada
