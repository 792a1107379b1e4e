// K3 — PCK / AUC / EPE accumulation as shardable integer counters, and the legacy evaluate_pck.
// The arithmetic of _calc_distances is reproduced step by step in the dtype numpy would promote to (the
// difference pred - gt in f32 when both are f32, the division and everything after it in f64 unless the
// normaliser is f32 too), rounded to f32 and compared with the f32 threshold, so hit counts are
// bit-exact; counters are int64 and order-independent, hence identical for any sharding.
#include <cstdlib>
#include <math_constants.h>

#include "lhn_common.cuh"

namespace lhn {
int num_sms();

constexpr int kMaxThr = 64;

struct PckArgs {
  const void* pred; int pred_dtype, pred_stride;
  const void* gt; int gt_dtype, gt_stride;
  const uint8_t* mask;
  const void* normalize; int norm_dtype;
  double norm_const;
  int64_t N; int K, T;
  float thr[kMaxThr];
  int all_f32;
  int diff_f32;               // pred and gt are both f32: numpy takes their difference in f32
  int sorted_thr;             // thr[] is non-decreasing (host-checked): histogram counting
  unsigned long long* counters;
};

__device__ __forceinline__ double ld_as_f64(const void* p, int dtype, int64_t i) {
  return dtype == LHN_F64 ? reinterpret_cast<const double*>(p)[i] : (double)reinterpret_cast<const float*>(p)[i];
}

// The grid stride is a multiple of K, so a thread meets ONE joint for its whole loop: `valid` and the fixed-point
// distance sum live in registers and the sample index advances without a division.  Thresholds in ascending order
// (every caller: one PCK threshold, or keypoint_auc's i / num_step) are counted as a HISTOGRAM of "thresholds passed" —
// one native 32-bit shared-memory add per element — and turned into per-threshold hit counts when the block flushes;
// unsorted thresholds take one add per passed threshold.  Every load of an element is issued before anything is
// decided, four elements per thread in flight.  Round 1: three or more 64-bit shared atomics (compare-and-swap loops)
// per element behind three DEPENDENT loads and a 64-bit division — 16 % of the HBM peak.
// FAST: every array is f32 with (x, y) pairs 8-byte aligned — the shape every caller on the hot path has (decoded f32
// points against f32 ground truth, f32 or constant normaliser): 64-bit loads, no dtype switches, f32 arithmetic.
template <bool FAST, int U>
__global__ void __launch_bounds__(256) pck_accumulate_kernel(const __grid_constant__ PckArgs a) {
  extern __shared__ unsigned long long sc[];   // [(T+2)*K] u64 block counters, then [(T+1)*K] u32 histogram
  const int K = a.K, T = a.T;
  const int ncnt = (T + 2) * K;
  unsigned int* hist = reinterpret_cast<unsigned int*>(sc + ncnt);
  for (int i = threadIdx.x; i < ncnt; i += blockDim.x) sc[i] = 0ull;
  for (int i = threadIdx.x; i < (T + 1) * K; i += blockDim.x) hist[i] = 0u;
  __syncthreads();
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  // the stride is rounded DOWN to a multiple of K, so k is loop-invariant and the threads at e0 >= stride (fewer than K)
  // take no element: every element is visited exactly once.  Uncapped grids have nthreads >= N*K, hence stride >= N*K.
  const int64_t stride = nthreads / K * K;
  const int64_t e0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = e0 < stride ? a.N * K : 0;
  const int k = (int)(e0 % K);
  const int64_t n_step = stride / K;
  int64_t n = e0 / K;
  unsigned int valid = 0;
  unsigned long long dsum = 0ull;
  unsigned int hit1 = 0;                               // T == 1 (PCK at one threshold): the count stays in a register
  const float thr0 = T > 0 ? a.thr[0] : 0.f;
  auto consume = [&](float d) {
    ++valid;
    dsum += epe_fix_term(d);                           // NaN, inf and d >= 2^43 add nothing
    if (T == 1) {
      hit1 += (d < thr0) ? 1u : 0u;
    } else if (a.sorted_thr) {
      int nh = 0;                                      // ascending thresholds: passed ones form a suffix
      for (int t = 0; t < T; ++t) nh += (d < a.thr[t]) ? 1 : 0;
      if (nh) atomicAdd(&hist[nh * K + k], 1u);
    } else {
      for (int t = 0; t < T; ++t)
        if (d < a.thr[t]) atomicAdd(reinterpret_cast<unsigned int*>(&sc[t * K + k]), 1u);
    }
  };
  if (FAST) {
    // four elements' loads (28 B each) are issued before any arithmetic: the shared atomics and the early-outs of
    // consume() would otherwise pin every load behind the previous element's decision
    // Running pointers, and a main loop over FULL batches without per-element bounds checks (then a plain tail): the
    // kernel is issue-bound — two IEEE divisions and a square root per 25-byte element — so the 64-bit index
    // arithmetic and predicates of a guarded batch (a quarter of the instructions) were worth removing.
    auto elem = [&](const float2 p, const float2 g, const float2 z, const unsigned char m) {
      if (!m || z.x == 0.f || z.y == 0.f) return;             // masked joint / _mask[normalize == 0 rows] = False
      const float fx = z.x < 0.f ? 1e6f : z.x, fy = z.y < 0.f ? 1e6f : z.y;      // normalize[normalize<=0] = 1e6
      const float qx = __fdiv_rn(__fsub_rn(p.x, g.x), fx), qy = __fdiv_rn(__fsub_rn(p.y, g.y), fy);
      consume(__fsqrt_rn(__fadd_rn(__fmul_rn(qx, qx), __fmul_rn(qy, qy))));
    };
    const float2* pp = reinterpret_cast<const float2*>(a.pred) + e0;
    const float2* gp = reinterpret_cast<const float2*>(a.gt) + e0;
    const float2* zp = reinterpret_cast<const float2*>(a.normalize) + n;    // the launcher takes this path only with a normaliser
    const unsigned char* mp = a.mask + e0;
    int64_t e = e0;
    for (; e + (U - 1) * stride < total; e += U * stride) {
      float2 p[U], g[U], z[U];
      unsigned char m[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        m[u] = mp[u * stride]; p[u] = __ldg(pp + u * stride); g[u] = __ldg(gp + u * stride); z[u] = __ldg(zp + u * n_step);
      }
      pp += U * stride; gp += U * stride; mp += U * stride; zp += U * n_step;
#pragma unroll
      for (int u = 0; u < U; ++u) elem(p[u], g[u], z[u], m[u]);
    }
    for (; e < total; e += stride, pp += stride, gp += stride, mp += stride, zp += n_step)
      elem(__ldg(pp), __ldg(gp), __ldg(zp), *mp);
  } else {
#pragma unroll 4
  for (int64_t e = e0; e < total; e += stride, n += n_step) {
    const bool m = a.mask[e] != 0;
    float d;
    double nx = a.norm_const, ny = a.norm_const;
    if (a.normalize) { nx = ld_as_f64(a.normalize, a.norm_dtype, 2 * n); ny = ld_as_f64(a.normalize, a.norm_dtype, 2 * n + 1); }
    if (a.all_f32) {
      const float* pp = reinterpret_cast<const float*>(a.pred) + e * a.pred_stride;
      const float* gp = reinterpret_cast<const float*>(a.gt) + e * a.gt_stride;
      const float p0 = pp[0], p1 = pp[1], g0 = gp[0], g1 = gp[1];
      const float fx = nx < 0.0 ? 1e6f : (float)nx, fy = ny < 0.0 ? 1e6f : (float)ny;   // normalize[normalize<=0] = 1e6
      const float qx = __fdiv_rn(__fsub_rn(p0, g0), fx);
      const float qy = __fdiv_rn(__fsub_rn(p1, g1), fy);
      d = __fsqrt_rn(__fadd_rn(__fmul_rn(qx, qx), __fmul_rn(qy, qy)));
    } else {
      const double px = ld_as_f64(a.pred, a.pred_dtype, e * a.pred_stride);
      const double py = ld_as_f64(a.pred, a.pred_dtype, e * a.pred_stride + 1);
      const double gx = ld_as_f64(a.gt, a.gt_dtype, e * a.gt_stride);
      const double gy = ld_as_f64(a.gt, a.gt_dtype, e * a.gt_stride + 1);
      const double dx = nx < 0.0 ? 1e6 : nx, dy = ny < 0.0 ? 1e6 : ny;
      // `preds - targets` comes first in numpy: two f32 arrays subtract in f32, and only the division by an f64
      // normaliser (or the python-float constant) promotes
      const double ex = a.diff_f32 ? (double)__fsub_rn((float)px, (float)gx) : __dsub_rn(px, gx);
      const double ey = a.diff_f32 ? (double)__fsub_rn((float)py, (float)gy) : __dsub_rn(py, gy);
      const double qx = __ddiv_rn(ex, dx), qy = __ddiv_rn(ey, dy);
      d = (float)__dsqrt_rn(__dadd_rn(__dmul_rn(qx, qx), __dmul_rn(qy, qy)));
    }
    if (!m || nx == 0.0 || ny == 0.0) continue;        // masked joint / _mask[normalize == 0 rows] = False
    consume(d);
  }
  }
  if (T == 1 && hit1) atomicAdd(reinterpret_cast<unsigned int*>(&sc[k]), hit1);
  if (valid) {
    atomicAdd(reinterpret_cast<unsigned int*>(&sc[T * K + k]), valid);      // low word: per-block counts stay < 2^32
    atomicAdd(&sc[(T + 1) * K + k], dsum);
  }
  __syncthreads();
  if (a.sorted_thr && T > 1) {
    // hits[t] = elements that passed at least T - t thresholds: a running sum down the histogram, one joint per thread
    for (int kk = threadIdx.x; kk < K; kk += blockDim.x) {
      unsigned long long run = 0ull;
      for (int nh = T; nh >= 1; --nh) { run += hist[nh * K + kk]; sc[(T - nh) * K + kk] = run; }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < ncnt; i += blockDim.x)
    if (sc[i]) atomicAdd(a.counters + i, sc[i]);
}

// ---- MPII PCKh counters (topdown_mpii_dataset.py:186-214): f64 throughout, `<=`, head-box norm * sc_bias ------
struct MpiiArgs {
  const float* pred; int pred_stride;
  const double* gt;        // [N,K,2] 1-based ground truth (pos_gt_src transposed)
  const double* head;      // [N,4] head box (x1, y1, x2, y2) (headboxes_src transposed)
  const uint8_t* visible;  // [N,K] 1 - jnt_missing
  int64_t N; int K, T;
  double sc_bias;
  double thr[kMaxThr];
  unsigned long long* counters;   // hits[T][K], count[K]
};

__global__ void __launch_bounds__(256) mpii_pckh_kernel(const __grid_constant__ MpiiArgs a) {
  extern __shared__ unsigned long long sc[];   // (T+1)*K
  const int K = a.K, T = a.T;
  const int ncnt = (T + 1) * K;
  for (int i = threadIdx.x; i < ncnt; i += blockDim.x) sc[i] = 0ull;
  __syncthreads();
  const int64_t total = a.N * K;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    if (!a.visible[e]) continue;
    const int64_t n = e / K;
    const int k = (int)(e - n * K);
    // preds[..., :2] + 1.0 stays f32 (NumPy keeps the array dtype), the difference with the f64 ground truth is f64
    const double dx = __dsub_rn((double)__fadd_rn(a.pred[e * a.pred_stride], 1.0f), a.gt[2 * e]);
    const double dy = __dsub_rn((double)__fadd_rn(a.pred[e * a.pred_stride + 1], 1.0f), a.gt[2 * e + 1]);
    const double err = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
    const double hx = __dsub_rn(a.head[4 * n + 2], a.head[4 * n]), hy = __dsub_rn(a.head[4 * n + 3], a.head[4 * n + 1]);
    const double hs = __dmul_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(hx, hx), __dmul_rn(hy, hy))), a.sc_bias);
    const double v = __ddiv_rn(err, hs);
    atomicAdd(&sc[T * K + k], 1ull);
    for (int t = 0; t < T; ++t)
      if (v <= a.thr[t]) atomicAdd(&sc[t * K + k], 1ull);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < ncnt; i += blockDim.x)
    if (sc[i]) atomicAdd(a.counters + i, sc[i]);
}

// ---- legacy evaluate_pck (evaluation.py:10-59): per-image reduction over the decoded joints -----
// pk/gk: [B*K,3] (x*fx, y*fy, maxval) already scaled (A1 + T2 from the heatmap kernel).
__global__ void __launch_bounds__(128) evaluate_pck_image_kernel(const float* __restrict__ pk,
                                                                 const float* __restrict__ gk,
                                                                 const float* __restrict__ bbox_wh,
                                                                 const float* __restrict__ weight,
                                                                 int64_t B, int K, float thr,
                                                                 float* __restrict__ pck) {
  const int lane = threadIdx.x & 31;
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= B) return;
  const float max_wh = fmaxf(bbox_wh[2 * b], bbox_wh[2 * b + 1]);
  int hits = 0;
  float wsum = 0.f;   // sum over the doubled [K,2] weight, f32 like torch
  for (int k = lane; k < K; k += 32) {
    const float w = weight ? weight[b * K + k] : 1.f;
    wsum += w;
    if (w == 1.f) {
      const float* p = pk + 3 * (b * K + k);
      const float* g = gk + 3 * (b * K + k);
      const float dx = __fsub_rn(p[0], g[0]), dy = __fsub_rn(p[1], g[1]);
      // torch.norm accumulates in double on CPU; coordinates are small integers * stride
      const float dist = (float)sqrt((double)dx * dx + (double)dy * dy);
      if (__fdiv_rn(dist, max_wh) < thr) hits += 1;
    }
  }
  hits = __reduce_add_sync(0xffffffffu, hits);
  wsum = warp_sum(wsum);
  if (lane == 0) pck[b] = __fmul_rn(__fdiv_rn((float)hits, __fmul_rn(wsum, 2.f)), 2.f);
}

__global__ void __launch_bounds__(1024) mean_f32_to_f64_kernel(const float* __restrict__ v, int64_t n,
                                                               double* __restrict__ out) {
  __shared__ double red[32];
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += (double)v[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    double t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
    t = warp_sum(t);
    if (threadIdx.x == 0) out[0] = t / (double)n;
  }
}

}  // namespace lhn

using namespace lhn;

extern "C" int lhn_pck_accumulate(const void* pred, int pred_dtype, int pred_stride, const void* gt,
                                  int gt_dtype, int gt_stride, const uint8_t* mask,
                                  const void* normalize, int norm_dtype, double norm_const, int64_t N,
                                  int K, const float* thr, int T, int64_t* counters,
                                  lhn_stream_t stream) {
  // an empty shard (N == 0) reads no element: its arrays may be null, as torch's empty CUDA tensors are
  if ((N > 0 && (!pred || !gt || !mask)) || !counters || N < 0 || K <= 0 || T < 0 || T > kMaxThr ||
      pred_stride < 2 || gt_stride < 2 || (T > 0 && !thr))
    return LHN_EINVAL;
  auto okdt = [](int d) { return d == LHN_F32 || d == LHN_F64; };
  if (!okdt(pred_dtype) || !okdt(gt_dtype) || (normalize && !okdt(norm_dtype))) return LHN_EDTYPE;
  if (N == 0) return LHN_OK;
  PckArgs a{};
  a.pred = pred; a.pred_dtype = pred_dtype; a.pred_stride = pred_stride;
  a.gt = gt; a.gt_dtype = gt_dtype; a.gt_stride = gt_stride;
  a.mask = mask; a.normalize = normalize; a.norm_dtype = norm_dtype; a.norm_const = norm_const;
  a.N = N; a.K = K; a.T = T;
  a.sorted_thr = 1;
  for (int i = 0; i < T; ++i) { a.thr[i] = thr[i]; if (i > 0 && !(thr[i] >= thr[i - 1])) a.sorted_thr = 0; }
  // numpy promotion: f32 only if every array operand is f32 (a python-float constant is f64)
  a.all_f32 = pred_dtype == LHN_F32 && gt_dtype == LHN_F32 && normalize && norm_dtype == LHN_F32;
  a.diff_f32 = pred_dtype == LHN_F32 && gt_dtype == LHN_F32;
  a.counters = reinterpret_cast<unsigned long long*>(counters);
  const int threads = 256;
  int64_t need = (N * K + threads - 1) / threads, cap = (int64_t)num_sms() * 8;
  int blocks = (int)(need < cap ? need : cap);
  size_t smem = (size_t)(T + 2) * K * sizeof(unsigned long long) + (size_t)(T + 1) * K * sizeof(unsigned int);
  if (smem > 48 * 1024) return LHN_EINVAL;
  auto al8 = [](const void* p) { return ((uintptr_t)p % 8) == 0; };
  // the f32 fast path needs a normaliser that is f32 (numpy then computes in f32) or absent with all-f32 points: with a
  // python-float constant numpy promotes to f64, so a constant normaliser keeps the general path
  const bool fast = a.all_f32 && normalize && pred_stride == 2 && gt_stride == 2 && al8(pred) && al8(gt) && al8(normalize);
  // (measured and not kept: eight elements per batch, 76 us against 67; a software-pipelined batch of four or of two,
  // 66.6 / 68.0 us; four resident CTAs per SM instead of a grid of eight, 66.9 us — profiles/r02_kernels.txt history)
  if (fast) pck_accumulate_kernel<true, 4><<<blocks, threads, smem, (cudaStream_t)stream>>>(a);
  else pck_accumulate_kernel<false, 4><<<blocks, threads, smem, (cudaStream_t)stream>>>(a);
  return check_launch();
}

// ---- _report_metric's final ratios on the device (no host round trip) ---------------------------------------
// One warp.  np.mean of the valid per-joint accuracies is numpy's pairwise sum (n < 8: sequential; n <= 128:
// eight strided accumulators combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the tail sequentially)
// divided by the count — restated literally so the f64 results equal the host expressions bit for bit.
__device__ double np_mean_valid(const double* acc, int n) {
  if (n <= 0) return 0.0;                       // keypoint_pck_accuracy: avg_acc = 0 when no joint is valid
  double res;
  if (n < 8) {
    res = 0.0;
    for (int i = 0; i < n; ++i) res += acc[i];
  } else {
    double r[8];
    for (int j = 0; j < 8; ++j) r[j] = acc[j];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
      for (int j = 0; j < 8; ++j) r[j] += acc[i + j];
    res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res += acc[i];
  }
  return res / (double)n;
}

constexpr int kMaxFinalizeJoints = 128;         // numpy's pairwise block: above it the summation tree changes

__global__ void metrics_finalize_kernel(const long long* __restrict__ c, int K, int T, double* __restrict__ out) {
  // counters: pck_hits[K], pck_valid[K], auc_hits[T][K], auc_valid[K], epe_valid[K], epe_fix[K]
  __shared__ double acc[kMaxFinalizeJoints];
  if (threadIdx.x != 0) return;
  auto avg_acc = [&](const long long* hits, const long long* valid, double* per_joint) {
    int n = 0;
    for (int k = 0; k < K; ++k) {
      const double a = valid[k] > 0 ? (double)hits[k] / (double)valid[k] : -1.0;     // _distance_acc
      if (per_joint) per_joint[k] = a;
      if (a >= 0.0) acc[n++] = a;
    }
    return np_mean_valid(acc, n);
  };
  out[0] = avg_acc(c, c + K, out + 3);                                                 // PCK (+ acc[K])
  double auc = 0.0;
  // auc += 1.0 / num_step * avg_acc: a rounded product, then a rounded sum (no FMA contraction)
  for (int t = 0; t < T; ++t)
    auc = __dadd_rn(auc, __dmul_rn(1.0 / (double)T, avg_acc(c + (int64_t)(2 + t) * K, c + (int64_t)(2 + T) * K, nullptr)));
  out[1] = auc;                                                                        // keypoint_auc
  long long cnt = 0, fix = 0;
  for (int k = 0; k < K; ++k) { cnt += c[(int64_t)(3 + T) * K + k]; fix += c[(int64_t)(4 + T) * K + k]; }
  out[2] = ((double)fix / 1048576.0) / (double)(cnt > 1 ? cnt : 1);                    // EPE from the fixed-point sum
}

extern "C" int lhn_metrics_finalize(const int64_t* counters, int K, int auc_steps, double* out, lhn_stream_t stream) {
  if (!counters || !out || K <= 0 || K > kMaxFinalizeJoints || auc_steps < 0) return LHN_EINVAL;
  metrics_finalize_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(reinterpret_cast<const long long*>(counters), K,
                                                             auc_steps, out);
  return check_launch();
}

extern "C" int64_t lhn_evaluate_pck_workspace_bytes(int64_t B, int K) {
  if (B < 0 || K <= 0) return LHN_EINVAL;
  return 2 * B * K * 3 * (int64_t)sizeof(float);
}

extern "C" int lhn_evaluate_pck(const void* pred_hm, const void* gt_hm, int dtype, int64_t B, int K,
                                int H, int W, const float* bbox_wh, const float* weight,
                                float image_w, float image_h, float thr, void* workspace,
                                int64_t workspace_bytes, float* pck_per_image, double* mean_out,
                                lhn_stream_t stream) {
  if (!pred_hm || !gt_hm || !bbox_wh || !workspace || !pck_per_image || !mean_out || B <= 0 || K <= 0)
    return LHN_EINVAL;
  if (workspace_bytes < lhn_evaluate_pck_workspace_bytes(B, K)) return LHN_EWORKSPACE;
  if ((uintptr_t)workspace % 4) return LHN_EALIGN;
  float* pk = (float*)workspace;
  float* gk = pk + B * K * 3;
  lhn_decode_params dp{};
  dp.mask_mode = LHN_MASK_ZERO; dp.refine = LHN_REFINE_NONE; dp.transform = LHN_XFORM_SCALE;
  dp.scale_x = image_w / (float)W; dp.scale_y = image_h / (float)H;   // tensor(image_size)/tensor([w,h])
  const int64_t HW = (int64_t)H * W;
  int rc = lhn_decode_heatmap(pred_hm, nullptr, nullptr, dtype, B, K, H, W, K * HW, HW, 0, 0, nullptr,
                              nullptr, &dp, nullptr, pk, nullptr, nullptr, nullptr, 0, nullptr, 0,
                              nullptr, nullptr, stream);
  if (rc) return rc;
  rc = lhn_decode_heatmap(gt_hm, nullptr, nullptr, dtype, B, K, H, W, K * HW, HW, 0, 0, nullptr,
                          nullptr, &dp, nullptr, gk, nullptr, nullptr, nullptr, 0, nullptr, 0,
                          nullptr, nullptr, stream);
  if (rc) return rc;
  const int threads = 128;
  int64_t blocks = (B * 32 + threads - 1) / threads;
  evaluate_pck_image_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(pk, gk, bbox_wh, weight,
                                                                                   B, K, thr, pck_per_image);
  rc = check_launch();
  if (rc) return rc;
  mean_f32_to_f64_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(pck_per_image, B, mean_out);
  return check_launch();
}

extern "C" int lhn_mpii_pckh_accumulate(const float* pred, int pred_stride, const double* gt, const double* head,
                                        const uint8_t* visible, int64_t N, int K, const double* thr, int T,
                                        double sc_bias, int64_t* counters, lhn_stream_t stream) {
  if (!pred || !gt || !head || !visible || !thr || !counters || N < 0 || K <= 0 || T <= 0 || T > kMaxThr ||
      pred_stride < 2 || !(sc_bias > 0.0))
    return LHN_EINVAL;
  if (N == 0) return LHN_OK;
  MpiiArgs a{};
  a.pred = pred; a.pred_stride = pred_stride; a.gt = gt; a.head = head; a.visible = visible;
  a.N = N; a.K = K; a.T = T; a.sc_bias = sc_bias;
  for (int t = 0; t < T; ++t) a.thr[t] = thr[t];
  a.counters = reinterpret_cast<unsigned long long*>(counters);
  const size_t smem = (size_t)(T + 1) * K * sizeof(unsigned long long);
  if (smem > 48 * 1024) return LHN_EINVAL;
  int64_t blocks = (N * K + 255) / 256;
  const int64_t cap = (int64_t)num_sms() * 4;
  if (blocks > cap) blocks = cap;
  mpii_pckh_kernel<<<(unsigned)blocks, 256, smem, (cudaStream_t)stream>>>(a);
  return check_launch();
}
