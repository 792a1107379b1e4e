// K2 — SimDR 1-D vector decode (+ optional vector_nms / bbox mask) and the KLDiscretLoss
// (SmoothL1) sums.  One warp owns one (b, k) pair: the x- and y-vector are streamed with 128-bit
// coalesced loads, reduced with redux/shuffles; nothing is staged in shared memory because every
// element is used exactly once (the 3-tap NMS neighbourhood comes from warp shuffles).
#include <math_constants.h>
#include <stdlib.h>

#include "lhn_common.cuh"

namespace lhn {
int num_sms();

thread_local lhn_simdr_launch_info g_simdr_launch = {};

// first-max argmax of one vector by one warp; NaN is maximal.
// NMS: value kept iff it equals max(v[i-1], v[i], v[i+1]) (max_pool1d k=3,s=1,p=1 with -inf
// padding) else 0; then multiplied by the [lo, hi) mask (result_parser.py:61-74,113-121).
// The value reported is the selected element itself (after NMS and the mask), as numpy's take_along_axis gives it:
// −0 and +0 tie (the key maps both to +0) but the score keeps the sign of the element at the first index.
template <typename T, bool NMS>
__device__ __forceinline__ void warp_vec_argmax(const T* __restrict__ v, int L, int lo, int hi,
                                                int lane, uint32_t& out_idx, float& out_val) {
  uint32_t bkey = 0u, bidx = 0xffffffffu;
  float bval = 0.f;                                          // this lane's first element of key bkey
  const bool vec = ((L & 3) == 0) && (reinterpret_cast<uintptr_t>(v) % (4 * sizeof(T)) == 0);
  if (vec && !NMS) {
    const int nq = L >> 2;
    float best = -CUDART_INF_F; bool has_nan = false; uint32_t nan_idx = 0xffffffffu;
#pragma unroll 4
    for (int q = lane; q < nq; q += 32) {
      const float4 a = ldg_stream4<T>(v + 4 * q);
      const uint32_t e = 4u * q;
      if (a.x > best) { best = a.x; bidx = e; }
      if (a.y > best) { best = a.y; bidx = e + 1; }
      if (a.z > best) { best = a.z; bidx = e + 2; }
      if (a.w > best) { best = a.w; bidx = e + 3; }
      if (!has_nan) {
        if (a.x != a.x) { has_nan = true; nan_idx = e; }
        else if (a.y != a.y) { has_nan = true; nan_idx = e + 1; }
        else if (a.z != a.z) { has_nan = true; nan_idx = e + 2; }
        else if (a.w != a.w) { has_nan = true; nan_idx = e + 3; }
      }
    }
    if (has_nan) { bkey = 0xffffffffu; bidx = nan_idx; bval = CUDART_NAN_F; }
    else { bkey = order_key(best); bval = best; }
  } else {
    // scalar path (also the NMS path: neighbours via an overlapping read)
    for (int i = lane; i < L; i += 32) {
      float x = Elem<T>::to_f32(v[i]);
      if (NMS) {
        const float l = i > 0 ? Elem<T>::to_f32(v[i - 1]) : -CUDART_INF_F;
        const float r = i + 1 < L ? Elem<T>::to_f32(v[i + 1]) : -CUDART_INF_F;
        // torch max_pool1d propagates NaN; eq(NaN, .) is false -> mask 0 -> NaN*0 = NaN
        float m = fmaxf(fmaxf(l, x), r);
        if (l != l || x != x || r != r) m = CUDART_NAN_F;
        x = x * ((m == x) ? 1.f : 0.f);
        x = x * ((i >= lo && i < hi) ? 1.f : 0.f);
      }
      const uint32_t kx = order_key(x);
      if (bidx == 0xffffffffu || kx > bkey) { bkey = kx; bidx = (uint32_t)i; bval = x; }
    }
    if (bidx == 0xffffffffu) bkey = 0u;
  }
  warp_argmax(bkey, bidx);
  if (bidx == 0xffffffffu) bidx = 0;
  out_idx = bidx;
  // the lane that scanned element bidx holds it as its own first maximum
  const int src = (vec && !NMS) ? (int)((bidx >> 2) & 31u) : (int)(bidx & 31u);
  out_val = __shfl_sync(0xffffffffu, bval, src);
}

// Fast path (no NMS, 16-byte aligned vectors): both vectors of a (b, k) pair are scanned in ONE loop so that all
// of their 128-bit loads are in flight together (one memory latency per pair instead of two), NaN detection is one
// NaN-propagating 3-input max per quad, and the exact first-NaN element is only looked up when one was seen.
struct LaneBest { float best; uint32_t q; };

// 4 instructions per quad: two NaN-propagating 3-input maxima (FMNMX3.NAN), one compare, one predicated move.
// `best` becomes NaN as soon as the lane meets one; `q` is the first quad that raised the running maximum.
__device__ __forceinline__ void lane_scan4(const float4& a, uint32_t q, LaneBest& s) {
  float m, r;
  asm("max.NaN.f32 %0, %1, %2, %3;" : "=f"(m) : "f"(a.x), "f"(a.y), "f"(a.z));
  asm("max.NaN.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(m), "f"(a.w), "f"(s.best));
  if (r != s.best) s.q = q;
  s.best = r;
}

// warp-wide (max, first quad holding it); then the winning quad is read again (L1/L2 hit) to name the element
template <typename T>
__device__ __forceinline__ void warp_finish(const T* __restrict__ v, int nq, int lane, LaneBest s, uint32_t& out_idx,
                                            float& out_val) {
  float wmax;
  asm volatile("redux.sync.max.NaN.f32 %0, %1, 0xffffffff;" : "=f"(wmax) : "f"(s.best));
  if (wmax != wmax) {                                      // rare: the first NaN of the vector is the argmax
    uint32_t first = 0xffffffffu;
    for (int q = lane; q < nq && first == 0xffffffffu; q += 32) {
      const float4 a = load4<T>(v + 4 * q);
      if (a.x != a.x) first = 4 * q;
      else if (a.y != a.y) first = 4 * q + 1;
      else if (a.z != a.z) first = 4 * q + 2;
      else if (a.w != a.w) first = 4 * q + 3;
    }
    out_idx = __reduce_min_sync(0xffffffffu, first);
    out_val = __uint_as_float(0x7fc00000u);
    return;
  }
  const uint32_t qsel = __reduce_min_sync(0xffffffffu, (s.best == wmax) ? s.q : 0xffffffffu);
  if (qsel == 0xffffffffu) {                               // every element is -inf: index 0
    out_idx = 0; out_val = Elem<T>::to_f32(v[0]);
    return;
  }
  const float4 a = load4<T>(v + 4 * qsel);
  // `==` treats -0 and +0 as equal, like torch/numpy; report the element actually selected
  if (a.x == wmax) { out_idx = 4 * qsel; out_val = a.x; }
  else if (a.y == wmax) { out_idx = 4 * qsel + 1; out_val = a.y; }
  else if (a.z == wmax) { out_idx = 4 * qsel + 2; out_val = a.z; }
  else { out_idx = 4 * qsel + 3; out_val = a.w; }
}

template <typename T>
__device__ __forceinline__ void warp_pair_argmax(const T* __restrict__ xv, const T* __restrict__ yv, int Lx, int Ly,
                                                 int lane, uint32_t& ix, float& mx, uint32_t& iy, float& my) {
  LaneBest sx{-CUDART_INF_F, 0xffffffffu}, sy = sx;
  const int nqx = Lx >> 2, nqy = Ly >> 2, nq = nqx > nqy ? nqx : nqy;
#pragma unroll 4
  for (int q = lane; q < nq; q += 32) {
    float4 a, b;
    const bool hx = q < nqx, hy = q < nqy;
    if (hx) a = ldg_stream4<T>(xv + 4 * q);
    if (hy) b = ldg_stream4<T>(yv + 4 * q);
    if (hx) lane_scan4(a, (uint32_t)q, sx);
    if (hy) lane_scan4(b, (uint32_t)q, sy);
  }
  warp_finish<T>(xv, nqx, lane, sx, ix, mx);
  warp_finish<T>(yv, nqy, lane, sy, iy, my);
}

// Loop-invariant divisors of the epilogue.  k, Lx / k and Ly / k are powers of two in every reference config
// (k = 2, 256- or 512-bin vectors), and dividing by a power of two is the same correctly rounded result as
// multiplying by its exact reciprocal — so the five IEEE divisions per pair (a fifth of the ring kernel's
// instructions, profiles/r01_simdr_ring_ncu_summary.txt) become multiplications; other sizes keep the divisions.
struct SimdrDiv {
  float fk, fxo, fyo;      // (float)k, (float)(Lx / k), (float)(Ly / k)
  float rk, rxo, ryo;      // their reciprocals (exact when pow2)
  bool pow2;
};
__device__ __forceinline__ bool is_pow2f(float v) { return v > 0.f && (__float_as_uint(v) & 0x007fffffu) == 0u && v < 1e30f && v > 1e-30f; }
__device__ __forceinline__ SimdrDiv simdr_div(int k, int Lx, int Ly) {
  SimdrDiv d;
  d.fk = (float)k; d.fxo = (float)(Lx / k); d.fyo = (float)(Ly / k);
  d.pow2 = is_pow2f(d.fk) && is_pow2f(d.fxo) && is_pow2f(d.fyo) && k < (1 << 24);
  d.rk = d.pow2 ? 1.f / d.fk : 0.f; d.rxo = d.pow2 ? 1.f / d.fxo : 0.f; d.ryo = d.pow2 ? 1.f / d.fyo : 0.f;
  return d;
}

// lane 0 of the warp that owns pair bk: preds = idx / k (int64 / int -> f64 -> f32: one rounding of the exact quotient,
// which is what the correctly rounded f32 division of the exactly representable operands gives),
// score = (max_x + max_y) / 2, transform_preds with output_size [Lx // k, Ly // k].
__device__ __forceinline__ void simdr_store(uint32_t ix, uint32_t iy, float mx, float my, int k, const SimdrDiv& dv,
                                            bool xform, float cx, float cy, float sc0, float sc1, float* __restrict__ out,
                                            int32_t* __restrict__ out_idx, int64_t bk) {
  float px, py;
  const bool small = ix < (1u << 24) && iy < (1u << 24) && k < (1 << 24);
  if (small && dv.pow2) {
    px = __fmul_rn((float)ix, dv.rk); py = __fmul_rn((float)iy, dv.rk);
  } else if (small) {
    px = __fdiv_rn((float)ix, dv.fk); py = __fdiv_rn((float)iy, dv.fk);
  } else {
    px = (float)((double)ix / (double)k); py = (float)((double)iy / (double)k);
  }
  const float score = __fmul_rn(__fadd_rn(mx, my), 0.5f);
  if (xform) {
    const float s0 = __fmul_rn(sc0, 200.f), s1 = __fmul_rn(sc1, 200.f);
    const float fx = dv.pow2 ? __fmul_rn(s0, dv.rxo) : __fdiv_rn(s0, dv.fxo);
    const float fy = dv.pow2 ? __fmul_rn(s1, dv.ryo) : __fdiv_rn(s1, dv.fyo);
    px = __fsub_rn(__fadd_rn(__fmul_rn(px, fx), cx), __fmul_rn(s0, 0.5f));
    py = __fsub_rn(__fadd_rn(__fmul_rn(py, fy), cy), __fmul_rn(s1, 0.5f));
  }
  float* o = out + 3 * bk;
  o[0] = px; o[1] = py; o[2] = score;
  if (out_idx) { out_idx[2 * bk] = (int32_t)ix; out_idx[2 * bk + 1] = (int32_t)iy; }
}

template <typename T, bool NMS>
__global__ void __launch_bounds__(256, 6) decode_simdr_kernel(const T* __restrict__ xv, const T* __restrict__ yv,
                                                           int64_t n_bk, int K, int Lx, int Ly, int k,
                                                           const float* __restrict__ center,
                                                           const float* __restrict__ scale,
                                                           const int32_t* __restrict__ ranges,
                                                           float* __restrict__ out,
                                                           int32_t* __restrict__ out_idx) {
  const int lane = threadIdx.x & 31;
  const int64_t wg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const SimdrDiv dv = simdr_div(k, Lx, Ly);
  for (int64_t bk = wg; bk < n_bk; bk += nw) {
    const int64_t b = bk / K;
    int x1 = 0, x2 = Lx, y1 = 0, y2 = Ly;
    if (NMS && ranges) { x1 = ranges[4 * b]; x2 = ranges[4 * b + 1]; y1 = ranges[4 * b + 2]; y2 = ranges[4 * b + 3]; }
    uint32_t ix, iy; float mx, my;
    // per-sample side inputs are requested before the vectors so their latency overlaps the scan
    float cx = 0.f, cy = 0.f, sc0 = 0.f, sc1 = 0.f;
    if (center) { cx = center[2 * b]; cy = center[2 * b + 1]; sc0 = scale[2 * b]; sc1 = scale[2 * b + 1]; }
    const T* xp = xv + bk * Lx;
    const T* yp = yv + bk * Ly;
    const bool fast = !NMS && ((Lx | Ly) & 3) == 0 &&
                      ((reinterpret_cast<uintptr_t>(xp) | reinterpret_cast<uintptr_t>(yp)) % (4 * sizeof(T)) == 0);
    if (fast) {
      warp_pair_argmax<T>(xp, yp, Lx, Ly, lane, ix, mx, iy, my);
    } else {
      warp_vec_argmax<T, NMS>(xp, Lx, x1, x2, lane, ix, mx);
      warp_vec_argmax<T, NMS>(yp, Ly, y1, y2, lane, iy, my);
    }
    if (lane == 0) simdr_store(ix, iy, mx, my, k, dv, center != nullptr, cx, cy, sc0, sc1, out, out_idx, bk);
  }
}

// ---- persistent ring variant (the fast path at scale) ------------------------------------------------------------
// The grid-stride kernel above has no load in flight while a warp reduces, re-reads the winning quad (two L2 round
// trips) and stores: at 48 warps x 4 KB per SM that duty cycle leaves ~100 KB in flight, marginal for 7 TB/s at the
// loaded latency.  Here every warp owns a private ring of `nstg` stages filled by TMA bulk copies (cp.async.bulk +
// mbarrier, L2 evict_first): while it scans one (b, k) pair out of shared memory the next nstg - 1 pairs are already
// in flight, and the winning quad is re-read from shared memory.  One CTA of 16 warps per SM, 3 stages of 4 KB at
// 2 x 512 f32 (16 warps x 3 stages x 4 KB = 192 KB per SM).  No CTA-wide barrier after set-up.
// Measured (profiles/r01_simdr_ring_sweep.txt): throughput follows the number of warps, not the number of stages —
// a pair costs a warp ~2.2k cycles of serial work (scan, two warp reductions, re-arm, five IEEE divisions in the
// epilogue; ~2.5k before the per-pair 64-bit index division was made incremental), so 8 warps run at 59 % of the HBM
// peak and 16 or 24 warps at 90 % (the grid-stride kernel: 82 %).
constexpr int kRingWarps = 16;
constexpr int kRingMaxStages = 4;
constexpr int kRingTriggerPair = 8;   // overlapped launches: warp 0 lets the successor grid in after this many pairs

template <typename T>
__global__ void __launch_bounds__(1024, 1)
decode_simdr_ring_kernel(const T* __restrict__ xv, const T* __restrict__ yv, int64_t n_bk, int K, int Lx, int Ly, int k,
                         const float* __restrict__ center, const float* __restrict__ scale, float* __restrict__ out,
                         int32_t* __restrict__ out_idx, int nstg, int pair_al, int overlap) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  unsigned char* wbase = smem_raw + (size_t)warp * nstg * pair_al;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)nwarps * nstg * pair_al) + warp * kRingMaxStages;
  const uint32_t xbytes = (uint32_t)Lx * sizeof(T), ybytes = (uint32_t)Ly * sizeof(T);
  // The next launch on the stream, if it carries LHN_FLAG_OVERLAP_PREVIOUS, takes over SMs as these CTAs retire.
  // A launch that itself overlaps its predecessor lets its successor in only after the predecessor has completed
  // (warp 0: griddepcontrol.wait, then the trigger, a few pairs into its loop), so launch i + 2 never runs beside
  // launch i — the rule that makes two rotating buffer sets sufficient (same scheme as lhn_heatmap_team.cuh).
  if (!overlap) asm volatile("griddepcontrol.launch_dependents;");
  if (lane == 0) {
    for (int s = 0; s < nstg; ++s) mbar_init(&bars[s], 1);
    fence_mbar_init();
  }
  __syncthreads();
  const uint64_t pol = policy_evict_first();
  SimdrDiv dv{};                                             // only lane 0 stores: only lane 0 pays for the reciprocals
  if (lane == 0) dv = simdr_div(k, Lx, Ly);
  const int64_t total = (int64_t)gridDim.x * nwarps;
  const int64_t gw = (int64_t)warp * gridDim.x + blockIdx.x;   // warp-major: the leftover pairs spread over all SMs
  auto issue = [&](int s, int64_t pair) {
    unsigned char* dst = wbase + (size_t)s * pair_al;
    mbar_arrive_expect_tx(&bars[s], xbytes + ybytes);
    tma_load_1d(dst, xv + pair * Lx, xbytes, &bars[s], pol);
    tma_load_1d(dst + xbytes, yv + pair * Ly, ybytes, &bars[s], pol);
  };
  if (lane == 0)
    for (int s = 0; s < nstg; ++s) {
      const int64_t pair = gw + (int64_t)s * total;
      if (pair < n_bk) issue(s, pair);
    }
  const int nqx = Lx >> 2, nqy = Ly >> 2, nq = nqx > nqy ? nqx : nqy;
  int s = 0, n_done = 0;
  uint32_t ph = 0;
  // b = bk / K advanced incrementally (the only 64-bit divisions: once per warp)
  int64_t b = gw / K;
  int kk = (int)(gw - b * K);
  const int64_t step_b = total / K;
  const int step_k = (int)(total - step_b * K);
  for (int64_t bk = gw; bk < n_bk; bk += total) {
    // per-sample side inputs: requested by lane 0 before the wait, consumed after the scan
    float cx = 0.f, cy = 0.f, sc0 = 0.f, sc1 = 0.f;
    if (center && lane == 0) { cx = center[2 * b]; cy = center[2 * b + 1]; sc0 = scale[2 * b]; sc1 = scale[2 * b + 1]; }
    b += step_b; kk += step_k;
    if (kk >= K) { kk -= K; ++b; }
    mbar_wait(&bars[s], ph);
    const T* xs = reinterpret_cast<const T*>(wbase + (size_t)s * pair_al);
    const T* ys = xs + Lx;
    LaneBest sx{-CUDART_INF_F, 0xffffffffu}, sy = sx;
#pragma unroll 4
    for (int q = lane; q < nq; q += 32) {
      if (q < nqx) lane_scan4(load4<T>(xs + 4 * q), (uint32_t)q, sx);
      if (q < nqy) lane_scan4(load4<T>(ys + 4 * q), (uint32_t)q, sy);
    }
    uint32_t ix, iy; float mx, my;
    warp_finish<T>(xs, nqx, lane, sx, ix, mx);
    warp_finish<T>(ys, nqy, lane, sy, iy, my);
    __syncwarp();                                             // every lane is done with stage s
    if (lane == 0) {
      const int64_t next = bk + (int64_t)nstg * total;
      if (next < n_bk) { fence_proxy_async(); issue(s, next); }
      simdr_store(ix, iy, mx, my, k, dv, center != nullptr, cx, cy, sc0, sc1, out, out_idx, bk);
    }
    if (++s == nstg) { s = 0; ph ^= 1u; }
    if (overlap && warp == 0 && ++n_done == kRingTriggerPair) {
      asm volatile("griddepcontrol.wait;" ::: "memory");
      asm volatile("griddepcontrol.launch_dependents;");
    }
  }
  if (overlap && warp == 0 && n_done < kRingTriggerPair) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;");
  }
}

// ---- KLDiscretLoss: SmoothL1(beta=1) sums per (b,k), then a fixed-order per-joint reduction -----
__device__ __forceinline__ float smooth_l1(float d) {
  const float a = fabsf(d);
  return a < 1.f ? 0.5f * d * d : a - 0.5f;
}

template <typename T>
__device__ __forceinline__ double warp_sl1_sum(const T* __restrict__ o, const T* __restrict__ t, int L, int lane) {
  float s0 = 0.f, s1 = 0.f;
  const bool vec = ((L & 3) == 0) &&
                   ((reinterpret_cast<uintptr_t>(o) | reinterpret_cast<uintptr_t>(t)) % (4 * sizeof(T)) == 0);
  if (vec) {
    const int nq = L >> 2;
#pragma unroll 4
    for (int q = lane; q < nq; q += 32) {
      const float4 a = ldg_stream4<T>(o + 4 * q), g = ldg_stream4<T>(t + 4 * q);
      s0 += smooth_l1(a.x - g.x); s1 += smooth_l1(a.y - g.y);
      s0 += smooth_l1(a.z - g.z); s1 += smooth_l1(a.w - g.w);
    }
  } else {
    for (int i = lane; i < L; i += 32) s0 += smooth_l1(Elem<T>::to_f32(o[i]) - Elem<T>::to_f32(t[i]));
  }
  return warp_sum((double)s0 + (double)s1);
}

template <typename T>
__global__ void __launch_bounds__(256) simdr_sl1_kernel(const T* __restrict__ ox, const T* __restrict__ oy,
                                                        const T* __restrict__ tx, const T* __restrict__ ty,
                                                        int64_t n_bk, int Lx, int Ly,
                                                        double* __restrict__ per_bk /* [n_bk,2] */) {
  asm volatile("griddepcontrol.launch_dependents;");          // the finalize cluster queues up behind this grid
  const int lane = threadIdx.x & 31;
  const int64_t wg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const bool vec = ((Lx | Ly) & 3) == 0 &&
                   ((reinterpret_cast<uintptr_t>(ox) | reinterpret_cast<uintptr_t>(oy) | reinterpret_cast<uintptr_t>(tx) |
                     reinterpret_cast<uintptr_t>(ty)) % (4 * sizeof(T)) == 0);
  for (int64_t bk = wg; bk < n_bk; bk += nw) {
    double sx, sy;
    if (vec) {
      // both vectors of the pair in ONE loop: all sixteen 128-bit loads of a 512-bin pair are in flight together
      const T* px = ox + bk * Lx; const T* qx = tx + bk * Lx;
      const T* py = oy + bk * Ly; const T* qy = ty + bk * Ly;
      const int nqx = Lx >> 2, nqy = Ly >> 2, nq = nqx > nqy ? nqx : nqy;
      float ax = 0.f, bx = 0.f, ay = 0.f, by = 0.f;
#pragma unroll 4
      for (int q = lane; q < nq; q += 32) {
        if (q < nqx) {
          const float4 a = ldg_stream4<T>(px + 4 * q), g = ldg_stream4<T>(qx + 4 * q);
          ax += smooth_l1(a.x - g.x); bx += smooth_l1(a.y - g.y); ax += smooth_l1(a.z - g.z); bx += smooth_l1(a.w - g.w);
        }
        if (q < nqy) {
          const float4 a = ldg_stream4<T>(py + 4 * q), g = ldg_stream4<T>(qy + 4 * q);
          ay += smooth_l1(a.x - g.x); by += smooth_l1(a.y - g.y); ay += smooth_l1(a.z - g.z); by += smooth_l1(a.w - g.w);
        }
      }
      sx = warp_sum((double)ax + (double)bx);
      sy = warp_sum((double)ay + (double)by);
    } else {
      sx = warp_sl1_sum<T>(ox + bk * Lx, tx + bk * Lx, Lx, lane);
      sy = warp_sl1_sum<T>(oy + bk * Ly, ty + bk * Ly, Ly, lane);
    }
    if (lane == 0) { per_bk[2 * bk] = sx; per_bk[2 * bk + 1] = sy; }
  }
}

// The same scan when the grid's warp count is a multiple of K (the host sizes it so): every row a warp meets belongs
// to ONE joint, so the lanes keep f64 running sums over the warp's rows and are added once, after the loop — no
// shuffle tree between rows (two f64 trees per 4 KB row were a quarter of the warp's instructions and held the next
// row's loads back) and K-fold fewer entries for the finalize.  Entry of warp w: (sum_x, sum_y, sum_weight).
template <typename T>
__global__ void __launch_bounds__(256) simdr_sl1_joint_kernel(const T* __restrict__ ox, const T* __restrict__ oy,
                                                              const T* __restrict__ tx, const T* __restrict__ ty,
                                                              const float* __restrict__ weight,
                                                              int64_t n_bk, int Lx, int Ly,
                                                              double* __restrict__ part /* [warps,3] */) {
  asm volatile("griddepcontrol.launch_dependents;");
  const int lane = threadIdx.x & 31;
  const int64_t wg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int nqx = Lx >> 2, nqy = Ly >> 2, nq = nqx > nqy ? nqx : nqy;
  double accx = 0.0, accy = 0.0, accw = 0.0;
  for (int64_t bk = wg; bk < n_bk; bk += nw) {
    const T* px = ox + bk * Lx; const T* qx = tx + bk * Lx;
    const T* py = oy + bk * Ly; const T* qy = ty + bk * Ly;
    float ax = 0.f, bx = 0.f, ay = 0.f, by = 0.f;
#pragma unroll 4
    for (int q = lane; q < nq; q += 32) {
      if (q < nqx) {
        const float4 a = ldg_stream4<T>(px + 4 * q), g = ldg_stream4<T>(qx + 4 * q);
        ax += smooth_l1(a.x - g.x); bx += smooth_l1(a.y - g.y); ax += smooth_l1(a.z - g.z); bx += smooth_l1(a.w - g.w);
      }
      if (q < nqy) {
        const float4 a = ldg_stream4<T>(py + 4 * q), g = ldg_stream4<T>(qy + 4 * q);
        ay += smooth_l1(a.x - g.x); by += smooth_l1(a.y - g.y); ay += smooth_l1(a.z - g.z); by += smooth_l1(a.w - g.w);
      }
    }
    accx += (double)ax + (double)bx;
    accy += (double)ay + (double)by;
    accw += (double)__ldg(weight + bk);                      // warp-uniform
  }
  accx = warp_sum(accx); accy = warp_sum(accy);
  if (lane == 0) { part[3 * wg] = accx; part[3 * wg + 1] = accy; part[3 * wg + 2] = accw; }
}

// One block.  The first T = (1024 / K) * K threads walk the [B*K] rows with a stride of T — a multiple of K, so a thread
// meets ONE joint and its loads are coalesced (a warp per joint walking b with a stride of K rows touched 32 sectors per
// load) — then the threads of a joint are added in thread order, the joints in joint order: a fixed summation order.
__global__ void __launch_bounds__(1024) simdr_loss_finalize_kernel(const double* __restrict__ per_bk,
                                                                   const float* __restrict__ weight,
                                                                   int64_t B, int K, int Lx, int Ly,
                                                                   float* __restrict__ loss) {
  __shared__ double s_x[1024], s_y[1024], s_w[1024];
  __shared__ double term[1024];
  const int tid = threadIdx.x;
  const int T = K <= (int)blockDim.x ? ((int)blockDim.x / K) * K : 0;
  if (T == 0) {                                               // more joints than threads: the plain loop
    if (tid == 0) {
      double t = 0.0;
      for (int jj = 0; jj < K; ++jj) {
        double sx = 0, sy = 0, sw = 0;
        for (int64_t b = 0; b < B; ++b) { sx += per_bk[2 * (b * K + jj)]; sy += per_bk[2 * (b * K + jj) + 1]; sw += (double)weight[b * K + jj]; }
        t += (sx / ((double)B * Lx) + sy / ((double)B * Ly)) * (sw / (double)B);
      }
      loss[0] = (float)(t / (double)K);
    }
    return;
  }
  double sx = 0, sy = 0, sw = 0;
  if (tid < T) {
    const int64_t n = B * K;
#pragma unroll 8
    for (int64_t i = tid; i < n; i += T) {                    // i % K == tid % K
      const double2 v = __ldcg(reinterpret_cast<const double2*>(per_bk + 2 * i));
      sx += v.x; sy += v.y; sw += (double)__ldg(weight + i);
    }
  }
  s_x[tid] = sx; s_y[tid] = sy; s_w[tid] = sw;
  __syncthreads();
  if (tid < K) {
    double ax = 0, ay = 0, aw = 0;
    for (int t = tid; t < T; t += K) { ax += s_x[t]; ay += s_y[t]; aw += s_w[t]; }
    term[tid] = (ax / ((double)B * Lx) + ay / ((double)B * Ly)) * (aw / (double)B);
  }
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int jj = 0; jj < K; ++jj) t += term[jj];
    loss[0] = (float)(t / (double)K);
  }
}

// The same sum on a cluster of 8 CTAs (one launch of 8 SMs instead of one: the single block spent ~6 us walking the
// [B*K] rows in 43 dependent rounds).  CTA r takes the rows r*T + tid + i*8T — 8T a multiple of K, so a thread still
// meets ONE joint — adds its threads per joint in thread order, and CTA 0 adds the eight per-joint partials in rank
// order through distributed shared memory: a fixed summation order again (a different one from the single block's;
// both agree with the f64 oracle to ~1e-15).  Launched with programmatic stream serialization: it is resident-ready
// when the last rows are written.
constexpr int kFinClusterMaxK = 128;
__global__ void __cluster_dims__(8, 1, 1) __launch_bounds__(1024)
simdr_loss_finalize_cluster_kernel(const double* __restrict__ per_bk, const float* __restrict__ weight,
                                   int64_t n, int64_t B, int K, int Lx, int Ly, float* __restrict__ loss) {
  // weight != nullptr: n = B*K rows of (sx, sy) + weight[row];  weight == nullptr: n per-warp entries of (sx, sy, sw)
  // written by simdr_sl1_joint_kernel.  Either way entry i belongs to joint i % K.
  __shared__ double s_x[1024], s_y[1024], s_w[1024];
  __shared__ double part[3][kFinClusterMaxK];
  __shared__ double term[kFinClusterMaxK];
  unsigned rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  const int tid = threadIdx.x;
  const int T = ((int)blockDim.x / K) * K;
  asm volatile("griddepcontrol.wait;" ::: "memory");
  double sx = 0, sy = 0, sw = 0;
  if (tid < T) {
    if (weight) {
#pragma unroll 8
      for (int64_t i = (int64_t)rank * T + tid; i < n; i += 8 * (int64_t)T) {
        const double2 v = __ldcg(reinterpret_cast<const double2*>(per_bk + 2 * i));
        sx += v.x; sy += v.y; sw += (double)__ldg(weight + i);
      }
    } else {
#pragma unroll 4
      for (int64_t i = (int64_t)rank * T + tid; i < n; i += 8 * (int64_t)T) {
        const double* e = per_bk + 3 * i;
        sx += __ldcg(e); sy += __ldcg(e + 1); sw += __ldcg(e + 2);
      }
    }
  }
  s_x[tid] = sx; s_y[tid] = sy; s_w[tid] = sw;
  __syncthreads();
  if (tid < K) {
    double ax = 0, ay = 0, aw = 0;
    for (int t = tid; t < T; t += K) { ax += s_x[t]; ay += s_y[t]; aw += s_w[t]; }
    part[0][tid] = ax; part[1][tid] = ay; part[2][tid] = aw;
  }
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  if (rank == 0 && tid < K) {
    double ax = 0, ay = 0, aw = 0;
    const unsigned base = (unsigned)__cvta_generic_to_shared(&part[0][0]);
    for (unsigned r = 0; r < 8; ++r) {
      double v[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        unsigned remote;
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(base + (unsigned)((c * kFinClusterMaxK + tid) * 8)), "r"(r));
        asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v[c]) : "r"(remote) : "memory");
      }
      ax += v[0]; ay += v[1]; aw += v[2];
    }
    term[tid] = (ax / ((double)B * Lx) + ay / ((double)B * Ly)) * (aw / (double)B);
  }
  // no CTA may exit while CTA 0 still reads its shared memory
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  if (rank == 0) {
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int jj = 0; jj < K; ++jj) t += term[jj];
      loss[0] = (float)(t / (double)K);
    }
  }
}

template <typename T>
static int launch_simdr(int dtype, const void* xv, const void* yv, int64_t n_bk, int K, int Lx, int Ly, int k,
                        const float* center, const float* scale, int nms, const int32_t* ranges,
                        float* out, int32_t* out_idx, int flags, cudaStream_t st) {
  // Ring kernel: no NMS, TMA-able vectors (16-byte multiples, 16-byte aligned bases), at least two stages per warp,
  // and enough pairs to give every warp of the persistent grid a few (below that the launch is latency-bound anyway).
  {
    const size_t xb = (size_t)Lx * sizeof(T), yb = (size_t)Ly * sizeof(T);
    const size_t pair_al = (xb + yb + 127) / 128 * 128;
    int warps = kRingWarps;
    if (const char* e = getenv("LHN_SIMDR_WARPS")) { const int w = atoi(e); if (w >= 1 && w <= 32) warps = w; }
    const size_t bar_bytes = (size_t)warps * kRingMaxStages * 8;
    int nstg = (int)((227 * 1024 - bar_bytes) / (warps * pair_al));
    if (nstg > kRingMaxStages) nstg = kRingMaxStages;
    if (const char* e = getenv("LHN_SIMDR_STAGES")) { const int g = atoi(e); if (g >= 2 && g <= nstg) nstg = g; }
    const char* env = getenv("LHN_SIMDR_RING");
    const bool ring_ok = !nms && !(env && env[0] == '0') && xb % 16 == 0 && yb % 16 == 0 &&
                         ((reinterpret_cast<uintptr_t>(xv) | reinterpret_cast<uintptr_t>(yv)) & 15) == 0 && nstg >= 2 &&
                         n_bk >= (int64_t)num_sms() * warps * 4;
    if (ring_ok) {
      const size_t smem = (size_t)warps * nstg * pair_al + bar_bytes;
      // per launch (the attribute is per device; a host call of ~1 us), as the team kernel does
      cudaError_t e = cudaFuncSetAttribute(decode_simdr_ring_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)smem);
      if (e != cudaSuccess) { set_last_error(e); return LHN_ECUDA; }
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)num_sms()); cfg.blockDim = dim3((unsigned)(warps * 32));
      cfg.dynamicSmemBytes = smem; cfg.stream = st;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[0].val.programmaticStreamSerializationAllowed = 1;
      const int overlap = (flags & LHN_FLAG_OVERLAP_PREVIOUS) ? 1 : 0;
      cfg.attrs = at; cfg.numAttrs = overlap;
      e = cudaLaunchKernelEx(&cfg, decode_simdr_ring_kernel<T>, (const T*)xv, (const T*)yv, n_bk, K, Lx, Ly, k, center, scale,
                             out, out_idx, nstg, (int)pair_al, overlap);
      if (e != cudaSuccess) { set_last_error(e); return LHN_ECUDA; }
      const int rc = check_launch();
      if (rc == LHN_OK) simdr_record(2, 1, dtype, warps, nstg, num_sms(), 1, 1, 0);
      return rc;
    }
  }
  const int threads = 256;
  // grid-stride over (b, k) pairs: exactly the resident CTAs (6 per SM at 40 registers), so there is no second wave
  int64_t need = (n_bk * 32 + threads - 1) / threads, cap = (int64_t)num_sms() * 6;
  int blocks = (int)(need < cap ? need : cap);
  if (nms)
    decode_simdr_kernel<T, true><<<blocks, threads, 0, st>>>((const T*)xv, (const T*)yv, n_bk, K, Lx, Ly, k,
                                                             center, scale, ranges, out, out_idx);
  else
    decode_simdr_kernel<T, false><<<blocks, threads, 0, st>>>((const T*)xv, (const T*)yv, n_bk, K, Lx, Ly, k,
                                                              center, scale, ranges, out, out_idx);
  const int rc = check_launch();
  if (rc == LHN_OK) {
    // the kernel's per-pair `fast` test: every row of an aligned base with L % 4 == 0 is aligned as well
    const bool fast = ((Lx | Ly) & 3) == 0 && ((reinterpret_cast<uintptr_t>(xv) | reinterpret_cast<uintptr_t>(yv)) %
                                              (4 * sizeof(T))) == 0;
    const int path = nms ? 4 : (fast ? 2 : 3);
    simdr_record(2, path, dtype, threads / 32, 0, blocks, path == 2, path == 2, 0);
  }
  return rc;
}

}  // namespace lhn

using namespace lhn;

extern "C" int lhn_decode_simdr(const void* x_vec, const void* y_vec, int dtype, int64_t B, int K,
                                int Lx, int Ly, int split_ratio, const float* center,
                                const float* scale, int nms, const int32_t* ranges, float* out,
                                int32_t* out_idx, lhn_stream_t stream) {
  return lhn_decode_simdr_flags(x_vec, y_vec, dtype, B, K, Lx, Ly, split_ratio, center, scale, nms, ranges, out,
                                out_idx, 0, stream);
}

extern "C" int lhn_decode_simdr_flags(const void* x_vec, const void* y_vec, int dtype, int64_t B, int K,
                                      int Lx, int Ly, int split_ratio, const float* center,
                                      const float* scale, int nms, const int32_t* ranges, float* out,
                                      int32_t* out_idx, int flags, lhn_stream_t stream) {
  g_simdr_launch = {};
  if (!x_vec || !y_vec || !out || B < 0 || K <= 0 || Lx <= 0 || Ly <= 0 || split_ratio <= 0 ||
      ((center == nullptr) != (scale == nullptr)))
    return LHN_EINVAL;
  const int64_t n = B * K;
  if (n == 0) return LHN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  switch (dtype) {
    case LHN_F32: return launch_simdr<float>(dtype, x_vec, y_vec, n, K, Lx, Ly, split_ratio, center, scale, nms, ranges, out, out_idx, flags, st);
    case LHN_BF16: return launch_simdr<__nv_bfloat16>(dtype, x_vec, y_vec, n, K, Lx, Ly, split_ratio, center, scale, nms, ranges, out, out_idx, flags, st);
    case LHN_F16: return launch_simdr<__half>(dtype, x_vec, y_vec, n, K, Lx, Ly, split_ratio, center, scale, nms, ranges, out, out_idx, flags, st);
    default: return LHN_EDTYPE;
  }
}

extern "C" int lhn_simdr_last_launch(lhn_simdr_launch_info* out) {
  if (!out) return LHN_EINVAL;
  *out = g_simdr_launch;
  return LHN_OK;
}

extern "C" int64_t lhn_simdr_loss_workspace_bytes(int64_t B, int K) {
  if (B < 0 || K <= 0) return LHN_EINVAL;
  return B * K * 2 * (int64_t)sizeof(double);
}

extern "C" int lhn_simdr_smoothl1(const void* out_x, const void* out_y, const void* tgt_x,
                                  const void* tgt_y, const float* weight, int dtype, int64_t B, int K,
                                  int Lx, int Ly, void* workspace, int64_t workspace_bytes, float* loss,
                                  lhn_stream_t stream) {
  g_simdr_launch = {};
  if (!out_x || !out_y || !tgt_x || !tgt_y || !weight || !workspace || !loss || B <= 0 || K <= 0 ||
      Lx <= 0 || Ly <= 0)
    return LHN_EINVAL;
  if (workspace_bytes < lhn_simdr_loss_workspace_bytes(B, K)) return LHN_EWORKSPACE;
  if ((uintptr_t)workspace % 16) return LHN_EALIGN;
  const int64_t n = B * K;
  const int threads = 256;
  int64_t need = (n * 32 + threads - 1) / threads, cap = (int64_t)num_sms() * 8;
  int blocks = (int)(need < cap ? need : cap);
  cudaStream_t st = (cudaStream_t)stream;
  double* per_bk = (double*)workspace;
  // read on every call, like LHN_SIMDR_RING / LHN_SIMDR_WARPS: 1 = rows + one block, 2 = rows + cluster (where the shape
  // allows the cluster finalise; otherwise rows + one block)
  const char* mode_env = getenv("LHN_SIMDR_LOSS_PATH");
  const int mode = mode_env ? atoi(mode_env) : 0;
  const size_t es = dtype == LHN_F32 ? 4 : 2;
  const bool vec = ((Lx | Ly) & 3) == 0 && (((uintptr_t)out_x | (uintptr_t)out_y | (uintptr_t)tgt_x | (uintptr_t)tgt_y) % (4 * es)) == 0;
  auto finalize_cluster = [&](const float* w, int64_t entries) -> int {
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[1];
    cfg.gridDim = dim3(8); cfg.blockDim = dim3(1024); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, simdr_loss_finalize_cluster_kernel, (const double*)per_bk, w, entries, B, K, Lx, Ly, loss);
    if (e != cudaSuccess) { cudaGetLastError(); return LHN_ECUDA; }
    return LHN_OK;
  };
  if (need > cap && vec && K <= kFinClusterMaxK && mode == 0) {
    // warps: a multiple of K (one joint per warp) and of 8 (whole CTAs), with rows / warps just under an integer so
    // every warp walks the same number of rows (43008 rows: 8736 warps x 4.92 rows instead of 9472 x 4.54)
    auto gcd = [](int64_t x, int64_t y) { while (y) { const int64_t t = x % y; x = y; y = t; } return x; };
    const int64_t unit = 8 * (int64_t)K / gcd(8, K);
    // ... and no more CTAs than are resident at once (6 per SM at 40 registers): a second, thin wave of CTAs would
    // walk its rows with a fraction of the loads in flight
    static int resident[3] = {0, 0, 0};
    const int di = dtype == LHN_F32 ? 0 : dtype == LHN_BF16 ? 1 : 2;
    if (!resident[di]) {
      int nb = 0;
      cudaError_t e = di == 0 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, simdr_sl1_joint_kernel<float>, threads, 0)
                    : di == 1 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, simdr_sl1_joint_kernel<__nv_bfloat16>, threads, 0)
                              : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, simdr_sl1_joint_kernel<__half>, threads, 0);
      if (e != cudaSuccess) { cudaGetLastError(); nb = 0; }
      resident[di] = nb > 0 ? nb : 4;
    }
    cap = (int64_t)num_sms() * resident[di];
    const int64_t rounds = (n + cap * 8 - 1) / (cap * 8);
    int64_t warps = (n + rounds - 1) / rounds;
    warps = (warps + unit - 1) / unit * unit;
    if (warps * 3 * (int64_t)sizeof(double) <= workspace_bytes && warps / 8 <= 2 * cap) {
      const int jb = (int)(warps / 8);
      switch (dtype) {
        case LHN_F32:
          simdr_sl1_joint_kernel<float><<<jb, threads, 0, st>>>((const float*)out_x, (const float*)out_y,
              (const float*)tgt_x, (const float*)tgt_y, weight, n, Lx, Ly, per_bk);
          break;
        case LHN_BF16:
          simdr_sl1_joint_kernel<__nv_bfloat16><<<jb, threads, 0, st>>>((const __nv_bfloat16*)out_x,
              (const __nv_bfloat16*)out_y, (const __nv_bfloat16*)tgt_x, (const __nv_bfloat16*)tgt_y, weight, n, Lx, Ly, per_bk);
          break;
        case LHN_F16:
          simdr_sl1_joint_kernel<__half><<<jb, threads, 0, st>>>((const __half*)out_x, (const __half*)out_y,
              (const __half*)tgt_x, (const __half*)tgt_y, weight, n, Lx, Ly, per_bk);
          break;
        default: return LHN_EDTYPE;
      }
      int rc = check_launch();
      if (rc) return rc;
      rc = finalize_cluster(nullptr, warps);
      if (rc == LHN_OK) simdr_record(3, 1, dtype, threads / 32, 0, jb, 1, 1, 0);
      return rc;
    }
  }
  switch (dtype) {
    case LHN_F32:
      simdr_sl1_kernel<float><<<blocks, threads, 0, st>>>((const float*)out_x, (const float*)out_y,
          (const float*)tgt_x, (const float*)tgt_y, n, Lx, Ly, per_bk);
      break;
    case LHN_BF16:
      simdr_sl1_kernel<__nv_bfloat16><<<blocks, threads, 0, st>>>((const __nv_bfloat16*)out_x,
          (const __nv_bfloat16*)out_y, (const __nv_bfloat16*)tgt_x, (const __nv_bfloat16*)tgt_y, n, Lx, Ly, per_bk);
      break;
    case LHN_F16:
      simdr_sl1_kernel<__half><<<blocks, threads, 0, st>>>((const __half*)out_x, (const __half*)out_y,
          (const __half*)tgt_x, (const __half*)tgt_y, n, Lx, Ly, per_bk);
      break;
    default: return LHN_EDTYPE;
  }
  int rc = check_launch();
  if (rc) return rc;
  if (K <= kFinClusterMaxK && n >= 8192 && mode != 1) {
    rc = finalize_cluster(weight, n);
    if (rc == LHN_OK) simdr_record(3, 2, dtype, threads / 32, 0, blocks, vec, vec, 0);
    return rc;
  }
  simdr_loss_finalize_kernel<<<1, 1024, 0, st>>>(per_bk, weight, B, K, Lx, Ly, loss);
  rc = check_launch();
  // the finalise walks the joints in one thread when they outnumber its 1024 threads
  if (rc == LHN_OK) simdr_record(3, K > 1024 ? 4 : 3, dtype, threads / 32, 0, blocks, vec, vec, 0);
  return rc;
}
