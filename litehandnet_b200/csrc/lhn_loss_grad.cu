// The fused heatmap loss and its gradient in ONE pass over the network output (the backward of the fused
// entry without a second read of the heatmaps).
//
// The balanced DistanceLoss scales the positives by 0.1/(N_pos+1) and the rest by 1/(N_neg+1), with N_pos
// counted over the whole batch — but N_pos counts `target > value`, and the target is rendered from the
// joints: it does not depend on the prediction.  So the kernel first counts the positives from the joints
// alone (a small window around each joint, exactly as the fused forward does), meets at a grid-wide barrier
// (persistent, cooperatively launched grid), and then streams every plane once: render the target into
// shared tables, accumulate the loss sums, write d loss / d output with 16-byte stores.  The first plane's
// loads are issued before the barrier, and each plane's f64 geometry is computed once, by one thread.  A last-CTA ticket adds the per-CTA rows in a fixed order and
// finalises the loss as lhn_loss_finalize does; bitwise reproducible for a given shape and device, and the
// workspace is left zeroed.
//
// The gradient assumes an upstream gradient `grad_scale` (what autograd will deliver to the loss).  The
// conditional backward compares the upstream value it actually receives with that assumption: bitwise
// equal -> nothing to do; otherwise it rewrites the gradient exactly as lhn_render_loss_backward would.
#include <math_constants.h>

#include <type_traits>

#include "lhn_common.cuh"

namespace lhn {
int num_sms();

constexpr int kGradThreads = 256;
constexpr int kGradWarps = kGradThreads / 32;
constexpr int kGradUnroll = 4;          // 16-byte chunks in flight per thread
constexpr int kGradGridCap = 4096;      // bound of the persistent grid (sizes the workspace without a device query)
constexpr int kWsRows = 256;            // workspace: [0] barrier, [64] ticket, [128] N_pos; rows from byte 256

struct LossGradArgs {
  const void* hm; void* grad;
  int64_t stride_b, stride_c;
  const float* joints; int joints_stride;
  const float* vis; int vis_stride;
  int64_t n_planes;
  int S, K, H, W, unbiased, loss_mode, sum_reduction;
  double feat_x, feat_y;
  float sigma[LHN_MAX_STACKS];
  float pos_radius[LHN_MAX_STACKS];
  float pos_value, scale;
  const float* grad_scale;        // one pass: the upstream value assumed (NULL = 1); conditional: grad_out
  // one pass
  float* out_weight; double* sums_out; float* loss_out; float* used_scale;
  unsigned int* barrier; unsigned int* ticket; unsigned long long* npos; double* rows;
  // conditional backward
  const double* sums; const float* used_in; int* recomputed;
};

// ---- 16-byte (or 8-, 4-, 2-byte) chunks of VE elements ---------------------------------------------------
template <typename T, int VE>
__device__ __forceinline__ uint4 ld_chunk(const T* p) {
  uint4 r = make_uint4(0u, 0u, 0u, 0u);
  if constexpr (VE * sizeof(T) == 16) {
    r = ldg_stream_u4(reinterpret_cast<const uint4*>(p));
  } else if constexpr (VE * sizeof(T) == 8) {
    const uint2 v = ldg_stream_u2(reinterpret_cast<const uint2*>(p));
    r.x = v.x; r.y = v.y;
  } else if constexpr (sizeof(T) == 4) {
    r.x = __float_as_uint(__ldg(reinterpret_cast<const float*>(p)));
  } else {
    r.x = __ldg(reinterpret_cast<const unsigned short*>(p));
  }
  return r;
}

template <typename T>
__device__ __forceinline__ float2 unpack2(uint32_t u) {
  if constexpr (sizeof(T) == 4) {
    return make_float2(__uint_as_float(u), 0.f);
  } else if constexpr (std::is_same<T, __nv_bfloat16>::value) {
    return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
  } else {
    return __half22float2(*reinterpret_cast<const __half2*>(&u));
  }
}

template <typename T, int VE>
__device__ __forceinline__ void unpack_chunk(const uint4& r, float (&v)[VE]) {
  if constexpr (sizeof(T) == 4) {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int j = 0; j < VE; ++j) v[j] = __uint_as_float(w[j]);
  } else if constexpr (VE == 1) {
    v[0] = unpack2<T>(r.x).x;
  } else {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int j = 0; j < VE / 2; ++j) { const float2 f = unpack2<T>(w[j]); v[2 * j] = f.x; v[2 * j + 1] = f.y; }
  }
}

template <typename T>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  if constexpr (std::is_same<T, __nv_bfloat16>::value) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
}

template <typename T, int VE>
__device__ __forceinline__ void st_chunk(T* p, const float (&r)[VE]) {
  if constexpr (VE == 1) {
    *p = Store4<T>::from(r[0]);
  } else if constexpr (sizeof(T) == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(r[0], r[1], r[2], r[3]);
  } else if constexpr (VE == 8) {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack2<T>(r[0], r[1]), pack2<T>(r[2], r[3]), pack2<T>(r[4], r[5]),
                                              pack2<T>(r[6], r[7]));
  } else {
    *reinterpret_cast<uint2*>(p) = make_uint2(pack2<T>(r[0], r[1]), pack2<T>(r[2], r[3]));
  }
}

// ---- per-plane geometry and Gaussian tables (as the fused forward and lhn_render_loss_backward) -----------
struct PlaneIdx { int64_t b; int c, s, k; };

__device__ __forceinline__ PlaneIdx plane_idx(const LossGradArgs& a, int64_t p) {
  PlaneIdx r;
  const int C = a.S * a.K;
  r.b = p / C;
  r.c = (int)(p - r.b * C);
  r.s = r.c / a.K; r.k = r.c - r.s * a.K;
  return r;
}

__device__ __forceinline__ RenderGeom plane_geom(const LossGradArgs& a, const PlaneIdx& q) {
  const float* jp = a.joints + (q.b * a.K + q.k) * (int64_t)a.joints_stride;
  return render_geom(jp[0], jp[1], a.vis[(q.b * a.K + q.k) * (int64_t)a.vis_stride], (double)a.sigma[q.s], a.unbiased,
                     a.feat_x, a.feat_y, 0, 0.0, 0.0, a.W, a.H);
}

// a plane's geometry with its stack index and 1 / (2 sigma^2), as the tables need them
struct PlaneRec {
  RenderGeom g;
  double inv2s2;
  int s;
};

__device__ __forceinline__ PlaneRec plane_rec(const LossGradArgs& a, int64_t p) {
  PlaneRec r;
  const PlaneIdx q = plane_idx(a, p);
  r.g = plane_geom(a, q);
  r.s = q.s;
  const double sig = (double)a.sigma[q.s];
  r.inv2s2 = 1.0 / (2.0 * sig * sig);
  return r;
}

__device__ __forceinline__ const void* plane_src(const LossGradArgs& a, int64_t p, size_t esz) {
  const PlaneIdx q = plane_idx(a, p);
  return reinterpret_cast<const unsigned char*>(a.hm) + (size_t)(q.b * a.stride_b + (int64_t)q.c * a.stride_c) * esz;
}

// One group of up to kGradUnroll chunks per thread, starting at chunk c0: gradient (and, with LOSS, the f32 loss sums
// of this thread).  Per element exactly the arithmetic of render_loss_backward_kernel.
template <typename T, int VE, bool LOSS>
__device__ __forceinline__ void process_group(const uint4 (&raw)[kGradUnroll], int c0, int nch, int W, T* dst,
                                              const float* ex, const float* ey, float wp, float wn, bool bal, float pv,
                                              float& sp, float& sn) {
#pragma unroll
  for (int u = 0; u < kGradUnroll; ++u) {
    const int c = c0 + u * kGradThreads;
    if (c < nch) {
      const int e0 = c * VE;
      const int row = e0 / W, col = e0 - row * W;
      float v[VE], r[VE];
      unpack_chunk<T, VE>(raw[u], v);
      const float gy = ey[row];
#pragma unroll
      for (int j = 0; j < VE; ++j) {
        const float gx = ex[col + j];
        const float g = gx * gy;
        const float d = fmaf(-gx, gy, v[j]);
        const bool pos = bal && g > pv;
        r[j] = (pos ? wp : wn) * d;
        if (LOSS) { const float l = d * d; sp += pos ? l : 0.f; sn += pos ? 0.f : l; }
      }
      st_chunk<T, VE>(dst + e0, r);
    }
  }
}

template <typename T, int VE>
__device__ __forceinline__ void load_group(uint4 (&raw)[kGradUnroll], const T* src, int c0, int nch) {
#pragma unroll
  for (int u = 0; u < kGradUnroll; ++u) {
    const int c = c0 + u * kGradThreads;
    if (c < nch) raw[u] = ld_chunk<T, VE>(src + (size_t)c * VE);
  }
}

__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ---- the one-pass kernel ----------------------------------------------------------------------------------
template <typename T, int VE>
__global__ void __launch_bounds__(kGradThreads, 3) render_loss_grad_kernel(const __grid_constant__ LossGradArgs a) {
  // dynamic shared memory: the geometry of up to kGradThreads of this CTA's planes (each computed ONCE, by one
  // thread: f64 geometry per thread and plane cost as much SM time as the stream itself), the tables [2][W+H], and
  // for the full-plane window of value <= 0 a [W+H] scratch per warp
  extern __shared__ double smem_d[];
  PlaneRec* geo = reinterpret_cast<PlaneRec*>(smem_d);
  float* tabs = reinterpret_cast<float*>(geo + kGradThreads);
  __shared__ double red[kGradWarps][3];
  __shared__ double s_sums[4];
  __shared__ unsigned int s_cnt, s_last;
  const int W = a.W, H = a.H, WH = W + H, HW = W * H;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nch = HW / VE;
  const int64_t n = a.n_planes, G = gridDim.x;
  const int64_t mine = n > (int64_t)blockIdx.x ? (n - 1 - blockIdx.x) / G + 1 : 0;   // planes blockIdx.x + i G
  const bool bal = a.loss_mode == LHN_LOSS_DISTANCE_BALANCE;
  const bool count = bal && a.pos_value < 1.f;            // value >= 1: no element can be positive
  const bool small = a.pos_value > 0.f && a.pos_value < 1.f;
  if (blockIdx.x == 0 && tid == 0 && a.used_scale) a.used_scale[0] = a.grad_scale ? a.grad_scale[0] : 1.f;

  // ---- geometry of this CTA's planes and N_pos, counted from the joints in the forward's window ---------
  if (tid == 0) s_cnt = 0u;
  unsigned int cnt = 0;
  for (int64_t i = tid; i < mine; i += kGradThreads) {
    const PlaneRec r = plane_rec(a, blockIdx.x + i * G);
    if (i < kGradThreads) geo[i] = r;
    if (count && small && r.g.on) {
      // one thread per plane: the window around the joint (5 x 5 for sigma 2, value 0.5)
      const float rad = a.pos_radius[r.s];
      const int x_lo = max(0, (int)ceilf(r.g.cx - rad)), x_hi = min(W - 1, (int)floorf(r.g.cx + rad));
      const int y_lo = max(0, (int)ceilf(r.g.cy - rad)), y_hi = min(H - 1, (int)floorf(r.g.cy + rad));
      for (int yy = y_lo; yy <= y_hi; ++yy) {
        const float gy = table_entry(r.g, W + yy, W, a.unbiased, r.inv2s2);
        for (int xx = x_lo; xx <= x_hi; ++xx)
          cnt += (table_entry(r.g, xx, W, a.unbiased, r.inv2s2) * gy > a.pos_value) ? 1u : 0u;
      }
    }
  }
  __syncthreads();                                          // geo[] and s_cnt visible
  if (count && !small) {
    // value <= 0: the window is the whole plane; a warp per plane with its tables in a scratch
    float* wt = tabs + (size_t)(2 + warp) * WH;
    for (int64_t i = warp; i < mine; i += kGradWarps) {
      const PlaneRec r = i < kGradThreads ? geo[i] : plane_rec(a, blockIdx.x + i * G);
      if (!(r.g.on || a.pos_value < 0.f)) continue;
      for (int j = lane; j < WH; j += 32) wt[j] = table_entry(r.g, j, W, a.unbiased, r.inv2s2);
      __syncwarp();
      for (int e = lane; e < HW; e += 32) {
        const int ry = e / W, rx = e - ry * W;
        cnt += (wt[rx] * wt[W + ry] > a.pos_value) ? 1u : 0u;
      }
      __syncwarp();
    }
  }
  // the first plane's loads go out before the grid barrier
  int64_t p = blockIdx.x;
  uint4 raw[kGradUnroll];
  if (p < n) load_group<T, VE>(raw, reinterpret_cast<const T*>(plane_src(a, p, sizeof(T))), tid, nch);
  if (count) {
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0 && cnt) atomicAdd(&s_cnt, cnt);
    __syncthreads();
    // grid-wide barrier: every CTA has added its count (the launch is cooperative: all CTAs are resident)
    if (tid == 0) {
      if (s_cnt) atomicAdd(a.npos, (unsigned long long)s_cnt);
      __threadfence();
      atomicAdd(a.barrier, 1u);
      while (ld_acquire_u32(a.barrier) < gridDim.x) __nanosleep(64);
    }
    __syncthreads();
  }
  if (tid == 0) {
    s_sums[0] = s_sums[1] = 0.0;
    s_sums[2] = count ? (double)__ldcg(a.npos) : 0.0;
    s_sums[3] = (double)n * (double)HW;
  }
  __syncthreads();
  float cpos, cneg;
  loss_coefs(s_sums, a.loss_mode, a.sum_reduction, a.scale, a.grad_scale, cpos, cneg);

  // ---- the stream: one read, one write per element --------------------------------------------------------
  double acc_sp = 0.0, acc_sn = 0.0;
  int64_t planes = 0;
  int buf = 0;
  T* grad = reinterpret_cast<T*>(a.grad);
  // tables of plane i are evaluated (into buffer i & 1) before the loads of plane i go out; one barrier per plane
  auto tables = [&](int64_t i, float* ex) -> float {
    if (i > 0 && i % kGradThreads == 0) {                   // the next kGradThreads planes' geometry
      __syncthreads();
      if (i + tid < mine) geo[tid] = plane_rec(a, blockIdx.x + (i + tid) * G);
      __syncthreads();
    }
    const PlaneRec& r = geo[i % kGradThreads];
    for (int j = tid; j < WH; j += kGradThreads) ex[j] = table_entry(r.g, j, W, a.unbiased, r.inv2s2);
    return r.g.w;
  };
  float wcur = p < n ? tables(0, tabs) : 0.f;
  for (; p < n; p += G, buf ^= 1, ++planes) {
    float* ex = tabs + (size_t)buf * WH;
    float w = wcur;
    if (tid == 0 && a.out_weight) a.out_weight[p] = w;
    if (a.loss_mode == LHN_LOSS_JOINTS_MSE) w *= w;
    const float wp = w * cpos, wn = w * cneg;
    __syncthreads();                    // tables of this plane visible; the other buffer is free (double-buffered)
    const T* src = reinterpret_cast<const T*>(plane_src(a, p, sizeof(T)));
    T* dst = grad + p * (int64_t)HW;
    float sp = 0.f, sn = 0.f;
    for (int c0 = tid; c0 < nch; c0 += kGradUnroll * kGradThreads) {
      if (c0 != tid) load_group<T, VE>(raw, src, c0, nch);
      process_group<T, VE, true>(raw, c0, nch, W, dst, ex, ex + W, wp, wn, bal, a.pos_value, sp, sn);
    }
    acc_sp += (double)sp * (double)w;
    acc_sn += (double)sn * (double)w;
    if (p + G < n) {
      wcur = tables(planes + 1, tabs + (size_t)(buf ^ 1) * WH);
      load_group<T, VE>(raw, reinterpret_cast<const T*>(plane_src(a, p + G, sizeof(T))), tid, nch);
    }
  }

  // ---- CTA row (fixed order), last-CTA ticket, finalisation ------------------------------------------------
  acc_sp = warp_sum(acc_sp); acc_sn = warp_sum(acc_sn);
  if (lane == 0) { red[warp][0] = acc_sp; red[warp][1] = acc_sn; }
  __syncthreads();
  if (tid == 0) {
    double r0 = 0.0, r1 = 0.0;
    for (int i = 0; i < kGradWarps; ++i) { r0 += red[i][0]; r1 += red[i][1]; }
    double* dst = a.rows + 4 * (size_t)blockIdx.x;
    __stcg(reinterpret_cast<double2*>(dst), make_double2(r0, r1));
    __stcg(reinterpret_cast<double2*>(dst) + 1, make_double2((double)planes * (double)HW, 0.0));
    __threadfence();
    s_last = (atomicAdd(a.ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  double v0 = 0.0, v1 = 0.0, v2 = 0.0;
  for (int c = tid; c < (int)gridDim.x; c += kGradThreads) {
    double2* row = reinterpret_cast<double2*>(a.rows + 4 * (size_t)c);
    const double2 x = __ldcg(row), y = __ldcg(row + 1);
    v0 += x.x; v1 += x.y; v2 += y.x;
    __stcg(row, make_double2(0.0, 0.0)); __stcg(row + 1, make_double2(0.0, 0.0));   // leave the workspace zeroed
  }
  v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2);
  __syncthreads();
  if (lane == 0) { red[warp][0] = v0; red[warp][1] = v1; red[warp][2] = v2; }
  __syncthreads();
  if (tid == 0) {
    double sp = 0.0, sn = 0.0, numel = 0.0;
    for (int i = 0; i < kGradWarps; ++i) { sp += red[i][0]; sn += red[i][1]; numel += red[i][2]; }
    const double npos = s_sums[2];
    if (a.sums_out) { a.sums_out[0] = sp; a.sums_out[1] = sn; a.sums_out[2] = npos; a.sums_out[3] = numel; }
    if (a.loss_out) {
      double v;                                             // lhn_loss_finalize
      if (a.loss_mode == LHN_LOSS_DISTANCE_BALANCE) v = 0.1 * sp / (npos + 1.0) + sn / (numel - npos + 1.0);
      else if (a.loss_mode == LHN_LOSS_JOINTS_MSE) v = 0.5 * (sp + sn) / numel;
      else v = (sp + sn) / numel;
      if (a.sum_reduction) v *= numel;
      a.loss_out[0] = (float)(v * (double)a.scale);
    }
    *a.barrier = 0u; *a.ticket = 0u; *a.npos = 0ull;
  }
}

// ---- conditional backward: a no-op when the upstream gradient is the one the forward assumed ---------------
template <typename T, int VE>
__global__ void __launch_bounds__(kGradThreads, 4) render_loss_backward_cond_kernel(const __grid_constant__ LossGradArgs a) {
  extern __shared__ float smem[];     // tables [2][W+H]
  const float go = a.grad_scale ? a.grad_scale[0] : 1.f;
  const bool same = __float_as_uint(go) == __float_as_uint(a.used_in[0]);
  if (blockIdx.x == 0 && threadIdx.x == 0 && a.recomputed) a.recomputed[0] = same ? 0 : 1;
  if (same) return;
  const int W = a.W, H = a.H, WH = W + H, HW = W * H, tid = threadIdx.x;
  const int nch = HW / VE;
  const bool bal = a.loss_mode == LHN_LOSS_DISTANCE_BALANCE;
  float cpos, cneg;
  loss_coefs(a.sums, a.loss_mode, a.sum_reduction, a.scale, a.grad_scale, cpos, cneg);
  T* grad = reinterpret_cast<T*>(a.grad);
  uint4 raw[kGradUnroll];
  int buf = 0;
  for (int64_t p = blockIdx.x; p < a.n_planes; p += gridDim.x, buf ^= 1) {
    const PlaneIdx q = plane_idx(a, p);
    const RenderGeom g = plane_geom(a, q);
    const double sig = (double)a.sigma[q.s], inv2s2 = 1.0 / (2.0 * sig * sig);
    float* ex = smem + (size_t)buf * WH;
    for (int i = tid; i < WH; i += kGradThreads) ex[i] = table_entry(g, i, W, a.unbiased, inv2s2);
    float w = g.w;
    if (a.loss_mode == LHN_LOSS_JOINTS_MSE) w *= w;
    const float wp = w * cpos, wn = w * cneg;
    __syncthreads();
    const T* src = reinterpret_cast<const T*>(plane_src(a, p, sizeof(T)));
    T* dst = grad + p * (int64_t)HW;
    float sp = 0.f, sn = 0.f;
    for (int c0 = tid; c0 < nch; c0 += kGradUnroll * kGradThreads) {
      load_group<T, VE>(raw, src, c0, nch);
      process_group<T, VE, false>(raw, c0, nch, W, dst, ex, ex + W, wp, wn, bal, a.pos_value, sp, sn);
    }
  }
}

}  // namespace lhn

using namespace lhn;

// validation and argument filling shared by both entries (no device access)
static int fill_grad_args(LossGradArgs& a, const void* hm, int dtype, int64_t B, int K, int H, int W, int64_t stride_b,
                          int64_t stride_c, const lhn_render_params* rp, const float* joints, int joints_stride,
                          const float* vis, int vis_stride, int sum_reduction, float scale, void* grad) {
  if (!hm || !rp || !joints || !vis || !grad || B < 0 || K <= 0 || H <= 0 || W <= 0 || joints_stride < 2 ||
      vis_stride < 1 || rp->image_w <= 0 || rp->image_h <= 0 || rp->loss_mode < 1 || rp->loss_mode > 3 ||
      rp->unbiased < 0 || rp->unbiased > 2)
    return LHN_EINVAL;
  if ((int64_t)H * W > 0x7fffffffLL) return LHN_EINVAL;
  const int S = rp->num_stacks > 0 ? rp->num_stacks : 1;
  if (S > LHN_MAX_STACKS) return LHN_EINVAL;
  if (dtype != LHN_F32 && dtype != LHN_BF16 && dtype != LHN_F16) return LHN_EDTYPE;
  a = LossGradArgs{};
  a.hm = hm; a.grad = grad; a.stride_b = stride_b; a.stride_c = stride_c;
  a.joints = joints; a.joints_stride = joints_stride; a.vis = vis; a.vis_stride = vis_stride;
  a.S = S; a.K = K; a.H = H; a.W = W; a.unbiased = rp->unbiased; a.loss_mode = rp->loss_mode;
  a.sum_reduction = sum_reduction; a.n_planes = B * S * K;
  if (rp->unbiased == 2) {
    if (W < 2 || H < 2) return LHN_EINVAL;
    a.feat_x = ((double)rp->image_w - 1.0) / (W - 1.0); a.feat_y = ((double)rp->image_h - 1.0) / (H - 1.0);
  } else {
    a.feat_x = (double)rp->image_w / W; a.feat_y = (double)rp->image_h / H;
  }
  a.pos_value = rp->pos_value; a.scale = scale;
  for (int i = 0; i < S; ++i) {
    if (!(rp->sigma[i] > 0.f)) return LHN_EINVAL;
    a.sigma[i] = rp->sigma[i];
    // the fused forward's window of the positives (lhn_heatmap_team.cuh, host side): same expression, same bits
    const double sg = (double)rp->sigma[i];
    a.pos_radius[i] = (a.pos_value > 0.f && a.pos_value < 1.f) ? (float)(sg * sqrt(-2.0 * log((double)a.pos_value)) * 1.001 + 0.01) : 0.f;
  }
  if (a.n_planes > 0x7fffffffLL) return LHN_EINVAL;
  return LHN_OK;
}

// elements per chunk: 16 bytes where rows and pointers allow it, else 4 elements, else scalar
static int chunk_elems(int dtype, int W, const LossGradArgs& a) {
  const int esz = dtype == LHN_F32 ? 4 : 2;
  auto aligned = [&](int ve) {
    const uintptr_t m = (uintptr_t)ve * esz;
    return (W % ve) == 0 && (uintptr_t)a.hm % m == 0 && (uintptr_t)a.grad % m == 0 &&
           ((uint64_t)a.stride_b * esz) % m == 0 && ((uint64_t)a.stride_c * esz) % m == 0;
  };
  if (esz == 2 && aligned(8)) return 8;
  if (aligned(4)) return 4;
  return 1;
}

template <typename T, int VE>
static int launch_grad(LossGradArgs& a, bool cond, size_t smem, cudaStream_t st) {
  auto kern = cond ? render_loss_backward_cond_kernel<T, VE> : render_loss_grad_kernel<T, VE>;
  // blocks per SM for this dynamic shared memory size, cached per instantiation
  static size_t cached_smem[2] = {(size_t)-1, (size_t)-1};
  static int cached_occ[2] = {0, 0};
  const int ci = cond ? 1 : 0;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_last_error(e); return LHN_ECUDA; }
  }
  if (cached_smem[ci] != smem) {
    int nb = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, kGradThreads, smem);
    if (e != cudaSuccess || nb < 1) { if (e != cudaSuccess) set_last_error(e); else set_last_error(cudaErrorInvalidConfiguration); return LHN_ECUDA; }
    cached_occ[ci] = nb; cached_smem[ci] = smem;
  }
  int64_t grid = (int64_t)num_sms() * cached_occ[ci];
  if (grid > kGradGridCap) grid = kGradGridCap;
  if (grid > a.n_planes) grid = a.n_planes;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kGradThreads);
  cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeCooperative;
  at[0].val.cooperative = 1;
  cfg.attrs = at; cfg.numAttrs = cond ? 0 : 1;            // the grid barrier needs every CTA resident
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a);
  if (e != cudaSuccess) { set_last_error(e); return LHN_ECUDA; }
  return check_launch();
}

static int dispatch_grad(LossGradArgs& a, int dtype, bool cond, cudaStream_t st) {
  const int ve = chunk_elems(dtype, a.W, a);
  const size_t WH = (size_t)a.W + a.H;
  const size_t smem = cond ? 2 * WH * sizeof(float) : kGradThreads * sizeof(PlaneRec) + (2 + kGradWarps) * WH * sizeof(float);
  switch (dtype) {
    case LHN_F32:
      return ve == 4 ? launch_grad<float, 4>(a, cond, smem, st) : launch_grad<float, 1>(a, cond, smem, st);
    case LHN_BF16:
      return ve == 8 ? launch_grad<__nv_bfloat16, 8>(a, cond, smem, st)
           : ve == 4 ? launch_grad<__nv_bfloat16, 4>(a, cond, smem, st) : launch_grad<__nv_bfloat16, 1>(a, cond, smem, st);
    default:
      return ve == 8 ? launch_grad<__half, 8>(a, cond, smem, st)
           : ve == 4 ? launch_grad<__half, 4>(a, cond, smem, st) : launch_grad<__half, 1>(a, cond, smem, st);
  }
}

extern "C" int64_t lhn_render_loss_grad_workspace_bytes(int64_t B, int K, int num_stacks) {
  if (B < 0 || K <= 0) return 0;
  const int64_t planes = B * K * (num_stacks > 0 ? num_stacks : 1);
  return kWsRows + 32 * (planes < kGradGridCap ? planes : (int64_t)kGradGridCap);
}

extern "C" int lhn_render_loss_grad(const void* hm, int dtype, int64_t B, int K, int H, int W, int64_t stride_b,
                                    int64_t stride_c, const lhn_render_params* rp, const float* joints,
                                    int joints_stride, const float* vis, int vis_stride, float* out_weight,
                                    void* workspace, int64_t workspace_bytes, double* sums, int sum_reduction,
                                    float loss_scale, float* loss, const float* grad_scale, float* used_scale,
                                    void* grad, lhn_stream_t stream) {
  if (!workspace) return LHN_EINVAL;
  LossGradArgs a;
  int rc = fill_grad_args(a, hm, dtype, B, K, H, W, stride_b, stride_c, rp, joints, joints_stride, vis, vis_stride,
                          sum_reduction, loss_scale, grad);
  if (rc) return rc;
  if (workspace_bytes < lhn_render_loss_grad_workspace_bytes(B, K, a.S)) return LHN_EWORKSPACE;
  if ((uintptr_t)workspace % 16 || (sums && (uintptr_t)sums % 8)) return LHN_EALIGN;
  if (a.n_planes == 0) return LHN_OK;
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  a.barrier = reinterpret_cast<unsigned int*>(ws);
  a.ticket = reinterpret_cast<unsigned int*>(ws + 64);
  a.npos = reinterpret_cast<unsigned long long*>(ws + 128);
  a.rows = reinterpret_cast<double*>(ws + kWsRows);
  a.out_weight = out_weight; a.sums_out = sums; a.loss_out = loss;
  a.grad_scale = grad_scale; a.used_scale = used_scale;
  return dispatch_grad(a, dtype, false, (cudaStream_t)stream);
}

extern "C" int lhn_render_loss_backward_cond(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                             int64_t stride_b, int64_t stride_c, const lhn_render_params* rp,
                                             const float* joints, int joints_stride, const float* vis,
                                             int vis_stride, const double* sums, int sum_reduction, float scale,
                                             const float* grad_out, const float* used_scale, int32_t* recomputed,
                                             void* grad, lhn_stream_t stream) {
  if (!sums || !used_scale) return LHN_EINVAL;
  LossGradArgs a;
  int rc = fill_grad_args(a, hm, dtype, B, K, H, W, stride_b, stride_c, rp, joints, joints_stride, vis, vis_stride,
                          sum_reduction, scale, grad);
  if (rc) return rc;
  if (a.n_planes == 0) return LHN_OK;
  a.sums = sums; a.grad_scale = grad_out; a.used_in = used_scale; a.recomputed = recomputed;
  return dispatch_grad(a, dtype, true, (cudaStream_t)stream);
}
