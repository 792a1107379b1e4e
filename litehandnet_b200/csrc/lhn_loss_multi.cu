// DistanceLoss / JointsDistanceLoss against explicit target tensors in ONE launch, for up to 8 tensor pairs at once
// (loss/heatmapLoss.py:195-265; SRHandNetLoss sums four scales, loss/loss.py:59-66: loss = sum_i w_i * L2_i).
//
// The un-fused criterion used to be three launches per tensor (per-plane partials -> cluster reduce -> finalise), i.e.
// twelve for SRHandNetLoss.  Here every CTA belongs to one tensor (CTAs are dealt out in proportion to the bytes of
// each tensor), a warp streams whole planes of `output` and `target` with 128-bit loads and keeps f64 sums, the CTA
// adds its warps in a fixed order and publishes one row, and the last CTA of the grid (ticket) adds the rows of every
// tensor in a fixed order, finalises each loss and their weighted sum.  Bitwise reproducible for a given shape and
// device; both inputs are read exactly once.
//
// lhn_render_loss_multi is the same kernel with the target rendered from the joints instead of read (RENDER = true):
// each warp evaluates its plane's separable tables ex[W], ey[H] into warp-private shared memory with render_geom /
// table_entry, and the target element is the f32 product ex[x] * ey[y] that lhn_render_targets writes.  The grid
// dealing, the per-element terms, the row publish and the last-CTA finalise are those of the explicit-target route.
#include <math_constants.h>

#include "lhn_common.cuh"

namespace lhn {

int num_sms();

constexpr int kLossMaxTensors = LHN_LOSS_MAX_TENSORS;
constexpr int kLossThreads = 256;
constexpr int kLossWarps = kLossThreads / 32;

struct LossTensor {
  const void* out;
  const void* tgt;
  const float* w;            // [n_planes]
  int64_t n_planes, HW;
  float loss_weight;
  int cta_begin;             // first CTA of this tensor; tensor i owns CTAs [cta_begin[i], cta_begin[i+1])
};

struct RenderScale {         // RENDER only: where plane (b, k) of this scale lives and how its target is drawn
  int64_t stride_b, stride_c;
  double feat_x, feat_y;
  float sigma;
  int H, W;
  float* w_out;              // optional [B*K]: target_weight after the visibility rule
};

struct LossMultiArgs {
  LossTensor t[kLossMaxTensors];
  RenderScale r[kLossMaxTensors];
  const float* joints; const float* vis;
  int joints_stride, vis_stride, K, unbiased, tab_stride;
  int n, cta_end;
  int loss_mode, sum_reduction, accumulate;
  float pos_value, scale;
  double* rows;              // [grid, 4]
  unsigned int* ticket;      // zero before the first launch; left zero
  double* sums_out;          // [n, 4] (S_pos, S_neg, N_pos, numel) per tensor (the backward needs them)
  float* per_tensor;         // optional [n]: each tensor's own loss (before loss_weight)
  float* loss_out;           // [1]
};

// RENDER: plane loads issued per lane before the plane's tables are evaluated (a first round of the stream)
constexpr int kRenderPrefetch = 4;

template <typename T, bool RENDER>
__device__ __forceinline__ void loss_multi_body(const LossMultiArgs& a) {
  __shared__ double red[kLossWarps][4];
  __shared__ double tloss[kLossMaxTensors];
  __shared__ unsigned int s_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int ti = 0;
#pragma unroll
  for (int i = 1; i < kLossMaxTensors; ++i)
    if (i < a.n && (int)blockIdx.x >= a.t[i].cta_begin) ti = i;
  const LossTensor& t = a.t[ti];
  const int cta_end = (ti + 1 < a.n) ? a.t[ti + 1].cta_begin : a.cta_end;
  const int64_t wstride = (int64_t)(cta_end - t.cta_begin) * kLossWarps;
  const int64_t HW = t.HW;
  const T* out = reinterpret_cast<const T*>(t.out);
  const T* tgt = reinterpret_cast<const T*>(t.tgt);
  const bool vec = (HW & 3) == 0 && ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(tgt)) % (4 * sizeof(T)) == 0);
  const bool vec8 = (HW & 7) == 0 && ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(tgt)) % 16 == 0);
  const bool bal = a.loss_mode == LHN_LOSS_DISTANCE_BALANCE;
  double acc_sp = 0.0, acc_sn = 0.0, acc_np = 0.0, acc_ne = 0.0;         // this lane's weighted sums
  float njx = 0.f, njy = 0.f, njv = 0.f;                                  // RENDER: the joint of the warp's next plane
  if constexpr (RENDER) {
    const int64_t p0 = (int64_t)((int)blockIdx.x - t.cta_begin) * kLossWarps + warp;
    if (p0 < t.n_planes) { njx = a.joints[p0 * a.joints_stride]; njy = a.joints[p0 * a.joints_stride + 1]; njv = a.vis[p0 * a.vis_stride]; }
  }
  for (int64_t p = (int64_t)((int)blockIdx.x - t.cta_begin) * kLossWarps + warp; p < t.n_planes; p += wstride) {
    float w;
    float sp0 = 0.f, sp1 = 0.f, sn0 = 0.f, sn1 = 0.f;
    int npos = 0;
    // per element: subtract, compare, ONE predicated fused multiply-add into the positive or the negative sum, one
    // predicated count (multiply / select / add / select / add was 8 issue slots; the 16-bit planes, twice the
    // elements per byte, were issue-bound at 75 % of the HBM peak)
    auto quad = [&](const float4& x, const float4& y) {
      const float d0 = x.x - y.x, d1 = x.y - y.y, d2 = x.z - y.z, d3 = x.w - y.w;
      const bool p0 = y.x > a.pos_value, p1 = y.y > a.pos_value, p2 = y.z > a.pos_value, p3 = y.w > a.pos_value;
      if (sizeof(T) == 2) {
        if (p0) { sp0 = __fmaf_rn(d0, d0, sp0); ++npos; } else sn0 = __fmaf_rn(d0, d0, sn0);
        if (p1) { sp1 = __fmaf_rn(d1, d1, sp1); ++npos; } else sn1 = __fmaf_rn(d1, d1, sn1);
        if (p2) { sp0 = __fmaf_rn(d2, d2, sp0); ++npos; } else sn0 = __fmaf_rn(d2, d2, sn0);
        if (p3) { sp1 = __fmaf_rn(d3, d3, sp1); ++npos; } else sn1 = __fmaf_rn(d3, d3, sn1);
      } else {
        // f32 planes are HBM-bound with issue slots to spare: the branch-free select form measured 4 % faster there
        const float l0 = d0 * d0, l1 = d1 * d1, l2 = d2 * d2, l3 = d3 * d3;
        sp0 += p0 ? l0 : 0.f; sn0 += p0 ? 0.f : l0;
        sp1 += p1 ? l1 : 0.f; sn1 += p1 ? 0.f : l1;
        sp0 += p2 ? l2 : 0.f; sn0 += p2 ? 0.f : l2;
        sp1 += p3 ? l3 : 0.f; sn1 += p3 ? 0.f : l3;
        npos += (int)p0 + (int)p1 + (int)p2 + (int)p3;
      }
    };
    if constexpr (!RENDER) {
      const T* o = out + p * HW;
      const T* g = tgt + p * HW;
      w = __ldg(t.w + p);
      if (sizeof(T) == 2 && vec8) {
        const int64_t n8 = HW >> 3;                       // 16-bit planes: 128-bit loads, eight elements per lane
#pragma unroll 4
        for (int64_t q = lane; q < n8; q += 32) {
          float4 x0, x1, y0, y1;
          ldg_stream8<T>(o + 8 * q, x0, x1);
          ldg_stream8<T>(g + 8 * q, y0, y1);
          quad(x0, y0); quad(x1, y1);
        }
      } else if (vec) {
        const int64_t nq = HW >> 2;
#pragma unroll 4
        for (int64_t q = lane; q < nq; q += 32) quad(ldg_stream4<T>(o + 4 * q), ldg_stream4<T>(g + 4 * q));
      } else {
        for (int64_t e = lane; e < HW; e += 32) {
          const float x = Elem<T>::to_f32(o[e]), y = Elem<T>::to_f32(g[e]);
          const float d = x - y, l = d * d;
          const bool pp = y > a.pos_value;
          sp0 += pp ? l : 0.f; sn0 += pp ? 0.f : l; npos += (int)pp;
        }
      }
    } else {
      const RenderScale& rs = a.r[ti];
      const int W = rs.W, H = rs.H, nq = (int)(HW >> 2), n8 = (int)(HW >> 3);
      const int64_t b = p / a.K;
      const int k = (int)(p - b * a.K);
      const T* o = out + b * rs.stride_b + (int64_t)k * rs.stride_c;
      const uintptr_t oa = reinterpret_cast<uintptr_t>(o);
      const bool rvec8 = sizeof(T) == 2 && (HW & 7) == 0 && oa % 16 == 0;
      const bool rvec = (HW & 3) == 0 && oa % (4 * sizeof(T)) == 0;
      // the plane's first loads go out before its tables are evaluated: the table work (W + H f64 entries per warp,
      // four times as much per element on a 16 x 16 plane as on 64 x 64) then overlaps the memory latency
      float4 x[kRenderPrefetch];
      if (rvec8) {
#pragma unroll
        for (int j = 0; j < kRenderPrefetch / 2; ++j)
          if (lane + 32 * j < n8) ldg_stream8<T>(o + 8 * (lane + 32 * j), x[2 * j], x[2 * j + 1]);
      } else if (rvec) {
#pragma unroll
        for (int j = 0; j < kRenderPrefetch; ++j)
          if (lane + 32 * j < nq) x[j] = ldg_stream4<T>(o + 4 * (lane + 32 * j));
      }
      extern __shared__ float4 ltab4[];
      float* ex = reinterpret_cast<float*>(ltab4) + warp * a.tab_stride;
      float* ey = ex + W;
      const float jx = njx, jy = njy, jv = njv;
      if (p + wstride < t.n_planes) {                   // the next plane's joint, while this one is worked on
        const int64_t pn = p + wstride;
        njx = a.joints[pn * a.joints_stride]; njy = a.joints[pn * a.joints_stride + 1]; njv = a.vis[pn * a.vis_stride];
      }
      const double sig = (double)rs.sigma;
      const RenderGeom gm = render_geom(jx, jy, jv, sig, a.unbiased, rs.feat_x, rs.feat_y, 0, 0.0, 0.0, W, H);
      w = gm.w;
      if (rs.w_out && lane == 0) rs.w_out[p] = w;
      const double inv2s2 = 1.0 / (2.0 * sig * sig);
      __syncwarp();                                     // every lane is done with the previous plane's tables
      for (int i = lane; i < W + H; i += 32) ex[i] = table_entry(gm, i, W, a.unbiased, inv2s2);
      __syncwarp();
      // target of elements 4 qi .. 4 qi + 3, as lhn_render_targets writes them; (row, cq) is quad qi's row and quad
      // column when W % 4 == 0, advanced by a fixed step instead of divided out per quad
      const int QR = W >> 2;
      auto tq = [&](int qi, int row, int cq) -> float4 {
        if ((W & 3) == 0) {
          const float4 gx = *reinterpret_cast<const float4*>(ex + 4 * cq);
          const float gy = ey[row];
          return make_float4(gx.x * gy, gx.y * gy, gx.z * gy, gx.w * gy);
        }
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int e = 4 * qi + j, yy = e / W;
          v[j] = ex[e - yy * W] * ey[yy];
        }
        return make_float4(v[0], v[1], v[2], v[3]);
      };
      const int start = rvec8 ? 2 * lane : lane, step = rvec8 ? 64 : 32;
      int row = 0, cq = 0, drow = 0, dcq = 0;
      if ((W & 3) == 0) { row = start / QR; cq = start - row * QR; drow = step / QR; dcq = step - drow * QR; }
      auto advance = [&]() { cq += dcq; row += drow; if (cq >= QR) { cq -= QR; ++row; } };
      if (rvec8) {
        auto oct = [&](int q, const float4& x0, const float4& x1) {
          const int r1 = cq + 1 < QR ? row : row + 1, c1 = cq + 1 < QR ? cq + 1 : 0;
          quad(x0, tq(2 * q, row, cq)); quad(x1, tq(2 * q + 1, r1, c1));
        };
#pragma unroll
        for (int j = 0; j < kRenderPrefetch / 2; ++j) {
          const int q = lane + 32 * j;
          if (q < n8) oct(q, x[2 * j], x[2 * j + 1]);
          advance();
        }
#pragma unroll 4
        for (int q = lane + 32 * (kRenderPrefetch / 2); q < n8; q += 32) {
          float4 x0, x1;
          ldg_stream8<T>(o + 8 * q, x0, x1);
          oct(q, x0, x1);
          advance();
        }
      } else if (rvec) {
#pragma unroll
        for (int j = 0; j < kRenderPrefetch; ++j) {
          if (lane + 32 * j < nq) quad(x[j], tq(lane + 32 * j, row, cq));
          advance();
        }
#pragma unroll 4
        for (int q = lane + 32 * kRenderPrefetch; q < nq; q += 32) {
          quad(ldg_stream4<T>(o + 4 * q), tq(q, row, cq));
          advance();
        }
      } else {
        for (int e = lane; e < (int)HW; e += 32) {
          const int yy = e / W;
          const float xo = Elem<T>::to_f32(o[e]), y = ex[e - yy * W] * ey[yy];
          const float d = xo - y, l = d * d;
          const bool pp = y > a.pos_value;
          sp0 += pp ? l : 0.f; sn0 += pp ? 0.f : l; npos += (int)pp;
        }
      }
    }
    // per-LANE f64 accumulators over the warp's planes (weighted): no shuffle between planes, so the next plane's
    // loads are not held behind a reduction; the lanes are added once, after the loop, in a fixed tree
    const double wp = (a.loss_mode == LHN_LOSS_JOINTS_MSE) ? (double)(w * w) : (double)w;
    if (bal) { acc_sp += ((double)sp0 + (double)sp1) * wp; acc_sn += ((double)sn0 + (double)sn1) * wp; acc_np += (double)npos; }
    else acc_sn += (((double)sp0 + (double)sp1) + ((double)sn0 + (double)sn1)) * wp;
    acc_ne += (double)HW;
  }
  acc_sp = warp_sum(acc_sp); acc_sn = warp_sum(acc_sn); acc_np = warp_sum(acc_np);     // acc_ne is warp-uniform
  if (lane == 0) { red[warp][0] = acc_sp; red[warp][1] = acc_sn; red[warp][2] = acc_np; red[warp][3] = acc_ne; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0;
    for (int i = 0; i < kLossWarps; ++i) { r0 += red[i][0]; r1 += red[i][1]; r2 += red[i][2]; r3 += red[i][3]; }
    double* dst = a.rows + 4 * (size_t)blockIdx.x;
    __stcg(reinterpret_cast<double2*>(dst), make_double2(r0, r1));
    __stcg(reinterpret_cast<double2*>(dst) + 1, make_double2(r2, r3));
    __threadfence();
    s_last = (atomicAdd(a.ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (!s_last) return;
  // ---- last CTA: a GROUP of warps adds the rows of one tensor (8 warps for one tensor, 2 each for four, ...):
  // thread-strided with every load in flight at once, a fixed shuffle tree per warp, then the group's warps in order.
  // (One warp per tensor walked 1184 rows in 37 dependent rounds — ~7 us of every launch.)
  __threadfence();
  int wpt = 1;                                                        // warps per tensor: a power of two <= 8 / n
  while (wpt * 2 * a.n <= kLossWarps) wpt *= 2;
  const int groups = kLossWarps / wpt, grp = warp / wpt, sub = warp % wpt;
  for (int i0 = 0; i0 < a.n; i0 += groups) {
    const int i = i0 + grp;
    double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
    if (i < a.n) {
      const int c0 = a.t[i].cta_begin, c1 = (i + 1 < a.n) ? a.t[i + 1].cta_begin : a.cta_end;
#pragma unroll 8
      for (int c = c0 + sub * 32 + lane; c < c1; c += wpt * 32) {
        const double2 x = __ldcg(reinterpret_cast<const double2*>(a.rows + 4 * (size_t)c));
        const double2 y = __ldcg(reinterpret_cast<const double2*>(a.rows + 4 * (size_t)c) + 1);
        v0 += x.x; v1 += x.y; v2 += y.x; v3 += y.y;
      }
      v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2); v3 = warp_sum(v3);
    }
    __syncthreads();                                                  // red[] is free (first round: read above)
    if (lane == 0) { red[warp][0] = v0; red[warp][1] = v1; red[warp][2] = v2; red[warp][3] = v3; }
    __syncthreads();
    if (i < a.n && sub == 0 && lane == 0) {
      v0 = v1 = v2 = v3 = 0.0;
      for (int w = 0; w < wpt; ++w) { v0 += red[warp + w][0]; v1 += red[warp + w][1]; v2 += red[warp + w][2]; v3 += red[warp + w][3]; }
      if (a.sums_out) { double* s = a.sums_out + 4 * i; s[0] = v0; s[1] = v1; s[2] = v2; s[3] = v3; }
      const double l = finalize_loss(v0, v1, v2, v3, a.loss_mode, a.sum_reduction);
      if (a.per_tensor) a.per_tensor[i] = (float)l;
      // each term rounded to f32 like the reference's 0-dim f32 loss tensors: loss += w_i * mse_i
      tloss[i] = (double)((float)l) * (double)a.t[i].loss_weight;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float total = 0.f;
    for (int i = 0; i < a.n; ++i) total += (float)tloss[i];
    total *= a.scale;
    if (a.loss_out) a.loss_out[0] = a.accumulate ? a.loss_out[0] + total : total;
    *a.ticket = 0u;
  }
}

template <typename T>
__global__ void __launch_bounds__(kLossThreads) loss_multi_kernel(const __grid_constant__ LossMultiArgs a) {
  loss_multi_body<T, false>(a);
}

// the rendered-target body holds the table geometry as well: capped at 80 registers (three CTAs per SM, no spills)
// it would otherwise take 110-120 and keep two
template <typename T>
__global__ void __launch_bounds__(kLossThreads, 3) render_loss_multi_kernel(const __grid_constant__ LossMultiArgs a) {
  loss_multi_body<T, true>(a);
}

template <typename T, bool RENDER>
static void (*loss_kernel())(LossMultiArgs) {
  if constexpr (RENDER) return render_loss_multi_kernel<T>;
  else return loss_multi_kernel<T>;
}

}  // namespace lhn

using namespace lhn;

static int64_t loss_multi_grid() { return (int64_t)num_sms() * 8; }

extern "C" int64_t lhn_loss_mse_workspace_bytes(void) { return 256 + (loss_multi_grid() + kLossMaxTensors) * 32; }

// Blocks of the kernel resident per SM (at most 8), per dtype and dynamic shared memory size.
template <bool RENDER>
static int resident_ctas(int di, size_t smem) {
  static int resident[3] = {0, 0, 0};
  static size_t resident_smem[3] = {0, 0, 0};
  if (!resident[di] || resident_smem[di] != smem) {
    int nb = 0;
    cudaError_t e = di == 0 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, loss_kernel<float, RENDER>(), kLossThreads, smem)
                  : di == 1 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, loss_kernel<__nv_bfloat16, RENDER>(), kLossThreads, smem)
                            : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, loss_kernel<__half, RENDER>(), kLossThreads, smem);
    if (e != cudaSuccess) { cudaGetLastError(); nb = 0; }
    resident[di] = nb > 0 ? (nb < 8 ? nb : 8) : 4;
    resident_smem[di] = smem;
  }
  return resident[di];
}

// Deals CTAs to the tensors (a.t[i].cta_begin, a.cta_end) from their plane counts and sizes; the caller has set
// a.n.  The grid: only as many CTAs as are resident at once (a second wave starts thin), and per tensor a warp
// count that puts planes / warps just under an integer, so every warp walks the same number of planes.
static int deal_ctas(LossMultiArgs& a, const int64_t* n_planes, const int64_t* plane_elems, int64_t grid_max) {
  const int n_tensors = a.n;
  double total_elems = 0.0;
  for (int i = 0; i < n_tensors; ++i) total_elems += (double)n_planes[i] * (double)plane_elems[i];
  // pass 1: CTAs in proportion to each tensor's elements, at least one, at most one per kLossWarps planes; pass 2: what
  // the capped (small) tensors left over goes to the others, so a small problem still gets a warp per plane
  int64_t wants[kLossMaxTensors], caps[kLossMaxTensors], used = 0;
  for (int i = 0; i < n_tensors; ++i) {
    wants[i] = (int64_t)((double)grid_max * ((double)n_planes[i] * (double)plane_elems[i] / total_elems));
    caps[i] = (n_planes[i] + kLossWarps - 1) / kLossWarps;
    if (wants[i] > caps[i]) wants[i] = caps[i];
    if (wants[i] < 1) wants[i] = 1;
    used += wants[i];
  }
  for (int i = 0; i < n_tensors && used < grid_max; ++i) {
    const int64_t more = caps[i] - wants[i] < grid_max - used ? caps[i] - wants[i] : grid_max - used;
    wants[i] += more; used += more;
  }
  int cta = 0;
  for (int i = 0; i < n_tensors; ++i) {
    a.t[i].n_planes = n_planes[i]; a.t[i].HW = plane_elems[i];
    a.t[i].cta_begin = cta;
    int64_t want = wants[i];
    {
      // planes / warps just under an integer: every warp walks the same number of planes
      const int64_t rounds = (n_planes[i] + want * kLossWarps - 1) / (want * kLossWarps);
      const int64_t warps = (n_planes[i] + rounds - 1) / rounds;
      want = (warps + kLossWarps - 1) / kLossWarps;
    }
    cta += (int)want;
  }
  a.cta_end = cta;
  return cta;
}

// The workspace, outputs and the launch, common to both entry points.
template <bool RENDER>
static int launch_loss_multi(LossMultiArgs& a, const int64_t* n_planes, const int64_t* plane_elems, int dtype,
                             size_t smem, void* workspace, double* sums, float* per_tensor_loss, float* loss,
                             lhn_stream_t stream) {
  const int di = dtype == LHN_F32 ? 0 : dtype == LHN_BF16 ? 1 : 2;
  const int64_t grid_max = (int64_t)num_sms() * resident_ctas<RENDER>(di, smem);
  const int cta = deal_ctas(a, n_planes, plane_elems, grid_max);
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  a.ticket = reinterpret_cast<unsigned int*>(ws);
  a.rows = reinterpret_cast<double*>(ws + 256);
  a.sums_out = sums; a.per_tensor = per_tensor_loss; a.loss_out = loss;
  if ((int64_t)cta > grid_max + kLossMaxTensors) return LHN_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  switch (dtype) {
    case LHN_F32: loss_kernel<float, RENDER>()<<<cta, kLossThreads, smem, st>>>(a); break;
    case LHN_BF16: loss_kernel<__nv_bfloat16, RENDER>()<<<cta, kLossThreads, smem, st>>>(a); break;
    default: loss_kernel<__half, RENDER>()<<<cta, kLossThreads, smem, st>>>(a); break;
  }
  return check_launch();
}

extern "C" int lhn_loss_mse_multi(int n_tensors, const void* const* outputs, const void* const* targets,
                                  const float* const* weights, const int64_t* n_planes, const int64_t* plane_elems,
                                  const float* loss_weights, int dtype, int loss_mode, float pos_value,
                                  int sum_reduction, float scale, void* workspace, int64_t workspace_bytes,
                                  double* sums, float* per_tensor_loss, float* loss, int accumulate,
                                  lhn_stream_t stream) {
  if (n_tensors < 1 || n_tensors > kLossMaxTensors || !outputs || !targets || !weights || !n_planes || !plane_elems ||
      !workspace || loss_mode < LHN_LOSS_DISTANCE || loss_mode > LHN_LOSS_JOINTS_MSE)
    return LHN_EINVAL;
  if (dtype != LHN_F32 && dtype != LHN_BF16 && dtype != LHN_F16) return LHN_EDTYPE;
  if (workspace_bytes < lhn_loss_mse_workspace_bytes()) return LHN_EWORKSPACE;
  if ((uintptr_t)workspace % 16 || (sums && (uintptr_t)sums % 8)) return LHN_EALIGN;
  LossMultiArgs a{};
  a.n = n_tensors;
  for (int i = 0; i < n_tensors; ++i) {
    if (!outputs[i] || !targets[i] || !weights[i] || n_planes[i] <= 0 || plane_elems[i] <= 0) return LHN_EINVAL;
    a.t[i].out = outputs[i]; a.t[i].tgt = targets[i]; a.t[i].w = weights[i];
    a.t[i].loss_weight = loss_weights ? loss_weights[i] : 1.f;
  }
  a.loss_mode = loss_mode; a.sum_reduction = sum_reduction; a.accumulate = accumulate;
  a.pos_value = pos_value; a.scale = scale;
  return launch_loss_multi<false>(a, n_planes, plane_elems, dtype, 0, workspace, sums, per_tensor_loss, loss, stream);
}

extern "C" int64_t lhn_render_loss_multi_workspace_bytes(void) { return lhn_loss_mse_workspace_bytes(); }

extern "C" int lhn_render_loss_multi(int n_scales, const lhn_loss_scale* scales, int dtype, int64_t B, int K,
                                     const lhn_render_params* rp, const float* joints, int joints_stride,
                                     const float* vis, int vis_stride, int sum_reduction, float scale,
                                     void* workspace, int64_t workspace_bytes, double* sums, float* per_scale_loss,
                                     float* loss, lhn_stream_t stream) {
  if (n_scales < 1 || n_scales > kLossMaxTensors || !scales || !rp || !joints || !vis || !workspace || B <= 0 ||
      K <= 0 || joints_stride < 2 || vis_stride < 1)
    return LHN_EINVAL;
  if (dtype != LHN_F32 && dtype != LHN_BF16 && dtype != LHN_F16) return LHN_EDTYPE;
  if (workspace_bytes < lhn_render_loss_multi_workspace_bytes()) return LHN_EWORKSPACE;
  if ((uintptr_t)workspace % 16 || (sums && (uintptr_t)sums % 8)) return LHN_EALIGN;
  LossMultiArgs a{};
  a.n = n_scales;
  int64_t n_planes[kLossMaxTensors], plane_elems[kLossMaxTensors];
  int tab = 0;
  for (int i = 0; i < n_scales; ++i) {
    const lhn_loss_scale& sc = scales[i];
    RenderScale& r = a.r[i];
    if (!sc.output || scale_geometry(rp, sc.H, sc.W, sc.sigma, r.feat_x, r.feat_y) != LHN_OK) return LHN_EINVAL;
    a.t[i].out = sc.output; a.t[i].loss_weight = sc.loss_weight;
    r.stride_b = sc.stride_b; r.stride_c = sc.stride_c; r.sigma = sc.sigma; r.H = sc.H; r.W = sc.W;
    r.w_out = sc.out_weight;
    n_planes[i] = B * K; plane_elems[i] = (int64_t)sc.H * sc.W;
    if (sc.H + sc.W > tab) tab = sc.H + sc.W;
  }
  a.joints = joints; a.joints_stride = joints_stride; a.vis = vis; a.vis_stride = vis_stride; a.K = K;
  a.unbiased = rp->unbiased; a.tab_stride = (tab + 3) & ~3;
  a.loss_mode = rp->loss_mode; a.sum_reduction = sum_reduction; a.accumulate = 0;
  a.pos_value = rp->pos_value; a.scale = scale;
  const size_t smem = (size_t)kLossWarps * a.tab_stride * sizeof(float);
  if (set_dynamic_smem(dtype == LHN_F32 ? (const void*)render_loss_multi_kernel<float>
                       : dtype == LHN_BF16 ? (const void*)render_loss_multi_kernel<__nv_bfloat16>
                                           : (const void*)render_loss_multi_kernel<__half>, smem) != LHN_OK)
    return LHN_EINVAL;
  return launch_loss_multi<true>(a, n_planes, plane_elems, dtype, smem, workspace, sums, per_scale_loss, loss, stream);
}
