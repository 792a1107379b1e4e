// Backward of the heatmap / SimDR losses (SURVEY §8f rank 1): d loss / d output as one streaming pass
// (128-bit loads of the output [and target], 128-bit stores of the gradient), so the drop-in losses can
// sit inside train_one_epoch (train/topdown_trainer.py:68-87) behind torch.autograd.Function.
//
// Every loss on the path is a weighted sum of squares (or SmoothL1) whose per-element coefficient is
// known from the forward's f64 sums (N_pos, numel), so the gradient is
//     grad[p, e] = gout * scale * coef(p, e) * (output[p, e] - target[p, e])
// with coef = 2 w f(e) for DistanceLoss (f = 1/numel, or the 0.1/(N_pos+1) | 1/(N_neg+1) balance factors,
// loss/heatmapLoss.py:249-262) and w^2 / numel for JointsDistanceLoss (heatmapLoss.py:195-225).
#include <math_constants.h>

#include "lhn_common.cuh"

namespace lhn {
int num_sms();

// ---- explicit target ----------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) loss_backward_kernel(const T* __restrict__ out, const T* __restrict__ tgt,
                                                            const float* __restrict__ weight, int64_t n_planes,
                                                            int64_t HW, int loss_mode, float pos_value,
                                                            const double* __restrict__ sums, int sum_reduction,
                                                            float scale, const float* __restrict__ grad_out,
                                                            T* __restrict__ grad) {
  float cpos, cneg;
  loss_coefs(sums, loss_mode, sum_reduction, scale, grad_out, cpos, cneg);
  const bool bal = loss_mode == LHN_LOSS_DISTANCE_BALANCE;
  const bool vec = (HW & 3) == 0 &&
                   ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(tgt) |
                     reinterpret_cast<uintptr_t>(grad)) % (4 * sizeof(T)) == 0);
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
  if (vec) {
    const int64_t QP = HW >> 2, nq = n_planes * QP;
    for (int64_t q = tid; q < nq; q += nthr) {
      const int64_t p = q / QP;
      float w = weight[p];
      if (loss_mode == LHN_LOSS_JOINTS_MSE) w *= w;
      const float4 a = ldg_stream4<T>(out + 4 * q), g = ldg_stream4<T>(tgt + 4 * q);
      const float wp = w * cpos, wn = w * cneg;
      float4 r;
      r.x = ((bal && g.x > pos_value) ? wp : wn) * (a.x - g.x);
      r.y = ((bal && g.y > pos_value) ? wp : wn) * (a.y - g.y);
      r.z = ((bal && g.z > pos_value) ? wp : wn) * (a.z - g.z);
      r.w = ((bal && g.w > pos_value) ? wp : wn) * (a.w - g.w);
      Store4<T>::st(grad + 4 * q, r);
    }
  } else {
    const int64_t n = n_planes * HW;
    for (int64_t e = tid; e < n; e += nthr) {
      const int64_t p = e / HW;
      float w = weight[p];
      if (loss_mode == LHN_LOSS_JOINTS_MSE) w *= w;
      const float a = Elem<T>::to_f32(out[e]), g = Elem<T>::to_f32(tgt[e]);
      grad[e] = Store4<T>::from(((bal && g > pos_value) ? w * cpos : w * cneg) * (a - g));
    }
  }
}

// ---- target rendered in-kernel from the joints (generateTarget.py:100-154), one CTA per plane ----------
struct RenderBwdArgs {
  const void* hm; void* grad;
  int64_t stride_b, stride_c;
  const float* joints; int joints_stride;
  const float* vis; int vis_stride;
  int64_t n_planes;
  int S, K, H, W, unbiased, loss_mode, sum_reduction;
  double feat_x, feat_y;
  float sigma[LHN_MAX_STACKS];
  float pos_value, scale;
  const double* sums; const float* grad_out;
};

// One plane of the rendered-target gradient, strided over threads t0, t0 + nt, ...: the per-element arithmetic that
// lhn_render_loss_backward and lhn_render_loss_backward_multi share, so the two write the same bits.
template <typename T>
__device__ __forceinline__ void render_grad_plane(const T* src, T* dst, const float* ex, const float* ey, int W, int H,
                                                  float wp, float wn, bool bal, float pos_value, int t0, int nt) {
  const bool vec = (W & 3) == 0 && (reinterpret_cast<uintptr_t>(src) % (4 * sizeof(T)) == 0) &&
                   (reinterpret_cast<uintptr_t>(dst) % (4 * sizeof(T)) == 0);
  if (vec) {
    const int QR = W >> 2, nq = (H * W) >> 2;
    for (int q = t0; q < nq; q += nt) {
      const int row = q / QR, cq = q - row * QR;
      const float4 gx = *reinterpret_cast<const float4*>(ex + 4 * cq);
      const float gy = ey[row];
      const float4 o = ldg_stream4<T>(src + 4 * q);
      const float g0 = gx.x * gy, g1 = gx.y * gy, g2 = gx.z * gy, g3 = gx.w * gy;
      float4 r;
      r.x = ((bal && g0 > pos_value) ? wp : wn) * fmaf(-gx.x, gy, o.x);
      r.y = ((bal && g1 > pos_value) ? wp : wn) * fmaf(-gx.y, gy, o.y);
      r.z = ((bal && g2 > pos_value) ? wp : wn) * fmaf(-gx.z, gy, o.z);
      r.w = ((bal && g3 > pos_value) ? wp : wn) * fmaf(-gx.w, gy, o.w);
      Store4<T>::st(dst + 4 * q, r);
    }
  } else {
    for (int e = t0; e < H * W; e += nt) {
      const int y = e / W, x = e - y * W;
      const float g = ex[x] * ey[y];
      dst[e] = Store4<T>::from(((bal && g > pos_value) ? wp : wn) * fmaf(-ex[x], ey[y], Elem<T>::to_f32(src[e])));
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(128) render_loss_backward_kernel(const __grid_constant__ RenderBwdArgs a) {
  extern __shared__ float tab[];   // ex[W], ey[H]
  const int W = a.W, H = a.H;
  float* ex = tab; float* ey = tab + W;
  const int64_t p = blockIdx.x;
  const int C = a.S * a.K;
  const int64_t b = p / C;
  const int c = (int)(p - b * C);
  const int s = c / a.K, k = c - s * a.K;
  const float* jp = a.joints + (b * a.K + k) * (int64_t)a.joints_stride;
  const double sig = (double)a.sigma[s];
  const RenderGeom g = render_geom(jp[0], jp[1], a.vis[(b * a.K + k) * (int64_t)a.vis_stride], sig, a.unbiased,
                                   a.feat_x, a.feat_y, 0, 0.0, 0.0, W, H);
  float w = g.w;
  const double inv2s2 = 1.0 / (2.0 * sig * sig);
  for (int i = threadIdx.x; i < W + H; i += blockDim.x) tab[i] = table_entry(g, i, W, a.unbiased, inv2s2);
  float cpos, cneg;
  loss_coefs(a.sums, a.loss_mode, a.sum_reduction, a.scale, a.grad_out, cpos, cneg);
  if (a.loss_mode == LHN_LOSS_JOINTS_MSE) w *= w;
  __syncthreads();
  const T* src = reinterpret_cast<const T*>(a.hm) + b * a.stride_b + (int64_t)c * a.stride_c;
  T* dst = reinterpret_cast<T*>(a.grad) + p * (int64_t)H * W;
  render_grad_plane<T>(src, dst, ex, ey, W, H, w * cpos, w * cneg, a.loss_mode == LHN_LOSS_DISTANCE_BALANCE,
                       a.pos_value, threadIdx.x, blockDim.x);
}

// ---- every scale of SRHandNetLoss in one launch (loss/loss.py:59-66): one WARP per plane ----------------
// Scale i's planes are warps [i * B * K, (i + 1) * B * K) of the grid.  A warp renders its plane's ex[W], ey[H]
// into warp-private shared memory and writes the gradient with render_grad_plane; the coefficient comes from the
// scale's own row of the forward's sums and its loss weight.  A 16 x 16 plane is 64 quads, two per lane: a
// 128-thread CTA per plane would leave half its threads without work.
constexpr int kBwdMultiWarps = 8;

struct RenderBwdScale {
  const void* hm; void* grad;
  int64_t stride_b, stride_c;
  double feat_x, feat_y;
  float sigma, scale;
  int H, W, sums_row;
};

struct RenderBwdMultiArgs {
  RenderBwdScale s[LHN_LOSS_MAX_TENSORS];
  int n, K;
  int64_t BK;
  const float* joints; int joints_stride;
  const float* vis; int vis_stride;
  int unbiased, loss_mode, sum_reduction, tab_stride;
  float pos_value;
  const double* sums; const float* grad_out;
  const float* used_in; int* recomputed;      // COND only: the upstream value the one-pass forward assumed
};

// COND: the backward of lhn_render_loss_grad_multi — nothing to do when grad_out is bitwise the value the forward's
// gradients assumed, else exactly the unconditional kernel's work (COND = false compiles to the code it had before)
template <typename T, bool COND>
__global__ void __launch_bounds__(kBwdMultiWarps * 32) render_loss_backward_multi_kernel(
    const __grid_constant__ RenderBwdMultiArgs a) {
  if constexpr (COND) {
    const float go = a.grad_out ? a.grad_out[0] : 1.f;
    const bool same = __float_as_uint(go) == __float_as_uint(a.used_in[0]);
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.recomputed) a.recomputed[0] = same ? 0 : 1;
    if (same) return;
  }
  extern __shared__ float4 btab4[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t gw = (int64_t)blockIdx.x * kBwdMultiWarps + warp;
  if (gw >= a.n * a.BK) return;
  const int i = (int)(gw / a.BK);
  const int64_t p = gw - i * a.BK;
  const RenderBwdScale& s = a.s[i];
  const int W = s.W, H = s.H;
  float* ex = reinterpret_cast<float*>(btab4) + warp * a.tab_stride;
  float* ey = ex + W;
  const int64_t b = p / a.K;
  const int k = (int)(p - b * a.K);
  const float* jp = a.joints + p * (int64_t)a.joints_stride;
  const double sig = (double)s.sigma;
  const RenderGeom g = render_geom(jp[0], jp[1], a.vis[p * (int64_t)a.vis_stride], sig, a.unbiased, s.feat_x,
                                   s.feat_y, 0, 0.0, 0.0, W, H);
  float w = g.w;
  const double inv2s2 = 1.0 / (2.0 * sig * sig);
  for (int e = lane; e < W + H; e += 32) ex[e] = table_entry(g, e, W, a.unbiased, inv2s2);
  float cpos, cneg;
  loss_coefs(a.sums + 4 * s.sums_row, a.loss_mode, a.sum_reduction, s.scale, a.grad_out, cpos, cneg);
  if (a.loss_mode == LHN_LOSS_JOINTS_MSE) w *= w;
  __syncwarp();
  const T* src = reinterpret_cast<const T*>(s.hm) + b * s.stride_b + (int64_t)k * s.stride_c;
  T* dst = reinterpret_cast<T*>(s.grad) + p * (int64_t)H * W;
  render_grad_plane<T>(src, dst, ex, ey, W, H, w * cpos, w * cneg, a.loss_mode == LHN_LOSS_DISTANCE_BALANCE,
                       a.pos_value, lane, 32);
}

// ---- KLDiscretLoss backward (centernet_simdr_loss.py:27-39): SmoothL1'(d) * mean_b(w)[j] / (K B L) ------
// One warp per (b, k) row of the x- or the y-vector (rows [0, BK) are x, [BK, 2 BK) are y): 128-bit loads of output and
// target, one 128-bit store of the gradient, the joint's coefficient computed once per row — ONE launch for both
// vectors (round 1: a scalar element loop with a 64-bit division per element, two launches: 22 % of the HBM peak).
template <typename T>
__global__ void __launch_bounds__(256) simdr_backward_kernel(const T* __restrict__ ox, const T* __restrict__ oy,
                                                             const T* __restrict__ tx, const T* __restrict__ ty,
                                                             const float* __restrict__ mean_w, int64_t BK, int K,
                                                             int Lx, int Ly, int64_t B, float scale,
                                                             const float* __restrict__ grad_out, T* __restrict__ gx,
                                                             T* __restrict__ gy) {
  const float g = scale * (grad_out ? grad_out[0] : 1.f);
  const int lane = threadIdx.x & 31;
  const int64_t wg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = wg; row < 2 * BK; row += nw) {
    const bool isx = row < BK;
    const int64_t bk = isx ? row : row - BK;
    const int Lv = isx ? Lx : Ly;
    const T* o = (isx ? ox : oy) + bk * Lv;
    const T* t = (isx ? tx : ty) + bk * Lv;
    T* gr = (isx ? gx : gy) + bk * Lv;
    const int j = (int)(bk % K);
    const float c = (float)((1.0 / ((double)K * (double)B * (double)Lv)) * (double)__ldg(mean_w + j)) * g;
    auto grad1 = [&](float d) {
      const float sl = fabsf(d) < 1.f ? d : (d > 0.f ? 1.f : -1.f);   // SmoothL1 beta = 1; NaN propagates through d
      return (d != d ? d : sl) * c;
    };
    const bool vec = (Lv & 3) == 0 && ((reinterpret_cast<uintptr_t>(o) | reinterpret_cast<uintptr_t>(t) |
                                        reinterpret_cast<uintptr_t>(gr)) % (4 * sizeof(T)) == 0);
    if (vec) {
      const int nq = Lv >> 2;
#pragma unroll 4
      for (int q = lane; q < nq; q += 32) {
        const float4 a = ldg_stream4<T>(o + 4 * q), b = ldg_stream4<T>(t + 4 * q);
        Store4<T>::st(gr + 4 * q, make_float4(grad1(a.x - b.x), grad1(a.y - b.y), grad1(a.z - b.z), grad1(a.w - b.w)));
      }
    } else {
      for (int e = lane; e < Lv; e += 32) gr[e] = Store4<T>::from(grad1(Elem<T>::to_f32(o[e]) - Elem<T>::to_f32(t[e])));
    }
  }
}

// mean_b w[b, j]: one warp per joint, f64 partial sums (more accurate than any f32 order; tensor.mean() agrees to 1e-7)
__global__ void __launch_bounds__(256) simdr_mean_weight_kernel(const float* __restrict__ weight, int64_t B, int K,
                                                                float* __restrict__ mean_w) {
  const int lane = threadIdx.x & 31;
  const int j = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (j >= K) return;
  double s = 0.0;
#pragma unroll 8
  for (int64_t b = lane; b < B; b += 32) s += (double)__ldg(weight + b * K + j);
  s = warp_sum(s);
  if (lane == 0) mean_w[j] = (float)(s / (double)B);
}

}  // namespace lhn

using namespace lhn;

extern "C" int lhn_loss_backward(const void* output, const void* target, const float* weight, int dtype,
                                 int64_t n_planes, int64_t plane_elems, int loss_mode, float pos_value,
                                 const double* sums, int sum_reduction, float scale, const float* grad_out,
                                 void* grad, lhn_stream_t stream) {
  if (!output || !target || !weight || !sums || !grad || n_planes < 0 || plane_elems <= 0 || loss_mode < 1 ||
      loss_mode > 3)
    return LHN_EINVAL;
  if (n_planes == 0) return LHN_OK;
  const int threads = 256;
  const int64_t work = (n_planes * plane_elems + 3) / 4;
  int64_t blocks = (work + threads - 1) / threads;
  const int64_t cap = (int64_t)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  cudaStream_t st = (cudaStream_t)stream;
#define LHN_BWD(T)                                                                                         \
  loss_backward_kernel<T><<<(unsigned)blocks, threads, 0, st>>>((const T*)output, (const T*)target, weight, \
      n_planes, plane_elems, loss_mode, pos_value, sums, sum_reduction, scale, grad_out, (T*)grad)
  switch (dtype) {
    case LHN_F32: LHN_BWD(float); break;
    case LHN_BF16: LHN_BWD(__nv_bfloat16); break;
    case LHN_F16: LHN_BWD(__half); break;
    default: return LHN_EDTYPE;
  }
#undef LHN_BWD
  return check_launch();
}

extern "C" int lhn_render_loss_backward(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                        int64_t stride_b, int64_t stride_c, const lhn_render_params* rp,
                                        const float* joints, int joints_stride, const float* vis,
                                        int vis_stride, const double* sums, int sum_reduction, float scale,
                                        const float* grad_out, void* grad, lhn_stream_t stream) {
  if (!hm || !rp || !joints || !vis || !sums || !grad || B < 0 || K <= 0 || H <= 0 || W <= 0 ||
      joints_stride < 2 || vis_stride < 1 || rp->image_w <= 0 || rp->image_h <= 0 || rp->loss_mode < 1 ||
      rp->loss_mode > 3)
    return LHN_EINVAL;
  const int S = rp->num_stacks > 0 ? rp->num_stacks : 1;
  if (S > LHN_MAX_STACKS) return LHN_EINVAL;
  RenderBwdArgs a{};
  a.hm = hm; a.grad = grad; a.stride_b = stride_b; a.stride_c = stride_c;
  a.joints = joints; a.joints_stride = joints_stride; a.vis = vis; a.vis_stride = vis_stride;
  a.S = S; a.K = K; a.H = H; a.W = W; a.unbiased = rp->unbiased; a.loss_mode = rp->loss_mode;
  a.sum_reduction = sum_reduction; a.n_planes = B * S * K;
  if (rp->unbiased < 0 || rp->unbiased > 2) return LHN_EINVAL;
  if (rp->unbiased == 2) {
    if (W < 2 || H < 2) return LHN_EINVAL;
    a.feat_x = ((double)rp->image_w - 1.0) / (W - 1.0); a.feat_y = ((double)rp->image_h - 1.0) / (H - 1.0);
  } else {
    a.feat_x = (double)rp->image_w / W; a.feat_y = (double)rp->image_h / H;
  }
  for (int i = 0; i < S; ++i) { if (!(rp->sigma[i] > 0.f)) return LHN_EINVAL; a.sigma[i] = rp->sigma[i]; }
  a.pos_value = rp->pos_value; a.scale = scale; a.sums = sums; a.grad_out = grad_out;
  if (a.n_planes == 0) return LHN_OK;
  if (a.n_planes > 0x7fffffffLL) return LHN_EINVAL;
  const size_t smem = (size_t)(W + H) * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
  switch (dtype) {
    case LHN_F32: render_loss_backward_kernel<float><<<(unsigned)a.n_planes, 128, smem, st>>>(a); break;
    case LHN_BF16: render_loss_backward_kernel<__nv_bfloat16><<<(unsigned)a.n_planes, 128, smem, st>>>(a); break;
    case LHN_F16: render_loss_backward_kernel<__half><<<(unsigned)a.n_planes, 128, smem, st>>>(a); break;
    default: return LHN_EDTYPE;
  }
  return check_launch();
}

// lhn_render_loss_backward_multi and, with used_scale != NULL, its conditional form
static int backward_multi(int n_scales, const lhn_loss_scale* scales, int dtype, int64_t B, int K,
                          const lhn_render_params* rp, const float* joints, int joints_stride, const float* vis,
                          int vis_stride, const double* sums, int sum_reduction, const float* grad_out,
                          const float* used_scale, int32_t* recomputed, lhn_stream_t stream) {
  if (n_scales < 1 || n_scales > LHN_LOSS_MAX_TENSORS || !scales || !rp || !joints || !vis || !sums || B <= 0 ||
      K <= 0 || joints_stride < 2 || vis_stride < 1)
    return LHN_EINVAL;
  if (dtype != LHN_F32 && dtype != LHN_BF16 && dtype != LHN_F16) return LHN_EDTYPE;
  RenderBwdMultiArgs a{};
  int tab = 0;
  for (int i = 0; i < n_scales; ++i) {
    const lhn_loss_scale& sc = scales[i];
    double fx, fy;
    if (!sc.output || scale_geometry(rp, sc.H, sc.W, sc.sigma, fx, fy) != LHN_OK) return LHN_EINVAL;
    if (!sc.grad) continue;                               // this scale's gradient is not wanted
    RenderBwdScale& s = a.s[a.n++];
    s.hm = sc.output; s.grad = sc.grad; s.stride_b = sc.stride_b; s.stride_c = sc.stride_c;
    s.feat_x = fx; s.feat_y = fy; s.sigma = sc.sigma; s.scale = sc.loss_weight; s.H = sc.H; s.W = sc.W;
    s.sums_row = i;
    if (sc.H + sc.W > tab) tab = sc.H + sc.W;
  }
  if (a.n == 0) return LHN_OK;
  a.K = K; a.BK = B * K;
  a.joints = joints; a.joints_stride = joints_stride; a.vis = vis; a.vis_stride = vis_stride;
  a.unbiased = rp->unbiased; a.loss_mode = rp->loss_mode; a.sum_reduction = sum_reduction;
  a.tab_stride = (tab + 3) & ~3; a.pos_value = rp->pos_value; a.sums = sums; a.grad_out = grad_out;
  a.used_in = used_scale; a.recomputed = recomputed;
  const int64_t blocks = (a.n * a.BK + kBwdMultiWarps - 1) / kBwdMultiWarps;
  if (blocks > 0x7fffffffLL) return LHN_EINVAL;
  const size_t smem = (size_t)kBwdMultiWarps * a.tab_stride * sizeof(float);
  const bool cond = used_scale != nullptr;
  void (*fn)(RenderBwdMultiArgs) =
      dtype == LHN_F32 ? (cond ? render_loss_backward_multi_kernel<float, true> : render_loss_backward_multi_kernel<float, false>)
    : dtype == LHN_BF16 ? (cond ? render_loss_backward_multi_kernel<__nv_bfloat16, true>
                                : render_loss_backward_multi_kernel<__nv_bfloat16, false>)
                        : (cond ? render_loss_backward_multi_kernel<__half, true> : render_loss_backward_multi_kernel<__half, false>);
  if (set_dynamic_smem((const void*)fn, smem) != LHN_OK) return LHN_EINVAL;
  fn<<<(unsigned)blocks, kBwdMultiWarps * 32, smem, (cudaStream_t)stream>>>(a);
  return check_launch();
}

extern "C" int lhn_render_loss_backward_multi(int n_scales, const lhn_loss_scale* scales, int dtype, int64_t B,
                                              int K, const lhn_render_params* rp, const float* joints,
                                              int joints_stride, const float* vis, int vis_stride,
                                              const double* sums, int sum_reduction, const float* grad_out,
                                              lhn_stream_t stream) {
  return backward_multi(n_scales, scales, dtype, B, K, rp, joints, joints_stride, vis, vis_stride, sums,
                        sum_reduction, grad_out, nullptr, nullptr, stream);
}

extern "C" int lhn_render_loss_backward_multi_cond(int n_scales, const lhn_loss_scale* scales, int dtype, int64_t B,
                                                   int K, const lhn_render_params* rp, const float* joints,
                                                   int joints_stride, const float* vis, int vis_stride,
                                                   const double* sums, int sum_reduction, const float* grad_out,
                                                   const float* used_scale, int32_t* recomputed,
                                                   lhn_stream_t stream) {
  if (!used_scale) return LHN_EINVAL;
  return backward_multi(n_scales, scales, dtype, B, K, rp, joints, joints_stride, vis, vis_stride, sums,
                        sum_reduction, grad_out, used_scale, recomputed, stream);
}

extern "C" int64_t lhn_simdr_backward_workspace_bytes(int K) { return K > 0 ? (int64_t)K * 4 : 0; }

extern "C" int lhn_simdr_smoothl1_backward(const void* out_x, const void* out_y, const void* tgt_x,
                                           const void* tgt_y, const float* weight, int dtype, int64_t B, int K,
                                           int Lx, int Ly, float scale, const float* grad_out, void* workspace,
                                           int64_t workspace_bytes, void* grad_x, void* grad_y,
                                           lhn_stream_t stream) {
  g_simdr_launch = {};
  if (!out_x || !out_y || !tgt_x || !tgt_y || !weight || !workspace || !grad_x || !grad_y || B <= 0 || K <= 0 ||
      Lx <= 0 || Ly <= 0)
    return LHN_EINVAL;
  if (workspace_bytes < (int64_t)K * 4) return LHN_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  float* mean_w = static_cast<float*>(workspace);
  simdr_mean_weight_kernel<<<(K * 32 + 255) / 256, 256, 0, st>>>(weight, B, K, mean_w);
  const int threads = 256;
  const int64_t rows = 2 * B * K;
  int64_t nb = (rows * 32 + threads - 1) / threads;
  const int64_t cap = (int64_t)num_sms() * 8;
  if (nb > cap) nb = cap;
#define LHN_SB(T)                                                                                               \
  simdr_backward_kernel<T><<<(unsigned)nb, threads, 0, st>>>((const T*)out_x, (const T*)out_y, (const T*)tgt_x, \
      (const T*)tgt_y, mean_w, B * K, K, Lx, Ly, B, scale, grad_out, (T*)grad_x, (T*)grad_y)
  switch (dtype) {
    case LHN_F32: LHN_SB(float); break;
    case LHN_BF16: LHN_SB(__nv_bfloat16); break;
    case LHN_F16: LHN_SB(__half); break;
    default: return LHN_EDTYPE;
  }
#undef LHN_SB
  const int rc = check_launch();
  if (rc == LHN_OK) {
    // the kernel's per-row `vec` test: with L % 4 == 0 every row of an aligned base is aligned
    const uintptr_t al = dtype == LHN_F32 ? 16 : 8;
    const bool vx = (Lx & 3) == 0 && (((uintptr_t)out_x | (uintptr_t)tgt_x | (uintptr_t)grad_x) % al) == 0;
    const bool vy = (Ly & 3) == 0 && (((uintptr_t)out_y | (uintptr_t)tgt_y | (uintptr_t)grad_y) % al) == 0;
    simdr_record(4, 1, dtype, threads / 32, 0, nb, vx, vy, 0);
  }
  return rc;
}
