// Un-fused drop-ins: masked MSE against an explicit target tensor, the deterministic loss
// reduction/finalisation, batched Gaussian target rendering (2-D and SimDR 1-D) and flip_back.
// All are single-pass, 128-bit vectorised streaming kernels; grids are sized as multiples of the
// SM count with grid-stride loops.
#include <math_constants.h>

#include <cooperative_groups.h>

#include "lhn_common.cuh"

namespace lhn {

// SM count of the CURRENT device, cached per device (a process may drive several GPUs)
static int g_num_sms[64] = {0};
int num_sms() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  if (g_num_sms[dev] == 0) {
    int n = 148;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    g_num_sms[dev] = n > 0 ? n : 148;
  }
  return g_num_sms[dev];
}

// ---- loss partials against an explicit target (heatmapLoss.py:242-265, :195-225) -------------
// one warp per plane: 2 streams of 128-bit loads, no shared memory needed
template <typename T>
__global__ void __launch_bounds__(256) loss_partials_kernel(const T* __restrict__ out,
                                                            const T* __restrict__ tgt,
                                                            const float* __restrict__ weight,
                                                            int64_t n_planes, int64_t HW,
                                                            int loss_mode, float pos_value,
                                                            double* __restrict__ partials) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const bool vec = (HW & 3) == 0 &&
                   ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(tgt)) % (4 * sizeof(T)) == 0);
  for (int64_t p = warp_global; p < n_planes; p += nwarps) {
    const T* o = out + p * HW;
    const T* t = tgt + p * HW;
    float sp0 = 0.f, sp1 = 0.f, sn0 = 0.f, sn1 = 0.f;
    int npos = 0;
    if (vec) {
      const int64_t nq = HW >> 2;
#pragma unroll 4
      for (int64_t q = lane; q < nq; q += 32) {
        const float4 a = ldg_stream4<T>(o + 4 * q);
        const float4 g = ldg_stream4<T>(t + 4 * q);
        const float d0 = a.x - g.x, d1 = a.y - g.y, d2 = a.z - g.z, d3 = a.w - g.w;
        const float l0 = d0 * d0, l1 = d1 * d1, l2 = d2 * d2, l3 = d3 * d3;
        const bool p0 = g.x > pos_value, p1 = g.y > pos_value, p2 = g.z > pos_value, p3 = g.w > pos_value;
        sp0 += p0 ? l0 : 0.f; sn0 += p0 ? 0.f : l0;
        sp1 += p1 ? l1 : 0.f; sn1 += p1 ? 0.f : l1;
        sp0 += p2 ? l2 : 0.f; sn0 += p2 ? 0.f : l2;
        sp1 += p3 ? l3 : 0.f; sn1 += p3 ? 0.f : l3;
        npos += (int)p0 + (int)p1 + (int)p2 + (int)p3;
      }
    } else {
      for (int64_t e = lane; e < HW; e += 32) {
        const float a = Elem<T>::to_f32(o[e]), g = Elem<T>::to_f32(t[e]);
        const float d = a - g, l = d * d;
        const bool pp = g > pos_value;
        sp0 += pp ? l : 0.f; sn0 += pp ? 0.f : l; npos += (int)pp;
      }
    }
    double sp = warp_sum((double)sp0 + (double)sp1);
    double sn = warp_sum((double)sn0 + (double)sn1);
    npos = __reduce_add_sync(0xffffffffu, npos);
    if (lane == 0) {
      const float w = weight[p];
      const double wp = (loss_mode == LHN_LOSS_JOINTS_MSE) ? (double)(w * w) : (double)w;
      double* dst = partials + 4 * p;
      if (loss_mode == LHN_LOSS_DISTANCE_BALANCE) { dst[0] = sp * wp; dst[1] = sn * wp; dst[2] = (double)npos; }
      else { dst[0] = 0.0; dst[1] = (sp + sn) * wp; dst[2] = 0.0; }
      dst[3] = (double)HW;
    }
  }
}

// ---- deterministic reduction: one thread-block cluster, fixed order, f64 --------------------------
// 8 CTAs of one cluster each reduce a contiguous slice of the per-plane partials; CTA 0 then reads the
// 8 slice sums through distributed shared memory in rank order.  One launch, no workspace, and the
// summation order is a pure function of (n_planes) — bitwise reproducible run to run.
constexpr int kReduceCtas = 8;
constexpr int kReduceThreads = 512;

__global__ void __cluster_dims__(kReduceCtas, 1, 1) __launch_bounds__(kReduceThreads)
loss_reduce_kernel(const double* __restrict__ partials, int64_t n_planes, double* __restrict__ sums,
                   int accumulate) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  __shared__ double red[4][kReduceThreads / 32];
  __shared__ double block_sum[4];
  const unsigned rank = cluster.block_rank();
  const int64_t per = (n_planes + kReduceCtas - 1) / kReduceCtas;
  const int64_t lo = rank * per, hi = (lo + per < n_planes) ? lo + per : n_planes;
  double acc[4] = {0, 0, 0, 0};
  for (int64_t p = lo + threadIdx.x; p < hi; p += kReduceThreads) {
    const double4 v = *reinterpret_cast<const double4*>(partials + 4 * p);
    acc[0] += v.x; acc[1] += v.y; acc[2] += v.z; acc[3] += v.w;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const double v = warp_sum(acc[i]);
    if (lane == 0) red[i][warp] = v;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      double v = lane < (kReduceThreads / 32) ? red[i][lane] : 0.0;
      v = warp_sum(v);
      if (lane == 0) block_sum[i] = v;
    }
  }
  cluster.sync();
  if (rank == 0 && threadIdx.x < 4) {
    double t = 0.0;
    for (unsigned r = 0; r < kReduceCtas; ++r) t += cluster.map_shared_rank(block_sum, r)[threadIdx.x];
    sums[threadIdx.x] = accumulate ? sums[threadIdx.x] + t : t;
  }
  cluster.sync();   // keep every CTA's shared memory alive until rank 0 has read it
}

__global__ void loss_finalize_kernel(const double* __restrict__ sums, int loss_mode, int sum_reduction,
                                     float scale, float* __restrict__ loss, int accumulate) {
  const double sp = sums[0], sn = sums[1], npos = sums[2], numel = sums[3];
  double v;
  if (loss_mode == LHN_LOSS_DISTANCE_BALANCE) v = 0.1 * sp / (npos + 1.0) + sn / (numel - npos + 1.0);
  else if (loss_mode == LHN_LOSS_JOINTS_MSE) v = 0.5 * (sp + sn) / numel;
  else v = (sp + sn) / numel;
  if (sum_reduction) v *= numel;
  const float r = (float)(v * (double)scale);
  loss[0] = accumulate ? loss[0] + r : r;
}

// ---- batched target rendering (generateTarget.py:100-154) --------------------------------------
// One CTA per plane: the separable factors are evaluated in f64 (as NumPy>=2 does for the
// unbiased branch), the plane is written with 128-bit stores.
struct RenderArgs {
  const float* joints; int joints_stride;
  const float* vis; int vis_stride;
  int64_t n_planes;
  int S, K, H, W;
  int unbiased;
  double feat_x, feat_y;
  float sigma[LHN_MAX_STACKS];
  float* target; float* target_weight;
};

__global__ void __launch_bounds__(128) render_targets_kernel(const __grid_constant__ RenderArgs a) {
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
  const float w = g.w;
  const double inv2s2 = 1.0 / (2.0 * sig * sig);
  for (int i = threadIdx.x; i < W + H; i += blockDim.x) tab[i] = table_entry(g, i, W, a.unbiased, inv2s2);
  __syncthreads();
  float* dst = a.target + p * (int64_t)H * W;
  if ((W & 3) == 0) {
    const int QR = W >> 2, nq = (H * W) >> 2;
    for (int q = threadIdx.x; q < nq; q += blockDim.x) {
      const int row = q / QR, cq = q - row * QR;
      const float4 gx = *reinterpret_cast<const float4*>(ex + 4 * cq);
      const float gy = ey[row];
      *reinterpret_cast<float4*>(dst + 4 * q) = make_float4(gx.x * gy, gx.y * gy, gx.z * gy, gx.w * gy);
    }
  } else {
    for (int e = threadIdx.x; e < H * W; e += blockDim.x) dst[e] = ex[e % W] * ey[e / W];
  }
  if (threadIdx.x == 0) a.target_weight[p] = w;
}

// ---- SimDR target (generate_simder.py:9-31): f32 arithmetic throughout ---------------------------
// One (sample, joint) per CTA; a thread writes four neighbouring positions with one 16-byte store (VEC) — the vectors are
// the only traffic.  exp runs in f64 on the f32 argument (rounded once, = the correctly rounded f32 exp numpy's result is
// compared against) but only where the result is not exactly 0: exp(a) < 2^-150 — half the smallest f32 denormal — for
// a < -104, so everything farther than ~14.4 sigma from the joint is a plain zero store (9 positions in 10 at sigma 2,
// 512 bins); without the cut the kernel sat on the FP64 pipe at 21 % of the HBM peak.
__device__ __forceinline__ float simdr_bin(int pos, float mu, float den) {
  const float d = __fsub_rn((float)pos, mu);
  const float arg = __fdiv_rn(-__fmul_rn(d, d), den);
  if (arg < -104.f) return 0.f;
  return (float)exp((double)arg);                                    // f32 argument, exp rounded once
}

// VEC: one (sample, joint) per WARP and a grid-stride loop over them; the next pair's joint is loaded while this one is
// written.  The warp first evaluates the window of bins that can be non-zero (|pos - mu| <= sqrt(104 * 2 sigma^2) + 1,
// 64 bins at sigma 2) ONE bin per lane into shared memory, then streams the vectors out as 16-byte stores that pick
// from the window or write the fill value.  Evaluating inside the store loop had each lane walk four divergent f64
// exps in turn — 8x the FP64 issue slots, and FP64 (64 lanes per SM) was what the kernel waited on.
constexpr int kSimdrWindowMax = 256;

template <bool VEC>
__global__ void __launch_bounds__(256) render_simdr_kernel(const float* __restrict__ joints, int js,
                                                           const float* __restrict__ vis, int vs,
                                                           int64_t n_bk, int Lx, int Ly, float kf,
                                                           float den, float* __restrict__ sx,
                                                           float* __restrict__ sy) {
  if (VEC) {
    __shared__ float win_all[8][kSimdrWindowMax];
    const int lane = threadIdx.x & 31;
    float* win = win_all[threadIdx.x >> 5];
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    int64_t bk = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (bk >= n_bk) return;
    const float reach = sqrtf(104.f * den) + 1.f;
    const int nw = 2 * (int)ceilf(reach) + 2;                       // host: nw <= kSimdrWindowMax on this path
    float jx = joints[bk * js], jy = joints[bk * js + 1], vv = vis[bk * vs];
    for (; bk < n_bk; bk += nwarps) {
      const bool on = vv > 0.f;
      const float mus[2] = {__fmul_rn(jx, kf), __fmul_rn(jy, kf)};
      const int64_t nb = bk + nwarps;
      if (nb < n_bk) { jx = joints[nb * js]; jy = joints[nb * js + 1]; vv = vis[nb * vs]; }
#pragma unroll
      for (int ax = 0; ax < 2; ++ax) {
        const float mu = mus[ax];
        const int L = ax ? Ly : Lx;
        float* dst = ax ? sy + bk * Ly : sx + bk * Lx;
        // a NaN joint makes every bin NaN (exp(NaN)); an infinite or far-away one makes every bin 0
        const float fill = (on && mu != mu) ? mu : 0.f;
        const bool near = on && fabsf(mu) < 1e9f;
        const int p0 = near ? (int)floorf(mu - reach) : 0;
        const unsigned span = near ? (unsigned)nw : 0u;
        if (near)
          for (int w = lane; w < nw; w += 32) {
            const int pos = p0 + w;
            if (pos >= 0 && pos < L) win[w] = simdr_bin(pos, mu, den);
          }
        __syncwarp();
        for (int q = lane; q < (L >> 2); q += 32) {
          const int pos = 4 * q;
          const int d = pos - p0;
          float4 v = make_float4(fill, fill, fill, fill);
          if (d > -4 && d < (int)span) {                 // 7 quads in 8 lie wholly outside the window: just the store
            const unsigned w = (unsigned)d;
            v.x = w < span ? win[w] : fill;
            v.y = w + 1u < span ? win[w + 1u] : fill;
            v.z = w + 2u < span ? win[w + 2u] : fill;
            v.w = w + 3u < span ? win[w + 3u] : fill;
          }
          __stcs(reinterpret_cast<float4*>(dst + pos), v);
        }
        __syncwarp();
      }
    }
  } else {
    const int64_t bk = blockIdx.x;
    if (bk >= n_bk) return;
    const bool on = vis[bk * vs] > 0.f;
    const float mux = __fmul_rn(joints[bk * js], kf), muy = __fmul_rn(joints[bk * js + 1], kf);
    float* dx = sx + bk * Lx; float* dy = sy + bk * Ly;
    for (int i = threadIdx.x; i < Lx + Ly; i += blockDim.x) {
      const bool isx = i < Lx;
      const int pos = isx ? i : i - Lx;
      const float v = on ? simdr_bin(pos, isx ? mux : muy, den) : 0.f;
      if (isx) dx[pos] = v; else dy[pos] = v;
    }
  }
}

// ---- flip_back (transforms.py:78-92) --------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) flip_back_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                        int64_t n_planes, int K, int H, int W,
                                                        const int32_t* __restrict__ flip_index) {
  const int64_t total = n_planes * H * W;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (int64_t)gridDim.x * blockDim.x) {
    const int x = (int)(e % W);
    const int64_t r = e / W;
    const int y = (int)(r % H);
    const int64_t p = r / H;
    const int k = (int)(p % K);
    const int64_t b = p / K;
    const int ks = flip_index ? flip_index[k] : k;
    out[e] = in[((b * K + ks) * H + y) * (int64_t)W + (W - 1 - x)];
  }
}

}  // namespace lhn

using namespace lhn;

extern "C" int lhn_loss_partials(const void* output, const void* target, const float* weight,
                                 int dtype, int64_t n_planes, int64_t plane_elems, int loss_mode,
                                 float pos_value, double* partials, lhn_stream_t stream) {
  if (!output || !target || !weight || !partials || n_planes < 0 || plane_elems <= 0 ||
      loss_mode < 1 || loss_mode > 3)
    return LHN_EINVAL;
  if (n_planes == 0) return LHN_OK;
  const int threads = 256;
  int64_t blocks_needed = (n_planes * 32 + threads - 1) / threads;
  int64_t cap = (int64_t)num_sms() * 8;
  int blocks = (int)(blocks_needed < cap ? blocks_needed : cap);
  cudaStream_t st = (cudaStream_t)stream;
  switch (dtype) {
    case LHN_F32:
      loss_partials_kernel<float><<<blocks, threads, 0, st>>>((const float*)output, (const float*)target,
          weight, n_planes, plane_elems, loss_mode, pos_value, partials);
      break;
    case LHN_BF16:
      loss_partials_kernel<__nv_bfloat16><<<blocks, threads, 0, st>>>((const __nv_bfloat16*)output,
          (const __nv_bfloat16*)target, weight, n_planes, plane_elems, loss_mode, pos_value, partials);
      break;
    case LHN_F16:
      loss_partials_kernel<__half><<<blocks, threads, 0, st>>>((const __half*)output, (const __half*)target,
          weight, n_planes, plane_elems, loss_mode, pos_value, partials);
      break;
    default: return LHN_EDTYPE;
  }
  return check_launch();
}

extern "C" int lhn_loss_reduce(const double* partials, int64_t n_planes, double* sums, int accumulate,
                               lhn_stream_t stream) {
  if (!partials || !sums || n_planes < 0) return LHN_EINVAL;
  if ((uintptr_t)partials % 32) return LHN_EALIGN;
  loss_reduce_kernel<<<kReduceCtas, kReduceThreads, 0, (cudaStream_t)stream>>>(partials, n_planes, sums, accumulate);
  return check_launch();
}

extern "C" int lhn_loss_finalize(const double* sums, int loss_mode, int sum_reduction, float scale,
                                 float* loss, int accumulate, lhn_stream_t stream) {
  if (!sums || !loss || loss_mode < 1 || loss_mode > 3) return LHN_EINVAL;
  loss_finalize_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(sums, loss_mode, sum_reduction, scale, loss, accumulate);
  return check_launch();
}

extern "C" int lhn_render_targets(const float* joints, int joints_stride, const float* vis,
                                  int vis_stride, int64_t B, int K, int H, int W,
                                  const lhn_render_params* rp, float* target, float* target_weight,
                                  lhn_stream_t stream) {
  if (!joints || !vis || !rp || !target || !target_weight || B < 0 || K <= 0 || H <= 0 || W <= 0 ||
      joints_stride < 2 || vis_stride < 1 || rp->image_w <= 0 || rp->image_h <= 0)
    return LHN_EINVAL;
  const int S = rp->num_stacks > 0 ? rp->num_stacks : 1;
  if (S > LHN_MAX_STACKS) return LHN_EINVAL;
  if ((uintptr_t)target % 16) return LHN_EALIGN;
  RenderArgs a{};
  a.joints = joints; a.joints_stride = joints_stride; a.vis = vis; a.vis_stride = vis_stride;
  a.S = S; a.K = K; a.H = H; a.W = W; a.unbiased = rp->unbiased;
  a.n_planes = B * S * K;
  if (rp->unbiased < 0 || rp->unbiased > 2) return LHN_EINVAL;
  if (rp->unbiased == 2) {
    if (W < 2 || H < 2) return LHN_EINVAL;
    a.feat_x = ((double)rp->image_w - 1.0) / (W - 1.0); a.feat_y = ((double)rp->image_h - 1.0) / (H - 1.0);
  } else {
    a.feat_x = (double)rp->image_w / W; a.feat_y = (double)rp->image_h / H;
  }
  for (int i = 0; i < S; ++i) { if (!(rp->sigma[i] > 0.f)) return LHN_EINVAL; a.sigma[i] = rp->sigma[i]; }
  a.target = target; a.target_weight = target_weight;
  if (a.n_planes == 0) return LHN_OK;
  if (a.n_planes > 0x7fffffffLL) return LHN_EINVAL;
  size_t smem = (size_t)(W + H) * sizeof(float);
  render_targets_kernel<<<(unsigned)a.n_planes, 128, smem, (cudaStream_t)stream>>>(a);
  return check_launch();
}

// Both render entry points: `den` is the Gaussian's denominator 2 sigma^2 as an f32, formed by the caller.
static int render_simdr_den(const float* joints, int joints_stride, const float* vis, int vis_stride, int64_t B, int K,
                            int Lx, int Ly, float split_ratio, float den, float* simdr_x, float* simdr_y,
                            lhn_stream_t stream) {
  if (!joints || !vis || !simdr_x || !simdr_y || B < 0 || K <= 0 || Lx <= 0 || Ly <= 0 ||
      joints_stride < 2 || vis_stride < 1 || !(den > 0.f) || !(den <= 3.4028235e38f))
    return LHN_EINVAL;
  const int64_t n = B * K;
  if (n == 0) return LHN_OK;
  if (n > 0x7fffffffLL) return LHN_EINVAL;
  const bool vec = Lx % 4 == 0 && Ly % 4 == 0 && ((uintptr_t)simdr_x % 16) == 0 && ((uintptr_t)simdr_y % 16) == 0 &&
                   2 * (int)ceilf(sqrtf(104.f * den) + 1.f) + 2 <= kSimdrWindowMax;
  const int64_t want = (n + 7) / 8, cap = (int64_t)num_sms() * 8;
  const int64_t ctas = vec ? (want < cap ? want : cap) : n;
  if (vec) render_simdr_kernel<true><<<(unsigned)ctas, 256, 0, (cudaStream_t)stream>>>(joints, joints_stride, vis, vis_stride,
      n, Lx, Ly, split_ratio, den, simdr_x, simdr_y);
  else render_simdr_kernel<false><<<(unsigned)ctas, 256, 0, (cudaStream_t)stream>>>(joints, joints_stride, vis, vis_stride,
      n, Lx, Ly, split_ratio, den, simdr_x, simdr_y);
  const int rc = check_launch();
  if (rc == LHN_OK) simdr_record(1, vec ? 1 : 2, LHN_F32, 8, 0, ctas, vec, vec, 0);
  return rc;
}

extern "C" int lhn_render_simdr(const float* joints, int joints_stride, const float* vis,
                                int vis_stride, int64_t B, int K, int Lx, int Ly, float split_ratio,
                                float sigma, float* simdr_x, float* simdr_y, lhn_stream_t stream) {
  g_simdr_launch = {};
  if (!(sigma > 0.f)) return LHN_EINVAL;
  return render_simdr_den(joints, joints_stride, vis, vis_stride, B, K, Lx, Ly, split_ratio, 2.f * sigma * sigma,
                          simdr_x, simdr_y, stream);
}

extern "C" int lhn_render_simdr_f64sigma(const float* joints, int joints_stride, const float* vis,
                                         int vis_stride, int64_t B, int K, int Lx, int Ly, float split_ratio,
                                         double sigma, float* simdr_x, float* simdr_y, lhn_stream_t stream) {
  g_simdr_launch = {};
  if (!(sigma > 0.0)) return LHN_EINVAL;
  // the reference's denominator: the Python float 2 * sigma ** 2 (f64), rounded to f32 once when numpy divides the f32
  // array by it.  2.f * s * s on an f32 sigma differs from it by one ulp for about half of all sigma (1.3, 2.1, 2.7, ...)
  return render_simdr_den(joints, joints_stride, vis, vis_stride, B, K, Lx, Ly, split_ratio,
                          (float)(2.0 * (sigma * sigma)), simdr_x, simdr_y, stream);
}

extern "C" int lhn_flip_back(const void* in, void* out, int dtype, int64_t B, int K, int H, int W,
                             const int32_t* flip_index, lhn_stream_t stream) {
  if (!in || !out || B < 0 || K <= 0 || H <= 0 || W <= 0) return LHN_EINVAL;
  const int64_t n_planes = B * K, total = n_planes * H * W;
  if (total == 0) return LHN_OK;
  int64_t need = (total + 255) / 256, cap = (int64_t)num_sms() * 16;
  int blocks = (int)(need < cap ? need : cap);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == LHN_F32)
    flip_back_kernel<float><<<blocks, 256, 0, st>>>((const float*)in, (float*)out, n_planes, K, H, W, flip_index);
  else if (dtype == LHN_BF16 || dtype == LHN_F16)
    flip_back_kernel<uint16_t><<<blocks, 256, 0, st>>>((const uint16_t*)in, (uint16_t*)out, n_planes, K, H, W, flip_index);
  else return LHN_EDTYPE;
  return check_launch();
}
