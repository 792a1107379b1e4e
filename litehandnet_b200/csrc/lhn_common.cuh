// Shared device helpers for liblhn.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/lhn.h"

namespace lhn {
// what the last SimDR call of this host thread launched (lhn_simdr_last_launch; defined in lhn_simdr.cu)
extern thread_local lhn_simdr_launch_info g_simdr_launch;
inline void simdr_record(int family, int path, int dtype, int warps, int stages, int64_t ctas, int vec_x, int vec_y,
                         int bn) {
  g_simdr_launch = lhn_simdr_launch_info{family, path, dtype, warps, stages, (int32_t)ctas, vec_x, vec_y, bn};
}
}  // namespace lhn

namespace lhn {

constexpr int kWarp = 32;

// thread-local last CUDA error text for lhn_last_cuda_error()
const char* set_last_error(cudaError_t e);
int check_launch();

// ---------------------------------------------------------------------------------------------
// element access
// ---------------------------------------------------------------------------------------------
template <typename T> struct Elem;
template <> struct Elem<float> {
  static __device__ __forceinline__ float to_f32(float v) { return v; }
};
template <> struct Elem<__nv_bfloat16> {
  static __device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
};
template <> struct Elem<__half> {
  static __device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
};

// 4 consecutive elements -> float4 (16 B for f32, 8 B for bf16/f16)
template <typename T> __device__ __forceinline__ float4 load4(const T* p);
template <> __device__ __forceinline__ float4 load4<float>(const float* p) {
  return *reinterpret_cast<const float4*>(p);
}
template <> __device__ __forceinline__ float4 load4<__nv_bfloat16>(const __nv_bfloat16* p) {
  uint2 r = *reinterpret_cast<const uint2*>(p);
  float4 o;
  o.x = __uint_as_float(r.x << 16); o.y = __uint_as_float(r.x & 0xffff0000u);
  o.z = __uint_as_float(r.y << 16); o.w = __uint_as_float(r.y & 0xffff0000u);
  return o;
}
template <> __device__ __forceinline__ float4 load4<__half>(const __half* p) {
  uint2 r = *reinterpret_cast<const uint2*>(p);
  float2 a = __half22float2(*reinterpret_cast<__half2*>(&r.x));
  float2 b = __half22float2(*reinterpret_cast<__half2*>(&r.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

// streaming 128-bit global load (read-once data: do not allocate in L1)
__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
  float4 r;
  asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ uint2 ldg_stream_u2(const uint2* p) {
  uint2 r;
  asm("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
template <typename T> __device__ __forceinline__ float4 ldg_stream4(const T* p);
template <> __device__ __forceinline__ float4 ldg_stream4<float>(const float* p) {
  return ldg_stream_f4(reinterpret_cast<const float4*>(p));
}
template <> __device__ __forceinline__ float4 ldg_stream4<__nv_bfloat16>(const __nv_bfloat16* p) {
  uint2 r = ldg_stream_u2(reinterpret_cast<const uint2*>(p));
  float4 o;
  o.x = __uint_as_float(r.x << 16); o.y = __uint_as_float(r.x & 0xffff0000u);
  o.z = __uint_as_float(r.y << 16); o.w = __uint_as_float(r.y & 0xffff0000u);
  return o;
}
template <> __device__ __forceinline__ float4 ldg_stream4<__half>(const __half* p) {
  uint2 r = ldg_stream_u2(reinterpret_cast<const uint2*>(p));
  float2 a = __half22float2(*reinterpret_cast<__half2*>(&r.x));
  float2 b = __half22float2(*reinterpret_cast<__half2*>(&r.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

// eight 16-bit elements with ONE 128-bit streaming load (a lane's 64-bit loads keep half the bytes in flight)
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p) {
  uint4 r;
  asm("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
template <typename T> __device__ __forceinline__ void ldg_stream8(const T* p, float4& lo, float4& hi);
template <> __device__ __forceinline__ void ldg_stream8<__nv_bfloat16>(const __nv_bfloat16* p, float4& lo, float4& hi) {
  const uint4 r = ldg_stream_u4(reinterpret_cast<const uint4*>(p));
  lo.x = __uint_as_float(r.x << 16); lo.y = __uint_as_float(r.x & 0xffff0000u);
  lo.z = __uint_as_float(r.y << 16); lo.w = __uint_as_float(r.y & 0xffff0000u);
  hi.x = __uint_as_float(r.z << 16); hi.y = __uint_as_float(r.z & 0xffff0000u);
  hi.z = __uint_as_float(r.w << 16); hi.w = __uint_as_float(r.w & 0xffff0000u);
}
template <> __device__ __forceinline__ void ldg_stream8<__half>(const __half* p, float4& lo, float4& hi) {
  uint4 r = ldg_stream_u4(reinterpret_cast<const uint4*>(p));
  const float2 a = __half22float2(*reinterpret_cast<__half2*>(&r.x)), b = __half22float2(*reinterpret_cast<__half2*>(&r.y));
  const float2 c = __half22float2(*reinterpret_cast<__half2*>(&r.z)), d = __half22float2(*reinterpret_cast<__half2*>(&r.w));
  lo = make_float4(a.x, a.y, b.x, b.y); hi = make_float4(c.x, c.y, d.x, d.y);
}
template <> __device__ __forceinline__ void ldg_stream8<float>(const float* p, float4& lo, float4& hi) {
  lo = ldg_stream_f4(reinterpret_cast<const float4*>(p)); hi = ldg_stream_f4(reinterpret_cast<const float4*>(p) + 1);
}

// ---------------------------------------------------------------------------------------------
// argmax with torch/numpy semantics: first maximal index; NaN is maximal; -0 == +0
// ---------------------------------------------------------------------------------------------
// Order-preserving map float -> uint32 (NaN -> 0xffffffff, -0 -> key(+0)).
__device__ __forceinline__ uint32_t order_key(float v) {
  if (v != v) return 0xffffffffu;
  uint32_t b = __float_as_uint(v + 0.0f);   // -0 + +0 = +0
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_to_float(uint32_t k) {
  if (k == 0xffffffffu) return __uint_as_float(0x7fc00000u);
  uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(b);
}
// warp-wide (max key, then min index among the maxima) using redux.sync
__device__ __forceinline__ void warp_argmax(uint32_t& key, uint32_t& idx) {
  uint32_t kmax = __reduce_max_sync(0xffffffffu, key);
  uint32_t cand = (key == kmax) ? idx : 0xffffffffu;
  idx = __reduce_min_sync(0xffffffffu, cand);
  key = kmax;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One joint's term of the fixed-point EPE sum (epe_fix counters): the f32 distance in 2^-20 px, rounded to nearest
// (a power of two, so d * 2^20 is exact).  A distance that is NaN, infinite or too large for the int64 term
// (d >= 2^43 px) adds nothing, and the joint still counts in epe_valid.  Every producer of the counters uses this.
__device__ __forceinline__ unsigned long long epe_fix_term(float d) {
  return d < 0x1p43f ? (unsigned long long)__float2ll_rn(d * 1048576.f) : 0ull;
}

// ---------------------------------------------------------------------------------------------
// Gaussian target geometry (generateTarget.py:100-154 MSRA, :162-243 UDP), shared by the fused kernel,
// the CTA-per-plane fallback, lhn_render_targets, the two-pass backward and the one-pass loss + gradient so
// that all five render the same target.  mode = lhn_render_params.unbiased: 1 = MSRA sub-pixel full plane, 0 = MSRA integer
// centre patch, 2 = UDP (integer patch position, sub-pixel Gaussian centre inside it).
// ---------------------------------------------------------------------------------------------
struct RenderGeom {
  double mux, muy;            // mode 1: the sub-pixel centre
  double ulx, uly, brx, bry;  // patch bounds [ul, br) (modes 0, 2) / visibility-rule bounds (mode 1)
  double x0x, x0y;            // modes 0, 2: centre inside the patch
  float w;                    // target weight after the visibility rule
  float cx, cy;               // centre in plane coordinates, f32 (window of the loss "positives")
  bool on;                    // w > 0.5: the plane carries a Gaussian
};

__device__ __forceinline__ RenderGeom render_geom(float jx, float jy, float w, double sig, int mode, double feat_x,
                                                  double feat_y, int feat_pow2, double inv_feat_x, double inv_feat_y,
                                                  int W, int H) {
  RenderGeom g;
  const double tmp = sig * 3.0;
  // joint / feat_stride in f64 (numpy promotes f32 / f64); a power-of-two stride multiplies exactly
  double mux, muy;
  if (feat_pow2) { mux = (double)jx * inv_feat_x; muy = (double)jy * inv_feat_y; }
  else { mux = (double)jx / feat_x; muy = (double)jy / feat_y; }
  g.x0x = g.x0y = 0.0;
  if (mode == 1) {
    g.ulx = mux - tmp; g.uly = muy - tmp; g.brx = mux + tmp + 1; g.bry = muy + tmp + 1;
    g.cx = (float)mux; g.cy = (float)muy;
  } else {
    const double mix = trunc(mux + 0.5), miy = trunc(muy + 0.5);      // int() truncates toward zero
    g.ulx = trunc(mix - tmp); g.uly = trunc(miy - tmp);
    g.brx = trunc(mix + tmp + 1); g.bry = trunc(miy + tmp + 1);
    const double half = floor((2 * tmp + 1) * 0.5);                   // size // 2
    g.x0x = half; g.x0y = half;
    if (mode == 2) { g.x0x += mux - mix; g.x0y += muy - miy; }        // UDP: x0 += mu_x_ac - mu_x
    g.cx = (float)(g.ulx + g.x0x); g.cy = (float)(g.uly + g.x0y);
    mux = mix; muy = miy;
  }
  g.mux = mux; g.muy = muy;
  if (g.ulx >= W || g.uly >= H || g.brx < 0 || g.bry < 0) w = 0.f;
  g.w = w;
  g.on = w > 0.5f;
  return g;
}

// exponent argument (<= 0) of table entry i (i < W: x table, else y table), or +1 for "no Gaussian here"
__device__ __forceinline__ double render_arg(const RenderGeom& g, int i, int W, int mode, double inv2s2) {
  const bool isx = i < W;
  const int pos = isx ? i : i - W;
  if (mode == 1) {
    const double d = (double)pos - (isx ? g.mux : g.muy);
    return -(d * d) * inv2s2;
  }
  const double ul = isx ? g.ulx : g.uly, br = isx ? g.brx : g.bry;
  if ((double)pos >= ul && (double)pos < br) {
    const double d = ((double)pos - ul) - (isx ? g.x0x : g.x0y);
    return -(d * d) * inv2s2;
  }
  return 1.0;
}

// fast f32 exp of a double argument: exp(a) = exp(ah) * (1 + al), ah = f32(a), al = a - ah
__device__ __forceinline__ float exp_f32_from_f64(double a) {
  const float ah = (float)a;
  const float al = (float)(a - (double)ah);
  const float v = expf(ah);
  return fmaf(v, al, v);
}

// Table entry i (i < W: x table, else y table) of the separable Gaussian: the one definition every kernel that
// renders the target calls, so that they all draw the same bits.  0 on a plane without a Gaussian and outside the
// patch (arg = +1).  `!(arg > 0)` passes a NaN argument (a NaN joint in mode 1) through as NaN, as the reference's
// np.exp does: the plane's target is NaN rather than silently 0.
__device__ __forceinline__ float table_entry(const RenderGeom& g, int i, int W, int mode, double inv2s2) {
  if (!g.on) return 0.f;
  const double arg = render_arg(g, i, W, mode, inv2s2);
  return !(arg > 0.0) ? exp_f32_from_f64(arg) : 0.f;
}

// Host: checks one scale of lhn_render_loss_multi / lhn_render_loss_backward_multi against the shared render
// parameters and gives its feature stride (image_size / [W, H], or (image_size - 1) / ([W, H] - 1) for UDP, as
// lhn_render_targets uses).
inline int scale_geometry(const lhn_render_params* rp, int H, int W, float sigma, double& feat_x, double& feat_y) {
  if (H <= 0 || W <= 0 || (int64_t)H * W > (1 << 30) || !(sigma > 0.f) || !(rp->image_w > 0.f) ||
      !(rp->image_h > 0.f) || rp->loss_mode < LHN_LOSS_DISTANCE || rp->loss_mode > LHN_LOSS_JOINTS_MSE ||
      rp->unbiased < 0 || rp->unbiased > 2)
    return LHN_EINVAL;
  if (rp->unbiased == 2) {
    if (W < 2 || H < 2) return LHN_EINVAL;
    feat_x = ((double)rp->image_w - 1.0) / (W - 1.0); feat_y = ((double)rp->image_h - 1.0) / (H - 1.0);
  } else {
    feat_x = (double)rp->image_w / W; feat_y = (double)rp->image_h / H;
  }
  return LHN_OK;
}

// Host: lets `kernel` take `smem` bytes of dynamic shared memory (above the 48 KB default only when asked for).
inline int set_dynamic_smem(const void* kernel, size_t smem) {
  if (smem <= 48 * 1024) return LHN_OK;
  if (smem > 227 * 1024) return LHN_EINVAL;
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();
    return LHN_EINVAL;
  }
  return LHN_OK;
}

// ---------------------------------------------------------------------------------------------
// gradient stores and loss coefficients, shared by lhn_backward.cu and lhn_loss_grad.cu so that the
// two-pass and the one-pass backward write bit-identical gradients
// ---------------------------------------------------------------------------------------------
template <typename T> struct Store4;
template <> struct Store4<float> {
  static __device__ __forceinline__ void st(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
  static __device__ __forceinline__ float from(float v) { return v; }
};
template <> struct Store4<__nv_bfloat16> {
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float4 v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 r;
    r.x = *reinterpret_cast<uint32_t*>(&a); r.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = r;
  }
  static __device__ __forceinline__ __nv_bfloat16 from(float v) { return __float2bfloat16_rn(v); }
};
template <> struct Store4<__half> {
  static __device__ __forceinline__ void st(__half* p, float4 v) {
    __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
    uint2 r;
    r.x = *reinterpret_cast<uint32_t*>(&a); r.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = r;
  }
  static __device__ __forceinline__ __half from(float v) { return __float2half_rn(v); }
};

// coefficients of the positive / negative elements from the forward sums (f64 -> f32 once)
__device__ __forceinline__ void loss_coefs(const double* sums, int loss_mode, int sum_reduction, float scale,
                                           const float* grad_out, float& cpos, float& cneg) {
  const double npos = sums[2], numel = sums[3];
  double cp, cn;
  if (loss_mode == LHN_LOSS_DISTANCE_BALANCE) { cp = 2.0 * 0.1 / (npos + 1.0); cn = 2.0 / (numel - npos + 1.0); }
  else if (loss_mode == LHN_LOSS_JOINTS_MSE) { cp = cn = 1.0 / numel; }
  else { cp = cn = 2.0 / numel; }
  if (sum_reduction) { cp *= numel; cn *= numel; }
  const double g = (double)scale * (grad_out ? (double)grad_out[0] : 1.0);
  cpos = (float)(cp * g); cneg = (float)(cn * g);
}

// one loss from its f64 sums (S_pos, S_neg, N_pos, numel): the finalise of lhn_loss_mse_multi, lhn_render_loss_multi
// and lhn_render_loss_grad_multi
__device__ __forceinline__ double finalize_loss(double sp, double sn, double npos, double numel, int loss_mode, int sum_reduction) {
  double v;
  if (loss_mode == LHN_LOSS_DISTANCE_BALANCE) v = 0.1 * sp / (npos + 1.0) + sn / (numel - npos + 1.0);
  else if (loss_mode == LHN_LOSS_JOINTS_MSE) v = 0.5 * (sp + sn) / numel;
  else v = (sp + sn) / numel;
  return sum_reduction ? v * numel : v;
}

// ---------------------------------------------------------------------------------------------
// mbarrier + TMA bulk copy (cp.async.bulk, 1-D: no tensor map needed for contiguous planes)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "LHN_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"   // suspend-time hint: fewer polling retries
      "@p bra LHN_DONE;\n"
      "bra LHN_WAIT;\n"
      "LHN_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity), "r"(2000u)
      : "memory");
}
// L2 eviction policy for read-once streams
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                            uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes),
      "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}

}  // namespace lhn
