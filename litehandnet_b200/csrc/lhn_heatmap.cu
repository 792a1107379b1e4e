// K1 — fused heatmap kernel: (flip-average) + argmax + sub-pixel refinement + back-transform,
// optionally fused with Gaussian target rendering, masked-MSE partial sums and PCK/AUC/EPE counters.
// One pass over every heatmap plane: the plane is pulled into shared memory by a TMA bulk copy
// (cp.async.bulk + mbarrier), reduced with warp redux/shuffles, and refined from the resident copy.
// sm_100a only; no tensor cores (nothing here is a dense contraction).
#include <stdlib.h>

#include "lhn_heatmap.cuh"

namespace lhn {

// what the last K1 call of this host thread launched (lhn_k1_last_launch); cleared by run_heatmap, filled by the
// launchers of both kernels
thread_local lhn_k1_launch_info g_k1_launch = {};

// ---- the kernel --------------------------------------------------------------------------------
template <typename T, int WT, bool FLIP, bool LOSS, int NT>
__global__ void __launch_bounds__(NT) heatmap_plane_kernel(const __grid_constant__ HmArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr bool kInPlace = std::is_same<T, float>::value;
  const int H = a.H, W = (WT > 0) ? WT : a.W, HW = a.HW;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int nwarps = NT / 32;

  SmemHeader* sh = reinterpret_cast<SmemHeader*>(smem_raw);
  size_t off = align_up(sizeof(SmemHeader), 16);
  float* ex = reinterpret_cast<float*>(smem_raw + off);
  float* ey = ex + W;
  off += align_up((size_t)(W + H) * sizeof(float), 16);
  off = align_up(off, 128);
  float* work = nullptr;
  if (!kInPlace) { work = reinterpret_cast<float*>(smem_raw + off); off += align_up((size_t)HW * sizeof(float), 128); }
  T* plane0 = reinterpret_cast<T*>(smem_raw + off);
  off += align_up((size_t)HW * sizeof(T), 128);
  T* plane1 = FLIP ? reinterpret_cast<T*>(smem_raw + off) : nullptr;
  // The decoded ("work") plane the epilogue refines from:
  //   f32, no flip : the TMA destination itself;
  //   f32, flip    : the average overwrites the FLIPPED plane in place, stored mirrored — the thread
  //                  that owns quad q is the only reader of the mirrored quad it overwrites, so there
  //                  is no race and the un-flipped plane stays intact for the loss;
  //   bf16/f16     : a separate f32 buffer.
  constexpr bool MIRROR = kInPlace && FLIP;
  if (kInPlace) work = reinterpret_cast<float*>(FLIP ? plane1 : plane0);
  auto widx = [&](int y, int x) { return y * W + (MIRROR ? (W - 1 - x) : x); };

  const int64_t p = blockIdx.x;
  const int64_t b = p / a.C;
  const int c = (int)(p - b * a.C);
  const int s = c / a.K;
  const int k = c - s * a.K;

  const T* g0 = reinterpret_cast<const T*>(a.hm) + b * a.stride_b + (int64_t)c * a.stride_c;
  const T* g1 = nullptr;
  if (FLIP) {
    int kf = a.flip_index ? a.flip_index[k] : k;
    g1 = reinterpret_cast<const T*>(a.hm_flip) + b * a.fstride_b + (int64_t)(s * a.K + kf) * a.fstride_c;
  }

  // ---- issue the plane loads -----------------------------------------------------------------
  const uint32_t plane_bytes = (uint32_t)HW * sizeof(T);
  if (a.use_tma) {
    if (tid == 0) {
      mbar_init(&sh->bar, 1);
      fence_mbar_init();
      uint64_t pol = policy_evict_first();
      mbar_arrive_expect_tx(&sh->bar, FLIP ? 2 * plane_bytes : plane_bytes);
      tma_load_1d(plane0, g0, plane_bytes, &sh->bar, pol);
      if (FLIP) tma_load_1d(plane1, g1, plane_bytes, &sh->bar, pol);
    }
  } else {
    for (int e = tid; e < HW; e += NT) {
      plane0[e] = g0[e];
      if (FLIP) plane1[e] = g1[e];
    }
  }

  // ---- per-plane render parameters + separable Gaussian tables (overlaps the load) -----------
  float w = 0.f, gcx = 0.f, gcy = 0.f;
  bool render_on = false;
  if (LOSS) {
    const float* jp = a.joints + (b * a.K + k) * (int64_t)a.joints_stride;
    const double sig = (double)a.sigma[s];
    const RenderGeom g = render_geom(jp[0], jp[1], a.vis[(b * a.K + k) * (int64_t)a.vis_stride], sig, a.unbiased,
                                     a.feat_x, a.feat_y, 0, 0.0, 0.0, W, H);
    w = g.w;
    render_on = g.on;
    gcx = g.cx; gcy = g.cy;
    const double inv2s2 = 1.0 / (2.0 * sig * sig);
    for (int i = tid; i < W + H; i += NT) ex[i] = table_entry(g, i, W, a.unbiased, inv2s2);   // ey follows ex
  }
  __syncthreads();   // tables (and the non-TMA copy) visible
  if (a.use_tma) mbar_wait(&sh->bar, 0);

  // ---- pass 1: one sweep over the plane -------------------------------------------------------
  // kUseS: without flip the loss sum S already turns non-finite when the plane holds a NaN/inf
  constexpr bool kUseS = LOSS && !FLIP;
  float S0 = 0.f, S1 = 0.f, nacc = 0.f;
  float best = -CUDART_INF_F;
  uint32_t bidx = 0xffffffffu;
  const bool vec_ok = (WT > 0) || ((W & 3) == 0);
  if (vec_ok) {
    const int QR = W >> 2;
    const int nq = HW >> 2;
#pragma unroll 4
    for (int q = tid; q < nq; q += NT) {
      const int row = q / QR;
      const int cq = q - row * QR;
      const float4 o = load4<T>(plane0 + 4 * q);
      float4 v = o;
      const int mq = row * W + (W - 4 - 4 * cq);     // mirrored quad
      if (FLIP) {
        const float4 f = load4<T>(plane1 + mq);
        v.x = __fmul_rn(__fadd_rn(o.x, f.w), 0.5f);
        v.y = __fmul_rn(__fadd_rn(o.y, f.z), 0.5f);
        v.z = __fmul_rn(__fadd_rn(o.z, f.y), 0.5f);
        v.w = __fmul_rn(__fadd_rn(o.w, f.x), 0.5f);
      }
      if (LOSS) {   // the loss is taken on the un-flipped network output
        const float4 gx = *reinterpret_cast<const float4*>(ex + 4 * cq);
        const float gy = ey[row];
        const float d0 = o.x - gx.x * gy, d1 = o.y - gx.y * gy, d2 = o.z - gx.z * gy, d3 = o.w - gx.w * gy;
        S0 = fmaf(d0, d0, S0); S1 = fmaf(d1, d1, S1); S0 = fmaf(d2, d2, S0); S1 = fmaf(d3, d3, S1);
      }
      if (!kUseS) {
        nacc = fmaf(v.x, 0.f, nacc); nacc = fmaf(v.y, 0.f, nacc);
        nacc = fmaf(v.z, 0.f, nacc); nacc = fmaf(v.w, 0.f, nacc);
      }
      if (MIRROR) *reinterpret_cast<float4*>(work + mq) = make_float4(v.w, v.z, v.y, v.x);
      else if (!kInPlace) *reinterpret_cast<float4*>(work + 4 * q) = v;
      const uint32_t e = 4u * q;
      if (v.x > best) { best = v.x; bidx = e; }
      if (v.y > best) { best = v.y; bidx = e + 1; }
      if (v.z > best) { best = v.z; bidx = e + 2; }
      if (v.w > best) { best = v.w; bidx = e + 3; }
    }
  } else {
    for (int e = tid; e < HW; e += NT) {
      const int row = e / W;
      const int col = e - row * W;
      const float o = Elem<T>::to_f32(plane0[e]);
      float v = o;
      if (FLIP) v = __fmul_rn(__fadd_rn(o, Elem<T>::to_f32(plane1[row * W + (W - 1 - col)])), 0.5f);
      if (LOSS) { float d = o - ex[col] * ey[row]; S0 = fmaf(d, d, S0); }
      if (!kUseS) nacc = fmaf(v, 0.f, nacc);
      if (MIRROR || !kInPlace) work[widx(row, col)] = v;
      if (v > best) { best = v; bidx = e; }
    }
  }

  // ---- block reduction ------------------------------------------------------------------------
  uint32_t key = order_key(best);
  warp_argmax(key, bidx);
  double ssum = 0.0;
  if (LOSS) ssum = warp_sum((double)S0 + (double)S1);
  if (lane == 0) { sh->red_key[warp] = key; sh->red_idx[warp] = bidx; sh->red_s[warp] = ssum; }
  // NaN/inf anywhere in the decoded plane (S may also overflow on huge finite values: that only
  // costs the slow path, never correctness)
  const bool nonfinite = kUseS ? !(fabsf(S0 + S1) < CUDART_INF_F) : (nacc != nacc);
  const int any_nonfinite = __syncthreads_or(nonfinite ? 1 : 0);

  if (warp == 0) {
    uint32_t k2 = lane < nwarps ? sh->red_key[lane] : 0u;
    uint32_t i2 = lane < nwarps ? sh->red_idx[lane] : 0xffffffffu;
    warp_argmax(k2, i2);
    if (i2 == 0xffffffffu) i2 = 0;     // every element is -inf: first index
    if (lane == 0) { sh->idx = i2; sh->maxval = key_to_float(k2); sh->nan_found = 0; sh->need_slow = 0; }
  }
  __syncthreads();

  if (any_nonfinite) {
    // rare: find the first NaN (np.argmax / torch.max treat NaN as maximal)
    uint32_t first_nan = 0xffffffffu;
    for (int e = tid; e < HW; e += NT) {
      const int y = e / W;
      const float v = work[widx(y, e - y * W)];
      if (v != v) { first_nan = (uint32_t)e; break; }
    }
    first_nan = __reduce_min_sync(0xffffffffu, first_nan);
    if (lane == 0) sh->red_idx[warp] = first_nan;
    __syncthreads();
    if (tid == 0) {
      uint32_t m = 0xffffffffu;
      for (int i = 0; i < nwarps; ++i) m = min(m, sh->red_idx[i]);
      if (m != 0xffffffffu) { sh->idx = m; sh->maxval = __uint_as_float(0x7fc00000u); sh->nan_found = 1; }
    }
    __syncthreads();
  }

  const uint32_t idx = sh->idx;
  const float maxval = sh->maxval;
  const int ipx = (int)(idx % (uint32_t)W), ipy = (int)(idx / (uint32_t)W);

  // masked integer coordinates (A1-A4)
  float cx = (float)ipx, cy = (float)ipy;
  const bool positive = maxval > 0.0f;   // false for NaN
  if (a.mask_mode == LHN_MASK_ZERO && !positive) { cx = 0.f; cy = 0.f; }
  if (a.mask_mode == LHN_MASK_NEG1 && !positive) { cx = -1.f; cy = -1.f; }

  const bool is_dark = (a.refine == LHN_REFINE_DARK) || (a.refine == LHN_REFINE_DARK_LEGACY);
  const bool legacy = a.refine == LHN_REFINE_DARK_LEGACY;
  const int px = (int)cx, py = (int)cy;      // int() of the (possibly masked) coordinates
  const bool dark_guard = is_dark && (1 < px) && (px < W - 2) && (1 < py) && (py < H - 2);

  if (is_dark) {
    if (warp == 0 && dark_guard) {
      if (legacy) dark_window<double, MIRROR>(work, H, W, px, py, a.ksize, a.tapsd, sh->hbuf, sh->hout, lane);
      else dark_window<float, MIRROR>(work, H, W, px, py, a.ksize, a.tapsf, reinterpret_cast<float*>(sh->hbuf), sh->hout, lane);
      // can the 1e-10 clamp (or a non-finite value) influence the 13 stencil points?
      float hv = lane < 25 ? sh->hout[lane] : CUDART_INF_F;
      const int dr = lane / 5 - 2, dc = lane % 5 - 2;
      const bool used = lane < 25 && (abs(dr) + abs(dc) <= 2);
      bool bad = used && !(hv >= 1e-9f);
      // origin_max is the plane max (np.max), which equals maxval (NaN included)
      bool ok_origin = legacy ? (maxval >= 1e-3f) : (maxval > 0.f);
      unsigned anybad = __ballot_sync(0xffffffffu, bad);
      if (lane == 0) sh->need_slow = (anybad != 0u || !ok_origin || any_nonfinite) ? 1 : 0;
    }
    __syncthreads();
    if (sh->need_slow) {
      // exact emulation: max of the blurred plane (NaN propagates like np.max)
      float m = -CUDART_INF_F;
      bool first = true;
      for (int e = tid; e < HW; e += NT) {
        int y = e / W, x = e - y * W;
        float v = legacy ? blur_at<double, MIRROR>(work, H, W, x, y, a.ksize, a.tapsd)
                         : blur_at<float, MIRROR>(work, H, W, x, y, a.ksize, a.tapsf);
        m = first ? v : nanmax(m, v);
        first = false;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = nanmax(m, __shfl_xor_sync(0xffffffffu, m, o));
      if (lane == 0) sh->red_b[warp] = (double)m;
      __syncthreads();
      if (tid == 0) {
        float mm = (float)sh->red_b[0];
        for (int i = 1; i < nwarps; ++i) mm = nanmax(mm, (float)sh->red_b[i]);
        sh->bmax = mm;
      }
      __syncthreads();
    }
  }

  // ---- epilogue: warp 0 -----------------------------------------------------------------------
  if (warp != 0) return;

  double S = 0.0;
  if (LOSS) {
    double t = lane < nwarps ? sh->red_s[lane] : 0.0;
    S = warp_sum(t);
  }

  // positives of the balanced loss live in a small window around the joint: sum them from smem
  double Spos = 0.0;
  int Npos = 0;
  if (LOSS && a.loss_mode == LHN_LOSS_DISTANCE_BALANCE) {
    const float* jp = a.joints + (b * a.K + k) * (int64_t)a.joints_stride;
    const float sig = a.sigma[s];
    int x_lo = 0, x_hi = W - 1, y_lo = 0, y_hi = H - 1;
    if (a.pos_value > 0.f && a.pos_value < 1.f) {
      // g > value  <=>  r^2 < -2 sigma^2 ln(value); per axis |d| < sqrt(-2 ln value) * sigma
      const float rad = sqrtf(-2.f * logf(a.pos_value)) * sig + 1.5f;
      const float mx = gcx, my = gcy;                     // Gaussian centre in plane coordinates
      x_lo = max(0, (int)floorf(mx - rad)); x_hi = min(W - 1, (int)ceilf(mx + rad));
      y_lo = max(0, (int)floorf(my - rad)); y_hi = min(H - 1, (int)ceilf(my + rad));
    } else if (a.pos_value >= 1.f) {
      x_hi = -1;   // g <= 1 always: no positives
    }
    if (render_on || a.pos_value < 0.f) {
      const int ww = x_hi - x_lo + 1, hh = y_hi - y_lo + 1;
      const int n = (ww > 0 && hh > 0) ? ww * hh : 0;
      for (int e = lane; e < n; e += kWarp) {
        int yy = y_lo + e / ww, xx = x_lo + e % ww;
        float g = ex[xx] * ey[yy];
        if (g > a.pos_value) {
          float o = Elem<T>::to_f32(plane0[yy * W + xx]);
          float d = o - g;
          Spos += (double)(d * d);
          Npos += 1;
        }
      }
      Spos = warp_sum(Spos);
      Npos = __reduce_add_sync(0xffffffffu, Npos);
    }
  }

  if (lane != 0) return;

  // ---- sub-pixel refinement (D1-D6) on the resident plane ------------------------------------
  float rx = cx, ry = cy;
  const float* P = work;
  switch (a.refine) {
    case LHN_REFINE_OFFSET_HALF:
    case LHN_REFINE_OFFSET: {
      const int xx = min(max(px, 0), W - 1), yy = min(max(py, 0), H - 1);
      // clamped neighbours; `>` false (equality, NaN) -> -0.25
      rx += (P[widx(yy, min(xx + 1, W - 1))] > P[widx(yy, max(xx - 1, 0))]) ? 0.25f : -0.25f;
      ry += (P[widx(min(yy + 1, H - 1), xx)] > P[widx(max(yy - 1, 0), xx)]) ? 0.25f : -0.25f;
      if (a.refine == LHN_REFINE_OFFSET_HALF) { rx += 0.5f; ry += 0.5f; }
      break;
    }
    case LHN_REFINE_SIGN:
    case LHN_REFINE_SIGN_ROUND: {
      int qx = px, qy = py;
      if (a.refine == LHN_REFINE_SIGN_ROUND) { qx = (int)floorf(cx + 0.5f); qy = (int)floorf(cy + 0.5f); }
      if (1 < qx && qx < W - 1 && 1 < qy && qy < H - 1) {
        float ddx = P[widx(qy, qx + 1)] - P[widx(qy, qx - 1)];
        float ddy = P[widx(qy + 1, qx)] - P[widx(qy - 1, qx)];
        // np.sign: +-1, 0 for 0, NaN for NaN
        float sxn = (ddx != ddx) ? ddx : (float)((ddx > 0.f) - (ddx < 0.f));
        float syn = (ddy != ddy) ? ddy : (float)((ddy > 0.f) - (ddy < 0.f));
        rx += sxn * 0.25f; ry += syn * 0.25f;
      }
      break;
    }
    case LHN_REFINE_DARK:
    case LHN_REFINE_DARK_LEGACY: {
      if (dark_guard) {
        float h[25];
        if (sh->need_slow) {
          const float bmax = sh->bmax;
          const float sc = legacy ? __fdiv_rn(maxval, __fadd_rn(bmax, 1e-6f)) : __fdiv_rn(maxval, bmax);
#pragma unroll
          for (int i = 0; i < 25; ++i) {
            float v = __fmul_rn(sh->hout[i], sc);
            v = (v != v) ? v : fmaxf(v, 1e-10f);     // np.maximum propagates NaN
            h[i] = logf(v);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 25; ++i) h[i] = logf(sh->hout[i]);
        }
#define HH(dy, dx) h[((dy) + 2) * 5 + (dx) + 2]
        const float ddx = __fmul_rn(0.5f, __fsub_rn(HH(0, 1), HH(0, -1)));
        const float ddy = __fmul_rn(0.5f, __fsub_rn(HH(1, 0), HH(-1, 0)));
        const float dxx = __fmul_rn(0.25f, __fadd_rn(__fsub_rn(HH(0, 2), __fmul_rn(2.f, HH(0, 0))), HH(0, -2)));
        const float dxy = __fmul_rn(0.25f, __fadd_rn(__fsub_rn(__fsub_rn(HH(1, 1), HH(-1, 1)), HH(1, -1)), HH(-1, -1)));
        const float dyy = __fmul_rn(0.25f, __fadd_rn(__fsub_rn(HH(2, 0), __fmul_rn(2.f, HH(0, 0))), HH(-2, 0)));
#undef HH
        const float det = __fsub_rn(__fmul_rn(dxx, dyy), __fmul_rn(dxy, dxy));
        if (det != 0.f) {   // true for NaN, as in numpy
          const float ox = -__fdiv_rn(__fsub_rn(__fmul_rn(dyy, ddx), __fmul_rn(dxy, ddy)), det);
          const float oy = -__fdiv_rn(__fsub_rn(__fmul_rn(dxx, ddy), __fmul_rn(dxy, ddx)), det);
          rx = __fadd_rn(rx, ox); ry = __fadd_rn(ry, oy);
        }
      }
      break;
    }
    default: break;
  }

  // ---- back-transform (T1/T2) -----------------------------------------------------------------
  float X = rx, Y = ry;
  if (a.transform == LHN_XFORM_CENTER_SCALE) {
    const float s0 = __fmul_rn(a.scale[2 * b], 200.0f), s1 = __fmul_rn(a.scale[2 * b + 1], 200.0f);
    const float dw = a.use_udp ? (float)(W - 1) : (float)W, dh = a.use_udp ? (float)(H - 1) : (float)H;
    const float fx = __fdiv_rn(s0, dw), fy = __fdiv_rn(s1, dh);
    X = __fsub_rn(__fadd_rn(__fmul_rn(rx, fx), a.center[2 * b]), __fmul_rn(s0, 0.5f));
    Y = __fsub_rn(__fadd_rn(__fmul_rn(ry, fy), a.center[2 * b + 1]), __fmul_rn(s1, 0.5f));
  } else if (a.transform == LHN_XFORM_SCALE) {
    X = __fmul_rn(rx, a.scale_x); Y = __fmul_rn(ry, a.scale_y);
  }

  if (a.out_hm) { float* o = a.out_hm + 3 * p; o[0] = rx; o[1] = ry; o[2] = maxval; }
  if (a.out_kpts) { float* o = a.out_kpts + 3 * p; o[0] = X; o[1] = Y; o[2] = maxval; }
  if (a.out_idx) a.out_idx[p] = (int32_t)idx;

  if (LOSS) {
    float wp = (a.loss_mode == LHN_LOSS_JOINTS_MSE) ? w * w : w;
    double* o = a.partials + 4 * p;
    double sall = S * (double)wp, spos = Spos * (double)wp;
    o[0] = spos; o[1] = sall - spos; o[2] = (double)Npos; o[3] = (double)HW;
    if (a.out_weight) a.out_weight[p] = w;
  }

  // ---- fused PCK / AUC / EPE counters (_calc_distances in f64, compared in f32) ----------------
  if (a.counters) {
    const int K = a.K;
    const int64_t bk = b * K + k;
    if (a.mask[bk]) {
      const double gx = (double)a.gt[2 * bk], gy = (double)a.gt[2 * bk + 1];
      const double ddx = (double)X - gx, ddy = (double)Y - gy;
      unsigned long long* cnt = reinterpret_cast<unsigned long long*>(a.counters);
      // PCK: normalize = max(bbox w, h) on both axes; ==0 masks the sample, <0 -> 1e6
      double nb = (double)fmaxf(a.bbox_wh[2 * b], a.bbox_wh[2 * b + 1]);
      if (nb != 0.0) {
        if (nb < 0.0) nb = 1e6;
        double qx = ddx / nb, qy = ddy / nb;
        float d = (float)sqrt(__dadd_rn(__dmul_rn(qx, qx), __dmul_rn(qy, qy)));
        atomicAdd(cnt + K + k, 1ull);
        if (d < a.pck_thr) atomicAdd(cnt + k, 1ull);
      }
      // AUC: normalize = auc_nor
      {
        double qx = ddx / (double)a.auc_nor, qy = ddy / (double)a.auc_nor;
        float d = (float)sqrt(__dadd_rn(__dmul_rn(qx, qx), __dmul_rn(qy, qy)));
        unsigned long long* auc = cnt + 2 * K;
        for (int t = 0; t < a.auc_steps; ++t) {
          float thr = (float)(1.0 * t / a.auc_steps);
          if (d < thr) atomicAdd(auc + (int64_t)t * K + k, 1ull);
        }
        atomicAdd(auc + (int64_t)a.auc_steps * K + k, 1ull);
      }
      // EPE: normalize = 1
      {
        float d = (float)sqrt(__dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy)));
        unsigned long long* epe = cnt + (int64_t)(3 + a.auc_steps) * K;
        atomicAdd(epe + k, 1ull);
        atomicAdd(epe + K + k, epe_fix_term(d));
      }
    }
  }
}

// ---- host-side launch ---------------------------------------------------------------------------
template <typename T, int WT, bool FLIP, bool LOSS>
static int launch_plane_kernel(const HmArgs& a, cudaStream_t st) {
  constexpr int NT = (WT == 128) ? 256 : 128;
  auto kern = heatmap_plane_kernel<T, WT, FLIP, LOSS, NT>;
  size_t smem = smem_bytes_for<T>(a.H, a.W, FLIP);
  if (smem > 227 * 1024) return LHN_EINVAL;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_last_error(e); return LHN_ECUDA; }
  }
  kern<<<(unsigned)a.n_planes, NT, smem, st>>>(a);
  const int rc = check_launch();
  if (rc == LHN_OK) {
    lhn_k1_launch_info& r = g_k1_launch;
    r = {};
    r.path = 2;
    r.dtype = std::is_same<T, float>::value ? LHN_F32 : std::is_same<T, __nv_bfloat16>::value ? LHN_BF16 : LHN_F16;
    r.flip = FLIP; r.loss = LOSS; r.counters = a.counters != nullptr;
    r.wc = WT; r.use_tma = a.use_tma; r.ctas = (int32_t)a.n_planes;
  }
  return rc;
}

template <typename T>
static int dispatch_shape(const HmArgs& a, bool flip, bool loss, cudaStream_t st) {
#define LHN_GO(WT)                                                                   \
  do {                                                                               \
    if (flip) return loss ? launch_plane_kernel<T, WT, true, true>(a, st)            \
                          : launch_plane_kernel<T, WT, true, false>(a, st);          \
    return loss ? launch_plane_kernel<T, WT, false, true>(a, st)                     \
                : launch_plane_kernel<T, WT, false, false>(a, st);                   \
  } while (0)
  if (a.W == 128) LHN_GO(128);
  LHN_GO(0);
#undef LHN_GO
}

static int run_heatmap(HmArgs& a, int dtype, cudaStream_t st, int* used_team_kernel = nullptr) {
  const bool flip = a.hm_flip != nullptr;
  const bool loss = a.loss_mode != LHN_LOSS_NONE;
  const size_t esz = dtype == LHN_F32 ? 4 : 2;
  g_k1_launch = {};
  // TMA bulk copies need 16-byte aligned sources and sizes
  auto aligned = [&](const void* base, int64_t sb, int64_t sc) {
    return ((uintptr_t)base % 16 == 0) && ((sb * esz) % 16 == 0) && ((sc * esz) % 16 == 0);
  };
  a.use_tma = (((size_t)a.HW * esz) % 16 == 0) && aligned(a.hm, a.stride_b, a.stride_c) &&
              (!flip || aligned(a.hm_flip, a.fstride_b, a.fstride_c));
  if ((uintptr_t)a.hm % esz) return LHN_EALIGN;
  if (dtype != LHN_F32 && dtype != LHN_BF16 && dtype != LHN_F16) return LHN_EDTYPE;
  // primary path: persistent warp-per-plane kernel; +1 = shape outside its envelope
  {
    const char* f = getenv("LHN_FORCE_CTA_KERNEL");
    a.force_cta_kernel = (f && f[0] == '1') ? 1 : 0;
  }
  if (a.refine == LHN_REFINE_DARK_UDP) {
    // one mirror reflection per side (cv2 BORDER_REFLECT_101 over a (k-1)/2 + 2 margin); team kernel only
    const int margin = ((a.ksize - 1) >> 1) + 2;
    if (a.H <= margin || a.W <= margin || a.force_cta_kernel) return LHN_EINVAL;
  }
  if (!a.force_cta_kernel) {
    const int rc = launch_heatmap_warp_kernel(a, dtype, st);
    if (rc <= 0) { if (used_team_kernel) *used_team_kernel = 1; return rc; }
    if (a.refine == LHN_REFINE_DARK_UDP) return LHN_EINVAL;      // the CTA-per-plane fallback has no UDP decode
  }
  if (a.fallback_partials) a.partials = a.fallback_partials;   // the CTA-per-plane kernel needs per-plane sums
  switch (dtype) {
    case LHN_F32: return dispatch_shape<float>(a, flip, loss, st);
    case LHN_BF16: return dispatch_shape<__nv_bfloat16>(a, flip, loss, st);
    case LHN_F16: return dispatch_shape<__half>(a, flip, loss, st);
    default: return LHN_EDTYPE;
  }
}

static int fill_decode(HmArgs& a, const lhn_decode_params* dp) {
  if (!dp) return LHN_EINVAL;
  if (dp->mask_mode < 0 || dp->mask_mode > 2 || dp->refine < 0 || dp->refine > 7 ||
      dp->transform < 0 || dp->transform > 2)
    return LHN_EINVAL;
  a.mask_mode = dp->mask_mode; a.refine = dp->refine; a.transform = dp->transform;
  a.use_udp = dp->use_udp; a.scale_x = dp->scale_x; a.scale_y = dp->scale_y;
  a.ksize = dp->blur_ksize;
  a.overlap_previous = (dp->flags & LHN_FLAG_OVERLAP_PREVIOUS) ? 1 : 0;
  a.spare_sms = (dp->flags >> 8) & 0xff;
  a.loss_accumulate = (dp->flags & LHN_FLAG_ACCUMULATE_LOSS) ? 1 : 0;
  if (dp->refine == LHN_REFINE_DARK || dp->refine == LHN_REFINE_DARK_LEGACY || dp->refine == LHN_REFINE_DARK_UDP) {
    if (a.ksize < 3 || a.ksize > LHN_MAX_TAPS || (a.ksize & 1) == 0) return LHN_EINVAL;
    for (int i = 0; i < a.ksize; ++i) { a.tapsd[i] = dp->taps[i]; a.tapsf[i] = (float)dp->taps[i]; }
  }
  if (dp->transform == LHN_XFORM_CENTER_SCALE && (!a.center || !a.scale)) return LHN_EINVAL;
  return LHN_OK;
}

static int fill_exchange(HmArgs& a, const lhn_exchange* x) {
  if (!x) return LHN_OK;
  if (x->world < 1 || x->world > LHN_XCH_MAX_RANKS || x->rank < 0 || x->rank >= x->world || x->seq == 0) return LHN_EINVAL;
  for (int r = 0; r < x->world; ++r) {
    if (!x->mailbox[r]) return LHN_EINVAL;
    if ((uintptr_t)x->mailbox[r] % 16) return LHN_EALIGN;
    a.xch.mail[r] = static_cast<unsigned char*>(x->mailbox[r]);
  }
  a.xch.world = x->world; a.xch.rank = x->rank; a.xch.timeout_ms = x->timeout_ms; a.xch.status = x->status;
  a.xch_seq = x->seq;
  a.xch_prev_block = static_cast<unsigned long long*>(x->prev_block);
  a.xch_prev_seq = x->prev_seq;
  a.xch_prev2_block = static_cast<unsigned long long*>(x->prev2_block);
  a.xch_prev2_seq = x->prev2_seq;
  if ((x->prev_block && x->prev_seq == 0) || (x->prev2_block && x->prev2_seq == 0)) return LHN_EINVAL;
  return LHN_OK;
}

}  // namespace lhn

using namespace lhn;

namespace lhn { int num_sms(); }

// workspace layout of the one-launch step: [ticket u32 | pad to 256 B][loss-sum rows x 4 f64: one per CTA is used,
// the region keeps its older size of one per team][partials of the three-launch fallback: n_planes x 4 f64]
static const int64_t kWsHeader = 256;
static int64_t ws_team_bytes() { return (int64_t)lhn::num_sms() * lhn::kMaxTeamsPerCta * 32; }

extern "C" int lhn_k1_last_launch(lhn_k1_launch_info* out) {
  if (!out) return LHN_EINVAL;
  *out = lhn::g_k1_launch;
  return LHN_OK;
}

extern "C" int64_t lhn_fused_workspace_bytes(int64_t B, int K, int num_stacks) {
  if (B < 0 || K <= 0) return 0;
  const int S = num_stacks > 0 ? num_stacks : 1;
  return kWsHeader + ws_team_bytes() + B * K * S * 32;
}

static int decode_heatmap_impl(const void* hm, const void* hm_flip, const int32_t* flip_index,
                               int dtype, int64_t B, int K, int H, int W, int64_t stride_b,
                               int64_t stride_c, int64_t flip_stride_b, int64_t flip_stride_c,
                               const float* center, const float* scale,
                               const lhn_decode_params* dp, float* out_hm, float* out_kpts,
                               int32_t* out_idx, const lhn_render_params* rp, const float* joints,
                               int joints_stride, const float* vis, int vis_stride,
                               float* out_weight, double* partials, bool fused, void* workspace,
                               int64_t workspace_bytes, double* sums, int sum_reduction,
                               float loss_scale, float* loss, lhn_stream_t stream, const lhn_exchange* xch = nullptr);

extern "C" int lhn_fused_render_loss_decode(const void* hm, const void* hm_flip,
                                            const int32_t* flip_index, int dtype, int64_t B, int K,
                                            int H, int W, int64_t stride_b, int64_t stride_c,
                                            int64_t flip_stride_b, int64_t flip_stride_c,
                                            const float* center, const float* scale,
                                            const lhn_decode_params* dp, float* out_hm,
                                            float* out_kpts, int32_t* out_idx,
                                            const lhn_render_params* rp, const float* joints,
                                            int joints_stride, const float* vis, int vis_stride,
                                            float* out_weight, double* partials, void* workspace,
                                            int64_t workspace_bytes, double* sums, int sum_reduction,
                                            float loss_scale, float* loss, lhn_stream_t stream) {
  if (!rp || rp->loss_mode == LHN_LOSS_NONE || !workspace) return LHN_EINVAL;
  if ((uintptr_t)workspace % 16) return LHN_EALIGN;
  return decode_heatmap_impl(hm, hm_flip, flip_index, dtype, B, K, H, W, stride_b, stride_c,
                             flip_stride_b, flip_stride_c, center, scale, dp, out_hm, out_kpts, out_idx,
                             rp, joints, joints_stride, vis, vis_stride, out_weight, partials, true,
                             workspace, workspace_bytes, sums, sum_reduction, loss_scale, loss, stream);
}

extern "C" int lhn_fused_render_loss_decode_xch(const void* hm, const void* hm_flip,
                                                const int32_t* flip_index, int dtype, int64_t B, int K,
                                                int H, int W, int64_t stride_b, int64_t stride_c,
                                                int64_t flip_stride_b, int64_t flip_stride_c,
                                                const float* center, const float* scale,
                                                const lhn_decode_params* dp, float* out_hm,
                                                float* out_kpts, int32_t* out_idx,
                                                const lhn_render_params* rp, const float* joints,
                                                int joints_stride, const float* vis, int vis_stride,
                                                float* out_weight, double* partials, void* workspace,
                                                int64_t workspace_bytes, double* sums, int sum_reduction,
                                                float loss_scale, float* loss, const lhn_exchange* xch,
                                                lhn_stream_t stream) {
  if (!rp || rp->loss_mode == LHN_LOSS_NONE || !workspace || !xch) return LHN_EINVAL;
  if ((uintptr_t)workspace % 16) return LHN_EALIGN;
  return decode_heatmap_impl(hm, hm_flip, flip_index, dtype, B, K, H, W, stride_b, stride_c,
                             flip_stride_b, flip_stride_c, center, scale, dp, out_hm, out_kpts, out_idx,
                             rp, joints, joints_stride, vis, vis_stride, out_weight, partials, true,
                             workspace, workspace_bytes, sums, sum_reduction, loss_scale, loss, stream, xch);
}

extern "C" int lhn_decode_heatmap(const void* hm, const void* hm_flip, const int32_t* flip_index,
                                  int dtype, int64_t B, int K, int H, int W, int64_t stride_b,
                                  int64_t stride_c, int64_t flip_stride_b, int64_t flip_stride_c,
                                  const float* center, const float* scale,
                                  const lhn_decode_params* dp, float* out_hm, float* out_kpts,
                                  int32_t* out_idx, const lhn_render_params* rp, const float* joints,
                                  int joints_stride, const float* vis, int vis_stride,
                                  float* out_weight, double* partials, lhn_stream_t stream) {
  return decode_heatmap_impl(hm, hm_flip, flip_index, dtype, B, K, H, W, stride_b, stride_c,
                             flip_stride_b, flip_stride_c, center, scale, dp, out_hm, out_kpts, out_idx,
                             rp, joints, joints_stride, vis, vis_stride, out_weight, partials, false,
                             nullptr, 0, nullptr, 0, 1.f, nullptr, stream);
}

static int decode_heatmap_impl(const void* hm, const void* hm_flip, const int32_t* flip_index,
                               int dtype, int64_t B, int K, int H, int W, int64_t stride_b,
                               int64_t stride_c, int64_t flip_stride_b, int64_t flip_stride_c,
                               const float* center, const float* scale,
                               const lhn_decode_params* dp, float* out_hm, float* out_kpts,
                               int32_t* out_idx, const lhn_render_params* rp, const float* joints,
                               int joints_stride, const float* vis, int vis_stride,
                               float* out_weight, double* partials, bool fused, void* workspace,
                               int64_t workspace_bytes, double* sums, int sum_reduction,
                               float loss_scale, float* loss, lhn_stream_t stream, const lhn_exchange* xch) {
  if (B < 0 || K <= 0 || H <= 0 || W <= 0) return LHN_EINVAL;
  if (B == 0) return LHN_OK;
  if (!hm) return LHN_EINVAL;
  HmArgs a{};
  const int S = (rp && rp->num_stacks > 0) ? rp->num_stacks : 1;
  if (S > LHN_MAX_STACKS) return LHN_EINVAL;
  a.hm = hm; a.hm_flip = hm_flip; a.flip_index = flip_index;
  a.stride_b = stride_b; a.stride_c = stride_c; a.fstride_b = flip_stride_b; a.fstride_c = flip_stride_c;
  a.C = S * K; a.K = K; a.H = H; a.W = W; a.HW = H * W;
  a.n_planes = B * a.C;
  a.center = center; a.scale = scale;
  a.out_hm = out_hm; a.out_kpts = out_kpts; a.out_idx = out_idx;
  int rc = fill_decode(a, dp);
  if (rc) return rc;
  a.loss_mode = rp ? rp->loss_mode : LHN_LOSS_NONE;
  if (a.loss_mode != LHN_LOSS_NONE) {
    if (a.loss_mode < 0 || a.loss_mode > 3 || !joints || !vis || (!partials && !fused) || joints_stride < 2 ||
        vis_stride < 1 || rp->image_w <= 0 || rp->image_h <= 0)
      return LHN_EINVAL;
    a.unbiased = rp->unbiased;
    if (rp->unbiased < 0 || rp->unbiased > 2) return LHN_EINVAL;
    if (rp->unbiased == 2) {   // UDP: feat_stride = (image_size - 1) / (heatmap_size - 1), generateTarget.py:208
      if (W < 2 || H < 2) return LHN_EINVAL;
      a.feat_x = ((double)rp->image_w - 1.0) / ((double)W - 1.0); a.feat_y = ((double)rp->image_h - 1.0) / ((double)H - 1.0);
    } else {
      a.feat_x = (double)rp->image_w / (double)W; a.feat_y = (double)rp->image_h / (double)H;
    }
    a.pos_value = rp->pos_value;
    for (int i = 0; i < S; ++i) { if (!(rp->sigma[i] > 0.f)) return LHN_EINVAL; a.sigma[i] = rp->sigma[i]; }
    a.joints = joints; a.joints_stride = joints_stride; a.vis = vis; a.vis_stride = vis_stride;
    a.out_weight = out_weight; a.partials = partials;
  }
  if (a.n_planes == 0) return LHN_OK;
  if (a.n_planes > 0x7fffffffLL) return LHN_EINVAL;
  if (!fused) return run_heatmap(a, dtype, (cudaStream_t)stream);
  // ---- one-launch step ------------------------------------------------------------------------------
  if (workspace_bytes < kWsHeader + ws_team_bytes() + a.n_planes * 32) return LHN_EWORKSPACE;
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  a.ticket = reinterpret_cast<unsigned int*>(ws);
  a.team_sums = reinterpret_cast<double*>(ws + kWsHeader);
  a.sums_out = sums; a.loss_out = loss; a.loss_scale = loss_scale; a.sum_reduction = sum_reduction;
  int used_team_kernel = 0;
  double* fallback_partials = partials ? partials : reinterpret_cast<double*>(ws + kWsHeader + ws_team_bytes());
  a.fallback_partials = fallback_partials;
  rc = fill_exchange(a, xch);
  if (rc) return rc;
  rc = run_heatmap(a, dtype, (cudaStream_t)stream, &used_team_kernel);
  if (rc || used_team_kernel) return rc;
  if (xch && xch->world > 1) return LHN_EINVAL;      // the in-kernel exchange lives in the team kernel only
  // CTA-per-plane fallback wrote per-plane partials: reduce + finalise as separate launches
  double* tmp_sums = sums ? sums : reinterpret_cast<double*>(ws + kWsHeader);
  rc = lhn_loss_reduce(fallback_partials, a.n_planes, tmp_sums, 0, stream);
  if (rc) return rc;
  if (loss) rc = lhn_loss_finalize(tmp_sums, a.loss_mode, sum_reduction, loss_scale, loss, a.loss_accumulate, stream);
  return rc;
}

static int decode_heatmap_pck_impl(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                   int64_t stride_b, int64_t stride_c, const float* center,
                                   const float* scale, const lhn_decode_params* dp, float* out_hm,
                                   float* out_kpts, int32_t* out_idx, const float* gt,
                                   const uint8_t* mask, const float* bbox_wh, float pck_thr,
                                   float auc_nor, int auc_steps, int64_t* counters, int64_t* totals,
                                   const lhn_exchange* xch, lhn_stream_t stream);

extern "C" int lhn_decode_heatmap_pck(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                      int64_t stride_b, int64_t stride_c, const float* center,
                                      const float* scale, const lhn_decode_params* dp, float* out_hm,
                                      float* out_kpts, int32_t* out_idx, const float* gt,
                                      const uint8_t* mask, const float* bbox_wh, float pck_thr,
                                      float auc_nor, int auc_steps, int64_t* counters,
                                      lhn_stream_t stream) {
  return decode_heatmap_pck_impl(hm, dtype, B, K, H, W, stride_b, stride_c, center, scale, dp, out_hm, out_kpts, out_idx,
                                 gt, mask, bbox_wh, pck_thr, auc_nor, auc_steps, counters, nullptr, nullptr, stream);
}

extern "C" int lhn_decode_heatmap_pck_xch(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                          int64_t stride_b, int64_t stride_c, const float* center,
                                          const float* scale, const lhn_decode_params* dp, float* out_hm,
                                          float* out_kpts, int32_t* out_idx, const float* gt,
                                          const uint8_t* mask, const float* bbox_wh, float pck_thr,
                                          float auc_nor, int auc_steps, int64_t* counters, int64_t* totals,
                                          const lhn_exchange* xch, lhn_stream_t stream) {
  if (!totals || !xch) return LHN_EINVAL;
  if ((int64_t)(auc_steps + 5) * K * 8 > LHN_XCH_PAYLOAD_BYTES) return LHN_EINVAL;
  return decode_heatmap_pck_impl(hm, dtype, B, K, H, W, stride_b, stride_c, center, scale, dp, out_hm, out_kpts, out_idx,
                                 gt, mask, bbox_wh, pck_thr, auc_nor, auc_steps, counters, totals, xch, stream);
}

static int decode_heatmap_pck_impl(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                   int64_t stride_b, int64_t stride_c, const float* center,
                                   const float* scale, const lhn_decode_params* dp, float* out_hm,
                                   float* out_kpts, int32_t* out_idx, const float* gt,
                                   const uint8_t* mask, const float* bbox_wh, float pck_thr,
                                   float auc_nor, int auc_steps, int64_t* counters, int64_t* totals,
                                   const lhn_exchange* xch, lhn_stream_t stream) {
  if (B < 0 || K <= 0 || H <= 0 || W <= 0 || auc_steps < 0 || !(auc_nor > 0.f)) return LHN_EINVAL;
  if (B == 0) return LHN_OK;
  if (!hm || !gt || !mask || !bbox_wh || !counters) return LHN_EINVAL;
  HmArgs a{};
  a.hm = hm; a.stride_b = stride_b; a.stride_c = stride_c;
  a.C = K; a.K = K; a.H = H; a.W = W; a.HW = H * W; a.n_planes = B * K;
  a.center = center; a.scale = scale;
  a.out_hm = out_hm; a.out_kpts = out_kpts; a.out_idx = out_idx;
  int rc = fill_decode(a, dp);
  if (rc) return rc;
  a.loss_mode = LHN_LOSS_NONE;
  a.gt = gt; a.mask = mask; a.bbox_wh = bbox_wh; a.pck_thr = pck_thr; a.auc_nor = auc_nor;
  a.auc_steps = auc_steps; a.counters = counters;
  if (auc_steps > 64) return LHN_EINVAL;
  for (int t = 0; t < auc_steps; ++t) a.auc_thr[t] = (float)(1.0 * t / auc_steps);
  if (a.n_planes == 0) return LHN_OK;
  if (a.n_planes > 0x7fffffffLL) return LHN_EINVAL;
  if (!xch) return run_heatmap(a, dtype, (cudaStream_t)stream);
  rc = fill_exchange(a, xch);
  if (rc) return rc;
  a.xch_totals = reinterpret_cast<long long*>(totals);
  int used_team_kernel = 0;
  rc = run_heatmap(a, dtype, (cudaStream_t)stream, &used_team_kernel);
  if (rc) return rc;
  return used_team_kernel ? LHN_OK : LHN_EINVAL;   // the in-kernel exchange lives in the team kernel only
}
