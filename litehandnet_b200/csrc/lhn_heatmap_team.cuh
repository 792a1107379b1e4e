// K1 (primary) — persistent fused heatmap kernel: sweeper warps + a lagging epilogue warp per TEAM.
//
// One CTA per SM, cut into teams of TW warps; every team owns a private stage (plane [+ flipped plane])
// filled by TMA bulk copies, and works as a two-stage pipeline with no CTA-wide barrier:
//
//   SWEEPERS (TW-1 warps)  wait for the stage's mbarrier; make ONE sweep over the plane (flip average,
//       Gaussian target + squared error as packed f32x2 FMAs, running NaN-propagating 3-input max; 128-bit
//       conflict-free shared-memory reads); combine the per-warp partials; resolve the argmax; compute the
//       DARK row sums around it straight from the stage; sum the loss "positives"; write a small plane
//       record; RELEASE the stage by re-arming it with the TMA load of the team's next plane; and, while
//       that load is in flight, evaluate the next plane's render parameters and Gaussian tables and run the
//       side-input ring (joints / visibility / center / scale prefetched four planes ahead with cp.async).
//   EPILOGUE warp (1 warp)  lags up to two planes behind on double-buffered records: column pass of the
//       blur, log, Taylor step, back-transform, stores, loss partial sums, PCK/AUC/EPE counters; at the end
//       it publishes the team's loss sums and the last team to finish reduces them in a fixed order and
//       finalises the loss (one launch per step, bitwise reproducible).
//
// The two sides hand records over through a full/empty mbarrier pair per buffer, so the latency-bound
// scalar epilogue (~4k cycles) overlaps the next plane's load and sweep instead of serialising with them.
// The rare exact-emulation path of DARK (1e-10 clamp reachable) re-reads the plane from global memory (L2).
#pragma once
#include <math.h>
#include <stdlib.h>

#include "lhn_heatmap.cuh"
#include "lhn_exchange.cuh"

namespace lhn {

constexpr int kMaxWarpsPerCta = 24;
constexpr int kMaxTeams = kMaxTeamsPerCta;

__device__ __forceinline__ void named_sync(int id, int nthreads) {
  if (nthreads == 32) { __syncwarp(); return; }      // a one-warp team needs no barrier unit
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- sm_100a packed-f32x2 / 3-input max / f32 warp-reduce primitives -------------------------------
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {   // FFMA2: 2 x fma.rn
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t fmul2(uint64_t a, uint64_t b) {               // FMUL2: 2 x mul.rn
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ float fmax3_nan(float a, float b, float c) {           // FMNMX3.NAN
  float d;
  asm("max.NaN.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ float redux_max_nan(float v) {                         // CREDUX.MAX.F32.NAN
  float d;
  asm volatile("redux.sync.max.NaN.f32 %0, %1, 0xffffffff;" : "=f"(d) : "f"(v));
  return d;
}
__device__ __forceinline__ void cp_async_4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// Phase timestamps for profiles/probes/trace_run.py (build with LHN_TRACE=1; compiled out otherwise).
// slots 0-5: first sweeper warp (S1 passed, plane landed, sweep done, S2 passed, staged, released);
// slots 8-11: epilogue warp (record received, blur/check done, Taylor done, plane finished).
#ifdef LHN_TRACE
static __device__ long long g_trace[148 * 12 * 16 * 16];
#define TRS(slot) do { if (role == 1 && lane == 0 && n_it < 16 && nteams <= 12) g_trace[((blockIdx.x * 12 + team) * 16 + n_it) * 16 + (slot)] = clock64(); } while (0)
#define TRE(slot) do { if (lane == 0 && n_it < 16 && nteams <= 12) g_trace[((blockIdx.x * 12 + team) * 16 + n_it) * 16 + (slot)] = clock64(); } while (0)
#else
#define TRS(slot) do { } while (0)
#define TRE(slot) do { } while (0)
#endif

// Record handed from the sweepers to the epilogue warp (double-buffered).
struct PlaneRec {
  uint32_t idx;               // first-maximal flat index
  float maxval;
  float rx, ry;               // coordinates after masking and the +-0.25 rules (DARK adds its offset later)
  float w;                    // target weight after the visibility rule
  float ssum;                 // sum of (output - target)^2 over the plane
  float spos;                 // ... over the positives (target > value)
  int npos;
  int flags;                  // bit 0: DARK guard passed, bit 1: a NaN was found, bits 8-9: window offset in its first quad
  int pad[3];
};

// per-team header at the start of the aux region
struct TeamHeader {
  uint64_t bar[4];            // TMA completion barriers of the stages
  uint64_t full[2];           // record n is complete          (sweepers -> epilogue warp)
  uint64_t empty[2];          // record/row-sum buffer is free (epilogue warp -> sweepers)
  uint32_t cta_done;          // team 0's header only: teams of this CTA that have published `tsum`
  uint32_t pad;
  double tsum[4];             // one-launch loss: this team's (S_pos, S_neg, N_pos, numel)
  float red_max[8];           // per-warp sweep partials: max (NaN-propagating), first quad holding it, sum
  uint32_t red_q[8];
  float red_s[8];
  // render parameters of the three table buffers (written by the epilogue warp two planes ahead)
  float w[3];
  float mx[3], my[3];
  int render_on[3];
  PlaneRec rec[2];
  // Per-plane side inputs (joint x/y, visibility, center, scale, gt x/y, bbox w/h), prefetched
  // kSideAhead planes ahead (two full plane periods before their first use) with 4-byte cp.async: under
  // a saturated memory system a plain global load costs microseconds, which must never sit on a team's
  // critical path.
  float side[8][12];
};
constexpr int kSideAhead = 4;
// Overlapped launches: team 0's epilogue warp lets the successor grid in after its third plane, or half-way through
// its planes in the exchanging variants (a.trigger_halfway; see the kernel).
// SD_MASK: the aligned 32-bit word that holds the plane's fused-metrics mask byte (cp.async moves >= 4 bytes)
enum { SD_JX = 0, SD_JY, SD_VIS, SD_CX, SD_CY, SD_SX, SD_SY, SD_GX, SD_GY, SD_BW, SD_BH, SD_MASK, SD_N };

template <typename T>
__device__ __forceinline__ float elem_f32(const T* p, int i) { return Elem<T>::to_f32(p[i]); }

// quads per row of the DARK tile: the (ksize+4)-wide window starts 0..3 columns into its first quad
__host__ __device__ constexpr int tile_quads(int td) { return (td + 6) >> 2; }

// WC:  compile-time square plane size (64 or 56: 89 of the reference's 108 configs) with a compile-time team
//      size (TWC warps = TWC-1 sweepers + 1 epilogue), so the sweep is a fully unrolled 128-bit loop with a
//      loop-invariant column quad per thread and immediate address offsets; 0 = run-time H, W and team size.
// KS:  DARK Gaussian size known at compile time (11: the Gen-2 decoder) or 0 = run-time size.
template <typename T, int WC, int TWC, bool FLIP, bool LOSS, int KS>
__global__ void __launch_bounds__(kMaxWarpsPerCta * 32, 1)
heatmap_team_kernel(const __grid_constant__ HmArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr bool FAST = WC > 0;
  const int H = FAST ? WC : a.H, W = FAST ? WC : a.W, HW = FAST ? WC * WC : a.HW;
  const int TW = FAST ? TWC : a.team_warps;          // warps per team
  const int NS = TW - 1;                             // sweeper warps
  const int ST = NS * 32;                            // sweeper threads
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int team = warp / TW, wt = warp - team * TW; // team in CTA, warp in team
  const int nteams = (blockDim.x >> 5) / TW;
  const int bar_id = 1 + team;                       // named barrier of this team's sweepers
  // Courier CTA of the exchanging launches (a.xch_courier: the grid's last CTA, on the one SM the host left without a
  // plane-carrying CTA).  It owns no planes: once the previous launch has completed it adds the block of two launches
  // back (all ranks' copies are in the mailbox by then) into the totals and sends the previous launch's block to the
  // peers.  On a plane-carrying CTA the same ~7 us held that CTA's SM, the successor grid's CTA there started late and,
  // the plane assignment being static, finished last: the delay was paid on every step (0.79 efficiency at 8 GPUs).
  const uint32_t wctas = gridDim.x - (uint32_t)a.xch_courier;      // plane-carrying CTAs
  if (a.xch_courier && blockIdx.x == wctas) {
    asm volatile("griddepcontrol.launch_dependents;");             // the plane-carrying CTAs pace the successor grid
    if (warp == 0 && (a.xch_prev_block || a.xch_prev2_block)) {
      const int n_blk = (a.auc_steps + 5) * a.K;
      asm volatile("griddepcontrol.wait;" ::: "memory");           // the previous launch is complete: its block is final
      if (a.xch_prev2_block) xch_consume_block_i64(a.xch, a.xch_prev2_seq, a.xch_prev2_block, n_blk, a.xch_totals, lane, smem_raw);
      __syncwarp();
      if (a.xch_prev_block && a.xch.world > 1)
        xch_publish(a.xch, a.xch_prev_seq, a.xch_prev_block, n_blk, lane, reinterpret_cast<unsigned long long*>(smem_raw));
    }
    return;
  }
  // Roles rotate over the warps of a team so that the epilogue warps of the CTA's teams are spread over
  // the four SM sub-partitions (warp w issues on SMSP w % 4): role 0 = epilogue, roles 1..TW-1 = sweepers.
  const int ew = (TW >= 4 ? team : (team >> 1)) % TW;
  const int role = (wt - ew + TW) % TW;
  const int sl = (role - 1) * 32 + lane;             // sweeper thread index (role >= 1)

  // ---- this team's private shared memory ----------------------------------------------------------
  unsigned char* tbase = smem_raw + (size_t)team * a.warp_smem;
  const int nstg = a.stages;                         // stages per team (1, 2 or 4): plane n lives in stage n % nstg
  unsigned char* aux = tbase + (size_t)nstg * a.stage_bytes;
  TeamHeader* th = reinterpret_cast<TeamHeader*>(aux);
  const size_t tab_bytes = align_up((size_t)(W + H) * 4, 16);
  float* tab0 = reinterpret_cast<float*>(aux + align_up(sizeof(TeamHeader), 16));   // two table buffers
  const int ksize = KS > 0 ? KS : a.ksize;
  const int TD = KS > 0 ? KS + 4 : a.tile_dim;       // DARK window side
  const int bb = (ksize - 1) >> 1;
  const int NQ = tile_quads(TD), TCW = 4 * NQ;       // DARK tile row = NQ quads
  const size_t tile_bytes = align_up((size_t)TD * TCW * 4, 16);
  unsigned char* tile0 = reinterpret_cast<unsigned char*>(tab0) + 3 * tab_bytes;        // two DARK tiles
  double* hbuf = reinterpret_cast<double*>(tile0 + 2 * tile_bytes);                     // row sums (epilogue warp)
  float* hout = reinterpret_cast<float*>(hbuf + (size_t)TD * 5);
  int* fidx = reinterpret_cast<int*>(hout + 32);     // this team's copy of flip_index[K]

  const uint32_t total_teams = wctas * nteams;
  // team-major numbering: the n_planes % total_teams leftover planes spread over all SMs instead of the first few
  const uint32_t gteam = team * wctas + blockIdx.x;
  const uint32_t n_planes = (uint32_t)a.n_planes;
  const uint32_t plane_bytes = (uint32_t)HW * sizeof(T);
  const uint32_t C = (uint32_t)a.C, K = (uint32_t)a.K;
  // plane -> (batch, channel) is advanced incrementally: no division in the loop
  const uint32_t step_b = total_teams / C, step_c = total_teams - step_b * C;

  auto split_channel = [&](uint32_t c, uint32_t& s, uint32_t& k) {
    if (C == K) { s = 0; k = c; } else { s = c / K; k = c - s * K; }
  };
  auto advance = [&](uint32_t& b, uint32_t& c) {
    b += step_b; c += step_c;
    if (c >= C) { c -= C; b += 1; }
  };
  auto gptr0 = [&](uint32_t b, uint32_t c) {
    return reinterpret_cast<const T*>(a.hm) + (int64_t)b * a.stride_b + (int64_t)c * a.stride_c;
  };
  auto gptr1 = [&](uint32_t b, uint32_t c) {
    uint32_t s, k;
    split_channel(c, s, k);
    const uint32_t kf = a.flip_index ? (uint32_t)fidx[k] : k;
    return reinterpret_cast<const T*>(a.hm_flip) + (int64_t)b * a.fstride_b + (int64_t)(s * K + kf) * a.fstride_c;
  };
  // KS > 0 is only instantiated for LHN_REFINE_DARK (the Gen-2 decoder): the other refinements, and the fused
  // metrics when a loss is fused (never together through the C ABI), are compiled out of those kernels — the
  // instruction footprint matters: 24 warps in different phases share a 32 KB L1.5 instruction cache.
  const bool is_dark = KS > 0 ? true : ((a.refine == LHN_REFINE_DARK) || (a.refine == LHN_REFINE_DARK_LEGACY));
  const bool legacy = KS > 0 ? false : (a.refine == LHN_REFINE_DARK_LEGACY);
  const bool udp = KS > 0 ? false : (a.refine == LHN_REFINE_DARK_UDP);   // post_dark_udp (top_down_eval.py:274-335)
  const bool has_counters = LOSS ? false : (a.counters != nullptr);

  // Side inputs of plane (b, c) -> ring slot `slot` (lanes 0..SD_N-1 of one warp; asynchronous).
  auto side_fetch = [&](uint32_t b, uint32_t c, int slot) {
    uint32_t s, k;
    split_channel(c, s, k);
    const int64_t bk = (int64_t)b * K + k;
    const float* src = nullptr;
    switch (lane) {
      case SD_JX: case SD_JY: if (LOSS) src = a.joints + bk * a.joints_stride + lane; break;
      case SD_VIS: if (LOSS) src = a.vis + bk * a.vis_stride; break;
      case SD_CX: case SD_CY: if (a.center) src = a.center + 2 * (int64_t)b + (lane - SD_CX); break;
      case SD_SX: case SD_SY: if (a.scale) src = a.scale + 2 * (int64_t)b + (lane - SD_SX); break;
      case SD_GX: case SD_GY: if (has_counters) src = a.gt + 2 * bk + (lane - SD_GX); break;
      case SD_BW: case SD_BH: if (has_counters) src = a.bbox_wh + 2 * (int64_t)b + (lane - SD_BW); break;
      case SD_MASK:
        if (has_counters) src = reinterpret_cast<const float*>(reinterpret_cast<uintptr_t>(a.mask + bk) & ~(uintptr_t)3);
        break;
      default: break;
    }
    if (src) cp_async_4(&th->side[slot][lane], src);
  };

  uint32_t p = gteam;
  uint32_t pb = p / C, pc = p - pb * C;            // the only division: once per team
  // The epilogue warp requests the side inputs of its first two planes before anything else: issued ahead of
  // the CTA's first bulk loads they return in ~1 us; queued behind 29 MB of plane traffic they take 5 us.
  uint32_t qb = pb, qc = pc, pq = p;               // cursor of the next plane to fetch (epilogue warp)
  if (role == 0) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      if (pq < n_planes) side_fetch(qb, qc, i);
      cp_async_commit();
      pq += total_teams; advance(qb, qc);
    }
  }

  // Fused metrics: one CTA-shared set of u64 counters in shared memory (same layout as the global ones, with
  // the AUC rows holding a histogram of "thresholds passed"), flushed once by the last epilogue warp of the CTA.
  unsigned long long* cta_cnt = reinterpret_cast<unsigned long long*>(smem_raw + (size_t)nteams * a.warp_smem);
  const int n_cnt = (!LOSS && a.counters) ? (a.auc_steps + 5) * (int)K : 0;
  unsigned int* cta_done = reinterpret_cast<unsigned int*>(cta_cnt + n_cnt);
  for (int i = threadIdx.x; i < n_cnt; i += blockDim.x) cta_cnt[i] = 0ull;
  if (threadIdx.x == 0 && !LOSS && a.counters) *cta_done = 0u;

  // Programmatic dependent launch.  A launch WITHOUT the overlap flag is ordered after everything before it on
  // the stream (a normal launch), so it lets its successor in at once.  A launch WITH the flag (promise: it
  // shares no buffer with the launch just before it) must not let ITS successor in before the launch two back
  // has completed: with two rotating buffer sets that one writes the successor's outputs, and small grids
  // (n_planes < SMs, spare SMs, little shared memory) could otherwise be co-resident three deep.  So in an
  // overlapped launch only the epilogue warp of team 0 triggers, after griddepcontrol.wait (= the predecessor
  // grid has completed and its writes are visible), a few planes into its loop — by then the predecessor is
  // long gone, and with one CTA per SM the successor cannot get an SM before this CTA retires anyway, so the
  // late trigger costs nothing.  Net contract: an overlapped launch runs after everything but its predecessor.
  if (!a.overlap_previous) asm volatile("griddepcontrol.launch_dependents;");

  // ---- one-time setup: barriers visible to the whole CTA before anybody waits on them ------------------
  if (wt == 0 && lane == 0) {
    for (int i = 0; i < nstg; ++i) mbar_init(&th->bar[i], 1);
    mbar_init(&th->full[0], 1); mbar_init(&th->full[1], 1);
    mbar_init(&th->empty[0], 1); mbar_init(&th->empty[1], 1);
    th->cta_done = 0u;
    fence_mbar_init();
  }
  __syncthreads();
#ifdef LHN_TRACE
  if (role == 1 && lane == 0 && nteams <= 12) {
    g_trace[((blockIdx.x * 12 + team) * 16 + 0) * 16 + 15] = clock64();
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    g_trace[((blockIdx.x * 12 + team) * 16 + 0) * 16 + 13] = (long long)gt;
  }
#endif
  if (p >= n_planes) return;                       // whole teams leave together

  // Render parameters + separable Gaussian factors of a plane (channel c, side-ring slot `slot`) into table
  // buffer `buf`, computed by `nthr` threads (thread index `t`).  exp() is evaluated on an f64 argument.
  auto prologue = [&](uint32_t c, int slot, int buf, int t, int nthr) {
    if (!LOSS) return;
    uint32_t s, k;
    split_channel(c, s, k);
    const float* sd = th->side[slot];
    const RenderGeom g = render_geom(sd[SD_JX], sd[SD_JY], sd[SD_VIS], (double)a.sigma[s], a.unbiased, a.feat_x, a.feat_y,
                                     a.feat_pow2, a.inv_feat_x, a.inv_feat_y, W, H);
    const bool render_on = g.on;
    if (t == 0) {
      th->w[buf] = g.w; th->mx[buf] = g.cx; th->my[buf] = g.cy; th->render_on[buf] = render_on ? 1 : 0;
    }
    const double i2 = a.inv2s2[s];
    float* tab = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(tab0) + (size_t)buf * tab_bytes);
    auto entry = [&](int i) -> float { return table_entry(g, i, W, a.unbiased, i2); };
    // four independent f64 chains per thread at a time: the loop is latency-bound, not throughput-bound
    const int n = W + H;
    int i0 = t;
    for (; i0 + 3 * nthr < n; i0 += 4 * nthr) {
      const float v0 = entry(i0), v1 = entry(i0 + nthr), v2 = entry(i0 + 2 * nthr), v3 = entry(i0 + 3 * nthr);
      tab[i0] = v0; tab[i0 + nthr] = v1; tab[i0 + 2 * nthr] = v2; tab[i0 + 3 * nthr] = v3;
    }
    for (; i0 < n; i0 += nthr) tab[i0] = entry(i0);
  };

  if (role == 0) {
    // =====================================================================================================
    // EPILOGUE WARP
    // =====================================================================================================
    double acc_sp = 0.0, acc_sn = 0.0, acc_np = 0.0, acc_ne = 0.0;   // this team's loss sums (lane 0)
    // side-input ring (kSideAhead planes ahead) and the tables of the first two planes; the sweepers start
    // on plane 0 as soon as its tables exist
#pragma unroll
    for (int i = 2; i < kSideAhead; ++i) {
      if (pq < n_planes) side_fetch(qb, qc, i);
      cp_async_commit();
      pq += total_teams; advance(qb, qc);
    }
    if (!LOSS) {
      // decode only: the sweepers need nothing from the side inputs (the epilogue does, for the back-transform), so
      // both record buffers are handed over at once — on a one-wave launch (BASELINE config 1: 64 samples) the
      // side-input round trip (~1.5 us cold) would otherwise sit in front of the first sweep
      if (lane == 0) { mbar_arrive(&th->empty[0]); mbar_arrive(&th->empty[1]); }
      cp_async_wait<kSideAhead - 2>();
      __syncwarp();
    } else {
      cp_async_wait<kSideAhead - 2>();               // the first two planes' side inputs have landed
      __syncwarp();
      if (!a.sweeper_tables) prologue(pc, 0, 0, lane, 32);
      __syncwarp();
      if (lane == 0) mbar_arrive(&th->empty[0]);
      if (!a.sweeper_tables && p + total_teams < n_planes) {
        uint32_t nb = pb, nc = pc;
        advance(nb, nc);
        prologue(nc, 1, 1, lane, 32);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&th->empty[1]);
    }

    int n_it = 0;
    // planes of this team: p, p + total_teams, ... < n_planes; the successor grid is let in after plane kTrig of team 0
    // plane 2 for plain launches (measured best: the earlier the successor grid is staged the better); half-way
    // for exchanging launches (measured at N = 8 on one box: 0.0515 ms per step half-way against 0.0540 early for the
    // counter exchange — the predecessor's completion includes its exchange and needs the slack)
    const int n_mine = (int)((n_planes - 1u - p) / total_teams + 1u);
    const int kTrig = a.trigger_halfway ? (n_mine >> 1) : (n_mine > a.trigger_plane ? a.trigger_plane : n_mine - 1);
    for (; p < n_planes; p += total_teams, ++n_it, advance(pb, pc)) {
      const int buf = n_it & 1;
      mbar_wait(&th->full[buf], (uint32_t)(n_it >> 1) & 1u);
      TRE(8);
      const PlaneRec* rec = &th->rec[buf];
      const uint32_t idx = rec->idx;
      const float maxval = rec->maxval;
      float rx = rec->rx, ry = rec->ry;
      float keepX = 0.f, keepY = 0.f;                  // image-space coordinates of this plane (lane 0)
      const bool dark_guard = (rec->flags & 1) != 0, any_nan = (rec->flags & 2) != 0;

      bool need_slow = false;
      float bmax = 0.f;
      if (dark_guard) {
        // row pass over the staged window (sequential FMA over the taps), then column pass (centre tap,
        // then symmetric pairs fused-added) — the summation order of cv2's separable filter
        const float* tile = reinterpret_cast<const float*>(tile0 + (size_t)buf * tile_bytes);
        const int xo = (rec->flags >> 8) & 3;
        if (legacy) {
          for (int e = lane; e < TD * 5; e += 32) {
            const int r = e / 5, c5 = e - r * 5;
            const float* trow = tile + r * TCW + xo + c5;
            double acc = 0.0;
            for (int j = 0; j < ksize; ++j) acc = __fma_rn(a.tapsd[j], (double)trow[j], acc);
            hbuf[e] = acc;
          }
          __syncwarp();
          if (lane < 25) {
            const int dr = lane / 5, c5 = lane - dr * 5;
            double acc = __dmul_rn(a.tapsd[bb], hbuf[(dr + bb) * 5 + c5]);
            for (int j = 1; j <= bb; ++j)
              acc = __fma_rn(a.tapsd[bb + j], __dadd_rn(hbuf[(dr + bb + j) * 5 + c5], hbuf[(dr + bb - j) * 5 + c5]), acc);
            hout[lane] = (float)acc;
          }
        } else {
          float* hb = reinterpret_cast<float*>(hbuf);
          if (KS > 0) {
            // (KS+4)*5 row sums over 32 lanes: the (up to 3) sums of a lane are independent FMA chains, interleaved
            constexpr int kN = (KS + 4) * 5, kPer = (kN + 31) / 32;
            float acc[kPer];
            const float* trow[kPer];
#pragma unroll
            for (int u = 0; u < kPer; ++u) {
              const int e = min(lane + 32 * u, kN - 1);
              const int r = e / 5, c5 = e - r * 5;
              trow[u] = tile + r * TCW + xo + c5;
              acc[u] = 0.f;
            }
#pragma unroll
            for (int j = 0; j < KS; ++j) {
#pragma unroll
              for (int u = 0; u < kPer; ++u) acc[u] = __fmaf_rn(a.tapsf[j], trow[u][j], acc[u]);   // taps: constant bank
            }
#pragma unroll
            for (int u = 0; u < kPer; ++u)
              if (lane + 32 * u < kN) hb[lane + 32 * u] = acc[u];
          } else {
            for (int e = lane; e < TD * 5; e += 32) {
              const int r = e / 5, c5 = e - r * 5;
              const float* trow = tile + r * TCW + xo + c5;
              float acc = 0.f;
              for (int j = 0; j < ksize; ++j) acc = __fmaf_rn(a.tapsf[j], trow[j], acc);
              hb[e] = acc;
            }
          }
          __syncwarp();
          if (lane < 25) {
            const int dr = lane / 5, c5 = lane - dr * 5;
            const float* hcol = hb + (dr + bb) * 5 + c5;
            float acc = __fmul_rn(a.tapsf[bb], hcol[0]);
            if (KS > 0) {
#pragma unroll
              for (int j = 1; j <= (KS - 1) / 2; ++j)
                acc = __fmaf_rn(a.tapsf[(KS - 1) / 2 + j], __fadd_rn(hcol[5 * j], hcol[-5 * j]), acc);
            } else {
              for (int j = 1; j <= bb; ++j) acc = __fmaf_rn(a.tapsf[bb + j], __fadd_rn(hcol[5 * j], hcol[-5 * j]), acc);
            }
            hout[lane] = acc;
          }
        }
        __syncwarp();
        if (udp) {
          // np.clip(., 0.001, 50) (NaN stays NaN), np.log
          float v = lane < 25 ? hout[lane] : 1.f;
          v = (v != v) ? v : fminf(fmaxf(v, 0.001f), 50.f);
          const float lv = logf(v);
          __syncwarp();
          if (lane < 25) hout[lane] = lv;
          __syncwarp();
        } else {
        // can the 1e-10 clamp of log() (or a non-finite value) touch the 13 stencil points?
        const float hv = lane < 25 ? hout[lane] : CUDART_INF_F;
        const int dr = lane / 5 - 2, dc = lane % 5 - 2;
        const bool used = lane < 25 && (abs(dr) + abs(dc) <= 2);
        const bool bad = used && !(hv >= 1e-9f);
        const bool ok_origin = legacy ? (maxval >= 1e-3f) : (maxval > 0.f);
        need_slow = __any_sync(0xffffffffu, bad) || !ok_origin || any_nan;
        if (need_slow) {
          // exact emulation: max of the whole blurred plane (NaN propagates like np.max).  The stage
          // belongs to the sweepers, so the decoded plane is re-read from global memory (L2-resident).
          const T* g0 = gptr0(pb, pc);
          const T* g1 = FLIP ? gptr1(pb, pc) : nullptr;
          auto gval = [&](int y, int x) -> float {
            float o = elem_f32<T>(g0, y * W + x);
            if (FLIP) o = __fmul_rn(__fadd_rn(o, elem_f32<T>(g1, y * W + (W - 1 - x))), 0.5f);
            return o;
          };
          float m = -CUDART_INF_F;
          bool first = true;
          for (int e = lane; e < HW; e += 32) {
            const int y = e / W, x = e - y * W;
            float v;
            if (legacy) {
              auto rowv = [&](int yy) {
                double r = 0.0;
                if (yy < 0 || yy >= H) return r;
                for (int j = 0; j < ksize; ++j) {
                  const int xx = x + j - bb;
                  r = __fma_rn(a.tapsd[j], (xx >= 0 && xx < W) ? (double)gval(yy, xx) : 0.0, r);
                }
                return r;
              };
              double acc = __dmul_rn(a.tapsd[bb], rowv(y));
              for (int j = 1; j <= bb; ++j) acc = __fma_rn(a.tapsd[bb + j], __dadd_rn(rowv(y + j), rowv(y - j)), acc);
              v = (float)acc;
            } else {
              auto rowv = [&](int yy) {
                float r = 0.f;
                if (yy < 0 || yy >= H) return r;
                for (int j = 0; j < ksize; ++j) {
                  const int xx = x + j - bb;
                  r = __fmaf_rn(a.tapsf[j], (xx >= 0 && xx < W) ? gval(yy, xx) : 0.f, r);
                }
                return r;
              };
              float acc = __fmul_rn(a.tapsf[bb], rowv(y));
              for (int j = 1; j <= bb; ++j) acc = __fmaf_rn(a.tapsf[bb + j], __fadd_rn(rowv(y + j), rowv(y - j)), acc);
              v = acc;
            }
            m = first ? v : nanmax(m, v);
            first = false;
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) m = nanmax(m, __shfl_xor_sync(0xffffffffu, m, o));
          bmax = m;
        }
        // log of the 25 blurred values in parallel, then the Taylor step on lane 0
        const float raw = lane < 25 ? hout[lane] : 1.f;
        float hval;
        if (need_slow) {
          const float sc = legacy ? __fdiv_rn(maxval, __fadd_rn(bmax, 1e-6f)) : __fdiv_rn(maxval, bmax);
          float v = __fmul_rn(raw, sc);
          v = (v != v) ? v : fmaxf(v, 1e-10f);          // np.maximum propagates NaN
          hval = logf(v);
        } else {
          hval = logf(raw);
        }
        __syncwarp();
        if (lane < 25) hout[lane] = hval;
        __syncwarp();
        }
      }
      // UDP, plane without a positive maximum (coordinates (-1, -1)): the reference's flat indexing into the
      // edge-padded batch reads i_, ix1, iy1, ix1y1 from this plane's pixel (0, 0) and ix1_, ix1_y1_, iy1_ from the
      // PREVIOUS plane's last row (the last plane's for plane 0).  Those three blurred values are computed here
      // from global memory (rare path); udp_deg = (own(0,0), prev(H-1,W-1), prev(H-1,0)).
      float udp_deg0 = 0.f, udp_deg1 = 0.f, udp_deg2 = 0.f;
      const bool udp_degenerate = udp && !dark_guard;
      if (udp_degenerate) {
        uint32_t qb2, qc2;
        if (p == 0) { qb2 = (uint32_t)((n_planes - 1) / C); qc2 = (n_planes - 1) - qb2 * C; }
        else if (pc == 0) { qb2 = pb - 1; qc2 = C - 1; }
        else { qb2 = pb; qc2 = pc - 1; }
        auto blur_at = [&](uint32_t bq, uint32_t cq, int y, int x) -> float {
          const T* g0 = gptr0(bq, cq);
          const T* g1 = FLIP ? gptr1(bq, cq) : nullptr;
          auto refl = [](int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); };
          // lanes 0..ksize-1: one window row each (sequential FMA over the taps), then the column pass on lane 0
          float rowv = 0.f;
          if (lane < ksize) {
            const int yy = refl(y + lane - bb, H);
            for (int j = 0; j < ksize; ++j) {
              const int xx = refl(x + j - bb, W);
              float o = elem_f32<T>(g0, yy * W + xx);
              if (FLIP) o = __fmul_rn(__fadd_rn(o, elem_f32<T>(g1, yy * W + (W - 1 - xx))), 0.5f);
              rowv = __fmaf_rn(a.tapsf[j], o, rowv);
            }
          }
          float acc = __fmul_rn(a.tapsf[bb], __shfl_sync(0xffffffffu, rowv, bb));
          for (int j = 1; j <= bb; ++j)
            acc = __fmaf_rn(a.tapsf[bb + j], __fadd_rn(__shfl_sync(0xffffffffu, rowv, bb + j),
                                                       __shfl_sync(0xffffffffu, rowv, bb - j)), acc);
          float v = (acc != acc) ? acc : fminf(fmaxf(acc, 0.001f), 50.f);
          return logf(v);
        };
        udp_deg0 = blur_at(pb, pc, 0, 0);
        udp_deg1 = blur_at(qb2, qc2, H - 1, W - 1);
        udp_deg2 = blur_at(qb2, qc2, H - 1, 0);
      }
      TRE(9);

      if (lane == 0) {
        if (udp) {
          // 3x3 stencil on the edge-padded log map: a neighbour beyond the plane is the border pixel itself
          const int px = (int)rx, py = (int)ry;
          auto LL = [&](int dy, int dx) -> float {
            const int yy = min(max(py + dy, 0), H - 1) - py, xx = min(max(px + dx, 0), W - 1) - px;
            return hout[(yy + 2) * 5 + xx + 2];
          };
          float i_, ix1, iy1, ix1y1, ix1_y1_, ix1_, iy1_;
          if (udp_degenerate) {
            i_ = ix1 = iy1 = ix1y1 = udp_deg0; ix1_y1_ = ix1_ = udp_deg1; iy1_ = udp_deg2;
          } else {
            i_ = LL(0, 0); ix1 = LL(0, 1); iy1 = LL(1, 0); ix1y1 = LL(1, 1);
            ix1_y1_ = LL(-1, -1); ix1_ = LL(0, -1); iy1_ = LL(-1, 0);
          }
          const float ddx = __fmul_rn(0.5f, __fsub_rn(ix1, ix1_));
          const float ddy = __fmul_rn(0.5f, __fsub_rn(iy1, iy1_));
          const float dxx = __fadd_rn(__fsub_rn(ix1, __fmul_rn(2.f, i_)), ix1_);
          const float dyy = __fadd_rn(__fsub_rn(iy1, __fmul_rn(2.f, i_)), iy1_);
          float t = __fsub_rn(ix1y1, ix1);
          t = __fsub_rn(t, iy1); t = __fadd_rn(t, i_); t = __fadd_rn(t, i_);
          t = __fsub_rn(t, ix1_); t = __fsub_rn(t, iy1_); t = __fadd_rn(t, ix1_y1_);
          const float dxy = __fmul_rn(0.5f, t);
          // (H + eps I)^-1 d in f64 (np.linalg.inv of the f64 matrix), coords (f32) -= that, rounded once
          const double eps = 1.1920928955078125e-07;
          const double ha = (double)dxx + eps, hd = (double)dyy + eps, hb = (double)dxy;
          const double det = __dsub_rn(__dmul_rn(ha, hd), __dmul_rn(hb, hb));
          const double ox = __dadd_rn(__dmul_rn(hd / det, (double)ddx), __dmul_rn(-hb / det, (double)ddy));
          const double oy = __dadd_rn(__dmul_rn(-hb / det, (double)ddx), __dmul_rn(ha / det, (double)ddy));
          rx = (float)((double)rx - ox); ry = (float)((double)ry - oy);
        } else if (dark_guard) {
#define HH(dy, dx) hout[((dy) + 2) * 5 + (dx) + 2]
          const float h00 = HH(0, 0);
          const float ddx = __fmul_rn(0.5f, __fsub_rn(HH(0, 1), HH(0, -1)));
          const float ddy = __fmul_rn(0.5f, __fsub_rn(HH(1, 0), HH(-1, 0)));
          const float dxx = __fmul_rn(0.25f, __fadd_rn(__fsub_rn(HH(0, 2), __fmul_rn(2.f, h00)), HH(0, -2)));
          const float dxy = __fmul_rn(0.25f, __fadd_rn(__fsub_rn(__fsub_rn(HH(1, 1), HH(-1, 1)), HH(1, -1)), HH(-1, -1)));
          const float dyy = __fmul_rn(0.25f, __fadd_rn(__fsub_rn(HH(2, 0), __fmul_rn(2.f, h00)), HH(-2, 0)));
#undef HH
          const float det = __fsub_rn(__fmul_rn(dxx, dyy), __fmul_rn(dxy, dxy));
          if (det != 0.f) {   // true for NaN, as in numpy
            const float ox = -__fdiv_rn(__fsub_rn(__fmul_rn(dyy, ddx), __fmul_rn(dxy, ddy)), det);
            const float oy = -__fdiv_rn(__fsub_rn(__fmul_rn(dxx, ddy), __fmul_rn(dxy, ddx)), det);
            rx = __fadd_rn(rx, ox); ry = __fadd_rn(ry, oy);
          }
        }
        TRE(10);
        // ---- back-transform (T1/T2) and stores --------------------------------------------------------
        uint32_t s, k;
        split_channel(pc, s, k);
        float X = rx, Y = ry;
        const float* sd = th->side[n_it & 7];
        if (a.transform == LHN_XFORM_CENTER_SCALE) {
          const float s0 = __fmul_rn(sd[SD_SX], 200.0f), s1 = __fmul_rn(sd[SD_SY], 200.0f);
          const float dw = a.use_udp ? (float)(W - 1) : (float)W, dh = a.use_udp ? (float)(H - 1) : (float)H;
          const float fx = __fdiv_rn(s0, dw), fy = __fdiv_rn(s1, dh);
          X = __fsub_rn(__fadd_rn(__fmul_rn(rx, fx), sd[SD_CX]), __fmul_rn(s0, 0.5f));
          Y = __fsub_rn(__fadd_rn(__fmul_rn(ry, fy), sd[SD_CY]), __fmul_rn(s1, 0.5f));
        } else if (a.transform == LHN_XFORM_SCALE) {
          X = __fmul_rn(rx, a.scale_x); Y = __fmul_rn(ry, a.scale_y);
        }
        if (a.out_hm) { float* o = a.out_hm + 3 * (int64_t)p; o[0] = rx; o[1] = ry; o[2] = maxval; }
        if (a.out_kpts) { float* o = a.out_kpts + 3 * (int64_t)p; o[0] = X; o[1] = Y; o[2] = maxval; }
        if (a.out_idx) a.out_idx[p] = (int32_t)idx;
        if (LOSS) {
          const float w = th->w[n_it % 3];
          const bool bal = a.loss_mode == LHN_LOSS_DISTANCE_BALANCE;
          const float wp = (a.loss_mode == LHN_LOSS_JOINTS_MSE) ? w * w : w;
          const double sall = (double)rec->ssum * (double)wp, spos = bal ? (double)rec->spos * (double)wp : 0.0;
          const double npos = bal ? (double)rec->npos : 0.0;
          if (a.partials) {
            *reinterpret_cast<double2*>(a.partials + 4 * (int64_t)p) = make_double2(spos, sall - spos);
            *reinterpret_cast<double2*>(a.partials + 4 * (int64_t)p + 2) = make_double2(npos, (double)HW);
          }
          acc_sp += spos; acc_sn += sall - spos; acc_np += npos; acc_ne += (double)HW;
          if (a.out_weight) a.out_weight[p] = w;
        }
        keepX = X; keepY = Y;
      }
      if (has_counters) {
        // fused PCK / AUC / EPE counters (_calc_distances in f64, compared in f32): lanes 0..2 take one
        // normaliser each (bbox, AUC constant, 1) so the three divide / sqrt chains run side by side
        const float Xb = __shfl_sync(0xffffffffu, keepX, 0), Yb = __shfl_sync(0xffffffffu, keepY, 0);
        uint32_t s_, k;
        split_channel(pc, s_, k);
        const float* sd = th->side[n_it & 7];
        // the mask byte came with the side inputs (four planes ahead): a plain load here waits microseconds behind
        // the plane traffic, once per plane, on the epilogue warp's critical path
        const uintptr_t maddr = reinterpret_cast<uintptr_t>(a.mask + ((int64_t)pb * K + k));
        const uint32_t mk = (__float_as_uint(sd[SD_MASK]) >> (8u * (uint32_t)(maddr & 3))) & 0xffu;
        if (mk) {
          const int Ki = (int)K;
          const double ddx = (double)Xb - (double)sd[SD_GX], ddy = (double)Yb - (double)sd[SD_GY];
          double nb = lane == 0 ? (double)fmaxf(sd[SD_BW], sd[SD_BH]) : (lane == 1 ? (double)a.auc_nor : 1.0);
          const bool counted = nb != 0.0;                   // normalize == 0 masks the sample out (PCK only)
          if (nb < 0.0) nb = 1e6;
          float d = 0.f;
          if (lane < 3 && counted) {
            const double qx = lane == 2 ? ddx : ddx / nb, qy = lane == 2 ? ddy : ddy / nb;
            d = (float)sqrt(__dadd_rn(__dmul_rn(qx, qx), __dmul_rn(qy, qy)));
          }
          // AUC: one threshold per lane, ballot -> how many of the (increasing) thresholds d is below
          const float d_auc = __shfl_sync(0xffffffffu, d, 1);
          int nh = 0;
          for (int t0 = 0; t0 < a.auc_steps; t0 += 32) {
            const int t = t0 + lane;
            nh += __popc(__ballot_sync(0xffffffffu, t < a.auc_steps && d_auc < a.auc_thr[t]));
          }
          // Plane counts of one CTA stay far below 2^32: they are bumped with the native 32-bit shared-memory
          // atomic on the low word of the 64-bit slot (a 64-bit shared atomicAdd is a compare-and-swap loop);
          // only the fixed-point EPE sum needs the 64-bit add.
          auto bump = [&](unsigned long long* slot) { atomicAdd(reinterpret_cast<unsigned int*>(slot), 1u); };
          if (lane == 0 && counted) {
            bump(cta_cnt + Ki + k);
            if (d < a.pck_thr) bump(cta_cnt + k);
          } else if (lane == 1) {
            bump(cta_cnt + (int64_t)(2 + nh) * Ki + k);
          } else if (lane == 2) {
            unsigned long long* epe = cta_cnt + (int64_t)(3 + a.auc_steps) * Ki;
            bump(epe + k);
            atomicAdd(epe + Ki + k, epe_fix_term(d));
          }
        }
      }
      TRE(11);
      // ---- side-input ring + the tables of plane n+2; then plane n+2 may start ------------------------------
      if (pq < n_planes) side_fetch(qb, qc, (n_it + kSideAhead) & 7);
      cp_async_commit();
      pq += total_teams; advance(qb, qc);
      cp_async_wait<kSideAhead - 2>();               // side inputs of plane n+2 have landed
      __syncwarp();
      if (!a.sweeper_tables && p + 2 * total_teams < n_planes) {
        uint32_t nb = pb, nc = pc;
        advance(nb, nc); advance(nb, nc);
        prologue(nc, (n_it + 2) & 7, (n_it + 2) % 3, lane, 32);
      }
      TRE(12);
      __syncwarp();
      if (lane == 0) mbar_arrive(&th->empty[buf]);   // release: record/tile buffer free, tables of n+2 ready
      if (a.overlap_previous && team == 0 && n_it == kTrig) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;");
      }
    }
    if (a.overlap_previous && team == 0 && n_it <= kTrig) {   // a single plane: trigger at the end
      asm volatile("griddepcontrol.wait;" ::: "memory");
      asm volatile("griddepcontrol.launch_dependents;");
    }

    if (has_counters) {
      // the last epilogue warp of the CTA to finish adds the CTA's counters to the global ones
      __syncwarp();
      unsigned int last = 0;
      if (lane == 0) {
        unsigned int active = 0;
        for (int t = 0; t < nteams; ++t) active += ((uint64_t)t * wctas + blockIdx.x < n_planes) ? 1u : 0u;
        __threadfence_block();
        last = (atomicAdd(cta_done, 1u) == active - 1u) ? 1u : 0u;
      }
      if (__shfl_sync(0xffffffffu, last, 0)) {
        __threadfence_block();
        const int Ki = (int)K, steps = a.auc_steps;
        unsigned long long* gcnt = reinterpret_cast<unsigned long long*>(a.counters);
        // rows outside the AUC histogram map one to one
        for (int e = lane; e < n_cnt; e += 32) {
          const int row = e / Ki;
          if (row >= 2 && row <= 2 + steps) continue;
          const unsigned long long v = cta_cnt[e];
          if (v) atomicAdd(gcnt + e, v);
        }
        // AUC: one joint per lane, a running sum down the histogram: auc_hits[t] = planes that passed at least
        // steps - t thresholds, auc_valid = all planes
        for (int k = lane; k < Ki; k += 32) {
          unsigned long long run = 0ull;
          for (int nh = steps; nh >= 0; --nh) {
            run += cta_cnt[(int64_t)(2 + nh) * Ki + k];
            const int row = nh >= 1 ? 2 + (steps - nh) : 2 + steps;
            if (run) atomicAdd(gcnt + (int64_t)row * Ki + k, run);
          }
        }
        if (a.xch.world > 0 && !a.xch_courier) {
          // (Without a courier CTA — LHN_XCH_COURIER=0.)  In-kernel all-reduce of the per-step blocks (lhn_decode_heatmap_pck_xch), pipelined over two launches: the
          // first CTA of this grid to finish CONSUMES the block of two launches back (every rank sent it during the
          // previous launch, so nothing is waited for: adds the ranks' blocks in rank order into the running totals)
          // and PUBLISHES the previous launch's block to every peer.  The last CTA of the grid would be the natural
          // place for an immediate exchange, but whoever exchanges holds its SM for the NVLink round trip, the successor
          // grid's CTA on that SM then starts late and — the plane assignment being static — finishes last again:
          // measured, the step went from 42 to 70 us (profiles/r02_xch_timing.txt).  The first CTA to finish runs
          // ~13 us ahead of the last (the grid's finish-time spread): ~7 us of sends and local adds fit in that slack.
          __threadfence();
          __syncwarp();
          unsigned int tk = 0;
          if (lane == 0) tk = atomicAdd(xch_ticket(a.xch, a.xch_seq), 1u);
          tk = __shfl_sync(0xffffffffu, tk, 0);
          if (tk == 0 && (a.xch_prev_block || a.xch_prev2_block)) {
            asm volatile("griddepcontrol.wait;" ::: "memory");   // the previous launch is complete: its block is final
            // every team of this CTA has finished: the stages' shared memory is free scratch for the gather
            if (a.xch_prev2_block) xch_consume_block_i64(a.xch, a.xch_prev2_seq, a.xch_prev2_block, n_cnt, a.xch_totals, lane, smem_raw);
            if (a.xch_prev_block && a.xch.world > 1) xch_publish(a.xch, a.xch_prev_seq, a.xch_prev_block, n_cnt, lane, cta_cnt);
          }
          if (tk == wctas - 1 && lane == 0) *xch_ticket(a.xch, a.xch_seq) = 0u;
        }
      }
    }
#ifdef LHN_TRACE
    if (lane == 0 && nteams <= 12) {
      g_trace[((blockIdx.x * 12 + team) * 16 + 0) * 16 + 14] = clock64();
      unsigned long long gt;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
      g_trace[((blockIdx.x * 12 + team) * 16 + 1) * 16 + 13] = (long long)gt;
    }
#endif
    // ---- one-launch loss: two fixed-order levels.  A team leaves its sums in shared memory; the last team of the
    // CTA to finish adds the CTA's teams (team order) and publishes ONE row; the last CTA adds the rows (lane-strided,
    // then a fixed tree) and finalises.  The whole grid waits for that last warp: 148 rows are one L2 round trip
    // (a row per team was ~47 dependent round trips, 4-5 us per launch: profiles/r01_batch_scaling.txt).
    if (LOSS && a.team_sums) {
      // the workspace is shared with the previous launch on the stream: it must have completed (it has, long
      // ago; this only orders the memory operations when the launches overlap)
      asm volatile("griddepcontrol.wait;" ::: "memory");
      TeamHeader* th0 = reinterpret_cast<TeamHeader*>(smem_raw + (size_t)nstg * a.stage_bytes);   // team 0's header
      unsigned int last = 0;
      if (lane == 0) {
        th->tsum[0] = acc_sp; th->tsum[1] = acc_sn; th->tsum[2] = acc_np; th->tsum[3] = acc_ne;
        unsigned int cta_teams = 0;
        for (int t = 0; t < nteams; ++t) cta_teams += ((uint64_t)t * wctas + blockIdx.x < n_planes) ? 1u : 0u;
        __threadfence_block();
        last = (atomicAdd(&th0->cta_done, 1u) == cta_teams - 1u) ? 1u : 0u;
      }
      if (!__shfl_sync(0xffffffffu, last, 0)) return;
      unsigned int ticket = 0;
      if (lane == 0) {
        __threadfence_block();
        double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
        for (int t = 0; t < nteams; ++t) {
          if ((uint64_t)t * wctas + blockIdx.x >= n_planes) break;
          const TeamHeader* tt = reinterpret_cast<const TeamHeader*>(reinterpret_cast<const unsigned char*>(th0) +
                                                                     (size_t)t * a.warp_smem);
          c0 += tt->tsum[0]; c1 += tt->tsum[1]; c2 += tt->tsum[2]; c3 += tt->tsum[3];
        }
        double* dst = a.team_sums + 4 * (size_t)blockIdx.x;
        __stcg(reinterpret_cast<double2*>(dst), make_double2(c0, c1));
        __stcg(reinterpret_cast<double2*>(dst) + 1, make_double2(c2, c3));
        __threadfence();
        ticket = atomicAdd(a.ticket, 1u);
      }
      ticket = __shfl_sync(0xffffffffu, ticket, 0);
      if (ticket == wctas - 1) {                            // every CTA of the grid owns at least one plane
        __threadfence();
        double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
        for (uint32_t t0 = lane; t0 < wctas; t0 += 160) {   // five rows per lane in flight: 148 SMs in one trip
          double2 x[5], y[5];
#pragma unroll
          for (int u = 0; u < 5; ++u) {
            const uint32_t t = t0 + 32u * u;
            x[u] = y[u] = make_double2(0.0, 0.0);               // rows past the end add +0.0
            if (t < wctas) {
              x[u] = __ldcg(reinterpret_cast<const double2*>(a.team_sums + 4 * (size_t)t));
              y[u] = __ldcg(reinterpret_cast<const double2*>(a.team_sums + 4 * (size_t)t) + 1);
            }
          }
#pragma unroll
          for (int u = 0; u < 5; ++u) { v0 += x[u].x; v1 += x[u].y; v2 += y[u].x; v3 += y[u].y; }
        }
        v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2); v3 = warp_sum(v3);
        if (a.xch.world > 1) {
          // batch-global loss (lhn_fused_render_loss_decode_xch): all-gather the four sums of every rank through the
          // peer mailboxes and add them in rank order — the same doubles in the same order on every rank
          unsigned long long* mine = reinterpret_cast<unsigned long long*>(xch_slot(a.xch, a.xch_seq, a.xch.rank, a.xch.rank));
          if (lane == 0) {
            mine[0] = (unsigned long long)__double_as_longlong(v0); mine[1] = (unsigned long long)__double_as_longlong(v1);
            mine[2] = (unsigned long long)__double_as_longlong(v2); mine[3] = (unsigned long long)__double_as_longlong(v3);
          }
          __syncwarp();
          const bool ok = xch_publish_and_wait(a.xch, a.xch_seq, mine, 4, lane, nullptr);
          if (ok) {
            double g0 = 0.0, g1 = 0.0, g2 = 0.0, g3 = 0.0;
            for (int r = 0; r < a.xch.world; ++r) {
              const volatile unsigned long long* src = reinterpret_cast<const volatile unsigned long long*>(xch_slot(a.xch, a.xch_seq, a.xch.rank, r));
              g0 += __longlong_as_double((long long)src[0]); g1 += __longlong_as_double((long long)src[1]);
              g2 += __longlong_as_double((long long)src[2]); g3 += __longlong_as_double((long long)src[3]);
            }
            v0 = g0; v1 = g1; v2 = g2; v3 = g3;
          }
        }
        if (lane == 0) {
          if (a.sums_out) { a.sums_out[0] = v0; a.sums_out[1] = v1; a.sums_out[2] = v2; a.sums_out[3] = v3; }
          if (a.loss_out) {
            double v;
            if (a.loss_mode == LHN_LOSS_DISTANCE_BALANCE) v = 0.1 * v0 / (v2 + 1.0) + v1 / (v3 - v2 + 1.0);
            else if (a.loss_mode == LHN_LOSS_JOINTS_MSE) v = 0.5 * (v0 + v1) / v3;
            else v = (v0 + v1) / v3;
            if (a.sum_reduction) v *= v3;
            const float lv = (float)(v * (double)a.loss_scale);
            a.loss_out[0] = a.loss_accumulate ? a.loss_out[0] + lv : lv;
          }
          *a.ticket = 0u;                                       // leave the workspace ready for the next launch
        }
      }
    }
    return;
  }

  // =======================================================================================================
  // SWEEPERS
  // =======================================================================================================
  uint64_t policy = 0;
  auto issue = [&](uint32_t b, uint32_t c, int stg) {   // one thread of the team
    unsigned char* dst = tbase + (size_t)stg * a.stage_bytes;
    mbar_arrive_expect_tx(&th->bar[stg], FLIP ? 2 * plane_bytes : plane_bytes);
    tma_load_1d(dst, gptr0(b, c), plane_bytes, &th->bar[stg], policy);
    if (FLIP) tma_load_1d(dst + (a.stage_bytes >> 1), gptr1(b, c), plane_bytes, &th->bar[stg], policy);
  };

  if (a.flip_index) {
    for (int i = sl; i < (int)K; i += ST) fidx[i] = a.flip_index[i];
    named_sync(bar_id, ST);
  }
  if (sl == 0) {
    policy = policy_evict_first();
    if (a.use_tma) {
      // Stagger the first loads of the CTA's teams: issued all at once they also all land at once (~5 us for
      // the 29 MB first wave) and the teams then sweep in lockstep while HBM idles.
      if (a.stagger_ns > 0 && team > 0) __nanosleep((unsigned)(team * a.stagger_ns));
      uint32_t ib = pb, ic = pc, ip = p;
      for (int i = 0; i < nstg && ip < n_planes; ++i, ip += total_teams, advance(ib, ic)) issue(ib, ic, i);
    }
  }
  int n_it = 0;                                    // team-local plane counter

  const int QR = W >> 2, nq = HW >> 2;
  const uint64_t half2 = pack2(0.5f, 0.5f);

  for (; p < n_planes; p += total_teams, ++n_it, advance(pb, pc)) {
    const int buf = n_it & 1, tb = n_it % 3, stg = n_it & (nstg - 1);
    const T* plane0 = reinterpret_cast<const T*>(tbase + (size_t)stg * a.stage_bytes);
    const T* plane1 = FLIP ? reinterpret_cast<const T*>(tbase + (size_t)stg * a.stage_bytes + (a.stage_bytes >> 1)) : nullptr;
    // the epilogue warp has written this plane's tables and is done with the record/tile buffer `buf`
    // (it finished plane n-2; it lags at most two planes)
    mbar_wait(&th->empty[buf], (uint32_t)(n_it >> 1) & 1u);
    if (LOSS && a.sweeper_tables) {
      // multi-stage teams: the plane is usually resident already and the sweepers have slack, the epilogue warp
      // has none — so the sweepers evaluate this plane's tables (its side inputs were published with `empty`)
      prologue(pc, n_it & 7, tb, sl, ST);
      named_sync(bar_id, ST);
    }
    TRS(0);
    const float* ex = reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(tab0) + (size_t)tb * tab_bytes);
    const float* ey = ex + W;

    // ---- wait for the plane ------------------------------------------------------------------------
    if (a.use_tma) {
      mbar_wait(&th->bar[stg], (uint32_t)(n_it / nstg) & 1u);
    } else {
      const T* g0 = gptr0(pb, pc);
      T* d0 = const_cast<T*>(plane0);
      for (int e = sl; e < HW; e += ST) d0[e] = g0[e];
      if (FLIP) {
        const T* g1 = gptr1(pb, pc);
        T* d1 = const_cast<T*>(plane1);
        for (int e = sl; e < HW; e += ST) d1[e] = g1[e];
      }
      named_sync(bar_id, ST);
    }
    TRS(1);

    // decoded values (flip average) of quad q = row * QR + cq
    auto avg_quad = [&](const float4& o, const float4& f) -> float4 {
      uint64_t lo = fmul2(pack2(__fadd_rn(o.x, f.w), __fadd_rn(o.y, f.z)), half2);
      uint64_t hi = fmul2(pack2(__fadd_rn(o.z, f.y), __fadd_rn(o.w, f.x)), half2);
      float4 v;
      unpack2(lo, v.x, v.y); unpack2(hi, v.z, v.w);
      return v;
    };
    auto load_quad = [&](int q) -> float4 {
      const int row = FAST ? (q / (WC > 0 ? WC / 4 : 1)) : (q / QR);
      const int cq = q - row * QR;
      const float4 o = load4<T>(plane0 + row * W + 4 * cq);
      if (!FLIP) return o;
      return avg_quad(o, load4<T>(plane1 + row * W + (W - 4 - 4 * cq)));
    };
    auto val = [&](int y, int x) -> float {
      float o = elem_f32<T>(plane0, y * W + x);
      if (FLIP) o = __fmul_rn(__fadd_rn(o, elem_f32<T>(plane1, y * W + (W - 1 - x))), 0.5f);
      return o;
    };

    // ---- pass 1: one sweep, split over the sweepers ----------------------------------------------------
    uint64_t S2acc = 0;                      // packed (S0, S1) squared-error accumulators
    float best = -CUDART_INF_F;              // NaN-propagating running max of this thread
    int bq = -1;                             // first quad that raised it
    // po / pf: pointers to the quad of the plane and to its mirror quad of the flipped plane
    auto sweep_quad = [&](int q, const T* po, const T* pf, const float* pgy, uint64_t ngx01, uint64_t ngx23) {
      const float4 o = load4<T>(po);
      float4 v = o;
      if (FLIP) v = avg_quad(o, load4<T>(pf));
      if (LOSS) {
        const float gy = *pgy;
        const uint64_t gy2 = pack2(gy, gy);
        const uint64_t d01 = ffma2(ngx01, gy2, pack2(o.x, o.y));     // o - gx*gy
        const uint64_t d23 = ffma2(ngx23, gy2, pack2(o.z, o.w));
        S2acc = ffma2(d01, d01, S2acc);
        S2acc = ffma2(d23, d23, S2acc);
      }
      const float m3 = fmax3_nan(v.x, v.y, v.z);
      const float r = fmax3_nan(m3, v.w, best);
      if (r != best) bq = q;                 // strictly greater (or NaN: resolved by the NaN path)
      best = r;
    };
    if (FAST) {
      // The first kAST sweeper threads (a multiple of the quads per row) take part: the column quad of a thread
      // is loop-invariant and every address is base + compile-time offset.
      constexpr int kQR = (WC > 0 ? WC : 4) / 4, kNQ = kQR * (WC > 0 ? WC : 4);
      constexpr int kST = (TWC > 1 ? TWC - 1 : 1) * 32;
      constexpr int kAST = kST / kQR * kQR, kRPI = kAST / kQR;      // active threads, rows per iteration
      constexpr int kFull = kNQ / kAST, kRem = kNQ - kFull * kAST;
      if (sl < kAST) {
        const int srow = sl / kQR, scq = sl - srow * kQR;
        uint64_t ngx01 = 0, ngx23 = 0;
        if (LOSS) {
          const float4 gx = *reinterpret_cast<const float4*>(ex + 4 * scq);
          ngx01 = pack2(-gx.x, -gx.y); ngx23 = pack2(-gx.z, -gx.w);
        }
        const T* po = plane0 + 4 * sl;
        const T* pf = FLIP ? plane1 + srow * WC + (WC - 4) - 4 * scq : nullptr;
        const float* pgy = ey + srow;
#pragma unroll (kFull <= 16 ? kFull : 8)
        for (int it = 0; it < kFull; ++it)
          sweep_quad(it * kAST + sl, po + it * kAST * 4, pf + it * kAST * 4, pgy + it * kRPI, ngx01, ngx23);
        if (kRem > 0 && sl < kRem)
          sweep_quad(kFull * kAST + sl, po + kFull * kAST * 4, pf + kFull * kAST * 4, pgy + kFull * kRPI, ngx01, ngx23);
      }
    } else {
      for (int q = sl; q < nq; q += ST) {
        const int row = q / QR, cq = q - row * QR;
        uint64_t ngx01 = 0, ngx23 = 0;
        if (LOSS) {
          const float4 gx = *reinterpret_cast<const float4*>(ex + 4 * cq);
          ngx01 = pack2(-gx.x, -gx.y); ngx23 = pack2(-gx.z, -gx.w);
        }
        sweep_quad(q, plane0 + 4 * q, FLIP ? plane1 + row * W + (W - 4 - 4 * cq) : nullptr, ey + row, ngx01, ngx23);
      }
    }
    TRS(2);

    // ---- per-warp partials -> shared, S2 ----------------------------------------------------------------
    {
      const float wmax = redux_max_nan(best);
      const uint32_t cand = (best == wmax) ? (uint32_t)bq : 0xffffffffu;   // -1 -> 0xffffffff
      const uint32_t wq = __reduce_min_sync(0xffffffffu, cand);
      float ssum = 0.f;
      if (LOSS) {
        float s0, s1;
        unpack2(S2acc, s0, s1);
        ssum = warp_sum(s0 + s1);
      }
      if (lane == 0) { th->red_max[role - 1] = wmax; th->red_q[role - 1] = wq; th->red_s[role - 1] = ssum; }
    }
    named_sync(bar_id, ST);
    TRS(3);

    // ---- every sweeper warp: the team-wide argmax (redundantly: cheaper than another barrier) ------------
    const float tm = lane < NS ? th->red_max[lane] : -CUDART_INF_F;
    const float tmax = redux_max_nan(tm);
    const uint32_t qsel = __reduce_min_sync(0xffffffffu, (lane < NS && tm == tmax) ? th->red_q[lane] : 0xffffffffu);
    const bool any_nan = tmax != tmax;
    uint32_t idx = 0;
    float maxval = tmax;
    if (any_nan) {
      // rare: the first NaN of the decoded plane is the argmax (np.argmax / torch.max semantics)
      uint32_t first_nan = 0xffffffffu;
      for (int q = lane; q < nq && first_nan == 0xffffffffu; q += 32) {
        const float4 v = load_quad(q);
        if (v.x != v.x) first_nan = 4 * q;
        else if (v.y != v.y) first_nan = 4 * q + 1;
        else if (v.z != v.z) first_nan = 4 * q + 2;
        else if (v.w != v.w) first_nan = 4 * q + 3;
      }
      idx = __reduce_min_sync(0xffffffffu, first_nan);
      maxval = __uint_as_float(0x7fc00000u);
    } else if (qsel != 0xffffffffu) {
      const float4 v = load_quad((int)qsel);
      // `==` treats -0 and +0 as equal, like torch/numpy; report the element actually selected
      if (v.x == tmax) { idx = 4 * qsel; maxval = v.x; }
      else if (v.y == tmax) { idx = 4 * qsel + 1; maxval = v.y; }
      else if (v.z == tmax) { idx = 4 * qsel + 2; maxval = v.z; }
      else { idx = 4 * qsel + 3; maxval = v.w; }
    } else {
      maxval = val(0, 0);                     // every element is -inf
    }

    // masked integer coordinates (A1-A4)
    const int ipy = FAST ? (int)(idx / (uint32_t)(WC > 0 ? WC : 1)) : (int)(idx / (uint32_t)W);
    const int ipx = (int)idx - ipy * W;
    float cx = (float)ipx, cy = (float)ipy;
    const bool positive = maxval > 0.0f;
    if (a.mask_mode == LHN_MASK_ZERO && !positive) { cx = 0.f; cy = 0.f; }
    if (a.mask_mode == LHN_MASK_NEG1 && !positive) { cx = -1.f; cy = -1.f; }
    const int px = (int)cx, py = (int)cy;
    // DARK: the reference's interior guard; UDP: every plane with a positive maximum (coordinates >= 0)
    const bool dark_guard = (is_dark && (1 < px) && (px < W - 2) && (1 < py) && (py < H - 2)) || (udp && px >= 0 && py >= 0);

    TRS(6);
    PlaneRec* rec = &th->rec[buf];
    const int wx0 = px - 2 - bb;                      // first window column (may be negative)
    const int c0 = wx0 & ~3, xo = wx0 & 3;            // its quad-aligned start and the offset inside it

    // ---- stage the DARK window: zero-padded (ksize+4) rows x NQ quads of the decoded plane -----------------
    if (dark_guard && udp) {
      // UDP blurs the plane with cv2's default BORDER_REFLECT_101: the window is addressed through the mirror
      float* tile = reinterpret_cast<float*>(tile0 + (size_t)buf * tile_bytes);
      auto refl = [](int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); };
      for (int e = sl; e < TD * TD; e += ST) {
        const int r = e / TD, c = e - r * TD;
        tile[r * TCW + c] = val(refl(py - 2 - bb + r, H), refl(px - 2 - bb + c, W));
      }
    } else if (dark_guard) {
      float* tile = reinterpret_cast<float*>(tile0 + (size_t)buf * tile_bytes);
      for (int e = sl; e < TD * NQ; e += ST) {
        const int r = e / NQ, cq = e - r * NQ;          // compile-time divisor when KS > 0
        const int y = py - 2 - bb + r, x = c0 + 4 * cq;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (y >= 0 && y < H && x >= 0 && x < W) v = load_quad(y * QR + (x >> 2));
        *reinterpret_cast<float4*>(tile + r * TCW + 4 * cq) = v;
      }
    }
    TRS(7);
    // ---- positives of the balanced loss: a small window around the joint, by the last sweeper warp ---------
    if (LOSS && role == TW - 1) {
      float Spos = 0.f;
      int Npos = 0;
      if (a.loss_mode == LHN_LOSS_DISTANCE_BALANCE) {
        uint32_t s, k;
        split_channel(pc, s, k);
        int x_lo = 0, x_hi = W - 1, y_lo = 0, y_hi = H - 1;
        if (a.pos_value > 0.f && a.pos_value < 1.f) {
          // g > value  <=>  r^2 < -2 sigma^2 ln(value): a.pos_radius = that radius + a rounding margin
          const float rad = a.pos_radius[s];
          const float mxf = th->mx[tb], myf = th->my[tb];
          x_lo = max(0, (int)ceilf(mxf - rad)); x_hi = min(W - 1, (int)floorf(mxf + rad));
          y_lo = max(0, (int)ceilf(myf - rad)); y_hi = min(H - 1, (int)floorf(myf + rad));
        } else if (a.pos_value >= 1.f) {
          x_hi = -1;
        }
        if (th->render_on[tb] || a.pos_value < 0.f) {
          float sp = 0.f;
          // one window element per lane (5 x 5 = 25 lanes for sigma = 2)
          const int ww = x_hi - x_lo + 1, wn = ww > 0 ? ww * (y_hi - y_lo + 1) : 0;
          for (int e = lane; e < wn; e += 32) {
            const int ry = e / ww, xx = x_lo + (e - ry * ww), yy = y_lo + ry;
            const float gxv = ex[xx], gyv = ey[yy];
            if (gxv * gyv > a.pos_value) {
              const float d = fmaf(-gxv, gyv, elem_f32<T>(plane0, yy * W + xx));
              sp = fmaf(d, d, sp);
              Npos += 1;
            }
          }
          Spos = warp_sum(sp);
          Npos = __reduce_add_sync(0xffffffffu, Npos);
        }
      }
      if (lane == 0) { rec->spos = Spos; rec->npos = Npos; }
    }
    // ---- the first sweeper warp: +-0.25 rules (neighbours read while the plane is resident) + the record ----
    if (role == 1 && lane == 0) {
      float rx = cx, ry = cy;
      if (KS > 0) {
        // DARK: no quarter offset
      } else if (a.refine == LHN_REFINE_OFFSET_HALF || a.refine == LHN_REFINE_OFFSET) {
        const int xx = min(max(px, 0), W - 1), yy = min(max(py, 0), H - 1);
        // clamped neighbours; `>` false (equality, NaN) -> -0.25
        rx += (val(yy, min(xx + 1, W - 1)) > val(yy, max(xx - 1, 0))) ? 0.25f : -0.25f;
        ry += (val(min(yy + 1, H - 1), xx) > val(max(yy - 1, 0), xx)) ? 0.25f : -0.25f;
        if (a.refine == LHN_REFINE_OFFSET_HALF) { rx += 0.5f; ry += 0.5f; }
      } else if (a.refine == LHN_REFINE_SIGN || a.refine == LHN_REFINE_SIGN_ROUND) {
        int qx = px, qy = py;
        if (a.refine == LHN_REFINE_SIGN_ROUND) { qx = (int)floorf(cx + 0.5f); qy = (int)floorf(cy + 0.5f); }
        if (1 < qx && qx < W - 1 && 1 < qy && qy < H - 1) {
          const float ddx = val(qy, qx + 1) - val(qy, qx - 1);
          const float ddy = val(qy + 1, qx) - val(qy - 1, qx);
          const float sxn = (ddx != ddx) ? ddx : (float)((ddx > 0.f) - (ddx < 0.f));   // np.sign
          const float syn = (ddy != ddy) ? ddy : (float)((ddy > 0.f) - (ddy < 0.f));
          rx += sxn * 0.25f; ry += syn * 0.25f;
        }
      }
      float S = 0.f;
      if (LOSS) for (int i = 0; i < NS; ++i) S += th->red_s[i];
      rec->idx = idx; rec->maxval = maxval; rec->rx = rx; rec->ry = ry;
      rec->ssum = S;
      rec->flags = (dark_guard ? 1 : 0) | (any_nan ? 2 : 0) | ((udp ? 0 : xo) << 8);
    }
    TRS(4);
    // S3: everything the epilogue needs is out of the stage — nobody reads it again
    named_sync(bar_id, ST);
    if (sl == 0) {
      // re-arm the stage with the plane `nstg` ahead, then hand the record to the epilogue warp
      if (a.use_tma && (uint64_t)p + (uint64_t)nstg * total_teams < n_planes) {
        uint32_t nb = pb, nc = pc;
        for (int i = 0; i < nstg; ++i) advance(nb, nc);
        fence_proxy_async();
        issue(nb, nc, stg);
      }
      mbar_arrive(&th->full[buf]);
    }
    TRS(5);

  }
}

// ---- host side ----------------------------------------------------------------------------------------
int num_sms();                       // lhn_loss_render.cu: SM count of the current device, cached per device
static int sm_count() { return num_sms(); }
extern thread_local lhn_k1_launch_info g_k1_launch;   // lhn_heatmap.cu: lhn_k1_last_launch()

template <typename T, int WC, int TWC, bool FLIP, bool LOSS, int KS>
static int launch_one(HmArgs& a, int nteams, size_t smem, cudaStream_t st) {
  auto kern = heatmap_team_kernel<T, WC, TWC, FLIP, LOSS, KS>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { set_last_error(e); return LHN_ECUDA; }
  // one CTA per SM; small problems still spread over as many SMs as they have planes (team-major numbering)
  int sms = sm_count() - a.spare_sms;
  if (sms < 1) sms = 1;
  if (a.xch_courier && sms < 2) a.xch_courier = 0;
  if (a.xch_courier) --sms;                                   // one SM carries the courier CTA instead of planes
  int64_t ctas = (a.n_planes < sms ? a.n_planes : sms) + a.xch_courier;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)ctas); cfg.blockDim = dim3((unsigned)(nteams * a.team_warps * 32));
  cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = a.overlap_previous ? 1 : 0;
  e = cudaLaunchKernelEx(&cfg, kern, a);
  if (e != cudaSuccess) { set_last_error(e); return LHN_ECUDA; }
  const int rc = check_launch();
  if (rc == LHN_OK) {
    lhn_k1_launch_info& r = g_k1_launch;
    r = {};
    r.path = 1;
    r.dtype = sizeof(T) == 4 ? LHN_F32 : std::is_same<T, __nv_bfloat16>::value ? LHN_BF16 : LHN_F16;
    r.flip = FLIP; r.loss = LOSS; r.counters = a.counters != nullptr;
    r.wc = WC; r.twc = TWC; r.ks = KS;
    r.team_warps = a.team_warps; r.nteams = nteams; r.stages = a.stages; r.sweeper_tables = a.sweeper_tables;
    r.use_tma = a.use_tma; r.ctas = (int32_t)ctas; r.stagger_ns = a.stagger_ns;
  }
  return rc;
}

template <typename T, bool FLIP, bool LOSS>
static int dispatch_variant(HmArgs& a, int wc, int nteams, size_t smem, cudaStream_t st) {
  // compile-time team size of the fixed-size paths (64x64, 56x56): stage > 16 KB (f32 + flip) -> 4 warps, else 2
  constexpr int TWF = (sizeof(T) == 4 && FLIP) ? 4 : 2;
  const bool ks11 = a.refine == LHN_REFINE_DARK && a.ksize == 11;
  // 128x128 (hourglass / srhandnet high-resolution maps): always 8-warp teams (7 sweepers), one 64 KB stage each.
  // On the run-time-size path this shape streamed at 85 % of the peak (profiles/r01_batch_scaling_cfg5.txt).
  // Instantiated for f32 without a flip plane only — the combination BASELINE config 5 uses and the GPU tests cover
  // ((2,4,128,128) decode / fused cases, the full-size config-5 property test); f32 + flip does not fit the team
  // kernel at this size, 2-byte inputs stay on the run-time-size path until they are measured and tested.
  if constexpr (sizeof(T) == 4 && !FLIP) {
    if (wc == 128 && a.team_warps == 8) {
      if (ks11) return launch_one<T, 128, 8, FLIP, LOSS, 11>(a, nteams, smem, st);
      return launch_one<T, 128, 8, FLIP, LOSS, 0>(a, nteams, smem, st);
    }
    // the lower scales of SRHandNet's output pyramid ([16,16,32,64], generateTarget.py:383-386): 1 / 4 KB planes,
    // 12 teams of 2 warps with up to 4 stages each
    if (wc == 32 && a.team_warps == 2) {
      if (ks11) return launch_one<T, 32, 2, FLIP, LOSS, 11>(a, nteams, smem, st);
      return launch_one<T, 32, 2, FLIP, LOSS, 0>(a, nteams, smem, st);
    }
    if (wc == 16 && a.team_warps == 2) {
      if (ks11) return launch_one<T, 16, 2, FLIP, LOSS, 11>(a, nteams, smem, st);
      return launch_one<T, 16, 2, FLIP, LOSS, 0>(a, nteams, smem, st);
    }
  }
  // 128x128 in bf16 / f16: 32 KB planes -> 6 teams of 4 warps without a flip plane, 3 teams of 8 warps with one
  if constexpr (sizeof(T) == 2) {
    if (wc == 128 && a.team_warps == (FLIP ? 8 : 4)) {
      if (ks11) return launch_one<T, 128, (FLIP ? 8 : 4), FLIP, LOSS, 11>(a, nteams, smem, st);
      return launch_one<T, 128, (FLIP ? 8 : 4), FLIP, LOSS, 0>(a, nteams, smem, st);
    }
  }
  if (wc == 64 && a.team_warps == TWF) {
    if (ks11) return launch_one<T, 64, TWF, FLIP, LOSS, 11>(a, nteams, smem, st);
    return launch_one<T, 64, TWF, FLIP, LOSS, 0>(a, nteams, smem, st);
  }
  if (wc == 56 && a.team_warps == TWF) {
    if (ks11) return launch_one<T, 56, TWF, FLIP, LOSS, 11>(a, nteams, smem, st);
    return launch_one<T, 56, TWF, FLIP, LOSS, 0>(a, nteams, smem, st);
  }
  if (ks11) return launch_one<T, 0, 0, FLIP, LOSS, 11>(a, nteams, smem, st);
  return launch_one<T, 0, 0, FLIP, LOSS, 0>(a, nteams, smem, st);
}

template <typename T>
int dispatch_team(HmArgs& a, bool flip, bool loss, int wc, int nteams, size_t smem, cudaStream_t st) {
  if (flip) return loss ? dispatch_variant<T, true, true>(a, wc, nteams, smem, st)
                        : dispatch_variant<T, true, false>(a, wc, nteams, smem, st);
  return loss ? dispatch_variant<T, false, true>(a, wc, nteams, smem, st)
              : dispatch_variant<T, false, false>(a, wc, nteams, smem, st);
}

#if defined(LHN_TEAM_DTYPE_TU) && defined(LHN_TRACE)
#ifdef LHN_TRACE_EXPORT
extern "C" __attribute__((visibility("default"))) int lhn_debug_trace(long long* host) {
  return (int)cudaMemcpyFromSymbol(host, g_trace, sizeof(g_trace));
}
#endif
#endif
#ifndef LHN_TEAM_DTYPE_TU
// instantiated per dtype in lhn_heatmap_team_{f32,bf16,f16}.cu so the three compile in parallel
extern template int dispatch_team<float>(HmArgs&, bool, bool, int, int, size_t, cudaStream_t);
extern template int dispatch_team<__nv_bfloat16>(HmArgs&, bool, bool, int, int, size_t, cudaStream_t);
extern template int dispatch_team<__half>(HmArgs&, bool, bool, int, int, size_t, cudaStream_t);

int launch_heatmap_warp_kernel(HmArgs& a, int dtype, cudaStream_t st) {
  const bool flip = a.hm_flip != nullptr;
  const bool loss = a.loss_mode != LHN_LOSS_NONE;
  const size_t esz = dtype == LHN_F32 ? 4 : 2;
  if ((a.W & 3) != 0) return 1;                       // quads must not straddle rows
  const size_t plane_bytes = (size_t)a.HW * esz;
  if (plane_bytes % 16) return 1;
  const size_t plane_al = align_up(plane_bytes, 128);
  a.stage_bytes = (int)(flip ? 2 * plane_al : plane_al);
  const bool is_dark = a.refine == LHN_REFINE_DARK || a.refine == LHN_REFINE_DARK_LEGACY ||
                       a.refine == LHN_REFINE_DARK_UDP;
  a.tile_dim = is_dark ? a.ksize + 4 : 0;
  const size_t aux = align_up(sizeof(TeamHeader), 16) + 3 * align_up((size_t)(a.W + a.H) * 4, 16) +
                     2 * align_up((size_t)a.tile_dim * 4 * tile_quads(a.tile_dim) * 4, 16) +
                     (size_t)a.tile_dim * 5 * 8 + 32 * 4 + align_up((size_t)a.K * 4, 16);
  // Teams: the serial epilogue of a plane costs ~4-5k cycles of one warp whatever the plane size, so small planes
  // need MANY epilogue warps: stages of <= 16 KB run up to 12 teams of 2 warps (1 sweeper + 1 epilogue), larger
  // ones 6 teams of 4 warps (3 sweepers + 1 epilogue) or 3 / 2 teams of 8 warps.  Spare shared memory then
  // multiplies the stages per team (2 or 4): the next planes of a team are already in flight while it sweeps.
  size_t budget = 227 * 1024;
  {
    // Experimental (profiles/r02_two_launch_interleave.txt): an OVERLAPPED launch may take only half of each SM's
    // shared memory, so that the successor launch becomes co-resident half-way through (the trigger point) and the
    // two launches' fill / drain bubbles interleave instead of coinciding.  LHN_CTAS_PER_SM=2 selects it.
    const char* cps = getenv("LHN_CTAS_PER_SM");
    if (cps && cps[0] == '2' && a.overlap_previous) budget = 113 * 1024;
  }
  const size_t aux_al = align_up(aux, 128);
  const size_t per_team = a.stage_bytes + aux_al;
  int nteams, tw;
  const char* pol = getenv("LHN_TEAM_POLICY");
  // measured (profiles/r01_configs.txt): for <= 16 KB stages up to 12 teams of 2 warps beat 6 teams of 4 warps
  // with two stages each (78 vs 67 % of peak at 64x64 f32 with loss + DARK); LHN_TEAM_POLICY=0 selects the latter
  const bool many_small = !(pol && pol[0] == '0');
  if (a.stage_bytes <= 16 * 1024 && many_small) { tw = 2; nteams = (int)(budget / per_team); if (nteams > kMaxTeams) nteams = kMaxTeams; }
  else if (6 * per_team <= budget) { tw = 4; nteams = 6; }
  else { tw = 8; nteams = (int)(budget / per_team); if (nteams > 3) nteams = 3; }
  if (nteams < 2) return 1;                           // plane pair too large: CTA-per-plane kernel
  int nstg = 1;
  while (nstg < 4 && (size_t)nteams * (2 * nstg * a.stage_bytes + aux_al) <= budget) nstg *= 2;
  const char* env = getenv("LHN_TEAM_STAGES");
  if (env && (atoi(env) == 1 || atoi(env) == 2 || atoi(env) == 4) && atoi(env) <= nstg) nstg = atoi(env);
  a.stages = nstg;
  {
    // measured (profiles/probes/stagger_sweep.sh): 600 ns between teams buys ~1.3 % on a cold launch of the
    // headline shape; pointless (and a visible delay) when a team only has a few planes
    const char* sg = getenv("LHN_STAGGER_NS");
    a.stagger_ns = sg ? atoi(sg) : ((a.n_planes >= (int64_t)8 * nteams * sm_count()) ? 600 : 0);
  }
  {
    const char* tg = getenv("LHN_TRIGGER");               // "half" / "early" / "p<n>": override the trigger point (experiments)
    if (a.xch.world > 0 && !loss && a.counters) {
      const char* cr = getenv("LHN_XCH_COURIER");             // "0": the first plane-carrying CTA to finish exchanges
      a.xch_courier = (cr && cr[0] == '0') ? 0 : 1;
    }
    // half-way only where a plane-carrying CTA exchanges (the batch-global loss; counters without a courier CTA): there
    // the predecessor's completion includes its exchange and needs the slack.  With the courier the early trigger is
    // best again (measured at 2 GPUs: 42.3 us per step early, 44.3 half-way; profiles/r02_courier.txt)
    a.trigger_halfway = tg ? (tg[0] == 'h') : (a.xch.world > 1 && !a.xch_courier);
    a.trigger_plane = (tg && tg[0] == 'p' && tg[1] >= '0' && tg[1] <= '9') ? (tg[1] - '0') : 2;
  }
  a.sweeper_tables = (nstg >= 2 && tw >= 4) ? 1 : 0;
  a.team_warps = tw;
  a.warp_smem = (int)((size_t)nstg * a.stage_bytes + aux_al);
  {
    // joint / feat_stride: a power-of-two stride (256/64, 224/56, ...) is an exact multiplication
    int ex = 0, ey = 0;
    a.feat_pow2 = (a.feat_x > 0 && a.feat_y > 0 && frexp(a.feat_x, &ex) == 0.5 && frexp(a.feat_y, &ey) == 0.5) ? 1 : 0;
    a.inv_feat_x = a.feat_x > 0 ? 1.0 / a.feat_x : 0.0;
    a.inv_feat_y = a.feat_y > 0 ? 1.0 / a.feat_y : 0.0;
  }
  for (int i = 0; i < LHN_MAX_STACKS; ++i) {
    const double sg = (double)a.sigma[i];
    a.inv2s2[i] = sg > 0 ? 1.0 / (2.0 * sg * sg) : 0.0;
    a.pos_radius[i] = (a.pos_value > 0.f && a.pos_value < 1.f && sg > 0)
                          ? (float)(sg * sqrt(-2.0 * log((double)a.pos_value)) * 1.001 + 0.01) : 0.f;
  }
  int wc = (a.W != a.H) ? 0 : ((a.W == 64 || a.W == 56 || a.W == 128 || a.W == 32 || a.W == 16) ? a.W : 0);
  {
    const char* nf = getenv("LHN_NO_FAST");              // tests: run the run-time-size instantiation on every shape
    if (nf && nf[0] == '1') wc = 0;
  }
  size_t smem = (size_t)nteams * a.warp_smem;
  if (a.counters) {
    // CTA-shared metric counters after the teams' regions; drop a team if they do not fit
    const size_t cnt_bytes = (size_t)(a.auc_steps + 5) * a.K * 8 + 16;
    while (nteams > 2 && (size_t)nteams * a.warp_smem + cnt_bytes > budget) --nteams;
    smem = (size_t)nteams * a.warp_smem + cnt_bytes;
    if (smem > budget) return 1;
    // the in-kernel exchange gathers every rank's block in the CTA's (by then idle) shared memory
    if (a.xch.world > 0 && smem < xch_scratch_bytes(a.xch.world, (a.auc_steps + 5) * a.K)) return LHN_EINVAL;
  }
  switch (dtype) {
    case LHN_F32: return dispatch_team<float>(a, flip, loss, wc, nteams, smem, st);
    case LHN_BF16: return dispatch_team<__nv_bfloat16>(a, flip, loss, wc, nteams, smem, st);
    case LHN_F16: return dispatch_team<__half>(a, flip, loss, wc, nteams, smem, st);
    default: return LHN_EDTYPE;
  }
}
#endif

}  // namespace lhn
