// SimDRLoss with its two linear heads fused (loss/centernet_simdr_loss.py:42-69):
//
//     pred_x | pred_y = heatmap.flatten(2) @ [Wx ; Wy]^T + [bx ; by]        [M, Kd] x [Kd, N],  M = B*K,  N = Lx + Ly
//     loss = (1/K) sum_j ( SmoothL1mean(pred_x[:, j], tx[:, j]) + SmoothL1mean(pred_y[:, j], ty[:, j]) ) * mean_b w[b, j]
//
// — the only dense contraction near the hot path (SURVEY.md §8a S3 / §8f rank 4).  One tcgen05 kernel: the GEMM
// accumulates in TMEM, the epilogue reads the accumulator tile with tcgen05.ld, adds the bias, takes SmoothL1 against
// the target and reduces it per row, so the predictions never reach HBM (the reference writes [B*K, N] f32 from cuBLAS
// and reads it back in the loss).  Optionally the epilogue also stores d loss / d pred (the clamp of the residual) for
// the backward, or the predictions themselves for inference.
//
// fp32 parity: the reference multiplies in fp32 (torch's default keeps TF32 off).  Operands are split into bf16 pairs
// x = hi + lo (|x - hi - lo| <= 2^-17 |x|) and each k-block issues three bf16 MMAs into the same fp32 accumulator —
// lo*hi + hi*lo + hi*hi — which leaves a relative error of ~1e-5 per PRODUCT with random sign, i.e. ~1e-7 on the loss.
//
// Structure (one 128 x BN output tile per CTA, 256 threads):
//   warp 0    TMA producer: four 2-D tiled loads per k-block (A_hi, A_lo, W_hi, W_lo; 128-byte swizzle) into a ring
//   warp 1    MMA issuer: one thread, 12 tcgen05.mma.cta_group::1.kind::f16 per k-block, tcgen05.commit frees the stage
//   warp 2    TMEM allocator (BN fp32 columns x 128 lanes)
//   warps 4-7 epilogue: tcgen05.ld 32x32b.x32 -> registers, bias + SmoothL1 + row sums, partial sums per (N tile, row)
// A second tiny kernel adds the partial sums in a fixed order (bitwise reproducible) and applies the joint weights.
#include <cuda.h>
#include <math_constants.h>
#include <stdlib.h>

#include "lhn_common.cuh"

namespace lhn {

int num_sms();

constexpr int kHeadsBM = 128;      // rows of the output tile = TMEM lanes
constexpr int kHeadsBK = 64;       // bf16 elements per k-block = one 128-byte swizzle row

struct HeadsArgs {
  const float* bias;               // [N]
  const float* tx;                 // [M, Lx]
  const float* ty;                 // [M, Ly]
  double* partial;                 // [N / BN, M, 2] f64 (sum_x, sum_y) per (N tile, row)
  float* dpred;                    // optional [M, N]: clamp(pred - target, -1, 1) = d SmoothL1 / d pred
  float* pred;                     // optional [M, N]
  int M, N, Kd, Lx, Ly;
};

// ---- PTX wrappers ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> f32, both operands K-major
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 consecutive fp32 columns of the accumulator: thread = lane (row), r[i] = column i
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor of a K-major bf16 tile stored as 128-byte rows with the 128-byte swizzle
// (what a TMA box {64, rows} with CU_TENSOR_MAP_SWIZZLE_128B writes): start address >> 4 in bits [0,14), leading byte
// offset (unused inside one swizzle atom; the canonical value 1) in [16,30), stride byte offset = 8 rows x 128 B
// = 1024 >> 4 in [32,46), descriptor version 1 in [46,48), layout type SWIZZLE_128B = 2 in [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}

__device__ __forceinline__ float smooth_l1_f(float d) {
  const float ad = fabsf(d);
  return ad < 1.f ? 0.5f * d * d : ad - 0.5f;
}

template <int BN>
struct HeadsTile {
  static constexpr int kStages = BN <= 80 ? 4 : 3;
  static constexpr uint32_t kABytes = kHeadsBM * kHeadsBK * 2;   // 16 KB
  static constexpr uint32_t kWBytes = BN * kHeadsBK * 2;
  static constexpr uint32_t kStageBytes = 2 * kABytes + 2 * kWBytes;
  static constexpr uint32_t kTmemCols = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));
  static constexpr size_t kSmemBytes = (size_t)kStages * kStageBytes + 1024 /* alignment slack */ + 256 /* barriers */;
};

template <int BN>
__global__ void __launch_bounds__(256, 1)
simdr_heads_kernel(const __grid_constant__ CUtensorMap tm_ahi, const __grid_constant__ CUtensorMap tm_alo,
                   const __grid_constant__ CUtensorMap tm_whi, const __grid_constant__ CUtensorMap tm_wlo,
                   const HeadsArgs a) {
  using Tile = HeadsTile<BN>;
  constexpr int kStages = Tile::kStages;
  extern __shared__ unsigned char smem_dyn[];
  // the 128-byte swizzle atoms (8 rows x 128 B) must start on 1024-byte boundaries
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)kStages * Tile::kStageBytes);
  uint64_t* empty = full + kStages;
  uint64_t* tmem_full = empty + kStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * kHeadsBM, n0 = blockIdx.x * BN;
  const int num_kb = a.Kd / kHeadsBK;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_ahi); prefetch_tmap(&tm_alo); prefetch_tmap(&tm_whi); prefetch_tmap(&tm_wlo);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(Tile::kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % kStages;
        const uint32_t ph = (uint32_t)(kb / kStages) & 1u;
        mbar_wait(&empty[s], ph ^ 1u);                        // the MMAs that read this slot have completed
        unsigned char* st = smem + (size_t)s * Tile::kStageBytes;
        mbar_arrive_expect_tx(&full[s], Tile::kStageBytes);
        const int k0 = kb * kHeadsBK;
        tma_load_2d(st, &tm_ahi, k0, m0, &full[s]);
        tma_load_2d(st + Tile::kABytes, &tm_alo, k0, m0, &full[s]);
        tma_load_2d(st + 2 * Tile::kABytes, &tm_whi, k0, n0, &full[s]);
        tma_load_2d(st + 2 * Tile::kABytes + Tile::kWBytes, &tm_wlo, k0, n0, &full[s]);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread) =====
    if (lane == 0) {
      // instruction descriptor: D = f32 (bits 4-5 = 1), A = B = bf16 (bits 7-9, 10-12 = 1), both K-major (bits 15, 16 = 0),
      // N >> 3 in bits 17-22, M >> 4 in bits 24-28
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(kHeadsBM >> 4) << 24);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % kStages;
        const uint32_t ph = (uint32_t)(kb / kStages) & 1u;
        mbar_wait(&full[s], ph);
        tc_fence_after();
        const uint32_t st = smem_u32(smem + (size_t)s * Tile::kStageBytes);
        const uint64_t d_ahi = umma_desc_sw128(st), d_alo = umma_desc_sw128(st + Tile::kABytes);
        const uint64_t d_whi = umma_desc_sw128(st + 2 * Tile::kABytes);
        const uint64_t d_wlo = umma_desc_sw128(st + 2 * Tile::kABytes + Tile::kWBytes);
#pragma unroll
        for (int k = 0; k < kHeadsBK / 16; ++k) {
          const uint64_t off = (uint64_t)(k * 2);            // 16 bf16 = 32 bytes further along K: start address + 32 >> 4
          umma_bf16(tmem_base, d_alo + off, d_whi + off, idesc, (kb | k) != 0 ? 1u : 0u);   // the small terms first
          umma_bf16(tmem_base, d_ahi + off, d_wlo + off, idesc, 1u);
          umma_bf16(tmem_base, d_ahi + off, d_whi + off, idesc, 1u);
        }
        tc_commit(&empty[s]);                                 // arrives when the MMAs above have read the slot
      }
      tc_commit(tmem_full);                                   // accumulator complete
    }
  } else if (warp >= 4) {
    // ===== epilogue: one accumulator row (TMEM lane) per thread =====
    const int q = warp & 3;                                   // warp w reaches TMEM lanes 32 (w % 4) .. +31
    const int row = m0 + 32 * q + lane;
    const bool row_ok = row < a.M;
    mbar_wait(tmem_full, 0u);
    tc_fence_after();
    float sx = 0.f, sy = 0.f;
    const float* txr = a.tx + (size_t)(row_ok ? row : 0) * a.Lx;
    const float* tyr = a.ty + (size_t)(row_ok ? row : 0) * a.Ly;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t r[32];
      tmem_ld_32x32(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)c0, r);
      tmem_ld_wait();
      if (row_ok) {
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const int col = n0 + c0 + i;                        // a group of 4 never straddles Lx (Lx % 4 == 0)
          if (c0 + i >= BN || col >= a.N) continue;           // BN = 80: the third chunk is half used; ragged last N tile
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(a.bias + col));
          const bool isx = col < a.Lx;
          const float4 t4 = isx ? __ldg(reinterpret_cast<const float4*>(txr + col))
                                : __ldg(reinterpret_cast<const float4*>(tyr + (col - a.Lx)));
          float4 p;
          p.x = __uint_as_float(r[i]) + b4.x; p.y = __uint_as_float(r[i + 1]) + b4.y;
          p.z = __uint_as_float(r[i + 2]) + b4.z; p.w = __uint_as_float(r[i + 3]) + b4.w;
          const float4 d = make_float4(p.x - t4.x, p.y - t4.y, p.z - t4.z, p.w - t4.w);
          const float s4 = (smooth_l1_f(d.x) + smooth_l1_f(d.y)) + (smooth_l1_f(d.z) + smooth_l1_f(d.w));
          if (isx) sx += s4; else sy += s4;
          if (a.dpred) {
            // clamp that keeps NaN, as torch's clamp and the SmoothL1 gradient do (fmaxf alone would return -1)
            auto clamp1 = [](float v) { return v != v ? v : fminf(fmaxf(v, -1.f), 1.f); };
            const float4 g = make_float4(clamp1(d.x), clamp1(d.y), clamp1(d.z), clamp1(d.w));
            *reinterpret_cast<float4*>(a.dpred + (size_t)row * a.N + col) = g;
          }
          if (a.pred) *reinterpret_cast<float4*>(a.pred + (size_t)row * a.N + col) = p;
        }
      }
    }
    if (row_ok) {
      double2* dst = reinterpret_cast<double2*>(a.partial + ((size_t)blockIdx.x * a.M + row) * 2);
      *dst = make_double2((double)sx, (double)sy);
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Tile::kTmemCols) : "memory");
  }
}

// loss = (1/K) sum_j ( Sx_j / (B Lx) + Sy_j / (B Ly) ) * ( sum_b w_bj / B ), Sx_j = sum over b and N tiles, in a fixed order
__global__ void __launch_bounds__(1024) simdr_heads_finalize_kernel(const double* __restrict__ partial, int n_tiles,
                                                                    const float* __restrict__ weight, int64_t B, int K,
                                                                    int Lx, int Ly, float* __restrict__ loss) {
  __shared__ double red[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int64_t M = B * K;
  double acc = 0.0;
  for (int j = warp; j < K; j += nwarps) {
    double sx = 0, sy = 0, sw = 0;
    for (int64_t b = lane; b < B; b += 32) {
      const int64_t row = b * K + j;
      for (int t = 0; t < n_tiles; ++t) {
        const double2 v = *reinterpret_cast<const double2*>(partial + ((size_t)t * M + row) * 2);
        sx += v.x; sy += v.y;
      }
      sw += (double)weight[row];
    }
    sx = warp_sum(sx); sy = warp_sum(sy); sw = warp_sum(sw);
    acc += (sx / ((double)B * Lx) + sy / ((double)B * Ly)) * (sw / (double)B);
  }
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < nwarps; ++i) t += red[i];
    loss[0] = (float)(t / (double)K);
  }
}

// x = hi + lo, both bf16 (round to nearest even): hi = bf16(x), lo = bf16(x - hi)
__global__ void __launch_bounds__(256) split_bf16_kernel(const float* __restrict__ x, int64_t n4, __nv_bfloat16* __restrict__ hi,
                                                         __nv_bfloat16* __restrict__ lo) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = ldg_stream_f4(reinterpret_cast<const float4*>(x) + i);
    const __nv_bfloat16 h0 = __float2bfloat16_rn(v.x), h1 = __float2bfloat16_rn(v.y), h2 = __float2bfloat16_rn(v.z),
                        h3 = __float2bfloat16_rn(v.w);
    const __nv_bfloat16 l0 = __float2bfloat16_rn(v.x - __bfloat162float(h0)), l1 = __float2bfloat16_rn(v.y - __bfloat162float(h1)),
                        l2 = __float2bfloat16_rn(v.z - __bfloat162float(h2)), l3 = __float2bfloat16_rn(v.w - __bfloat162float(h3));
    auto pack = [](__nv_bfloat16 a, __nv_bfloat16 b) {
      return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
    };
    reinterpret_cast<uint2*>(hi)[i] = make_uint2(pack(h0, h1), pack(h2, h3));
    reinterpret_cast<uint2*>(lo)[i] = make_uint2(pack(l0, l1), pack(l2, l3));
  }
}

// ---- host ----------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// bf16 [rows, cols] row-major -> tiled map with a {64, box_rows} box and the 128-byte swizzle
static bool make_tmap(CUtensorMap* tm, const void* base, int64_t rows, int64_t cols, int box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  const cuuint32_t box[2] = {(cuuint32_t)kHeadsBK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// N tile: 128 columns unless that leaves more than half of the SMs idle and 64 still fits in one wave.  An 80-column
// tile (LHN_HEADS_BN=80) fills 143 of 148 SMs at the reference's training shape (M = 1344, N = 1024) where 128 fills
// 88 — and is NOT faster (54.2 against 53.3 us, 212 against 176 us at M = 5376, profiles/r02_simdr_heads_bn80.txt): the
// kernel is bound by L2 -> shared-memory traffic, and narrower tiles re-read the A operand more often.
static int pick_bn(int64_t M, int N) {
  const char* env = getenv("LHN_HEADS_BN");
  if (env && (atoi(env) == 64 || atoi(env) == 80 || atoi(env) == 128)) return atoi(env);
  const int64_t mt = (M + kHeadsBM - 1) / kHeadsBM, sms = num_sms();
  const int64_t c128 = mt * ((N + 127) / 128), c64 = mt * ((N + 63) / 64);
  if (c128 * 2 <= sms && c64 <= sms) return 64;
  return 128;
}

template <int BN>
static int launch_heads(const CUtensorMap& ahi, const CUtensorMap& alo, const CUtensorMap& whi, const CUtensorMap& wlo,
                        const HeadsArgs& a, cudaStream_t st) {
  auto kern = simdr_heads_kernel<BN>;
  const size_t smem = HeadsTile<BN>::kSmemBytes;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { set_last_error(e); return LHN_ECUDA; }
  dim3 grid((unsigned)((a.N + BN - 1) / BN), (unsigned)((a.M + kHeadsBM - 1) / kHeadsBM));
  kern<<<grid, 256, smem, st>>>(ahi, alo, whi, wlo, a);
  return check_launch();
}

}  // namespace lhn

using namespace lhn;

extern "C" int lhn_split_bf16(const float* x, int64_t n, void* hi, void* lo, lhn_stream_t stream) {
  if (!x || !hi || !lo || n < 0 || (n & 3)) return LHN_EINVAL;
  if (((uintptr_t)x % 16) || ((uintptr_t)hi % 8) || ((uintptr_t)lo % 8)) return LHN_EALIGN;
  if (n == 0) return LHN_OK;
  const int64_t n4 = n >> 2;
  int64_t blocks = (n4 + 255) / 256;
  const int64_t cap = (int64_t)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  split_bf16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, n4, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo);
  return check_launch();
}

extern "C" int64_t lhn_simdr_heads_workspace_bytes(int64_t B, int K, int Lx, int Ly) {
  if (B <= 0 || K <= 0 || Lx <= 0 || Ly <= 0) return LHN_EINVAL;
  return (int64_t)((Lx + Ly + 63) / 64) * B * K * 2 * (int64_t)sizeof(double);     // the narrowest N tile is 64 columns
}

// The same from the f32 heatmaps: splits them into the workspace first (one more streaming launch, no host round trip).
// workspace: lhn_simdr_heads_f32_workspace_bytes(B, K, Kd, Lx, Ly) = partial sums + 2 x bf16 [B*K, Kd].
extern "C" int64_t lhn_simdr_heads_f32_workspace_bytes(int64_t B, int K, int Kd, int Lx, int Ly) {
  const int64_t p = lhn_simdr_heads_workspace_bytes(B, K, Lx, Ly);
  if (p < 0 || Kd <= 0) return LHN_EINVAL;
  return (p + 255) / 256 * 256 + 2 * B * K * (int64_t)Kd * 2;
}

extern "C" int lhn_simdr_heads_loss(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo,
                                    const float* bias, const float* target_x, const float* target_y,
                                    const float* weight, int64_t B, int K, int Kd, int Lx, int Ly, void* workspace,
                                    int64_t workspace_bytes, float* loss, float* dpred, float* pred,
                                    lhn_stream_t stream);

extern "C" int lhn_simdr_heads_loss_f32(const float* heatmap, const void* w_hi, const void* w_lo, const float* bias,
                                        const float* target_x, const float* target_y, const float* weight, int64_t B,
                                        int K, int Kd, int Lx, int Ly, void* workspace, int64_t workspace_bytes,
                                        float* loss, float* dpred, float* pred, lhn_stream_t stream) {
  g_simdr_launch = {};
  if (!heatmap || !workspace || B <= 0 || K <= 0 || Kd <= 0 || (Kd & 3)) return LHN_EINVAL;
  const int64_t need = lhn_simdr_heads_f32_workspace_bytes(B, K, Kd, Lx, Ly);
  if (need < 0) return LHN_EINVAL;
  if (workspace_bytes < need) return LHN_EWORKSPACE;
  if ((uintptr_t)workspace % 256 || (uintptr_t)heatmap % 16) return LHN_EALIGN;
  const int64_t p = (lhn_simdr_heads_workspace_bytes(B, K, Lx, Ly) + 255) / 256 * 256;
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  void* a_hi = ws + p;
  void* a_lo = ws + p + B * K * (int64_t)Kd * 2;
  int rc = lhn_split_bf16(heatmap, B * K * (int64_t)Kd, a_hi, a_lo, stream);
  if (rc) return rc;
  return lhn_simdr_heads_loss(a_hi, a_lo, w_hi, w_lo, bias, target_x, target_y, weight, B, K, Kd, Lx, Ly, workspace, p, loss,
                              dpred, pred, stream);
}

extern "C" int lhn_simdr_heads_loss(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo,
                                    const float* bias, const float* target_x, const float* target_y,
                                    const float* weight, int64_t B, int K, int Kd, int Lx, int Ly, void* workspace,
                                    int64_t workspace_bytes, float* loss, float* dpred, float* pred,
                                    lhn_stream_t stream) {
  g_simdr_launch = {};
  if (!a_hi || !a_lo || !w_hi || !w_lo || !bias || !target_x || !target_y || !weight || !workspace || !loss || B <= 0 ||
      K <= 0 || Kd <= 0 || Lx <= 0 || Ly <= 0)
    return LHN_EINVAL;
  const int N = Lx + Ly;
  const int64_t M = B * K;
  // k-blocks of 64, N tiles of 64 or 128, float4 groups that do not straddle the x | y boundary
  if (Kd % kHeadsBK || N % 64 || (Lx & 3) || (Ly & 3) || M > 0x7fffffffLL) return LHN_EINVAL;
  if (workspace_bytes < lhn_simdr_heads_workspace_bytes(B, K, Lx, Ly)) return LHN_EWORKSPACE;
  auto al16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
  if (!al16(a_hi) || !al16(a_lo) || !al16(w_hi) || !al16(w_lo) || !al16(bias) || !al16(target_x) || !al16(target_y) ||
      !al16(workspace) || (dpred && !al16(dpred)) || (pred && !al16(pred)))
    return LHN_EALIGN;
  const int bn = pick_bn(M, N);
  CUtensorMap ahi, alo, whi, wlo;
  if (!make_tmap(&ahi, a_hi, M, Kd, kHeadsBM) || !make_tmap(&alo, a_lo, M, Kd, kHeadsBM) ||
      !make_tmap(&whi, w_hi, N, Kd, bn) || !make_tmap(&wlo, w_lo, N, Kd, bn))
    return LHN_ECUDA;
  HeadsArgs a{};
  a.bias = bias; a.tx = target_x; a.ty = target_y; a.partial = (double*)workspace; a.dpred = dpred; a.pred = pred;
  a.M = (int)M; a.N = N; a.Kd = Kd; a.Lx = Lx; a.Ly = Ly;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = bn == 128 ? launch_heads<128>(ahi, alo, whi, wlo, a, st)
                     : (bn == 80 ? launch_heads<80>(ahi, alo, whi, wlo, a, st) : launch_heads<64>(ahi, alo, whi, wlo, a, st));
  if (rc) return rc;
  simdr_heads_finalize_kernel<<<1, 1024, 0, st>>>((const double*)workspace, (N + bn - 1) / bn, weight, B, K, Lx, Ly, loss);
  rc = check_launch();
  if (rc == LHN_OK) {
    const int stages = bn == 128 ? HeadsTile<128>::kStages : (bn == 80 ? HeadsTile<80>::kStages : HeadsTile<64>::kStages);
    simdr_record(5, 1, LHN_BF16, 8, stages, (int64_t)((N + bn - 1) / bn) * ((M + kHeadsBM - 1) / kHeadsBM), 1, 1, bn);
  }
  return rc;
}
