/*
 * lhn.h — C ABI of liblhn.so: the B200-native heatmap encode/decode hot path of
 * Runki2018/litehandnet (render + target-weight MSE loss + heatmap/SimDR decode + PCK/EPE/AUC).
 *
 * The reference has no FFI: its boundary is plain Python callables (SURVEY.md §8b).  Each entry
 * point below names the reference function(s) whose arithmetic it replaces (file:line relative to
 * the reference root); the Python mirror in litehandnet_b200/ keeps the reference's names and
 * signatures and calls these through ctypes with raw device pointers (INTEGRATION.md).
 *
 * Conventions (all entry points):
 *   - every pointer is a DEVICE pointer unless its comment says "host";
 *   - returns 0 on success, a negative LHN_E* code on a rejected call; never throws, never
 *     allocates, never synchronises the stream, keeps no global state; re-entrant and thread-safe
 *     for distinct streams/workspaces;
 *   - the caller owns every buffer, including the workspace whose size lhn_*_workspace_bytes gives;
 *   - `stream` is a cudaStream_t (NULL = legacy default stream);
 *   - a "plane" is one H x W slice; heatmap tensors are [B, C, H, W] with the plane contiguous,
 *     batch stride `stride_b` and channel stride `stride_c` in ELEMENTS (so channel-sliced views
 *     such as model_output[:, :num_joints] need no copy).  C = S*K for the stacked hourglass shape
 *     [B, S, K, H, W]; joint k of stack s is channel s*K + k.
 */
#ifndef LHN_H_
#define LHN_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LHN_API __attribute__((visibility("default")))

typedef void* lhn_stream_t; /* cudaStream_t */

/* error codes */
#define LHN_OK 0
#define LHN_EINVAL (-1)      /* bad shape / null pointer / bad enum */
#define LHN_EDTYPE (-2)      /* unsupported dtype */
#define LHN_EALIGN (-3)      /* pointer not aligned as required */
#define LHN_EWORKSPACE (-4)  /* workspace too small */
#define LHN_ECUDA (-5)       /* launch failed; see lhn_last_cuda_error() */

/* element types of heatmaps / vectors */
#define LHN_F32 0
#define LHN_BF16 1
#define LHN_F16 2
#define LHN_F64 3 /* metrics inputs only */

/* argmax masking convention (SURVEY §8a A1-A4) */
#define LHN_MASK_NONE 0 /* A4: result_parser.py:76-90, SPheatmapParser.py:44-56 (topk k=1) */
#define LHN_MASK_ZERO 1 /* A1/A3: evaluation.py:62-89, transforms.py:47-75 (coords*0 if max<=0) */
#define LHN_MASK_NEG1 2 /* A2: top_down_eval.py:199-231 (coords=-1 if max<=0) */

/* sub-pixel refinement (SURVEY §8a D1-D6) */
#define LHN_REFINE_NONE 0
#define LHN_REFINE_OFFSET_HALF 1 /* D1: heatmap_post_processing.py:6-33 (+-0.25 clamped, then +0.5) */
#define LHN_REFINE_OFFSET 2      /* D2: SPheatmapParser.py:140-167, HeatmapParser.py:197-223 */
#define LHN_REFINE_SIGN 3        /* D3: top_down_eval.py:440-452 (guarded, sign(0)=0) */
#define LHN_REFINE_SIGN_ROUND 4  /* D4: transforms.py:18-44 (px=floor(x+0.5)) */
#define LHN_REFINE_DARK 5        /* D5: top_down_eval.py:233-272,338-372,433-439 (f32 blur) */
#define LHN_REFINE_DARK_LEGACY 6 /* D6: heatmap_post_processing.py:35-91 (f64 blur, +1e-6) */
#define LHN_REFINE_DARK_UDP 7    /* D7: post_dark_udp, top_down_eval.py:274-335 (reflect-101 blur of the whole plane,
                                    clip [0.001, 50], log, edge-padded 3x3 stencil, (H + eps I)^-1 in f64); use with
                                    use_udp = 1 and LHN_MASK_NEG1 as keypoints_from_heatmaps(use_udp=True) does */

/* heatmap -> image coordinates (SURVEY §8a T1-T2) */
#define LHN_XFORM_NONE 0
#define LHN_XFORM_CENTER_SCALE 1 /* T1: post_transforms.py:6-48 transform_preds */
#define LHN_XFORM_SCALE 2        /* T2: coords * (scale_x, scale_y) — SPheatmapParser.py:203,
                                    result_parser.py:248, evaluation.py:34-36 */

/* loss reductions (SURVEY §8a L1-L3) */
#define LHN_LOSS_NONE 0
#define LHN_LOSS_DISTANCE 1         /* L1: DistanceLoss L2 balance=False, heatmapLoss.py:242-265 */
#define LHN_LOSS_DISTANCE_BALANCE 2 /* L2: DistanceLoss L2 balance=True */
#define LHN_LOSS_JOINTS_MSE 3       /* L3: JointsDistanceLoss mse, heatmapLoss.py:195-225 */

/* lhn_decode_params.flags */
#define LHN_FLAG_OVERLAP_PREVIOUS 1 /* This launch touches no buffer (inputs, outputs, workspace) that the previous
                                       launch on the same stream writes: it may begin while that launch is still
                                       draining (programmatic dependent launch), which hides the ~10 us launch gap
                                       of back-to-back steps over rotating buffers.  It is still ordered after
                                       every EARLIER launch: an overlapped launch lets its own successor in only
                                       after its predecessor has completed, so a launch never runs beside the one
                                       two back and two rotating buffer sets are enough.  Stream order is unchanged
                                       for everything launched afterwards. */

#define LHN_FLAG_ACCUMULATE_LOSS 2  /* lhn_fused_render_loss_decode adds the finalised loss into loss[0] instead of
                                       overwriting it: the epoch sum of train_one_epoch's loss_dict['sum'] += v
                                       (train/topdown_trainer.py:82-84) kept on the device, all-reduced once per
                                       epoch (train/distributed_utils.py:65-76) instead of once per step. */
#define LHN_FLAG_SPARE_SMS(n) (((n) & 0xff) << 8) /* leave n SMs to other work: the persistent kernel otherwise
                                       fills every SM (216 KB of shared memory each), so a concurrent NCCL kernel —
                                       the 32-byte all-reduce of the previous step's loss sums — could not start
                                       before it ends.  The kernel is HBM-bound: 4 of 148 SMs cost < 1 %. */

#define LHN_LOSS_MAX_TENSORS 8
#define LHN_MAX_TAPS 31
#define LHN_MAX_STACKS 8

/* ---- cross-GPU exchange inside the kernel (NVLink / NVSwitch peer memory) ----------------------------------------
 * The path's only cross-rank data are a few hundred counters or four loss sums per step (SURVEY.md §8e).  A
 * persistent kernel that owns every SM leaves no room for a concurrent NCCL kernel, so the per-step all-reduce is
 * done by the kernel itself: the last CTA of the grid stores this rank's block into every peer's MAILBOX (plain
 * stores to peer-mapped memory, then a release flag), waits for the peers' flags in its own mailbox and adds the
 * blocks in rank order — integers bit-exact, doubles in one fixed order, identical on every rank.
 * Each rank owns one mailbox of LHN_XCH_MAILBOX_BYTES, zeroed once, mapped into every peer (symmetric memory or
 * cudaIpc).  `seq` is the step number (1, 2, 3, ... — the same on every rank for the same step; slots rotate with it,
 * LHN_XCH_SLOTS deep, which the launch ordering of LHN_FLAG_OVERLAP_PREVIOUS makes sufficient).  A peer that does not
 * arrive within timeout_ms sets *status = 1 and the kernel finishes with the local block only. */
#define LHN_XCH_MAX_RANKS 8
#define LHN_XCH_SLOTS 4
#define LHN_XCH_PAYLOAD_BYTES 8192
#define LHN_XCH_CTRL_BYTES 4096   /* flags u32 [slots][ranks], then the launch ticket */
#define LHN_XCH_MAILBOX_BYTES (LHN_XCH_SLOTS * LHN_XCH_MAX_RANKS * LHN_XCH_PAYLOAD_BYTES + LHN_XCH_CTRL_BYTES)
typedef struct {
  void* mailbox[LHN_XCH_MAX_RANKS]; /* mailbox of rank r as mapped into THIS process; mailbox[rank] is the local one */
  int32_t world, rank;
  uint32_t seq;                     /* step number >= 1 */
  uint32_t timeout_ms;              /* 0 = 2000 */
  int32_t* status;                  /* device int32 (local), or NULL */
  /* lhn_decode_heatmap_pck_xch / lhn_exchange_flush only — the pipelined counter exchange: */
  void* prev_block;                 /* per-step block of the PREVIOUS exchanging launch (this launch publishes it), or NULL */
  uint32_t prev_seq;                /* ... and that launch's step number */
  uint32_t prev2_seq;               /* step number of the launch before that */
  void* prev2_block;                /* ... and its block (published by the previous launch; this launch adds every
                                       rank's copy into the totals and zeroes it), or NULL */
} lhn_exchange;

/* Decode parameters. */
typedef struct {
  int32_t mask_mode;  /* LHN_MASK_* */
  int32_t refine;     /* LHN_REFINE_* */
  int32_t transform;  /* LHN_XFORM_* */
  int32_t use_udp;    /* T1: divide by (W-1),(H-1) instead of W,H (post_transforms.py:37-39) */
  int32_t blur_ksize; /* DARK Gaussian kernel size (odd, 3..31): 11 for D5, 19 for D6 */
  int32_t flags;      /* LHN_FLAG_* (0 = none) */
  float scale_x, scale_y;         /* LHN_XFORM_SCALE factors */
  double taps[LHN_MAX_TAPS];      /* cv2.getGaussianKernel(blur_ksize, 0) in double; host fills it
                                     with lhn_gaussian_taps() */
} lhn_decode_params;

/* Render + loss parameters (fused op and lhn_render_targets). */
typedef struct {
  int32_t loss_mode;    /* LHN_LOSS_* (LHN_LOSS_NONE = decode only) */
  int32_t unbiased;     /* 1: R1 MSRA sub-pixel full-plane Gaussian, generateTarget.py:100-123;
                           0: R2 MSRA integer-centre (2*3*sigma+1)^2 patch, generateTarget.py:124-154;
                           2: UDP GaussianHeatmap — integer patch position, sub-pixel centre inside it,
                              feat_stride = (image_size-1)/(heatmap_size-1), generateTarget.py:162-243 */
  int32_t num_stacks;   /* S >= 1 (R3: sigma list -> [B,S,K,H,W], generateTarget.py:252-268) */
  int32_t reserved;
  float image_w, image_h;        /* cfg image_size; feat_stride = image_size / [W, H] */
  float pos_value;               /* DistanceLoss `value` (0.5): positives are target > value */
  float sigma[LHN_MAX_STACKS];   /* per stack */
} lhn_render_params;

/* ---- host helpers ------------------------------------------------------------------------- */

/* Library/ABI version (major*100 + minor). */
LHN_API int lhn_version(void);
/* Text of the last CUDA error seen by this thread's failed launch (host pointer, static storage). */
LHN_API const char* lhn_last_cuda_error(void);
/* Fill taps[0..ksize) with cv2.getGaussianKernel(ksize, sigma<=0, CV_64F) (host pointer). */
LHN_API int lhn_gaussian_taps(int ksize, double* taps);

/* Which code path the last K1 call of THIS host thread launched (lhn_decode_heatmap, lhn_decode_heatmap_pck,
 * lhn_fused_render_loss_decode and their _xch variants).  Cleared on entry to every such call that reaches the
 * launcher, filled after a successful launch; a rejected call leaves path == 0.  For tests that must know which
 * instantiation, team geometry and copy path a shape takes; nothing in the library reads it. */
typedef struct {
  int32_t path;            /* 0 = nothing launched / rejected, 1 = persistent team kernel, 2 = CTA-per-plane kernel */
  int32_t dtype;           /* LHN_F32 / LHN_BF16 / LHN_F16 */
  int32_t flip, loss, counters;   /* flip plane present, loss fused, PCK/AUC/EPE counters fused (0/1) */
  int32_t wc;              /* compile-time plane width of the instantiation (team: 128/64/56/32/16; CTA: 128), 0 = run-time size */
  int32_t twc;             /* compile-time team width in warps, 0 = run-time */
  int32_t ks;              /* compile-time DARK window: 11, or 0 = run-time */
  int32_t team_warps, nteams, stages, sweeper_tables;   /* team kernel geometry (0 on the CTA-per-plane kernel) */
  int32_t use_tma;         /* planes loaded by TMA bulk copies (1) or element copies (0) */
  int32_t ctas;            /* grid size */
  int32_t stagger_ns;      /* delay between the first loads of consecutive teams (team kernel) */
} lhn_k1_launch_info;
LHN_API int lhn_k1_last_launch(lhn_k1_launch_info* out);

/* Which code path the last SimDR call of THIS host thread launched (lhn_render_simdr(_f64sigma), lhn_decode_simdr(_flags),
 * lhn_simdr_smoothl1, lhn_simdr_smoothl1_backward, lhn_simdr_heads_loss(_f32)).  Cleared on entry to each of them,
 * filled after a successful launch; a rejected call leaves family == 0.  For tests that must know which kernel and
 * geometry a shape takes; nothing in the library reads it. */
typedef struct {
  int32_t family;          /* 0 = nothing launched / rejected, 1 render, 2 decode, 3 loss, 4 backward, 5 heads */
  int32_t path;            /* render: 1 windowed (warp per joint), 2 plain (CTA per joint);
                              decode: 1 TMA ring, 2 pair scan, 3 scalar scan, 4 NMS;
                              loss: 1 joint-per-warp + cluster finalise, 2 rows + cluster finalise,
                                    3 rows + one-block finalise, 4 rows + single-thread loop (K > 1024);
                              backward, heads: 1 */
  int32_t dtype;           /* LHN_F32 / LHN_BF16 / LHN_F16 of the vectors (heads: LHN_BF16 operands) */
  int32_t warps;           /* warps per CTA of the main kernel */
  int32_t stages;          /* decode ring / heads mbarrier ring stages, else 0 */
  int32_t ctas;            /* grid size of the main kernel */
  int32_t vec_x, vec_y;    /* 128-bit path over the x / y vectors (backward per vector; loss: one flag for both) */
  int32_t bn;              /* heads: N tile width, else 0 */
} lhn_simdr_launch_info;
LHN_API int lhn_simdr_last_launch(lhn_simdr_launch_info* out);

/* ---- K1: heatmap decode, optionally fused with target render + masked MSE partial sums -------
 *
 * Replaces, in ONE pass over each heatmap plane:
 *   decode : _get_max_preds / get_coordinates_from_heatmap / get_max_preds / topk(k=1) (A1-A4),
 *            the +-0.25 rules and DARK (D1-D6), flip_back + averaging (F1/F2: transforms.py:78-92),
 *            transform_preds (T1) or the plain scale (T2);
 *   render : TopDownGenerateTarget._msra_generate_target (R1/R2/R3) evaluated in registers;
 *   loss   : the per-plane sums of DistanceLoss / JointsDistanceLoss (L1-L3) against that target.
 *
 * hm            [B, C, H, W] dtype (C = S*K), strides in elements.
 * hm_flip       same layout or NULL; when given the kernel decodes
 *               (hm[b,c] + hm_flip[b, s*K+flip_index[k], :, ::-1]) * 0.5 (f32).
 * flip_index    int32 [K] or NULL (identity).
 * center, scale f32 [B,2] (T1) or NULL.
 * out_hm        f32 [B*C, 3] (x, y, maxval) in heatmap space, or NULL.
 * out_kpts      f32 [B*C, 3] (X, Y, maxval) after the transform, or NULL.
 * out_idx       int32 [B*C] first-maximal flat index (NaN counts as maximal), or NULL.
 * Render/loss inputs (ignored when rp == NULL or rp->loss_mode == LHN_LOSS_NONE):
 * joints        f32 [B, K, joints_stride] (x, y in image pixels in columns 0,1).
 * vis           f32 [B, K, vis_stride] (column 0 = visibility / weight).
 * out_weight    f32 [B*C] target_weight after the visibility rule, or NULL.
 * partials      f64 [B*C, 4] per-plane (w^p*S_pos, w^p*S_neg, N_pos, H*W); reduce with
 *               lhn_loss_reduce + lhn_loss_finalize (or use lhn_fused_render_loss_decode below).  The loss is taken on `hm` (not the flip
 *               average), as the training loss is.
 */
LHN_API int lhn_decode_heatmap(const void* hm, const void* hm_flip, const int32_t* flip_index,
                               int dtype, int64_t B, int K, int H, int W,
                               int64_t stride_b, int64_t stride_c,
                               int64_t flip_stride_b, int64_t flip_stride_c,
                               const float* center, const float* scale,
                               const lhn_decode_params* dp,
                               float* out_hm, float* out_kpts, int32_t* out_idx,
                               const lhn_render_params* rp,
                               const float* joints, int joints_stride,
                               const float* vis, int vis_stride,
                               float* out_weight, double* partials,
                               lhn_stream_t stream);

/* ---- the headline step in ONE launch ------------------------------------------------------------
 * lhn_decode_heatmap (with the fused render + loss) followed by lhn_loss_reduce and
 * lhn_loss_finalize, as a single kernel: every team of the persistent kernel keeps its own f64
 * loss sums; the last team of a CTA adds the CTA's teams in team order and publishes one row, the
 * last CTA adds the rows in a fixed order (bitwise reproducible for a given shape and device) and
 * finalises the loss.  Replaces the same reference calls as lhn_decode_heatmap +
 * DistanceLoss.forward / JointsDistanceLoss.forward (heatmapLoss.py:242-265, :195-225).
 *
 * workspace  device buffer of lhn_fused_workspace_bytes(B, K, num_stacks) bytes; zero it ONCE
 *            (cudaMemsetAsync) before the first call — every call leaves it zeroed.  One workspace
 *            per concurrently running stream.
 * partials   optional here (NULL = do not write the per-plane sums).
 * sums       f64 [4] = (S_pos, S_neg, N_pos, numel) of the whole call, or NULL: all-reduce these across
 *            ranks and call lhn_loss_finalize for a batch-sharded loss with global counts.
 * loss       f32 [1] = loss_scale * f(sums) as lhn_loss_finalize (sum_reduction as there), or NULL.
 * Shapes outside the persistent kernel's envelope (a plane pair larger than half the shared memory)
 * run the same arithmetic as three launches; results are identical. */
LHN_API int64_t lhn_fused_workspace_bytes(int64_t B, int K, int num_stacks);
LHN_API int lhn_fused_render_loss_decode(const void* hm, const void* hm_flip,
                                         const int32_t* flip_index, int dtype, int64_t B, int K, int H,
                                         int W, int64_t stride_b, int64_t stride_c,
                                         int64_t flip_stride_b, int64_t flip_stride_c,
                                         const float* center, const float* scale,
                                         const lhn_decode_params* dp, float* out_hm, float* out_kpts,
                                         int32_t* out_idx, const lhn_render_params* rp,
                                         const float* joints, int joints_stride, const float* vis,
                                         int vis_stride, float* out_weight, double* partials,
                                         void* workspace, int64_t workspace_bytes, double* sums,
                                         int sum_reduction, float loss_scale, float* loss,
                                         lhn_stream_t stream);

/* The same with the loss sums all-reduced over the ranks INSIDE the kernel (lhn_exchange, above): `sums` and `loss`
 * then hold the batch-GLOBAL (S_pos, S_neg, N_pos, numel) and the loss a single process would compute on the
 * concatenated batch (global N_pos, loss/heatmapLoss.py:253-258) — one launch per step, no NCCL call. */
LHN_API int lhn_fused_render_loss_decode_xch(const void* hm, const void* hm_flip,
                                         const int32_t* flip_index, int dtype, int64_t B, int K, int H,
                                         int W, int64_t stride_b, int64_t stride_c,
                                         int64_t flip_stride_b, int64_t flip_stride_c,
                                         const float* center, const float* scale,
                                         const lhn_decode_params* dp, float* out_hm, float* out_kpts,
                                         int32_t* out_idx, const lhn_render_params* rp,
                                         const float* joints, int joints_stride, const float* vis,
                                         int vis_stride, float* out_weight, double* partials,
                                         void* workspace, int64_t workspace_bytes, double* sums,
                                         int sum_reduction, float loss_scale, float* loss,
                                         const lhn_exchange* xch, lhn_stream_t stream);

/* ---- loss against an explicit target tensor (the un-fused drop-in) ----------------------------
 * DistanceLoss.forward(output, target, target_weight) / JointsDistanceLoss.forward
 * (heatmapLoss.py:242-265, :195-225).  output/target [P, HW] contiguous planes (any leading
 * dims flattened), weight f32 [P].  Writes partials f64 [P,4] as above (pos = target > pos_value).
 */
LHN_API int lhn_loss_partials(const void* output, const void* target, const float* weight,
                              int dtype, int64_t n_planes, int64_t plane_elems, int loss_mode,
                              float pos_value, double* partials, lhn_stream_t stream);

/* Deterministic fixed-order reduction of partials[P,4] to sums[4] = (S_pos, S_neg, N_pos, numel)
 * in f64.  `accumulate` != 0 adds into sums (multi-tensor losses), else overwrites. */
LHN_API int lhn_loss_reduce(const double* partials, int64_t n_planes, double* sums, int accumulate,
                            lhn_stream_t stream);

/* loss[0] (f32) = scale * f(sums):
 *   LHN_LOSS_DISTANCE          (S_pos+S_neg)/numel                       (reduction='mean')
 *   LHN_LOSS_DISTANCE_BALANCE  0.1*S_pos/(N_pos+1) + S_neg/(N_neg+1)
 *   LHN_LOSS_JOINTS_MSE        0.5*(S_pos+S_neg)/numel
 * sum_reduction != 0 multiplies by numel (reduction='sum').  `accumulate` adds into loss[0]. */
LHN_API int lhn_loss_finalize(const double* sums, int loss_mode, int sum_reduction, float scale,
                              float* loss, int accumulate, lhn_stream_t stream);

/* ---- backward of the losses (SURVEY §8f rank 1: lets the drop-in losses sit in train_one_epoch,
 * train/topdown_trainer.py:68-87, behind torch.autograd.Function) ---------------------------------
 * grad[p,e] = grad_out[0] * scale * coef(p,e) * (output[p,e] - target[p,e]), coef from the forward's
 * f64 sums (S_pos, S_neg, N_pos, numel):
 *   LHN_LOSS_DISTANCE          2 w / numel
 *   LHN_LOSS_DISTANCE_BALANCE  2 w * 0.1/(N_pos+1) where target > pos_value, else 2 w / (N_neg+1)
 *   LHN_LOSS_JOINTS_MSE        w^2 / numel
 * (x numel when sum_reduction != 0) — the derivative of DistanceLoss.forward / JointsDistanceLoss.forward
 * (heatmapLoss.py:242-265, :195-225) as torch autograd computes it.  grad_out: f32 [1] device pointer
 * (the upstream gradient of the scalar loss) or NULL (= 1).  grad: same dtype and [P, HW] layout as
 * output.  One pass: reads output and target once, writes grad once. */
LHN_API int lhn_loss_backward(const void* output, const void* target, const float* weight, int dtype,
                              int64_t n_planes, int64_t plane_elems, int loss_mode, float pos_value,
                              const double* sums, int sum_reduction, float scale, const float* grad_out,
                              void* grad, lhn_stream_t stream);

/* The same with the target rendered in-kernel from the joints (the backward of the fused entry):
 * hm [B, S*K, H, W] with element strides as lhn_decode_heatmap, rp->loss_mode selects the loss;
 * grad is contiguous [B, S*K, H, W] of the heatmap dtype. */
LHN_API int lhn_render_loss_backward(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                     int64_t stride_b, int64_t stride_c, const lhn_render_params* rp,
                                     const float* joints, int joints_stride, const float* vis,
                                     int vis_stride, const double* sums, int sum_reduction, float scale,
                                     const float* grad_out, void* grad, lhn_stream_t stream);

/* The fused loss AND its gradient in one pass over hm (one read, one write): the same inputs as
 * lhn_render_loss_backward, plus what lhn_fused_render_loss_decode reports for the loss — out_weight
 * [B*S*K] (optional), sums f64 [4] = (S_pos, S_neg, N_pos, numel) (optional), loss f32 [1] (optional,
 * as lhn_loss_finalize with sum_reduction and loss_scale).  N_pos is counted from the joints before the
 * first gradient element is written, so it equals the fused forward's.  grad (contiguous [B, S*K, H, W],
 * heatmap dtype) is d loss / d hm for an upstream gradient grad_scale[0] (f32 [1] device pointer, NULL = 1):
 * coefficient (float)(c * loss_scale * grad_scale[0]) — bit-identical to lhn_render_loss_backward run
 * with grad_out = grad_scale on these sums.  used_scale (f32 [1], optional) receives the value assumed.
 * workspace: lhn_render_loss_grad_workspace_bytes(B, K, num_stacks) bytes, 16-byte aligned, zero before
 * the first call and left zero.  One cooperative launch (a grid-wide barrier after the count). */
LHN_API int64_t lhn_render_loss_grad_workspace_bytes(int64_t B, int K, int num_stacks);
LHN_API int lhn_render_loss_grad(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                 int64_t stride_b, int64_t stride_c, const lhn_render_params* rp,
                                 const float* joints, int joints_stride, const float* vis, int vis_stride,
                                 float* out_weight, void* workspace, int64_t workspace_bytes, double* sums,
                                 int sum_reduction, float loss_scale, float* loss, const float* grad_scale,
                                 float* used_scale, void* grad, lhn_stream_t stream);

/* The backward of lhn_render_loss_grad: if grad_out[0] (NULL = 1) is bitwise equal to used_scale[0], the
 * gradient already in `grad` is the answer and nothing is written; otherwise grad is overwritten exactly
 * as lhn_render_loss_backward(grad_out) would.  recomputed (int32 [1], optional) receives 0 or 1.  One
 * launch of about one wave either way. */
LHN_API int lhn_render_loss_backward_cond(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                          int64_t stride_b, int64_t stride_c, const lhn_render_params* rp,
                                          const float* joints, int joints_stride, const float* vis,
                                          int vis_stride, const double* sums, int sum_reduction, float scale,
                                          const float* grad_out, const float* used_scale, int32_t* recomputed,
                                          void* grad, lhn_stream_t stream);

/* KLDiscretLoss backward (centernet_simdr_loss.py:27-39): grad_x[b,j,i] = grad_out * scale *
 * SmoothL1'(out_x - tgt_x) * mean_b(weight[b,j]) / (K * B * Lx), likewise grad_y.  workspace:
 * lhn_simdr_backward_workspace_bytes(K) bytes. */
LHN_API int64_t lhn_simdr_backward_workspace_bytes(int K);
LHN_API int lhn_simdr_smoothl1_backward(const void* out_x, const void* out_y, const void* tgt_x,
                                        const void* tgt_y, const float* weight, int dtype, int64_t B,
                                        int K, int Lx, int Ly, float scale, const float* grad_out,
                                        void* workspace, int64_t workspace_bytes, void* grad_x,
                                        void* grad_y, lhn_stream_t stream);

/* ---- render (the un-fused drop-in; write-bound) -----------------------------------------------
 * TopDownGenerateTarget (generateTarget.py:100-154,245-300) for a batch: target f32
 * [B, S, K, H, W] contiguous, target_weight f32 [B, S, K]. */
LHN_API int lhn_render_targets(const float* joints, int joints_stride, const float* vis,
                               int vis_stride, int64_t B, int K, int H, int W,
                               const lhn_render_params* rp, float* target, float* target_weight,
                               lhn_stream_t stream);

/* GenerateSimDR._generate_sa_simdr (generate_simder.py:9-31): simdr_x f32 [B,K,Lx],
 * simdr_y f32 [B,K,Ly]; Lx = int(image_w*k), Ly = int(image_h*k).  The Gaussian's denominator is
 * 2.f * sigma * sigma in f32 arithmetic. */
LHN_API int lhn_render_simdr(const float* joints, int joints_stride, const float* vis,
                             int vis_stride, int64_t B, int K, int Lx, int Ly, float split_ratio,
                             float sigma, float* simdr_x, float* simdr_y, lhn_stream_t stream);
/* The same with sigma as a double, bit for bit the reference: it divides by the Python float
 * 2 * sigma ** 2, formed in f64 and rounded to f32 once, and this entry point forms
 * (float)(2.0 * sigma * sigma) the same way.  An f32 sigma cannot reproduce that denominator: for about
 * half of all sigma (1.3, 2.1, 2.7, 3.3, ...) 2.f * s * s is one f32 ulp away from it. */
LHN_API int lhn_render_simdr_f64sigma(const float* joints, int joints_stride, const float* vis,
                                      int vis_stride, int64_t B, int K, int Lx, int Ly, float split_ratio,
                                      double sigma, float* simdr_x, float* simdr_y, lhn_stream_t stream);

/* ---- K2: SimDR --------------------------------------------------------------------------------
 * keypoints_from_simdr (top_down_eval.py:466-500): x = argmax(x_vec)/k, y = argmax(y_vec)/k,
 * score = (max_x+max_y)/2, transform_preds with output_size [Lx//k, Ly//k] (center==NULL: none).
 * With `nms` != 0 applies ResultParser.vector_nms (result_parser.py:61-74) first and, when
 * `ranges` (int32 [B,4] = x1,x2,y1,y2 bins) is given, the bbox mask of
 * get_coordinates_from_vectors (result_parser.py:92-129) — without mutating the inputs.
 * out f32 [B*K,3]; out_idx int32 [B*K,2] or NULL. */
LHN_API int lhn_decode_simdr(const void* x_vec, const void* y_vec, int dtype, int64_t B, int K,
                             int Lx, int Ly, int split_ratio, const float* center,
                             const float* scale, int nms, const int32_t* ranges, float* out,
                             int32_t* out_idx, lhn_stream_t stream);
/* The same with `flags` (LHN_FLAG_OVERLAP_PREVIOUS: this launch shares no buffer with the previous launch on the
 * stream — e.g. a loop over rotating batches — and may start while that one drains; honoured by the
 * persistent ring kernel, ignored by the small-batch / NMS path). */
LHN_API int lhn_decode_simdr_flags(const void* x_vec, const void* y_vec, int dtype, int64_t B, int K,
                                   int Lx, int Ly, int split_ratio, const float* center,
                                   const float* scale, int nms, const int32_t* ranges, float* out,
                                   int32_t* out_idx, int flags, lhn_stream_t stream);

/* KLDiscretLoss.forward (centernet_simdr_loss.py:27-39): per-joint SmoothL1(beta=1) sums.
 * out/target [B,K,L*]; weight f32 [B,K]; joint_sums f64 [K,3] = (sum_x, sum_y, sum_w) must be
 * zeroed by the caller (the kernel adds per-(b,k) partials in a fixed order per joint).
 * loss[0] = (1/K) sum_j (sum_x/(B*Lx) + sum_y/(B*Ly)) * (sum_w/B). */
LHN_API int64_t lhn_simdr_loss_workspace_bytes(int64_t B, int K);
LHN_API int lhn_simdr_smoothl1(const void* out_x, const void* out_y, const void* tgt_x,
                               const void* tgt_y, const float* weight, int dtype, int64_t B, int K,
                               int Lx, int Ly, void* workspace, int64_t workspace_bytes, float* loss,
                               lhn_stream_t stream);

/* DistanceLoss / JointsDistanceLoss against explicit target tensors in ONE launch, for n_tensors <= LHN_LOSS_MAX_TENSORS
 * (output, target, weight) triples at once (loss/heatmapLoss.py:195-265; SRHandNetLoss._forward_only_heatmap,
 * loss/loss.py:59-66: loss = sum_i loss_weights[i] * L2(outputs[i], targets[i], w[i])).
 * outputs[i] / targets[i]: n_planes[i] contiguous planes of plane_elems[i] elements, all of `dtype`; weights[i] f32
 * [n_planes[i]].  The arrays of pointers / sizes are HOST arrays.  sums (optional) f64 [n_tensors, 4] receives each
 * tensor's (S_pos, S_neg, N_pos, numel) for the backward; per_tensor_loss (optional) f32 [n_tensors]; loss f32 [1]
 * = scale * sum_i loss_weights[i] * loss_i (added to loss[0] when accumulate != 0).  workspace: zeroed once,
 * lhn_loss_mse_workspace_bytes() bytes, 16-byte aligned; the kernel leaves it ready for the next launch. */
LHN_API int64_t lhn_loss_mse_workspace_bytes(void);
LHN_API int lhn_loss_mse_multi(int n_tensors, const void* const* outputs, const void* const* targets,
                               const float* const* weights, const int64_t* n_planes, const int64_t* plane_elems,
                               const float* loss_weights, int dtype, int loss_mode, float pos_value,
                               int sum_reduction, float scale, void* workspace, int64_t workspace_bytes,
                               double* sums, float* per_tensor_loss, float* loss, int accumulate,
                               lhn_stream_t stream);

/* ---- the multi-scale loss with every scale's target rendered in-kernel ---------------------------------------------
 * SRHandNetLoss._forward_only_heatmap (loss/loss.py:59-66) from the joints: loss = scale * sum_i loss_weight_i *
 * f32(L_i), L_i = DistanceLoss / JointsDistanceLoss (heatmapLoss.py:195-265) of scale i's output against the target
 * lhn_render_targets would draw for it (rp->unbiased, rp->pos_value, rp->loss_mode and rp->image_w / image_h shared;
 * the scale's own H, W, sigma and feature stride; target_weight after the visibility rule of ITS plane size).  The
 * targets are never materialised.  All scales share joints f32 [B, K, joints_stride] and vis f32 [B, K, vis_stride]
 * (column 0); rp->num_stacks and rp->sigma are not read.  `scales` is a HOST array of n_scales <=
 * LHN_LOSS_MAX_TENSORS descriptors. */
typedef struct {
  const void* output;      /* [B, K, H, W] of `dtype`, planes contiguous, element strides stride_b / stride_c */
  void* grad;              /* backward, one pass: contiguous [B, K, H, W] of `dtype`, or NULL to skip this scale's
                              gradient; forward: unused */
  float* out_weight;       /* forward, one pass: f32 [B*K] target_weight of this scale, or NULL; backward: unused */
  int64_t stride_b, stride_c;
  int32_t H, W;
  float sigma;
  float loss_weight;       /* forward: the weight of this scale's term; backward: its gradient's scale; one pass:
                              both */
} lhn_loss_scale;

/* Forward, ONE launch: the grid dealing, fixed-order two-level reduction and last-CTA finalise of
 * lhn_loss_mse_multi (bitwise reproducible for a given shape and device).  sums (optional) f64 [n_scales, 4] =
 * (S_pos, S_neg, N_pos, numel) per scale, which the backward needs; per_scale_loss (optional) f32 [n_scales] = L_i;
 * loss (optional) f32 [1].  workspace: lhn_render_loss_multi_workspace_bytes() bytes, 16-byte aligned, zeroed once
 * and left zero (the same size and contract as lhn_loss_mse_multi's, so one buffer may serve both on one stream). */
LHN_API int64_t lhn_render_loss_multi_workspace_bytes(void);
LHN_API int lhn_render_loss_multi(int n_scales, const lhn_loss_scale* scales, int dtype, int64_t B, int K,
                                  const lhn_render_params* rp, const float* joints, int joints_stride,
                                  const float* vis, int vis_stride, int sum_reduction, float scale,
                                  void* workspace, int64_t workspace_bytes, double* sums, float* per_scale_loss,
                                  float* loss, lhn_stream_t stream);
/* Backward, ONE launch writing every scale's gradient (scales with grad == NULL are skipped): bit for bit
 * lhn_render_loss_backward on scale i with sums + 4 i and scale = loss_weight_i, for an upstream gradient
 * grad_out[0] (f32 [1] device pointer, NULL = 1). */
LHN_API int lhn_render_loss_backward_multi(int n_scales, const lhn_loss_scale* scales, int dtype, int64_t B, int K,
                                           const lhn_render_params* rp, const float* joints, int joints_stride,
                                           const float* vis, int vis_stride, const double* sums, int sum_reduction,
                                           const float* grad_out, lhn_stream_t stream);

/* The loss AND every wanted scale's gradient in one pass over the outputs (one read, one write): the inputs of
 * lhn_render_loss_multi, and it writes what that entry point writes — out_weight per scale, sums [n_scales, 4] with
 * N_pos and numel bit for bit its values (S_pos, S_neg may differ in the last bits), per_scale_loss, loss.  Scale i's
 * grad (NULL = not wanted; the scale is still read for its loss) receives d loss / d output for an upstream gradient
 * grad_scale[0] (f32 [1] device pointer, NULL = 1), loss_weight_i being both the term's weight and the gradient's
 * scale: bit for bit what lhn_render_loss_backward_multi writes from these sums with grad_out = grad_scale.  `scale`
 * multiplies the reported loss only, as in lhn_render_loss_multi.  used_scale (f32 [1], optional) receives the
 * upstream value assumed.  Two launches: the balanced loss's N_pos per scale is counted from the joints alone (skipped
 * for the other modes and for pos_value >= 1), then one warp per plane streams every scale behind that count.
 * workspace: lhn_render_loss_grad_multi_workspace_bytes(n_scales, B, K) bytes (0 for invalid arguments), 16-byte
 * aligned, zero before the first call and left zero; bitwise reproducible for a given shape and device. */
LHN_API int64_t lhn_render_loss_grad_multi_workspace_bytes(int n_scales, int64_t B, int K);
LHN_API int lhn_render_loss_grad_multi(int n_scales, const lhn_loss_scale* scales, int dtype, int64_t B, int K,
                                       const lhn_render_params* rp, const float* joints, int joints_stride,
                                       const float* vis, int vis_stride, int sum_reduction, float scale,
                                       void* workspace, int64_t workspace_bytes, double* sums, float* per_scale_loss,
                                       float* loss, const float* grad_scale, float* used_scale, lhn_stream_t stream);
/* The backward of lhn_render_loss_grad_multi: lhn_render_loss_backward_multi's arguments plus used_scale (required)
 * and recomputed (int32 [1], optional).  If grad_out[0] (NULL = 1) is bitwise equal to used_scale[0], the gradients
 * already in the scales' grad buffers are the answer and nothing is written (recomputed = 0); otherwise every wanted
 * gradient is rewritten exactly as lhn_render_loss_backward_multi would (recomputed = 1).  With no gradient wanted it
 * launches nothing. */
LHN_API int lhn_render_loss_backward_multi_cond(int n_scales, const lhn_loss_scale* scales, int dtype, int64_t B,
                                                int K, const lhn_render_params* rp, const float* joints,
                                                int joints_stride, const float* vis, int vis_stride,
                                                const double* sums, int sum_reduction, const float* grad_out,
                                                const float* used_scale, int32_t* recomputed, lhn_stream_t stream);

/* ---- SimDRLoss with its two nn.Linear heads fused (centernet_simdr_loss.py:42-69) -------------------------------
 * pred_x | pred_y = heatmap.flatten(2) @ [Wx ; Wy]^T + [bx ; by], then KLDiscretLoss (:27-39) — ONE tcgen05 kernel:
 * the predictions stay in tensor memory, the epilogue takes SmoothL1 against the targets and row-reduces it; a
 * second tiny launch adds the partial sums in a fixed order and applies the joint weights.
 *
 * fp32 parity: operands are passed as bf16 pairs x = hi + lo made by lhn_split_bf16 (x f32 [n], n % 4 == 0,
 * 16-byte aligned; hi / lo bf16 [n]); the kernel issues lo*hi + hi*lo + hi*hi into one fp32 accumulator.
 *   a_hi / a_lo  bf16 [B*K, Kd]   the heatmaps flattened (Kd = H*W, a multiple of 64)
 *   w_hi / w_lo  bf16 [Lx+Ly, Kd] rows 0..Lx-1 = x_shared_decoder.weight, then y_shared_decoder.weight
 *   bias f32 [Lx+Ly]; target_x f32 [B,K,Lx], target_y f32 [B,K,Ly]; weight f32 [B,K]; (Lx+Ly) % 64 == 0, Lx % 4 == 0
 *   loss f32 [1];  dpred (optional) f32 [B*K, Lx+Ly] = clamp(pred - target, -1, 1) = d SmoothL1 / d pred for the
 *   backward;  pred (optional) f32 [B*K, Lx+Ly] = the predictions (inference).  All pointers 16-byte aligned. */
LHN_API int lhn_split_bf16(const float* x, int64_t n, void* hi, void* lo, lhn_stream_t stream);
LHN_API int64_t lhn_simdr_heads_workspace_bytes(int64_t B, int K, int Lx, int Ly);
/* lhn_simdr_heads_loss straight from the f32 heatmaps [B,K,H*W]: the bf16 split of the heatmaps goes into the workspace
 * (lhn_simdr_heads_f32_workspace_bytes bytes, 256-byte aligned) as a first streaming launch — one call per step. */
LHN_API int64_t lhn_simdr_heads_f32_workspace_bytes(int64_t B, int K, int Kd, int Lx, int Ly);
LHN_API int lhn_simdr_heads_loss_f32(const float* heatmap, const void* w_hi, const void* w_lo, const float* bias,
                                     const float* target_x, const float* target_y, const float* weight, int64_t B,
                                     int K, int Kd, int Lx, int Ly, void* workspace, int64_t workspace_bytes,
                                     float* loss, float* dpred, float* pred, lhn_stream_t stream);
LHN_API int lhn_simdr_heads_loss(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo,
                                 const float* bias, const float* target_x, const float* target_y,
                                 const float* weight, int64_t B, int K, int Kd, int Lx, int Ly, void* workspace,
                                 int64_t workspace_bytes, float* loss, float* dpred, float* pred,
                                 lhn_stream_t stream);

/* ---- K3: metrics ------------------------------------------------------------------------------
 * _calc_distances + _distance_acc (top_down_eval.py:12-62) as shardable counters.
 * pred [N,K,pred_stride] / gt [N,K,gt_stride] (x,y in columns 0,1), dtype f32 or f64 each;
 * mask uint8 [N,K]; normalize [N,2] (norm_dtype) or NULL -> the constant `norm_const` on both
 * axes.  The distance is computed in f64 unless pred, gt and normalize are all f32 (numpy
 * promotion), rounded to f32 and compared with (float)thr[t].
 * counters int64 [(T+2)*K]: hits[t][k] (t<T), valid[k], dist_fix[k] = sum of valid distances
 * in 2^-20 fixed point.  ADDS into counters (zero them first; all-reduce them across ranks
 * with ncclSum for the sharded evaluation — SURVEY §8e). */
LHN_API int lhn_pck_accumulate(const void* pred, int pred_dtype, int pred_stride, const void* gt,
                               int gt_dtype, int gt_stride, const uint8_t* mask,
                               const void* normalize, int norm_dtype, double norm_const, int64_t N,
                               int K, const float* thr /* host, T floats */, int T,
                               int64_t* counters, lhn_stream_t stream);

/* Kpt2dDataset._report_metric's final ratios (datasets/base_dataset.py:193-261) from the fused counter block of
 * lhn_decode_heatmap_pck / MetricAccumulator, on the device: no device->host copy or sync per metric call.
 * counters int64 [(auc_steps+5)*K] (after the cross-rank ncclSum, if sharded).
 * out f64 [3 + K]: out[0] = PCK = keypoint_pck_accuracy's avg_acc (top_down_eval.py:65-101: mean of the per-joint
 * hits/valid that are >= 0, numpy's pairwise summation order), out[1] = keypoint_auc (:167-196: sum_t avg_acc_t /
 * auc_steps), out[2] = EPE (:104-126, from the 2^-20 px fixed-point sum), out[3..3+K) = the per-joint PCK
 * accuracies (-1 where a joint has no valid sample).  K <= 128.  f64 results equal the host expressions exactly. */
LHN_API int lhn_metrics_finalize(const int64_t* counters, int K, int auc_steps, double* out, lhn_stream_t stream);

/* MPII PCKh counters (datasets/datasets/body/topdown_mpii_dataset.py:186-214, duplicate in
 * topdown_mpii_action_dataset.py:176-204): pred f32 [N,K,pred_stride] 0-based (the kernel adds the reference's
 * +1.0 in f32), gt f64 [N,K,2] (pos_gt_src transposed), head f64 [N,4] = (x1,y1,x2,y2) of headboxes_src,
 * visible uint8 [N,K] = 1 - jnt_missing.  err / (|head box| * sc_bias) <= thr[t] in f64 (thr: host, T <= 64
 * doubles).  counters int64 [(T+1)*K]: hits[t][k], count[k]; ADDS (shardable). */
LHN_API int lhn_mpii_pckh_accumulate(const float* pred, int pred_stride, const double* gt,
                                     const double* head, const uint8_t* visible, int64_t N, int K,
                                     const double* thr /* host */, int T, double sc_bias,
                                     int64_t* counters, lhn_stream_t stream);

/* Fused decode + metrics counters for the sharded evaluation (BASELINE config 4): as
 * lhn_decode_heatmap (decode only) and, per plane, the three _report_metric accumulations
 * (base_dataset.py:193-261): PCK@pck_thr / max(bbox w,h), AUC thresholds i/auc_steps / auc_nor,
 * EPE.  gt f32 [B,K,2], mask uint8 [B,K] (fetched as the aligned 32-bit words that hold its bytes: the
 * buffer must be readable up to the next 4-byte boundary, which every cudaMalloc'd block is), bbox_wh f32 [B,2].
 * counters int64 [(1 + auc_steps + 4) * K] laid out as
 *   pck_hits[K], pck_valid[K], auc_hits[auc_steps][K], auc_valid[K], epe_valid[K], epe_fix[K]. */
LHN_API int lhn_decode_heatmap_pck(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                   int64_t stride_b, int64_t stride_c, const float* center,
                                   const float* scale, const lhn_decode_params* dp, float* out_hm,
                                   float* out_kpts, int32_t* out_idx, const float* gt,
                                   const uint8_t* mask, const float* bbox_wh, float pck_thr,
                                   float auc_nor, int auc_steps, int64_t* counters,
                                   lhn_stream_t stream);

/* The same with the per-step counter block all-reduced over the ranks INSIDE the kernel, pipelined over two launches:
 * `counters` is this rank's block for THIS step (zero at entry; rotate LHN_XCH_SLOTS blocks).  The launch carries one
 * extra CTA — the courier, on one SM that gets no planes — which, once the previous launch has completed, (a) adds
 * every rank's copy of xch->prev2_block's step (sent during the previous launch, so nothing is waited for) in rank
 * order into `totals` int64 [(auc_steps+5)*K] and zeroes that block, (b) sends xch->prev_block — the previous launch's
 * block — to every peer.  lhn_exchange_flush(xch, n, totals) completes the (up to two) steps still in flight when a
 * sequence ends; after it every rank holds the same running totals, equal bit for bit to a single-process evaluation
 * (datasets/base_dataset.py:193-261 on the gathered results).  Why a courier and why pipelined: whoever exchanges
 * holds its SM for the NVLink round trip, and a plane-carrying CTA that does so delays its SM's CTA of the next launch
 * on every step (DESIGN.md §6; LHN_XCH_COURIER=0 in the environment selects that older variant, where the first
 * plane-carrying CTA to finish exchanges). */
LHN_API int lhn_decode_heatmap_pck_xch(const void* hm, int dtype, int64_t B, int K, int H, int W,
                                   int64_t stride_b, int64_t stride_c, const float* center,
                                   const float* scale, const lhn_decode_params* dp, float* out_hm,
                                   float* out_kpts, int32_t* out_idx, const float* gt,
                                   const uint8_t* mask, const float* bbox_wh, float pck_thr,
                                   float auc_nor, int auc_steps, int64_t* counters,
                                   int64_t* totals, const lhn_exchange* xch,
                                          lhn_stream_t stream);
LHN_API int lhn_exchange_flush(const lhn_exchange* xch, int n, int64_t* totals, lhn_stream_t stream);

/* evaluate_pck (evaluation.py:10-59): argmax (A1) on pred and gt heatmap batches [B,K,H,W],
 * * image_size/[W,H], distance / max(bbox[:,0,2:]), per-image hits/(2*sum w)*2 in f32.
 * bbox_wh f32 [B,2]; weight f32 [B,K] or NULL (ones).  pck_per_image f32 [B]; mean_out f64 [1]
 * = mean over images (np.mean), NaN if an image has no weight, as the reference. */
LHN_API int64_t lhn_evaluate_pck_workspace_bytes(int64_t B, int K);
LHN_API int lhn_evaluate_pck(const void* pred_hm, const void* gt_hm, int dtype, int64_t B, int K,
                             int H, int W, const float* bbox_wh, const float* weight,
                             float image_w, float image_h, float thr, void* workspace,
                             int64_t workspace_bytes, float* pck_per_image, double* mean_out,
                             lhn_stream_t stream);

/* flip_back (transforms.py:78-92) materialised: out[b,k,y,x] = in[b,flip_index[k],y,W-1-x]. */
LHN_API int lhn_flip_back(const void* in, void* out, int dtype, int64_t B, int K, int H, int W,
                          const int32_t* flip_index, lhn_stream_t stream);

/* ---- region-map bbox decode (SURVEY §8f rank 4) -------------------------------------------------
 * The bbox branch of the legacy parsers: centre-map NMS -> top-k candidate centres -> size lookup ->
 * (centre refinement) -> box filter + IoU NMS, one CTA per image, everything on the device.
 *   LHN_REGION_SH  HeatmapParser_SH.heatmap_nms / candidate_bbox / non_max_suppression
 *                  (utils/SPheatmapParser.py:32-41,58-99,101-138): size = clip(avgpool(size)[y,x], 0, 0.99) *
 *                  image_size, centre = (idx % W, idx // W) * (image_size / [W, H]);
 *   LHN_REGION_RP  ResultParser.heatmap_nms / candidate_bbox / non_max_suppression
 *                  (utils/result_parser.py:50-59,131-175,177-215) with cfg['DARK'] = True: candidate centres
 *                  refined by the legacy DARK (blur_ksize = 19, f64 blur) on the NMS'd centre map — every
 *                  candidate on the same un-blurred map, the reference's CUDA semantics — then centre and
 *                  avgpool size both * (stride_x, stride_y).  refine = LHN_REFINE_NONE skips the refinement;
 *   LHN_REGION_CS  cs_from_region_map + non_max_suppression (utils/evaluation.py:94-212): no centre NMS
 *                  (nms_kernel = 0), size = mean of the size maps over the clipped window [c-6, c+7) *
 *                  image_w / W, only candidates with confidence > cand_thr get centre and size.
 * top-k follows torch.topk: descending, NaN greatest; EQUAL values (whose order torch leaves unspecified) come
 * lowest index first.  The IoU NMS is torchvision.ops.nms: f32 arithmetic, IoU compared with the double
 * threshold, candidates already in descending score order. */
#define LHN_REGION_SH 0
#define LHN_REGION_RP 1
#define LHN_REGION_CS 2
#define LHN_MAX_CANDIDATES 32

typedef struct {
  int32_t mode;            /* LHN_REGION_* */
  int32_t nms_kernel;      /* centre-map MaxPool2d window (odd, stride 1, padding (k-1)/2; pcfg nms_kernel = 11);
                              0 = use the centre map as it is */
  int32_t num_candidates;  /* top-k size N <= LHN_MAX_CANDIDATES (pcfg num_candidates = 10; evaluate_ap k = 20) */
  int32_t max_num_bbox;    /* boxes kept per image <= N (pcfg max_num_bbox = 1) */
  int32_t avg_kernel;      /* SH / RP: AvgPool2d window of the size maps (pcfg region_avg_kernel = 3) */
  int32_t refine;          /* RP: LHN_REFINE_NONE or LHN_REFINE_DARK_LEGACY */
  int32_t blur_ksize;      /* RP + DARK: 19 (pcfg blue_kernel) */
  int32_t reserved;
  float image_w, image_h;  /* SH, CS */
  float stride_x, stride_y;/* RP: feature_stride */
  float cand_thr;          /* CS: detection threshold inside cs_from_region_map */
  float det_thr;           /* box filter: confidence > det_thr (pcfg detection_threshold = 0.1) */
  float min_wh, max_wh;    /* box filter: min_wh < w, h < max_wh (2, 4096) */
  double iou_thr;          /* pcfg iou_threshold = 0.6 */
  double taps[LHN_MAX_TAPS]; /* lhn_gaussian_taps(blur_ksize) */
} lhn_region_params;

/* center [B,1,H,W] (batch stride center_stride_b elements, plane contiguous), size [B,2,H,W] (strides
 * size_stride_b / size_stride_c) — e.g. the two channel slices of one region map [B,3,H,W].
 * nms_out    NULL, or a tensor like `center` (same dtype and batch stride) that receives the NMS'd centre map;
 *            it MAY be `center` itself: the reference masks its argument in place (heatmaps *= mask).
 * candidates f32 [B, N, 5] (x, y, w, h, confidence) or NULL.
 * boxes      f32 [B, max_num_bbox, 5], zero-filled past counts[b]; counts int32 [B]. */
LHN_API int lhn_region_bbox_decode(const void* center, const void* size, int dtype, int64_t B, int H, int W,
                                   int64_t center_stride_b, int64_t size_stride_b, int64_t size_stride_c,
                                   const lhn_region_params* rp, void* nms_out, float* candidates,
                                   float* boxes, int32_t* counts, lhn_stream_t stream);

/* The width / height planes of SRHandNet's region-map target (SRHandNetGenerateTarget._region_generate_target,
 * datasets/data_pipeline/generateTarget.py:350-365): out[b, c, y, x] = gamma[b, c] inside the window
 * rect[b] = (x1, x2, y1, y2) (int32, half-open, already clipped to the plane), else 0; c = 0 width ratio,
 * 1 height ratio.  out f32, plane contiguous, out_stride_b elements between images (>= 2*H*W, so the two planes
 * can be written straight into channels K+1, K+2 of a [B, K+3, H, W] target).  The centre plane (channel K) is
 * lhn_render_targets on the box centre. */
LHN_API int lhn_render_region_wh(const int32_t* rect, const float* gamma, int64_t B, int H, int W, float* out,
                                 int64_t out_stride_b, lhn_stream_t stream);

/* non_max_suppression alone (utils/result_parser.py:177-215, utils/SPheatmapParser.py:101-138,
 * utils/evaluation.py:170-212) on given candidates f32 [B, N, 5] (x, y, w, h, confidence), N <= LHN_MAX_CANDIDATES:
 * confidence > det_thr, min_wh < w, h < max_wh, torchvision.ops.nms with iou_thr, first max_num kept.
 * boxes f32 [B, max_num, 5] zero-filled past counts[b]; counts int32 [B]. */
LHN_API int lhn_box_nms(const float* candidates, int64_t B, int N, float det_thr, float min_wh, float max_wh,
                        double iou_thr, int max_num, float* boxes, int32_t* counts, lhn_stream_t stream);

/* heatmap_nms alone (utils/result_parser.py:50-59, utils/SPheatmapParser.py:32-41) on [B, C, H, W] planes:
 * out = hm * eq(maxpool_k(hm), hm).  out has the same dtype and strides as hm and may alias it. */
LHN_API int lhn_heatmap_nms(const void* hm, void* out, int dtype, int64_t B, int C, int H, int W,
                            int64_t stride_b, int64_t stride_c, int nms_kernel, lhn_stream_t stream);

/* ResultParser.vector_nms (utils/result_parser.py:61-74): out = v * eq(max_pool1d(v, 3, 1, 1), v) on n_rows
 * contiguous rows of length L.  out must NOT alias v. */
LHN_API int lhn_vector_nms(const void* v, void* out, int dtype, int64_t n_rows, int L, lhn_stream_t stream);

/* The +-0.25 rule at GIVEN integer positions (HeatmapParser.adjust_keypoints, utils/HeatmapParser.py:197-223,
 * whose grouped candidates are not plane argmaxima): for point i on plane (bc[2i], bc[2i+1]) of hm [B,C,H,W],
 * xx = int(x), yy = int(y); x += 0.25 if hm[yy, min(xx+1, W-1)] > hm[yy, max(xx-1, 0)] else -0.25, likewise y;
 * refine = LHN_REFINE_OFFSET, or LHN_REFINE_OFFSET_HALF (then + 0.5).  xy f32 [n, xy_stride] updated in place. */
LHN_API int lhn_refine_points(const void* hm, int dtype, int64_t B, int C, int H, int W, int64_t stride_b,
                              int64_t stride_c, const int32_t* bc, float* xy, int xy_stride, int64_t n,
                              int refine, lhn_stream_t stream);

/* The legacy DARK at GIVEN positions (adjust_keypoints_by_DARK, utils/heatmap_post_processing.py:35-76, which
 * refines around int(keypoints) wherever the caller puts them — e.g. the top-k candidates of
 * ResultParser.candidate_bbox): per point the plane (bc[2i], bc[2i+1]) is blurred (f64, zero-padded, dp->blur_ksize =
 * 19), scaled by max / (max(blurred) + 1e-6), log, Taylor step under the 1 < p < size - 2 guard.  One CTA per point;
 * two points on the same plane may run concurrently (the plane is only read).  xy f32 [n, xy_stride] updated in
 * place.  dp->refine must be LHN_REFINE_DARK_LEGACY. */
LHN_API int lhn_dark_refine_points(const void* hm, int dtype, int64_t B, int C, int H, int W, int64_t stride_b,
                                   int64_t stride_c, const int32_t* bc, float* xy, int xy_stride, int64_t n,
                                   const lhn_decode_params* dp, lhn_stream_t stream);

/* Bbox-restricted keypoint decode (ResultParser._get_first_result, utils/result_parser.py:288-306):
 * for image b only the window roi[b] = (x0, y0, x1, y1) (int32 [B,4], 0 <= x0 < x1 <= W) of each plane takes
 * part: first-index argmax of the cropped plane (A4), then LHN_REFINE_NONE / _OFFSET / _OFFSET_HALF /
 * _DARK_LEGACY evaluated ON THE CROP (neighbours clamp, and the blur zero-pads, at the window's border), then
 * (x + x0, y + y0) * (scale_x, scale_y).  dp: refine, blur_ksize, taps, scale_x/scale_y are read.
 * out f32 [B*K, 3] (X, Y, score); out_idx int32 [B*K] flat index inside the crop, or NULL. */
LHN_API int lhn_decode_heatmap_roi(const void* hm, int dtype, int64_t B, int K, int H, int W, int64_t stride_b,
                                   int64_t stride_c, const int32_t* roi, const lhn_decode_params* dp,
                                   float* out, int32_t* out_idx, lhn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LHN_H_ */
