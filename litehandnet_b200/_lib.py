"""ctypes binding of liblhn.so — the thin layer that hands raw device pointers to the kernels.

There is NO fallback: if the library is missing or a call is rejected this raises.  The library is
built in-tree by ``litehandnet_b200.build`` (``__graft_entry__.build()``) into
``litehandnet_b200/lib/liblhn.so`` and declared in ``include/lhn.h``.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LHN_LIB", os.path.join(_HERE, "lib", "liblhn.so"))

# ---- constants mirrored from include/lhn.h -------------------------------------------------------
F32, BF16, F16, F64 = 0, 1, 2, 3
MASK_NONE, MASK_ZERO, MASK_NEG1 = 0, 1, 2
REFINE_NONE, REFINE_OFFSET_HALF, REFINE_OFFSET, REFINE_SIGN, REFINE_SIGN_ROUND, REFINE_DARK, \
    REFINE_DARK_LEGACY, REFINE_DARK_UDP = range(8)
XFORM_NONE, XFORM_CENTER_SCALE, XFORM_SCALE = 0, 1, 2
LOSS_NONE, LOSS_DISTANCE, LOSS_DISTANCE_BALANCE, LOSS_JOINTS_MSE = 0, 1, 2, 3
FLAG_OVERLAP_PREVIOUS = 1
FLAG_ACCUMULATE_LOSS = 2
MAX_TAPS, MAX_STACKS = 31, 8
LOSS_MAX_TENSORS = 8
XCH_MAX_RANKS, XCH_SLOTS, XCH_PAYLOAD_BYTES, XCH_CTRL_BYTES = 8, 4, 8192, 4096
XCH_MAILBOX_BYTES = XCH_SLOTS * XCH_MAX_RANKS * XCH_PAYLOAD_BYTES + XCH_CTRL_BYTES
REGION_SH, REGION_RP, REGION_CS = 0, 1, 2
MAX_CANDIDATES = 32

ERRORS = {-1: "LHN_EINVAL (bad shape / null pointer / bad enum)", -2: "LHN_EDTYPE (unsupported dtype)",
          -3: "LHN_EALIGN (misaligned pointer)", -4: "LHN_EWORKSPACE (workspace too small)",
          -5: "LHN_ECUDA (launch failed)"}

EXPORTS = [
    "lhn_version", "lhn_last_cuda_error", "lhn_gaussian_taps", "lhn_decode_heatmap",
    "lhn_decode_heatmap_pck", "lhn_loss_partials", "lhn_loss_reduce", "lhn_loss_finalize", "lhn_loss_mse_workspace_bytes", "lhn_loss_mse_multi",
    "lhn_render_targets", "lhn_render_simdr", "lhn_render_simdr_f64sigma", "lhn_decode_simdr", "lhn_decode_simdr_flags", "lhn_simdr_loss_workspace_bytes",
    "lhn_simdr_smoothl1", "lhn_split_bf16", "lhn_simdr_heads_workspace_bytes", "lhn_simdr_heads_loss",
    "lhn_simdr_heads_f32_workspace_bytes", "lhn_simdr_heads_loss_f32", "lhn_pck_accumulate", "lhn_metrics_finalize", "lhn_evaluate_pck_workspace_bytes",
    "lhn_evaluate_pck", "lhn_flip_back", "lhn_fused_workspace_bytes", "lhn_fused_render_loss_decode",
    "lhn_fused_render_loss_decode_xch", "lhn_decode_heatmap_pck_xch", "lhn_exchange_flush",
    "lhn_loss_backward", "lhn_render_loss_backward", "lhn_simdr_backward_workspace_bytes",
    "lhn_render_loss_grad_workspace_bytes", "lhn_render_loss_grad", "lhn_render_loss_backward_cond",
    "lhn_simdr_smoothl1_backward", "lhn_mpii_pckh_accumulate", "lhn_region_bbox_decode", "lhn_heatmap_nms",
    "lhn_vector_nms", "lhn_refine_points", "lhn_decode_heatmap_roi", "lhn_box_nms", "lhn_render_region_wh", "lhn_dark_refine_points",
    "lhn_k1_last_launch", "lhn_simdr_last_launch",
    "lhn_render_loss_multi_workspace_bytes", "lhn_render_loss_multi", "lhn_render_loss_backward_multi",
    "lhn_render_loss_grad_multi_workspace_bytes", "lhn_render_loss_grad_multi", "lhn_render_loss_backward_multi_cond",
]


class DecodeParams(C.Structure):
    _fields_ = [("mask_mode", C.c_int32), ("refine", C.c_int32), ("transform", C.c_int32),
                ("use_udp", C.c_int32), ("blur_ksize", C.c_int32), ("flags", C.c_int32),
                ("scale_x", C.c_float), ("scale_y", C.c_float), ("taps", C.c_double * MAX_TAPS)]


class RenderParams(C.Structure):
    _fields_ = [("loss_mode", C.c_int32), ("unbiased", C.c_int32), ("num_stacks", C.c_int32),
                ("reserved", C.c_int32), ("image_w", C.c_float), ("image_h", C.c_float),
                ("pos_value", C.c_float), ("sigma", C.c_float * MAX_STACKS)]


class LossScale(C.Structure):
    """lhn_loss_scale: one scale of lhn_render_loss_multi / lhn_render_loss_backward_multi."""
    _fields_ = [("output", C.c_void_p), ("grad", C.c_void_p), ("out_weight", C.c_void_p), ("stride_b", C.c_int64),
                ("stride_c", C.c_int64), ("H", C.c_int32), ("W", C.c_int32), ("sigma", C.c_float),
                ("loss_weight", C.c_float)]


class Exchange(C.Structure):
    _fields_ = [("mailbox", C.c_void_p * XCH_MAX_RANKS), ("world", C.c_int32), ("rank", C.c_int32),
                ("seq", C.c_uint32), ("timeout_ms", C.c_uint32), ("status", C.c_void_p), ("prev_block", C.c_void_p),
                ("prev_seq", C.c_uint32), ("prev2_seq", C.c_uint32), ("prev2_block", C.c_void_p)]


class RegionParams(C.Structure):
    _fields_ = [("mode", C.c_int32), ("nms_kernel", C.c_int32), ("num_candidates", C.c_int32),
                ("max_num_bbox", C.c_int32), ("avg_kernel", C.c_int32), ("refine", C.c_int32),
                ("blur_ksize", C.c_int32), ("reserved", C.c_int32), ("image_w", C.c_float), ("image_h", C.c_float),
                ("stride_x", C.c_float), ("stride_y", C.c_float), ("cand_thr", C.c_float), ("det_thr", C.c_float),
                ("min_wh", C.c_float), ("max_wh", C.c_float), ("iou_thr", C.c_double),
                ("taps", C.c_double * MAX_TAPS)]


class K1LaunchInfo(C.Structure):
    """lhn_k1_launch_info: which K1 code path the last call on this thread launched (tests only)."""
    _fields_ = [(n, C.c_int32) for n in ("path", "dtype", "flip", "loss", "counters", "wc", "twc", "ks", "team_warps",
                                          "nteams", "stages", "sweeper_tables", "use_tma", "ctas", "stagger_ns")]


class SimdrLaunchInfo(C.Structure):
    """lhn_simdr_launch_info: which SimDR kernel and geometry the last SimDR call on this thread launched (tests only)."""
    _fields_ = [(n, C.c_int32) for n in ("family", "path", "dtype", "warps", "stages", "ctas", "vec_x", "vec_y", "bn")]


class LhnError(RuntimeError):
    pass


_lib = None


def _declare(lib):
    vp, i32, i64, f32, f64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double
    lib.lhn_version.restype = C.c_int
    lib.lhn_last_cuda_error.restype = C.c_char_p
    lib.lhn_gaussian_taps.argtypes = [i32, C.POINTER(C.c_double)]
    lib.lhn_k1_last_launch.argtypes = [C.POINTER(K1LaunchInfo)]
    lib.lhn_simdr_last_launch.argtypes = [C.POINTER(SimdrLaunchInfo)]
    lib.lhn_decode_heatmap.argtypes = [vp, vp, vp, i32, i64, i32, i32, i32, i64, i64, i64, i64, vp, vp,
                                       C.POINTER(DecodeParams), vp, vp, vp, C.POINTER(RenderParams),
                                       vp, i32, vp, i32, vp, vp, vp]
    lib.lhn_fused_workspace_bytes.argtypes = [i64, i32, i32]
    lib.lhn_fused_workspace_bytes.restype = i64
    lib.lhn_fused_render_loss_decode.argtypes = [vp, vp, vp, i32, i64, i32, i32, i32, i64, i64, i64, i64, vp, vp,
                                                 C.POINTER(DecodeParams), vp, vp, vp, C.POINTER(RenderParams),
                                                 vp, i32, vp, i32, vp, vp, vp, i64, vp, i32, f32, vp, vp]
    lib.lhn_fused_render_loss_decode_xch.argtypes = [vp, vp, vp, i32, i64, i32, i32, i32, i64, i64, i64, i64, vp, vp,
                                                     C.POINTER(DecodeParams), vp, vp, vp, C.POINTER(RenderParams),
                                                     vp, i32, vp, i32, vp, vp, vp, i64, vp, i32, f32, vp,
                                                     C.POINTER(Exchange), vp]
    lib.lhn_decode_heatmap_pck_xch.argtypes = [vp, i32, i64, i32, i32, i32, i64, i64, vp, vp,
                                               C.POINTER(DecodeParams), vp, vp, vp, vp, vp, vp, f32, f32,
                                               i32, vp, vp, C.POINTER(Exchange), vp]
    lib.lhn_exchange_flush.argtypes = [C.POINTER(Exchange), i32, vp, vp]
    lib.lhn_loss_backward.argtypes = [vp, vp, vp, i32, i64, i64, i32, f32, vp, i32, f32, vp, vp, vp]
    lib.lhn_render_loss_backward.argtypes = [vp, i32, i64, i32, i32, i32, i64, i64, C.POINTER(RenderParams),
                                             vp, i32, vp, i32, vp, i32, f32, vp, vp, vp]
    lib.lhn_render_loss_grad_workspace_bytes.argtypes = [i64, i32, i32]
    lib.lhn_render_loss_grad_workspace_bytes.restype = i64
    lib.lhn_render_loss_grad.argtypes = [vp, i32, i64, i32, i32, i32, i64, i64, C.POINTER(RenderParams),
                                         vp, i32, vp, i32, vp, vp, i64, vp, i32, f32, vp, vp, vp, vp, vp]
    lib.lhn_render_loss_backward_cond.argtypes = [vp, i32, i64, i32, i32, i32, i64, i64, C.POINTER(RenderParams),
                                                  vp, i32, vp, i32, vp, i32, f32, vp, vp, vp, vp, vp]
    lib.lhn_simdr_backward_workspace_bytes.argtypes = [i32]
    lib.lhn_simdr_backward_workspace_bytes.restype = i64
    lib.lhn_simdr_smoothl1_backward.argtypes = [vp, vp, vp, vp, vp, i32, i64, i32, i32, i32, f32, vp, vp, i64,
                                                vp, vp, vp]
    lib.lhn_mpii_pckh_accumulate.argtypes = [vp, i32, vp, vp, vp, i64, i32, C.POINTER(C.c_double), i32, f64, vp, vp]
    lib.lhn_decode_heatmap_pck.argtypes = [vp, i32, i64, i32, i32, i32, i64, i64, vp, vp,
                                           C.POINTER(DecodeParams), vp, vp, vp, vp, vp, vp, f32, f32,
                                           i32, vp, vp]
    lib.lhn_loss_partials.argtypes = [vp, vp, vp, i32, i64, i64, i32, f32, vp, vp]
    lib.lhn_loss_reduce.argtypes = [vp, i64, vp, i32, vp]
    lib.lhn_loss_mse_workspace_bytes.argtypes = []
    lib.lhn_loss_mse_workspace_bytes.restype = i64
    lib.lhn_loss_mse_multi.argtypes = [i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(i64), C.POINTER(i64),
                                       C.POINTER(f32), i32, i32, f32, i32, f32, vp, i64, vp, vp, vp, i32, vp]
    lib.lhn_render_loss_multi_workspace_bytes.argtypes = []
    lib.lhn_render_loss_multi_workspace_bytes.restype = i64
    lib.lhn_render_loss_multi.argtypes = [i32, C.POINTER(LossScale), i32, i64, i32, C.POINTER(RenderParams), vp, i32,
                                          vp, i32, i32, f32, vp, i64, vp, vp, vp, vp]
    lib.lhn_render_loss_backward_multi.argtypes = [i32, C.POINTER(LossScale), i32, i64, i32, C.POINTER(RenderParams),
                                                   vp, i32, vp, i32, vp, i32, vp, vp]
    lib.lhn_render_loss_grad_multi_workspace_bytes.argtypes = [i32, i64, i32]
    lib.lhn_render_loss_grad_multi_workspace_bytes.restype = i64
    lib.lhn_render_loss_grad_multi.argtypes = [i32, C.POINTER(LossScale), i32, i64, i32, C.POINTER(RenderParams), vp,
                                               i32, vp, i32, i32, f32, vp, i64, vp, vp, vp, vp, vp, vp]
    lib.lhn_render_loss_backward_multi_cond.argtypes = [i32, C.POINTER(LossScale), i32, i64, i32,
                                                        C.POINTER(RenderParams), vp, i32, vp, i32, vp, i32, vp, vp, vp,
                                                        vp]
    lib.lhn_loss_finalize.argtypes = [vp, i32, i32, f32, vp, i32, vp]
    lib.lhn_render_targets.argtypes = [vp, i32, vp, i32, i64, i32, i32, i32, C.POINTER(RenderParams),
                                       vp, vp, vp]
    lib.lhn_render_simdr.argtypes = [vp, i32, vp, i32, i64, i32, i32, i32, f32, f32, vp, vp, vp]
    lib.lhn_render_simdr_f64sigma.argtypes = [vp, i32, vp, i32, i64, i32, i32, i32, f32, f64, vp, vp, vp]
    lib.lhn_decode_simdr.argtypes = [vp, vp, i32, i64, i32, i32, i32, i32, vp, vp, i32, vp, vp, vp, vp]
    lib.lhn_decode_simdr_flags.argtypes = [vp, vp, i32, i64, i32, i32, i32, i32, vp, vp, i32, vp, vp, vp, i32, vp]
    lib.lhn_simdr_loss_workspace_bytes.argtypes = [i64, i32]
    lib.lhn_simdr_loss_workspace_bytes.restype = i64
    lib.lhn_simdr_smoothl1.argtypes = [vp, vp, vp, vp, vp, i32, i64, i32, i32, i32, vp, i64, vp, vp]
    lib.lhn_pck_accumulate.argtypes = [vp, i32, i32, vp, i32, i32, vp, vp, i32, f64, i64, i32,
                                       C.POINTER(C.c_float), i32, vp, vp]
    lib.lhn_metrics_finalize.argtypes = [vp, i32, i32, vp, vp]
    lib.lhn_split_bf16.argtypes = [vp, i64, vp, vp, vp]
    lib.lhn_simdr_heads_workspace_bytes.argtypes = [i64, i32, i32, i32]
    lib.lhn_simdr_heads_workspace_bytes.restype = i64
    lib.lhn_simdr_heads_f32_workspace_bytes.argtypes = [i64, i32, i32, i32, i32]
    lib.lhn_simdr_heads_f32_workspace_bytes.restype = i64
    lib.lhn_simdr_heads_loss_f32.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, i32, vp, i64, vp, vp, vp, vp]
    lib.lhn_simdr_heads_loss.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, i32, vp, i64, vp, vp, vp, vp]
    lib.lhn_evaluate_pck_workspace_bytes.argtypes = [i64, i32]
    lib.lhn_evaluate_pck_workspace_bytes.restype = i64
    lib.lhn_evaluate_pck.argtypes = [vp, vp, i32, i64, i32, i32, i32, vp, vp, f32, f32, f32, vp, i64,
                                     vp, vp, vp]
    lib.lhn_flip_back.argtypes = [vp, vp, i32, i64, i32, i32, i32, vp, vp]
    lib.lhn_region_bbox_decode.argtypes = [vp, vp, i32, i64, i32, i32, i64, i64, i64, C.POINTER(RegionParams),
                                           vp, vp, vp, vp, vp]
    lib.lhn_render_region_wh.argtypes = [vp, vp, i64, i32, i32, vp, i64, vp]
    lib.lhn_dark_refine_points.argtypes = [vp, i32, i64, i32, i32, i32, i64, i64, vp, vp, i32, i64,
                                           C.POINTER(DecodeParams), vp]
    lib.lhn_box_nms.argtypes = [vp, i64, i32, f32, f32, f32, f64, i32, vp, vp, vp]
    lib.lhn_heatmap_nms.argtypes = [vp, vp, i32, i64, i32, i32, i32, i64, i64, i32, vp]
    lib.lhn_vector_nms.argtypes = [vp, vp, i32, i64, i32, vp]
    lib.lhn_refine_points.argtypes = [vp, i32, i64, i32, i32, i32, i64, i64, vp, vp, i32, i64, i32, vp]
    lib.lhn_decode_heatmap_roi.argtypes = [vp, i32, i64, i32, i32, i32, i64, i64, vp, C.POINTER(DecodeParams),
                                           vp, vp, vp]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is C.c_int and name not in ("lhn_version",):
            fn.restype = C.c_int


def lib():
    """Load liblhn.so once.  Raises LhnError (never falls back) if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LhnError(f"{LIB_PATH} not found: build it with `python -m litehandnet_b200.build` "
                           "(there is no CPU or PyTorch fallback for this path)")
        handle = C.CDLL(LIB_PATH)
        _declare(handle)
        _lib = handle
    return _lib


_ext = False


def ext():
    """The torch-extension shim (csrc/ext/lhn_torch_ext.cpp, built in-tree by litehandnet_b200.build) or None when it
    is absent or LHN_NO_EXT=1.  It is a faster route to the SAME library (a few microseconds of host time per call
    instead of 20-30 through ctypes); the kernels and their results are identical."""
    global _ext
    if _ext is False:
        _ext = None
        if os.environ.get("LHN_NO_EXT") != "1":
            import glob
            import importlib.util
            cands = glob.glob(os.path.join(_HERE, "lib", "lhn_torch_ext*.so"))
            if cands:
                lib()                                            # liblhn.so first (the shim links against it)
                spec = importlib.util.spec_from_file_location("lhn_torch_ext", cands[0])
                mod = importlib.util.module_from_spec(spec)
                spec.loader.exec_module(mod)
                _ext = mod
    return _ext


def check(rc, what):
    if rc != 0:
        msg = ERRORS.get(rc, f"error {rc}")
        if rc == -5:
            msg += ": " + (lib().lhn_last_cuda_error() or b"").decode()
        raise LhnError(f"{what}: {msg}")


def require_cuda(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise LhnError(f"{name} must be a CUDA tensor (this path has no CPU fallback)")
    return t


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream(device=None):
    """Raw handle of torch's current stream on `device` (default: the current device; ops wrappers run under a
    guard for their tensors' device, so the default is that device)."""
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class on_device:
    """`with on_device(dev):` — no-op when `dev` is already current, else torch.cuda.device(dev).  The library
    launches on the CURRENT device, so every launch on tensors of another device must run under this."""
    __slots__ = ("dev", "ctx")

    def __init__(self, dev):
        self.dev, self.ctx = dev, None

    def __enter__(self):
        if self.dev.index is not None and self.dev.index != torch.cuda.current_device():
            self.ctx = torch.cuda.device(self.dev)
            self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
            self.ctx = None
        return False


def dtype_code(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    if t.dtype == torch.float16:
        return F16
    if t.dtype == torch.float64:
        return F64
    raise LhnError(f"unsupported dtype {t.dtype}")


_TAPS_CACHE = {}


def gaussian_taps(ksize):
    """cv2.getGaussianKernel(ksize, 0, CV_64F) as computed by the library (host)."""
    if ksize not in _TAPS_CACHE:
        arr = (C.c_double * MAX_TAPS)()
        check(lib().lhn_gaussian_taps(int(ksize), arr), "lhn_gaussian_taps")
        _TAPS_CACHE[ksize] = list(arr)[:ksize]
    return _TAPS_CACHE[ksize]
