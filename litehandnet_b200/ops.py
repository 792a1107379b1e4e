"""Tensor-level wrappers over the C ABI (include/lhn.h).  Every function takes CUDA tensors, launches
on ``torch.cuda.current_stream()`` and returns CUDA tensors; nothing here synchronises or falls back.
"""
import ctypes as C
import functools

import torch

from . import _lib as L


def _cuda_tensors(values):
    for v in values:
        if isinstance(v, torch.Tensor):
            if v.is_cuda:
                yield v
        elif isinstance(v, dict):
            yield from _cuda_tensors(v.values())


def _on_device(fn):
    """Run the wrapped launch on the device of its tensors: all CUDA tensor arguments must live on ONE device;
    if that is not the current device the call runs under ``torch.cuda.device(dev)``, so the library's launch,
    ``torch.cuda.current_stream()`` (L.stream()) and every output allocation refer to the tensors' device — the
    reference calls set_device only in its DDP entry points, a single process may well drive several GPUs."""
    @functools.wraps(fn)
    def wrapper(*args, **kw):
        dev = None
        for t in _cuda_tensors(args):
            if dev is None:
                dev = t.device
            elif t.device != dev:
                raise L.LhnError(f"{fn.__name__}: tensors on different devices ({dev} and {t.device})")
        for t in _cuda_tensors(kw.values()):
            if dev is None:
                dev = t.device
            elif t.device != dev:
                raise L.LhnError(f"{fn.__name__}: tensors on different devices ({dev} and {t.device})")
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kw)
        with torch.cuda.device(dev):
            return fn(*args, **kw)
    return wrapper


_REFINE_KSIZE = {L.REFINE_DARK: 11, L.REFINE_DARK_LEGACY: 19, L.REFINE_DARK_UDP: 11}


_DP_CACHE = {}


def _decode_params(mask_mode, refine, transform, scale_xy=(1.0, 1.0), blur_ksize=None, use_udp=False, flags=0):
    """lhn_decode_params for one call; the library only reads it, so equal arguments share one cached struct (building
    it costs ~4 us of host time per launch otherwise)."""
    key = (int(mask_mode), int(refine), int(transform), float(scale_xy[0]), float(scale_xy[1]),
           int(blur_ksize) if blur_ksize else 0, bool(use_udp), int(flags))
    dp = _DP_CACHE.get(key)
    if dp is None:
        if len(_DP_CACHE) > 256:
            _DP_CACHE.clear()
        dp = _DP_CACHE[key] = _build_decode_params(mask_mode, refine, transform, scale_xy, blur_ksize, use_udp, flags)
    return dp


def _build_decode_params(mask_mode, refine, transform, scale_xy, blur_ksize, use_udp, flags):
    dp = L.DecodeParams()
    dp.mask_mode, dp.refine, dp.transform, dp.use_udp = int(mask_mode), int(refine), int(transform), int(bool(use_udp))
    dp.scale_x, dp.scale_y = float(scale_xy[0]), float(scale_xy[1])
    dp.flags = int(flags)
    if refine in _REFINE_KSIZE:
        k = int(blur_ksize) if blur_ksize else _REFINE_KSIZE[refine]
        dp.blur_ksize = k
        for i, t in enumerate(L.gaussian_taps(k)):
            dp.taps[i] = t
    return dp


def _render_params(loss_mode, image_size, sigma, unbiased=True, pos_value=0.5):
    rp = L.RenderParams()
    sig = list(sigma) if isinstance(sigma, (list, tuple)) else [sigma]
    if len(sig) > L.MAX_STACKS:
        raise L.LhnError(f"at most {L.MAX_STACKS} stacked sigmas")
    # unbiased: False/0 = MSRA integer-centre patch, True/1 = MSRA sub-pixel plane, 'udp'/2 = UDP GaussianHeatmap
    mode = 2 if (unbiased == 2 or (isinstance(unbiased, str) and unbiased.lower() == "udp")) else int(bool(unbiased))
    rp.loss_mode, rp.unbiased, rp.num_stacks = int(loss_mode), mode, len(sig)
    rp.image_w, rp.image_h = float(image_size[0]), float(image_size[1])
    rp.pos_value = float(pos_value)
    for i, s in enumerate(sig):
        rp.sigma[i] = float(s)
    return rp


def _plane_view(hm, name):
    """[B,C,H,W] or [B,S,K,H,W] tensor with contiguous planes -> (tensor, B, C, H, W, stride_b, stride_c)."""
    L.require_cuda(hm, name)
    if hm.dim() == 5:
        B, S, K, H, W = hm.shape
        if not hm[0].is_contiguous():
            hm = hm.contiguous()
        return hm, B, S * K, H, W, hm.stride(0), hm.stride(2)
    if hm.dim() != 4:
        raise L.LhnError(f"{name} must be [B,K,H,W] or [B,S,K,H,W], got {tuple(hm.shape)}")
    B, Cc, H, W = hm.shape
    if hm.stride(3) != 1 or hm.stride(2) != W or (Cc > 1 and hm.stride(1) < H * W):
        hm = hm.contiguous()
    return hm, B, Cc, H, W, hm.stride(0), hm.stride(1) if Cc > 1 else H * W


def _f32c(t, name):
    if t is None:
        return None
    L.require_cuda(t, name)
    if t.dtype == torch.float32 and t.is_contiguous():
        return t
    return t.to(torch.float32).contiguous()


def _ext_ready(t, dtype=None):
    """A tensor the extension shim takes as is (CUDA, contiguous, right dtype), or None."""
    return t is None or (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous() and (dtype is None or t.dtype == dtype))


def decode_heatmap(hm, mask_mode, refine, transform=L.XFORM_NONE, center=None, scale=None,
                   scale_xy=(1.0, 1.0), hm_flip=None, flip_index=None, blur_ksize=None, use_udp=False,
                   want_idx=True, render=None, joints=None, vis=None, out=None, overlap_previous=False):
    """K1 (see _decode_heatmap_ctypes for the arguments).  Plain decode calls on ready-to-use tensors go through the
    torch-extension shim (same library entry point, ~4x less host time per call: the reference decodes 32-64 samples per
    call, test.py:114-126, where the Python wrapper costs more than the kernel); everything else through ctypes."""
    e = L.ext()
    if (e is not None and render is None and not out and isinstance(hm, torch.Tensor) and hm.is_cuda and hm.dim() == 4 and
            hm.stride(3) == 1 and hm.stride(2) == hm.shape[3] and (hm.shape[1] == 1 or hm.stride(1) >= hm.shape[2] * hm.shape[3]) and
            _ext_ready(center, torch.float32) and _ext_ready(scale, torch.float32) and _ext_ready(flip_index, torch.int32) and
            (hm_flip is None or (isinstance(hm_flip, torch.Tensor) and hm_flip.is_cuda and hm_flip.stride(3) == 1 and
                                 hm_flip.stride(2) == hm.shape[3]))):
        dp = _decode_params(mask_mode, refine, transform, scale_xy, blur_ksize, use_udp,
                            flags=L.FLAG_OVERLAP_PREVIOUS if overlap_previous else 0)
        try:
            r = e.decode_heatmap(hm, hm_flip, flip_index, center, scale, C.addressof(dp), bool(want_idx))
        except RuntimeError as err:
            raise L.LhnError(str(err).split("\n")[0]) from None
        return dict(hm_kpts=r[0], kpts=r[1], idx=r[2] if want_idx else None)
    return _decode_heatmap_ctypes(hm, mask_mode, refine, transform, center, scale, scale_xy, hm_flip, flip_index, blur_ksize,
                                  use_udp, want_idx, render, joints, vis, out, overlap_previous)


@_on_device
def _decode_heatmap_ctypes(hm, mask_mode, refine, transform=L.XFORM_NONE, center=None, scale=None,
                           scale_xy=(1.0, 1.0), hm_flip=None, flip_index=None, blur_ksize=None, use_udp=False,
                           want_idx=True, render=None, joints=None, vis=None, out=None, overlap_previous=False):
    """K1.  Returns dict(hm_kpts [B,C,3], kpts [B,C,3], idx [B,C] int32[, weight [B,C], partials [B*C,4]]).

    render: None or dict(loss_mode, image_size, sigma, unbiased, pos_value) to fuse the target render +
    masked-MSE partial sums against joints [B,K,>=2] / vis [B,K,>=1] (column 0 = visibility).
    out: optional dict of preallocated contiguous outputs (hm_kpts, kpts, idx, partials, weight) to
    write into instead of allocating (steady-state loops, chunked pipelines).
    overlap_previous: this call touches no buffer the previous launch on the stream writes (rotating buffer sets),
    so its kernel may start while that one drains (LHN_FLAG_OVERLAP_PREVIOUS).
    """
    out = out or {}
    hm, B, Cc, H, W, sb, sc = _plane_view(hm, "heatmaps")
    dev = hm.device
    fb = fc = 0
    if hm_flip is not None:
        hm_flip, B2, C2, H2, W2, fb, fc = _plane_view(hm_flip, "flipped heatmaps")
        if (B2, C2, H2, W2) != (B, Cc, H, W) or hm_flip.dtype != hm.dtype:
            raise L.LhnError("flipped heatmaps must match heatmaps in shape and dtype")
    S = 1
    rp = None
    partials = weight = None
    if render is not None and render.get("loss_mode", L.LOSS_NONE) != L.LOSS_NONE:
        rp = _render_params(render["loss_mode"], render["image_size"], render["sigma"],
                            render.get("unbiased", True), render.get("pos_value", 0.5))
        S = rp.num_stacks
        joints = _f32c(joints, "joints")
        vis = _f32c(vis, "vis")
        if joints.dim() != 3 or joints.shape[0] != B or joints.shape[2] < 2:
            raise L.LhnError("joints must be [B,K,>=2]")
        if vis.dim() == 2:
            vis = vis.unsqueeze(-1).contiguous()
        partials = out.get("partials")
        if partials is None:
            partials = torch.empty((B * Cc, 4), dtype=torch.float64, device=dev)
        weight = out.get("weight")
        if weight is None:
            weight = torch.empty((B, Cc), dtype=torch.float32, device=dev)
    if Cc % S:
        raise L.LhnError("channel count is not a multiple of the number of stacks")
    K = Cc // S
    if flip_index is not None:
        flip_index = L.require_cuda(flip_index, "flip_index").to(torch.int32).contiguous()
        if flip_index.numel() != K:
            raise L.LhnError("flip_index must have K entries")
    center = _f32c(center, "center")
    scale = _f32c(scale, "scale")
    dp = _decode_params(mask_mode, refine, transform, scale_xy, blur_ksize, use_udp,
                        flags=L.FLAG_OVERLAP_PREVIOUS if overlap_previous else 0)
    out_hm = out.get("hm_kpts")
    if out_hm is None:
        out_hm = torch.empty((B, Cc, 3), dtype=torch.float32, device=dev)
    out_k = out.get("kpts")
    if out_k is None:
        out_k = torch.empty((B, Cc, 3), dtype=torch.float32, device=dev)
    out_idx = out.get("idx")
    if out_idx is None and want_idx:
        out_idx = torch.empty((B, Cc), dtype=torch.int32, device=dev)
    for name, t, dt, n in (("hm_kpts", out_hm, torch.float32, B * Cc * 3), ("kpts", out_k, torch.float32, B * Cc * 3),
                           ("idx", out_idx, torch.int32, B * Cc), ("partials", partials, torch.float64, B * Cc * 4),
                           ("weight", weight, torch.float32, B * Cc)):
        if t is not None and (t.dtype != dt or t.numel() != n or not t.is_contiguous() or t.device != dev):
            raise L.LhnError(f"preallocated output '{name}' has the wrong dtype/size/layout/device")
    rc = L.lib().lhn_decode_heatmap(
        L.ptr(hm), L.ptr(hm_flip), L.ptr(flip_index), L.dtype_code(hm), B, K, H, W, sb, sc, fb, fc,
        L.ptr(center), L.ptr(scale), C.byref(dp), L.ptr(out_hm), L.ptr(out_k), L.ptr(out_idx),
        C.byref(rp) if rp is not None else None,
        L.ptr(joints), joints.shape[2] if joints is not None else 0,
        L.ptr(vis), vis.shape[2] if vis is not None else 0,
        L.ptr(weight), L.ptr(partials), L.stream())
    L.check(rc, "lhn_decode_heatmap")
    res = dict(hm_kpts=out_hm, kpts=out_k, idx=out_idx)
    if partials is not None:
        res["partials"], res["weight"] = partials, weight
    return res


_WORKSPACES = {}


def fused_workspace(device, B, K, S=1, stream_key=None):
    """Zero-initialised workspace of the one-launch step, cached per (device, stream, size): the kernel
    leaves it zeroed, so it is memset only once."""
    need = int(L.lib().lhn_fused_workspace_bytes(int(B), int(K), int(S)))
    if stream_key is None:
        stream_key = torch.cuda.current_stream(device).cuda_stream
    key = (str(device), stream_key)
    ws = _WORKSPACES.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.zeros(need, dtype=torch.uint8, device=device)
        _WORKSPACES[key] = ws
    return ws


@_on_device
def fused_render_loss_decode(hm, mask_mode, refine, transform, center, scale, render, joints, vis,
                             hm_flip=None, flip_index=None, blur_ksize=None, use_udp=False, scale_xy=(1.0, 1.0),
                             want_idx=True, want_partials=False, reduction="mean", loss_scale=1.0,
                             want_loss=True, out=None, workspace=None, overlap_previous=False):
    """The headline step in ONE launch (lhn_fused_render_loss_decode): as decode_heatmap(render=...) plus
    the deterministic loss reduction and finalisation.  Returns dict(hm_kpts, kpts, idx, weight,
    sums f64[4], loss f32[1] (if want_loss)[, partials])."""
    out = out or {}
    hm, B, Cc, H, W, sb, sc = _plane_view(hm, "heatmaps")
    dev = hm.device
    fb = fc = 0
    if hm_flip is not None:
        hm_flip, B2, C2, H2, W2, fb, fc = _plane_view(hm_flip, "flipped heatmaps")
        if (B2, C2, H2, W2) != (B, Cc, H, W) or hm_flip.dtype != hm.dtype:
            raise L.LhnError("flipped heatmaps must match heatmaps in shape and dtype")
    if render is None or render.get("loss_mode", L.LOSS_NONE) == L.LOSS_NONE:
        raise L.LhnError("fused_render_loss_decode needs a loss mode")
    rp = _render_params(render["loss_mode"], render["image_size"], render["sigma"],
                        render.get("unbiased", True), render.get("pos_value", 0.5))
    S = rp.num_stacks
    if Cc % S:
        raise L.LhnError("channel count is not a multiple of the number of stacks")
    K = Cc // S
    joints = _f32c(joints, "joints")
    vis = _f32c(vis, "vis")
    if joints.dim() != 3 or joints.shape[0] != B or joints.shape[2] < 2:
        raise L.LhnError("joints must be [B,K,>=2]")
    if vis.dim() == 2:
        vis = vis.unsqueeze(-1).contiguous()
    if flip_index is not None:
        flip_index = L.require_cuda(flip_index, "flip_index").to(torch.int32).contiguous()
        if flip_index.numel() != K:
            raise L.LhnError("flip_index must have K entries")
    center = _f32c(center, "center")
    scale = _f32c(scale, "scale")
    dp = _decode_params(mask_mode, refine, transform, scale_xy, blur_ksize, use_udp,
                        flags=L.FLAG_OVERLAP_PREVIOUS if overlap_previous else 0)

    def _get(name, shape, dtype, want=True):
        t = out.get(name)
        if t is None and want:
            t = torch.empty(shape, dtype=dtype, device=dev)
        if t is not None and (t.dtype != dtype or t.numel() != int(torch.Size(shape).numel()) or
                              not t.is_contiguous() or t.device != dev):
            raise L.LhnError(f"preallocated output '{name}' has the wrong dtype/size/layout/device")
        return t

    out_hm = _get("hm_kpts", (B, Cc, 3), torch.float32)
    out_k = _get("kpts", (B, Cc, 3), torch.float32)
    out_idx = _get("idx", (B, Cc), torch.int32, want_idx)
    weight = _get("weight", (B, Cc), torch.float32)
    partials = _get("partials", (B * Cc, 4), torch.float64, want_partials)
    sums = _get("sums", (4,), torch.float64)
    loss = _get("loss", (1,), torch.float32, want_loss)
    ws = workspace if workspace is not None else fused_workspace(dev, B, K, S)
    rc = L.lib().lhn_fused_render_loss_decode(
        L.ptr(hm), L.ptr(hm_flip), L.ptr(flip_index), L.dtype_code(hm), B, K, H, W, sb, sc, fb, fc,
        L.ptr(center), L.ptr(scale), C.byref(dp), L.ptr(out_hm), L.ptr(out_k), L.ptr(out_idx),
        C.byref(rp), L.ptr(joints), joints.shape[2], L.ptr(vis), vis.shape[2], L.ptr(weight), L.ptr(partials),
        L.ptr(ws), ws.numel(), L.ptr(sums), int(reduction == "sum"), float(loss_scale), L.ptr(loss), L.stream())
    L.check(rc, "lhn_fused_render_loss_decode")
    res = dict(hm_kpts=out_hm, kpts=out_k, idx=out_idx, weight=weight, sums=sums)
    if loss is not None:
        res["loss"] = loss
    if partials is not None:
        res["partials"] = partials
    return res


def _mask_u8(mask):
    """Boolean joint mask as the uint8 bytes the kernels read: a bool tensor is reinterpreted in place (no
    conversion kernel in front of every launch — it cost ~15 us per call and broke the launch overlap); anything
    else is `!= 0`."""
    mask = L.require_cuda(mask, "mask")
    if mask.dtype == torch.bool:
        return mask.contiguous().view(torch.uint8)
    if mask.dtype == torch.uint8:
        return mask.contiguous()
    return (mask != 0).contiguous().view(torch.uint8)


@_on_device
def decode_heatmap_pck(hm, mask_mode, refine, center, scale, gt, mask, bbox_wh, counters,
                       pck_thr=0.2, auc_nor=30.0, auc_steps=20, blur_ksize=None, overlap_previous=False, out=None):
    """K1 + fused PCK/AUC/EPE counters (BASELINE config 4).  `counters` int64 [(auc_steps+5)*K] is
    ADDED to.  Returns dict(hm_kpts, kpts, idx).  out: optional preallocated hm_kpts / kpts / idx."""
    out = out or {}
    hm, B, K, H, W, sb, sc = _plane_view(hm, "heatmaps")
    dev = hm.device
    dp = _decode_params(mask_mode, refine, L.XFORM_CENTER_SCALE, (1, 1), blur_ksize,
                        flags=L.FLAG_OVERLAP_PREVIOUS if overlap_previous else 0)
    center, scale = _f32c(center, "center"), _f32c(scale, "scale")
    gt = _f32c(gt, "gt")
    bbox_wh = _f32c(bbox_wh, "bbox_wh")
    mask = _mask_u8(mask)
    if counters.dtype != torch.int64 or counters.numel() != (auc_steps + 5) * K or not counters.is_contiguous():
        raise L.LhnError("counters must be a contiguous int64 tensor of (auc_steps+5)*K entries")
    out_hm, out_k, out_idx = out.get("hm_kpts"), out.get("kpts"), out.get("idx")
    if out_hm is None:
        out_hm = torch.empty((B, K, 3), dtype=torch.float32, device=dev)
    if out_k is None:
        out_k = torch.empty((B, K, 3), dtype=torch.float32, device=dev)
    if out_idx is None:
        out_idx = torch.empty((B, K), dtype=torch.int32, device=dev)
    for name, t, dt, n in (("hm_kpts", out_hm, torch.float32, B * K * 3), ("kpts", out_k, torch.float32, B * K * 3),
                           ("idx", out_idx, torch.int32, B * K)):
        if t.dtype != dt or t.numel() != n or not t.is_contiguous() or t.device != dev:
            raise L.LhnError(f"preallocated output '{name}' has the wrong dtype/size/layout/device")
    rc = L.lib().lhn_decode_heatmap_pck(
        L.ptr(hm), L.dtype_code(hm), B, K, H, W, sb, sc, L.ptr(center), L.ptr(scale), C.byref(dp),
        L.ptr(out_hm), L.ptr(out_k), L.ptr(out_idx), L.ptr(gt), L.ptr(mask), L.ptr(bbox_wh),
        float(pck_thr), float(auc_nor), int(auc_steps), L.ptr(counters), L.stream())
    L.check(rc, "lhn_decode_heatmap_pck")
    return dict(hm_kpts=out_hm, kpts=out_k, idx=out_idx)


@_on_device
def loss_partials(output, target, weight, loss_mode, pos_value=0.5):
    """Per-plane sums of DistanceLoss / JointsDistanceLoss against an explicit target tensor."""
    L.require_cuda(output, "output")
    L.require_cuda(target, "target")
    if target.shape != output.shape:
        raise L.LhnError("output and target shapes differ")
    if target.dtype != output.dtype:
        target = target.to(output.dtype)
    output, target = output.contiguous(), target.contiguous()
    H, W = output.shape[-2:]
    P = output.numel() // (H * W)
    weight = _f32c(weight, "target_weight").reshape(-1)
    if weight.numel() != P:
        raise L.LhnError(f"target_weight has {weight.numel()} entries for {P} planes")
    partials = torch.empty((P, 4), dtype=torch.float64, device=output.device)
    rc = L.lib().lhn_loss_partials(L.ptr(output), L.ptr(target), L.ptr(weight), L.dtype_code(output), P,
                                   H * W, int(loss_mode), float(pos_value), L.ptr(partials), L.stream())
    L.check(rc, "lhn_loss_partials")
    return partials


_LOSS_WS = {}


def _loss_workspace(device):
    """Zeroed once per (device, stream); lhn_loss_mse_multi leaves its ticket at zero."""
    key = (str(device), torch.cuda.current_stream(device).cuda_stream)
    ws = _LOSS_WS.get(key)
    if ws is None:
        ws = _LOSS_WS[key] = torch.zeros(int(L.lib().lhn_loss_mse_workspace_bytes()), dtype=torch.uint8, device=device)
    return ws


@_on_device
def loss_mse_multi(outputs, targets, weights, loss_mode, pos_value=0.5, reduction="mean", loss_weights=None, scale=1.0):
    """lhn_loss_mse_multi: DistanceLoss / JointsDistanceLoss of up to 8 (output, target, weight) triples in ONE launch.
    Returns (loss f32[1] = scale * sum_i loss_weights[i] * loss_i, sums f64 [n,4], per_tensor f32 [n])."""
    n = len(outputs)
    if n < 1 or n > L.LOSS_MAX_TENSORS or len(targets) != n or len(weights) != n:
        raise L.LhnError(f"loss_mse_multi takes 1..{L.LOSS_MAX_TENSORS} (output, target, weight) triples")
    dt = outputs[0].dtype
    keep, po, pt, pw, npl, hw = [], [], [], [], [], []
    for o, t, w in zip(outputs, targets, weights):
        L.require_cuda(o, "output")
        L.require_cuda(t, "target")
        if t.shape != o.shape:
            raise L.LhnError("output and target shapes differ")
        if o.dtype != dt:
            raise L.LhnError("all outputs must share one dtype")
        o = o.detach().contiguous()
        t = t.detach().to(dt).contiguous()
        H, W = o.shape[-2:]
        P = o.numel() // (H * W)
        w = _f32c(w.detach(), "target_weight").reshape(-1)
        if w.numel() != P:
            raise L.LhnError(f"target_weight has {w.numel()} entries for {P} planes")
        keep += [o, t, w]
        po.append(o.data_ptr()); pt.append(t.data_ptr()); pw.append(w.data_ptr()); npl.append(P); hw.append(H * W)
    dev = outputs[0].device
    lw = [1.0] * n if loss_weights is None else [float(x) for x in loss_weights]
    sums = torch.empty((n, 4), dtype=torch.float64, device=dev)
    per = torch.empty(n, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    ws = _loss_workspace(dev)
    VP, I64, F32 = C.c_void_p * n, C.c_int64 * n, C.c_float * n
    rc = L.lib().lhn_loss_mse_multi(n, VP(*po), VP(*pt), VP(*pw), I64(*npl), I64(*hw), F32(*lw), L.dtype_code(keep[0]),
                                    int(loss_mode), float(pos_value), int(reduction == "sum"), float(scale), L.ptr(ws),
                                    ws.numel(), L.ptr(sums), L.ptr(per), L.ptr(loss), 0, L.stream())
    L.check(rc, "lhn_loss_mse_multi")
    return loss, sums, per


def _loss_scales(outputs, joints, vis, render, loss_weights, what):
    """Checks the per-scale inputs of the multi-scale rendered-target loss and builds its lhn_loss_scale array.
    Returns (scales, keep-alive list, dtype code, B, K, render params, joints, vis)."""
    n = len(outputs)
    if n < 1 or n > L.LOSS_MAX_TENSORS:
        raise L.LhnError(f"{what} takes 1..{L.LOSS_MAX_TENSORS} scales, got {n}")
    joints = _f32c(joints, "joints")
    vis = _f32c(vis, "vis")
    if vis.dim() == 2:
        vis = vis.unsqueeze(-1).contiguous()
    sig = list(render["sigma"]) if isinstance(render["sigma"], (list, tuple)) else [render["sigma"]] * n
    if len(sig) != n:
        raise L.LhnError(f"{what}: {len(sig)} sigmas for {n} scales")
    lw = [1.0] * n if loss_weights is None else [float(x) for x in loss_weights]
    if len(lw) != n:
        raise L.LhnError(f"{what}: {len(lw)} loss weights for {n} scales")
    rp = _render_params(render["loss_mode"], render["image_size"], 1.0, render.get("unbiased", True),
                        render.get("pos_value", 0.5))
    scales = (L.LossScale * n)()
    keep = []
    B = K = None
    for i, o in enumerate(outputs):
        L.require_cuda(o, f"output {i}")
        if o.device != joints.device:
            raise L.LhnError(f"{what}: output {i} is on {o.device}, the joints on {joints.device}")
        if o.dtype != outputs[0].dtype:
            raise L.LhnError(f"{what}: all outputs must share one dtype ({outputs[0].dtype} and {o.dtype})")
        if o.dim() != 4:
            raise L.LhnError(f"{what}: output {i} must be [B,K,H,W], got {tuple(o.shape)}")
        v, Bi, Ki, H, W, sb, sc = _plane_view(o.detach(), f"output {i}")
        if B is None:
            B, K = Bi, Ki
        elif (Bi, Ki) != (B, K):
            raise L.LhnError(f"{what}: output {i} is [{Bi},{Ki},..], output 0 [{B},{K},..]: B and K must agree")
        keep.append(v)
        s = scales[i]
        s.output, s.stride_b, s.stride_c, s.H, s.W = v.data_ptr(), sb, sc, H, W
        s.sigma, s.loss_weight = float(sig[i]), lw[i]
    if joints.dim() != 3 or joints.shape[0] != B or joints.shape[1] != K or joints.shape[2] < 2:
        raise L.LhnError(f"{what}: joints must be [B={B}, K={K}, >=2], got {tuple(joints.shape)}")
    if vis.dim() != 3 or vis.shape[0] != B or vis.shape[1] != K:
        raise L.LhnError(f"{what}: joints_visible must be [B={B}, K={K}(, >=1)], got {tuple(vis.shape)}")
    return scales, keep, L.dtype_code(keep[0]), B, K, rp, joints, vis


@_on_device
def render_loss_multi(outputs, joints, vis, render, loss_weights=None, reduction="mean", want_weights=True):
    """lhn_render_loss_multi: sum_i loss_weights[i] * DistanceLoss / JointsDistanceLoss of outputs[i] against the
    target rendered in-kernel from the joints (SRHandNetLoss's scales, loss/loss.py:59-66), in ONE launch.
    outputs: up to 8 [B,K,H_i,W_i] tensors of one dtype (channel-sliced views need no copy); joints [B,K,>=2],
    vis [B,K(,>=1)]; render = dict(loss_mode, image_size, sigma (one for every scale, or a list of one per scale),
    unbiased, pos_value).  Returns (loss f32[1], sums f64 [n,4], per_scale f32 [n], weights: a list of [B,K] f32
    target_weight tensors, or None)."""
    scales, keep, dt, B, K, rp, joints, vis = _loss_scales(outputs, joints, vis, render, loss_weights,
                                                           "render_loss_multi")
    n = len(outputs)
    dev = keep[0].device
    weights = None
    if want_weights:
        weights = [torch.empty((B, K), dtype=torch.float32, device=dev) for _ in range(n)]
        for s, w in zip(scales, weights):
            s.out_weight = w.data_ptr()
    sums = torch.empty((n, 4), dtype=torch.float64, device=dev)
    per = torch.empty(n, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    ws = _loss_workspace(dev)
    rc = L.lib().lhn_render_loss_multi(n, scales, dt, B, K, C.byref(rp), L.ptr(joints), joints.shape[2], L.ptr(vis),
                                       vis.shape[2], int(reduction == "sum"), 1.0, L.ptr(ws), ws.numel(), L.ptr(sums),
                                       L.ptr(per), L.ptr(loss), L.stream())
    L.check(rc, "lhn_render_loss_multi")
    return loss, sums, per, weights


@_on_device
def render_loss_backward_multi(outputs, joints, vis, render, sums, loss_weights=None, reduction="mean",
                               grad_out=None, needs=None):
    """lhn_render_loss_backward_multi: d loss / d outputs[i] for render_loss_multi's loss, every scale in ONE launch.
    sums: the forward's f64 [n,4]; grad_out: the upstream gradient (CUDA tensor of one element, None = 1); needs: a
    list of n booleans, the scales whose gradient is wanted (None = all).  Returns a list of contiguous gradients
    like the outputs, None where not wanted."""
    scales, keep, dt, B, K, rp, joints, vis = _loss_scales(outputs, joints, vis, render, loss_weights,
                                                           "render_loss_backward_multi")
    n = len(outputs)
    sums = L.require_cuda(sums, "sums")
    if sums.dtype != torch.float64 or sums.numel() != 4 * n or not sums.is_contiguous():
        raise L.LhnError(f"sums must be a contiguous f64 [{n},4] tensor")
    grads = []
    for i, o in enumerate(outputs):
        if needs is None or needs[i]:
            g = torch.empty(o.shape, dtype=o.dtype, device=o.device)
            scales[i].grad = g.data_ptr()
            grads.append(g)
        else:
            grads.append(None)
    if all(g is None for g in grads):
        return grads
    gkeep, gp = _grad_out_ptr(grad_out, keep[0].device)
    rc = L.lib().lhn_render_loss_backward_multi(n, scales, dt, B, K, C.byref(rp), L.ptr(joints), joints.shape[2],
                                                L.ptr(vis), vis.shape[2], L.ptr(sums), int(reduction == "sum"), gp,
                                                L.stream())
    L.check(rc, "lhn_render_loss_backward_multi")
    return grads


_GRAD_MULTI_WS = {}


def render_loss_grad_multi_workspace(device, n, B, K):
    """Zeroed once per (device, stream), grown when a larger shape comes; lhn_render_loss_grad_multi leaves it zeroed."""
    need = int(L.lib().lhn_render_loss_grad_multi_workspace_bytes(int(n), int(B), int(K)))
    key = (str(device), torch.cuda.current_stream(device).cuda_stream)
    ws = _GRAD_MULTI_WS.get(key)
    if ws is None or ws.numel() < need:
        ws = _GRAD_MULTI_WS[key] = torch.zeros(need, dtype=torch.uint8, device=device)
    return ws


@_on_device
def render_loss_grad_multi(outputs, joints, vis, render, loss_weights=None, reduction="mean", grad_scale=None,
                           needs=None, want_weights=True, workspace=None):
    """render_loss_multi's loss and render_loss_backward_multi's gradients in ONE pass over the outputs
    (lhn_render_loss_grad_multi).  The gradients are those of an upstream gradient ``grad_scale`` (float or one-element
    CUDA tensor; None = 1); needs: a list of n booleans, the scales whose gradient is wanted (None = all; the others are
    still read for the loss).  Returns (loss f32[1], sums f64 [n,4], per_scale f32 [n], gradients: a list of
    contiguous tensors like the outputs, None where not wanted, used_scale f32[1], weights: a list of [B,K] f32
    target_weight tensors, or None)."""
    scales, keep, dt, B, K, rp, joints, vis = _loss_scales(outputs, joints, vis, render, loss_weights,
                                                           "render_loss_grad_multi")
    n = len(outputs)
    dev = keep[0].device
    grads = []
    for i, o in enumerate(outputs):
        if needs is None or needs[i]:
            g = torch.empty(o.shape, dtype=o.dtype, device=dev)
            scales[i].grad = g.data_ptr()
            grads.append(g)
        else:
            grads.append(None)
    weights = None
    if want_weights:
        weights = [torch.empty((B, K), dtype=torch.float32, device=dev) for _ in range(n)]
        for s, w in zip(scales, weights):
            s.out_weight = w.data_ptr()
    sums = torch.empty((n, 4), dtype=torch.float64, device=dev)
    per = torch.empty(n, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    used = torch.empty(1, dtype=torch.float32, device=dev)
    gkeep, gp = (None, None) if grad_scale is None else _scale_tensor(grad_scale, dev)
    ws = workspace if workspace is not None else render_loss_grad_multi_workspace(dev, n, B, K)
    rc = L.lib().lhn_render_loss_grad_multi(n, scales, dt, B, K, C.byref(rp), L.ptr(joints), joints.shape[2],
                                            L.ptr(vis), vis.shape[2], int(reduction == "sum"), 1.0, L.ptr(ws),
                                            ws.numel(), L.ptr(sums), L.ptr(per), L.ptr(loss), gp, L.ptr(used),
                                            L.stream())
    L.check(rc, "lhn_render_loss_grad_multi")
    return loss, sums, per, grads, used, weights


@_on_device
def render_loss_backward_multi_cond(outputs, joints, vis, render, sums, grads, used_scale, loss_weights=None,
                                    reduction="mean", grad_out=None, recomputed=None):
    """Backward of render_loss_grad_multi (lhn_render_loss_backward_multi_cond): ``grads`` (its list, None where not
    wanted) are left as they are when grad_out (None = 1) is bitwise the ``used_scale`` the forward assumed, else
    overwritten as render_loss_backward_multi would write them.  recomputed: optional int32 [1] CUDA tensor, set to 0
    or 1.  Returns grads."""
    scales, keep, dt, B, K, rp, joints, vis = _loss_scales(outputs, joints, vis, render, loss_weights,
                                                           "render_loss_backward_multi_cond")
    n = len(outputs)
    sums = L.require_cuda(sums, "sums")
    if sums.dtype != torch.float64 or sums.numel() != 4 * n or not sums.is_contiguous():
        raise L.LhnError(f"sums must be a contiguous f64 [{n},4] tensor")
    if len(grads) != n:
        raise L.LhnError(f"{len(grads)} gradients for {n} scales")
    for i, (o, g) in enumerate(zip(outputs, grads)):
        if g is None:
            continue
        if g.shape != o.shape or g.dtype != o.dtype or not g.is_contiguous() or g.device != o.device:
            raise L.LhnError(f"gradient {i} must be a contiguous tensor of output {i}'s shape, dtype and device")
        scales[i].grad = g.data_ptr()
    if recomputed is not None and (recomputed.dtype != torch.int32 or recomputed.numel() != 1):
        raise L.LhnError("recomputed must be an int32 tensor of one element")
    gkeep, gp = _grad_out_ptr(grad_out, keep[0].device)
    rc = L.lib().lhn_render_loss_backward_multi_cond(n, scales, dt, B, K, C.byref(rp), L.ptr(joints),
                                                     joints.shape[2], L.ptr(vis), vis.shape[2], L.ptr(sums),
                                                     int(reduction == "sum"), gp, L.ptr(used_scale),
                                                     L.ptr(recomputed), L.stream())
    L.check(rc, "lhn_render_loss_backward_multi_cond")
    return grads


def _grad_out_ptr(grad_out, device):
    if grad_out is None:
        return None, None
    g = L.require_cuda(grad_out, "grad_output").detach().to(torch.float32).reshape(1).contiguous()
    return g, L.ptr(g)


@_on_device
def loss_backward(output, target, weight, loss_mode, sums, pos_value=0.5, reduction="mean", scale=1.0,
                  grad_out=None):
    """d loss / d output for the explicit-target losses (lhn_loss_backward); returns a tensor like output."""
    L.require_cuda(output, "output")
    L.require_cuda(target, "target")
    if target.dtype != output.dtype:
        target = target.to(output.dtype)
    output, target = output.contiguous(), target.contiguous()
    H, W = output.shape[-2:]
    P = output.numel() // (H * W)
    weight = _f32c(weight, "target_weight").reshape(-1)
    grad = torch.empty_like(output)
    keep, gp = _grad_out_ptr(grad_out, output.device)
    rc = L.lib().lhn_loss_backward(L.ptr(output), L.ptr(target), L.ptr(weight), L.dtype_code(output), P, H * W,
                                   int(loss_mode), float(pos_value), L.ptr(sums), int(reduction == "sum"),
                                   float(scale), gp, L.ptr(grad), L.stream())
    L.check(rc, "lhn_loss_backward")
    return grad


@_on_device
def render_loss_backward(hm, joints, vis, render, sums, reduction="mean", scale=1.0, grad_out=None):
    """d loss / d hm for the fused (render-in-kernel) losses (lhn_render_loss_backward)."""
    hm_v, B, Cc, H, W, sb, sc = _plane_view(hm, "heatmaps")
    rp = _render_params(render["loss_mode"], render["image_size"], render["sigma"],
                        render.get("unbiased", True), render.get("pos_value", 0.5))
    K = Cc // rp.num_stacks
    joints = _f32c(joints, "joints")
    vis = _f32c(vis, "vis")
    if vis.dim() == 2:
        vis = vis.unsqueeze(-1).contiguous()
    grad = torch.empty(hm.shape, dtype=hm.dtype, device=hm.device)
    keep, gp = _grad_out_ptr(grad_out, hm.device)
    rc = L.lib().lhn_render_loss_backward(L.ptr(hm_v), L.dtype_code(hm_v), B, K, H, W, sb, sc, C.byref(rp),
                                          L.ptr(joints), joints.shape[2], L.ptr(vis), vis.shape[2], L.ptr(sums),
                                          int(reduction == "sum"), float(scale), gp, L.ptr(grad), L.stream())
    L.check(rc, "lhn_render_loss_backward")
    return grad


_GRAD_WS = {}
_SCALES = {}


def render_loss_grad_workspace(device, B, K, S=1):
    """Zeroed once per (device, stream, size); lhn_render_loss_grad leaves it zeroed."""
    need = int(L.lib().lhn_render_loss_grad_workspace_bytes(int(B), int(K), int(S)))
    key = (str(device), torch.cuda.current_stream(device).cuda_stream)
    ws = _GRAD_WS.get(key)
    if ws is None or ws.numel() < need:
        ws = _GRAD_WS[key] = torch.zeros(need, dtype=torch.uint8, device=device)
    return ws


def _scale_tensor(v, device):
    """A float or a one-element CUDA tensor -> (keep-alive f32 [1] tensor on `device`, pointer)."""
    if isinstance(v, torch.Tensor):
        t = L.require_cuda(v, "grad_scale").detach().to(torch.float32).reshape(1).contiguous()
        return t, L.ptr(t)
    key = (str(device), float(v))
    t = _SCALES.get(key)
    if t is None:                                  # a constant: filled once, the library only reads it
        if len(_SCALES) > 64:
            _SCALES.clear()
        t = _SCALES[key] = torch.full((1,), float(v), dtype=torch.float32, device=device)
    return t, L.ptr(t)


@_on_device
def render_loss_grad(hm, joints, vis, render, reduction="mean", loss_scale=1.0, grad_scale=None, workspace=None):
    """The fused loss and d loss / d hm in ONE pass over hm (lhn_render_loss_grad).  The gradient is the one
    lhn_render_loss_backward computes for an upstream gradient ``grad_scale`` (float or 0-dim CUDA tensor;
    None = 1).  Returns dict(loss f32[1], sums f64[4], weight [B, S*K], grad like hm (contiguous),
    used_scale f32[1])."""
    hm_v, B, Cc, H, W, sb, sc = _plane_view(hm, "heatmaps")
    dev = hm.device
    rp = _render_params(render["loss_mode"], render["image_size"], render["sigma"],
                        render.get("unbiased", True), render.get("pos_value", 0.5))
    S = rp.num_stacks
    if Cc % S:
        raise L.LhnError("channel count is not a multiple of the number of stacks")
    K = Cc // S
    joints = _f32c(joints, "joints")
    vis = _f32c(vis, "vis")
    if joints.dim() != 3 or joints.shape[0] != B or joints.shape[2] < 2:
        raise L.LhnError("joints must be [B,K,>=2]")
    if vis.dim() == 2:
        vis = vis.unsqueeze(-1).contiguous()
    grad = torch.empty(hm.shape, dtype=hm.dtype, device=dev)
    weight = torch.empty((B, Cc), dtype=torch.float32, device=dev)
    sums = torch.empty(4, dtype=torch.float64, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    used = torch.empty(1, dtype=torch.float32, device=dev)
    keep, gp = (None, None) if grad_scale is None else _scale_tensor(grad_scale, dev)
    ws = workspace if workspace is not None else render_loss_grad_workspace(dev, B, K, S)
    rc = L.lib().lhn_render_loss_grad(L.ptr(hm_v), L.dtype_code(hm_v), B, K, H, W, sb, sc, C.byref(rp),
                                      L.ptr(joints), joints.shape[2], L.ptr(vis), vis.shape[2], L.ptr(weight),
                                      L.ptr(ws), ws.numel(), L.ptr(sums), int(reduction == "sum"), float(loss_scale),
                                      L.ptr(loss), gp, L.ptr(used), L.ptr(grad), L.stream())
    L.check(rc, "lhn_render_loss_grad")
    return dict(loss=loss, sums=sums, weight=weight, grad=grad, used_scale=used)


@_on_device
def render_loss_backward_cond(hm, joints, vis, render, sums, grad, used_scale, reduction="mean", scale=1.0,
                              grad_out=None, recomputed=None):
    """Backward of render_loss_grad (lhn_render_loss_backward_cond): ``grad`` is left as it is when grad_out
    (None = 1) is bitwise the ``used_scale`` the forward assumed, else overwritten as render_loss_backward would
    write it.  recomputed: optional int32 [1] CUDA tensor, set to 0 or 1.  Returns grad."""
    hm_v, B, Cc, H, W, sb, sc = _plane_view(hm, "heatmaps")
    rp = _render_params(render["loss_mode"], render["image_size"], render["sigma"],
                        render.get("unbiased", True), render.get("pos_value", 0.5))
    K = Cc // rp.num_stacks
    joints = _f32c(joints, "joints")
    vis = _f32c(vis, "vis")
    if vis.dim() == 2:
        vis = vis.unsqueeze(-1).contiguous()
    if grad.shape != hm.shape or grad.dtype != hm.dtype or not grad.is_contiguous():
        raise L.LhnError("grad must be a contiguous tensor of the heatmaps' shape and dtype")
    if recomputed is not None and (recomputed.dtype != torch.int32 or recomputed.numel() != 1):
        raise L.LhnError("recomputed must be an int32 tensor of one element")
    keep, gp = _grad_out_ptr(grad_out, hm.device)
    rc = L.lib().lhn_render_loss_backward_cond(L.ptr(hm_v), L.dtype_code(hm_v), B, K, H, W, sb, sc, C.byref(rp),
                                               L.ptr(joints), joints.shape[2], L.ptr(vis), vis.shape[2], L.ptr(sums),
                                               int(reduction == "sum"), float(scale), gp, L.ptr(used_scale),
                                               L.ptr(recomputed), L.ptr(grad), L.stream())
    L.check(rc, "lhn_render_loss_backward_cond")
    return grad


@_on_device
def simdr_smoothl1_backward(out_x, out_y, tgt_x, tgt_y, weight, scale=1.0, grad_out=None):
    dt = out_x.dtype
    out_x, out_y = out_x.contiguous(), out_y.to(dt).contiguous()
    tgt_x, tgt_y = tgt_x.to(dt).contiguous(), tgt_y.to(dt).contiguous()
    B, K, Lx = out_x.shape
    Ly = out_y.shape[2]
    weight = _f32c(weight, "target_weight").reshape(B, K)
    nbytes = int(L.lib().lhn_simdr_backward_workspace_bytes(K))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=out_x.device)
    gx, gy = torch.empty_like(out_x), torch.empty_like(out_y)
    keep, gp = _grad_out_ptr(grad_out, out_x.device)
    rc = L.lib().lhn_simdr_smoothl1_backward(L.ptr(out_x), L.ptr(out_y), L.ptr(tgt_x), L.ptr(tgt_y), L.ptr(weight),
                                             L.dtype_code(out_x), B, K, Lx, Ly, float(scale), gp, L.ptr(ws), nbytes,
                                             L.ptr(gx), L.ptr(gy), L.stream())
    L.check(rc, "lhn_simdr_smoothl1_backward")
    return gx, gy


@_on_device
def loss_reduce(partials, sums=None, accumulate=False):
    if sums is None:
        sums = torch.empty(4, dtype=torch.float64, device=partials.device)
    L.check(L.lib().lhn_loss_reduce(L.ptr(partials), partials.shape[0], L.ptr(sums), int(accumulate),
                                    L.stream()), "lhn_loss_reduce")
    return sums


@_on_device
def loss_finalize(sums, loss_mode, reduction="mean", scale=1.0, out=None, accumulate=False):
    if out is None:
        out = torch.empty(1, dtype=torch.float32, device=sums.device)
    L.check(L.lib().lhn_loss_finalize(L.ptr(sums), int(loss_mode), int(reduction == "sum"), float(scale),
                                      L.ptr(out), int(accumulate), L.stream()), "lhn_loss_finalize")
    return out


@_on_device
def render_targets(joints, vis, image_size, heatmap_size, sigma, unbiased=True):
    """Batched TopDownGenerateTarget: target [B,(S,)K,H,W] f32, target_weight [B,(S,)K,1] f32."""
    joints = _f32c(joints, "joints")
    vis = _f32c(vis, "vis")
    if vis.dim() == 2:
        vis = vis.unsqueeze(-1).contiguous()
    B, K = joints.shape[:2]
    W, H = int(heatmap_size[0]), int(heatmap_size[1])
    rp = _render_params(L.LOSS_NONE, image_size, sigma, unbiased)
    S = rp.num_stacks
    stacked = isinstance(sigma, (list, tuple))
    shape = (B, S, K, H, W) if stacked else (B, K, H, W)
    target = torch.empty(shape, dtype=torch.float32, device=joints.device)
    tw = torch.empty(shape[:-2] + (1,), dtype=torch.float32, device=joints.device)
    rc = L.lib().lhn_render_targets(L.ptr(joints), joints.shape[2], L.ptr(vis), vis.shape[2], B, K, H, W,
                                    C.byref(rp), L.ptr(target), L.ptr(tw), L.stream())
    L.check(rc, "lhn_render_targets")
    return target, tw


@_on_device
def render_simdr(joints, vis, image_size, k=2, sigma=2):
    joints = _f32c(joints, "joints")
    vis = _f32c(vis, "vis")
    if vis.dim() == 2:
        vis = vis.unsqueeze(-1).contiguous()
    B, K = joints.shape[:2]
    Lx, Ly = int(image_size[0] * k), int(image_size[1] * k)
    sx = torch.empty((B, K, Lx), dtype=torch.float32, device=joints.device)
    sy = torch.empty((B, K, Ly), dtype=torch.float32, device=joints.device)
    # sigma as a double: the reference's denominator 2 * sigma ** 2 is formed in f64 and rounded to f32 once
    rc = L.lib().lhn_render_simdr_f64sigma(L.ptr(joints), joints.shape[2], L.ptr(vis), vis.shape[2], B, K, Lx, Ly,
                                           float(k), float(sigma), L.ptr(sx), L.ptr(sy), L.stream())
    L.check(rc, "lhn_render_simdr_f64sigma")
    return sx, sy


@_on_device
def decode_simdr(x_vec, y_vec, k=2, center=None, scale=None, nms=False, ranges=None, want_idx=False,
                 overlap_previous=False, out=None):
    """K2.  overlap_previous: as in decode_heatmap (rotating buffers; honoured by the ring kernel).
    out: optional preallocated contiguous f32 [B,K,3]."""
    L.require_cuda(x_vec, "x_vectors")
    L.require_cuda(y_vec, "y_vectors")
    if y_vec.dtype != x_vec.dtype:
        y_vec = y_vec.to(x_vec.dtype)
    x_vec, y_vec = x_vec.contiguous(), y_vec.contiguous()
    B, K, Lx = x_vec.shape
    Ly = y_vec.shape[2]
    center, scale = _f32c(center, "center"), _f32c(scale, "scale")
    if ranges is not None:
        ranges = L.require_cuda(ranges, "ranges").to(torch.int32).contiguous()
    if out is None:
        out = torch.empty((B, K, 3), dtype=torch.float32, device=x_vec.device)
    elif out.dtype != torch.float32 or out.numel() != B * K * 3 or not out.is_contiguous() or out.device != x_vec.device:
        raise L.LhnError("preallocated output has the wrong dtype/size/layout/device")
    idx = torch.empty((B, K, 2), dtype=torch.int32, device=x_vec.device) if want_idx else None
    rc = L.lib().lhn_decode_simdr_flags(L.ptr(x_vec), L.ptr(y_vec), L.dtype_code(x_vec), B, K, Lx, Ly, int(k),
                                        L.ptr(center), L.ptr(scale), int(bool(nms)), L.ptr(ranges), L.ptr(out),
                                        L.ptr(idx), L.FLAG_OVERLAP_PREVIOUS if overlap_previous else 0, L.stream())
    L.check(rc, "lhn_decode_simdr")
    return (out, idx) if want_idx else out


@_on_device
def simdr_smoothl1(out_x, out_y, tgt_x, tgt_y, weight):
    for n, t in (("output_x", out_x), ("output_y", out_y), ("target_x", tgt_x), ("target_y", tgt_y)):
        L.require_cuda(t, n)
    dt = out_x.dtype
    out_x, out_y = out_x.contiguous(), out_y.to(dt).contiguous()
    tgt_x, tgt_y = tgt_x.to(dt).contiguous(), tgt_y.to(dt).contiguous()
    B, K, Lx = out_x.shape
    Ly = out_y.shape[2]
    weight = _f32c(weight, "target_weight").reshape(B, K)
    nbytes = L.lib().lhn_simdr_loss_workspace_bytes(B, K)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=out_x.device)
    loss = torch.empty(1, dtype=torch.float32, device=out_x.device)
    rc = L.lib().lhn_simdr_smoothl1(L.ptr(out_x), L.ptr(out_y), L.ptr(tgt_x), L.ptr(tgt_y), L.ptr(weight),
                                    L.dtype_code(out_x), B, K, Lx, Ly, L.ptr(ws), nbytes, L.ptr(loss),
                                    L.stream())
    L.check(rc, "lhn_simdr_smoothl1")
    return loss


@_on_device
def split_bf16(x):
    """lhn_split_bf16: f32 tensor -> (hi, lo) bf16 tensors of the same shape with x = hi + lo + O(2^-17 |x|)."""
    L.require_cuda(x, "x")
    x = x.detach()
    if x.dtype != torch.float32 or not x.is_contiguous():
        x = x.to(torch.float32).contiguous()
    if x.numel() % 4:
        raise L.LhnError("split_bf16 needs a multiple of 4 elements")
    hi = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    lo = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    L.check(L.lib().lhn_split_bf16(L.ptr(x), x.numel(), L.ptr(hi), L.ptr(lo), L.stream()), "lhn_split_bf16")
    return hi, lo


@_on_device
def simdr_heads_loss(heatmap, w_split, bias, tgt_x, tgt_y, weight, want_dpred=False, want_pred=False):
    """lhn_simdr_heads_loss: SimDRLoss.forward with both linear heads in ONE tcgen05 kernel (the predictions stay in
    tensor memory).  heatmap f32 [B,K,H,W]; w_split = split_bf16(cat([Wx, Wy])) ([Lx+Ly, H*W] each); bias f32 [Lx+Ly];
    tgt_x [B,K,Lx], tgt_y [B,K,Ly], weight [B,K(,1)].  Returns (loss f32[1], dpred or None, pred or None)."""
    L.require_cuda(heatmap, "heatmap")
    B, K = heatmap.shape[:2]
    Kd = heatmap[0, 0].numel()
    w_hi, w_lo = w_split
    N = w_hi.shape[0]
    tgt_x, tgt_y = _f32c(tgt_x, "simdr_x"), _f32c(tgt_y, "simdr_y")
    Lx, Ly = tgt_x.shape[-1], tgt_y.shape[-1]
    if Lx + Ly != N or w_hi.shape[1] != Kd or tgt_x.shape[:2] != (B, K) or tgt_y.shape[:2] != (B, K):
        raise L.LhnError("simdr_heads_loss: shapes of the heads, the heatmap and the targets do not agree")
    hm = heatmap.detach()
    if hm.dtype != torch.float32 or not hm.is_contiguous():
        hm = hm.to(torch.float32).contiguous()
    bias = _f32c(bias, "bias")
    weight = _f32c(weight, "target_weight").reshape(B, K)
    dev = heatmap.device
    # one C call: the bf16 split of the heatmaps goes into the workspace, then the GEMM + loss kernel and its finalise
    nbytes = int(L.lib().lhn_simdr_heads_f32_workspace_bytes(B, K, Kd, Lx, Ly))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    dpred = torch.empty((B * K, N), dtype=torch.float32, device=dev) if want_dpred else None
    pred = torch.empty((B * K, N), dtype=torch.float32, device=dev) if want_pred else None
    L.check(L.lib().lhn_simdr_heads_loss_f32(L.ptr(hm), L.ptr(w_hi), L.ptr(w_lo), L.ptr(bias), L.ptr(tgt_x), L.ptr(tgt_y),
                                             L.ptr(weight), B, K, Kd, Lx, Ly, L.ptr(ws), nbytes, L.ptr(loss), L.ptr(dpred),
                                             L.ptr(pred), L.stream()), "lhn_simdr_heads_loss_f32")
    return loss, dpred, pred


@_on_device
def pck_accumulate(pred, gt, mask, thr, normalize=None, norm_const=1.0, counters=None):
    """Adds hits[T,K], valid[K], dist_fix[K] (int64, [(T+2)*K]) for one shard of samples."""
    L.require_cuda(pred, "pred")
    L.require_cuda(gt, "gt")
    if pred.dtype not in (torch.float32, torch.float64):
        pred = pred.float()
    if gt.dtype not in (torch.float32, torch.float64):
        gt = gt.float()
    pred, gt = pred.contiguous(), gt.contiguous()
    N, K = pred.shape[:2]
    mask = _mask_u8(mask)
    if normalize is not None:
        L.require_cuda(normalize, "normalize")
        if normalize.dtype not in (torch.float32, torch.float64):
            normalize = normalize.double()
        normalize = normalize.contiguous()
    T = len(thr)
    if counters is None:
        counters = torch.zeros((T + 2) * K, dtype=torch.int64, device=pred.device)
    thr_arr = (C.c_float * max(T, 1))(*[float(t) for t in thr])
    rc = L.lib().lhn_pck_accumulate(L.ptr(pred), L.dtype_code(pred), pred.shape[2], L.ptr(gt),
                                    L.dtype_code(gt), gt.shape[2], L.ptr(mask), L.ptr(normalize),
                                    L.dtype_code(normalize) if normalize is not None else L.F64,
                                    float(norm_const), N, K, thr_arr, T, L.ptr(counters), L.stream())
    L.check(rc, "lhn_pck_accumulate")
    return counters


@_on_device
def metrics_finalize(counters, K, auc_steps=20, out=None):
    """lhn_metrics_finalize: f64 [3 + K] = (PCK, AUC, EPE, per-joint PCK accuracies) from the fused counter block,
    computed on the device (no sync, no device->host copy)."""
    L.require_cuda(counters, "counters")
    if counters.dtype != torch.int64 or not counters.is_contiguous() or counters.numel() != (auc_steps + 5) * K:
        raise L.LhnError("counters must be a contiguous int64 tensor of (auc_steps+5)*K entries")
    if out is None:
        out = torch.empty(3 + K, dtype=torch.float64, device=counters.device)
    L.check(L.lib().lhn_metrics_finalize(L.ptr(counters), int(K), int(auc_steps), L.ptr(out), L.stream()),
            "lhn_metrics_finalize")
    return out


@_on_device
def evaluate_pck(pred_hm, gt_hm, bbox_wh, weight, image_size, thr):
    L.require_cuda(pred_hm, "pred_keypoints_hm")
    L.require_cuda(gt_hm, "gt_keypoints_hm")
    if gt_hm.dtype != pred_hm.dtype:
        gt_hm = gt_hm.to(pred_hm.dtype)
    pred_hm, gt_hm = pred_hm.contiguous(), gt_hm.contiguous()
    B, K, H, W = pred_hm.shape
    bbox_wh = _f32c(bbox_wh, "bbox")
    weight = None if weight is None else _f32c(weight, "target_weight").reshape(B, K)
    nbytes = L.lib().lhn_evaluate_pck_workspace_bytes(B, K)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=pred_hm.device)
    pck = torch.empty(B, dtype=torch.float32, device=pred_hm.device)
    mean = torch.empty(1, dtype=torch.float64, device=pred_hm.device)
    rc = L.lib().lhn_evaluate_pck(L.ptr(pred_hm), L.ptr(gt_hm), L.dtype_code(pred_hm), B, K, H, W,
                                  L.ptr(bbox_wh), L.ptr(weight), float(image_size[0]), float(image_size[1]),
                                  float(thr), L.ptr(ws), nbytes, L.ptr(pck), L.ptr(mean), L.stream())
    L.check(rc, "lhn_evaluate_pck")
    return pck, mean


@_on_device
def flip_back(x, flip_index=None):
    L.require_cuda(x, "output_flipped")
    x = x.contiguous()
    B, K, H, W = x.shape
    if flip_index is not None:
        flip_index = L.require_cuda(flip_index, "flip_index").to(torch.int32).contiguous()
    out = torch.empty_like(x)
    L.check(L.lib().lhn_flip_back(L.ptr(x), L.ptr(out), L.dtype_code(x), B, K, H, W, L.ptr(flip_index),
                                  L.stream()), "lhn_flip_back")
    return out


# ---- region-map bbox decode and point / window restricted refinements (SURVEY §8f rank 4) --------------------
def region_bbox_decode(center, size, mode, nms_kernel=11, num_candidates=10, max_num_bbox=1, avg_kernel=3,
                       refine=L.REFINE_NONE, blur_ksize=19, image_size=(256, 256), stride=(4.0, 4.0), cand_thr=0.1,
                       det_thr=0.1, iou_thr=0.6, min_wh=2.0, max_wh=4096.0, nms_inplace=False, want_nms=False):
    """lhn_region_bbox_decode.  center [B,1,H,W] and size [B,2,H,W] may be channel slices of one region map
    (no copy).  Returns dict(candidates [B,N,5], boxes [B,max_num_bbox,5], counts [B] int32[, nms [B,1,H,W]]).
    nms_inplace: write the NMS'd centre map over `center` (the reference's in-place heatmaps *= mask)."""
    L.require_cuda(center, "center_maps")
    L.require_cuda(size, "size_maps")
    if center.dim() != 4 or center.shape[1] != 1 or size.dim() != 4 or size.shape[1] != 2:
        raise L.LhnError("center_maps must be [B,1,H,W] and size_maps [B,2,H,W]")
    B, _, H, W = center.shape
    if size.shape[0] != B or tuple(size.shape[2:]) != (H, W) or size.dtype != center.dtype:
        raise L.LhnError("size_maps must match center_maps in batch, plane size and dtype")

    def planes_ok(t):
        return t.stride(3) == 1 and t.stride(2) == W

    if not planes_ok(center):
        if nms_inplace:
            raise L.LhnError("in-place NMS needs contiguous centre planes")
        center = center.contiguous()
    if not planes_ok(size) or size.stride(1) < H * W:
        size = size.contiguous()
    rp = L.RegionParams()
    rp.mode, rp.nms_kernel, rp.num_candidates, rp.max_num_bbox = int(mode), int(nms_kernel), int(num_candidates), int(max_num_bbox)
    rp.avg_kernel, rp.refine, rp.blur_ksize = int(avg_kernel), int(refine), int(blur_ksize)
    rp.image_w, rp.image_h = float(image_size[0]), float(image_size[1])
    rp.stride_x, rp.stride_y = float(stride[0]), float(stride[1])
    rp.cand_thr, rp.det_thr, rp.min_wh, rp.max_wh, rp.iou_thr = float(cand_thr), float(det_thr), float(min_wh), float(max_wh), float(iou_thr)
    if refine == L.REFINE_DARK_LEGACY:
        for i, t in enumerate(L.gaussian_taps(int(blur_ksize))):
            rp.taps[i] = t
    dev = center.device
    nms = None
    if nms_inplace:
        nms = center
    elif want_nms:
        nms = torch.empty((B, 1, H, W), dtype=center.dtype, device=dev)
        if nms.stride(0) != center.stride(0):
            center = center.contiguous()
    cand = torch.empty((B, int(num_candidates), 5), dtype=torch.float32, device=dev)
    boxes = torch.empty((B, int(max_num_bbox), 5), dtype=torch.float32, device=dev)
    counts = torch.empty((B,), dtype=torch.int32, device=dev)
    L.check(L.lib().lhn_region_bbox_decode(L.ptr(center), L.ptr(size), L.dtype_code(center), B, H, W,
                                           center.stride(0), size.stride(0), size.stride(1), C.byref(rp),
                                           L.ptr(nms), L.ptr(cand), L.ptr(boxes), L.ptr(counts), L.stream()),
            "lhn_region_bbox_decode")
    r = dict(candidates=cand, boxes=boxes, counts=counts)
    if nms is not None:
        r["nms"] = nms
    return r


@_on_device
def box_nms(candidates, det_thr=0.1, iou_thr=0.6, max_num=1, min_wh=2.0, max_wh=4096.0):
    """lhn_box_nms on candidates [B,N,5] -> (boxes [B,max_num,5], counts [B] int32)."""
    c = _f32c(candidates, "candidates")
    if c.dim() != 3 or c.shape[2] != 5 or c.shape[1] > L.MAX_CANDIDATES:
        raise L.LhnError(f"candidates must be [B, N <= {L.MAX_CANDIDATES}, 5]")
    B, N = c.shape[:2]
    max_num = min(int(max_num), N)
    boxes = torch.empty((B, max_num, 5), dtype=torch.float32, device=c.device)
    counts = torch.empty((B,), dtype=torch.int32, device=c.device)
    L.check(L.lib().lhn_box_nms(L.ptr(c), B, N, float(det_thr), float(min_wh), float(max_wh), float(iou_thr), max_num,
                                L.ptr(boxes), L.ptr(counts), L.stream()), "lhn_box_nms")
    return boxes, counts


@_on_device
def heatmap_nms(hm, nms_kernel=11, inplace=False):
    """lhn_heatmap_nms: hm * eq(maxpool_k(hm), hm) on [B,C,H,W]; inplace=True overwrites hm as the reference does."""
    L.require_cuda(hm, "heatmaps")
    if hm.dim() != 4:
        raise L.LhnError("heatmaps must be [B,C,H,W]")
    B, Cc, H, W = hm.shape
    ok = hm.stride(3) == 1 and hm.stride(2) == W and (Cc == 1 or hm.stride(1) >= H * W)
    if not ok:
        if inplace:
            raise L.LhnError("in-place NMS needs contiguous planes")
        hm = hm.contiguous()
    out = hm if inplace else torch.empty_strided(hm.shape, hm.stride(), dtype=hm.dtype, device=hm.device)
    L.check(L.lib().lhn_heatmap_nms(L.ptr(hm), L.ptr(out), L.dtype_code(hm), B, Cc, H, W, hm.stride(0),
                                    hm.stride(1) if Cc > 1 else H * W, int(nms_kernel), L.stream()), "lhn_heatmap_nms")
    return out


@_on_device
def vector_nms(v):
    """lhn_vector_nms on [..., L] (returns a new tensor)."""
    L.require_cuda(v, "vector")
    v = v.contiguous()
    out = torch.empty_like(v)
    Ln = v.shape[-1]
    L.check(L.lib().lhn_vector_nms(L.ptr(v), L.ptr(out), L.dtype_code(v), v.numel() // max(Ln, 1), Ln, L.stream()),
            "lhn_vector_nms")
    return out


@_on_device
def refine_points(hm, bc, xy, plus_half=False):
    """lhn_refine_points: the +-0.25 rule at given positions.  bc int32 [n,2] (image, channel), xy f32 [n,>=2]
    (updated in place and returned)."""
    hm, B, Cc, H, W, sb, sc = _plane_view(hm, "heatmaps")
    bc = L.require_cuda(bc, "bc").to(torch.int32).contiguous()
    L.require_cuda(xy, "xy")
    if xy.dtype != torch.float32 or not xy.is_contiguous() or xy.dim() != 2 or xy.shape[1] < 2:
        raise L.LhnError("xy must be a contiguous f32 [n,>=2] tensor")
    n = xy.shape[0]
    if bc.shape != (n, 2):
        raise L.LhnError("bc must be [n,2]")
    L.check(L.lib().lhn_refine_points(L.ptr(hm), L.dtype_code(hm), B, Cc, H, W, sb, sc, L.ptr(bc), L.ptr(xy),
                                      xy.shape[1], n, L.REFINE_OFFSET_HALF if plus_half else L.REFINE_OFFSET,
                                      L.stream()), "lhn_refine_points")
    return xy


@_on_device
def decode_heatmap_roi(hm, roi, refine, scale_xy=(1.0, 1.0), blur_ksize=None, want_idx=False):
    """lhn_decode_heatmap_roi: per-image window roi int32 [B,4] = (x0, y0, x1, y1) -> [B,K,3] (X, Y, score)."""
    hm, B, Cc, H, W, sb, sc = _plane_view(hm, "heatmaps")
    roi = L.require_cuda(roi, "roi").to(torch.int32).contiguous()
    if roi.shape != (B, 4):
        raise L.LhnError("roi must be [B,4]")
    dp = _decode_params(L.MASK_NONE, refine, L.XFORM_SCALE, scale_xy, blur_ksize)
    out = torch.empty((B, Cc, 3), dtype=torch.float32, device=hm.device)
    idx = torch.empty((B, Cc), dtype=torch.int32, device=hm.device) if want_idx else None
    L.check(L.lib().lhn_decode_heatmap_roi(L.ptr(hm), L.dtype_code(hm), B, Cc, H, W, sb, sc, L.ptr(roi), C.byref(dp),
                                           L.ptr(out), L.ptr(idx), L.stream()), "lhn_decode_heatmap_roi")
    return (out, idx) if want_idx else out


@_on_device
def render_region_wh(rect, gamma, H, W, out=None):
    """lhn_render_region_wh: rect int32 [B,4] = (x1, x2, y1, y2), gamma f32 [B,2] -> [B,2,H,W] f32; `out` may be a
    two-channel slice of a larger contiguous [B,C,H,W] target."""
    rect = L.require_cuda(rect, "rect").to(torch.int32).contiguous()
    gamma = _f32c(gamma, "gamma")
    B = rect.shape[0]
    if rect.shape != (B, 4) or gamma.shape != (B, 2):
        raise L.LhnError("rect must be [B,4] and gamma [B,2]")
    if out is None:
        out = torch.empty((B, 2, H, W), dtype=torch.float32, device=rect.device)
    if out.dtype != torch.float32 or tuple(out.shape) != (B, 2, H, W) or out.stride(3) != 1 or out.stride(2) != W \
            or out.stride(1) != H * W:
        raise L.LhnError("out must be an f32 [B,2,H,W] view with contiguous planes")
    L.check(L.lib().lhn_render_region_wh(L.ptr(rect), L.ptr(gamma), B, H, W, L.ptr(out), out.stride(0) if B > 1 else 2 * H * W,
                                         L.stream()), "lhn_render_region_wh")
    return out


@_on_device
def dark_refine_points(hm, bc, xy, blur_ksize=19):
    """lhn_dark_refine_points: the legacy DARK at given positions.  bc int32 [n,2] (image, channel), xy f32 [n,>=2]
    (updated in place and returned)."""
    hm, B, Cc, H, W, sb, sc = _plane_view(hm, "heatmaps")
    bc = L.require_cuda(bc, "bc").to(torch.int32).contiguous()
    L.require_cuda(xy, "xy")
    if xy.dtype != torch.float32 or not xy.is_contiguous() or xy.dim() != 2 or xy.shape[1] < 2:
        raise L.LhnError("xy must be a contiguous f32 [n,>=2] tensor")
    n = xy.shape[0]
    if bc.shape != (n, 2):
        raise L.LhnError("bc must be [n,2]")
    dp = _decode_params(L.MASK_NONE, L.REFINE_DARK_LEGACY, L.XFORM_NONE, blur_ksize=blur_ksize)
    L.check(L.lib().lhn_dark_refine_points(L.ptr(hm), L.dtype_code(hm), B, Cc, H, W, sb, sc, L.ptr(bc), L.ptr(xy),
                                           xy.shape[1], n, C.byref(dp), L.stream()), "lhn_dark_refine_points")
    return xy
