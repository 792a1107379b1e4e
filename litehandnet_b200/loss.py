"""Drop-in mirrors of the reference's loss modules (loss/heatmapLoss.py, loss/centernet_simdr_loss.py,
loss/loss.py, loss/__init__.py) — same class names, constructor arguments, call signatures, return
types and error behaviour; the arithmetic runs in the CUDA library.

Scope (SURVEY.md §8a L1-L5): L2-type DistanceLoss (balance on/off, mean/sum), JointsDistanceLoss mse,
KLDiscretLoss, SimDRLoss, TopdownHeatmapLoss, SRHandNetLoss (heatmap-only branch), get_loss.

Autograd (SURVEY §8f rank 1): every loss is a torch.autograd.Function whose backward is one streaming CUDA
kernel (lhn_loss_backward / lhn_render_loss_backward / lhn_simdr_smoothl1_backward) driven by the forward's
f64 sums, so ``loss, d = criterion(outputs, meta); loss.backward()`` works as in
train/topdown_trainer.py:68-87.  Gradients flow to the network output only (targets and weights are data).
"""
import torch
from torch import nn

from . import _lib as L
from . import ops


def _as_cuda(t, device):
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(t)
    return t.to(device)          # the reference moves meta['target'] to the output's device (loss.py:97-98)


class _HeatmapLossFn(torch.autograd.Function):
    """forward: ONE launch (lhn_loss_mse_multi: streaming sums, fixed-order two-level reduction, finalisation);
    backward: lhn_loss_backward."""

    @staticmethod
    def forward(ctx, output, target, weight, mode, value, reduction):
        loss, sums, _ = ops.loss_mse_multi([output], [target], [weight], mode, value, reduction)
        sums = sums[0]
        ctx.save_for_backward(output.detach(), target, weight, sums)
        ctx.cfg = (mode, value, reduction)
        return loss[0]

    @staticmethod
    def backward(ctx, grad_out):
        output, target, weight, sums = ctx.saved_tensors
        mode, value, reduction = ctx.cfg
        g = ops.loss_backward(output, target, weight, mode, sums, value, reduction, 1.0, grad_out)
        return g, None, None, None, None, None


class _MultiHeatmapLossFn(torch.autograd.Function):
    """sum_i loss_weight[i] * DistanceLoss(outputs[i], targets[i], w[i]) in ONE launch (SRHandNetLoss's four scales,
    loss/loss.py:59-66); backward: one lhn_loss_backward per tensor, scaled by its loss weight."""

    @staticmethod
    def forward(ctx, mode, value, reduction, loss_weights, n, *tensors):
        outputs, targets, weights = tensors[:n], tensors[n:2 * n], tensors[2 * n:3 * n]
        loss, sums, _ = ops.loss_mse_multi(list(outputs), list(targets), list(weights), mode, value, reduction, loss_weights)
        ctx.save_for_backward(*[o.detach() for o in outputs], *targets, *weights, sums)
        ctx.cfg = (mode, value, reduction, [float(x) for x in loss_weights], n)
        return loss[0]

    @staticmethod
    def backward(ctx, grad_out):
        mode, value, reduction, lw, n = ctx.cfg
        saved = ctx.saved_tensors
        outputs, targets, weights, sums = saved[:n], saved[n:2 * n], saved[2 * n:3 * n], saved[3 * n]
        grads = []
        for i in range(n):
            if ctx.needs_input_grad[5 + i]:
                grads.append(ops.loss_backward(outputs[i], targets[i], weights[i], mode, sums[i], value, reduction, lw[i], grad_out))
            else:
                grads.append(None)
        return (None, None, None, None, None, *grads, *([None] * (2 * n)))


class _FusedMultiHeatmapLossFn(torch.autograd.Function):
    """SRHandNetLoss's scales with every target rendered in-kernel from the joints: ONE launch forward
    (lhn_render_loss_multi), ONE launch backward (lhn_render_loss_backward_multi) for the outputs that need a
    gradient."""

    @staticmethod
    def forward(ctx, render, reduction, loss_weights, joints, vis, *outputs):
        outs = [o.detach() for o in outputs]
        loss, sums, _, _ = ops.render_loss_multi(outs, joints, vis, render, loss_weights, reduction, want_weights=False)
        ctx.save_for_backward(joints, vis, sums, *outs)
        ctx.cfg = (render, reduction, loss_weights)
        return loss[0]

    @staticmethod
    def backward(ctx, grad_out):
        joints, vis, sums, *outs = ctx.saved_tensors
        render, reduction, lw = ctx.cfg
        grads = ops.render_loss_backward_multi(outs, joints, vis, render, sums, lw, reduction, grad_out,
                                               needs=list(ctx.needs_input_grad[5:]))
        return (None, None, None, None, None, *grads)


class _FusedMultiHeatmapLossOnePassFn(torch.autograd.Function):
    """SRHandNetLoss's scales with the gradients written in the forward (lhn_render_loss_grad_multi: one read of the
    outputs, one write of the gradients of those that need one).  The gradients assume the upstream value
    ``expected``; the backward (lhn_render_loss_backward_multi_cond) returns them as they are when autograd delivers
    exactly that value, and rewrites them as the two-launch backward would otherwise.  The gradient buffers are
    allocated here, in the forward."""

    @staticmethod
    def forward(ctx, render, reduction, loss_weights, expected, joints, vis, *outputs):
        outs = [o.detach() for o in outputs]
        loss, sums, _, grads, used, _ = ops.render_loss_grad_multi(outs, joints, vis, render, loss_weights, reduction,
                                                                   expected, needs=list(ctx.needs_input_grad[6:]),
                                                                   want_weights=False)
        ctx.save_for_backward(joints, vis, sums, used, *outs)
        # the gradients are intermediates, kept on ctx and released in backward: handed back with no other reference,
        # autograd adopts them as the outputs' .grad instead of copying them
        ctx.grads = grads
        ctx.cfg = (render, reduction, loss_weights)
        return loss[0]

    @staticmethod
    def backward(ctx, grad_out):
        joints, vis, sums, used, *outs = ctx.saved_tensors
        grads, ctx.grads = ctx.grads, None
        render, reduction, lw = ctx.cfg
        ops.render_loss_backward_multi_cond(outs, joints, vis, render, sums, grads, used, lw, reduction, grad_out,
                                            recomputed=_ONE_PASS_PROBE.get("recomputed"))
        return (None, None, None, None, None, None, *grads)


class _FusedHeatmapLossFn(torch.autograd.Function):
    """The fused entry: target rendered in-kernel from the joints, one launch forward
    (lhn_fused_render_loss_decode without a refinement), lhn_render_loss_backward backward."""

    @staticmethod
    def forward(ctx, output, joints, vis, render, reduction):
        r = ops.fused_render_loss_decode(output.detach(), L.MASK_NEG1, L.REFINE_NONE, L.XFORM_NONE, None, None,
                                         render, joints, vis, want_idx=False, reduction=reduction)
        ctx.save_for_backward(output.detach(), joints, vis, r["sums"])
        ctx.cfg = (render, reduction)
        ctx.mark_non_differentiable(r["weight"])
        return r["loss"][0], r["weight"]

    @staticmethod
    def backward(ctx, grad_out, _grad_w):
        output, joints, vis, sums = ctx.saved_tensors
        render, reduction = ctx.cfg
        return ops.render_loss_backward(output, joints, vis, render, sums, reduction, 1.0, grad_out), None, None, None, None


class _FusedHeatmapLossOnePassFn(torch.autograd.Function):
    """The fused entry with the gradient written in the forward (lhn_render_loss_grad: one read of the output,
    one write of the gradient).  The gradient assumes the upstream value ``expected``; the backward
    (lhn_render_loss_backward_cond) returns it as is when autograd delivers exactly that value, and rewrites it
    as the two-pass backward would otherwise.  The gradient buffer is allocated here, in the forward."""

    @staticmethod
    def forward(ctx, output, joints, vis, render, reduction, expected):
        r = ops.render_loss_grad(output.detach(), joints, vis, render, reduction, 1.0, expected)
        ctx.save_for_backward(output.detach(), joints, vis, r["sums"], r["used_scale"])
        # the gradient is an intermediate, kept on ctx and released in backward: handed back with no other
        # reference, autograd adopts it as output.grad instead of copying it
        ctx.grad = r["grad"]
        ctx.cfg = (render, reduction)
        ctx.mark_non_differentiable(r["weight"])
        return r["loss"][0], r["weight"]

    @staticmethod
    def backward(ctx, grad_out, _grad_w):
        output, joints, vis, sums, used = ctx.saved_tensors
        grad, ctx.grad = ctx.grad, None
        render, reduction = ctx.cfg
        g = ops.render_loss_backward_cond(output, joints, vis, render, sums, grad, used, reduction, 1.0, grad_out,
                                          recomputed=_ONE_PASS_PROBE.get("recomputed"))
        del grad
        return g, None, None, None, None, None


# tests: an int32 [1] CUDA tensor under "recomputed" receives which branch the conditional backward took
_ONE_PASS_PROBE = {}


class _SimDRLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, out_x, out_y, tgt_x, tgt_y, weight):
        ctx.save_for_backward(out_x.detach(), out_y.detach(), tgt_x, tgt_y, weight)
        return ops.simdr_smoothl1(out_x.detach(), out_y.detach(), tgt_x, tgt_y, weight)[0]

    @staticmethod
    def backward(ctx, grad_out):
        out_x, out_y, tgt_x, tgt_y, weight = ctx.saved_tensors
        gx, gy = ops.simdr_smoothl1_backward(out_x, out_y, tgt_x, tgt_y, weight, 1.0, grad_out)
        return gx, gy.to(out_y.dtype), None, None, None


class _SimDRHeadsLossFn(torch.autograd.Function):
    """SimDRLoss.forward with the two linear heads fused into the loss kernel (lhn_simdr_heads_loss).  When a
    gradient is needed the kernel's epilogue also stores g = d SmoothL1 / d pred = clamp(pred - target, -1, 1); the
    backward scales its rows by grad * mean_b(w[b, j]) / (B * L * K) and takes the three plain GEMMs of a linear layer
    (d heatmap = G W, d W = G^T A, d b = column sums of G) from the library."""

    @staticmethod
    def forward(ctx, heatmap, wx, bx, wy, by, tgt_x, tgt_y, weight, w_split):
        need = any(ctx.needs_input_grad[:5])
        bias = torch.cat([bx.detach(), by.detach()])
        loss, dpred, _ = ops.simdr_heads_loss(heatmap.detach(), w_split, bias, tgt_x, tgt_y, weight, want_dpred=need)
        if need:
            ctx.save_for_backward(heatmap.detach(), wx.detach(), wy.detach(), weight, dpred)
            ctx.Lx, ctx.Ly = tgt_x.shape[-1], tgt_y.shape[-1]
        return loss[0]

    @staticmethod
    def backward(ctx, grad_out):
        heatmap, wx, wy, weight, g = ctx.saved_tensors
        B, K = heatmap.shape[:2]
        Lx, Ly = ctx.Lx, ctx.Ly
        A = heatmap.reshape(B * K, -1).float()
        mw = weight.reshape(B, K).float().mean(0)                          # mean_b w[b, j]
        row = (grad_out.float() * mw / float(K * B)).repeat(B)              # coefficient of row b*K + j, without 1/L
        g = g * row[:, None]
        gx, gy = g[:, :Lx] * (1.0 / Lx), g[:, Lx:] * (1.0 / Ly)
        d_hm = d_wx = d_bx = d_wy = d_by = None
        if ctx.needs_input_grad[0]:
            d_hm = (gx @ wx.float() + gy @ wy.float()).reshape(heatmap.shape).to(heatmap.dtype)
        if ctx.needs_input_grad[1]:
            d_wx = gx.t() @ A
        if ctx.needs_input_grad[2]:
            d_bx = gx.sum(0)
        if ctx.needs_input_grad[3]:
            d_wy = gy.t() @ A
        if ctx.needs_input_grad[4]:
            d_by = gy.sum(0)
        return d_hm, d_wx, d_bx, d_wy, d_by, None, None, None, None


class DistanceLoss(nn.Module):
    """loss/heatmapLoss.py:228-265.  Only loss_type 'L2' is on the path (every config uses it)."""

    def __init__(self, loss_type='L2', reduction='mean', balance=True, value=0.5):
        super().__init__()
        assert reduction in ['mean', 'sum', None], f"Error: {reduction=}"
        if loss_type.lower() != 'l2':
            raise NotImplementedError("only DistanceLoss(loss_type='L2') is on the B200 hot path "
                                      "(SURVEY.md §2 row 1); L1/SmoothL1 are unused by every config")
        if reduction is None:
            raise NotImplementedError("reduction=None (unreduced loss map) is not on the hot path")
        self.reduction = reduction
        self.value = value
        self.balance = balance

    @property
    def _mode(self):
        return L.LOSS_DISTANCE_BALANCE if self.balance else L.LOSS_DISTANCE

    def forward(self, output, target, target_weight):
        """output/target [N,K,H,W] or [N,S,K,H,W]; target_weight [N,K,1] / [N,S,K,1] -> 0-dim f32."""
        L.require_cuda(output, "output")
        target = _as_cuda(target, output.device)
        target_weight = _as_cuda(target_weight, output.device)
        return _HeatmapLossFn.apply(output, target, target_weight, self._mode, self.value, self.reduction)

    def forward_fused(self, output, joints_3d, joints_3d_visible, image_size, sigma=2,
                      unbiased_encoding=True, one_pass=False, expected_grad_out=1.0):
        """Additive fused entry (SURVEY §8b): render the target in-kernel from the joints instead of
        reading a target tensor.  Returns (loss, target_weight [.., 1]).

        one_pass=True (when a gradient is needed): the loss and d loss / d output come from ONE pass over the
        output, and ``loss.backward()`` returns that gradient without reading the output again — provided the
        upstream gradient of the loss is bitwise ``expected_grad_out`` (a float, or a 0-dim CUDA tensor such as
        a gradient scaler's scale times the loss weight).  Any other upstream value is still correct: the
        backward then recomputes the gradient as the default route does.  The gradient buffer (one tensor
        like ``output``) is allocated in the forward rather than in the backward."""
        L.require_cuda(output, "output")
        render = dict(loss_mode=self._mode, image_size=image_size, sigma=sigma, unbiased=unbiased_encoding,
                      pos_value=self.value)
        joints = _as_cuda(joints_3d, output.device)
        vis = _as_cuda(joints_3d_visible, output.device)
        if one_pass and torch.is_grad_enabled() and output.requires_grad:
            loss, weight = _FusedHeatmapLossOnePassFn.apply(output, joints, vis, render, self.reduction,
                                                            expected_grad_out)
        else:
            loss, weight = _FusedHeatmapLossFn.apply(output, joints, vis, render, self.reduction)
        return loss, weight.unsqueeze(-1)


class JointsDistanceLoss(nn.Module):
    """loss/heatmapLoss.py:175-225 (HRNet per-joint 0.5*MSE; the weight multiplies both operands)."""

    def __init__(self, use_target_weight=True, loss_type='mse'):
        super().__init__()
        assert loss_type.lower() in ['mse', 'mae', 'smoothl1']
        if loss_type.lower() != 'mse':
            raise NotImplementedError("only JointsDistanceLoss(loss_type='mse') is on the hot path")
        self.use_target_weight = use_target_weight

    def forward(self, output, target, target_weight=None):
        L.require_cuda(output, "output")
        if self.use_target_weight:
            if target_weight is None:
                raise NameError
            w = _as_cuda(target_weight, output.device)
        else:
            w = torch.ones(output.shape[:2], device=output.device)
        return _HeatmapLossFn.apply(output, _as_cuda(target, output.device), w, L.LOSS_JOINTS_MSE, 0.5, "mean")


class KLDiscretLoss(nn.Module):
    """loss/centernet_simdr_loss.py:6-39 — despite the name: per-joint SmoothL1 mean, times the
    batch-mean of the weight."""

    def forward(self, output_x, output_y, target_x, target_y, target_weight):
        L.require_cuda(output_x, "output_x")
        dev = output_x.device
        return _SimDRLossFn.apply(output_x, _as_cuda(output_y, dev), _as_cuda(target_x, dev),
                                  _as_cuda(target_y, dev), _as_cuda(target_weight, dev))


class SimDRLoss(nn.Module):
    """loss/centernet_simdr_loss.py:42-69.  Same parameters as the reference (two nn.Linear heads, so checkpoints
    load unchanged); the forward is ONE tcgen05 kernel that multiplies the flattened heatmaps with both heads and
    takes KLDiscretLoss in its epilogue (lhn_simdr_heads_loss: the [B*K, k*W_img] predictions never reach HBM).
    ``fused=False`` keeps the reference's structure (cuBLAS heads, then lhn_simdr_smoothl1); shapes outside the
    fused kernel's envelope (H*W not a multiple of 64, non-f32 heatmaps) take that route too."""

    def __init__(self, cfg=None):
        super().__init__()
        image_size = cfg.DATASET.image_size
        heatmap_size = cfg.DATASET.heatmap_size
        k = cfg.PIPELINE.simdr_split_ratio
        self.simdr_width = int(k * image_size[0])
        self.simdr_height = int(k * image_size[1])
        in_features = int(heatmap_size[0] * heatmap_size[1])
        self.x_shared_decoder = nn.Linear(in_features, self.simdr_width)
        self.y_shared_decoder = nn.Linear(in_features, self.simdr_height)
        self.loss = KLDiscretLoss()
        self.fused = True
        self._split = None                   # (key, (w_hi, w_lo)): bf16 pair of cat([Wx, Wy]), rebuilt when the weights change

    def _weight_split(self):
        wx, wy = self.x_shared_decoder.weight, self.y_shared_decoder.weight
        key = (wx.data_ptr(), wx._version, wy.data_ptr(), wy._version, wx.device)
        if self._split is None or self._split[0] != key:
            self._split = (key, ops.split_bf16(torch.cat([wx.detach(), wy.detach()]).float().contiguous()))
        return self._split[1]

    def _fusable(self, heatmap):
        n = self.simdr_width + self.simdr_height
        return (self.fused and heatmap.is_cuda and heatmap.dtype == torch.float32 and heatmap.dim() == 4 and
                heatmap[0, 0].numel() % 64 == 0 and n % 64 == 0 and self.simdr_width % 4 == 0 and self.simdr_height % 4 == 0
                and self.x_shared_decoder.weight.dtype == torch.float32)

    def forward(self, heatmap, simdr_x, simdr_y, target_weight):
        if self._fusable(heatmap):
            dev = heatmap.device
            return _SimDRHeadsLossFn.apply(heatmap, self.x_shared_decoder.weight, self.x_shared_decoder.bias,
                                           self.y_shared_decoder.weight, self.y_shared_decoder.bias,
                                           _as_cuda(simdr_x, dev), _as_cuda(simdr_y, dev), _as_cuda(target_weight, dev),
                                           self._weight_split())
        pred_x = self.x_shared_decoder(heatmap.flatten(start_dim=2))
        pred_y = self.y_shared_decoder(heatmap.flatten(start_dim=2))
        return self.loss(pred_x, pred_y, simdr_x, simdr_y, target_weight)


class TopdownHeatmapLoss(nn.Module):
    """loss/loss.py:69-114.  criterion(output, meta) -> (loss, {name: float}).

    Fused entry (additive): when ``meta`` has no 'target' but has 'joints_3d' / 'joints_3d_visible',
    the target is rendered in-kernel (cfg.PIPELINE sigma / unbiased_encoding, cfg.DATASET.image_size)."""

    def __init__(self, cfg):
        super().__init__()
        loss_type = cfg.LOSS.get('dl_type', 'L2')
        balance = cfg.MODEL.name != 'atthandnet'
        self.heatmap_loss = DistanceLoss(loss_type=loss_type, reduction='mean', balance=balance)
        if cfg.PIPELINE.simdr_split_ratio > 0:
            self.simdr_loss = SimDRLoss(cfg)
        else:
            self.simdr_loss = None
        self.loss_weight = cfg.LOSS.loss_weight
        self.auto_weight = cfg.LOSS.auto_weight
        if self.auto_weight:
            params = torch.ones(len(self.loss_weight), requires_grad=True)
            self.p = nn.Parameter(params, requires_grad=True)
        self._image_size = cfg.DATASET.get('image_size', None)
        self._sigma = cfg.PIPELINE.get('sigma', 2)
        self._unbiased = cfg.PIPELINE.get('unbiased_encoding', True)
        # fused entry: loss and gradient in one pass over the output (DistanceLoss.forward_fused(one_pass=True))
        self.one_pass_grad = bool(cfg.LOSS.get('one_pass_grad', False))

    def forward(self, output, meta):
        loss_dict = {}
        device = output.device
        if 'target' in meta:
            target = meta['target'].to(device)
            target_weight = meta['target_weight'].to(device)
            hl = self.heatmap_loss(output, target, target_weight)
        else:
            # the in-kernel render multiplies no per-joint weights into target_weight (generateTarget.py:156-157);
            # every hand dataset forces them off (freihand_dataset.py:62) — refuse rather than silently ignore
            ann = meta.get('ann_info', {}) if hasattr(meta, 'get') else {}
            if meta.get('use_different_joint_weights', False) or (hasattr(ann, 'get') and ann.get('use_different_joint_weights', False)):
                raise NotImplementedError("use_different_joint_weights: render the targets with TopDownGenerateTarget "
                                          "and pass meta['target'] / meta['target_weight'] instead of the fused entry")
            # autograd delivers loss_weight[0] (as f32) to the heatmap term of `loss` below
            hl, target_weight = self.heatmap_loss.forward_fused(
                output, meta['joints_3d'], meta['joints_3d_visible'], self._image_size, self._sigma,
                self._unbiased, one_pass=self.one_pass_grad, expected_grad_out=float(self.loss_weight[0]))
        loss_dict['heatmap'] = self.loss_weight[0] * hl
        if self.simdr_loss is not None:
            simdr_x = meta['simdr_x'].to(device)
            simdr_y = meta['simdr_y'].to(device)
            loss_dict['simdr'] = self.loss_weight[1] * self.simdr_loss(output, simdr_x, simdr_y, target_weight)
        loss = 0
        for k, v in loss_dict.items():
            loss += v
            loss_dict[k] = v.item()          # .item() syncs: the reference contract
        return loss, loss_dict


class SRHandNetLoss(nn.Module):
    """loss/loss.py:7-66, heatmap-only branch (_forward_only_heatmap): sum_i loss_weight[i] *
    DistanceLoss(outputs[i], targets[i], w[i]) over the 4 scales.  The region-map branch
    (pred_bbox with 24 channels) is out of scope (SURVEY §2 row 3/4).

    Fused entry (additive): when ``meta`` has no 'target' but has 'joints_3d' / 'joints_3d_visible', every scale's
    target is rendered in-kernel — one launch forward, one backward — with SRHandNetGenerateTarget's settings:
    cfg.DATASET.image_size, cfg.PIPELINE.sigma (one for every scale, or a list of one per scale; default
    [2, 2, 2, 2]), cfg.PIPELINE.unbiased_encoding (default False) or UDP when cfg.PIPELINE.encoding == 'UDP'.  The
    plane sizes are those of the outputs.  cfg.LOSS.one_pass_grad = True (default False) computes the loss and the
    gradients in one pass over the outputs when a gradient is needed (SRHandNetLoss.forward_fused(one_pass=True))."""

    def __init__(self, cfg):
        super().__init__()
        out_c = cfg.MODEL.get('output_channel', 24)
        pred_bbox = cfg.MODEL.get('pred_bbox', False)
        self.mse_loss = DistanceLoss(loss_type='L2', reduction='mean')
        if pred_bbox and out_c == 24:
            raise NotImplementedError("SRHandNetLoss region-map branch is out of the hot-path scope")
        self.smoothl1_loss = None
        self.num_out = 4
        self.loss_weight = cfg.LOSS.loss_weight
        assert len(self.loss_weight) == self.num_out
        dataset = cfg.get('DATASET', None) or {}
        pipeline = cfg.get('PIPELINE', None) or {}
        self._image_size = dataset.get('image_size', None)
        self._heatmap_size = dataset.get('heatmap_size', None)
        self._sigma = pipeline.get('sigma', [2, 2, 2, 2])
        self._unbiased = 'udp' if pipeline.get('encoding', 'MSRA') == 'UDP' else pipeline.get('unbiased_encoding', False)
        # fused entry: loss and gradients in one pass over the outputs (forward_fused(one_pass=True))
        self.one_pass_grad = bool(cfg.LOSS.get('one_pass_grad', False))

    def forward(self, outputs, meta):
        if 'target' not in meta and 'joints_3d' in meta and 'joints_3d_visible' in meta:
            # the in-kernel render multiplies no per-joint weights into target_weight (generateTarget.py:156-157);
            # every hand dataset forces them off (freihand_dataset.py:62) — refuse rather than silently ignore
            ann = meta.get('ann_info', {}) if hasattr(meta, 'get') else {}
            if meta.get('use_different_joint_weights', False) or (hasattr(ann, 'get') and ann.get('use_different_joint_weights', False)):
                raise NotImplementedError("use_different_joint_weights: render the targets with SRHandNetGenerateTarget "
                                          "and pass meta['target'] / meta['target_weight'] instead of the fused entry")
            hs = self._heatmap_size
            if isinstance(hs, (list, tuple)) and len(hs) and isinstance(hs[0], (list, tuple)):
                got = [[int(outputs[i].shape[-1]), int(outputs[i].shape[-2])] for i in range(self.num_out)]
                if [[int(x) for x in h] for h in hs] != got:
                    raise ValueError(f"cfg.DATASET.heatmap_size {hs} does not match the outputs' [W, H] {got}")
            if self._image_size is None:
                raise ValueError("the fused SRHandNetLoss entry needs cfg.DATASET.image_size")
            # the loss weights are applied inside the kernel: autograd delivers 1 to this loss
            return self.forward_fused(outputs, meta['joints_3d'], meta['joints_3d_visible'], self._image_size,
                                      self._sigma, self._unbiased, one_pass=self.one_pass_grad)
        target = meta['target']
        target_weight = meta['target_weight']
        return self._forward_only_heatmap(outputs, target, target_weight)

    def forward_fused(self, outputs, joints_3d, joints_3d_visible, image_size, sigmas=(2, 2, 2, 2),
                      unbiased_encoding=False, one_pass=False, expected_grad_out=1.0):
        """The loss of ``forward`` with every scale's target rendered in-kernel from the joints (image_size [w, h];
        sigmas: one for every scale or one per scale; unbiased_encoding False / True / 'udp').  Returns
        (loss, dict(kpt_loss=float)).

        one_pass=True (when grad is enabled and an output requires a gradient): the loss and d loss / d outputs come
        from ONE pass over the outputs, and ``loss.backward()`` returns those gradients without reading the outputs
        again — provided the upstream gradient of the loss is bitwise ``expected_grad_out`` (a float, or a 0-dim CUDA
        tensor such as a gradient scaler's scale).  Any other upstream value is still correct: the backward then
        recomputes the gradients as the default route does.  The gradient buffers are allocated in the forward rather
        than in the backward."""
        outs = [outputs[i] for i in range(self.num_out)]
        for o in outs:
            L.require_cuda(o, "output")
        device = outs[-1].device
        render = dict(loss_mode=self.mse_loss._mode, image_size=tuple(image_size),
                      sigma=list(sigmas) if isinstance(sigmas, (list, tuple)) else sigmas,
                      unbiased=unbiased_encoding, pos_value=self.mse_loss.value)
        joints = _as_cuda(joints_3d, device)
        vis = _as_cuda(joints_3d_visible, device)
        lw = [float(x) for x in self.loss_weight]
        if one_pass and torch.is_grad_enabled() and any(o.requires_grad for o in outs):
            loss = _FusedMultiHeatmapLossOnePassFn.apply(render, self.mse_loss.reduction, lw, expected_grad_out,
                                                         joints, vis, *outs)
        else:
            loss = _FusedMultiHeatmapLossFn.apply(render, self.mse_loss.reduction, lw, joints, vis, *outs)
        return loss, dict(kpt_loss=loss.item())

    def _forward_only_heatmap(self, outputs, targets, target_weight):
        device = outputs[-1].device
        ws = [_as_cuda(target_weight[i] if isinstance(target_weight, (list, tuple)) else target_weight, device)
              for i in range(self.num_out)]
        tg = [_as_cuda(targets[i], device) for i in range(self.num_out)]
        outs = [outputs[i] for i in range(self.num_out)]
        for o in outs:
            L.require_cuda(o, "output")
        # the four scales in ONE launch (it used to be 4 x 3)
        loss = _MultiHeatmapLossFn.apply(self.mse_loss._mode, self.mse_loss.value, self.mse_loss.reduction,
                                         [float(x) for x in self.loss_weight], self.num_out, *outs, *tg, *ws)
        return loss, dict(kpt_loss=loss.item())


srhandnetloss = SRHandNetLoss
topdownheatmaploss = TopdownHeatmapLoss


def get_loss(cfg):
    """loss/__init__.py:18-19."""
    return {"srhandnetloss": SRHandNetLoss, "topdownheatmaploss": TopdownHeatmapLoss}[cfg.LOSS.type.lower()](cfg)
