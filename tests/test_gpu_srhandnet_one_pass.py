"""GPU: SRHandNetLoss's multi-scale loss and its gradients in one pass over the outputs (lhn_render_loss_grad_multi:
a count launch and a stream launch) and its conditional backward (lhn_render_loss_backward_multi_cond), against the
two-launch route (lhn_render_loss_multi + lhn_render_loss_backward_multi) and through the criterion with
cfg.LOSS.one_pass_grad."""
import numpy as np
import pytest
import torch

from oracle.ref_loader import _AttrDict
from litehandnet_b200 import _lib as L
from litehandnet_b200 import ops, synth
from litehandnet_b200 import loss as LS

pytestmark = pytest.mark.gpu
DEV = "cuda"
IMG = (256, 256)
LW = [0.3, 0.3, 0.5, 1.0]
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
# the plane-size sets of tests/test_gpu_srhandnet_fused.py: name -> (plane sizes, per-scale sigmas, loss weights);
# W = 14 and 28 take the kernels' unaligned-row paths
SETS = {
    "16-16-32-64": ([16, 16, 32, 64], [2, 2, 3, 4], LW),
    "14-14-28-56": ([14, 14, 28, 56], [2, 2, 3, 4], LW),
    "single-64": ([64], [2], [1.0]),
    "eight": ([16, 16, 32, 64, 14, 28, 56, 8], [2, 2, 3, 4, 2, 3, 4, 1.5], [0.3, 0.3, 0.5, 1.0, 0.2, 0.4, 0.6, 0.8]),
}


def _joints(B, K, seed):
    """The joint edges of tests/test_gpu_srhandnet_fused.py: outside the image at every scale, outside on the right,
    a weight that differs by scale, an invisible joint."""
    j, v = synth.hand_joints(B, K, IMG, seed=seed)
    j, v = j.clone(), v.clone()
    j[0, 0, :2] = torch.tensor([-300.0, -300.0])
    j[0, 1, :2] = torch.tensor([IMG[0] + 240.0, 10.0])
    j[min(1, B - 1), 2, :2] = torch.tensor([-80.0, 100.0])
    v[0, 3] = 0.0
    return j.to(DEV), v.to(DEV)


def _outputs(B, K, sizes, dtype, seed, extra=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    outs = [(torch.rand((B, K + extra, s, s), generator=g) * 0.9).to(DTYPES[dtype]).to(DEV) for s in sizes]
    return [o[:, :K] for o in outs] if extra else outs


def _render(unbiased, mode, sigmas, value=0.5):
    return dict(loss_mode=mode, image_size=IMG, sigma=sigmas, unbiased=unbiased, pos_value=value)


def _bits(t):
    return t.contiguous().view(torch.int32 if t.element_size() == 4 else torch.int16)


def _same(a, b):
    """Bit for bit (NaN included)."""
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(_bits(a), _bits(b))


def _rel(a, b):
    a, b = float(a), float(b)
    if np.isnan(a) and np.isnan(b):
        return 0.0
    return abs(a - b) / max(abs(b), 1e-30)


def _check(outs, j, v, render, lw, reduction, grad_scale=None, needs=None):
    """One pass against the two-launch route: gradients bit-identical, N_pos and numel bit-equal, S_pos and S_neg
    within 1e-5 of S_pos + S_neg, the losses within 1e-5 relative, the weights equal, used_scale as assumed."""
    gs = None if grad_scale is None else torch.tensor([grad_scale], device=DEV)
    loss, sums, per, grads, used, weights = ops.render_loss_grad_multi(outs, j, v, render, lw, reduction, gs, needs)
    loss_r, sums_r, per_r, w_r = ops.render_loss_multi(outs, j, v, render, lw, reduction)
    grads_r = ops.render_loss_backward_multi(outs, j, v, render, sums_r, lw, reduction, gs, needs)
    for i, (g, gr) in enumerate(zip(grads, grads_r)):
        if gr is None:
            assert g is None, i
            continue
        assert g.is_contiguous() and g.shape == outs[i].shape
        assert _same(g, gr), (i, (g.float() - gr.float()).abs().max().item())
    a, b = sums.cpu().numpy(), sums_r.cpu().numpy()
    assert np.array_equal(a[:, 2:], b[:, 2:]), (a, b)
    for i in range(len(outs)):
        tot = abs(b[i, 0]) + abs(b[i, 1])
        if np.isfinite(tot):
            assert abs(a[i, 0] - b[i, 0]) <= 1e-5 * tot and abs(a[i, 1] - b[i, 1]) <= 1e-5 * tot, (i, a[i], b[i])
        assert _rel(per[i].item(), per_r[i].item()) <= 1e-5, (i, per[i].item(), per_r[i].item())
    assert _rel(loss.item(), loss_r.item()) <= 1e-5, (loss.item(), loss_r.item())
    assert all(torch.equal(x, y) for x, y in zip(weights, w_r))
    assert used.item() == (1.0 if grad_scale is None else np.float32(grad_scale))
    return loss, sums, grads


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("unbiased", [0, 1, 2])
@pytest.mark.parametrize("name", list(SETS))
def test_against_two_launch_route(name, unbiased, dtype):
    sizes, sigmas, lw = SETS[name]
    for (B, K), (mode, reduction) in zip([(1, 21), (3, 16), (64, 21)],
                                         [(L.LOSS_DISTANCE_BALANCE, "mean"), (L.LOSS_DISTANCE, "sum"),
                                          (L.LOSS_DISTANCE_BALANCE, "sum")]):
        outs = _outputs(B, K, sizes, dtype, seed=B + K + unbiased)
        j, v = _joints(B, K, seed=B * 7 + unbiased)
        _check(outs, j, v, _render(unbiased, mode, sigmas), lw, reduction)


@pytest.mark.parametrize("mode", [L.LOSS_DISTANCE, L.LOSS_DISTANCE_BALANCE, L.LOSS_JOINTS_MSE])
@pytest.mark.parametrize("value", [0.5, 0.05, 0.0, -0.25, 1.0])
def test_settings(mode, value):
    """The window (0.5, 0.05), the whole plane (0, and a negative value that counts the planes without a Gaussian too)
    and no positives (1.0); both reductions; a non-unit gradient scale."""
    sizes, sigmas, lw = SETS["16-16-32-64"]
    outs = _outputs(5, 21, sizes, "f32", seed=11)
    j, v = _joints(5, 21, seed=12)
    for unbiased in (0, 1):
        render = _render(unbiased, mode, sigmas, value)
        for reduction in ("mean", "sum"):
            for gs in (None, 0.37):
                _, sums, _ = _check(outs, j, v, render, lw, reduction, gs)
                if mode == L.LOSS_DISTANCE_BALANCE and value >= 1.0:
                    assert (sums[:, 2] == 0).all()


@pytest.mark.parametrize("unbiased", [0, 1, 2])
def test_non_finite_joints(unbiased):
    """NaN and +-inf joints: N_pos (NaN is never a positive) and the gradient bits of the two-launch route."""
    sizes, sigmas, lw = SETS["16-16-32-64"]
    B, K = 4, 21
    for dtype in ("f32", "bf16"):
        outs = _outputs(B, K, sizes, dtype, seed=21)
        j, v = _joints(B, K, seed=22)
        for bad in (float("nan"), float("inf"), float("-inf")):
            jb = j.clone()
            jb[2, 5, 0] = bad
            jb[3, 7, 1] = bad
            for value in (0.5, 0.0):
                _check(outs, jb, v, _render(unbiased, L.LOSS_DISTANCE_BALANCE, sigmas, value), lw, "mean")


@pytest.mark.parametrize("dtype", list(DTYPES))
def test_strided_views_and_gradient_subset(dtype):
    """out[:, :K] of a K+3-channel tensor gives the bits of contiguous copies; scales without a wanted gradient are
    still read for the loss."""
    for name in ("16-16-32-64", "14-14-28-56"):
        sizes, sigmas, lw = SETS[name]
        views = _outputs(3, 21, sizes, dtype, seed=31, extra=3)
        assert not views[0].is_contiguous()
        copies = [x.contiguous() for x in views]
        j, v = _joints(3, 21, seed=32)
        render = _render(1, L.LOSS_DISTANCE_BALANCE, sigmas)
        a = ops.render_loss_grad_multi(views, j, v, render, lw, "mean")
        b = ops.render_loss_grad_multi(copies, j, v, render, lw, "mean")
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
        assert all(_same(x, y) for x, y in zip(a[3], b[3]))
        _check(views, j, v, render, lw, "mean")
        needs = [True, False, True, False]
        loss, sums, grads = _check(views, j, v, render, lw, "mean", 0.37, needs)
        assert grads[1] is None and grads[3] is None
        assert torch.equal(sums, a[1]) and torch.equal(loss, a[0])


def test_reproducible_and_workspace_left_zero():
    sizes, sigmas, lw = SETS["16-16-32-64"]
    j, v = _joints(64, 21, seed=62)
    for dtype in DTYPES:
        outs = _outputs(64, 21, sizes, dtype, seed=61)
        for mode, value in ((L.LOSS_DISTANCE_BALANCE, 0.5), (L.LOSS_DISTANCE_BALANCE, 0.0), (L.LOSS_JOINTS_MSE, 0.5)):
            render = _render(1, mode, sigmas, value)
            ws = torch.zeros(int(L.lib().lhn_render_loss_grad_multi_workspace_bytes(4, 64, 21)), dtype=torch.uint8,
                             device=DEV)
            first = ops.render_loss_grad_multi(outs, j, v, render, lw, "mean", workspace=ws)
            torch.cuda.synchronize()
            assert int(ws.count_nonzero()) == 0
            second = ops.render_loss_grad_multi(outs, j, v, render, lw, "mean", workspace=ws)
            torch.cuda.synchronize()
            assert int(ws.count_nonzero()) == 0
            for x, y in zip(first[:3], second[:3]):
                assert _same(x, y)
            assert all(_same(x, y) for x, y in zip(first[3], second[3]))


def test_conditional_backward():
    sizes, sigmas, lw = SETS["16-16-32-64"]
    outs = _outputs(8, 21, sizes, "f32", seed=71)
    j, v = _joints(8, 21, seed=72)
    render = _render(0, L.LOSS_DISTANCE_BALANCE, sigmas)
    loss, sums, per, grads, used, _ = ops.render_loss_grad_multi(outs, j, v, render, lw, "mean", None,
                                                                 needs=[True, True, False, True])
    rec = torch.full((1,), -1, dtype=torch.int32, device=DEV)
    # upstream equal to the value assumed: nothing is written (NaN sentinels survive)
    for g in grads:
        if g is not None:
            g.fill_(float("nan"))
    ops.render_loss_backward_multi_cond(outs, j, v, render, sums, grads, used, lw, "mean",
                                        torch.ones(1, device=DEV), recomputed=rec)
    assert rec.item() == 0
    assert all(torch.isnan(g).all() for g in grads if g is not None)
    ops.render_loss_backward_multi_cond(outs, j, v, render, sums, grads, used, lw, "mean", None, recomputed=rec)
    assert rec.item() == 0
    # any other upstream value: every wanted gradient is rewritten as the two-launch backward writes it
    go = torch.tensor([0.37], device=DEV)
    ops.render_loss_backward_multi_cond(outs, j, v, render, sums, grads, used, lw, "mean", go, recomputed=rec)
    assert rec.item() == 1
    want = ops.render_loss_backward_multi(outs, j, v, render, sums, lw, "mean", go, needs=[True, True, False, True])
    assert grads[2] is None and want[2] is None
    assert all(_same(g, w) for g, w in zip(grads, want) if g is not None)


def _cfg(sizes, sigma, one_pass):
    loss = dict(loss_weight=list(LW))
    if one_pass is not None:
        loss["one_pass_grad"] = one_pass
    return _AttrDict(MODEL=dict(output_channel=21, pred_bbox=False), LOSS=loss,
                     DATASET=dict(image_size=list(IMG), heatmap_size=[[s, s] for s in sizes]),
                     PIPELINE=dict(sigma=list(sigma), unbiased_encoding=False))


class _Net(torch.nn.Module):
    """Four heads over one shared parameter set (the _Net of tests/test_gpu_srhandnet_fused.py)."""

    def __init__(self, sizes, K, seed):
        super().__init__()
        g = torch.Generator(device="cpu").manual_seed(seed)
        self.base = torch.nn.ParameterList([torch.nn.Parameter(torch.rand((1, K, s, s), generator=g) * 0.9)
                                            for s in sizes])
        self.gain = torch.nn.Parameter(torch.ones(1, K, 1, 1))

    def forward(self, B):
        return [(b * self.gain).expand(B, -1, -1, -1).contiguous() for b in self.base]


@pytest.mark.parametrize("name", ["16-16-32-64", "14-14-28-56"])
def test_criterion_one_sgd_step(name):
    sizes, sigmas, _ = SETS[name]
    B, K = 6, 21
    j, v = _joints(B, K, seed=81)
    meta = dict(joints_3d=j, joints_3d_visible=v)
    nets = [_Net(sizes, K, seed=82).to(DEV) for _ in range(2)]
    crits = [LS.SRHandNetLoss(_cfg(sizes, sigmas, True)), LS.SRHandNetLoss(_cfg(sizes, sigmas, None))]
    assert crits[0].one_pass_grad and not crits[1].one_pass_grad
    losses = []
    for net, crit in zip(nets, crits):
        opt = torch.optim.SGD(net.parameters(), lr=10.0)
        opt.zero_grad()
        loss, ld = crit(net(B), meta)
        assert ld["kpt_loss"] == loss.item()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert _rel(losses[0], losses[1]) <= 1e-5
    for a, b in zip(nets[0].parameters(), nets[1].parameters()):
        assert torch.equal(a, b), (a - b).abs().max().item()


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    return r, [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and
               "kernel" in e.name.lower()]


def test_criterion_launches():
    sizes, sigmas, lw = SETS["16-16-32-64"]
    outs = [o.requires_grad_(True) for o in _outputs(64, 21, sizes, "f32", seed=91)]
    j, v = _joints(64, 21, seed=92)
    crit = LS.SRHandNetLoss(_cfg(sizes, sigmas, True))
    meta = dict(joints_3d=j, joints_3d_visible=v)
    one = torch.ones((), device=DEV)
    crit(outs, meta)[0].backward(one)                                     # warm-up
    for o in outs:
        o.grad = None
    torch.cuda.synchronize()
    # no gradient wanted: the forward kernel alone
    with torch.no_grad():
        _, fwd = _kernels(lambda: crit(outs, meta))
    assert len(fwd) == 1 and "render_loss_multi_kernel" in fwd[0], fwd
    # with a gradient: the count and the stream kernel forward, one conditional kernel backward
    (loss, _), fwd = _kernels(lambda: crit(outs, meta))
    assert len(fwd) == 2 and sum("render_count_multi_kernel" in n for n in fwd) == 1 and \
        sum("render_loss_grad_multi_kernel" in n for n in fwd) == 1, fwd
    _, bwd = _kernels(lambda: loss.backward(one))
    assert len(bwd) == 1 and "render_loss_backward_multi_kernel" in bwd[0] and "true" in bwd[0], bwd
    assert all(o.grad is not None for o in outs)
    # the unbalanced loss needs no N_pos: the stream kernel alone
    render = _render(0, L.LOSS_DISTANCE, sigmas)
    for o in outs:
        o.grad = None
    (loss, fwd) = _kernels(lambda: LS._FusedMultiHeatmapLossOnePassFn.apply(render, "mean", lw, 1.0, j, v, *outs))
    assert len(fwd) == 1 and "render_loss_grad_multi_kernel" in fwd[0], fwd
    probe = torch.full((1,), -1, dtype=torch.int32, device=DEV)
    LS._ONE_PASS_PROBE["recomputed"] = probe
    try:
        loss.backward(one)
    finally:
        LS._ONE_PASS_PROBE.clear()
    assert probe.item() == 0
    want = ops.render_loss_backward_multi([o.detach() for o in outs], j, v, render,
                                          ops.render_loss_multi([o.detach() for o in outs], j, v, render, lw)[1], lw)
    assert all(_same(o.grad, w) for o, w in zip(outs, want))


def test_full_size():
    sizes, sigmas, lw = SETS["16-16-32-64"]
    outs = _outputs(1024, 21, sizes, "f32", seed=3)
    j, v = _joints(1024, 21, seed=4)
    _check(outs, j, v, _render(1, L.LOSS_DISTANCE_BALANCE, sigmas), lw, "mean")
