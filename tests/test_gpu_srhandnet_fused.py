"""GPU: SRHandNetLoss's multi-scale loss with every scale's target rendered in-kernel (lhn_render_loss_multi, one
launch) and its gradient (lhn_render_loss_backward_multi, one launch), against the f64 oracle, the explicit-target
route (lhn_render_targets per scale + lhn_loss_mse_multi), the per-scale backward (lhn_render_loss_backward) and the
drop-in criterion fed with rendered targets."""
import numpy as np
import pytest
import torch

from oracle import np_oracle as O
from oracle.ref_loader import _AttrDict
from litehandnet_b200 import _lib as L
from litehandnet_b200 import ops, synth
from litehandnet_b200 import loss as LS
from litehandnet_b200.render import render_srhandnet_targets

pytestmark = pytest.mark.gpu
DEV = "cuda"
IMG = (256, 256)
LW = [0.3, 0.3, 0.5, 1.0]
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
# name -> (plane sizes, per-scale sigmas, loss weights); W = 14 and 28 take the kernel's unaligned-row path
SETS = {
    "16-16-32-64": ([16, 16, 32, 64], [2, 2, 3, 4], LW),
    "14-14-28-56": ([14, 14, 28, 56], [2, 2, 3, 4], LW),
    "single-64": ([64], [2], [1.0]),
    "eight": ([16, 16, 32, 64, 14, 28, 56, 8], [2, 2, 3, 4, 2, 3, 4, 1.5], [0.3, 0.3, 0.5, 1.0, 0.2, 0.4, 0.6, 0.8]),
}


def _joints(B, K, seed):
    j, v = synth.hand_joints(B, K, IMG, seed=seed)
    j, v = j.clone(), v.clone()
    j[0, 0, :2] = torch.tensor([-300.0, -300.0])               # outside the image at every scale
    j[0, 1, :2] = torch.tensor([IMG[0] + 240.0, 10.0])         # outside on the right
    # 80 px outside: weight 0 on a 64 x 64 plane (stride 4, sigma 4), 1 on 16 x 16 (stride 16, sigma 2) — the
    # weight differs by scale
    j[min(1, B - 1), 2, :2] = torch.tensor([-80.0, 100.0])
    v[0, 3] = 0.0                                              # invisible
    return j.to(DEV), v.to(DEV)


def _outputs(B, K, sizes, dtype, seed, extra=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    outs = [(torch.rand((B, K + extra, s, s), generator=g) * 0.9).to(DTYPES[dtype]).to(DEV) for s in sizes]
    return [o[:, :K] for o in outs] if extra else outs


def _render(unbiased, balance, sigmas, value=0.5):
    return dict(loss_mode=L.LOSS_DISTANCE_BALANCE if balance else L.LOSS_DISTANCE, image_size=IMG, sigma=sigmas,
                unbiased=unbiased, pos_value=value)


def _oracle(outs, j, v, sigmas, unbiased, balance, reduction, lw):
    """Per scale O.render_targets + O.distance_loss_l2 (outputs upcast to f64, targets f32) -> (total, per-scale
    losses, per-scale weights)."""
    j3 = j.cpu().numpy()
    v3 = np.repeat(v.cpu().numpy()[..., :1], 3, -1)
    per, ws = [], []
    for o, s in zip(outs, sigmas):
        H, W = o.shape[-2:]
        with np.errstate(all="ignore"):
            t, w = O.render_targets(j3, v3, IMG, (W, H), s, unbiased=unbiased)
            per.append(float(O.distance_loss_l2(o.float().cpu().numpy(), t, w, balance, 0.5, reduction)))
        ws.append(np.asarray(w, np.float32).reshape(w.shape[0], w.shape[1]))
    return sum(float(a) * b for a, b in zip(lw, per)), per, ws


def _bits(t):
    return t.contiguous().view(torch.int32 if t.element_size() == 4 else torch.int16)


def _same(a, b):
    """Bit for bit (NaN included)."""
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(_bits(a), _bits(b))


def _rel(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-30)


def _check_backward(outs, j, v, render, sums, lw, reduction):
    """The one-launch backward is bitwise one lhn_render_loss_backward per scale on that scale's sums row."""
    for go in (1.0, 0.37):
        gt = torch.tensor([go], device=DEV)
        grads = ops.render_loss_backward_multi(outs, j, v, render, sums, lw, reduction, gt)
        for i, (o, g) in enumerate(zip(outs, grads)):
            r1 = dict(render, sigma=render["sigma"][i])
            want = ops.render_loss_backward(o, j, v, r1, sums[i].contiguous(), reduction, lw[i], gt)
            assert g.shape == o.shape and g.dtype == o.dtype and g.is_contiguous()
            assert _same(g, want), (i, go, (g.float() - want.float()).abs().max().item())


def _check_explicit(outs, j, v, render, lw, reduction, loss, sums, weights):
    """f32: the explicit-target route renders each scale's target (lhn_render_targets) and reads it back."""
    tg, tw = [], []
    for o, s in zip(outs, render["sigma"]):
        H, W = o.shape[-2:]
        t, w = ops.render_targets(j, v, IMG, (W, H), s, render["unbiased"])
        tg.append(t); tw.append(w)
    l2, s2, _ = ops.loss_mse_multi(outs, tg, tw, render["loss_mode"], render["pos_value"], reduction, lw)
    a, b = sums.cpu().numpy(), s2.cpu().numpy()
    assert np.array_equal(a[:, 2:], b[:, 2:]), (a, b)                   # N_pos and numel bit-exact
    for i in range(len(outs)):
        total = abs(b[i, 0]) + abs(b[i, 1])
        if np.isfinite(total) and total > 0:
            assert abs(a[i, 0] - b[i, 0]) <= 1e-6 * total and abs(a[i, 1] - b[i, 1]) <= 1e-6 * total, (i, a[i], b[i])
    if np.isfinite(l2.item()):
        assert _rel(loss.item(), l2.item()) <= 1e-6, (loss.item(), l2.item())
    for w, t in zip(weights, tw):
        assert torch.equal(w, t.reshape(w.shape))


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("unbiased", [0, 1, 2])
@pytest.mark.parametrize("name", list(SETS))
def test_against_oracle(name, unbiased, dtype):
    sizes, sigmas, lw = SETS[name]
    for (B, K), (balance, reduction) in zip([(1, 21), (3, 16), (64, 21)], [(True, "mean"), (False, "sum"), (True, "sum")]):
        if unbiased == 2 and min(sizes) < 2:
            continue
        outs = _outputs(B, K, sizes, dtype, seed=B + K + unbiased)
        j, v = _joints(B, K, seed=B * 7 + unbiased)
        render = _render(unbiased, balance, sigmas)
        loss, sums, per, weights = ops.render_loss_multi(outs, j, v, render, lw, reduction)
        want, want_per, want_w = _oracle(outs, j, v, sigmas, unbiased, balance, reduction, lw)
        assert _rel(loss.item(), want) <= 1e-5, (name, B, K, loss.item(), want)
        for i in range(len(sizes)):
            assert _rel(per[i].item(), want_per[i]) <= 1e-5, (i, per[i].item(), want_per[i])
            assert np.array_equal(weights[i].cpu().numpy(), want_w[i]), i
        _check_backward(outs, j, v, render, sums, lw, reduction)
        if dtype == "f32":
            _check_explicit(outs, j, v, render, lw, reduction, loss, sums, weights)


@pytest.mark.parametrize("mode", [L.LOSS_DISTANCE, L.LOSS_DISTANCE_BALANCE, L.LOSS_JOINTS_MSE])
@pytest.mark.parametrize("value", [0.5, 0.05])
def test_loss_modes_against_explicit_route(mode, value):
    sizes, sigmas, lw = SETS["16-16-32-64"]
    outs = _outputs(5, 21, sizes, "f32", seed=11)
    j, v = _joints(5, 21, seed=12)
    render = dict(_render(1, True, sigmas, value), loss_mode=mode)
    for reduction in ("mean", "sum"):
        loss, sums, _, weights = ops.render_loss_multi(outs, j, v, render, lw, reduction)
        _check_explicit(outs, j, v, render, lw, reduction, loss, sums, weights)
        _check_backward(outs, j, v, render, sums, lw, reduction)


def test_large_batch():
    """B = 1024: the explicit-target route and the f64 loss of the same targets (lhn_render_targets draws the
    oracle's targets pixel for pixel, tests/test_gpu_render_conformance.py), computed on the device."""
    sizes, sigmas, lw = SETS["16-16-32-64"]
    outs = _outputs(1024, 21, sizes, "f32", seed=3)
    j, v = _joints(1024, 21, seed=4)
    render = _render(1, True, sigmas)
    loss, sums, per, weights = ops.render_loss_multi(outs, j, v, render, lw, "mean")
    want = 0.0
    for i, (o, s) in enumerate(zip(outs, sigmas)):
        t, w = ops.render_targets(j, v, IMG, (o.shape[-1], o.shape[-2]), s, 1)
        ell = (o.double() - t.double()) ** 2 * w.double()[..., None]
        pos = t > 0.5
        n_pos, numel = int(pos.sum()), ell.numel()
        li = (ell[pos].sum() * (0.1 / (n_pos + 1)) + ell[~pos].sum() / (numel - n_pos + 1)).item()
        assert _rel(per[i].item(), li) <= 1e-5
        want += lw[i] * li
    assert _rel(loss.item(), want) <= 1e-5
    _check_explicit(outs, j, v, render, lw, "mean", loss, sums, weights)
    _check_backward(outs, j, v, render, sums, lw, "mean")


@pytest.mark.parametrize("unbiased", [0, 1, 2])
def test_geometry_edges(unbiased):
    """Joints outside the image, invisible, weight differing by scale, NaN and +-inf.  A NaN or infinite joint is
    compared with the explicit-target route (the reference's int() raises on it in modes 0 and 2); in mode 1 with the
    oracle as well.  A NaN in one scale's output makes that scale's loss NaN and leaves the others' bits alone."""
    sizes, sigmas, lw = SETS["16-16-32-64"]
    B, K = 4, 21
    outs = _outputs(B, K, sizes, "f32", seed=21)
    j, v = _joints(B, K, seed=22)
    render = _render(unbiased, True, sigmas)
    base, base_sums, base_per, base_w = ops.render_loss_multi(outs, j, v, render, LW, "mean")
    w = [x.cpu().numpy() for x in base_w]
    assert w[0][1, 2] == 1.0 and w[3][1, 2] == 0.0                  # the 80 px joint: in at 16 x 16, out at 64 x 64
    assert all(x[0, 0] == 0.0 and x[0, 1] == 0.0 and x[0, 3] == 0.0 for x in w)
    if unbiased == 1:
        want, want_per, _ = _oracle(outs, j, v, sigmas, unbiased, True, "mean", LW)
        assert _rel(base.item(), want) <= 1e-5
    for bad in (float("nan"), float("inf"), float("-inf")):
        jb = j.clone()
        jb[2, 5, 0] = bad
        jb[3, 7, 1] = bad
        loss, sums, per, weights = ops.render_loss_multi(outs, jb, v, render, LW, "mean")
        _check_explicit(outs, jb, v, render, LW, "mean", loss, sums, weights)
        _check_backward(outs, jb, v, render, sums, LW, "mean")
        if unbiased == 1:
            want, want_per, want_w = _oracle(outs, jb, v, sigmas, 1, True, "mean", LW)
            got = per.cpu().numpy()
            assert np.array_equal(np.isnan(got), np.isnan(np.asarray(want_per))), (bad, got, want_per)
            for i in range(len(sizes)):
                assert np.array_equal(weights[i].cpu().numpy(), want_w[i])
                if np.isfinite(want_per[i]):
                    assert _rel(got[i], want_per[i]) <= 1e-5
    for hit in range(len(sizes)):
        o2 = [o.clone() for o in outs]
        o2[hit][1, 4, 3, 3] = float("nan")
        loss, sums, per, _ = ops.render_loss_multi(o2, j, v, render, LW, "mean")
        p, bp = per.cpu().numpy(), base_per.cpu().numpy()
        assert np.isnan(p[hit]) and np.isnan(loss.item())
        others = [i for i in range(len(sizes)) if i != hit]
        assert np.array_equal(p[others], bp[others])
        assert torch.equal(sums[others], base_sums[others])


@pytest.mark.parametrize("dtype", list(DTYPES))
def test_strided_views(dtype):
    """out[:, :K] of a K+3-channel tensor (the layout SRHandNet's outputs have with region maps) needs no copy and
    gives the bits of contiguous copies, forward and backward."""
    for name in ("16-16-32-64", "14-14-28-56"):
        sizes, sigmas, lw = SETS[name]
        views = _outputs(3, 21, sizes, dtype, seed=31, extra=3)
        assert not views[0].is_contiguous()
        copies = [x.contiguous() for x in views]
        j, v = _joints(3, 21, seed=32)
        render = _render(1, True, sigmas)
        a = ops.render_loss_multi(views, j, v, render, lw, "mean")
        b = ops.render_loss_multi(copies, j, v, render, lw, "mean")
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
        ga = ops.render_loss_backward_multi(views, j, v, render, a[1], lw, "mean")
        gb = ops.render_loss_backward_multi(copies, j, v, render, b[1], lw, "mean")
        assert all(torch.equal(x, y) for x, y in zip(ga, gb))


def _torch_oracle_loss(outs64, j, v, sigmas, unbiased, balance, reduction, lw):
    """The oracle's loss restated in torch float64 so autograd can differentiate it (targets from O.render_targets)."""
    j3 = j.cpu().numpy()
    v3 = np.repeat(v.cpu().numpy()[..., :1], 3, -1)
    total = 0.0
    for o, s, wgt in zip(outs64, sigmas, lw):
        H, W = o.shape[-2:]
        t, w = O.render_targets(j3, v3, IMG, (W, H), s, unbiased=unbiased)
        t = torch.from_numpy(np.asarray(t, np.float32)).to(DEV)
        w = torch.from_numpy(np.asarray(w, np.float64)).to(DEV).reshape(o.shape[0], o.shape[1], 1, 1)
        ell = (o - t.double()) ** 2 * w
        numel = ell.numel()
        if balance:
            pos = t > 0.5
            n_pos = int(pos.sum())
            li = ell[pos].sum() * (0.1 / (n_pos + 1)) + ell[~pos].sum() / (numel - n_pos + 1)
        else:
            li = ell.sum() / numel
        total = total + wgt * (li * numel if reduction == "sum" else li)
    return total


@pytest.mark.parametrize("unbiased", [0, 1, 2])
@pytest.mark.parametrize("balance,reduction", [(True, "mean"), (False, "sum")])
def test_backward_against_f64_autograd(unbiased, balance, reduction):
    for name in ("16-16-32-64", "14-14-28-56"):
        sizes, sigmas, lw = SETS[name]
        outs = _outputs(3, 21, sizes, "f32", seed=41)
        j, v = _joints(3, 21, seed=42)
        render = _render(unbiased, balance, sigmas)
        _, sums, _, _ = ops.render_loss_multi(outs, j, v, render, lw, reduction)
        grads = ops.render_loss_backward_multi(outs, j, v, render, sums, lw, reduction)
        o64 = [o.double().requires_grad_(True) for o in outs]
        _torch_oracle_loss(o64, j, v, sigmas, unbiased, balance, reduction, lw).backward()
        for g, o in zip(grads, o64):
            ref = o.grad
            scale = ref.abs().max().item()
            assert (g.double() - ref).abs().max().item() <= 1e-5 * scale


def test_autograd_function_grads_only_where_required():
    sizes, sigmas, lw = SETS["16-16-32-64"]
    outs = _outputs(2, 21, sizes, "f32", seed=51)
    outs = [o.clone().requires_grad_(i != 1) for i, o in enumerate(outs)]
    j, v = _joints(2, 21, seed=52)
    render = _render(0, True, sigmas)
    loss = LS._FusedMultiHeatmapLossFn.apply(render, "mean", lw, j, v, *outs)
    loss.backward()
    assert outs[1].grad is None
    _, sums, _, _ = ops.render_loss_multi([o.detach() for o in outs], j, v, render, lw, "mean")
    for i in (0, 2, 3):
        want = ops.render_loss_backward(outs[i].detach(), j, v, dict(render, sigma=sigmas[i]), sums[i].contiguous(),
                                        "mean", lw[i], torch.ones(1, device=DEV))
        assert torch.equal(outs[i].grad, want)
    got = ops.render_loss_backward_multi([o.detach() for o in outs], j, v, render, sums, lw, "mean",
                                         needs=[True, False, True, False])
    assert got[1] is None and got[3] is None and torch.equal(got[0], outs[0].grad)


def test_determinism_and_workspace_reuse():
    sizes, sigmas, lw = SETS["16-16-32-64"]
    j, v = _joints(64, 21, seed=62)
    render = _render(1, True, sigmas)
    for dtype in DTYPES:
        outs = _outputs(64, 21, sizes, dtype, seed=61)
        a = ops.render_loss_multi(outs, j, v, render, lw, "mean")
        b = ops.render_loss_multi(outs, j, v, render, lw, "mean")      # on the workspace the first call left
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
        # the explicit-target loss shares the workspace on this stream and still agrees with itself
        tg = [ops.render_targets(j, v, IMG, (s, s), sg, 1) for s, sg in zip(sizes, sigmas)]
        c = ops.loss_mse_multi(outs, [t for t, _ in tg], [w for _, w in tg], L.LOSS_DISTANCE_BALANCE, 0.5, "mean", lw)
        d = ops.loss_mse_multi(outs, [t for t, _ in tg], [w for _, w in tg], L.LOSS_DISTANCE_BALANCE, 0.5, "mean", lw)
        assert torch.equal(c[1], d[1])
        e = ops.render_loss_multi(outs, j, v, render, lw, "mean")
        assert torch.equal(a[1], e[1])


def _cfg(sizes, sigma=(2, 2, 2, 2), unbiased=False, encoding=None, heatmap_size=True):
    pipe = dict(sigma=list(sigma), unbiased_encoding=unbiased)
    if encoding:
        pipe["encoding"] = encoding
    ds = dict(image_size=list(IMG))
    if heatmap_size:
        ds["heatmap_size"] = [[s, s] for s in sizes]
    return _AttrDict(MODEL=dict(output_channel=21, pred_bbox=False), LOSS=dict(loss_weight=list(LW)),
                     DATASET=ds, PIPELINE=pipe)


class _Net(torch.nn.Module):
    """Four heads over one shared parameter set: the gradient of every scale reaches the same parameters."""

    def __init__(self, sizes, K, seed):
        super().__init__()
        g = torch.Generator(device="cpu").manual_seed(seed)
        self.base = torch.nn.ParameterList([torch.nn.Parameter(torch.rand((1, K, s, s), generator=g) * 0.9)
                                            for s in sizes])
        self.gain = torch.nn.Parameter(torch.ones(1, K, 1, 1))

    def forward(self, B):
        return [(b * self.gain).expand(B, -1, -1, -1).contiguous() for b in self.base]


@pytest.mark.parametrize("name", ["16-16-32-64", "14-14-28-56"])
@pytest.mark.parametrize("unbiased", [False, True, "udp"])
def test_srhandnet_loss_end_to_end(name, unbiased):
    sizes, sigmas, _ = SETS[name]
    B, K = 6, 21
    enc = "UDP" if unbiased == "udp" else None
    cfg = _cfg(sizes, sigmas, unbiased if unbiased != "udp" else False, enc)
    j, v = _joints(B, K, seed=71)
    bbox = np.tile(np.array([[40.0, 40.0, 150.0, 150.0]], np.float32), (B, 1))
    tg, tw = render_srhandnet_targets(j, v, bbox, IMG, [[s, s] for s in sizes], sigmas, pred_bbox=False,
                                      unbiased_encoding=unbiased)
    nets = [_Net(sizes, K, seed=72).to(DEV) for _ in range(2)]
    crit = LS.SRHandNetLoss(cfg)
    fused, ld_f = crit(nets[0](B), dict(joints_3d=j, joints_3d_visible=v))
    ref, ld_r = crit(nets[1](B), dict(target=tg, target_weight=tw))
    assert set(ld_f) == {"kpt_loss"} and ld_f["kpt_loss"] == fused.item()
    assert _rel(fused.item(), ref.item()) <= 1e-6, (fused.item(), ref.item())
    for net, l in zip(nets, (fused, ref)):
        opt = torch.optim.SGD(net.parameters(), lr=10.0)
        opt.zero_grad()
        l.backward()
        opt.step()
    for a, b in zip(nets[0].parameters(), nets[1].parameters()):
        assert torch.allclose(a, b, rtol=1e-6, atol=0.0), (a - b).abs().max().item()
    # forward_fused is the same loss without a cfg
    again, _ = LS.SRHandNetLoss(_AttrDict(MODEL=dict(output_channel=21), LOSS=dict(loss_weight=list(LW)))).forward_fused(
        nets[0](B), j, v, IMG, sigmas, unbiased)
    loss2, _, _, _ = ops.render_loss_multi(nets[0](B), j, v, _render(unbiased, True, sigmas), LW, "mean")
    assert again.item() == loss2.item()


def test_srhandnet_loss_settings_and_refusals():
    sizes = [16, 16, 32, 64]
    B, K = 3, 21
    outs = _outputs(B, K, sizes, "f32", seed=81)
    j, v = _joints(B, K, seed=82)
    meta = dict(joints_3d=j, joints_3d_visible=v)
    # defaults: SRHandNetGenerateTarget's sigma [2, 2, 2, 2] and integer-centre encoding; a scalar sigma
    cfg = _AttrDict(MODEL=dict(output_channel=21), LOSS=dict(loss_weight=list(LW)), DATASET=dict(image_size=list(IMG)))
    got, _ = LS.SRHandNetLoss(cfg)(outs, meta)
    want = ops.render_loss_multi(outs, j, v, _render(False, True, [2, 2, 2, 2]), LW, "mean")[0]
    assert got.item() == want.item()
    cfg.PIPELINE = _AttrDict(sigma=3, unbiased_encoding=True)
    got, _ = LS.SRHandNetLoss(cfg)(outs, meta)
    assert got.item() == ops.render_loss_multi(outs, j, v, _render(True, True, 3), LW, "mean")[0].item()
    # the heatmap sizes of the cfg are [W, H] and must match the outputs
    with pytest.raises(ValueError):
        LS.SRHandNetLoss(_cfg([16, 16, 32, 32]))(outs, meta)
    rect = [torch.rand((B, K, s, 2 * s), device=DEV) for s in sizes]
    cfg_r = _cfg(sizes)
    cfg_r.DATASET.heatmap_size = [[2 * s, s] for s in sizes]
    LS.SRHandNetLoss(cfg_r)(rect, meta)
    with pytest.raises(ValueError):
        LS.SRHandNetLoss(_cfg(sizes))(rect, meta)
    crit = LS.SRHandNetLoss(_cfg(sizes))
    with pytest.raises(NotImplementedError):
        crit(outs, dict(meta, use_different_joint_weights=True))
    with pytest.raises(NotImplementedError):
        crit(outs, dict(meta, ann_info=dict(use_different_joint_weights=True)))
    with pytest.raises(L.LhnError):                                       # B differs
        crit([outs[0][:2]] + outs[1:], meta)
    with pytest.raises(L.LhnError):                                       # K differs
        crit([outs[0][:, :20]] + outs[1:], meta)
    with pytest.raises(L.LhnError):                                       # joints of another batch
        crit(outs, dict(joints_3d=j[:2], joints_3d_visible=v[:2]))
    with pytest.raises(L.LhnError):                                       # CPU outputs
        crit([o.cpu() for o in outs], meta)
    with pytest.raises(L.LhnError):                                       # mixed dtypes
        crit([outs[0].half()] + outs[1:], meta)
    with pytest.raises(L.LhnError):
        ops.render_loss_multi(outs, j.cpu(), v.cpu(), _render(0, True, 2), LW)
    with pytest.raises(L.LhnError):
        ops.render_loss_multi(outs * 3, j, v, _render(0, True, 2))          # 12 scales
    with pytest.raises(L.LhnError):
        ops.render_loss_multi(outs, j, v, _render(0, True, [2, 2, 2]), LW)  # 3 sigmas for 4 scales


def test_one_launch_each():
    sizes, sigmas, lw = SETS["16-16-32-64"]
    outs = [o.requires_grad_(True) for o in _outputs(64, 21, sizes, "f32", seed=91)]
    j, v = _joints(64, 21, seed=92)
    crit = LS.SRHandNetLoss(_cfg(sizes, sigmas))
    meta = dict(joints_3d=j, joints_3d_visible=v)
    one = torch.ones((), device=DEV)
    crit(outs, meta)[0].backward(one)                                     # warm-up
    for o in outs:
        o.grad = None
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        loss, _ = crit(outs, meta)
        torch.cuda.synchronize()
    fwd = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "kernel" in e.name.lower()]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        loss.backward(one)
        torch.cuda.synchronize()
    bwd = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "kernel" in e.name.lower()]
    assert len(fwd) == 1 and "loss_multi_kernel" in fwd[0], fwd
    assert len(bwd) == 1 and "render_loss_backward_multi_kernel" in bwd[0], bwd
