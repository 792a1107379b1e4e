"""GPU: the fused heatmap loss and its gradient in one pass (lhn_render_loss_grad) and its conditional backward
(lhn_render_loss_backward_cond), against the two-pass route (lhn_fused_render_loss_decode, then
lhn_render_loss_backward) and the NumPy oracle."""
import numpy as np
import pytest
import torch

from oracle import np_oracle as O
from oracle.ref_loader import _AttrDict
from litehandnet_b200 import _lib as L
from litehandnet_b200 import ops, synth
from litehandnet_b200 import loss as LS

pytestmark = pytest.mark.gpu
DEV = "cuda"
IMG = (256, 256)
MAX_REL = {"loss": 0.0, "sums": 0.0, "oracle": 0.0}       # largest relative differences seen (printed at the end)

DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
# name -> (heatmap shape, sigma); "sliced" is out[:, :21] of a 24-channel tensor
SHAPES = {
    "16x21x64": ((16, 21, 64, 64), 2),
    "stacked": ((3, 2, 21, 64, 64), [2, 3]),
    "5x6x56": ((5, 6, 56, 56), 2),
    "128": ((2, 4, 128, 128), 2),
    "28": ((3, 5, 28, 28), 2),
    "14": ((3, 5, 14, 14), 2),
    "sliced": ((4, 24, 64, 64), 2),
}


def _inputs(name, dtype, seed=0):
    shape, sigma = SHAPES[name]
    g = torch.Generator(device="cpu").manual_seed(seed)
    hm = (torch.rand(shape, generator=g) * 0.9).to(DTYPES[dtype]).to(DEV)
    if name == "sliced":
        hm = hm[:, :21]
    B, K = hm.shape[0], hm.shape[-3]
    W, H = hm.shape[-1], hm.shape[-2]
    joints, vis = synth.hand_joints(B, K, IMG, seed=seed + 7)
    joints, vis = joints.clone(), vis.clone()
    joints[0, 0, :2] = torch.tensor([-80.0, -80.0])            # outside the image
    joints[0, 1, :2] = torch.tensor([IMG[0] + 40.0, 10.0])      # outside on the right
    joints[min(1, B - 1), 2, :2] = torch.tensor([-3.0, 100.0])  # just outside: its Gaussian still reaches in
    vis[0, 3] = 0.0                                             # invisible
    return hm, joints.to(DEV), vis.to(DEV), sigma


def _render(mode, sigma, unbiased, value):
    return dict(loss_mode=mode, image_size=IMG, sigma=sigma, unbiased=unbiased, pos_value=value)


def _two_pass(hm, j, v, render, reduction, loss_scale, grad_scale):
    f = ops.fused_render_loss_decode(hm, L.MASK_NEG1, L.REFINE_NONE, L.XFORM_NONE, None, None, render, j, v,
                                     want_idx=False, reduction=reduction, loss_scale=loss_scale)
    go = torch.tensor([1.0 if grad_scale is None else float(grad_scale)], device=DEV)
    g = ops.render_loss_backward(hm, j, v, render, f["sums"], reduction, loss_scale, go)
    return f, g


def _rel(a, b):
    a, b = float(a), float(b)
    return abs(a - b) / max(abs(b), 1e-30)


def _check_case(hm, j, v, render, reduction="mean", loss_scale=1.0, grad_scale=None):
    one = ops.render_loss_grad(hm, j, v, render, reduction, loss_scale, grad_scale)
    f, g2 = _two_pass(hm, j, v, render, reduction, loss_scale, grad_scale)
    torch.cuda.synchronize()
    # 1. the gradient is bit-identical to the two-pass backward on the forward's sums
    assert one["grad"].shape == hm.shape and one["grad"].dtype == hm.dtype
    assert torch.equal(one["grad"], g2), f"grad differs: max {(one['grad'].float() - g2.float()).abs().max().item()}"
    # 2. N_pos, numel and target_weight bit-equal to the fused forward
    s1, s2 = one["sums"].cpu().numpy(), f["sums"].cpu().numpy()
    assert s1[2] == s2[2] and s1[3] == s2[3], (s1, s2)
    assert torch.equal(one["weight"], f["weight"])
    # 3. loss and S_pos / S_neg within 1e-5 relative of the fused forward; relative to S_pos + S_neg, because the
    #    forward derives S_neg as S_all - S_pos (an S_neg of ~0 comes back as rounding residue of that difference)
    total = abs(s2[0]) + abs(s2[1])
    for k in (0, 1):
        if total > 0.0:
            r = abs(s1[k] - s2[k]) / total
            MAX_REL["sums"] = max(MAX_REL["sums"], r)
            assert r <= 1e-5, (k, s1, s2)
    r = _rel(one["loss"].item(), f["loss"].item())
    MAX_REL["loss"] = max(MAX_REL["loss"], r)
    assert r <= 1e-5, (one["loss"].item(), f["loss"].item())
    expect = 1.0 if grad_scale is None else float(grad_scale)
    assert one["used_scale"].item() == np.float32(expect)
    return one, f


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("name", list(SHAPES))
def test_one_pass_matches_two_pass(name, dtype):
    hm, j, v, sigma = _inputs(name, dtype)
    _check_case(hm, j, v, _render(L.LOSS_DISTANCE_BALANCE, sigma, True, 0.5))
    _check_case(hm, j, v, _render(L.LOSS_DISTANCE_BALANCE, sigma, 2, 0.05), "sum", 0.7, 0.25)


@pytest.mark.parametrize("unbiased", [0, 1, 2])
@pytest.mark.parametrize("mode", [L.LOSS_DISTANCE, L.LOSS_DISTANCE_BALANCE, L.LOSS_JOINTS_MSE])
@pytest.mark.parametrize("reduction", ["mean", "sum"])
def test_one_pass_settings(unbiased, mode, reduction):
    hm, j, v, sigma = _inputs("16x21x64", "f32", seed=3)
    for value in (0.5, 0.05, 0.0, 1.0):
        _check_case(hm, j, v, _render(mode, sigma, unbiased, value), reduction, 1.0, torch.tensor(1.5, device=DEV))


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("value", [0.5, 0.05, 0.0, 1.0])
def test_one_pass_values_dtypes(dtype, value):
    for name in ("stacked", "28", "14"):
        hm, j, v, sigma = _inputs(name, dtype, seed=5)
        _check_case(hm, j, v, _render(L.LOSS_DISTANCE_BALANCE, sigma, 1, value))


@pytest.mark.parametrize("balance", [True, False])
@pytest.mark.parametrize("reduction", ["mean", "sum"])
def test_one_pass_against_oracle(balance, reduction):
    hm, j, v, sigma = _inputs("16x21x64", "f32", seed=11)
    mode = L.LOSS_DISTANCE_BALANCE if balance else L.LOSS_DISTANCE
    one = ops.render_loss_grad(hm, j, v, _render(mode, sigma, True, 0.5), reduction)
    tg, tw = O.render_targets(j.cpu().numpy(), v.cpu().numpy(), IMG, (64, 64), sigma, True)
    out = hm.cpu().numpy()
    ref = O.distance_loss_l2(out, tg, tw, balance, 0.5, reduction)
    r = _rel(one["loss"].item(), ref)
    MAX_REL["oracle"] = max(MAX_REL["oracle"], r)
    assert r <= 1e-5, (one["loss"].item(), ref)
    gref = O.distance_loss_l2_grad(out, tg, tw, balance, 0.5, reduction)
    gd = np.abs(one["grad"].cpu().numpy().astype(np.float64) - gref).max()
    MAX_REL["oracle"] = max(MAX_REL["oracle"], gd / np.abs(gref).max())
    assert gd <= 1e-5 * np.abs(gref).max(), gd


def test_one_pass_reproducible_and_workspace_zero():
    hm, j, v, sigma = _inputs("stacked", "bf16")
    render = _render(L.LOSS_DISTANCE_BALANCE, sigma, True, 0.5)
    a = ops.render_loss_grad(hm, j, v, render)
    b = ops.render_loss_grad(hm, j, v, render)
    torch.cuda.synchronize()
    assert torch.equal(a["loss"], b["loss"]) and torch.equal(a["sums"], b["sums"]) and torch.equal(a["grad"], b["grad"])
    B, S, K = hm.shape[:3]
    ws = ops.render_loss_grad_workspace(hm.device, B, K, S)
    assert int(ws.count_nonzero()) == 0


def _dist_loss(balance=True, reduction="mean"):
    return LS.DistanceLoss(reduction=reduction, balance=balance)


def test_autograd_conditional_backward():
    hm, j, v, sigma = _inputs("16x21x64", "f32", seed=2)
    crit = _dist_loss()
    probe = torch.full((1,), -1, dtype=torch.int32, device=DEV)
    LS._ONE_PASS_PROBE["recomputed"] = probe
    try:
        for factor in (None, 0.7):
            x1 = hm.clone().requires_grad_(True)
            x2 = hm.clone().requires_grad_(True)
            l1, w1 = crit.forward_fused(x1, j, v, IMG, sigma, True, one_pass=True)
            l2, w2 = crit.forward_fused(x2, j, v, IMG, sigma, True)
            assert torch.equal(l1, l2) or _rel(l1.item(), l2.item()) <= 1e-5
            assert torch.equal(w1, w2)
            if factor is None:
                l1.backward(); l2.backward()
            else:
                (l1 * factor).backward(); (l2 * factor).backward()
            torch.cuda.synchronize()
            assert probe.item() == (0 if factor is None else 1)
            assert torch.equal(x1.grad, x2.grad)
    finally:
        LS._ONE_PASS_PROBE.clear()


def _cfg(K=21, hm=(64, 64), loss_weight=(1.0, 1.0), one_pass=False):
    return _AttrDict(
        DATASET=dict(image_size=list(IMG), heatmap_size=list(hm), num_joints=K),
        PIPELINE=dict(unbiased_encoding=True, kernel=(11, 11), use_udp=False, simdr_split_ratio=0, sigma=2),
        MODEL=dict(name="litehandnet"),
        LOSS=dict(type="TopdownHeatmapLoss", loss_weight=list(loss_weight), auto_weight=False, one_pass_grad=one_pass))


@pytest.mark.parametrize("loss_weight", [1.0, 0.3])
def test_criterion_expected_upstream_is_loss_weight(loss_weight):
    """TopdownHeatmapLoss passes float32(loss_weight[0]) as the expected upstream value: autograd delivers exactly
    that to the heatmap term, so the backward is the no-op branch."""
    hm, j, v, _ = _inputs("16x21x64", "f32", seed=4)
    crit = LS.get_loss(_cfg(loss_weight=(loss_weight, 1.0), one_pass=True))
    assert crit.one_pass_grad
    probe = torch.full((1,), -1, dtype=torch.int32, device=DEV)
    LS._ONE_PASS_PROBE["recomputed"] = probe
    try:
        x = hm.clone().requires_grad_(True)
        loss, _ = crit(x, dict(joints_3d=j, joints_3d_visible=v))
        loss.backward()
        torch.cuda.synchronize()
        assert probe.item() == 0
    finally:
        LS._ONE_PASS_PROBE.clear()
    ref = LS.get_loss(_cfg(loss_weight=(loss_weight, 1.0)))
    y = hm.clone().requires_grad_(True)
    loss2, _ = ref(y, dict(joints_3d=j, joints_3d_visible=v))
    loss2.backward()
    assert torch.equal(x.grad, y.grad)


def test_training_step_through_one_pass_criterion():
    """train_one_epoch's pattern with one_pass_grad on: parameter gradients agree with the default criterion's,
    and five SGD steps reduce the loss."""
    torch.manual_seed(0)
    N, K, H, W = 4, 21, 64, 64
    crit_ref = LS.get_loss(_cfg(K=K, hm=(W, H)))
    crit = LS.get_loss(_cfg(K=K, hm=(W, H)))
    crit.one_pass_grad = True
    model = torch.nn.Conv2d(3, K, 3, padding=1).to(DEV)
    opt = torch.optim.SGD(model.parameters(), lr=0.5)
    img = torch.randn(N, 3, H, W, device=DEV)
    joints, vis = synth.hand_joints(N, K, IMG, seed=81)
    meta = dict(joints_3d=joints, joints_3d_visible=vis)
    grads = []
    for c in (crit_ref, crit):
        opt.zero_grad()
        loss, d = c(model(img), meta)
        loss.backward()
        grads.append([p.grad.clone() for p in model.parameters()])
        assert isinstance(d["heatmap"], float) and np.isfinite(d["heatmap"])
    for a, b in zip(*grads):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-7)
    opt.zero_grad()
    l0 = float(crit(model(img), meta)[0].detach())
    for _ in range(5):
        opt.zero_grad()
        loss, _ = crit(model(img), meta)
        loss.backward()
        opt.step()
    assert float(loss.detach()) < l0


def test_no_grad_uses_loss_only_path(monkeypatch):
    hm, j, v, sigma = _inputs("16x21x64", "f32", seed=6)
    crit = _dist_loss()
    ref, wref = crit.forward_fused(hm, j, v, IMG, sigma, True)

    def _fail(*a, **k):
        raise AssertionError("the one-pass kernel (and its gradient buffer) must not run without a gradient")
    monkeypatch.setattr(ops, "render_loss_grad", _fail)
    x = hm.clone().requires_grad_(True)
    with torch.no_grad():
        loss, w = crit.forward_fused(x, j, v, IMG, sigma, True, one_pass=True)
    assert torch.equal(loss, ref) and torch.equal(w, wref)
    loss, w = crit.forward_fused(hm, j, v, IMG, sigma, True, one_pass=True)      # no requires_grad
    assert torch.equal(loss, ref)


@pytest.mark.parametrize("dtype", ["f32"])
def test_full_size(dtype):
    g = torch.Generator(device="cpu").manual_seed(1)
    hm = (torch.rand((1024, 21, 64, 64), generator=g) * 0.9).to(DTYPES[dtype]).to(DEV)
    joints, vis = synth.hand_joints(1024, 21, IMG, seed=17)
    render = _render(L.LOSS_DISTANCE_BALANCE, 2, True, 0.5)
    _check_case(hm, joints.to(DEV), vis.to(DEV), render)


def test_report_largest_differences():
    print(f"\nlargest relative differences: {MAX_REL}")
