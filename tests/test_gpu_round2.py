"""GPU: round-2 additions — lhn_metrics_finalize, the single-launch un-fused criterion, multi-tensor losses."""
import numpy as np
import pytest
import torch

from oracle import np_oracle as O
from litehandnet_b200 import _lib as L
from litehandnet_b200 import metrics as M
from litehandnet_b200 import ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _fin(K, N, mask_prob, T=20, dead=(), first=False):
    # the first four cases keep the ids they had before T and `dead` were parameters
    return pytest.param(K, N, mask_prob, T, dead, id=f"{K}-{N}-{mask_prob}" + ("" if first else f"-T{T}-dead{len(dead)}"))


# np.mean's pairwise sum changes form at 8 averaged joints (eight accumulators, then a tail) and ends at 128; joints
# without a valid sample (`dead`) are left out of the mean, so they move the count across those edges
FINALIZE_CASES = [
    _fin(16, 512, 0.9, first=True), _fin(21, 300, 0.5, first=True), _fin(7, 40, 0.9, dead=(3,), first=True),
    _fin(16, 64, 0.0, first=True),
    _fin(1, 64, 0.9), _fin(8, 64, 0.9), _fin(9, 64, 0.9), _fin(9, 64, 0.9, dead=(4,)), _fin(15, 64, 0.9),
    _fin(16, 64, 0.9, T=1, dead=(0,)), _fin(17, 64, 0.9), _fin(17, 64, 0.9, dead=(16,)), _fin(17, 64, 0.9, T=0, dead=(1, 2)),
    _fin(64, 32, 0.9, T=64), _fin(64, 32, 0.9, dead=tuple(range(55))), _fin(127, 16, 0.9), _fin(128, 16, 0.9),
    _fin(128, 16, 0.9, T=1, dead=tuple(range(0, 128, 2))), _fin(128, 16, 0.9, dead=tuple(range(121))),
    _fin(128, 8, 0.0, T=64),
]


@pytest.mark.parametrize("K,N,mask_prob,T,dead", FINALIZE_CASES)
def test_metrics_finalize_equals_host_expressions(K, N, mask_prob, T, dead):
    """lhn_metrics_finalize (device) == _report_metric's NumPy expressions on the same counters, bit for bit
    (datasets/base_dataset.py:193-261, top_down_eval.py:44-62,167-196), and == the oracle on the decoded points.
    K from 1 to 128, T = 0, 1, 20 and 64 AUC steps, all-zero counters."""
    hm, cen = synth.blob_heatmaps(N, K, 64, 64, seed=11, device=DEV)
    c, s = synth.bbox_center_scale(N, seed=12, device=DEV)
    gt, mask, wh = synth.pck_inputs(cen, seed=13, device=DEV, mask_prob=mask_prob)
    for k in dead:
        mask[:, k] = False                                  # a joint without any valid sample: acc = -1, left out of the mean
    acc = M.MetricAccumulator(K, device=DEV, auc_steps=T)
    r = acc.update_from_heatmaps(hm, c, s, gt, mask, wh, post_process="default")
    host = acc.compute()
    dev = acc.compute(on_device=True)
    for name in ("PCK", "AUC", "EPE"):
        assert float(host[name]) == float(dev[name]), (name, host[name], dev[name])
    full = acc.compute_device().cpu().numpy()
    cnt = acc.counters.cpu().numpy().reshape(-1, K)
    want_acc = np.array([h / v if v > 0 else -1 for h, v in zip(cnt[0], cnt[1])])
    assert np.array_equal(full[3:], want_acc)
    if mask_prob > 0:
        p64 = r["kpts"][..., :2].double().cpu().numpy()
        t = wh.max(1).values.double().cpu().numpy()
        _, pck, _ = O.keypoint_pck_accuracy(p64, gt.cpu().numpy(), mask.cpu().numpy(), 0.2, np.stack([t, t], 1))
        np.testing.assert_allclose(dev["PCK"], pck, rtol=1e-12)
        if T:
            np.testing.assert_allclose(dev["AUC"], O.keypoint_auc(p64, gt.cpu().numpy(), mask.cpu().numpy(), 30, T),
                                       rtol=1e-12)
        n_avg = int((cnt[1] > 0).sum())
        assert n_avg == K - len(dead)                         # the number of averaged joints the case aims at
    else:
        assert not cnt.any()
        assert dev["PCK"] == 0 and dev["AUC"] == 0 and dev["EPE"] == 0


def test_metrics_finalize_rejects_bad_arguments():
    cnt = torch.zeros(25 * 16, dtype=torch.int64, device=DEV)
    with pytest.raises(L.LhnError):
        ops.metrics_finalize(cnt, 15)
    with pytest.raises(L.LhnError):
        ops.metrics_finalize(cnt.int(), 16)
    with pytest.raises(L.LhnError):                         # past numpy's 128-element pairwise block
        ops.metrics_finalize(torch.zeros(25 * 129, dtype=torch.int64, device=DEV), 129)


# ---- SimDRLoss heads fused into one tcgen05 kernel (centernet_simdr_loss.py:42-69) ---------------------------
def _heads_case(B, K, HW, Lx, Ly, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    side = int(round(HW ** 0.5))
    hm, _ = synth.blob_heatmaps(B, K, side, side, seed=seed, device=DEV)
    wx = (torch.rand(Lx, HW, generator=g, device=DEV) * 2 - 1) * HW ** -0.5       # nn.Linear's default init range
    wy = (torch.rand(Ly, HW, generator=g, device=DEV) * 2 - 1) * HW ** -0.5
    bx = (torch.rand(Lx, generator=g, device=DEV) * 2 - 1) * HW ** -0.5
    by = (torch.rand(Ly, generator=g, device=DEV) * 2 - 1) * HW ** -0.5
    j, v = synth.hand_joints(B, K, (Lx // 2, Ly // 2), seed=seed + 1, device=DEV)
    tx, ty = ops.render_simdr(j, v, (Lx // 2, Ly // 2), 2, 2)
    w = v[..., :1].contiguous()
    return hm, wx, bx, wy, by, tx, ty, w


def _heads_reference(hm, wx, bx, wy, by, tx, ty, w):
    """SimDRLoss.forward literally, in float64 (the fp32 reference's own rounding is ~1e-7 of this)."""
    A = hm.flatten(2).double()
    px = A @ wx.double().t() + bx.double()
    py = A @ wy.double().t() + by.double()
    sl1 = torch.nn.SmoothL1Loss(reduction="mean")
    K = hm.shape[1]
    loss = 0
    for k in range(K):
        loss = loss + (sl1(px[:, k], tx[:, k].double()) * w[:, k].squeeze().double()).mean()
        loss = loss + (sl1(py[:, k], ty[:, k].double()) * w[:, k].squeeze().double()).mean()
    return loss / K, torch.cat([px, py], -1)


@pytest.mark.parametrize("B,K,HW,Lx,Ly", [(64, 21, 4096, 512, 512), (5, 21, 4096, 512, 512), (8, 16, 3136, 448, 448),
                                          (3, 2, 256, 64, 192)])
def test_simdr_heads_fused_forward(B, K, HW, Lx, Ly):
    hm, wx, bx, wy, by, tx, ty, w = _heads_case(B, K, HW, Lx, Ly, seed=40 + B)
    ref_loss, ref_pred = _heads_reference(hm, wx, bx, wy, by, tx, ty, w)
    split = ops.split_bf16(torch.cat([wx, wy]).contiguous())
    loss, dpred, pred = ops.simdr_heads_loss(hm, split, torch.cat([bx, by]), tx, ty, w, want_dpred=True, want_pred=True)
    np.testing.assert_allclose(float(loss.item()), float(ref_loss.item()), rtol=1e-5)
    # predictions: bf16x3 leaves ~2^-17 per product; bound relative to the magnitude of the summed terms
    mag = (hm.flatten(2).double().abs() @ torch.cat([wx, wy]).double().abs().t()).reshape(B * K, -1)
    err = (pred.double() - ref_pred.reshape(B * K, -1)).abs()
    assert float((err / mag).max()) < 2e-5, float((err / mag).max())
    want_g = (ref_pred.reshape(B * K, -1) - torch.cat([tx, ty], -1).reshape(B * K, -1).double()).clamp(-1, 1)
    assert float((dpred.double() - want_g).abs().max()) < 1e-4
    # deterministic (fixed-order reduction)
    loss2, _, _ = ops.simdr_heads_loss(hm, split, torch.cat([bx, by]), tx, ty, w)
    assert torch.equal(loss, loss2)


def test_split_bf16_is_a_17_bit_split():
    x = torch.randn(4096, device=DEV) * torch.logspace(-6, 6, 4096, device=DEV)
    hi, lo = ops.split_bf16(x)
    rec = hi.float() + lo.float()
    assert float(((rec - x).abs() / x.abs().clamp_min(1e-30)).max()) <= 2.0 ** -16
    assert torch.equal(hi, x.to(torch.bfloat16))


def test_simdr_loss_module_fused_matches_unfused_and_backward():
    """The drop-in SimDRLoss (reference parameters) — fused forward/backward against the reference's structure
    (nn.Linear heads + KLDiscretLoss) in float64 autograd."""
    from litehandnet_b200 import loss as LS
    from oracle.ref_loader import _AttrDict
    cfg = _AttrDict(DATASET=dict(image_size=[256, 256], heatmap_size=[64, 64]), PIPELINE=dict(simdr_split_ratio=2))
    B, K = 6, 21
    hm, wx, bx, wy, by, tx, ty, w = _heads_case(B, K, 4096, 512, 512, seed=77)
    crit = LS.SimDRLoss(cfg).to(DEV)
    with torch.no_grad():
        crit.x_shared_decoder.weight.copy_(wx); crit.x_shared_decoder.bias.copy_(bx)
        crit.y_shared_decoder.weight.copy_(wy); crit.y_shared_decoder.bias.copy_(by)
    hm_f = hm.clone().requires_grad_(True)
    loss = crit(hm_f, tx, ty, w)
    (loss * 3.0).backward()
    # float64 autograd through the literal module structure
    hm_d = hm.double().clone().requires_grad_(True)
    wxd, bxd, wyd, byd = [t.double().clone().requires_grad_(True) for t in (wx, bx, wy, by)]
    px = hm_d.flatten(2) @ wxd.t() + bxd
    py = hm_d.flatten(2) @ wyd.t() + byd
    sl1 = torch.nn.SmoothL1Loss(reduction="mean")
    ref = 0
    for k in range(K):
        ref = ref + (sl1(px[:, k], tx[:, k].double()) * w[:, k].squeeze().double()).mean()
        ref = ref + (sl1(py[:, k], ty[:, k].double()) * w[:, k].squeeze().double()).mean()
    ref = ref / K
    (ref * 3.0).backward()
    np.testing.assert_allclose(float(loss.item()), float(ref.item()), rtol=1e-5)

    def close(a, b, what):
        scale = float(b.abs().max())
        assert float((a.double() - b).abs().max()) <= 2e-5 * scale + 1e-12, what

    close(hm_f.grad, hm_d.grad, "d heatmap")
    close(crit.x_shared_decoder.weight.grad, wxd.grad, "d Wx")
    close(crit.y_shared_decoder.weight.grad, wyd.grad, "d Wy")
    close(crit.x_shared_decoder.bias.grad, bxd.grad, "d bx")
    close(crit.y_shared_decoder.bias.grad, byd.grad, "d by")
    # the un-fused route (cuBLAS heads + lhn_simdr_smoothl1) gives the same loss
    crit.fused = False
    np.testing.assert_allclose(float(crit(hm, tx, ty, w).item()), float(ref.item()), rtol=1e-5)
    # weights changed in place -> the cached bf16 split is rebuilt
    crit.fused = True
    with torch.no_grad():
        crit.x_shared_decoder.weight.mul_(0.5)
    l2 = crit(hm, tx, ty, w)
    ref2, _ = _heads_reference(hm, wx * 0.5, bx, wy, by, tx, ty, w)
    np.testing.assert_allclose(float(l2.item()), float(ref2.item()), rtol=1e-5)


@pytest.mark.parametrize("bn", ["64", "80", "128"])
def test_simdr_heads_tile_straddles_the_xy_boundary(bn, monkeypatch):
    """Lx = 448 = 3.5 tiles of 128 columns (5.6 of 80: the last N tile is ragged too): one tile holds x columns and y
    columns (per-column target select)."""
    monkeypatch.setenv("LHN_HEADS_BN", bn)
    B, K, HW, Lx, Ly = 40, 16, 3136, 448, 448
    hm, wx, bx, wy, by, tx, ty, w = _heads_case(B, K, HW, Lx, Ly, seed=91)
    ref_loss, _ = _heads_reference(hm, wx, bx, wy, by, tx, ty, w)
    loss, dpred, pred = ops.simdr_heads_loss(hm, ops.split_bf16(torch.cat([wx, wy]).contiguous()), torch.cat([bx, by]), tx, ty, w,
                                             want_dpred=True, want_pred=True)
    np.testing.assert_allclose(float(loss.item()), float(ref_loss.item()), rtol=1e-5)
    _, ref_pred = _heads_reference(hm, wx, bx, wy, by, tx, ty, w)
    mag = (hm.flatten(2).double().abs() @ torch.cat([wx, wy]).double().abs().t()).reshape(B * K, -1)
    assert float(((pred.double() - ref_pred.reshape(B * K, -1)).abs() / mag).max()) < 2e-5      # every column of every tile


# ---- the un-fused criterion in ONE launch, several tensors at once (lhn_loss_mse_multi) ----------------------
@pytest.mark.parametrize("mode", [L.LOSS_DISTANCE_BALANCE, L.LOSS_DISTANCE, L.LOSS_JOINTS_MSE])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_loss_mse_multi_matches_three_launch_path_and_oracle(mode, dtype):
    shapes = [(6, 21, 16, 16), (6, 21, 16, 16), (6, 21, 32, 32), (6, 21, 64, 64)]       # SRHandNet's four scales
    g = torch.Generator(device=DEV).manual_seed(3)
    outs, tgts, ws = [], [], []
    for i, (B, K, H, W) in enumerate(shapes):
        j, v = synth.hand_joints(B, K, (256, 256), seed=20 + i, device=DEV)
        t, tw = ops.render_targets(j, v, (256, 256), (W, H), 2.0 if H > 16 else 1.0, True)
        o = (t + torch.randn(t.shape, generator=g, device=DEV) * 0.1).to(dtype)
        outs.append(o); tgts.append(t.to(dtype)); ws.append(tw)
    lw = [0.3, 0.3, 0.5, 1.0]
    loss, sums, per = ops.loss_mse_multi(outs, tgts, ws, mode, 0.5, "mean", lw)
    want_total = 0.0
    for i in range(4):
        partials = ops.loss_partials(outs[i], tgts[i], ws[i], mode, 0.5)
        s3 = ops.loss_reduce(partials)
        l3 = ops.loss_finalize(s3, mode, "mean")
        np.testing.assert_allclose(sums[i].cpu().numpy(), s3.cpu().numpy(), rtol=1e-6)   # f32 partial sums: fused multiply-adds and another summation order
        np.testing.assert_allclose(float(per[i].item()), float(l3.item()), rtol=1e-6)
        o64, t64, w64 = outs[i].float().cpu().numpy(), tgts[i].float().cpu().numpy(), ws[i].cpu().numpy()
        if mode == L.LOSS_JOINTS_MSE:
            ref = O.joints_distance_loss_mse(o64, t64, w64)
        else:
            ref = O.distance_loss_l2(o64, t64, w64, balance=(mode == L.LOSS_DISTANCE_BALANCE))
        np.testing.assert_allclose(float(per[i].item()), float(ref), rtol=1e-5)
        want_total += lw[i] * float(ref)
    np.testing.assert_allclose(float(loss.item()), want_total, rtol=1e-5)
    loss2, _, _ = ops.loss_mse_multi(outs, tgts, ws, mode, 0.5, "mean", lw)
    assert torch.equal(loss, loss2), "fixed-order reduction: bitwise reproducible"


def test_loss_mse_multi_single_large_tensor_and_sum_reduction():
    B, K = 300, 21
    j, v = synth.hand_joints(B, K, (256, 256), seed=31, device=DEV)
    t, tw = ops.render_targets(j, v, (256, 256), (64, 64), 2.0, True)
    o = t + torch.randn(t.shape, generator=torch.Generator(device=DEV).manual_seed(4), device=DEV) * 0.05
    for red in ("mean", "sum"):
        loss, sums, _ = ops.loss_mse_multi([o], [t], [tw], L.LOSS_DISTANCE_BALANCE, 0.5, red)
        ref = O.distance_loss_l2(o.cpu().numpy(), t.cpu().numpy(), tw.cpu().numpy(), balance=True, reduction=red)
        np.testing.assert_allclose(float(loss.item()), float(ref), rtol=1e-5)
    with pytest.raises(L.LhnError):
        ops.loss_mse_multi([o] * 9, [t] * 9, [tw] * 9, L.LOSS_DISTANCE)


# ---- the torch-extension shim: same library entry point, same results as the ctypes route ---------------------
def test_torch_extension_route_equals_ctypes_route():
    assert L.ext() is not None, "the extension shim must be built in-tree (litehandnet_b200.build)"
    hm, cen = synth.blob_heatmaps(16, 21, 64, 64, seed=5, device=DEV, zero_frac=0.05, tie_frac=0.05)
    hf = synth.flipped_blob_heatmaps(cen, 64, 64, seed=6, device=DEV)
    c, s = synth.bbox_center_scale(16, seed=7, device=DEV)
    for refine in (L.REFINE_SIGN, L.REFINE_DARK, L.REFINE_OFFSET_HALF):
        for flip in (None, hf):
            a = ops.decode_heatmap(hm, L.MASK_NEG1, refine, L.XFORM_CENTER_SCALE, c, s, hm_flip=flip)
            b = ops._decode_heatmap_ctypes(hm, L.MASK_NEG1, refine, L.XFORM_CENTER_SCALE, c, s, hm_flip=flip)
            for k in ("hm_kpts", "kpts", "idx"):
                assert torch.equal(a[k], b[k]), (refine, k)
    # channel slice (stride_c != H*W) and bf16 go through the shim as well
    big = torch.cat([hm, hm.flip(1)], 1)
    a = ops.decode_heatmap(big[:, :21], L.MASK_ZERO, L.REFINE_NONE)
    b = ops._decode_heatmap_ctypes(hm, L.MASK_ZERO, L.REFINE_NONE)
    assert torch.equal(a["kpts"], b["kpts"])
    a = ops.decode_heatmap(hm.bfloat16(), L.MASK_NEG1, L.REFINE_SIGN, L.XFORM_CENTER_SCALE, c, s, want_idx=False)
    b = ops._decode_heatmap_ctypes(hm.bfloat16(), L.MASK_NEG1, L.REFINE_SIGN, L.XFORM_CENTER_SCALE, c, s)
    assert a["idx"] is None and torch.equal(a["kpts"], b["kpts"])
    with pytest.raises(L.LhnError):
        ops.decode_heatmap(hm.cpu(), L.MASK_NEG1, L.REFINE_SIGN)
    with pytest.raises(L.LhnError):                       # f64 heatmaps: rejected by the shim, as an LhnError
        ops.decode_heatmap(hm.double(), L.MASK_NEG1, L.REFINE_SIGN)


# ---- low-precision inputs at the sizes that are measured (VERDICT r1 weak #9) ---------------------------------
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("B,HW,flip,sigma", [(1024, 64, True, 2), (1024, 56, False, 2), (96, 128, False, 4)])
def test_low_precision_fused_at_measured_sizes(dt, B, HW, flip, sigma):
    """bf16 / f16 network outputs through the one-launch fused step (render + balanced loss + [flip] + DARK) at the
    batch sizes of the roofline rows: oracle = the reference pipeline on the upcast f32 tensors, all samples."""
    from conftest import assert_coords_close, xform_magnitude
    from oracle import cpu_path
    from litehandnet_b200 import fused
    K = 21
    img = (4 * HW, 4 * HW)
    hm, cen = synth.blob_heatmaps(B, K, HW, HW, seed=61, device=DEV, sigma=float(sigma), zero_frac=0.01)
    hm = hm.to(dt)
    hf = synth.flipped_blob_heatmaps(cen, HW, HW, seed=62, device=DEV, sigma=float(sigma)).to(dt) if flip else None
    j, v = synth.hand_joints(B, K, img, seed=63, device=DEV)
    c, s = synth.bbox_center_scale(B, seed=64, device=DEV)
    out = fused.fused_render_loss_decode(hm, j, v, c, s, hm_flip=hf, image_size=img, sigma=sigma)
    runner = cpu_path.FusedCpuRunner(hm.float().cpu().numpy(), None if hf is None else hf.float().cpu().numpy(),
                                     j.cpu().numpy(), v.cpu().numpy(), c.cpu().numpy(), s.cpu().numpy(),
                                     image_size=img, sigma=sigma, kernel=11)
    try:
        with np.errstate(all="ignore"):
            preds, loss, _ = runner.run()
        ridx = runner.last_idx
    finally:
        runner.close()
    assert np.array_equal(out["idx"].cpu().numpy(), ridx), "argmax (first index on the many bf16/f16 ties)"
    got = out["preds"].cpu().numpy()
    assert_coords_close(got[..., :2], preds[..., :2], what=f"{dt} {HW}x{HW}", mag=xform_magnitude(c.cpu().numpy(), s.cpu().numpy()))
    assert np.array_equal(got[..., 2], preds[..., 2], equal_nan=True)
    np.testing.assert_allclose(float(out["loss"].item()), float(loss), rtol=1e-5)


# ---- compile-time instantiations added in round 2: 32x32 / 16x16 f32, 128x128 bf16 / f16 (+ flip) ---------------
@pytest.mark.parametrize("HW,dt,flip,sigma,B", [(32, torch.float32, False, 1.5, 300), (16, torch.float32, False, 1.0, 700),
                                                (128, torch.bfloat16, True, 4, 24), (128, torch.float16, True, 4, 24),
                                                (32, torch.float32, True, 1.5, 50)])
def test_fused_step_on_the_new_compile_time_shapes(HW, dt, flip, sigma, B, monkeypatch):
    from conftest import assert_coords_close, xform_magnitude
    from oracle import cpu_path
    from litehandnet_b200 import fused
    K = 21
    img = (4 * HW, 4 * HW)
    # (no exact-tie planes here: a tie puts the argmax on an isolated noise spike, where DARK's 2x2 solve is
    # ill-conditioned and amplifies 1-ulp differences of the blur to tenths of a pixel — in the reference too)
    hm, cen = synth.blob_heatmaps(B, K, HW, HW, seed=71, device=DEV, sigma=float(sigma), margin=min(4.0, HW / 8), zero_frac=0.02)
    hm = hm.to(dt)
    hf = synth.flipped_blob_heatmaps(cen, HW, HW, seed=72, device=DEV, sigma=float(sigma)).to(dt) if flip else None
    j, v = synth.hand_joints(B, K, img, seed=73, device=DEV)
    c, s = synth.bbox_center_scale(B, seed=74, device=DEV)
    out = fused.fused_render_loss_decode(hm, j, v, c, s, hm_flip=hf, image_size=img, sigma=sigma)
    # the compile-time instantiation and the run-time-size one do the same arithmetic: bitwise equal, ties included
    hm_t, _ = synth.blob_heatmaps(B, K, HW, HW, seed=75, device=DEV, sigma=float(sigma), margin=min(4.0, HW / 8), zero_frac=0.02,
                                  tie_frac=0.05)
    hm_t = hm_t.to(dt)
    fast = fused.fused_render_loss_decode(hm_t, j, v, c, s, hm_flip=hf, image_size=img, sigma=sigma)
    monkeypatch.setenv("LHN_NO_FAST", "1")
    slow = fused.fused_render_loss_decode(hm_t, j, v, c, s, hm_flip=hf, image_size=img, sigma=sigma)
    monkeypatch.delenv("LHN_NO_FAST")
    assert torch.equal(fast["idx"], slow["idx"]) and torch.equal(fast["preds"], slow["preds"]), "fast != run-time-size path"
    assert torch.equal(fast["loss_sums"], slow["loss_sums"])
    runner = cpu_path.FusedCpuRunner(hm.float().cpu().numpy(), None if hf is None else hf.float().cpu().numpy(),
                                     j.cpu().numpy(), v.cpu().numpy(), c.cpu().numpy(), s.cpu().numpy(),
                                     image_size=img, sigma=sigma, kernel=11)
    try:
        with np.errstate(all="ignore"):
            preds, loss, _ = runner.run()
        ridx = runner.last_idx
    finally:
        runner.close()
    assert np.array_equal(out["idx"].cpu().numpy(), ridx)
    got = out["preds"].cpu().numpy()
    assert_coords_close(got[..., :2], preds[..., :2], what=f"{dt} {HW}x{HW} flip={flip}",
                        mag=xform_magnitude(c.cpu().numpy(), s.cpu().numpy()))
    assert np.array_equal(got[..., 2], preds[..., 2], equal_nan=True)
    np.testing.assert_allclose(float(out["loss"].item()), float(loss), rtol=1e-5)
    # decode only ('default' refinement) on the same shapes
    r = ops.decode_heatmap(hm, L.MASK_NEG1, L.REFINE_SIGN, L.XFORM_CENTER_SCALE, c, s, hm_flip=hf)
    avg = hm.float().cpu().numpy() if hf is None else O.flip_average(hm.float().cpu().numpy(), hf.float().cpu().numpy(), ())
    with np.errstate(all="ignore"):
        _, p, mv = O.keypoints_from_heatmaps(avg, c.cpu().numpy(), s.cpu().numpy(), "default", 11)
    assert np.array_equal(r["idx"].cpu().numpy(), avg.reshape(B, K, -1).argmax(-1))
    assert_coords_close(r["kpts"].cpu().numpy()[..., :2], p, what="decode default", mag=xform_magnitude(c.cpu().numpy(), s.cpu().numpy()))


def test_fused_criterion_refuses_joint_weights():
    """ADVICE r1: the in-kernel render applies no per-joint weights (generateTarget.py:156-157) — refuse, do not ignore."""
    from litehandnet_b200 import loss as LS
    from oracle.ref_loader import _AttrDict
    cfg = _AttrDict(DATASET=dict(image_size=[256, 256], heatmap_size=[64, 64], num_joints=21),
                    PIPELINE=dict(unbiased_encoding=True, kernel=(11, 11), use_udp=False, simdr_split_ratio=0, sigma=2),
                    MODEL=dict(name="litehandnet"), LOSS=dict(type="TopdownHeatmapLoss", loss_weight=[1.0, 1.0], auto_weight=False))
    crit = LS.get_loss(cfg)
    hm, _ = synth.blob_heatmaps(2, 21, 64, 64, seed=1, device=DEV)
    j, v = synth.hand_joints(2, 21, seed=2, device=DEV)
    loss, d = crit(hm, dict(joints_3d=j, joints_3d_visible=v))
    assert np.isfinite(d["heatmap"])
    with pytest.raises(NotImplementedError):
        crit(hm, dict(joints_3d=j, joints_3d_visible=v, use_different_joint_weights=True))
    with pytest.raises(NotImplementedError):
        crit(hm, dict(joints_3d=j, joints_3d_visible=v, ann_info=dict(use_different_joint_weights=True)))


@pytest.mark.parametrize("sigma,isz,k", [(2, (256, 256), 2), (3, (256, 192), 2), (10, (256, 256), 2), (2, (255, 253), 1)])
def test_render_simdr_window_edges(sigma, isz, k):
    """generate_simder.py:9-31 with the joints a data pipeline can hand over: on a bin, between bins, at and beyond the
    borders, far outside, infinite, NaN, invisible.  sigma 2/3 take the windowed path (lhn_loss_render.cu), sigma 10 the
    window is wider than the kernel's buffer and (255, 253) is not 16-byte tileable: both take the plain path."""
    rng = np.random.default_rng(7)
    B, K = 6, 21
    j = np.zeros((B, K, 3), np.float32)
    j[..., 0] = rng.uniform(-40, isz[0] + 40, (B, K))
    j[..., 1] = rng.uniform(-40, isz[1] + 40, (B, K))
    j[0, 0, :2] = (0.0, isz[1] - 1); j[0, 1, :2] = (isz[0] - 0.5, 0.25); j[0, 2, :2] = (-14.4 * sigma / k, isz[1] + 14.4 * sigma / k)
    j[0, 3, :2] = (-1e12, 1e12); j[0, 4, :2] = (np.inf, -np.inf); j[0, 5, :2] = (np.nan, 10.0); j[0, 6, :2] = (17.0, np.nan)
    j[0, 7, :2] = (3e9, 64.0)
    v = (rng.uniform(size=(B, K, 1)) < 0.8).astype(np.float32)
    v[0, :8] = 1
    with np.errstate(all="ignore"):
        want_x, want_y = O.render_simdr_batch(j, v, isz, k, sigma)
    sx, sy = ops.render_simdr(torch.from_numpy(j).to(DEV), torch.from_numpy(v).to(DEV), isz, k, sigma)
    nump = lambda t: t.cpu().numpy()
    np.testing.assert_allclose(nump(sx), want_x, rtol=1e-5, atol=1e-7, equal_nan=True)
    np.testing.assert_allclose(nump(sy), want_y, rtol=1e-5, atol=1e-7, equal_nan=True)
    assert np.all(nump(sx)[want_x > 1e-30] > 0) and np.all(nump(sy)[want_y > 1e-30] > 0)   # the cut removes only what rounds to 0


@pytest.mark.parametrize("B,K,Lx,Ly,dt", [(1024, 21, 64, 48, torch.float32), (700, 17, 128, 128, torch.float32),
                                          (1024, 16, 64, 64, torch.bfloat16), (96, 21, 512, 512, torch.float32),
                                          (420, 21, 64, 64, torch.float32)])
def test_simdr_smoothl1_large_batches_take_the_joint_per_warp_path(B, K, Lx, Ly, dt):
    """KLDiscretLoss (loss/simdrLoss.py) at sizes where lhn_simdr_smoothl1 runs one joint per warp with per-lane f64
    sums and the cluster finalise (B*K rows > the resident warps; (96, 21) stays on the row-per-warp path with the
    one-block finalise, (420, 21) on the row-per-warp path with the cluster finalise):
    against the NumPy oracle on the same values, weights with zeros and non-unit values."""
    g = torch.Generator(device=DEV).manual_seed(B + K)
    ox = torch.randn(B, K, Lx, generator=g, device=DEV) * 0.7
    oy = torch.randn(B, K, Ly, generator=g, device=DEV) * 0.7
    tx = torch.rand(B, K, Lx, generator=g, device=DEV)
    ty = torch.rand(B, K, Ly, generator=g, device=DEV)
    ox[0, 0, :5] = 3.0; oy[1, 2, -3:] = -2.5                      # |d| > 1: the linear branch
    w = (torch.rand(B, K, 1, generator=g, device=DEV) < 0.8).float() * (0.5 + torch.rand(B, K, 1, generator=g, device=DEV))
    ox, oy, tx, ty = (t.to(dt) for t in (ox, oy, tx, ty))
    got = float(ops.simdr_smoothl1(ox, oy, tx, ty, w).item())
    f = lambda t: t.float().cpu().numpy()
    want = float(O.kl_discret_loss(f(ox), f(oy), f(tx), f(ty), f(w)))
    np.testing.assert_allclose(got, want, rtol=2e-6)
    # run-to-run: the summation order is fixed
    assert float(ops.simdr_smoothl1(ox, oy, tx, ty, w).item()) == got
