"""GPU parity tests proper: the CUDA path (through the C ABI) against the numpy oracle on the same
seeded inputs and against the committed golden vectors (outputs of the executed reference).

Bars (north_star): argmax indices and PCK hit counts bit-exact; float coordinates and losses within
1e-5 relative (assert_coords_close adds a 2e-5 px absolute floor for coordinates near zero).
"""
import numpy as np
import pytest
import torch

from conftest import assert_coords_close, load_golden
from oracle import np_oracle as O
from litehandnet_b200 import synth

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def ops():
    from litehandnet_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def L():
    from litehandnet_b200 import _lib
    return _lib


def cu(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def nump(t):
    return t.detach().cpu().numpy()


def synth_case(N=8, K=21, H=64, W=64, seed=0, **kw):
    hm, cen = synth.blob_heatmaps(N, K, H, W, seed=seed, zero_frac=0.03, tie_frac=0.03, **kw)
    center, scale = synth.bbox_center_scale(N, seed=seed + 1)
    return hm.numpy(), cen, center.numpy(), scale.numpy()


# ---- argmax conventions (A1-A4) ---------------------------------------------------------------
@pytest.mark.parametrize("case", ["decode_64.npz", "decode_56.npz", "decode_mpii16.npz"])
def test_argmax_golden(ops, L, case):
    g = load_golden(case)
    hm = cu(g["hm"])
    for mode, name in ((L.MASK_ZERO, "zero"), (L.MASK_NEG1, "neg1"), (L.MASK_NONE, "none")):
        r = ops.decode_heatmap(hm, mode, L.REFINE_NONE)
        assert np.array_equal(nump(r["idx"]), g["ref_argmax_idx"]), "argmax index must be bit-exact"
        p, mv, _ = O.max_preds(g["hm"], name)
        k = nump(r["hm_kpts"])
        assert np.array_equal(k[..., :2], p)
        assert np.array_equal(k[..., 2:], mv, equal_nan=True)
    r = ops.decode_heatmap(hm, L.MASK_ZERO, L.REFINE_NONE)
    assert np.array_equal(nump(r["hm_kpts"])[..., :2], g["ref_a1_preds"])
    assert np.array_equal(nump(r["hm_kpts"])[..., 2:], g["ref_a1_maxvals"], equal_nan=True)


@pytest.mark.parametrize("shape", [(4, 21, 64, 64), (3, 5, 56, 56), (2, 4, 128, 128), (3, 6, 14, 14),
                                   (2, 3, 28, 28), (2, 7, 32, 32), (2, 3, 16, 16), (1, 2, 48, 64)])
def test_argmax_shapes_ties_nan(ops, L, shape):
    N, K, H, W = shape
    hm, _, _, _ = synth_case(N, K, H, W, seed=H + W)
    hm[0, 0] = 0.0                                     # all-zero plane -> idx 0
    hm[0, 1] = -1.0                                    # constant negative plane
    hm[-1, -1, H // 2, W // 3] = np.nan                # NaN is maximal
    hm[-1, -1, H - 1, W - 1] = np.nan                  # first NaN wins
    hm[-1, 0] = -np.inf                                # all -inf -> idx 0
    hm[0, -1, 1, 2] = np.inf
    hm[0, -1, 3, 1] = np.inf                           # first +inf wins
    r = ops.decode_heatmap(cu(hm), L.MASK_NONE, L.REFINE_NONE)
    idx, mv = O.argmax_planes(hm)
    assert np.array_equal(nump(r["idx"]), idx)
    assert np.array_equal(nump(r["hm_kpts"])[..., 2], mv, equal_nan=True)


def test_argmax_every_position_and_4way_ties(ops, L):
    H = W = 64
    rng = np.random.default_rng(5)
    hm = rng.uniform(0, 0.5, (8, 32, H, W)).astype(np.float32)
    flat = hm.reshape(8 * 32, -1)
    for p in range(flat.shape[0]):
        pos = rng.choice(H * W, size=4, replace=False)
        flat[p, pos] = 0.75                            # exact 4-way tie: lowest flat index wins
    r = ops.decode_heatmap(cu(hm), L.MASK_NEG1, L.REFINE_NONE)
    assert np.array_equal(nump(r["idx"]).reshape(-1), np.argmax(flat, 1))


def test_channel_sliced_view_needs_no_copy(ops, L):
    hm, _, _, _ = synth_case(3, 24, 64, 64, seed=9)
    full = cu(hm)
    r = ops.decode_heatmap(full[:, :21], L.MASK_NEG1, L.REFINE_NONE)     # model_output[:, :num_joints]
    assert np.array_equal(nump(r["idx"]), O.argmax_planes(hm[:, :21])[0])


# ---- refinements + back-transform ---------------------------------------------------------------
@pytest.mark.parametrize("case", ["decode_64.npz", "decode_56.npz", "decode_mpii16.npz"])
def test_gen2_decode_golden(ops, L, case):
    g = load_golden(case)
    hm, c, s = cu(g["hm"]), cu(g["center"]), cu(g["scale"])
    for refine, tag in ((L.REFINE_SIGN, "default"), (L.REFINE_NONE, "none"), (L.REFINE_DARK, "unbiased")):
        r = ops.decode_heatmap(hm, L.MASK_NEG1, refine, L.XFORM_CENTER_SCALE, c, s)
        hk, k = nump(r["hm_kpts"]), nump(r["kpts"])
        if refine == L.REFINE_DARK:
            assert_coords_close(hk[..., :2], g[f"ref_g2_{tag}_hm_preds"], what=f"{tag} hm_preds")
            assert_coords_close(k[..., :2], g[f"ref_g2_{tag}_preds"], what=f"{tag} preds")
        else:   # quarter-offset arithmetic is exact
            assert np.array_equal(hk[..., :2], g[f"ref_g2_{tag}_hm_preds"], equal_nan=True)
            assert np.array_equal(k[..., :2], g[f"ref_g2_{tag}_preds"], equal_nan=True)
        assert np.array_equal(hk[..., 2:], g[f"ref_g2_{tag}_maxvals"], equal_nan=True)


@pytest.mark.parametrize("case", ["decode_64.npz", "decode_56.npz", "decode_mpii16.npz"])
def test_legacy_decode_golden(ops, L, case):
    g = load_golden(case)
    hm = cu(g["hm"])
    H, W = g["hm"].shape[2:]
    isz = g["image_size"]
    stride = (float(isz[0] // W), float(isz[1] // H))
    r = ops.decode_heatmap(hm, L.MASK_NONE, L.REFINE_OFFSET_HALF, L.XFORM_SCALE, scale_xy=stride)
    assert np.array_equal(nump(r["hm_kpts"]), g["ref_legacy_offset_hm"], equal_nan=True)
    assert np.array_equal(nump(r["kpts"]), g["ref_legacy_offset_img"], equal_nan=True)
    r = ops.decode_heatmap(hm, L.MASK_NONE, L.REFINE_DARK_LEGACY, L.XFORM_SCALE, scale_xy=stride)
    assert_coords_close(nump(r["hm_kpts"]), g["ref_legacy_dark_hm"], what="legacy dark hm")
    assert_coords_close(nump(r["kpts"]), g["ref_legacy_dark_img"], what="legacy dark img")
    r = ops.decode_heatmap(hm, L.MASK_NONE, L.REFINE_OFFSET, L.XFORM_SCALE,
                           scale_xy=(float(isz[0]) / W, float(isz[1]) / H))
    assert np.array_equal(nump(r["kpts"]), g["ref_parse_sh"], equal_nan=True)
    r = ops.decode_heatmap(hm, L.MASK_ZERO, L.REFINE_SIGN_ROUND, L.XFORM_CENTER_SCALE, cu(g["center"]), cu(g["scale"]))
    assert_coords_close(nump(r["kpts"])[..., :2], g["ref_final_preds"], rtol=1e-5, atol=1e-4, what="final_preds")


def test_sp_parser_known_answer(ops, L):
    hm = torch.zeros((2, 4, 64, 64), device=DEV)
    hm[..., 3, 3] = 1; hm[..., 3, 2] = 0.5; hm[..., 2, 3] = 0.5
    r = ops.decode_heatmap(hm, L.MASK_NONE, L.REFINE_OFFSET, L.XFORM_SCALE, scale_xy=(4.0, 4.0))
    assert np.array_equal(nump(r["kpts"])[0, 0], np.array([11.0, 11.0, 1.0], np.float32))


@pytest.mark.parametrize("shape", [(16, 21, 64, 64), (4, 8, 56, 56), (2, 4, 128, 128), (4, 5, 28, 28)])
def test_decode_variants_vs_oracle(ops, L, shape):
    N, K, H, W = shape
    hm, _, center, scale = synth_case(N, K, H, W, seed=3 * H)
    t, c, s = cu(hm), cu(center), cu(scale)
    with np.errstate(all="ignore"):
        # D3 + T1
        hp, p, mv = O.keypoints_from_heatmaps(hm, center, scale, "default")
        r = ops.decode_heatmap(t, L.MASK_NEG1, L.REFINE_SIGN, L.XFORM_CENTER_SCALE, c, s)
        assert np.array_equal(nump(r["hm_kpts"])[..., :2], hp) and np.array_equal(nump(r["kpts"])[..., :2], p)
        # D5 + T1
        hp, p, mv = O.keypoints_from_heatmaps(hm, center, scale, "unbiased", 11)
        r = ops.decode_heatmap(t, L.MASK_NEG1, L.REFINE_DARK, L.XFORM_CENTER_SCALE, c, s)
        assert_coords_close(nump(r["hm_kpts"])[..., :2], hp, what="dark hm")
        assert_coords_close(nump(r["kpts"])[..., :2], p, what="dark img")
        # D1, D6 (legacy)
        r = ops.decode_heatmap(t, L.MASK_NONE, L.REFINE_OFFSET_HALF)
        assert np.array_equal(nump(r["hm_kpts"]), O.get_pred_kpt(hm, dark=False))
        r = ops.decode_heatmap(t, L.MASK_NONE, L.REFINE_DARK_LEGACY)
        assert_coords_close(nump(r["hm_kpts"]), O.get_pred_kpt(hm, dark=True), what="legacy dark")
        # D2, D4
        r = ops.decode_heatmap(t, L.MASK_NONE, L.REFINE_OFFSET, L.XFORM_SCALE, scale_xy=(256.0 / W, 256.0 / H))
        assert np.array_equal(nump(r["kpts"]), O.parse_sh(hm, (256, 256)))
        r = ops.decode_heatmap(t, L.MASK_ZERO, L.REFINE_SIGN_ROUND, L.XFORM_CENTER_SCALE, c, s)
        assert np.array_equal(nump(r["kpts"])[..., :2], O.get_final_preds(hm, center, scale))


def test_dark_clamp_slow_path(ops, L):
    """Planes where the 1e-10 clamp of log() binds: isolated spikes, tiny and negative planes."""
    H = W = 64
    hm = np.zeros((1, 6, H, W), np.float32)
    hm[0, 0, 20, 30] = 1.0                                    # single spike on zeros
    hm[0, 1, 10, 12] = 1e-6; hm[0, 1, 10, 13] = 5e-7          # tiny values
    hm[0, 2] = -0.5; hm[0, 2, 30, 30] = -0.1                  # all negative (legacy: no mask)
    hm[0, 3, 40, 40] = 0.8; hm[0, 3, 41, 40] = 0.4; hm[0, 3, 40, 41] = 0.3
    hm[0, 4, 5:9, 5:9] = 0.2; hm[0, 4, 6, 6] = 0.3
    hm[0, 5, 33, 31] = 1e-12
    with np.errstate(all="ignore"):
        for refine, mask, legacy in ((L.REFINE_DARK, "neg1", False), (L.REFINE_DARK_LEGACY, "none", True)):
            co, mv, _ = O.max_preds(hm, mask)
            want = O.refine_dark(np.concatenate([co, mv], 2), hm, 19 if legacy else 11, legacy)
            r = ops.decode_heatmap(cu(hm), L.MASK_NEG1 if mask == "neg1" else L.MASK_NONE, refine)
            assert_coords_close(nump(r["hm_kpts"]), want, rtol=1e-5, atol=1e-4, what=f"slow path legacy={legacy}")


# ---- flip test ------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,pairs", [(21, ()), (16, synth.MPII_FLIP_PAIRS)])
def test_flip_average_decode(ops, L, K, pairs):
    N, H, W = 6, 64, 64
    hm, cen, center, scale = synth_case(N, K, H, W, seed=17)
    hf = synth.flipped_blob_heatmaps(cen, H, W, seed=18, flip_pairs=pairs).numpy()
    fi = list(range(K))
    for a, b in pairs:
        fi[a], fi[b] = fi[b], fi[a]
    avg = O.flip_average(hm, hf, pairs)
    assert np.array_equal(nump(ops.flip_back(cu(hf), cu(np.array(fi, np.int32)))), O.flip_back(hf, pairs))
    with np.errstate(all="ignore"):
        hp, p, mv = O.keypoints_from_heatmaps(avg, center, scale, "unbiased", 11)
    r = ops.decode_heatmap(cu(hm), L.MASK_NEG1, L.REFINE_DARK, L.XFORM_CENTER_SCALE, cu(center), cu(scale),
                           hm_flip=cu(hf), flip_index=cu(np.array(fi, np.int32)))
    assert np.array_equal(nump(r["idx"]), O.argmax_planes(avg)[0]), "argmax of the average must be bit-exact"
    assert np.array_equal(nump(r["hm_kpts"])[..., 2:], mv)
    assert_coords_close(nump(r["hm_kpts"])[..., :2], hp, what="flip dark hm")
    assert_coords_close(nump(r["kpts"])[..., :2], p, what="flip dark img")


# ---- fused render + loss + decode (the headline path) ----------------------------------------------
@pytest.mark.parametrize("flip", [False, True])
@pytest.mark.parametrize("unbiased", [True, False])
def test_fused_render_loss_decode(ops, L, flip, unbiased):
    N, K, H, W = 12, 21, 64, 64
    hm, cen, center, scale = synth_case(N, K, H, W, seed=23)
    hf = synth.flipped_blob_heatmaps(cen, H, W, seed=24).numpy() if flip else None
    j, v = synth.hand_joints(N, K, seed=25, outside_frac=0.05, vis_prob=0.9)
    v[0, 0, 0] = 0.3
    jn, vn = j.numpy(), v.numpy()
    tg, tw = O.render_targets(jn, vn, (256, 256), (W, H), 2, unbiased)
    for mode, bal in ((L.LOSS_DISTANCE_BALANCE, True), (L.LOSS_DISTANCE, False)):
        want = O.distance_loss_l2(hm, tg, tw, balance=bal)
        r = ops.decode_heatmap(cu(hm), L.MASK_NEG1, L.REFINE_DARK, L.XFORM_CENTER_SCALE, cu(center), cu(scale),
                               hm_flip=None if hf is None else cu(hf),
                               render=dict(loss_mode=mode, image_size=(256, 256), sigma=2, unbiased=unbiased),
                               joints=cu(jn), vis=cu(vn))
        loss = nump(ops.loss_finalize(ops.loss_reduce(r["partials"]), mode))[0]
        np.testing.assert_allclose(loss, want, rtol=1e-5)
        assert np.array_equal(nump(r["weight"]), tw.reshape(N, K))
    want = O.joints_distance_loss_mse(hm, tg, tw)
    r = ops.decode_heatmap(cu(hm), L.MASK_NEG1, L.REFINE_NONE,
                           render=dict(loss_mode=L.LOSS_JOINTS_MSE, image_size=(256, 256), sigma=2, unbiased=unbiased),
                           joints=cu(jn), vis=cu(vn))
    np.testing.assert_allclose(nump(ops.loss_finalize(ops.loss_reduce(r["partials"]), L.LOSS_JOINTS_MSE))[0],
                               want, rtol=1e-5)
    avg = hm if hf is None else O.flip_average(hm, hf, ())
    assert np.array_equal(nump(r["idx"]) if hf is None else O.argmax_planes(avg)[0], O.argmax_planes(avg)[0])


@pytest.mark.parametrize("shape,flip", [((37, 21, 64, 64), True), ((1000, 21, 64, 64), True), ((9, 16, 56, 56), False),
                                        ((3, 4, 128, 128), True), ((2, 3, 21, 64, 64), False)])
def test_one_launch_step_equals_three_launches(ops, L, shape, flip):
    """lhn_fused_render_loss_decode (kernel-side fixed-order reduction + finalisation) against
    lhn_decode_heatmap -> lhn_loss_reduce -> lhn_loss_finalize; also the CTA-per-plane fallback shape
    (128x128 f32 with flip), a stacked [N,S,K,H,W] shape, determinism and the self-resetting workspace."""
    stacked = len(shape) == 5
    N, K, H, W = (shape[0], shape[2], shape[3], shape[4]) if stacked else shape
    S = shape[1] if stacked else 1
    hm, cen = synth.blob_heatmaps(N, S * K, H, W, seed=41, zero_frac=0.03, tie_frac=0.03)
    hf = synth.flipped_blob_heatmaps(cen, H, W, seed=42) if flip else None
    center, scale = synth.bbox_center_scale(N, seed=43)
    j, v = synth.hand_joints(N, K, (4 * W, 4 * H), seed=44, outside_frac=0.05, vis_prob=0.9)
    sig = [2.0, 3.0, 2.5][:S] if stacked else 2
    render = dict(loss_mode=L.LOSS_DISTANCE_BALANCE, image_size=(4 * W, 4 * H), sigma=sig, unbiased=True)
    args = (cu(hm.numpy()), L.MASK_NEG1, L.REFINE_DARK, L.XFORM_CENTER_SCALE, cu(center.numpy()), cu(scale.numpy()))
    kw = dict(hm_flip=None if hf is None else cu(hf.numpy()), blur_ksize=11)
    a = ops.decode_heatmap(*args, render=render, joints=cu(j.numpy()), vis=cu(v.numpy()), **kw)
    sums3 = ops.loss_reduce(a["partials"])
    loss3 = ops.loss_finalize(sums3, L.LOSS_DISTANCE_BALANCE, "mean", 0.7)
    ws = torch.zeros(int(L.lib().lhn_fused_workspace_bytes(N, K, S)), dtype=torch.uint8, device=DEV)
    b = ops.fused_render_loss_decode(*args, render, cu(j.numpy()), cu(v.numpy()), loss_scale=0.7, want_partials=True,
                                     workspace=ws, **kw)
    torch.cuda.synchronize()
    for k in ("hm_kpts", "kpts", "idx", "weight", "partials"):
        assert torch.equal(a[k], b[k]), k
    np.testing.assert_allclose(nump(b["sums"]), nump(sums3), rtol=1e-12)
    assert nump(b["sums"])[2] == nump(sums3)[2] and nump(b["sums"])[3] == nump(sums3)[3]      # integer counts
    np.testing.assert_allclose(nump(b["loss"]), nump(loss3), rtol=2e-7)
    assert int(torch.count_nonzero(ws[:256])) == 0, "the ticket must be left at zero"
    c = ops.fused_render_loss_decode(*args, render, cu(j.numpy()), cu(v.numpy()), loss_scale=0.7, workspace=ws, **kw)
    assert torch.equal(b["sums"], c["sums"]) and torch.equal(b["loss"], c["loss"]), "reduction must be reproducible"
    assert "partials" not in c
    # sums only (multi-GPU form): no loss pointer
    d = ops.fused_render_loss_decode(*args, render, cu(j.numpy()), cu(v.numpy()), want_loss=False, workspace=ws, **kw)
    assert torch.equal(d["sums"], b["sums"]) and "loss" not in d


def test_fused_golden_loss(ops, L):
    g = load_golden("render_loss_64.npz")
    hm = np.nan_to_num(load_golden("decode_64.npz")["hm"], nan=0.25, posinf=1.0, neginf=-1.0)
    for unb, tag in ((True, "unbiased"), (False, "int")):
        for mode, key in ((L.LOSS_DISTANCE_BALANCE, f"ref_distance_loss_{tag}_bal"),
                          (L.LOSS_DISTANCE, f"ref_distance_loss_{tag}_nobal"),
                          (L.LOSS_JOINTS_MSE, f"ref_joints_mse_{tag}")):
            r = ops.decode_heatmap(cu(hm), L.MASK_NEG1, L.REFINE_NONE,
                                   render=dict(loss_mode=mode, image_size=(256, 256), sigma=2, unbiased=unb),
                                   joints=cu(g["joints_3d"]), vis=cu(g["joints_3d_visible"]))
            loss = nump(ops.loss_finalize(ops.loss_reduce(r["partials"]), mode))[0]
            assert np.isfinite(g[key])
            np.testing.assert_allclose(loss, g[key], rtol=1e-5)


def test_fused_stacked_sigmas(ops, L):
    """[N,S,K,H,W] hourglass shape with a sigma list (generateTarget.py:252-268)."""
    N, S, K, H, W = 4, 2, 21, 64, 64
    hm, _, _, _ = synth_case(N, S * K, H, W, seed=31)
    hm5 = hm.reshape(N, S, K, H, W)
    j, v = synth.hand_joints(N, K, seed=32)
    tg, tw = O.render_targets(j.numpy(), v.numpy(), (256, 256), (W, H), [2, 3], True)
    want = O.distance_loss_l2(hm5, tg, tw, True)
    r = ops.decode_heatmap(cu(hm5), L.MASK_NEG1, L.REFINE_NONE,
                           render=dict(loss_mode=L.LOSS_DISTANCE_BALANCE, image_size=(256, 256), sigma=[2, 3]),
                           joints=cu(j.numpy()), vis=cu(v.numpy()))
    np.testing.assert_allclose(nump(ops.loss_finalize(ops.loss_reduce(r["partials"]), L.LOSS_DISTANCE_BALANCE))[0],
                               want, rtol=1e-5)


# ---- un-fused loss / render ------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(6, 21, 64, 64), (3, 2, 21, 64, 64), (4, 6, 56, 56), (3, 5, 14, 14)])
def test_loss_against_explicit_target(ops, L, shape):
    rng = np.random.default_rng(41)
    out = rng.uniform(0, 1, shape).astype(np.float32)
    tgt = rng.uniform(0, 1, shape).astype(np.float32) ** 4
    w = (rng.uniform(0, 1, shape[:-2] + (1,)) > 0.2).astype(np.float32)
    for mode, want in ((L.LOSS_DISTANCE_BALANCE, O.distance_loss_l2(out, tgt, w, True)),
                       (L.LOSS_DISTANCE, O.distance_loss_l2(out, tgt, w, False))):
        p = ops.loss_partials(cu(out), cu(tgt), cu(w), mode)
        np.testing.assert_allclose(nump(ops.loss_finalize(ops.loss_reduce(p), mode))[0], want, rtol=1e-5)
    if len(shape) == 4:
        p = ops.loss_partials(cu(out), cu(tgt), cu(w), L.LOSS_JOINTS_MSE)
        np.testing.assert_allclose(nump(ops.loss_finalize(ops.loss_reduce(p), L.LOSS_JOINTS_MSE))[0],
                                   O.joints_distance_loss_mse(out, tgt, w), rtol=1e-5)


@pytest.mark.parametrize("case", ["render_loss_64.npz", "render_loss_56.npz"])
def test_render_golden(ops, L, case):
    g = load_golden(case)
    isz = tuple(int(x) for x in g["image_size"]); hs = tuple(int(x) for x in g["heatmap_size"])
    for unb, tag in ((True, "unbiased"), (False, "int")):
        t, w = ops.render_targets(cu(g["joints_3d"]), cu(g["joints_3d_visible"]), isz, hs, 2, unb)
        assert np.array_equal(nump(w), g[f"ref_weight_{tag}"]), "target_weight must match exactly"
        np.testing.assert_allclose(nump(t), g[f"ref_target_{tag}"], rtol=1e-5, atol=1e-7)
    sx, sy = ops.render_simdr(cu(g["joints_3d"]), cu(g["joints_3d_visible"]), isz, 2, 2)
    np.testing.assert_allclose(nump(sx)[:, 0], g["ref_simdr_x_row0"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(nump(sy)[:, 0], g["ref_simdr_y_row0"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(nump(sx).sum(-1), g["ref_simdr_x_sum"], rtol=1e-5)


def test_render_multi_sigma_and_edges(ops, L):
    j, v = synth.hand_joints(32, 21, seed=51, outside_frac=0.3, vis_prob=0.7)
    for unb in (True, False):
        want_t, want_w = O.render_targets(j.numpy(), v.numpy(), (256, 256), (64, 64), [2, 3, 4], unb)
        t, w = ops.render_targets(cu(j.numpy()), cu(v.numpy()), (256, 256), (64, 64), [2, 3, 4], unb)
        assert np.array_equal(nump(w), want_w)
        np.testing.assert_allclose(nump(t), want_t, rtol=1e-5, atol=1e-7)


# ---- SimDR -----------------------------------------------------------------------------------------
def test_udp_render_loss_and_backward(ops, L):
    """UDP encoding (SURVEY §8f rank 3, render side): lhn_render_targets, the fused loss on UDP targets and its
    backward against the executed reference (tests/golden/render_udp.npz) and the oracle."""
    g = load_golden("render_udp.npz")
    isz, hsz = tuple(int(v) for v in g["image_size"]), tuple(int(v) for v in g["heatmap_size"])
    j, v = cu(g["joints_3d"]), cu(g["joints_3d_visible"])
    for sg, tag in ((2, "s2"), (1.5, "s15"), ([2, 3], "list")):
        t, w = ops.render_targets(j, v, isz, hsz, sg, "udp")
        assert np.array_equal(nump(w), g[f"ref_weight_{tag}"])
        assert np.abs(nump(t) - g[f"ref_target_{tag}"]).max() <= 1.2e-7
    # non-integer 3*sigma in the MSRA integer-centre branch as well (patch centre != rounded joint)
    t, w = ops.render_targets(j, v, isz, hsz, 1.5, False)
    rt, rw = O.render_targets(g["joints_3d"], g["joints_3d_visible"], isz, hsz, 1.5, False)
    assert np.array_equal(nump(w), rw) and np.abs(nump(t) - rt).max() <= 1.2e-7
    for sg, tag, mode in ((2, "s2", "udp"), (1.5, "s15", "udp"), (1.5, None, False)):
        render = dict(loss_mode=L.LOSS_DISTANCE_BALANCE, image_size=isz, sigma=sg, unbiased=mode)
        r = ops.fused_render_loss_decode(cu(g["hm"]), L.MASK_NEG1, L.REFINE_NONE, L.XFORM_NONE, None, None, render, j, v)
        tg, tw = O.render_targets(g["joints_3d"], g["joints_3d_visible"], isz, hsz, sg, mode)
        want = O.distance_loss_l2(g["hm"], tg, tw, True)
        np.testing.assert_allclose(nump(r["loss"])[0], want, rtol=1e-5)
        if tag == "s2":
            np.testing.assert_allclose(nump(r["loss"])[0], g["ref_loss_bal_s2"], rtol=1e-5)
        grad = ops.render_loss_backward(cu(g["hm"]), j, v, render, r["sums"])
        ref = O.distance_loss_l2_grad(g["hm"], tg, tw, True)
        assert np.abs(nump(grad) - ref).max() <= 1e-5 * np.abs(ref).max()


@pytest.mark.parametrize("shape", [(5, 21, 64, 64), (4, 6, 56, 56), (3, 4, 28, 28)])
def test_misaligned_base_pointer_takes_the_non_tma_path(ops, L, shape):
    """A heatmap tensor whose base address is only 4-byte aligned cannot be fetched with TMA bulk copies: the
    kernel stages the plane with plain loads instead.  Same results as the aligned tensor, bit for bit."""
    N, K, H, W = shape
    hm, cen, center, scale = synth_case(N, K, H, W, seed=61)
    hf = synth.flipped_blob_heatmaps(cen, H, W, seed=62).numpy()
    j, v = synth.hand_joints(N, K, (4 * W, 4 * H), seed=63)
    render = dict(loss_mode=L.LOSS_DISTANCE_BALANCE, image_size=(4 * W, 4 * H), sigma=2, unbiased=True)

    def shifted(a):                      # the same values at a base address that is 4 (mod 16)
        buf = torch.empty(a.size + 1, dtype=torch.float32, device=DEV)
        view = buf[1:].view(a.shape)
        view.copy_(cu(a))
        assert view.data_ptr() % 16 == 4
        return view

    args = (L.MASK_NEG1, L.REFINE_DARK, L.XFORM_CENTER_SCALE, cu(center), cu(scale))
    a = ops.decode_heatmap(cu(hm), *args, hm_flip=cu(hf), render=render, joints=cu(j.numpy()), vis=cu(v.numpy()))
    b = ops.decode_heatmap(shifted(hm), *args, hm_flip=shifted(hf), render=render, joints=cu(j.numpy()), vis=cu(v.numpy()))
    for k in ("hm_kpts", "kpts", "idx", "weight", "partials"):
        assert torch.equal(a[k], b[k]), k


def test_simdr_decode_and_loss(ops, L):
    g = load_golden("render_loss_64.npz")
    xv, yv = g["simdr_xv"], g["simdr_yv"]
    r, idx = ops.decode_simdr(cu(xv), cu(yv), 2, cu(g["center"]), cu(g["scale"]), want_idx=True)
    assert np.array_equal(nump(r), g["ref_simdr_decode"]), "SimDR decode is exact arithmetic"
    assert np.array_equal(nump(idx)[..., 0], xv.argmax(-1)) and np.array_equal(nump(idx)[..., 1], yv.argmax(-1))
    sx, sy = O.render_simdr_batch(g["joints_3d"], g["joints_3d_visible"], (256, 256), 2, 2)
    loss = nump(ops.simdr_smoothl1(cu(xv), cu(yv), cu(sx), cu(sy), cu(g["ref_weight_unbiased"])))[0]
    np.testing.assert_allclose(loss, g["ref_kld_loss"], rtol=1e-5)


@pytest.mark.parametrize("B,K,Lx,Ly", [(64, 21, 512, 512), (5, 16, 448, 448), (3, 4, 100, 36)])
def test_simdr_vs_oracle(ops, L, B, K, Lx, Ly):
    xv, _ = synth.simdr_vectors(B, K, Lx, seed=61)
    _, yv = synth.simdr_vectors(B, K, Ly, seed=62)
    xv, yv = xv.numpy(), yv.numpy()
    xv[0, 0, 7] = np.nan; yv[0, 0] = 0.0; xv[1, 1, 3] = xv[1, 1].max(); xv[1, 1, 9] = xv[1, 1, 3]
    center, scale = [t.numpy() for t in synth.bbox_center_scale(B, seed=63)]
    want = O.keypoints_from_simdr(xv, yv, center, scale, 2)
    got = nump(ops.decode_simdr(cu(xv), cu(yv), 2, cu(center), cu(scale)))
    assert np.array_equal(got, want, equal_nan=True)
    # vector_nms + bbox-masked argmax (result_parser.py:61-129)
    rng = np.random.default_rng(64)
    x1 = rng.integers(0, Lx // 2, B); x2 = x1 + rng.integers(1, Lx // 2, B)
    y1 = rng.integers(0, Ly // 2, B); y2 = y1 + rng.integers(1, Ly // 2, B)
    ranges = np.stack([x1, x2, y1, y2], 1).astype(np.int32)
    xv = np.nan_to_num(xv)
    want = O.coordinates_from_vectors(xv, yv, ranges, 2)
    got = nump(ops.decode_simdr(cu(xv), cu(yv), 2, nms=True, ranges=cu(ranges)))
    assert np.array_equal(got, want)


@pytest.mark.parametrize("B,K,Lx,Ly,dtype", [(512, 21, 512, 512, "f32"), (700, 16, 448, 448, "f32"), (600, 21, 256, 512, "f32"),
                                             (1024, 21, 512, 512, "bf16"), (1030, 21, 64, 32, "f16")])
def test_simdr_ring_kernel_vs_oracle(ops, L, B, K, Lx, Ly, dtype, monkeypatch):
    """Batches large enough for the persistent TMA-ring kernel (>= 148 * 16 * 4 pairs): exact equality with the
    oracle incl. NaN / all-zero / tied / -inf vectors and a ragged pair count, and with the grid-stride kernel
    (LHN_SIMDR_RING=0) on the same inputs."""
    assert B * K >= 148 * 16 * 4
    xv, _ = synth.simdr_vectors(B, K, Lx, seed=71)
    _, yv = synth.simdr_vectors(B, K, Ly, seed=72)
    td = dict(f32=torch.float32, bf16=torch.bfloat16, f16=torch.float16)[dtype]
    xv, yv = xv.to(td).float().numpy(), yv.to(td).float().numpy()      # values exactly representable in `dtype`
    xv[0, 0, 7] = np.nan; yv[0, 0] = 0.0
    xv[1, 1, 3] = xv[1, 1].max(); xv[1, 1, 9] = xv[1, 1, 3]
    yv[2, 2] = -np.inf
    xv[-1, -1, Lx - 1] = 9.0; yv[-1, -1, 0] = 9.0; yv[-1, -1, Ly - 1] = 9.0
    xv[3, 0, 5] = np.nan; xv[3, 0, 2] = np.nan
    xv[4, 0] = -0.0; xv[4, 0, 17] = 0.0
    center, scale = [t.numpy() for t in synth.bbox_center_scale(B, seed=73)]
    with np.errstate(all="ignore"):
        want = O.keypoints_from_simdr(xv, yv, center, scale, 2)
    xt, yt = cu(xv).to(td), cu(yv).to(td)
    got, idx = ops.decode_simdr(xt, yt, 2, cu(center), cu(scale), want_idx=True)
    assert np.array_equal(nump(got), want, equal_nan=True)
    assert np.array_equal(nump(idx)[..., 0], np.argmax(xv, -1)) and np.array_equal(nump(idx)[..., 1], np.argmax(yv, -1))
    monkeypatch.setenv("LHN_SIMDR_RING", "0")
    got0, idx0 = ops.decode_simdr(xt, yt, 2, cu(center), cu(scale), want_idx=True)
    monkeypatch.delenv("LHN_SIMDR_RING")
    assert torch.equal(idx, idx0) and np.array_equal(nump(got), nump(got0), equal_nan=True)
    # lhn_decode_simdr_flags: back-to-back launches on disjoint outputs that may overlap (LHN_FLAG_OVERLAP_PREVIOUS)
    outs = [ops.decode_simdr(xt, yt, 2, cu(center), cu(scale), want_idx=True, overlap_previous=True) for _ in range(4)]
    for g_, i_ in outs:
        assert torch.equal(i_, idx) and np.array_equal(nump(g_), nump(got), equal_nan=True)
    # no transform
    got2 = ops.decode_simdr(xt, yt, 2)
    with np.errstate(all="ignore"):
        want2 = np.concatenate([np.stack([np.argmax(xv, -1), np.argmax(yv, -1)], -1).astype(np.float32) / 2,
                                ((xv.max(-1) + yv.max(-1)) / 2)[..., None]], -1)
    want2[..., 2] = want[..., 2]
    assert np.array_equal(nump(got2), want2.astype(np.float32), equal_nan=True)


# ---- metrics ---------------------------------------------------------------------------------------
def _counters_to_pck(cnt, T, K):
    cnt = cnt.reshape(T + 2, K)
    return cnt[:T], cnt[T], cnt[T + 1]


def test_pck_counters_golden(ops, L):
    g = load_golden("metrics_16.npz")
    K = g["preds"].shape[1]
    p64 = g["preds"].astype(np.float64)
    t = g["bbox_wh"].max(1).astype(np.float64)
    nor = np.stack([t, t], 1)
    cnt = nump(ops.pck_accumulate(cu(p64), cu(g["gt"]), cu(g["mask"]), [0.2], normalize=cu(nor)))
    hits, valid, _ = _counters_to_pck(cnt, 1, K)
    acc, avg, n = O.pck_from_counters(hits[0], valid)
    assert np.array_equal(acc, g["ref_pck_acc"]) and avg == g["ref_pck_avg"] and n == g["ref_pck_cnt"]
    # AUC: 20 thresholds, constant normaliser 30 (python float -> f64 arithmetic)
    thr = [1.0 * i / 20 for i in range(20)]
    cnt = nump(ops.pck_accumulate(cu(p64), cu(g["gt"]), cu(g["mask"]), thr, norm_const=30.0))
    hits, valid, _ = _counters_to_pck(cnt, 20, K)
    auc = sum(1.0 / 20 * O.pck_from_counters(hits[i], valid)[1] for i in range(20))
    assert auc == g["ref_auc"]
    # EPE: constant normaliser 1 given as an f32 array of ones in the reference
    ones = np.ones((len(p64), 2), np.float32)
    cnt = nump(ops.pck_accumulate(cu(p64), cu(g["gt"]), cu(g["mask"]), [], normalize=cu(ones)))
    _, valid, fix = _counters_to_pck(cnt, 0, K)
    np.testing.assert_allclose(fix.sum() / 1048576.0 / max(1, valid.sum()), g["ref_epe"], rtol=1e-5)
    # all-f32 promotion
    cnt = nump(ops.pck_accumulate(cu(g["preds"]), cu(g["gt"]), cu(g["mask"]), [0.2], normalize=cu(nor.astype(np.float32))))
    hits, valid, _ = _counters_to_pck(cnt, 1, K)
    acc, avg, _ = O.pck_from_counters(hits[0], valid)
    assert np.array_equal(acc, g["ref_pck_f32_acc"]) and avg == g["ref_pck_f32_avg"]


def test_pck_counters_sharded_equal_monolithic(ops, L):
    """Eight even shards of 4096 x 16, and uneven shards of 21-joint samples past the capped grid (8 * SMs blocks of
    256 threads), one shard past it by itself, with the cap not a multiple of 21: the grid stride must still visit
    every element once."""
    cap = 8 * torch.cuda.get_device_properties(0).multi_processor_count * 256
    S = cap // 21
    assert cap % 21 and (S + 3) * 21 > cap
    for N, K, bounds in ((4096, 16, [int(s[0]) for s in np.array_split(np.arange(4096), 8)] + [4096]),
                         (2 * S + 5, 21, [0, 7, S + 10, 2 * S + 4, 2 * S + 5])):
        rng = np.random.default_rng(72)
        pred = rng.uniform(0, 256, (N, K, 2)).astype(np.float32)
        gt = (pred + rng.normal(0, 12, (N, K, 2))).astype(np.float32)
        mask = rng.uniform(0, 1, (N, K)) < 0.9
        nor = np.repeat(rng.uniform(60, 200, (N, 1)), 2, 1)
        thr = [0.05, 0.1, 0.2, 0.5]
        mono = nump(ops.pck_accumulate(cu(pred.astype(np.float64)), cu(gt), cu(mask), thr, normalize=cu(nor)))
        sharded = torch.zeros((len(thr) + 2) * K, dtype=torch.int64, device=DEV)
        for a, b in zip(bounds[:-1], bounds[1:]):
            ops.pck_accumulate(cu(pred[a:b].astype(np.float64)), cu(gt[a:b]), cu(mask[a:b]), thr,
                               normalize=cu(nor[a:b]), counters=sharded)
        assert np.array_equal(mono, nump(sharded)), (N, K)
        hits, valid = O.pck_counters(pred.astype(np.float64), gt, mask, thr, nor)
        assert np.array_equal(mono.reshape(len(thr) + 2, K)[:len(thr)], hits), (N, K)
        assert np.array_equal(mono.reshape(len(thr) + 2, K)[len(thr)], valid), (N, K)


def test_fused_decode_pck_counters(ops, L):
    """BASELINE config 4 path: decode + PCK@0.2 / AUC / EPE counters in one kernel."""
    N, K, H, W = 64, 16, 64, 64
    hm, cen = synth.blob_heatmaps(N, K, H, W, seed=81)
    center, scale = synth.bbox_center_scale(N, fixed=True)
    gt, mask, wh = synth.pck_inputs(cen, seed=82)
    mask[3] = False; wh[5] = 0.0
    cnt = torch.zeros((20 + 5) * K, dtype=torch.int64, device=DEV)
    r = ops.decode_heatmap_pck(cu(hm.numpy()), L.MASK_NEG1, L.REFINE_SIGN, center.to(DEV), scale.to(DEV),
                               gt.to(DEV), mask.to(DEV), wh.to(DEV), cnt)
    _, preds, _ = O.keypoints_from_heatmaps(hm.numpy(), center.numpy(), scale.numpy(), "default")
    assert np.array_equal(nump(r["kpts"])[..., :2], preds)
    c = nump(cnt).reshape(25, K)
    info = dict(O.report_metric(preds.astype(np.float64), gt.numpy(), mask.numpy(),
                                bbox_wh=wh.numpy().astype(np.float64)))
    acc, pck, _ = O.pck_from_counters(c[0], c[1])
    assert pck == info["PCK"], "PCK hit counts must be bit-exact"
    auc = sum(1.0 / 20 * O.pck_from_counters(c[2 + i], c[22])[1] for i in range(20))
    assert auc == info["AUC"]
    np.testing.assert_allclose(c[24].sum() / 1048576.0 / max(1, c[23].sum()), info["EPE"], rtol=1e-5)


def test_evaluate_pck_golden(ops, L):
    g = load_golden("metrics_16.npz")
    bbox_wh = g["pck_bbox"][:, 0, 2:]
    pck, mean = ops.evaluate_pck(cu(g["pck_pred_hm"]), cu(g["pck_gt_hm"]), cu(bbox_wh), cu(g["pck_tw"]), (256, 256), 0.2)
    np.testing.assert_allclose(nump(mean)[0], g["ref_evaluate_pck_w"], rtol=1e-6, equal_nan=True)
    pck, mean = ops.evaluate_pck(cu(g["pck_pred_hm"]), cu(g["pck_gt_hm"]), cu(bbox_wh), None, (256, 256), 0.02)
    np.testing.assert_allclose(nump(mean)[0], g["ref_evaluate_pck_now"], rtol=1e-6, equal_nan=True)


# ---- low-precision inputs: oracle = reference arithmetic on the upcast f32 tensor -------------------
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
def test_low_precision_inputs(ops, L, dt):
    N, K, H, W = 6, 21, 64, 64
    hm, cen, center, scale = synth_case(N, K, H, W, seed=91)
    t = cu(hm).to(dt)
    up = nump(t.float())
    hf = cu(synth.flipped_blob_heatmaps(cen, H, W, seed=92).numpy()).to(dt)
    with np.errstate(all="ignore"):
        r = ops.decode_heatmap(t, L.MASK_NEG1, L.REFINE_DARK, L.XFORM_CENTER_SCALE, cu(center), cu(scale))
        assert np.array_equal(nump(r["idx"]), O.argmax_planes(up)[0]), "bf16/f16 ties: first index"
        hp, p, mv = O.keypoints_from_heatmaps(up, center, scale, "unbiased", 11)
        assert_coords_close(nump(r["kpts"])[..., :2], p, what="lowp dark")
        avg = O.flip_average(up, nump(hf.float()), ())
        r = ops.decode_heatmap(t, L.MASK_NEG1, L.REFINE_SIGN, L.XFORM_CENTER_SCALE, cu(center), cu(scale), hm_flip=hf)
        assert np.array_equal(nump(r["idx"]), O.argmax_planes(avg)[0])
        hp, p, mv = O.keypoints_from_heatmaps(avg, center, scale, "default")
        assert np.array_equal(nump(r["kpts"])[..., :2], p)
    j, v = synth.hand_joints(N, K, seed=93)
    tg, tw = O.render_targets(j.numpy(), v.numpy(), (256, 256), (W, H), 2, True)
    r = ops.decode_heatmap(t, L.MASK_NEG1, L.REFINE_NONE, hm_flip=hf,
                           render=dict(loss_mode=L.LOSS_DISTANCE_BALANCE, image_size=(256, 256), sigma=2),
                           joints=cu(j.numpy()), vis=cu(v.numpy()))
    np.testing.assert_allclose(nump(ops.loss_finalize(ops.loss_reduce(r["partials"]), L.LOSS_DISTANCE_BALANCE))[0],
                               O.distance_loss_l2(up, tg, tw, True), rtol=1e-5)


# ---- error behaviour: loud, never a fallback -------------------------------------------------------
def test_rejects_cpu_tensors_and_bad_args(ops, L):
    with pytest.raises(L.LhnError):
        ops.decode_heatmap(torch.zeros(1, 1, 64, 64), L.MASK_NONE, L.REFINE_NONE)
    with pytest.raises(L.LhnError):
        ops.decode_heatmap(torch.zeros(1, 1, 64, 64, device=DEV), L.MASK_NONE, L.REFINE_NONE, L.XFORM_CENTER_SCALE)
    with pytest.raises(L.LhnError):
        ops.decode_heatmap(torch.zeros(1, 1, 64, 64, device=DEV, dtype=torch.float64), L.MASK_NONE, L.REFINE_NONE)
    r = ops.decode_heatmap(torch.zeros(0, 21, 64, 64, device=DEV), L.MASK_NONE, L.REFINE_NONE)
    assert r["idx"].shape == (0, 21)
