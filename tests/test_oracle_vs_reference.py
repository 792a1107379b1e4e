"""CPU, only where the original project's source tree is present (LHN_REFERENCE_ROOT, or the copy staged in
oracle/_ref): the numpy oracle against the EXECUTED, unmodified reference on fresh seeds.  Skipped without it;
tests/test_oracle_golden.py checks the oracle against the reference's stored outputs everywhere."""
import numpy as np
import pytest
import torch

from oracle import np_oracle as O
from oracle import ref_loader
from litehandnet_b200 import synth
from conftest import assert_coords_close

pytestmark = pytest.mark.skipif(not ref_loader.available(),
                                reason="the original project's sources are not present (set LHN_REFERENCE_ROOT)")


@pytest.fixture(scope="module")
def ref():
    return ref_loader.load()


def _hm(N, K, H, W, seed):
    hm, cen = synth.blob_heatmaps(N, K, H, W, seed=seed, zero_frac=0.1, tie_frac=0.1)
    return hm.numpy(), cen


@pytest.mark.parametrize("shape,seed", [((4, 21, 64, 64), 101), ((3, 21, 56, 56), 102), ((3, 16, 64, 64), 103)])
@pytest.mark.parametrize("pp", ["default", "unbiased"])
def test_keypoints_from_heatmaps_live(ref, shape, seed, pp):
    N, K, H, W = shape
    hm, _ = _hm(N, K, H, W, seed)
    c, s = synth.bbox_center_scale(N, seed=seed + 1)
    c, s = c.numpy(), s.numpy()
    with np.errstate(all="ignore"):
        r_hp, r_p, r_mv = ref.top_down_eval.keypoints_from_heatmaps(hm.copy(), c, s, post_process=pp, kernel=11)
        hp, p, mv = O.keypoints_from_heatmaps(hm, c, s, pp, 11)
    assert np.array_equal(mv, r_mv, equal_nan=True)
    if pp == "default":
        assert np.array_equal(hp, r_hp) and np.array_equal(p, r_p)
    else:
        assert_coords_close(hp, r_hp, what="hm_preds")
        assert_coords_close(p, r_p, what="preds")


@pytest.mark.parametrize("seed", [111, 112])
def test_argmax_and_legacy_live(ref, seed):
    hm, _ = _hm(4, 21, 64, 64, seed)
    t = torch.from_numpy(hm)
    r_p, r_mv = ref.evaluation.get_coordinates_from_heatmap(t)
    p, mv, idx = O.max_preds(hm, "zero")
    assert np.array_equal(p, r_p.numpy()) and np.array_equal(mv, r_mv.numpy(), equal_nan=True)
    assert np.array_equal(idx, hm.reshape(4, 21, -1).argmax(-1))
    rp = ref_loader.make_result_parser(ref, dark=False)
    k = rp.get_pred_kpt(t.clone(), resized=True)
    assert np.array_equal(O.get_pred_kpt(hm, dark=False, resized=True, feature_stride=(4, 4)), np.asarray(k))
    rpd = ref_loader.make_result_parser(ref, dark=True)
    with np.errstate(all="ignore"):
        kd = rpd.get_pred_kpt(t.clone(), resized=False)
        assert_coords_close(O.get_pred_kpt(hm, dark=True, resized=False, feature_stride=(4, 4)), np.asarray(kd),
                            what="legacy dark")


@pytest.mark.parametrize("unbiased", [True, False])
def test_render_and_balanced_loss_live(ref, unbiased):
    K, H, W = 21, 64, 64
    joints, vis = synth.hand_joints(6, K, (256, 256), seed=120)
    joints, vis = joints.numpy(), vis.numpy()
    gen = ref.generateTarget.TopDownGenerateTarget(sigma=2, unbiased_encoding=unbiased)
    tg, tw = [], []
    for b in range(6):
        res = dict(joints_3d=joints[b].copy(), joints_3d_visible=vis[b].copy(),
                   ann_info=dict(num_joints=K, image_size=np.array([256, 256]), heatmap_size=np.array([W, H]),
                                 joint_weights=None, use_different_joint_weights=False))
        out = gen(res)
        tg.append(out["target"]); tw.append(out["target_weight"])
    tg, tw = np.stack(tg), np.stack(tw)
    o_tg, o_tw = O.render_targets(joints, vis, (256, 256), (W, H), 2, unbiased)
    assert np.array_equal(o_tw, tw)
    assert np.abs(o_tg - tg).max() <= 1.2e-7                      # 1 ulp of f32 (NumPy-version dependent)
    hm, _ = _hm(6, K, H, W, 121)
    crit = ref.loss.heatmapLoss.DistanceLoss(loss_type="L2", balance=True) if hasattr(ref.loss, "heatmapLoss") \
        else ref.loss.DistanceLoss(loss_type="L2", balance=True)
    r = float(crit(torch.from_numpy(hm), torch.from_numpy(tg), torch.from_numpy(tw)))
    o = float(O.distance_loss_l2(hm, o_tg, o_tw, balance=True))
    assert abs(o - r) <= 1e-5 * abs(r)


def test_metrics_live(ref):
    rng = np.random.default_rng(130)
    N, K = 64, 16
    gt = rng.uniform(0, 256, (N, K, 2)).astype(np.float32)
    pred = (gt + rng.normal(0, 8, gt.shape)).astype(np.float64)
    mask = rng.random((N, K)) < 0.9
    norm = np.tile(rng.uniform(60, 200, (N, 1)).astype(np.float32), (1, 2))
    T = ref.top_down_eval
    r_acc, r_avg, r_cnt = T.keypoint_pck_accuracy(pred, gt, mask, 0.2, norm.copy())
    acc, avg, cnt = O.keypoint_pck_accuracy(pred, gt, mask, 0.2, norm.copy())
    assert np.array_equal(acc, r_acc) and avg == r_avg and cnt == r_cnt
    assert O.keypoint_auc(pred, gt, mask, 30) == T.keypoint_auc(pred, gt, mask, 30)
    assert O.keypoint_epe(pred, gt, mask) == T.keypoint_epe(pred, gt, mask)


def test_simdr_live(ref):
    xv, yv = synth.simdr_vectors(8, 21, 512, seed=140)
    c, s = synth.bbox_center_scale(8, seed=141)
    r = ref.top_down_eval.keypoints_from_simdr(xv.numpy(), yv.numpy(), c.numpy(), s.numpy(), k=2)
    o = O.keypoints_from_simdr(xv.numpy(), yv.numpy(), c.numpy(), s.numpy(), 2)
    assert np.array_equal(o, r)


def test_get_final_preds_anisotropic_live(ref):
    """utils/transforms.py:18-44 with the cv2-affine transform_preds: only scale[0] enters (SURVEY §8a T3)."""
    for shape, seed in (((3, 16, 64, 64), 150), ((2, 16, 64, 48), 151)):
        hm, _ = _hm(*shape, seed)
        rng = np.random.default_rng(seed)
        c = rng.uniform(60, 200, (shape[0], 2)).astype(np.float32)
        s = np.stack([rng.uniform(0.6, 1.6, shape[0]), rng.uniform(0.6, 1.6, shape[0])], 1).astype(np.float32)
        r = ref.transforms.get_final_preds(torch.from_numpy(hm.copy()), c, s)
        o = O.get_final_preds(hm, c, s)
        assert_coords_close(o, r, rtol=1e-5, atol=1e-4, what="final_preds (anisotropic scale)")


def test_anisotropic_scales_live(ref):
    """transform_preds (post_transforms.py:6-48) uses both scale components; the synthetic boxes elsewhere are
    square, so pin the anisotropic case for the Gen-2 heatmap / SimDR / UDP decoders here."""
    rng = np.random.default_rng(160)
    N = 4
    hm, _ = _hm(N, 21, 64, 48, 161)
    c = rng.uniform(60, 200, (N, 2)).astype(np.float32)
    s = np.stack([rng.uniform(0.6, 1.6, N), rng.uniform(0.6, 1.6, N)], 1).astype(np.float32)
    T = ref.top_down_eval
    with np.errstate(all="ignore"):
        for pp in ("default", "unbiased"):
            r = T.keypoints_from_heatmaps(hm.copy(), c, s, post_process=pp, kernel=11)
            o = O.keypoints_from_heatmaps(hm, c, s, pp, 11)
            assert_coords_close(o[1], r[1], what=f"preds {pp}")
        r = T.keypoints_from_heatmaps(hm.copy(), c, s, kernel=11, use_udp=True)
        o = O.keypoints_from_heatmaps_udp(hm, c, s, 11)
        assert np.array_equal(o[0], r[0], equal_nan=True) and np.array_equal(o[1], r[1], equal_nan=True)
    xv, yv = synth.simdr_vectors(N, 21, 448, seed=162)
    assert np.array_equal(O.keypoints_from_simdr(xv.numpy(), yv.numpy(), c, s, 2),
                          T.keypoints_from_simdr(xv.numpy(), yv.numpy(), c, s, k=2))


def test_region_bbox_decode_live(ref):
    """SURVEY §8f rank 4, live: the oracle against the executed bbox branch of HeatmapParser_SH, ResultParser (DARK)
    and utils/evaluation.py on freshly seeded region maps (other seeds than the golden fixture)."""
    import torch
    from oracle import make_golden as M
    from conftest import canon_candidates
    for seed in (5, 6):
        c, s = M.region_maps(4, seed)
        SH = ref.SPheatmapParser.HeatmapParser_SH()
        cn = SH.heatmap_nms(c.clone())
        on = O.heatmap_nms(c.numpy())
        assert np.array_equal(cn.numpy(), on)
        cand = SH.candidate_bbox(cn.clone(), s.clone(), (256, 256))
        oc = O.candidate_bbox(on, s.numpy(), "sh", (256, 256))
        (a, da), (b, db) = canon_candidates(oc), canon_candidates(cand.numpy())
        assert np.array_equal(da, db) and np.array_equal(a[da], b[db])
        SH.max_num_bbox = 10
        for thr in (0.6, 0.2):
            SH.iou_threshold = thr
            assert SH.non_max_suppression(cand) == O.box_nms(cand.numpy(), 0.1, thr, 10)
        RP = ref_loader.make_result_parser(ref, dark=True)
        RP.num_candidates = 1
        s40 = s * 40
        c1 = RP.candidate_bbox(RP.heatmap_nms(c.clone()), s40.clone())
        with np.errstate(all="ignore"):
            o1 = O.candidate_bbox(on, s40.numpy(), "rp", num_candidates=1)
        assert_coords_close(o1, c1.numpy(), what="rp cand1")
        ev = ref.evaluation
        cc = ev.cs_from_region_map(torch.cat([c, s40], 1), 256, 20, 0.1)
        oc2 = O.candidate_bbox(c.numpy(), s40.numpy(), "cs", (256, 256), num_candidates=20, thr=0.1)
        (a, da), (b, db) = canon_candidates(oc2), canon_candidates(cc.numpy())
        assert np.array_equal(da, db)
        assert_coords_close(a[da], b[db], what="cs cand")
        hm = torch.rand(4, 5, 64, 64, generator=torch.Generator().manual_seed(seed))
        for dark, P in ((False, ref_loader.make_result_parser(ref, dark=False)), (True, RP)):
            for j, bb in enumerate(M.FIRST_RESULT_BOXES):
                r = P._get_first_result(list(bb), hm.clone(), j % 4)
                with np.errstate(all="ignore"):
                    o = O.get_first_result(list(bb), hm.numpy(), j % 4, dark=dark)
                assert_coords_close(o, r.numpy(), what=f"first_result dark={dark} box {j}")
