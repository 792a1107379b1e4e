"""Generate tests/golden/*.npz by EXECUTING the unmodified reference (test infrastructure).

Run here (the container that has /root/reference):  python -m oracle.make_golden
The fixtures travel to the GPU box; the reference does not.  Every array named ``ref_*`` is an
output of a reference function; the rest are the seeded inputs it was run on.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_loader  # noqa: E402
from oracle import np_oracle as O  # noqa: E402  (only to place the synthetic blobs inside the decoded windows)
from litehandnet_b200 import synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def _ann(K, image_size, heatmap_size):
    return dict(num_joints=K, image_size=np.array(image_size), heatmap_size=np.array(heatmap_size),
                joint_weights=None, use_different_joint_weights=False)


def decode_case(ref, name, N, K, H, W, seed, image_size):
    T = ref.top_down_eval
    hm, cen = synth.blob_heatmaps(N, K, H, W, seed=seed, zero_frac=0.08, tie_frac=0.08)
    # hand-made edge planes: negative-only plane, NaN plane, border maxima, flat plateau
    hm[0, 0] = -hm[0, 0].abs() - 0.1
    hm[0, 1, 5, 7] = float("nan")
    hm[0, 2] = 0.0; hm[0, 2, 0, 0] = 1.0
    hm[0, 3] = 0.0; hm[0, 3, H - 1, W - 1] = 1.0
    hm[0, 4] = 0.0; hm[0, 4, 10:13, 20:23] = 0.7
    n1 = N - 1
    hm[n1, 5] = 0.0; hm[n1, 5, 2, 2] = 0.9; hm[n1, 5, 2, 3] = 0.5; hm[n1, 5, 3, 2] = 0.4
    hm[n1, 4 if N > 1 else 6] = 0.0; hm[n1, 4 if N > 1 else 6, 1, W - 2] = 0.9
    hmn = hm.numpy()
    center, scale = [t.numpy() for t in synth.bbox_center_scale(N, seed=seed + 1)]
    d = dict(hm=hmn, center=center, scale=scale, image_size=np.array(image_size))
    with np.errstate(all="ignore"):
        for pp, tag in (("default", "default"), ("unbiased", "unbiased"), (None, "none")):
            a = T.keypoints_from_heatmaps(hmn.copy(), center, scale, post_process=pp, kernel=11)
            d[f"ref_g2_{tag}_hm_preds"], d[f"ref_g2_{tag}_preds"], d[f"ref_g2_{tag}_maxvals"] = a
        d["ref_argmax_idx"] = np.argmax(hmn.reshape(N, K, -1), 2)
        a = ref.evaluation.get_coordinates_from_heatmap(torch.from_numpy(hmn.copy()))
        d["ref_a1_preds"], d["ref_a1_maxvals"] = a[0].numpy(), a[1].numpy()
        a = ref.transforms.get_max_preds(hmn.copy())
        d["ref_a3_preds"], d["ref_a3_maxvals"] = a
        stride = (image_size[0] // W, image_size[1] // H)
        for dark in (False, True):
            rp = ref_loader.make_result_parser(ref, image_size=image_size, hm_size=(W, H), dark=dark)
            for resized in (False, True):
                k = rp.get_pred_kpt(torch.from_numpy(hmn.copy()), resized=resized)
                d[f"ref_legacy_{'dark' if dark else 'offset'}_{'img' if resized else 'hm'}"] = \
                    np.asarray(k, dtype=np.float32)
        k, bb = ref.SPheatmapParser.HeatmapParser_SH().parse(torch.from_numpy(hmn.copy()),
                                                            image_size=image_size)
        assert bb is None
        d["ref_parse_sh"] = k.numpy()
        d["ref_final_preds"] = ref.transforms.get_final_preds(torch.from_numpy(hmn.copy()),
                                                              center, scale)
        pairs = synth.MPII_FLIP_PAIRS if K >= 16 else ((0, 1), (2, 3))
        d["flip_pairs"] = np.array(pairs)
        d["ref_flip_back"] = ref.transforms.flip_back(hmn.copy(), pairs)
    np.savez_compressed(os.path.join(OUT, name), **d)
    return hm, cen, center, scale


def render_loss_case(ref, name, N, K, H, W, seed, image_size, hm):
    G = ref.generateTarget.TopDownGenerateTarget
    L = ref.loss
    j, v = synth.hand_joints(N, K, image_size=image_size, seed=seed, outside_frac=0.12, vis_prob=0.8)
    v[0, 0, 0] = 0.3                       # fractional visibility: weight kept, target zero
    jn, vn = j.numpy(), v.numpy()
    # losses are taken on a NaN/inf-free copy of the decode fixture (loss_input = nan_to_num(hm))
    hm = torch.nan_to_num(hm, nan=0.25, posinf=1.0, neginf=-1.0)
    d = dict(joints_3d=jn, joints_3d_visible=vn, image_size=np.array(image_size),
             heatmap_size=np.array([W, H]))
    for unb, tag in ((True, "unbiased"), (False, "int")):
        g = G(sigma=2, unbiased_encoding=unb)
        tg, tw = [], []
        for b in range(N):
            out = g(dict(joints_3d=jn[b], joints_3d_visible=vn[b], ann_info=_ann(K, image_size, (W, H))))
            tg.append(out["target"]); tw.append(out["target_weight"])
        tg, tw = np.stack(tg), np.stack(tw)
        d[f"ref_target_{tag}"] = tg; d[f"ref_weight_{tag}"] = tw
        o = hm.clone()
        for bal in (True, False):
            d[f"ref_distance_loss_{tag}_{'bal' if bal else 'nobal'}"] = np.float32(
                L.DistanceLoss("L2", "mean", bal)(o.clone(), torch.from_numpy(tg), torch.from_numpy(tw)).item())
        d[f"ref_joints_mse_{tag}"] = np.float32(
            L.JointsDistanceLoss()(o.clone(), torch.from_numpy(tg), torch.from_numpy(tw)).item())
    # 5-D hourglass shape [N,S,K,H,W] with a sigma list (generateTarget.py:252-268)
    g = G(sigma=[2, 2], unbiased_encoding=True)
    tg, tw = [], []
    for b in range(N):
        out = g(dict(joints_3d=jn[b], joints_3d_visible=vn[b], ann_info=_ann(K, image_size, (W, H))))
        tg.append(out["target"]); tw.append(out["target_weight"])
    tg, tw = np.stack(tg), np.stack(tw)
    o5 = torch.stack([hm, hm * 0.5], 1)
    d["ref_distance_loss_5d_bal"] = np.float32(
        L.DistanceLoss("L2", "mean", True)(o5.clone(), torch.from_numpy(tg), torch.from_numpy(tw)).item())
    # SimDR render + KLDiscretLoss + decode
    k = 2
    S = ref.generate_simder.GenerateSimDR(sigma=2, k=k)
    sx, sy = [], []
    for b in range(N):
        out = S(dict(joints_3d=jn[b], joints_3d_visible=vn[b], ann_info=dict(image_size=np.array(image_size))))
        sx.append(out["simdr_x"]); sy.append(out["simdr_y"])
    sx, sy = np.stack(sx), np.stack(sy)
    # stored as the argmax/max summary + a few full rows (the full vectors are regenerated by the oracle)
    d["ref_simdr_x_row0"] = sx[:, 0]; d["ref_simdr_y_row0"] = sy[:, 0]
    d["ref_simdr_x_sum"] = sx.sum(-1); d["ref_simdr_y_sum"] = sy.sum(-1)
    xv, yv = synth.simdr_vectors(N, K, sx.shape[-1], seed=seed + 3, k=k)
    d["simdr_xv"], d["simdr_yv"] = xv.numpy(), yv.numpy()
    d["ref_kld_loss"] = np.float32(L.KLDiscretLoss()(
        xv, yv, torch.from_numpy(sx), torch.from_numpy(sy), torch.from_numpy(d["ref_weight_unbiased"])).item())
    center, scale = [t.numpy() for t in synth.bbox_center_scale(N, seed=seed + 1)]
    d["center"], d["scale"] = center, scale
    d["ref_simdr_decode"] = ref.top_down_eval.keypoints_from_simdr(xv.numpy(), yv.numpy(), center, scale, k)
    np.savez_compressed(os.path.join(OUT, name), **d)


def keep_argmax_shrink(hm, bits=16):
    """Heatmaps [..., H, W] f32 with the low `bits` mantissa bits of every value cleared except each plane's maximum,
    which stays exact.  A plane whose maximum is unique keeps its argmax, its maximum and that uniqueness, the only
    things evaluate_pck reads from a heatmap (utils/evaluation.py:62-89); the noise then compresses, which keeps
    the evaluate_pck case of metrics_16.npz under 1 MB."""
    f = np.ascontiguousarray(hm, np.float32).reshape(-1, hm.shape[-2] * hm.shape[-1])
    out = (f.view(np.uint32) & np.uint32((0xFFFFFFFF << bits) & 0xFFFFFFFF)).view(np.float32).copy()
    rows, i = np.arange(len(f)), f.argmax(1)
    out[rows, i] = f[rows, i]
    return out.reshape(hm.shape)


def metrics_case(ref, name, N, K, seed):
    T = ref.top_down_eval
    H = W = 64
    hm, cen = synth.blob_heatmaps(N, K, H, W, seed=seed)
    center, scale = [t.numpy() for t in synth.bbox_center_scale(N, fixed=True)]
    _, preds, _ = T.keypoints_from_heatmaps(hm.numpy().copy(), center, scale, post_process="default")
    gt, mask, wh = synth.pck_inputs(cen, seed=seed + 1)
    mask[3] = False                                   # a sample with no visible joint
    mask[:, 2] = False                                # a joint never visible -> acc = -1
    wh[5] = 0.0                                       # normalize == 0 -> sample masked out
    gtn, m, whn = gt.numpy(), mask.numpy(), wh.numpy()
    pred64 = preds.astype(np.float64)                 # as after the JSON round trip
    t = np.max(whn, axis=1).astype(np.float64)
    thr_bbox = np.stack([t, t], 1)
    d = dict(preds=preds, gt=gtn, mask=m, bbox_wh=whn)
    acc, avg, cnt = T.keypoint_pck_accuracy(pred64, gtn, m, 0.2, thr_bbox.copy())
    d["ref_pck_acc"], d["ref_pck_avg"], d["ref_pck_cnt"] = acc, np.float64(avg), np.int64(cnt)
    head = (t * 0.3)
    acc, avg, cnt = T.keypoint_pck_accuracy(pred64, gtn, m, 0.5, np.stack([head, head], 1))
    d["head_size"] = head
    d["ref_pckh_acc"], d["ref_pckh_avg"] = acc, np.float64(avg)
    d["ref_auc"] = np.float64(T.keypoint_auc(pred64, gtn, m, 30))
    d["ref_epe"] = np.float64(T.keypoint_epe(pred64, gtn, m))
    # all-f32 call (numpy promotion keeps f32 arithmetic)
    acc, avg, cnt = T.keypoint_pck_accuracy(preds, gtn, m, 0.2, thr_bbox.astype(np.float32))
    d["ref_pck_f32_acc"], d["ref_pck_f32_avg"] = acc, np.float64(avg)
    # legacy evaluate_pck on heatmap pairs (small: first 6 samples, first 8 joints)
    n2, k2 = 6, 8
    ghm, _ = synth.blob_heatmaps(n2, k2, H, W, seed=seed + 2,
                                 centers=cen[:n2, :k2] + torch.randn(n2, k2, 2) * 2)
    phm = hm[:n2, :k2].contiguous()
    bbox = torch.cat([torch.full((n2, 1, 2), 128.), torch.rand(n2, 1, 2) * 140 + 60], -1)
    tw = mask[:n2, :k2].float()[..., None]
    tw[0, 0, 0] = 0.5
    phm, ghm = torch.from_numpy(keep_argmax_shrink(phm.numpy())), torch.from_numpy(keep_argmax_shrink(ghm.numpy()))
    d["pck_pred_hm"], d["pck_gt_hm"], d["pck_bbox"], d["pck_tw"] = \
        phm.numpy(), ghm.numpy(), bbox.numpy(), tw.numpy()
    with np.errstate(all="ignore"):
        d["ref_evaluate_pck_w"] = np.float64(ref.evaluation.evaluate_pck(phm, ghm, bbox, 256, tw, 0.2))
        d["ref_evaluate_pck_now"] = np.float64(ref.evaluation.evaluate_pck(phm, ghm, bbox, 256, None, 0.02))
    np.savez_compressed(os.path.join(OUT, name), **d)


def udp_case(ref, name, seed):
    """UDP GaussianHeatmap targets (generateTarget.py:162-243) for two sigmas incl. a non-integer 3*sigma, joints
    outside the image and invisible joints; plus DistanceLoss on them."""
    N, K, H, W = 3, 8, 64, 48
    isz = (192, 256)
    joints, vis = synth.hand_joints(N, K, isz, seed=seed, vis_prob=0.85, outside_frac=0.15)
    d = dict(joints_3d=joints.numpy(), joints_3d_visible=vis.numpy(), image_size=np.array(isz), heatmap_size=np.array([W, H]))
    for sg, tag in ((2, "s2"), (1.5, "s15"), ([2, 3], "list")):
        gen = ref.generateTarget.TopDownGenerateTarget(sigma=sg, encoding="UDP", target_type="GaussianHeatmap")
        tg, tw = [], []
        for b in range(N):
            out = gen(dict(joints_3d=joints[b].numpy().copy(), joints_3d_visible=vis[b].numpy().copy(),
                           ann_info=_ann(K, isz, (W, H))))
            tg.append(out["target"]); tw.append(out["target_weight"])
        d[f"ref_target_{tag}"], d[f"ref_weight_{tag}"] = np.stack(tg), np.stack(tw)
    hm, _ = synth.blob_heatmaps(N, K, H, W, seed=seed + 1)
    d["hm"] = hm.numpy()
    HL = ref.loss.heatmapLoss
    d["ref_loss_bal_s2"] = np.float32(HL.DistanceLoss(loss_type="L2", balance=True)(
        hm, torch.from_numpy(d["ref_target_s2"]), torch.from_numpy(d["ref_weight_s2"])).item())
    np.savez_compressed(os.path.join(OUT, name), **d)


def udp_decode_case(ref, name, seed):
    """keypoints_from_heatmaps(use_udp=True) = _get_max_preds + post_dark_udp + transform_preds(use_udp)
    (top_down_eval.py:274-335, 427-431): blobs + noise, all-zero and negative planes (incl. the first and the last
    plane of the batch: the reference then indexes the previous / the last plane's padding), border maxima, ties."""
    T = ref.top_down_eval
    N, K, H, W = 3, 7, 56, 56
    hm, _ = synth.blob_heatmaps(N, K, H, W, seed=seed, zero_frac=0.1, tie_frac=0.1)
    hm = hm.numpy()
    hm[0, 0] = 0.0                                    # first plane of the batch without a positive maximum
    hm[N - 1, K - 1] = -0.25                          # and the last one
    hm[1, 0] = 0.0; hm[1, 1] = 0.0                    # two degenerate planes in a row
    hm[0, 1] = 0.0; hm[0, 1, 0, 0] = 1.0              # maxima on the corners / edges
    hm[0, 2] = 0.0; hm[0, 2, H - 1, W - 1] = 0.7
    hm[0, 3] = 0.0; hm[0, 3, 0, 20] = 0.5
    hm[0, 4] = 0.0; hm[0, 4, 30, W - 1] = 0.9
    hm[0, 1:5] += np.random.default_rng(seed).random((4, H, W)).astype(np.float32) * 0.01
    center, scale = [t.numpy() for t in synth.bbox_center_scale(N, seed=seed + 1)]
    d = dict(hm=hm, center=center, scale=scale)
    for k in (11, 17):                                # k=17 is the reference's "sigma=3" setting
        with np.errstate(all="ignore"):
            hp, p, mv = T.keypoints_from_heatmaps(hm.copy(), center, scale, post_process="default", kernel=k, use_udp=True)
        d[f"ref_udp_hm_preds_k{k}"], d[f"ref_udp_preds_k{k}"], d["ref_udp_maxvals"] = hp, p, mv
    np.savez_compressed(os.path.join(OUT, name), **d)


def mpii_case(name, seed):
    """MPII PCKh (datasets/datasets/body/topdown_mpii_dataset.py:126-249).  The dataset class cannot be imported
    (xtcocotools, json_tricks) and its mpii_gt_val.mat is not in the tree, so the method's own source is compiled
    from the reference file and executed on a fake `self` with a synthetic gt_dict standing in for loadmat()."""
    import ast
    import textwrap
    from collections import OrderedDict
    path = os.path.join(ref_loader.REF_ROOT, "datasets/datasets/body/topdown_mpii_dataset.py")
    src = open(path).read()
    fn = None
    for node in ast.walk(ast.parse(src)):
        if isinstance(node, ast.FunctionDef) and node.name == "evaluate":
            fn = textwrap.dedent(ast.get_source_segment(src, node))
    rng = np.random.default_rng(seed)
    N, K = 40, 16
    names = np.array([["rank", "rkne", "rhip", "lhip", "lkne", "lank", "pelv", "thor", "neck", "head", "rwri", "relb", "rsho",
                       "lsho", "lelb", "lwri"]], dtype=object)
    pos_gt = rng.uniform(20, 400, (K, 2, N))
    head = np.zeros((2, 2, N)); head[0] = rng.uniform(50, 200, (2, N)); head[1] = head[0] + rng.uniform(15, 60, (2, N))
    missing = (rng.random((K, N)) < 0.15).astype(np.float64)
    gt_dict = dict(dataset_joints=names, jnt_missing=missing, pos_gt_src=pos_gt, headboxes_src=head)
    preds = (np.transpose(pos_gt, (2, 0, 1)) - 1.0 + rng.normal(0, 8, (N, K, 2))).astype(np.float32)
    preds = np.concatenate([preds, rng.random((N, K, 1)).astype(np.float32)], axis=2)
    ids = list(rng.permutation(N)) + [3, 7]           # shuffled, two duplicates
    order = [int(i) for i in ids]
    results = [dict(preds=preds[order[a:a + 16]], bbox_ids=order[a:a + 16]) for a in range(0, len(order), 16)]

    class _Self:
        ann_file = "/nonexistent/mpii_val.json"

        @staticmethod
        def _sort_and_unique_bboxes(kpts, key="bbox_id"):
            kpts = sorted(kpts, key=lambda x: x[key])
            for i in range(len(kpts) - 1, 0, -1):
                if kpts[i][key] == kpts[i - 1][key]:
                    del kpts[i]
            return kpts

    ns = dict(np=np, OrderedDict=OrderedDict, osp=os.path, loadmat=lambda f: gt_dict, savemat=lambda *a, **k: None)
    exec(fn, ns)
    out = ns["evaluate"](_Self(), results, None, "PCKh")
    d = dict(preds=preds, bbox_ids=np.array(order), dataset_joints=names.astype(str), jnt_missing=missing,
             pos_gt_src=pos_gt, headboxes_src=head,
             ref_names=np.array(list(out.keys())), ref_values=np.array([float(v) for v in out.values()], dtype=np.float64))
    np.savez_compressed(os.path.join(OUT, name), **d)
    return out


def backward_case(ref, name, seed):
    """Gradients of the reference losses by torch autograd on the CPU (SURVEY §8f rank 1): the explicit-target
    heatmap losses on a rendered target, and KLDiscretLoss on SimDR vectors."""
    N, K, H, W = 2, 4, 32, 32
    hm, _ = synth.blob_heatmaps(N, K, H, W, seed=seed, sigma=1.5, margin=3.0)
    joints, vis = synth.hand_joints(N, K, (128, 128), seed=seed + 1, vis_prob=0.8)
    gen = ref.generateTarget.TopDownGenerateTarget(sigma=1.5, unbiased_encoding=True)
    tg, tw = [], []
    for b in range(N):
        res = dict(joints_3d=joints[b].numpy().copy(), joints_3d_visible=vis[b].numpy().copy(),
                   ann_info=_ann(K, (128, 128), (W, H)))
        out = gen(res)
        tg.append(out["target"]); tw.append(out["target_weight"])
    tg, tw = torch.from_numpy(np.stack(tg)), torch.from_numpy(np.stack(tw))
    tw[0, 1, 0] = 0.5                                  # a fractional weight: w vs w^2 must differ
    d = dict(hm=hm.numpy(), target=tg.numpy(), target_weight=tw.numpy(), joints_3d=joints.numpy(),
             joints_3d_visible=vis.numpy(), sigma=np.float32(1.5), image_size=np.array([128, 128]))
    HL = ref.loss.heatmapLoss if hasattr(ref.loss, "heatmapLoss") else ref.loss
    for tag, crit in (("bal", HL.DistanceLoss(loss_type="L2", balance=True)),
                      ("nobal", HL.DistanceLoss(loss_type="L2", balance=False)),
                      ("sum", HL.DistanceLoss(loss_type="L2", balance=True, reduction="sum")),
                      ("jmse", HL.JointsDistanceLoss(use_target_weight=True, loss_type="mse"))):
        x = hm.clone().requires_grad_(True)
        loss = crit(x, tg, tw)
        (loss * 0.7).backward()                        # a non-unit upstream gradient
        d[f"ref_loss_{tag}"] = np.float32(loss.item())
        d[f"ref_grad_{tag}"] = x.grad.numpy()
    # KLDiscretLoss
    xv, yv = synth.simdr_vectors(N, K, 96, seed=seed + 2)
    tx, ty = synth.simdr_vectors(N, K, 96, seed=seed + 3)
    xv, yv = xv * 3.0, yv * 3.0                       # some |d| > 1 so both SmoothL1 branches are hit
    SL = ref.loss.centernet_simdr_loss if hasattr(ref.loss, "centernet_simdr_loss") else ref.loss
    px, py = xv.clone().requires_grad_(True), yv.clone().requires_grad_(True)
    loss = SL.KLDiscretLoss()(px, py, tx, ty, tw)
    (loss * 1.3).backward()
    d.update(simdr_out_x=xv.numpy(), simdr_out_y=yv.numpy(), simdr_tgt_x=tx.numpy(), simdr_tgt_y=ty.numpy(),
             ref_loss_simdr=np.float32(loss.item()), ref_grad_simdr_x=px.grad.numpy(), ref_grad_simdr_y=py.grad.numpy())
    np.savez_compressed(os.path.join(OUT, name), **d)


def region_maps(B, seed, H=64, W=64, npk=3):
    """Centre map = noise U(0,0.3) + npk Gaussian blobs (sigma 2) per image; size maps U(0,1)."""
    g = torch.Generator().manual_seed(seed)
    c = torch.rand(B, 1, H, W, generator=g) * 0.3
    ys, xs = torch.meshgrid(torch.arange(float(H)), torch.arange(float(W)), indexing="ij")
    for i in range(B):
        for _ in range(npk):
            cx = torch.rand(1, generator=g).item() * W
            cy = torch.rand(1, generator=g).item() * H
            a = 0.4 + torch.rand(1, generator=g).item()
            c[i, 0] += a * torch.exp(-((xs - cx) ** 2 + (ys - cy) ** 2) / 8)
    s = torch.rand(B, 2, H, W, generator=g)
    return c, s


def _boxes_to_arrays(lists, max_num):
    """list over images of None | [[x,y,w,h,conf], ...] -> (boxes f32 [B,max_num,5] zero-filled, counts int32 [B])."""
    B = len(lists)
    boxes = np.zeros((B, max_num, 5), np.float32)
    counts = np.zeros(B, np.int32)
    for i, l in enumerate(lists):
        if l is not None:
            counts[i] = len(l)
            boxes[i, :len(l)] = np.asarray(l, np.float32)
    return boxes, counts


FIRST_RESULT_BOXES = [[80., 124., 58.02, 102.15, 1.3], [10., 250., 30., 40., 1.], [300., 300., 10., 10., 1.],
                      [128., 128., 400., 400., 1.], [5.0, 5.0, 3., 3., 1.], [200.5, 31.25, 77.7, 20.1, 0.4]]


def region_case(ref, name, seed):
    """SURVEY §8f rank 4: the bbox branch of the legacy parsers executed on seeded region maps.
    HeatmapParser_SH (utils/SPheatmapParser.py:32-138,169-206), ResultParser with cfg['DARK'] = True
    (utils/result_parser.py:50-59,131-229,288-306), cs_from_region_map / non_max_suppression
    (utils/evaluation.py:94-212)."""
    B = 6
    c, s = region_maps(B, seed)
    c[1, 0, 10, 10:13] = 2.0                       # a plateau: three equal maxima inside one window all survive the NMS
    c[2] = 0                                       # an empty centre map: no candidate passes the threshold
    c[2, 0, 40, 20] = 0.05
    s40 = s * 40
    d = dict(center=c.numpy().copy(), size=s.numpy().copy())
    SH = ref.SPheatmapParser.HeatmapParser_SH()
    cn = SH.heatmap_nms(c.clone())
    d["ref_nms"] = cn.numpy().copy()
    cand = SH.candidate_bbox(cn.clone(), s.clone(), (256, 256))
    d["ref_sh_cand"] = cand.numpy().copy()
    d["ref_sh_boxes"], d["ref_sh_counts"] = _boxes_to_arrays(SH.non_max_suppression(cand), 1)
    SH.max_num_bbox = 10
    for thr in (0.6, 0.3, 0.1):
        SH.iou_threshold = thr
        bx, ct = _boxes_to_arrays(SH.non_max_suppression(cand), 10)
        d[f"ref_sh_boxes10_iou{int(thr * 10)}"], d[f"ref_sh_counts10_iou{int(thr * 10)}"] = bx, ct
    # the whole parse() call, centre maps mutated in place by the reference
    # keypoint heatmaps: blobs + noise whose centres lie inside the bbox window that image j is decoded in below
    # (a window holding only noise makes the DARK Taylor step ill-conditioned: no parity to speak of)
    rng = np.random.default_rng(seed + 1)
    centers = np.zeros((B, 5, 2), np.float32)
    for j in range(B):
        x0, y0, x1, y1 = O.first_result_roi(FIRST_RESULT_BOXES[j], (64, 64), 4, 1.3)
        centers[j, :, 0] = (x0 + x1) / 2 + (rng.random(5) - 0.5) * 0.5 * (x1 - x0)
        centers[j, :, 1] = (y0 + y1) / 2 + (rng.random(5) - 0.5) * 0.5 * (y1 - y0)
    hm, _ = synth.blob_heatmaps(B, 5, 64, 64, seed=seed + 1, centers=torch.from_numpy(centers))
    d["kpt_hm"] = hm.numpy().copy()
    d["kpt_centers"] = centers
    SH = ref.SPheatmapParser.HeatmapParser_SH()
    c_in = c.clone()
    kpt, boxes = SH.parse(hm.clone(), c_in, s.clone(), (256, 256))
    d["ref_parse_kpt"] = kpt.numpy().copy()
    d["ref_parse_boxes"], d["ref_parse_counts"] = _boxes_to_arrays(boxes, 1)
    d["ref_parse_center_after"] = c_in.numpy().copy()
    # ResultParser, DARK = True.  One candidate: the executed method as is.  Ten candidates: on CPU tensors the
    # reference's blur aliases the centre map and re-blurs it once per candidate; the CUDA semantics (a fresh copy
    # each time) are obtained by executing its own adjust_keypoints_by_DARK per candidate on un-aliased inputs.
    RP = ref_loader.make_result_parser(ref, dark=True)
    cn2 = RP.heatmap_nms(c.clone())
    RP.num_candidates = 1
    d["ref_rp_cand1"] = RP.candidate_bbox(cn2.clone(), s40.clone()).numpy().copy()
    d["ref_rp_boxes1"], d["ref_rp_counts1"] = _boxes_to_arrays(
        RP.non_max_suppression(torch.from_numpy(d["ref_rp_cand1"])), 1)
    tv, ti = torch.topk(cn2.reshape(B, -1), 10)
    xy = np.zeros((B, 10, 2), np.float32)
    for i in range(10):
        kp = torch.stack([(ti[:, i] % 64).float(), torch.div(ti[:, i], 64, rounding_mode="trunc").float()], 1)[:, None, :]
        xy[:, i] = ref.heatmap_post_processing.adjust_keypoints_by_DARK(kp.clone(), cn2.clone())[:, 0, :]
    d["ref_rp_xy10"] = xy * 4
    d["ref_rp_topk_idx"] = ti.numpy().copy()
    d["ref_rp_topk_val"] = tv.numpy().copy()
    # cs_from_region_map + non_max_suppression (evaluation.py)
    ev = ref.evaluation
    region = torch.cat([c, s40], 1)
    for K, thr in ((20, 0.1), (5, 0.5)):
        cc = ev.cs_from_region_map(region.clone(), 256, K, thr)
        d[f"ref_cs_cand_k{K}"] = cc.numpy().copy()
        d[f"ref_cs_boxes_k{K}"], d[f"ref_cs_counts_k{K}"] = _boxes_to_arrays(ev.non_max_suppression(cc, 0.6, 0.1, 3), 3)
    # bbox-restricted keypoint decode
    RPn = ref_loader.make_result_parser(ref, dark=False)
    for dark, P in ((False, RPn), (True, RP)):
        out = np.zeros((len(FIRST_RESULT_BOXES), 5, 3), np.float32)
        for j, bb in enumerate(FIRST_RESULT_BOXES):
            out[j] = P._get_first_result(list(bb), hm.clone(), j % B).numpy()[0]
        d[f"ref_first_result_dark{int(dark)}"] = out
    d["first_result_boxes"] = np.asarray(FIRST_RESULT_BOXES, np.float64)
    # the reference's own fixture (utils/SPheatmapParser.py:221-233)
    c_hm = torch.zeros(2, 1, 64, 64); c_hm[..., 3, 3] = 1
    s_hm = torch.zeros(2, 2, 64, 64); s_hm[..., 0:7, 0:7] = 1.
    k_hm = torch.zeros((2, 4, 64, 64)); k_hm[..., 3, 3] = 1; k_hm[..., 3, 2] = 0.5; k_hm[..., 2, 3] = 0.5
    _, b = ref.SPheatmapParser.HeatmapParser_SH().parse(k_hm, c_hm, s_hm, (256, 256))
    d["ref_main_boxes"], _ = _boxes_to_arrays(b, 1)
    np.savez_compressed(os.path.join(OUT, name), **d)


def srhandnet_case(ref, name, seed):
    """R3b: SRHandNetGenerateTarget (generateTarget.py:303-426) executed per sample: four scales, region map on/off,
    integer-centre and sub-pixel encodings, boxes inside, across and outside the image."""
    rng = np.random.default_rng(seed)
    N, K = 4, 5
    hs = [[16, 16], [16, 16], [32, 32], [64, 64]]
    j = np.zeros((N, K, 3), np.float32); j[..., :2] = rng.uniform(-30, 290, (N, K, 2))
    v = np.zeros((N, K, 3), np.float32); v[..., :2] = (rng.random((N, K, 1)) < 0.85)
    bbox = np.stack([rng.uniform(0, 200, N), rng.uniform(0, 200, N), rng.uniform(10, 200, N), rng.uniform(10, 200, N)], 1).astype(np.float32)
    bbox[1] = (-150.0, 40.0, 60.0, 60.0)          # centre left of the image: the slice's upper bound goes negative
    bbox[2] = (250.0, 250.0, 30.0, 500.0)         # height ratio clipped to 1, window cut by the border
    bbox[3] = (400.0, 10.0, 20.0, 20.0)           # outside on the right: empty window
    d = dict(joints_3d=j, joints_3d_visible=v, bbox=bbox, heatmap_sizes=np.asarray(hs), sigmas=np.asarray([2, 2, 2, 2]))
    G = ref.generateTarget
    for pred_bbox in (True, False):
        for unb in (False, True):
            T = G.SRHandNetGenerateTarget(pred_bbox=pred_bbox, sigma=[2, 2, 2, 2], unbiased_encoding=unb)
            for i in range(len(hs)):
                d[f"ref_t_bbox{int(pred_bbox)}_unb{int(unb)}_s{i}"] = []
                d[f"ref_w_bbox{int(pred_bbox)}_unb{int(unb)}_s{i}"] = []
            for n in range(N):
                res = dict(joints_3d=j[n].copy(), joints_3d_visible=v[n].copy(), bbox=bbox[n].copy(),
                           ann_info=dict(image_size=np.array([256, 256]), heatmap_size=np.array(hs), num_joints=K,
                                         joint_weights=np.ones((K, 1), np.float32), use_different_joint_weights=False))
                out = T(res)
                for i in range(len(hs)):
                    d[f"ref_t_bbox{int(pred_bbox)}_unb{int(unb)}_s{i}"].append(out["target"][i])
                    d[f"ref_w_bbox{int(pred_bbox)}_unb{int(unb)}_s{i}"].append(out["target_weight"][i])
    d = {k: np.asarray(x) for k, x in d.items()}
    np.savez_compressed(os.path.join(OUT, name), **d)


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    ref = ref_loader.load()
    hm, _, _, _ = decode_case(ref, "decode_64.npz", N=2, K=8, H=64, W=64, seed=11, image_size=(256, 256))
    decode_case(ref, "decode_56.npz", N=2, K=6, H=56, W=56, seed=12, image_size=(224, 224))
    decode_case(ref, "decode_mpii16.npz", N=1, K=16, H=64, W=64, seed=13, image_size=(256, 256))
    render_loss_case(ref, "render_loss_64.npz", N=2, K=8, H=64, W=64, seed=21, image_size=(256, 256), hm=hm)
    hm56, _ = synth.blob_heatmaps(2, 6, 56, 56, seed=12)
    render_loss_case(ref, "render_loss_56.npz", N=2, K=6, H=56, W=56, seed=22, image_size=(224, 224), hm=hm56)
    metrics_case(ref, "metrics_16.npz", N=48, K=16, seed=31)
    backward_case(ref, "loss_backward.npz", seed=41)
    udp_case(ref, "render_udp.npz", seed=51)
    udp_decode_case(ref, "decode_udp.npz", seed=61)
    mpii_case("mpii_pckh.npz", seed=71)
    region_case(ref, "region_bbox.npz", seed=81)
    srhandnet_case(ref, "render_srhandnet.npz", seed=91)
    # the reference's only hand-derivable known answer (utils/SPheatmapParser.py:221-233)
    kpt_hm = torch.zeros((2, 4, 64, 64)); kpt_hm[..., 3, 3] = 1; kpt_hm[..., 3, 2] = 0.5; kpt_hm[..., 2, 3] = 0.5
    k, _ = ref.SPheatmapParser.HeatmapParser_SH().parse(kpt_hm.clone(), image_size=(256, 256))
    np.savez_compressed(os.path.join(OUT, "sp_parser_main.npz"), ref_kpt=k.numpy())
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
