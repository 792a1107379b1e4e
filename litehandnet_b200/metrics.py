"""Drop-in mirrors of the reference's metric functions, accumulated on the GPU as shardable integer
counters (SURVEY.md §8a M1-M5, §8e):

  utils/evaluation.py:10                                   evaluate_pck
  utils/post_processing/evaluation/top_down_eval.py:65     keypoint_pck_accuracy
  utils/post_processing/evaluation/top_down_eval.py:104    keypoint_epe
  utils/post_processing/evaluation/top_down_eval.py:167    keypoint_auc
  datasets/base_dataset.py:193                             Kpt2dDataset._report_metric (arithmetic)

Hit counts are bit-exact: the normalised distance is evaluated in the dtype numpy would promote to,
rounded to f32 and compared with the f32 threshold, exactly as _calc_distances/_distance_acc do.
The final ratios (hits/valid, means) are taken on the host from the int64 counters with the
reference's own expressions, so sharded and monolithic evaluation give identical numbers.
"""
from collections import OrderedDict

import numpy as np
import torch

from . import _lib as L
from . import ops
from .decode import _device, _up


def _counters(pred, gt, mask, thr, normalize=None, norm_const=1.0, counters=None):
    p, _ = _up(pred)
    g, _ = _up(gt)
    m, _ = _up(np.asarray(mask, dtype=bool) if not isinstance(mask, torch.Tensor) else mask)
    n = None
    if normalize is not None:
        n, _ = _up(normalize)
    return ops.pck_accumulate(p, g, m, thr, n, norm_const, counters)


def _acc_from(hits, valid):
    """_distance_acc per joint + the averaging of keypoint_pck_accuracy (top_down_eval.py:44-101)."""
    hits = np.asarray(hits, dtype=np.int64); valid = np.asarray(valid, dtype=np.int64)
    acc = np.array([h / v if v > 0 else -1 for h, v in zip(hits, valid)])
    valid_acc = acc[acc >= 0]
    cnt = len(valid_acc)
    avg_acc = valid_acc.mean() if cnt > 0 else 0
    return acc, avg_acc, cnt


def keypoint_pck_accuracy(pred, gt, mask, thr, normalize):
    """-> (acc [K], avg_acc, cnt).  pred/gt [N,K,2], mask [N,K] bool, normalize [N,2].  Unlike the
    reference, `normalize` is not mutated (the reference overwrites entries <= 0 with 1e6)."""
    K = pred.shape[1]
    c = _counters(pred, gt, mask, [thr], normalize=normalize).cpu().numpy().reshape(3, K)
    return _acc_from(c[0], c[1])


def keypoint_auc(pred, gt, mask, normalize, num_step=20):
    """normalize is a scalar (30 px in _report_metric); thresholds i/num_step."""
    K = pred.shape[1]
    thr = [1.0 * i / num_step for i in range(num_step)]
    c = _counters(pred, gt, mask, thr, normalize=None, norm_const=float(normalize)).cpu().numpy().reshape(num_step + 2, K)
    auc = 0
    for i in range(num_step):
        auc += 1.0 / num_step * _acc_from(c[i], c[num_step])[1]
    return auc


def keypoint_epe(pred, gt, mask):
    """Mean end-point error over the visible joints.  The distances are summed in 2^-20 px fixed point
    (int64: exact, order-independent, shardable); the reference sums f32 distances.  A distance that is NaN,
    infinite or at least 2^43 px (a NaN or inf prediction, say) cannot be held in that sum: it adds nothing and the
    joint still counts, where the reference would return NaN or inf."""
    K = pred.shape[1]
    n = pred.shape[0]
    dev_pred, _ = _up(pred)
    ones = torch.ones((n, 2), dtype=torch.float32, device=dev_pred.device)   # np.ones(..., float32) in the reference
    c = _counters(dev_pred, gt, mask, [], normalize=ones).cpu().numpy().reshape(2, K)
    return (c[1].sum() / 1048576.0) / max(1, int(c[0].sum()))


class MetricAccumulator:
    """Streaming / sharded form of Kpt2dDataset._report_metric: call update() per batch (on each rank),
    all_reduce() once, then compute().  Counter layout = lhn_decode_heatmap_pck's:
    pck_hits[K], pck_valid[K], auc_hits[steps][K], auc_valid[K], epe_valid[K], epe_fix[K]."""

    def __init__(self, num_joints, device="cuda", pck_thr=0.2, auc_nor=30.0, auc_steps=20):
        self.K, self.pck_thr, self.auc_nor, self.steps = num_joints, pck_thr, auc_nor, auc_steps
        self.counters = torch.zeros((auc_steps + 5) * num_joints, dtype=torch.int64, device=device)

    def update_from_heatmaps(self, heatmaps, center, scale, gt, mask, bbox_wh, post_process="default", kernel=11):
        """Fused decode + counters in one kernel (BASELINE config 4).  Returns the decode dict."""
        refine = {"unbiased": L.REFINE_DARK, "default": L.REFINE_SIGN, None: L.REFINE_NONE}[post_process]
        return ops.decode_heatmap_pck(heatmaps, L.MASK_NEG1, refine, center, scale, gt, mask, bbox_wh,
                                      self.counters, self.pck_thr, self.auc_nor, self.steps, kernel)

    def update_from_preds(self, preds, gt, mask, bbox_wh):
        """Counters from already-decoded predictions [N,K,>=2].  As in _report_metric the predictions
        enter the distance arithmetic as float64 (they come back from JSON there)."""
        K, T = self.K, self.steps
        dev = self.counters.device
        preds = preds.to(dev).double().contiguous()
        bb = torch.as_tensor(bbox_wh).to(dev)
        nor = bb.max(dim=1, keepdim=True).values.expand(-1, 2).to(torch.float64).contiguous()
        c = self.counters.view(T + 5, K)
        pck = ops.pck_accumulate(preds, gt, mask, [self.pck_thr], nor).view(3, K)
        auc = ops.pck_accumulate(preds, gt, mask, [1.0 * i / T for i in range(T)], None, self.auc_nor).view(T + 2, K)
        ones = torch.ones((preds.shape[0], 2), dtype=torch.float32, device=dev)
        epe = ops.pck_accumulate(preds, gt, mask, [], ones).view(2, K)
        c[0] += pck[0]; c[1] += pck[1]
        c[2:2 + T] += auc[:T]; c[2 + T] += auc[T]
        c[3 + T] += epe[0]; c[4 + T] += epe[1]

    def all_reduce(self, group=None):
        """ncclAllReduce(int64, SUM) of the counter block — the path's only exchange step."""
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(self.counters, op=dist.ReduceOp.SUM, group=group)
        return self.counters

    def compute_device(self):
        """f64 [3 + K] device tensor (PCK, AUC, EPE, per-joint PCK accuracies): lhn_metrics_finalize, no sync and
        no device->host copy — for loops that log or all-gather the metrics without leaving the stream."""
        return ops.metrics_finalize(self.counters, self.K, self.steps)

    def compute(self, metrics=("PCK", "AUC", "EPE"), on_device=False):
        """-> OrderedDict like dataset.evaluate() (freihand_dataset.py:177-178).  on_device=True takes the ratios
        from lhn_metrics_finalize (one 24-byte device->host read) instead of finishing the counters in NumPy;
        the two are bit-identical."""
        if on_device:
            v = self.compute_device()[:3].cpu().numpy()
            return OrderedDict((m, float(v[i])) for i, m in enumerate(("PCK", "AUC", "EPE")) if m in metrics)
        K, T = self.K, self.steps
        c = self.counters.cpu().numpy().reshape(T + 5, K)
        out = OrderedDict()
        if "PCK" in metrics:
            out["PCK"] = _acc_from(c[0], c[1])[1]
        if "AUC" in metrics:
            out["AUC"] = sum(1.0 / T * _acc_from(c[2 + i], c[2 + T])[1] for i in range(T))
        if "EPE" in metrics:
            out["EPE"] = (c[4 + T].sum() / 1048576.0) / max(1, int(c[3 + T].sum()))
        return out


def report_metric(outputs, gts, masks, bbox_wh=None, head_size=None, metrics=("PCK", "AUC", "EPE"),
                  pck_thr=0.2, pckh_thr=0.5, auc_nor=30):
    """datasets/base_dataset.py:193-261 arithmetic on arrays instead of the JSON/db round trip:
    outputs [N,K,2] (f64 in the reference after JSON), gts [N,K,2] f32, masks [N,K] bool,
    bbox_wh [N,2] (PCK normaliser max(w,h)), head_size [N] (PCKh).  Returns [(name, value), ...]."""
    outputs = np.asarray(outputs, dtype=np.float64) if not isinstance(outputs, torch.Tensor) else outputs.double()
    info_str = []
    if 'PCK' in metrics:
        t = np.max(np.asarray(bbox_wh, dtype=np.float64), axis=1)
        _, pck, _ = keypoint_pck_accuracy(outputs, gts, masks, pck_thr, np.stack([t, t], axis=1))
        info_str.append(('PCK', pck))
    if 'PCKh' in metrics:
        hs = np.asarray(head_size, dtype=np.float64)
        _, pckh, _ = keypoint_pck_accuracy(outputs, gts, masks, pckh_thr, np.stack([hs, hs], axis=1))
        info_str.append(('PCKh', pckh))
    if 'AUC' in metrics:
        info_str.append(('AUC', keypoint_auc(outputs, gts, masks, auc_nor)))
    if 'EPE' in metrics:
        info_str.append(('EPE', keypoint_epe(outputs, gts, masks)))
    return info_str


def evaluate_results(results, db, metric='PCK', pck_thr=0.2, pckh_thr=0.5, auc_nor=30):
    """dataset.evaluate(results, res_folder, metric) without the JSON detour (SURVEY §8f rank 2):
    datasets/datasets/hand/freihand_dataset.py:111-183 + base_dataset.py:193-284.

    results: list of TopDownDecoder.decode() dicts (preds [N,K,3], boxes [N,6], image_paths, bbox_ids) — NumPy
    arrays or CUDA tensors; db: the dataset's list of annotation dicts ('joints_3d' [K,3], 'joints_3d_visible'
    [K,3], 'bbox' [x,y,w,h], optional 'head_size'), sorted by bbox_id as the reference's _get_db leaves it.
    The predictions are sorted by bbox_id and de-duplicated (_sort_and_unique_bboxes keeps the first of equal
    ids), the distances are taken in float64 (the reference reads the points back from JSON) and the hit
    counts come from lhn_pck_accumulate.  Returns an OrderedDict like the reference."""
    metrics = metric if isinstance(metric, (list, tuple)) else [metric]
    for m in metrics:
        if m not in ('PCK', 'PCKh', 'AUC', 'EPE'):
            raise KeyError(f'metric {m} is not supported')
    dev = _device()
    preds = torch.cat([_up(r['preds'], torch.float32)[0] for r in results], 0)
    ids = torch.as_tensor(np.concatenate([np.asarray(r['bbox_ids']).reshape(-1) for r in results])).to(dev)
    order = torch.sort(ids, stable=True).indices                  # stable: the first of equal ids stays first
    ids_s = ids[order]
    keep = torch.ones_like(ids_s, dtype=torch.bool)
    keep[1:] = ids_s[1:] != ids_s[:-1]
    preds = preds[order][keep]
    assert preds.shape[0] == len(db), (preds.shape[0], len(db))
    gts = torch.as_tensor(np.stack([np.asarray(it['joints_3d'], dtype=np.float32)[:, :2] for it in db])).to(dev)
    masks = torch.as_tensor(np.stack([np.asarray(it['joints_3d_visible'])[:, 0] > 0 for it in db])).to(dev)
    bbox_wh = head = None
    if 'PCK' in metrics:
        bbox_wh = np.stack([np.asarray(it['bbox'], dtype=np.float64)[2:] for it in db])
    if 'PCKh' in metrics:
        head = np.asarray([it['head_size'] for it in db], dtype=np.float64)
    return OrderedDict(report_metric(preds[..., :2].double(), gts, masks, bbox_wh, head, metrics, pck_thr, pckh_thr,
                                     auc_nor))


def mpii_pckh_counters(preds, gt_dict, thresholds, counters=None, sc_bias=0.6):
    """Shardable int64 counters of the MPII PCKh arithmetic (lhn_mpii_pckh_accumulate): hits[T][K], count[K].
    preds [N,K,>=2] 0-based (CUDA or NumPy); gt_dict arrays cover the same N samples (or a shard of them)."""
    import ctypes as C
    dev = _device()
    p, _ = _up(preds, torch.float32)
    p = p.contiguous()
    N, K = p.shape[0], p.shape[1]
    gt = torch.as_tensor(np.ascontiguousarray(np.transpose(np.asarray(gt_dict['pos_gt_src'], dtype=np.float64), (2, 0, 1)))).to(dev)
    hb = np.asarray(gt_dict['headboxes_src'], dtype=np.float64)                       # [corner, xy, N]
    head = torch.as_tensor(np.ascontiguousarray(np.concatenate([hb[0].T, hb[1].T], axis=1))).to(dev)   # [N,4]
    vis = torch.as_tensor(np.ascontiguousarray((1 - np.asarray(gt_dict['jnt_missing'])).T != 0)).to(dev).to(torch.uint8)
    T = len(thresholds)
    if counters is None:
        counters = torch.zeros((T + 1) * K, dtype=torch.int64, device=dev)
    thr = (C.c_double * T)(*[float(t) for t in thresholds])
    L.check(L.lib().lhn_mpii_pckh_accumulate(L.ptr(p), p.shape[2], L.ptr(gt), L.ptr(head), L.ptr(vis), N, K, thr, T,
                                             float(sc_bias), L.ptr(counters), L.stream()), "lhn_mpii_pckh_accumulate")
    return counters


def mpii_evaluate(results, gt_dict, metric='PCKh'):
    """TopDownMpiiDataset.evaluate (datasets/datasets/body/topdown_mpii_dataset.py:126-249) with the contents of
    mpii_gt_val.mat handed in as ``gt_dict`` (dataset_joints, jnt_missing, pos_gt_src, headboxes_src): results are
    sorted / de-duplicated by bbox_id, the hit counts come from the GPU, the name/value table is the reference's."""
    metrics = metric if isinstance(metric, (list, tuple)) else [metric]
    for m in metrics:
        if m not in ('PCKh',):
            raise KeyError(f'metric {m} is not supported')
    dev = _device()
    preds = torch.cat([_up(r['preds'], torch.float32)[0] for r in results], 0)
    ids = torch.as_tensor(np.concatenate([np.asarray(r['bbox_ids']).reshape(-1) for r in results])).to(dev)
    order = torch.sort(ids, stable=True).indices
    ids_s = ids[order]
    keep = torch.ones_like(ids_s, dtype=torch.bool)
    keep[1:] = ids_s[1:] != ids_s[:-1]
    preds = preds[order][keep].contiguous()
    thr = MPII_THRESHOLDS
    K = preds.shape[1]
    c = mpii_pckh_counters(preds, gt_dict, thr).cpu().numpy().reshape(len(thr) + 1, K)
    return mpii_table(c, gt_dict['dataset_joints'])


# PCKh@0.5, then the rows of pckAll (np.arange(0, 0.5 + 0.01, 0.01)) in the reference's evaluate
MPII_THRESHOLDS = [0.5] + [float(t) for t in np.arange(0, 0.5 + 0.01, 0.01)]


def mpii_table(counters, dataset_joints):
    """The name/value table of TopDownMpiiDataset.evaluate from the counters [len(MPII_THRESHOLDS) + 1, K]
    (hits per threshold, then the joint count) of mpii_pckh_counters."""
    c = np.asarray(counters).astype(np.float64)
    jnt_count = c[-1]
    PCKh = 100. * c[0] / jnt_count
    pck10 = (100. * c[1 + 10] / jnt_count).astype(np.float32)                  # pckAll is a float32 table
    names = np.asarray(dataset_joints)
    J = {n: np.where(names == n)[1][0] for n in ('head', 'lsho', 'lelb', 'lwri', 'lhip', 'lkne', 'lank', 'rsho',
                                                 'relb', 'rwri', 'rkne', 'rank', 'rhip')}
    PCKh = np.ma.array(PCKh, mask=False); PCKh.mask[6:8] = True
    jc = np.ma.array(jnt_count, mask=False); jc.mask[6:8] = True
    ratio = jc / np.sum(jc).astype(np.float64)
    return OrderedDict([('Head', PCKh[J['head']]), ('Shoulder', 0.5 * (PCKh[J['lsho']] + PCKh[J['rsho']])),
                        ('Elbow', 0.5 * (PCKh[J['lelb']] + PCKh[J['relb']])), ('Wrist', 0.5 * (PCKh[J['lwri']] + PCKh[J['rwri']])),
                        ('Hip', 0.5 * (PCKh[J['lhip']] + PCKh[J['rhip']])), ('Knee', 0.5 * (PCKh[J['lkne']] + PCKh[J['rkne']])),
                        ('Ankle', 0.5 * (PCKh[J['lank']] + PCKh[J['rank']])), ('PCKh', np.sum(PCKh * ratio)),
                        ('PCKh@0.1', np.sum(pck10 * ratio))])


def evaluate_pck(pred_keypoints_hm, gt_keypoints_hm, bbox, image_size=256, target_weight=None, thr=0.2):
    """utils/evaluation.py:10-59 -> python float (NaN if an image has zero total weight, as the
    reference).  bbox [B, n_hand, 4] (cx, cy, w, h); only hand 0 is used (:23)."""
    p, _ = _up(pred_keypoints_hm)
    g, _ = _up(gt_keypoints_hm)
    bb, _ = _up(bbox, torch.float32)
    bb = bb[:, 0, 2:].contiguous()
    w = None
    if target_weight is not None:
        w, _ = _up(target_weight, torch.float32)
    isz = (image_size, image_size) if np.isscalar(image_size) else tuple(image_size)
    _, mean = ops.evaluate_pck(p, g, bb, w, isz, thr)
    return float(mean.item())
