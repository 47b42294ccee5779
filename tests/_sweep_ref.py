"""Reference of the score x IoU threshold sweep (analyze.det_seg_scores_sweep, ampis_eval_images_sweep_host) in numpy,
sharing none of its code: for every image and score threshold the predictions are filtered with numpy's own
``scores > s`` on the caller's array, the kept list goes through tests/_dataset_ref.image() (sparse incidence
product, first arg-max per ground-truth row) and the cell is counted from its per-row results:

- TP = rows whose best IoU is strictly above the IoU threshold, FN = the other rows;
- FP = kept predictions that no TP row chose;
- seg TP / FP / FN = sums over the TP rows of intersection, prediction area - intersection, GT area - intersection.

Identical kept lists (several score thresholds between the same two scores) are evaluated once."""
import numpy as np

from tests import _dataset_ref as D


def image_sweep(gt, pred, scores, score_thresholds, iou_thresholds):
    """int64 arrays of one image: n_pred [K] and cells [K, T, 6] (det TP / FP / FN, seg TP / FP / FN)."""
    K, T = len(score_thresholds), len(iou_thresholds)
    G = len(gt)
    n_pred = np.zeros(K, np.int64)
    cells = np.zeros((K, T, 6), np.int64)
    seen = {}
    for k, s in enumerate(score_thresholds):
        with np.errstate(over='ignore'):
            keep = np.flatnonzero(scores > float(s))
        n_pred[k] = len(keep)
        key = keep.tobytes()
        if key not in seen:
            res = D.image(list(gt), [pred[i] for i in keep], D.MODE_IOU)
            seen[key] = res
        res = seen[key]
        area = res['area'].astype(np.int64)
        for j, t in enumerate(iou_thresholds):
            m = res['best_score'] > float(t)
            col = res['best_col'][m].astype(np.int64)
            inter = res['best_inter'][m].astype(np.int64)
            a_gt = area[:G][m]
            a_pr = area[G + col]
            tp = int(m.sum())
            cells[k, j] = [tp, len(keep) - len(np.unique(col)), G - tp,
                           inter.sum(), (a_pr - inter).sum(), (a_gt - inter).sum()]
    return n_pred, cells


def sweep(gt_lists, pred_lists, scores, score_thresholds, iou_thresholds):
    """The dict of analyze.det_seg_scores_sweep for a list of images."""
    K, T = len(score_thresholds), len(iou_thresholds)
    per = [image_sweep(g, p, np.asarray(s), score_thresholds, iou_thresholds)
           for g, p, s in zip(gt_lists, pred_lists, scores)]
    n_pred = np.stack([p[0] for p in per]) if per else np.zeros((0, K), np.int64)
    cells = np.stack([p[1] for p in per]) if per else np.zeros((0, K, T, 6), np.int64)
    out = {'n_pred': n_pred, 'totals': cells[..., :3].sum(axis=0), 'seg_totals': cells[..., 3:].sum(axis=0)}
    for c, k in enumerate(('det_tp', 'det_fp', 'det_fn', 'seg_tp', 'seg_fp', 'seg_fn')):
        out[k] = cells[..., c]
    tp, fp, fn = (out['totals'][..., c].astype(np.float64) for c in range(3))
    with np.errstate(invalid='ignore', divide='ignore'):
        out['det_precision'] = tp / (tp + fp)
        out['det_recall'] = tp / (tp + fn)
    return out


SWEEP_KEYS = ('n_pred', 'det_tp', 'det_fp', 'det_fn', 'seg_tp', 'seg_fp', 'seg_fn', 'totals', 'seg_totals')


def assert_same(got, ref, what=''):
    """Every count equal, precision / recall equal bit for bit with NaN where the reference has NaN."""
    for k in SWEEP_KEYS:
        assert np.asarray(got[k]).shape == ref[k].shape, (what, k, np.asarray(got[k]).shape, ref[k].shape)
        assert np.array_equal(np.asarray(got[k], np.int64), ref[k]), (what, k)
    for k in ('det_precision', 'det_recall'):
        a, b = np.asarray(got[k], np.float64), ref[k]
        assert np.array_equal(np.isnan(a), np.isnan(b)), (what, k)
        assert np.array_equal(a[~np.isnan(a)].view(np.uint64), b[~np.isnan(b)].view(np.uint64)), (what, k)
