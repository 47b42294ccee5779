"""Instance matching and detection/segmentation scores -- drop-in for ``ampis.analyze``
(reference ampis/analyze.py:19-339) on the GPU.

The reference loops over ground-truth masks in Python and calls pycocotools' RLE.iou on
chunks of 80 predictions (analyze.py:149-164), then RLE.merge/RLE.area per match
(analyze.py:315-321).  Here one fused kernel (csrc/intersect.cu) produces, per ground-truth
mask, the first-arg-max prediction, its IoU and its intersection, so the matcher and all
det/seg scores are read off a single pass.  ``interval`` is accepted for signature
compatibility; it never affected results (SURVEY.md Appendix B.14).
"""
import os
from pathlib import Path

import numpy as np
import torch

from . import engine
from .containers import Instances
from .structures import InstanceSet, RLEMasks, masks_to_rle, masks_to_bitmask_array  # noqa: F401 (re-exported like ampis.analyze)


def align_instance_sets(a, b):
    """Reorder *b* to match *a* by file name, keeping common files only (analyze.py:19-51)."""
    bdict = {Path(item.filepath).name: item for item in b}
    a_ordered, b_ordered = [], []
    for item in a:
        x = bdict.get(Path(item.filepath).name, None)
        if x is not None:
            a_ordered.append(item)
            b_ordered.append(x)
    return a_ordered, b_ordered


def _check_same_size(*mask_lists):
    sizes = [m['size'] for ml in mask_lists for m in ml]
    if not sizes:
        return
    a = np.asarray(sizes, np.int64).reshape(len(sizes), -1)[:, :2]
    bad = np.nonzero((a != a[0]).any(axis=1))[0]
    if len(bad):
        raise ValueError('masks of different image sizes cannot be compared (%s vs %s)'
                         % (tuple(a[0].tolist()), tuple(a[bad[0]].tolist())))


def _rows_vs_cols(rows_rle, cols_rle, mode, dense=False, crowded=None):
    """One image: rows x cols through the table API, kernel by kernel. Returns host arrays + device handles.
    crowded: True when the caller already knows the image belongs to the tensor-core contraction (the one-call
    entry flagged it); None = decide here from the operand fill."""
    _check_same_size(rows_rle, cols_rle)
    # measured as bounding-box windows (the smallest storage, the fastest culled walk) ...
    table = engine.table_from_rle(list(rows_rle) + list(cols_rle), layout=engine.MATCH_LAYOUT, paint=False)
    # ... unless the image is crowded (operand fill above the measured crossover): then linear spans and the
    # tensor-core contraction.  The results are identical either way.
    if crowded is None:
        crowded = min(len(rows_rle), len(cols_rle)) >= engine.MMA_MIN_SIDE and \
            engine.operand_fill(table) >= engine.MMA_FILL_THRESHOLD
    if crowded and table.layout == engine.LAYOUT_CROP:
        table.relayout(engine.LAYOUT_SPAN)
    table.paint()
    groups = engine.Groups.interleaved(table.device, [len(rows_rle)], [len(cols_rle)], dense=dense or crowded)
    res = engine.intersect(table, groups, mode, kernel='mma' if crowded else 'rows')
    return table, groups, res


#: one library call per image (engine.eval_image) instead of the table API driven kernel by kernel from Python
FUSED_CALL = os.environ.get('AMPIS_FUSED_CALL', '1') != '0'


def _image_rows(rows_rle, cols_rle, mode):
    """Per-row arg-max results of one image as host arrays: (best_col int64, best_score float64, best_inter int64,
    areas uint32 of rows then columns).  Normally ONE call into the library (ampis_eval_images_host: bounding-box
    windows, candidate-pair join, culled AND+popc).  A crowded image -- candidate pairs above
    engine.CROWD_PAIR_FRACTION of all pairs, decided on the device right after the join, before any intersection is
    computed -- comes back flagged and goes through the table API with the tensor-core contraction instead, which is
    where the time goes on such images.  Identical results either way.  The last result is cached on the identity of
    the string objects, so a loop over IoU thresholds evaluates the image once."""
    G = len(rows_rle)
    if FUSED_CALL:
        crowd = engine.CROWD_PAIR_FRACTION if min(G, len(cols_rle)) >= engine.MMA_MIN_SIDE else -1.0
        r = engine.eval_images([rows_rle], [cols_rle], mode, crowd_frac=crowd, cache=True)
        if not r.crowded:                 # copies: the cached arrays stay untouched
            return r.best_col.astype(np.int64), r.best_score.copy(), r.best_inter.astype(np.int64), r.area.copy()
        table, groups, res = _rows_vs_cols(rows_rle, cols_rle, mode, crowded=True)
        return (res.best_col[:G].cpu().numpy().astype(np.int64), res.best_score[:G].cpu().numpy(),
                res.best_inter[:G].cpu().numpy().view(np.uint32).astype(np.int64), table.areas_np())
    table, groups, res = _rows_vs_cols(rows_rle, cols_rle, mode)
    return (res.best_col[:G].cpu().numpy().astype(np.int64), res.best_score[:G].cpu().numpy(),
            res.best_inter[:G].cpu().numpy().view(np.uint32).astype(np.int64), table.areas_np())


def _piecewise_iou(a, b, interval=80):
    """len(a) x len(b) float64 IoU matrix (analyze.py:54-112)."""
    imax, jmax = len(a), len(b)
    if imax == 0 or jmax == 0:
        return np.zeros((imax, jmax))
    if FUSED_CALL:
        r = engine.eval_image(a, b, engine.MODE_IOU, dense_iou=True)
        if not (min(imax, jmax) >= engine.MMA_MIN_SIDE and r.fill() >= engine.MMA_FILL_THRESHOLD):
            return r.iou                  # crowded images go on to the tensor-core contraction, as in _image_rows
    table, groups, res = _rows_vs_cols(a, b, engine.MODE_IOU, dense=True)
    return engine.iou_matrix(table, res, groups, 0).cpu().numpy()


def sparse_iou(a, b, size=None):
    """The non-zero cells of ``_piecewise_iou(a, b)`` without forming the dense matrix: a dict with
    ``row``, ``col`` (int64, sorted by row then column), ``inter`` (uint32 intersections), ``iou``
    (float64, the same values the dense matrix holds) and ``shape``.  Not a function of the reference:
    on images with thousands of instances (spheroidite: 5,000 x 5,000) the dense matrix is 200 MB of
    zeros around a few thousand overlapping pairs; this is the bbox-pruned form (grid-pruned crop rows
    kernel, engine.SparseRows)."""
    from .structures import masks_to_rle
    a, b = (masks_to_rle(m, size) if len(m) else [] for m in (a, b))
    out = {'row': np.zeros(0, np.int64), 'col': np.zeros(0, np.int64), 'inter': np.zeros(0, np.uint32),
           'iou': np.zeros(0), 'shape': (len(a), len(b))}
    if len(a) == 0 or len(b) == 0:
        return out
    _check_same_size(a, b)
    table = engine.table_from_rle(list(a) + list(b), layout=engine.LAYOUT_CROP)
    groups = engine.Groups.interleaved(table.device, [len(a)], [len(b)])
    capacity = 16 * (len(a) + len(b))
    while True:
        sp = engine.SparseRows(table.device, capacity)
        engine.intersect_rows(table, groups, engine.MODE_IOU, sparse=sp)
        n = int(sp.count.item())
        if n <= capacity:
            break
        capacity = n
    r, c, v = (x.cpu().numpy() for x in sp.triplets())
    area = table.areas_np().astype(np.uint32)
    with np.errstate(over='ignore'):
        union = area[r] + area[len(a) + c] - v.astype(np.uint32)          # uint32 wrap-around like rleIou
    out.update(row=r, col=c, inter=v.astype(np.uint32), iou=v.astype(np.float64) / union.astype(np.float64))
    return out


def _match_from_rows(best_col, best_iou, n_pred, iou_thresh):
    """The bookkeeping of analyze.py:166-179 on the per-GT (arg-max, max IoU) arrays."""
    matched = best_iou > iou_thresh
    gt_idx = np.flatnonzero(matched)
    if len(gt_idx):
        cols = best_col[gt_idx]
        tp = np.empty((len(gt_idx), 2), int)
        tp[:, 0] = gt_idx
        tp[:, 1] = cols
        pred_matched = np.zeros(n_pred, bool)
        pred_matched[cols] = True
        fp = np.flatnonzero(~pred_matched)
    else:
        tp = np.asarray([], int)
        fp = np.arange(n_pred)
    return {'tp': tp, 'fn': np.flatnonzero(~matched), 'fp': fp, 'iou': best_iou[gt_idx]}


def _rows_of_image(gt, pred):
    """(best_col, best_iou, best_inter, areas) of one image; the conventions of analyze.py:115-181 for empty sides."""
    G = len(gt)
    if G == 0 or len(pred) == 0:
        return np.full(G, -1, np.int64), np.zeros(G), np.zeros(G, np.int64), None
    return _image_rows(gt, pred, engine.MODE_IOU)


def _piecewise_rle_match(gt, pred, iou_thresh=0.5, interval=80, _details=None):
    """Per-GT arg-max matching on RLE lists (analyze.py:115-181).

    For each ground-truth mask the prediction with the highest IoU is taken (first one on ties,
    only IoUs strictly above 0 count); it is a match when that IoU is strictly above
    *iou_thresh*.  Several ground-truth masks may match the same prediction."""
    best_col, best_iou, best_inter, areas = _rows_of_image(gt, pred)
    if _details is not None:
        _details.update(best_col=best_col, best_iou=best_iou, best_inter=best_inter, areas=areas)
    return _match_from_rows(best_col, best_iou, len(pred), iou_thresh)


def rle_instance_matcher(gt, pred, iou_thresh=0.5, size=None):
    """Instance matching of two mask sets (analyze.py:184-223)."""
    gt = masks_to_rle(gt, size)
    pred = masks_to_rle(pred, size)
    return _piecewise_rle_match(gt, pred, iou_thresh)


#: legacy name of the matcher in older AMPIS releases (SURVEY.md F3)
fast_instance_match = rle_instance_matcher


def det_seg_scores(gt, pred, iou_thresh=0.5, size=None):
    """Detection and segmentation precision / recall of one image (analyze.py:226-339): eleven keys --
    ``det_precision``, ``det_recall`` (floats), per-match ``seg_precision``, ``seg_recall``, ``seg_tp``,
    ``seg_fp``, ``seg_fn`` and the matcher's ``det_tp``, ``det_fn``, ``det_fp``, ``det_tp_iou``.  The
    intersection of every matched pair is a by-product of the row kernel, so there is no second pass
    of merges.  Raises ZeroDivisionError like the reference when TP+FP or TP+FN is zero."""
    gtmasks, predmasks = masks_to_rle(gt, size), masks_to_rle(pred, size)
    G, P = len(gtmasks), len(predmasks)
    best_col, best_iou, best_inter, areas = _rows_of_image(gtmasks, predmasks)     # the matching is done once, below
    return _scores_from_rows(G, P, best_col, best_iou, best_inter,
                             None if areas is None else areas[:G], None if areas is None else areas[G:], iou_thresh)


def _scores_from_rows(G, P, best_col, best_iou, best_inter, areas_gt, areas_pred, iou_thresh):
    """The dict of det_seg_scores from one image's row results (analyze.py:300-339)."""
    det = _match_from_rows(best_col, best_iou, P, iou_thresh)
    tp = np.asarray(det['tp'])
    n_tp, n_fn, n_fp = len(tp), len(det['fn']), len(det['fp'])
    out = {'det_precision': n_tp / (n_tp + n_fp), 'det_recall': n_tp / (n_tp + n_fn)}     # ZeroDivisionError as in the reference
    if n_tp:
        gi, pi = tp[:, 0], tp[:, 1]
        inter = best_inter[gi].astype(np.int64)
        a_gt, a_pr = areas_gt[gi].astype(np.int64), areas_pred[pi].astype(np.int64)
    else:
        inter = a_gt = a_pr = np.array([], np.int64)
    with np.errstate(invalid='ignore', divide='ignore'):
        out['seg_precision'] = inter / a_pr       # TP / (TP + FP) with FP = area(pred) - TP: the integer sum is the area
        out['seg_recall'] = inter / a_gt
    out.update(det_tp=tp, det_fn=det['fn'], det_fp=det['fp'], seg_tp=inter, seg_fn=a_gt - inter, seg_fp=a_pr - inter,
               det_tp_iou=det['iou'])
    return out


def det_seg_scores_batch(gt_list, pred_list, iou_thresh=0.5, size=None):
    """``det_seg_scores`` for many images at once -- not in the reference API, which scores one image
    per Python call (Colab cell 44 loops over the dataset: ``[det_seg_scores(g, p) for g, p in zip(gt, pred)]``).
    All images go through ONE library call (engine.eval_images -> ampis_eval_images_host: the strings are picked up
    where Python keeps them, one upload, one launch of each kernel, one download) and the bookkeeping of
    analyze.py:300-339 is done for all images at once on flat arrays; the result is the list of per-image dicts the
    loop would have produced, key for key and bit for bit.  Images with no ground truth or no predictions raise
    ZeroDivisionError like the per-image function."""
    assert len(gt_list) == len(pred_list)
    gts = [masks_to_rle(g, size) for g in gt_list]
    prs = [masks_to_rle(p, size) for p in pred_list]
    n_img = len(gts)
    if n_img == 0:
        return []
    if sum(map(len, gts)) + sum(map(len, prs)) == 0:
        raise ZeroDivisionError('division by zero')
    # the crowd gate only matters when some image is large enough for the contraction to pay off
    big = max(min(len(g), len(p)) for g, p in zip(gts, prs)) >= engine.MMA_MIN_SIDE
    r = engine.eval_images(gts, prs, engine.MODE_IOU, crowd_frac=engine.CROWD_PAIR_FRACTION if big else -1.0)
    if r.crowded:                          # crowded batch: image by image (each picks its kernel)
        return [det_seg_scores(g, p, iou_thresh) for g, p in zip(gts, prs)]
    return _scores_from_rows_batch(r, iou_thresh)


def _scores_from_rows_batch(r, iou_thresh):
    """analyze.py:166-179 + 300-339 for all images of an engine.ImagesRows at once: every array is formed over the
    concatenated rows / predictions and cut into per-image views at the end (the per-image Python work is a dozen
    slices)."""
    n_img = len(r.n_rows)
    G, P = r.n_rows.astype(np.int64), r.n_cols.astype(np.int64)
    row_off, mask_off = r.row_off, r.mask_off
    pred_off = np.zeros(n_img + 1, np.int64)
    np.cumsum(P, out=pred_off[1:])
    matched = r.best_score > iou_thresh
    # index arrays once, then gathers (a boolean mask costs a pass over all rows every time it is applied); rows and
    # predictions are grouped by image, so "image of item k" is a repeat of the per-image counts
    images = np.arange(n_img)
    before = np.zeros(len(matched) + 1, np.int64)            # matched rows before each row
    np.cumsum(matched, out=before[1:])
    n_tp = before[row_off[1:]] - before[row_off[:-1]]
    n_fn = G - n_tp
    mi = np.flatnonzero(matched)
    m_img = np.repeat(images, n_tp)
    m_gt = mi - np.repeat(row_off[:-1], n_tp)
    m_pr = r.best_col[mi].astype(np.int64)
    pm = np.zeros(int(pred_off[-1]) + 1, np.int64)           # 1 at every matched prediction (+ a sentinel slot)
    pm[pred_off[m_img] + m_pr] = 1
    used_before = np.zeros(len(pm) + 1, np.int64)            # matched predictions before each prediction
    np.cumsum(pm, out=used_before[1:])
    n_fp = P - (used_before[pred_off[1:]] - used_before[pred_off[:-1]])
    fp_local = (np.flatnonzero(pm[:-1] == 0) - np.repeat(pred_off[:-1], n_fp)).astype(int)
    fn_local = (np.flatnonzero(~matched) - np.repeat(row_off[:-1], n_fn)).astype(int)
    bad = np.nonzero((n_tp + n_fp == 0) | (n_tp + n_fn == 0))[0]
    if len(bad):
        raise ZeroDivisionError('division by zero')      # image %d has no ground truth or no predictions
    tp = np.stack([m_gt, m_pr], axis=1).astype(int)
    inter = r.best_inter[mi].astype(np.int64)
    a_gt = r.area[mask_off[m_img] + m_gt].astype(np.int64)
    a_pr = r.area[mask_off[m_img] + G[m_img] + m_pr].astype(np.int64)
    seg_fn, seg_fp = a_gt - inter, a_pr - inter
    with np.errstate(invalid='ignore', divide='ignore'):
        seg_p = inter / a_pr          # TP / (TP + FP) with FP = area(pred) - TP: the integer sum is the area
        seg_r = inter / a_gt
    iou = r.best_score[mi]
    t_off = np.zeros(n_img + 1, np.int64)
    np.cumsum(n_tp, out=t_off[1:])
    fp_off = np.zeros(n_img + 1, np.int64)
    np.cumsum(n_fp, out=fp_off[1:])
    fn_off = np.zeros(n_img + 1, np.int64)
    np.cumsum(n_fn, out=fn_off[1:])
    empty_tp = np.asarray([], int)
    out = []
    t_cut, fp_cut, fn_cut = t_off.tolist(), fp_off.tolist(), fn_off.tolist()      # Python ints: cheap in the loop
    for g in range(n_img):
        a, b = t_cut[g], t_cut[g + 1]
        ntp, nfp, nfn = b - a, fp_cut[g + 1] - fp_cut[g], fn_cut[g + 1] - fn_cut[g]
        out.append({'det_precision': ntp / (ntp + nfp), 'det_recall': ntp / (ntp + nfn),
                    'seg_precision': seg_p[a:b], 'seg_recall': seg_r[a:b],
                    'det_tp': tp[a:b] if ntp else empty_tp,
                    'det_fn': fn_local[fn_cut[g]:fn_cut[g + 1]],
                    'det_fp': fp_local[fp_cut[g]:fp_cut[g + 1]],
                    'seg_tp': inter[a:b], 'seg_fn': seg_fn[a:b], 'seg_fp': seg_fp[a:b], 'det_tp_iou': iou[a:b]})
    return out


_SCORE_DTYPES = (np.float16, np.float32, np.float64)


def _sorted_thresholds(thresholds, what):
    """(thresholds ascending as float64, position of each caller's threshold in that order).  NaN is refused."""
    th = np.asarray(thresholds, np.float64).reshape(-1)
    if len(th) == 0:
        raise ValueError('%s: at least one threshold is needed' % what)
    if np.isnan(th).any():
        raise ValueError('%s: NaN is not a threshold' % what)
    order = np.argsort(th, kind='stable')
    pos = np.empty(len(th), np.int64)
    pos[order] = np.arange(len(th))
    return th[order], pos


def _score_array(s):
    """A float16/32/64 numpy or torch array of scores as a 1-D numpy array of the same dtype (TypeError otherwise)."""
    if isinstance(s, torch.Tensor):
        if s.dtype not in (torch.float16, torch.float32, torch.float64):
            raise TypeError('scores must be float16, float32 or float64, not %s' % s.dtype)
        s = s.detach().cpu().numpy()
    elif not isinstance(s, np.ndarray) or s.dtype.type not in _SCORE_DTYPES:
        raise TypeError('scores must be float16, float32 or float64 numpy or torch arrays, not %r'
                        % (getattr(s, 'dtype', type(s)),))
    return s.reshape(-1)


def _score_levels(scores, sorted_th):
    """Per prediction, the number of sorted thresholds strictly below its score, as numpy decides ``scores > t`` for a
    Python float t: the threshold is rounded to the scores' dtype (NumPy 2), NaN scores are never above it.  So a
    prediction is kept at sorted threshold k iff its level > k.  scores: one array of one float dtype."""
    with np.errstate(over='ignore'):
        th = sorted_th.astype(scores.dtype)                  # rounding is monotone: still sorted
    lv = np.searchsorted(th, scores, side='left')
    lv[np.isnan(scores)] = 0
    return lv.astype(np.uint16)


def _image_levels(sc, sorted_th):
    """Levels of the per-image score arrays sc (concatenated, uint16) and the kept counts int64 [n, K] (instances whose
    level exceeds k), one numpy pass per score dtype."""
    n, K = len(sc), len(sorted_th)
    lens = np.fromiter(map(len, sc), np.int64, n)
    dtypes = [s.dtype for s in sc]
    kinds = sorted(set(dtypes), key=str)
    if len(kinds) <= 1:
        levels = _score_levels(np.concatenate(sc) if n else np.zeros(0), sorted_th)
    else:
        levels = np.zeros(int(lens.sum()), np.uint16)
        code = np.asarray([kinds.index(d) for d in dtypes])
        for c, dt in enumerate(kinds):
            levels[np.repeat(code == c, lens)] = _score_levels(np.concatenate([s for s in sc if s.dtype == dt]), sorted_th)
    img = np.repeat(np.arange(n), lens)
    hist = np.bincount(img * (K + 1) + levels, minlength=n * (K + 1)).reshape(n, K + 1)
    kept = np.cumsum(hist[:, ::-1], axis=1)[:, ::-1][:, 1:]                 # [n, K]: sum over levels > k
    return levels, kept


def _image_scores(p):
    inst = p if type(p) == Instances else p.instances if type(p) == InstanceSet else None
    if inst is None or getattr(inst, 'scores', None) is None:
        raise ValueError('scores are needed for predictions given as %s' % type(p).__name__)
    return inst.scores


def _reorder(a, pos, axis):
    """a with axis `axis` in the order pos (no copy when pos is the identity: thresholds that came sorted)."""
    return a if np.array_equal(pos, np.arange(len(pos))) else np.take(a, pos, axis=axis)


def det_seg_scores_sweep(gt_list, pred_list, score_thresholds, iou_thresholds=None, scores=None, size=None):
    """Detection and segmentation counts of a list of images over a grid of prediction-score cut-offs x IoU
    thresholds, from one evaluation.  Cell (k, j) of image i is ``det_seg_scores(gt_i, kept, iou_thresh=t_j)`` with
    ``kept = pred_i[scores_i > s_k]`` (numpy's comparison on the caller's scores: NaN is never kept), reduced to counts.
    AMPIS's matcher is kept (per-GT first arg-max, several GTs may share a prediction, strict ``>``); this is not
    COCO AP.  An image with no ground truth or nothing kept gets its counts instead of a ZeroDivisionError.

    gt_list / pred_list: per image, any mask container of det_seg_scores_batch (a single image is a list of one).
    scores: per image, a float16/32/64 numpy or torch array with one score per prediction; None takes
    ``instances.scores`` of InstanceSet / Instances predictions (RLE lists need scores).  iou_thresholds: None = the
    ten COCO thresholds 0.50:0.05:0.95; each must be >= 0.

    Returns a dict: ``score_thresholds`` and ``iou_thresholds`` as given (float64), ``n_pred`` int64 [n, K] (kept
    predictions), ``det_tp`` / ``det_fp`` / ``det_fn`` int64 [n, K, T] (``len`` of det_seg_scores' arrays),
    ``seg_tp`` / ``seg_fp`` / ``seg_fn`` int64 [n, K, T] (sums of det_seg_scores' arrays), ``totals`` int64 [K, T, 3]
    (TP / FP / FN over the dataset), ``seg_totals`` int64 [K, T, 3] and ``det_precision`` / ``det_recall`` float64
    [K, T] from the totals (NaN where the denominator is 0).  One library call (engine.eval_images_sweep)."""
    from . import batch
    if len(gt_list) != len(pred_list):
        raise ValueError('%d ground-truth images against %d prediction images' % (len(gt_list), len(pred_list)))
    s_th = np.asarray(score_thresholds, np.float64).reshape(-1)
    i_th = np.asarray(batch.COCO_THRESHOLDS if iou_thresholds is None else iou_thresholds, np.float64).reshape(-1)
    s_sorted, s_pos = _sorted_thresholds(s_th, 'score_thresholds')
    i_sorted, i_pos = _sorted_thresholds(i_th, 'iou_thresholds')
    if i_sorted[0] < 0:
        raise ValueError('iou_thresholds must not be negative')
    if len(s_th) > 65535 or len(i_th) > 256:
        raise ValueError('at most 65,535 score thresholds and 256 IoU thresholds')
    if scores is None:
        scores = [_image_scores(p) for p in pred_list]
    if len(scores) != len(pred_list):
        raise ValueError('%d score arrays for %d images' % (len(scores), len(pred_list)))
    rle = lambda m: [] if type(m) == list and not m else masks_to_rle(m, size)
    gts, prs = [rle(g) for g in gt_list], [rle(p) for p in pred_list]
    sc = [_score_array(s) for s in scores]
    for i, (p, s) in enumerate(zip(prs, sc)):
        if len(s) != len(p):
            raise ValueError('image %d: %d scores for %d predictions' % (i, len(s), len(p)))
    n, K, T = len(gts), len(s_th), len(i_th)
    levels, kept = _image_levels(sc, s_sorted)
    r = engine.eval_images_sweep(gts, prs, levels, K, i_sorted)
    # back to the caller's order of thresholds
    order = lambda a, ks: _reorder(_reorder(a, s_pos, ks), i_pos, ks + 1)
    totals, seg_totals = order(r.totals, 0), order(r.seg_totals, 0)
    tp, fp, fn = (totals[..., c].astype(np.float64) for c in range(3))
    with np.errstate(invalid='ignore', divide='ignore'):
        out = {'score_thresholds': s_th, 'iou_thresholds': i_th, 'n_pred': _reorder(kept, s_pos, 1), 'totals': totals,
               'seg_totals': seg_totals, 'det_precision': tp / (tp + fp), 'det_recall': tp / (tp + fn)}
    counts = order(r.counts, 1).astype(np.int64)
    seg = order(r.seg, 1)
    for c, k in enumerate(('det_tp', 'det_fp', 'det_fn')):
        out[k] = counts[..., c]
    for c, k in enumerate(('seg_tp', 'seg_fp', 'seg_fn')):
        out[k] = seg[..., c]
    return out


def merge_boxes(box1, box2):
    """Smallest [r1, r2, c1, c2] box enclosing both (analyze.py:342-376)."""
    r11, r12, c11, c12 = box1
    r21, r22, c21, c22 = box2
    return np.array([min(r11, r21), max(r12, r22), min(c11, c21), max(c12, c22)])


def _min_euclid(a, b):
    """Minimum Euclidean distance from each row of *a* (n x 2) to the rows of *b* (m x 2), float64
    tensor (analyze.py:379-413).  Tensor plumbing on whatever device the inputs live on; the
    mask-level path (mask_edge_distance) uses the dedicated kernel instead of an n x m table."""
    a = a.unsqueeze(1)
    square_diffs = torch.pow(a.double() - b.double(), 2)
    distances = torch.sqrt(square_diffs.sum(axis=2))
    return distances.min(axis=1)[0]


def mask_edge_distance(gt_mask, pred_mask, gt_box, pred_box, matches, device='auto'):
    """Distances from false-positive pixels to the nearest ground-truth pixel and from
    false-negative pixels to the nearest predicted pixel, per matched pair, inside the merged
    box of the pair (analyze.py:416-499).  Boxes are index boxes [r1, r2, c1, c2].

    Returns two lists of float64 tensors in the reference's order (np.where / torch.where order
    of the cropped window).  device='cuda' returns CUDA tensors, anything else CPU tensors --
    the arithmetic always runs on the GPU (csrc/edge.cu); the reference's n x m distance table
    is replaced by a search over boundary pixels, which gives the same minima."""
    if type(gt_mask) == RLEMasks:
        gt_mask = gt_mask.rle
    if type(pred_mask) == RLEMasks:
        pred_mask = pred_mask.rle
    matches = np.asarray(matches).reshape(-1, 2)
    n = len(matches)
    if n == 0:
        return [], []
    _check_same_size(gt_mask, pred_mask)
    h, w = int(gt_mask[0]['size'][0]), int(gt_mask[0]['size'][1])
    gi, pi = matches[:, 0].astype(np.int64), matches[:, 1].astype(np.int64)
    ug, inv_g = np.unique(gi, return_inverse=True)
    up, inv_p = np.unique(pi, return_inverse=True)
    table = engine.table_from_rle([gt_mask[i] for i in ug] + [pred_mask[i] for i in up])
    win = np.zeros((n, 4), np.int64)
    for k in range(n):
        box = merge_boxes(gt_box[gi[k]], pred_box[pi[k]])
        if (np.asarray(box) < 0).any():
            raise ValueError('negative box indices are not supported')
        r1, r2, c1, c2 = [int(v) for v in box]
        win[k] = (min(r1, h), min(r2, h), min(c1, w), min(c2, w))     # numpy slicing clips at the frame
    if (win[:, 1] - win[:, 0]).max() > 32767 or (win[:, 3] - win[:, 2]).max() > 32767:
        raise ValueError('merged boxes larger than 32767 pixels a side are not supported')
    counts, d_fp, d_fn, off_fp, off_fn = engine.edge_distances(table, inv_g, len(ug) + inv_p, win)
    on_gpu = str(device).lower() == 'cuda'
    if not on_gpu:
        d_fp, d_fn = d_fp.cpu(), d_fn.cpu()
    FP = [d_fp[off_fp[k]:off_fp[k + 1]].clone() for k in range(n)]
    FN = [d_fn[off_fn[k]:off_fn[k + 1]].clone() for k in range(n)]
    return FP, FN


_DET_COLORS = {'TP': (0.5, 0., 1.), 'FP': (0., 1., 1.), 'FN': (1., 0., 0.)}


def _boxes_array(instances):
    b = instances.boxes
    return b if type(b) == np.ndarray else b.tensor.numpy()


def det_perf_iset(gt, pred, match_results=None, colormap=None, tp_gt=False):
    """Detection outcome of an image as one InstanceSet for display (analyze.py:502-586): the matched
    instances (taken from the predictions, or from the ground truth with *tp_gt*), then the
    unmatched predictions (FP), then the unmatched ground truth (FN), each group in its colour.
    Returns ``(iset, colormap)`` when no colormap was passed, else ``iset``.  Host bookkeeping over
    the matcher's output."""
    if match_results is None:
        match_results = rle_instance_matcher(gt, pred)
    default_colors = colormap is None
    if default_colors:
        colormap = {k: np.asarray(v, np.float64) for k, v in _DET_COLORS.items()}
    size = gt.instances.image_size
    sources = {'gt': (masks_to_rle(gt.instances.masks, size), _boxes_array(gt.instances)),
               'pred': (masks_to_rle(pred.instances.masks, size), _boxes_array(pred.instances))}
    tp = match_results['tp']
    parts = [('TP', 'gt', tp[:, 0]) if tp_gt else ('TP', 'pred', tp[:, 1]),
             ('FP', 'pred', match_results['fp']),
             ('FN', 'gt', match_results['fn'])]
    masks, boxes, colors = [], [], []
    for kind, side, idx in parts:
        rles, bb = sources[side]
        masks += [rles[i] for i in idx]
        boxes.append(bb[idx])
        colors.append(np.tile(colormap[kind], (len(idx), 1)))
    masks = RLEMasks(masks)
    iset = InstanceSet()
    iset.instances = Instances(image_size=masks.rle[0]['size'], masks=masks, boxes=np.concatenate(boxes, axis=0),
                               colors=np.concatenate(colors, axis=0))
    return (iset, colormap) if default_colors else iset


_SEG_COLORS_ALL = np.array([[0., 0., 0.], [0.153, 0.153, 0.000], [0.286, 1., 0.], [1., 0.857, 0.], [1., 0., 0.],
                            [0., 0.571, 1.], [0., 1., 0.571], [0.285, 0., 1.]])
_SEG_COLORS_REDUCED = np.array([[0.5, 0., 1.], [1., 0., 0.], [0., 1., 1.], [1., 1., 0.]])


def seg_perf_iset(gt_masks, pred_masks, match_results=None, mode='reduced'):
    """Pixel-level TP / FN / FP classes of the matched pairs as an InstanceSet of class masks
    (analyze.py:589-699).  The reference decodes every mask to a full frame, forms the three
    boolean stacks, OR-reduces them and re-encodes; here the projection, the class logic and the
    RLE encoding all run on packed bits on the GPU (csrc/rle_encode.cu), nothing is decoded."""
    if match_results is None:
        match_results = rle_instance_matcher(gt_masks, pred_masks)
    g_rle, p_rle = masks_to_rle(gt_masks), masks_to_rle(pred_masks)
    _check_same_size(g_rle, p_rle)
    h, w = int(g_rle[0]['size'][0]), int(g_rle[0]['size'][1])
    tp_idx = np.asarray(match_results['tp']).reshape(-1, 2)
    gi, pi = tp_idx[:, 0].astype(np.int64), tp_idx[:, 1].astype(np.int64)
    ug, inv_g = np.unique(gi, return_inverse=True)
    up, inv_p = np.unique(pi, return_inverse=True)
    table = engine.table_from_rle([g_rle[i] for i in ug] + [p_rle[i] for i in up])
    rles = engine.project_pairs(table, inv_g, len(ug) + inv_p, h, w, 'all' if mode == 'all' else 'reduced')
    if mode == 'all':
        colors = [_SEG_COLORS_ALL[1:], ['Other', 'TP', 'FN', 'TP+FN', 'FP', 'TP+FP', 'FN+FP', 'TP+FN+FP']]
    else:
        colors = [_SEG_COLORS_REDUCED, ['TP', 'FN', 'FP', 'other']]
    masks = RLEMasks(rles)
    i = InstanceSet()
    i.instances = Instances(image_size=masks.rle[0]['size'], **{'masks': masks, 'colors': colors[0],
                                                                'boxes': np.zeros((len(masks), 4))})
    return i, colors
