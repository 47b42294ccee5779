"""Reference of the many-image evaluation entry (``ampis_eval_images_host`` / ``engine.eval_images``) in numpy and
scipy, sharing none of its code: every mask is decoded into pixel indices, the intersections of an image are the
sparse product I = A B^T of its incidence matrices (masks x pixels), and the per-row results are read off I with the
conventions of DESIGN.md section 3:

- area = row sums of the incidence matrix; bbox = (x0, y0, x1, y1) inclusive, (0, 0, -1, -1) for an empty mask;
- IoU mode: IoU = I / (a_r + a_c - I) in float64, 0.0 where I == 0; best_col = first maximum under strict ``>``
  starting from 0.0, -1 when no column overlaps the row;
- satellite mode: best_col = first maximum of I (0 when no column overlaps, -1 without columns), score = I / a_r with
  numpy's float64 division (NaN for a zero-area satellite);
- TP / FP / FN per image and threshold: a row is a true positive when its score is strictly above the threshold
  (thresholds as stored, e.g. ``batch.COCO_THRESHOLDS``); FP = columns no true positive claims; FN = the other rows.
"""
import numpy as np
import scipy.sparse as sp

from oracle import cocomask as rle

MODE_IOU, MODE_SAT = 0, 1


def _counts(m):
    c = m['counts']
    return rle.counts_from_string(c if isinstance(c, bytes) else bytes(c, 'ascii') if isinstance(c, str) else bytes(c))


def pixels(m):
    """Column-major pixel indices of one compressed RLE dict, and whether its runs sum to h * w."""
    cnt = _counts(m).astype(np.int64)
    h, w = int(m['size'][0]), int(m['size'][1])
    ends = np.cumsum(cnt)
    ones = cnt[1::2]
    starts = (ends - cnt)[1::2]
    total = int(ones.sum())
    idx = np.arange(total, dtype=np.int64) + np.repeat(starts - (np.cumsum(ones) - ones), ones)
    return idx, int(ends[-1]) if len(ends) else 0, h, w


def incidence(masks, hw):
    """(CSR incidence matrix masks x pixels, area int64, bbox int32 [n, 4], valid bool [n]) of masks of size hw."""
    h, w = hw
    ind, ptr = [], [0]
    n = len(masks)
    area = np.zeros(n, np.int64)
    bbox = np.tile(np.array([0, 0, -1, -1], np.int32), (n, 1))
    valid = np.ones(n, bool)
    for k, m in enumerate(masks):
        idx, total, mh, mw = pixels(m)
        assert (mh, mw) == (h, w)
        valid[k] = total == h * w
        ind.append(idx)
        ptr.append(ptr[-1] + len(idx))
        area[k] = len(idx)
        if len(idx):
            x, y = idx // h, idx % h
            bbox[k] = [x.min(), y.min(), x.max(), y.max()]
    data = np.ones(ptr[-1], np.int64)
    A = sp.csr_matrix((data, np.concatenate(ind) if ind else np.zeros(0, np.int64), np.asarray(ptr, np.int64)),
                      shape=(n, max(h * w, 1)))
    return A, area, bbox, valid


def image(rows, cols, mode):
    """Per-row and per-mask results of one image (rows then columns in the mask arrays)."""
    G, P = len(rows), len(cols)
    hw = tuple(int(v) for v in (rows or cols)[0]['size']) if G + P else (0, 0)
    A, a_r, bb_r, ok_r = incidence(rows, hw)
    B, a_c, bb_c, ok_c = incidence(cols, hw)
    best_col = np.full(G, -1, np.int32)
    best_inter = np.zeros(G, np.uint32)
    best_score = np.zeros(G, np.float64)
    if G and P:
        I = (A @ B.T).tocoo()
        r, c, v = I.row.astype(np.int64), I.col.astype(np.int64), I.data.astype(np.int64)
        keep = v > 0
        r, c, v = r[keep], c[keep], v[keep]
        if mode == MODE_IOU:
            s = v / (a_r[r] + a_c[c] - v).astype(np.float64)
        else:
            s = v.astype(np.float64)
        order = np.lexsort((c, -s, r))              # per row: highest score first, lowest column among equals
        r, c, v = r[order], c[order], v[order]
        first = np.ones(len(r), bool)
        first[1:] = r[1:] != r[:-1]
        rr = r[first]
        best_col[rr] = c[first]
        best_inter[rr] = v[first]
        if mode == MODE_IOU:
            best_score[rr] = s[order][first]
        else:
            best_col[best_col < 0] = 0              # np.argmax of a row of zeros
    if mode == MODE_SAT:
        with np.errstate(invalid='ignore', divide='ignore'):
            best_score = best_inter.astype(np.float64) / a_r.astype(np.float64)
    return dict(best_col=best_col, best_inter=best_inter, best_score=best_score,
                area=np.concatenate([a_r, a_c]).astype(np.uint32), bbox=np.concatenate([bb_r, bb_c]),
                status=(~np.concatenate([ok_r, ok_c])).astype(np.int32), n_rows=G, n_cols=P, hw=hw)


def counts(res, thresholds):
    """int32 [T, 3] TP / FP / FN of one image result of image() (IoU mode) at every threshold."""
    out = np.zeros((len(thresholds), 3), np.int32)
    G, P = res['n_rows'], res['n_cols']
    for t, th in enumerate(thresholds):
        m = res['best_score'] > th
        tp = int(m.sum())
        out[t] = [tp, P - len(np.unique(res['best_col'][m])), G - tp]
    return out


def dataset(rows_lists, cols_lists, mode, thresholds=None):
    """The outputs of the many-image entry for a list of images, concatenated in image order like
    engine.ImagesRows: best_col / best_inter / best_score over all rows, area / bbox / status over all masks, and
    (IoU mode, thresholds given) grp_counts int32 [n_images, T, 3] and totals int64 [T, 3]."""
    per = [image(list(r), list(c), mode) for r, c in zip(rows_lists, cols_lists)]
    cat = lambda k, dt, shape: np.concatenate([p[k] for p in per]) if per else np.zeros(shape, dt)
    out = dict(best_col=cat('best_col', np.int32, 0), best_inter=cat('best_inter', np.uint32, 0),
               best_score=cat('best_score', np.float64, 0), area=cat('area', np.uint32, 0),
               bbox=cat('bbox', np.int32, (0, 4)), status=cat('status', np.int32, 0), images=per)
    if thresholds is not None:
        gc = np.stack([counts(p, thresholds) for p in per]) if per else np.zeros((0, len(thresholds), 3), np.int32)
        out['grp_counts'] = gc
        out['totals'] = gc.astype(np.int64).sum(axis=0)
    return out
