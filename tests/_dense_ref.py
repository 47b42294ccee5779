"""Exact reference of the dense intersection kernels (intersect_mma.cu, intersect_mma2.cu, intersect_tma.cu) and of
the per-row results read off their matrices (rows_from_imat_kernel), sharing no code with the package.

The intersection matrix is a sparse product of pixel-incidence matrices, I = A · Bᵀ in int64, where A[r, k] = 1 when
row mask r covers pixel k.  That is neither the AND+popc of the culled kernels nor the u8 contraction of the tensor
cores, and it stays fast on blob masks of 1024² frames.  The row rules are the reference's (DESIGN.md §3
"Exactness"): IoU = I / (a_r + a_c - I) in float64 with 0.0 where I = 0, the first strict maximum above 0 (best
column -1 when every IoU is 0); satellites take the first maximum of I from index 0, score I / area(s) (NaN for a
zero-area satellite) and best column -1 only when there are no particles."""
import numpy as np
import scipy.sparse as sp


def counts_of(rle_dict):
    """Run counts (uint32) of one compressed COCO RLE dict, through the oracle's string decoder."""
    from oracle import cocomask
    c = rle_dict['counts']
    return cocomask.counts_from_string(c if isinstance(c, bytes) else c.encode('ascii'))


def incidence(masks, hw=None):
    """CSR int64 [n, h·w] pixel incidence of n masks in column-major pixel order (the order of RLE counts).

    masks: bool [n, h, w]; a list of compressed RLE dicts; or a list of uint32 run-count arrays with hw = h·w."""
    if isinstance(masks, np.ndarray):
        n, h, w = masks.shape
        flat = masks.transpose(0, 2, 1).reshape(n, h * w)
        return sp.csr_matrix(flat.astype(np.int64))
    masks = list(masks)
    if masks and isinstance(masks[0], dict):
        hw = int(masks[0]['size'][0]) * int(masks[0]['size'][1])
        masks = [counts_of(m) for m in masks]
    assert hw is not None, 'run counts need the frame size h·w'
    starts, lens, per = [], [], np.zeros(len(masks), np.int64)
    for i, c in enumerate(masks):
        c = np.asarray(c, np.int64)
        end = np.cumsum(c)
        assert len(c) == 0 or end[-1] == hw, 'run counts of mask %d do not sum to h·w' % i
        s, ln = (end - c)[1::2], c[1::2]               # 1-runs: every second run, starting with the second
        starts.append(s)
        lens.append(ln)
        per[i] = ln.sum()
    s = np.concatenate(starts) if starts else np.zeros(0, np.int64)
    ln = np.concatenate(lens) if lens else np.zeros(0, np.int64)
    # pixel k of run j: s_j + (k - first pixel of run j); one repeat and one arange for all runs
    first = np.zeros(len(ln) + 1, np.int64)
    np.cumsum(ln, out=first[1:])
    cols = np.repeat(s - first[:-1], ln) + np.arange(int(first[-1]), dtype=np.int64)
    indptr = np.zeros(len(masks) + 1, np.int64)
    np.cumsum(per, out=indptr[1:])
    return sp.csr_matrix((np.ones(len(cols), np.int64), cols, indptr), shape=(len(masks), hw))


def intersections(rows, cols, hw=None):
    """Exact int64 [G, P] intersection matrix: rows and cols as incidence() takes them."""
    A, B = incidence(rows, hw), incidence(cols, hw)
    if A.shape[0] == 0 or B.shape[0] == 0:
        return np.zeros((A.shape[0], B.shape[0]), np.int64)
    assert A.shape[1] == B.shape[1], 'rows and columns of one image share one frame'
    return np.asarray((A @ B.T).toarray(), np.int64)


def areas(masks, hw=None):
    """int64 pixel counts of masks as incidence() takes them."""
    return np.asarray(incidence(masks, hw).sum(axis=1), np.int64).reshape(-1)


def rows_iou(I, area_r, area_c):
    """(best_col int64 [G], best_inter int64 [G], best_score float64 [G], iou float64 [G, P]) of the IoU rows."""
    I = np.asarray(I, np.int64)
    G, P = I.shape
    union = np.asarray(area_r, np.int64)[:, None] + np.asarray(area_c, np.int64)[None, :] - I
    with np.errstate(invalid='ignore', divide='ignore'):
        iou = np.where(I > 0, I.astype(np.float64) / union.astype(np.float64), 0.0)
    if P == 0:
        return np.full(G, -1, np.int64), np.zeros(G, np.int64), np.zeros(G), iou
    best = iou.argmax(axis=1)                     # first maximum
    top = iou[np.arange(G), best]
    best = np.where(top > 0, best, -1)            # strict '>' against a running maximum that starts at 0.0
    inter = np.where(best >= 0, I[np.arange(G), np.maximum(best, 0)], 0)
    return best.astype(np.int64), inter.astype(np.int64), top, iou


def rows_sat(I, area_r):
    """(best_col int64 [S], best_inter int64 [S], best_score float64 [S]) of the satellite rows."""
    I = np.asarray(I, np.int64)
    S, P = I.shape
    a = np.asarray(area_r, np.int64).astype(np.float64)
    if P == 0:
        best, inter = np.full(S, -1, np.int64), np.zeros(S, np.int64)
    else:
        best = I.argmax(axis=1).astype(np.int64)  # first maximum of I from index 0 (all-zero rows: index 0)
        inter = I[np.arange(S), best]
    with np.errstate(invalid='ignore', divide='ignore'):
        score = inter.astype(np.float64) / a      # 0 / 0 = NaN for a zero-area satellite
    return best, inter, score
