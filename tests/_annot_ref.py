"""Exact references of the annotation kernels -- labelling (label.cu), rleFrPoly (poly.cu poly_to_rle_kernel) and
boundary distances (edge.cu) -- that stay fast at frame scale, in numpy and scipy only, sharing no code with the
package.

The oracle's own forms cannot serve at these sizes: R.annotations_from_label_image makes one full-frame pass per
label, and R.mask_edge_distance builds an n x m distance table per pair.  The forms below cost O(h·w log) for a whole
label image and one Euclidean distance transform per pair; tests/test_annot_ref_oracle.py pins each to the oracle.

* Label images.  'binary': scipy.ndimage.label with a 3x3 structure, renumbered by the raster index of each
  component's first pixel (scipy's own numbering is not relied on).  'label': the distinct values in ascending
  order, a leading 0 skipped.  Per label: the tight box and the RLE counts read off the segments of equal value of
  the column-major flattening, sorted stably by label.
* Edge distances.  Per pair, both masks cropped to the merged window (numpy slicing clips it at the frame); the
  distance transform of the other mask's complement gives, for every false-positive (false-negative) pixel in
  row-major order, a nearest pixel of the other mask; the distance is np.sqrt of the exact integer squared distance.
* rleFrPoly.  The x5 up-sampled DDA boundary and its crossings of pixel-column centres, restated from
  maskapi_ref.c with the same double operations; positions >= h·w are dropped as the kernel drops them, so the
  count is the one the kernel compares with its limit of 8192.  Counts follow by the parity rule of DESIGN.md §3:
  a position survives iff it occurs an odd number of times, and h·w closes the last run."""
import numpy as np
import scipy.ndimage as ndi


# ---- label images -> instances ------------------------------------------------------------------------------------

def dense_labels(ann, binary):
    """(int64 [h, w] labels 0..n in the reference's instance order, n)."""
    ann = np.asarray(ann)
    assert ann.ndim == 2
    if binary:
        lab, n = ndi.label(ann.astype(bool), structure=np.ones((3, 3), int))
        vals, first = np.unique(lab.ravel(), return_index=True)
        keep = vals != 0
        vals, first = vals[keep], first[keep]
        new = np.zeros(n + 1, np.int64)
        new[vals[np.argsort(first)]] = np.arange(1, len(vals) + 1)
        return new[lab], int(len(vals))
    vals, inv = np.unique(ann.ravel(), return_inverse=True)
    inv = inv.reshape(ann.shape).astype(np.int64)
    if len(vals) and vals[0] == 0:
        return inv, int(len(vals) - 1)
    return inv + 1, int(len(vals))


def label_instances(ann, binary):
    """Instances of an annotation image in the reference's order: (int64 [n, 4] boxes x0, y0, x1, y1 with inclusive
    maxima, as engine.label_image_to_instances returns them; list of n uint32 RLE count arrays)."""
    dense, n = dense_labels(ann, binary)
    h, w = dense.shape
    hw = h * w
    boxes = np.zeros((n, 4), np.int64)
    for i, sl in enumerate(ndi.find_objects(dense, max_label=n)):
        boxes[i] = (sl[1].start, sl[0].start, sl[1].stop - 1, sl[0].stop - 1)
    if n == 0:
        return boxes, []
    f = dense.ravel(order='F')                                   # column-major: COCO pixel order
    start = np.flatnonzero(np.r_[True, f[1:] != f[:-1]])
    end = np.r_[start[1:], hw]
    val = f[start]
    fg = val != 0
    start, end, val = start[fg], end[fg], val[fg]
    order = np.argsort(val, kind='stable')
    start, end, val = start[order], end[order], val[order]
    k = np.bincount(val, minlength=n + 1)[1:]                    # segments per label, every label has one
    # per label l the boundary list [0, s_1, e_1, ..., s_k, e_k, h·w]; its differences are the counts
    glen = 2 * k + 2
    g0 = np.zeros(n, np.int64)
    np.cumsum(glen[:-1], out=g0[1:])
    E = np.empty(int(glen.sum()), np.int64)
    E[g0] = 0
    E[g0 + glen - 1] = hw
    b = np.stack([start, end], axis=1).ravel()
    E[np.arange(len(b)) + 2 * np.repeat(val - 1, 2) + 1] = b
    D = np.diff(E)
    keep = np.ones(len(D), bool)
    keep[(g0 + glen - 1)[:-1]] = False                           # h·w of one label -> 0 of the next
    last = g0 + glen - 2
    ends_frame = D[last] == 0                                    # a label holding the last pixel has no closing 0
    keep[last[ends_frame]] = False
    D = D[keep].astype(np.uint32)
    return boxes, np.split(D, np.cumsum(2 * k + 1 - ends_frame)[:-1])


# ---- boundary distances -------------------------------------------------------------------------------------------

def _window(gt_box, pred_box, h, w):
    """The merged box [r1, r2, c1, c2] of the pair, clipped at the frame as numpy slicing clips it."""
    r1, r2 = int(min(gt_box[0], pred_box[0])), int(max(gt_box[1], pred_box[1]))
    c1, c2 = int(min(gt_box[2], pred_box[2])), int(max(gt_box[3], pred_box[3]))
    assert min(r1, r2, c1, c2) >= 0, 'negative box indices'
    return min(r1, h), min(r2, h), min(c1, w), min(c2, w)


def boundary(m):
    """Pixels of the bool crop *m* with a 4-neighbour outside the set or outside the crop (the kernel's candidates)."""
    inner = np.zeros_like(m)
    inner[1:-1, 1:-1] = m[1:-1, 1:-1] & m[:-2, 1:-1] & m[2:, 1:-1] & m[1:-1, :-2] & m[1:-1, 2:]
    return m & ~inner


def _crops(gt, pred, gt_box, pred_box, pair):
    gi, pi = int(pair[0]), int(pair[1])
    h, w = gt[gi].shape
    r1, r2, c1, c2 = _window(gt_box[gi], pred_box[pi], h, w)
    return np.asarray(gt[gi][r1:r2, c1:c2], bool), np.asarray(pred[pi][r1:r2, c1:c2], bool)


def edge_counts(gt, pred, gt_box, pred_box, matches):
    """int64 [n, 4] per pair: false positives, false negatives, boundary pixels of gt and of pred in the window --
    the queries and the candidates of the kernel.  gt, pred: sequences of bool [h, w] masks; boxes [r1, r2, c1, c2]."""
    out = []
    for pair in np.asarray(matches).reshape(-1, 2):
        g, p = _crops(gt, pred, gt_box, pred_box, pair)
        out.append((int((p & ~g).sum()), int((g & ~p).sum()), int(boundary(g).sum()), int(boundary(p).sum())))
    return np.asarray(out, np.int64).reshape(-1, 4)


def _nearest(q, other):
    if not q.any():
        return np.zeros(0, np.float64)
    if not other.any():
        return None
    _, (ir, ic) = ndi.distance_transform_edt(~other, return_indices=True)
    rr, cc = np.nonzero(q)
    dr = rr.astype(np.int64) - ir[rr, cc]
    dc = cc.astype(np.int64) - ic[rr, cc]
    return np.sqrt((dr * dr + dc * dc).astype(np.float64))


def edge_distances(gt, pred, gt_box, pred_box, matches):
    """(fp, fn): per pair the float64 distances of R.mask_edge_distance, in its order.  An entry is None where the
    pair has queries but no pixel of the other mask in the window (the public call raises RuntimeError there)."""
    fp_all, fn_all = [], []
    for pair in np.asarray(matches).reshape(-1, 2):
        g, p = _crops(gt, pred, gt_box, pred_box, pair)
        fp_all.append(_nearest(p & ~g, g))
        fn_all.append(_nearest(g & ~p, p))
    return fp_all, fn_all


# ---- rleFrPoly ----------------------------------------------------------------------------------------------------

def _trunc_to_int(v):
    """C's (int) truncation as maskapi_ref.c's trunc_to_int does it: out of range and NaN -> INT_MIN."""
    v = np.asarray(v, np.float64)
    ok = (v > -2147483649.0) & (v < 2147483648.0)
    return np.where(ok, np.trunc(np.where(ok, v, 0.0)), -2147483648.0).astype(np.int64)


def poly_crossings(xy, h, w):
    """int64 crossing positions (column-major pixel index < h·w) of one polygon [x0, y0, x1, y1, ...], in the order
    rleFrPoly records them.  len() is the count poly_to_rle_kernel compares with its limit."""
    xy = np.asarray(xy, np.float64).ravel()
    x = _trunc_to_int(5.0 * xy[0::2] + 0.5)
    y = _trunc_to_int(5.0 * xy[1::2] + 0.5)
    xs, ys, xe, ye = x, y, np.roll(x, -1), np.roll(y, -1)
    dx, dy = np.abs(xe - xs), np.abs(ys - ye)
    hor = dx >= dy
    flip = (hor & (xs > xe)) | (~hor & (ys > ye))
    xs, xe = np.where(flip, xe, xs), np.where(flip, xs, xe)
    ys, ye = np.where(flip, ye, ys), np.where(flip, ys, ye)
    L = np.maximum(dx, dy)
    with np.errstate(divide='ignore', invalid='ignore'):
        s = np.where(hor, (ye - ys).astype(np.float64) / dx, (xe - xs).astype(np.float64) / dy)
    n_pts = L + 1
    e = np.repeat(np.arange(len(x)), n_pts)
    d = np.arange(int(n_pts.sum())) - np.repeat(np.cumsum(n_pts) - n_pts, n_pts)
    t = np.where(flip[e], L[e] - d, d)
    with np.errstate(invalid='ignore'):
        along = _trunc_to_int(np.where(hor[e], ys[e], xs[e]) + s[e] * t + 0.5)
    u = np.where(hor[e], t + xs[e], along)
    v = np.where(hor[e], along, t + ys[e])
    u0, u1, v0, v1 = u[:-1], u[1:], v[:-1], v[1:]
    moved = u1 != u0
    xd = np.where(u1 < u0, u1, u1 - 1).astype(np.float64)
    xd = (xd + 0.5) / 5.0 - 0.5
    yd = np.minimum(v0, v1).astype(np.float64)
    yd = np.ceil(np.clip((yd + 0.5) / 5.0 - 0.5, 0.0, float(h)))
    ok = moved & (np.floor(xd) == xd) & (xd >= 0) & (xd <= w - 1)
    pos = xd[ok].astype(np.int64) * int(h) + yd[ok].astype(np.int64)
    return pos[pos < int(h) * int(w)]


def counts_from_crossings(pos, h, w):
    """uint32 RLE counts from crossing positions: odd multiplicity survives, h·w closes the last run."""
    vals, mult = np.unique(np.asarray(pos, np.int64), return_counts=True)
    kept = vals[mult % 2 == 1]
    return np.diff(np.r_[0, kept, int(h) * int(w)]).astype(np.uint32)


def poly_counts(xy, h, w):
    return counts_from_crossings(poly_crossings(xy, h, w), h, w)
