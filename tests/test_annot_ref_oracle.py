"""CPU tests of tests/_annot_ref.py, the scalable references of the annotation kernels, against the oracle on small
inputs: label instances against R.annotations_from_label_image (both formats), edge distances against
R.mask_edge_distance (shared masks, windows sticking out of the frame, empty sets), and rleFrPoly crossings turned
into counts by the parity rule against rle.frPyObjects (integer, half-integer and out-of-frame vertices, degenerate
rings).  Frames include empty and full images, 1 x n and n x 1 frames, and pixel 0 or the last pixel set."""
import numpy as np
import pytest

from tests import _annot_ref as A
from tests import _util as U


def _label_images(rng, h, w):
    """Random images of the kinds the labelling trips on, as int64 [h, w]."""
    yield np.zeros((h, w), np.int64)
    yield np.ones((h, w), np.int64)
    for p in (0.2, 0.45, 0.7):
        yield (rng.random((h, w)) < p).astype(np.int64)
    a = np.zeros((h, w), np.int64)
    a[0, 0] = 1
    yield a
    a = np.zeros((h, w), np.int64)
    a[-1, -1] = 1
    yield a
    a = (rng.random((h, w)) < 0.4).astype(np.int64)
    a[0, 0] = a[-1, -1] = 1
    yield a
    yield (np.add.outer(np.arange(h), np.arange(w)) % 2 == 0).astype(np.int64)       # checkerboard
    a = np.zeros((h, w), np.int64)
    a[:, w // 2:] = 1                                            # full height: runs cross column ends
    yield a
    vals = np.array([0, 0, 3, 4, 9, 500, 70000, (1 << 24) - 1])
    yield rng.choice(vals, size=(h, w))
    yield rng.choice(vals[2:], size=(h, w))                      # no 0
    yield rng.integers(0, 4, (h, w)) * 7


SHAPES = [(1, 1), (1, 37), (37, 1), (2, 2), (5, 7), (16, 16), (33, 65), (64, 33), (97, 130)]


@pytest.mark.parametrize('h,w', SHAPES)
def test_label_instances_equal_the_oracle(h, w):
    from oracle import ampis_ref as R
    from oracle import cocomask as rle
    rng = np.random.default_rng(h * 1000 + w)
    for k, img in enumerate(_label_images(rng, h, w)):
        for binary in (True, False):
            boxes, counts = A.label_instances(img, binary)
            want = R.annotations_from_label_image(img, binary)
            tag = (h, w, k, binary)
            assert len(counts) == len(want) == len(boxes), tag
            assert [rle.string_from_counts(c) for c in counts] == [m['counts'] for _, m in want], tag
            if want:
                assert boxes.dtype == np.int64
                assert np.array_equal(boxes.astype(np.float64), np.stack([b for b, _ in want])), tag
            for c in counts:
                assert c.dtype == np.uint32 and int(c.sum()) == h * w, tag


def test_label_instances_known_answer():
    """Components numbered by their first pixel in raster order, diagonal neighbours joined; boxes x0, y0, x1, y1;
    counts in column-major order with a leading zero-length run when pixel 0 is set."""
    img = np.array([[1, 0, 0, 1],
                    [0, 1, 0, 0],
                    [1, 0, 0, 1]])
    dense, n = A.dense_labels(img, True)
    assert n == 3 and dense.tolist() == [[1, 0, 0, 2], [0, 1, 0, 0], [1, 0, 0, 3]]
    boxes, counts = A.label_instances(img, True)
    assert boxes.tolist() == [[0, 0, 1, 2], [3, 0, 3, 0], [3, 2, 3, 2]]
    assert [c.tolist() for c in counts] == [[0, 1, 1, 1, 1, 1, 7], [9, 1, 2], [11, 1]]
    dense, n = A.dense_labels(np.array([[5, 0], [0, 9]]), False)
    assert n == 2 and dense.tolist() == [[1, 0], [0, 2]]
    dense, n = A.dense_labels(np.array([[5, 7], [7, 9]]), False)
    assert n == 3 and dense.tolist() == [[1, 2], [2, 3]]


def _encode(rle, masks):
    return [rle.encode(np.asfortranarray(m.astype(np.uint8))) for m in masks]


@pytest.mark.parametrize('seed', range(6))
def test_edge_distances_equal_the_oracle(seed):
    from oracle import ampis_ref as R
    from oracle import cocomask as rle
    rng = np.random.default_rng(100 + seed)
    h, w = [(1, 40), (40, 1), (23, 31), (48, 64), (61, 47), (9, 130)][seed]
    n = 8
    g = U.rand_masks(rng, n, h, w, p_empty=0.1)
    p = np.roll(g, int(rng.integers(1, 4)), axis=2) | (rng.random((n, h, w)) < 0.03)
    g[0], p[0] = True, False                       # FN only, no pred pixel: a None entry
    g[1, 0, 0] = p[1, -1, -1] = True
    g[2] = False
    g[2, -1, -1] = True
    p[2] = True                                    # full frame against one pixel
    gb, pb = [], []
    for masks, boxes in ((g, gb), (p, pb)):
        for m in masks:
            rr, cc = np.nonzero(m)
            if len(rr) == 0 or rng.random() < 0.3:   # loose box sticking out of the frame
                boxes.append([int(rng.integers(0, 3)), h + int(rng.integers(0, 6)), int(rng.integers(0, 3)),
                              w + int(rng.integers(0, 9))])
            else:
                boxes.append([rr.min(), rr.max() + 1, cc.min(), cc.max() + 1])
    gb, pb = np.asarray(gb), np.asarray(pb)
    # shared masks, reverse order, every mask against itself and its neighbour
    matches = np.array([[i, j] for i in range(n) for j in (i, (i + 1) % n)])[::-1]
    ge, pe = _encode(rle, g), _encode(rle, p)
    fp, fn = A.edge_distances(g, p, gb, pb, matches)
    counts = A.edge_counts(g, p, gb, pb, matches)
    n_none = 0
    for k, (gi, pi) in enumerate(matches):
        one = np.array([[gi, pi]])
        try:
            wfp, wfn = R.mask_edge_distance(ge, pe, gb, pb, one)
        except RuntimeError:
            assert fp[k] is None or fn[k] is None, k
            n_none += 1
            continue
        assert fp[k] is not None and fn[k] is not None, k
        assert fp[k].dtype == np.float64 and np.array_equal(fp[k], wfp[0]), k
        assert np.array_equal(fn[k], wfn[0]), k
        assert counts[k, 0] == len(fp[k]) and counts[k, 1] == len(fn[k]), k
    assert n_none >= 1


def test_boundary_is_the_set_minus_its_4_interior():
    m = np.zeros((6, 7), bool)
    m[1:5, 1:6] = True
    b = A.boundary(m)
    assert b.sum() == 2 * 4 + 2 * 5 - 4 and not b[2:4, 2:5].any()
    assert A.boundary(np.ones((3, 3), bool)).sum() == 8                # the crop edge counts as outside
    assert A.boundary(np.ones((1, 5), bool)).sum() == 5


def _polys(rng, h, w):
    """Polygons of the kinds rleFrPoly trips on."""
    out = []
    for _ in range(25):
        k = int(rng.integers(3, 40))
        kind = rng.integers(0, 4)
        if kind == 0:                              # integer vertices, also outside and on the frame edge
            pts = rng.integers(-4, max(h, w) + 5, (k, 2)).astype(np.float64)
        elif kind == 1:                            # half-integer vertices
            pts = rng.integers(-4, max(h, w) + 5, (k, 2)) + 0.5
        elif kind == 2:                            # star around a random centre, maybe far outside
            ang = np.sort(rng.uniform(0, 2 * np.pi, k))
            r = rng.uniform(0.2, 0.8) * max(h, w) * rng.uniform(0.3, 1.0, k)
            c = rng.uniform(-0.5, 1.5, 2) * [w, h]
            pts = np.stack([c[0] + r * np.cos(ang), c[1] + r * np.sin(ang)], 1)
        else:                                      # vertices snapped to the frame edges
            pts = rng.choice([0.0, 0.5, float(w) - 0.5, float(w)], (k, 2))
            pts[:, 1] = rng.choice([0.0, 0.5, float(h) - 0.5, float(h)], k)
        out.append(pts.ravel())
    out.append(np.array([0.0, 0.0, w, 0.0, w, h, 0.0, h]))                     # whole frame
    out.append(np.array([-3.0, -3.0, w + 3, -3.0, w + 3, h + 3, -3.0, h + 3]))  # beyond the frame
    out.append(np.array([w + 1.0, 0.0, w + 5.0, 0.0, w + 5.0, h]))              # wholly outside
    out.append(np.array([5.0, 5.0, 5.0, 5.0, 5.0, 5.0]))                        # a point
    out.append(np.array([1.0, 1.0, 7.0, 3.0, 1.0, 1.0, 7.0, 3.0]))             # a line walked twice
    out.append(np.array([0.0, 0.0, 3.0, 0.0, 3.0, 3.0, 3.0, 3.0, 0.0, 3.0]))   # a repeated vertex
    return out


@pytest.mark.parametrize('h,w', [(1, 1), (1, 30), (30, 1), (7, 9), (37, 53), (64, 64), (128, 96)])
def test_poly_crossings_to_counts_equal_frpyobjects(h, w):
    from oracle import cocomask as rle
    rng = np.random.default_rng(h * 7 + w)
    for i, xy in enumerate(_polys(rng, h, w)):
        pos = A.poly_crossings(xy, h, w)
        assert pos.dtype == np.int64 and (pos < h * w).all() and (pos >= 0).all()
        got = rle.string_from_counts(A.poly_counts(xy, h, w))
        assert got == rle.frPyObjects([list(xy)], h, w)[0]['counts'], (h, w, i)
