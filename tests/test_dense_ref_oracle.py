"""CPU tests of tests/_dense_ref.py, the exact reference of the dense intersection kernels: its sparse-product
intersections against the oracle's run-walk merges, its IoU rows against the oracle's rleIou and the reference's
matcher (tests/_util.py one-shot forms and oracle/ampis_ref.py loops), its satellite rows against the reference's
satellite matcher -- with empty masks, duplicate masks (ties), and images without rows or columns."""
import numpy as np
import pytest

from tests import _dense_ref as D
from tests import _util as U


def _enc(rle, frames):
    return [rle.encode(np.asfortranarray(f.astype(np.uint8))) for f in frames]


def _masks(rng, n, h, w):
    """Blobs, plus masks of the kinds kernels trip on: empty, full frame, one pixel, stripes that wrap column ends,
    the last pixel only, noise."""
    m = U.rand_masks(rng, n, h, w, p_empty=0.1)
    for i, k in enumerate(rng.integers(0, 9, n)):
        if k == 0:
            m[i] = True
        elif k == 1:
            m[i] = False
            m[i, rng.integers(0, h), rng.integers(0, w)] = True
        elif k == 2:
            m[i] = False
            m[i, rng.integers(0, h):, rng.integers(0, w):] = True
        elif k == 3:
            m[i] = False
            m[i, -1, -1] = True
        elif k == 4:
            m[i] = rng.random((h, w)) < 0.5
    return m


@pytest.mark.parametrize('seed', range(4))
def test_intersections_and_areas_equal_the_oracle(seed):
    """I = A · Bᵀ equals merge_area(intersect=True) of every pair, from bool stacks, RLE dicts and run counts alike;
    areas equal rle.area."""
    from oracle import cocomask as rle
    rng = np.random.default_rng(seed)
    h, w = int(rng.integers(1, 60)) | 1, int(rng.integers(1, 60)) | 1          # odd frames
    G, P = int(rng.integers(0, 14)), int(rng.integers(0, 14))
    rows, cols = _masks(rng, G, h, w), _masks(rng, P, h, w)
    er, ec = _enc(rle, rows), _enc(rle, cols)
    I = D.intersections(rows, cols)
    assert I.shape == (G, P) and I.dtype == np.int64
    want = np.array([[int(rle.merge_area(a, b, intersect=True)) for b in ec] for a in er], np.int64).reshape(G, P)
    assert np.array_equal(I, want)
    assert np.array_equal(D.intersections(er, ec), want)
    counts = lambda es: [D.counts_of(e) for e in es]
    assert np.array_equal(D.intersections(counts(er), counts(ec), hw=h * w), want)
    assert np.array_equal(D.areas(rows), rle.area(er).astype(np.int64).reshape(-1))
    assert np.array_equal(D.areas(er), D.areas(rows))


@pytest.mark.parametrize('seed', range(4))
def test_iou_rows_equal_the_oracle_matcher(seed):
    """The IoU matrix equals the oracle's rleIou bit for bit; the rows equal match_from_iou and the reference's loop
    over 80-column chunks (first strict maximum, -1 where every IoU is 0), including duplicate columns."""
    from oracle import ampis_ref as R
    from oracle import cocomask as rle
    rng = np.random.default_rng(10 + seed)
    h, w = int(rng.integers(3, 50)) | 1, int(rng.integers(3, 50)) | 1
    G, P = int(rng.integers(1, 30)), int(rng.integers(1, 100))
    rows, cols = _masks(rng, G, h, w), _masks(rng, P, h, w)
    dup = rng.integers(0, P, P // 3)
    cols[rng.integers(0, P, len(dup))] = cols[dup]                  # duplicate columns: IoU ties
    er, ec = _enc(rle, rows), _enc(rle, cols)
    I = D.intersections(er, ec)
    best, inter, top, iou = D.rows_iou(I, D.areas(er), D.areas(ec))
    assert np.array_equal(iou, U.iou_matrix_one_shot(rle, er, ec))
    for th in (0.0, 0.3, 0.5, 0.75):
        want = U.match_from_iou(iou, th)
        m = top > th
        assert np.array_equal(np.stack([np.nonzero(m)[0], best[m]], axis=1).reshape(-1, 2),
                              np.asarray(want['tp']).reshape(-1, 2))
        assert np.array_equal(top[m], want['iou'])
        lit = R.piecewise_rle_match(er, ec, th)
        assert np.array_equal(np.asarray(lit['tp']).reshape(-1, 2), np.asarray(want['tp']).reshape(-1, 2))
        assert np.array_equal(lit['iou'], top[m])
    assert np.array_equal(inter, np.where(best >= 0, I[np.arange(G), np.maximum(best, 0)], 0))


@pytest.mark.parametrize('seed', range(4))
def test_satellite_rows_equal_the_oracle_matcher(seed):
    """First maximum of I from index 0, score I / area(s) with NaN for zero-area satellites: equal to the one-shot
    form and to the reference's S x N loop of merges, with duplicate particles and empty satellites."""
    from oracle import ampis_ref as R
    from oracle import cocomask as rle
    rng = np.random.default_rng(20 + seed)
    h, w = int(rng.integers(3, 50)) | 1, int(rng.integers(3, 50)) | 1
    S, P = int(rng.integers(2, 25)), int(rng.integers(1, 40))
    sats, parts = _masks(rng, S, h, w), _masks(rng, P, h, w)
    sats[rng.integers(0, S, 2)] = False                              # zero-area satellites
    parts[rng.integers(0, P, P // 2)] = parts[rng.integers(0, P, P // 2)]    # duplicate particles
    parts[-1, 0, :] = True
    sats[0] = parts[-1]                                              # one satellite certainly matches
    es, ep = _enc(rle, sats), _enc(rle, parts)
    I = D.intersections(es, ep)
    best, inter, score = D.rows_sat(I, D.areas(es))
    assert np.array_equal(inter, I[np.arange(S), best])
    zero = D.areas(es) == 0
    assert np.isnan(score[zero]).all() and (best[zero] == 0).all() and not np.isnan(score[~zero]).any()
    for th in (0.0, 0.5, 0.9):
        for want in (U.satellite_match_one_shot(rle, ep, es, th), R.rle_satellite_match(ep, es, th)):
            with np.errstate(invalid='ignore'):
                m = score > th
            assert np.array_equal(np.stack([np.nonzero(m)[0], best[m]], axis=1), want['satellite_matches'])
            assert np.array_equal(score[m], want['intersection_scores'])
            assert np.array_equal(np.nonzero(~m)[0], want['satellites_unmatched'])


def test_rows_of_images_without_rows_or_columns():
    """P = 0: every row -1 with intersection 0 (satellite scores 0 / area, NaN for an empty satellite); G = 0: empty."""
    I = np.zeros((3, 0), np.int64)
    best, inter, top, iou = D.rows_iou(I, [5, 0, 7], [])
    assert best.tolist() == [-1] * 3 and inter.tolist() == [0] * 3 and top.tolist() == [0.0] * 3 and iou.shape == (3, 0)
    best, inter, score = D.rows_sat(I, [5, 0, 7])
    assert best.tolist() == [-1] * 3 and inter.tolist() == [0] * 3
    assert np.array_equal(score, [0.0, np.nan, 0.0], equal_nan=True)
    for b in (D.rows_iou(np.zeros((0, 4), np.int64), [], [1, 2, 3, 4])[0], D.rows_sat(np.zeros((0, 4), np.int64), [])[0]):
        assert b.shape == (0,)
    assert D.intersections(np.zeros((0, 5, 3), bool), np.ones((2, 5, 3), bool)).shape == (0, 2)
    assert D.intersections(np.ones((2, 5, 3), bool), np.zeros((0, 5, 3), bool)).shape == (2, 0)
