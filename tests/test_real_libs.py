"""Differential tests of the oracle (and, with a GPU, of the CUDA path) against the REAL third-party code the
reference calls -- pycocotools.mask (2.0.4 pinned at /root/reference/docker/env.yml:21) and scikit-image 0.18.3 --
whenever they are importable.  Neither is in this image nor installable offline (DESIGN.md section 4), so today every
test here SKIPS; the day a wheel appears they lift "parity unpinned" without a line of new code (SURVEY 8c: "probe at
runtime and prefer it").

What each test pins, by reference call site:
  test_codec_area_bbox_decode     RLE.decode / RLE.area / RLE.toBbox / RLE.encode  (structures.py:568,571,752,761;
                                  data_utils.py:275,423) on every shipped RLE string
  test_iou_and_merge              RLE.iou, RLE.merge(intersect=True) (analyze.py:108,158,315; powder.py:82)
  test_fr_polygons                RLE.frPyObjects (structures.py:677) on every shipped VIA polygon
  test_regionprops_and_label      skimage.measure.regionprops_table (structures.py:505-508), skimage.measure.label
                                  (data_utils.py:409-424), skimage.draw.polygon2mask (structures.py:693-715)
  test_gpu_path_against_real_pycocotools   the drop-in functions themselves against the reference's loops run on
                                  the real pycocotools (GPU only)

Inputs: the frozen fixtures under tests/golden/ (3,411 RLE strings cut from the reference's shipped prediction
pickles, 238 polygons of its VIA validation file).
"""
import numpy as np
import pytest

from oracle import ampis_ref as R
from oracle import cocomask as rle
from tests import _util as U


def _real_mask():
    return pytest.importorskip('pycocotools.mask', reason='pycocotools is not installed (parity stays unpinned)')


def _fixture_strings():
    """Every RLE dict of the golden fixtures."""
    out = []
    g = U.load('powder_match.npz')
    for k in range(len(g['names'])):
        _, gt, pr = U.powder_match_image(k)
        out += list(gt) + list(pr)
    s = U.load('powder_satellite.npz')
    for k in range(len(s['names'])):
        out += list(U.powder_satellite_image(k)[2])
    m = U.load('spheroidite_measure.npz')
    for k in range(len(m['names'])):
        out += U.unpack_strings(m['%d_blob' % k], m['%d_off' % k], m['%d_size' % k])
    return out


def _fixture_polygons():
    """(flat [x0, y0, ...] polygon, (h, w)) pairs of the golden fixture."""
    out = []
    p = U.load('powder_polygons.npz')
    for k in range(int(p['n_images'])):
        xy, off, size = p['%d_poly_xy' % k], p['%d_poly_off' % k], tuple(int(v) for v in p['%d_size' % k])
        out += [(xy[off[i]:off[i + 1]].tolist(), size) for i in range(len(off) - 1)]
    return out


def test_codec_area_bbox_decode():
    M = _real_mask()
    masks = _fixture_strings()
    assert len(masks) >= 3000
    for i in range(0, len(masks), 200):
        blk = masks[i:i + 200]
        assert np.array_equal(M.area(blk), rle.area(blk))
        assert np.array_equal(M.toBbox(blk), np.stack([rle.to_bbox(m) for m in blk]))
    for m in masks[::37]:
        d = M.decode(m)
        assert np.array_equal(d, rle.decode(m))
        assert M.encode(np.asfortranarray(d))['counts'] == rle.encode(np.asfortranarray(d))['counts'] == m['counts']


def test_iou_and_merge():
    M = _real_mask()
    for k in range(5):
        _, gt, pr = U.powder_match_image(k)
        want = M.iou(pr, gt, np.zeros(len(gt), np.uint8))
        assert np.array_equal(want, rle.iou(pr, gt, np.zeros(len(gt), np.uint8)))
        for g_, p_ in zip(*np.nonzero(want.T)):
            a = M.area(M.merge([gt[g_], pr[p_]], intersect=True))
            assert int(a) == int(rle.merge_area(gt[g_], pr[p_], intersect=True))
            assert M.merge([gt[g_], pr[p_]], intersect=False)['counts'] == rle.merge([gt[g_], pr[p_]], False)['counts']


def test_fr_polygons():
    M = _real_mask()
    polys = _fixture_polygons()
    assert len(polys) >= 200
    for poly, (h, w) in polys:
        want = M.frPyObjects([poly], h, w)[0]
        got = rle.frPyObjects([poly], h, w)[0]
        assert got['counts'] == want['counts'], poly[:6]


def test_regionprops_and_label():
    sk = pytest.importorskip('skimage.measure', reason='scikit-image is not installed (parity stays unpinned)')
    draw = pytest.importorskip('skimage.draw')
    keys = ['area', 'equivalent_diameter', 'major_axis_length', 'minor_axis_length', 'perimeter', 'solidity',
            'orientation', 'eccentricity', 'convex_area', 'extent']
    m = U.load('spheroidite_measure.npz')
    for k in range(len(m['names'])):
        masks = U.unpack_strings(m['%d_blob' % k], m['%d_off' % k], m['%d_size' % k])
        for mk in masks[:60]:
            img = rle.decode(mk).astype(int)
            if not img.any():
                continue
            want = sk.regionprops_table(img, properties=keys)
            got = R.regionprops_one(img.astype(bool))
            for key in keys:
                assert np.allclose(got[key], want[key][0], rtol=1e-6, atol=1e-9), key      # north_star: 1e-6 relative
    a = U.load('spheroidite_annotations.npz')
    for k in range(len(a['names'])):
        shape = tuple(int(v) for v in a['%d_shape' % k])
        ann = np.unpackbits(a['%d_bits' % k])[:shape[0] * shape[1]].reshape(shape).astype(bool)
        assert np.array_equal(sk.label(ann), R.label_binary(ann))
    for poly, (h, w) in _fixture_polygons()[:150]:
        xy = np.asarray(poly).reshape(-1, 2)
        want = draw.polygon2mask((h, w), xy[:, ::-1])
        assert np.array_equal(want, R.poly2mask([poly], (h, w))[0])


@pytest.mark.gpu
def test_gpu_path_against_real_pycocotools():
    """The drop-in functions against the reference's own loops (analyze.py:149-172, 300-339; powder.py:80-112) driven
    by the REAL pycocotools: every key of det_seg_scores and of _rle_satellite_match on the shipped images."""
    M = _real_mask()
    from ampis_b200 import analyze as A
    from ampis_b200.applications import powder as P
    import oracle.ampis_ref as ref
    real = ref.rle
    ref.rle = M                                       # the restated loops call whatever `rle` names
    try:
        for k in range(5):
            _, gt, pr = U.powder_match_image(k)
            want, got = ref.det_seg_scores(gt, pr, 0.5), A.det_seg_scores(gt, pr, 0.5)
            for key in want:
                assert np.array_equal(np.asarray(want[key]), np.asarray(got[key])), (k, key)
            assert np.array_equal(A._piecewise_iou(gt, pr), ref.piecewise_iou(gt, pr))
        _, part, sat = U.powder_satellite_image(1)
        M.merge_area = lambda a, b, intersect=True: M.area(M.merge([a, b], intersect=intersect))
        want, got = ref.rle_satellite_match(part, sat, 0.5), P._rle_satellite_match(part, sat, 0.5)
        for key in ('satellite_matches', 'satellites_unmatched', 'particles_unmatched', 'intersection_scores'):
            assert np.array_equal(want[key], got[key]), key
    finally:
        ref.rle = real
