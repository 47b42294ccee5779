"""CPU tests of the restatement of the remaining skimage 0.18.3 region properties
(tests/_rprops_ref.py): closed forms on squares, lines and frames, the 8-connected hole
fill, the Crofton LUT against the transition-count form the GPU uses, symmetries of the Hu invariants,
and -- when scikit-image is installed -- the real regionprops_table."""
import numpy as np
import pytest

from oracle import ampis_ref as R
from tests import _rprops_ref as M
from tests import _util as U

DIAGONAL_LEAK = np.array([[1, 1, 1, 0],
                          [1, 0, 1, 0],
                          [1, 1, 0, 1],
                          [0, 0, 1, 1]], bool)


def _S(p, n):
    return sum(k ** p for k in range(n))


def _crofton_from_transitions(img):
    t = M.crofton_transitions(img)
    return np.pi / 8 * (t[0] + t[1] + (t[2] + t[3]) / np.sqrt(2))


@pytest.mark.parametrize('n', [1, 2, 5, 10])
def test_square_moments_closed_form(n):
    p = M.regionprops_more(np.ones((n, n), bool), ['moments', 'moments_central'])
    for a in range(4):
        for b in range(4):
            assert p['moments'][a, b] == _S(a, n) * _S(b, n)
            if a % 2 or b % 2:
                assert abs(p['moments_central'][a, b]) < 1e-9 * max(1, _S(a, n) * _S(b, n))


@pytest.mark.parametrize('n', [1, 2, 3, 7, 20])
def test_square_feret(n):
    assert M.regionprops_more(np.ones((n, n), bool), ['feret_diameter_max'])['feret_diameter_max'] == \
        np.sqrt(n * n + (n - 1) ** 2)


def test_line_and_pixel_feret():
    assert M.regionprops_more(np.ones((1, 7), bool), ['feret_diameter_max'])['feret_diameter_max'] == 7.0
    assert M.regionprops_more(np.ones((7, 1), bool), ['feret_diameter_max'])['feret_diameter_max'] == 7.0
    assert M.regionprops_more(np.ones((1, 1), bool), ['feret_diameter_max'])['feret_diameter_max'] == 1.0


def test_frame_is_filled_and_diagonal_leak_is_not():
    f = np.ones((9, 12), bool)
    f[2:-2, 3:-3] = False
    p = M.regionprops_more(f, ['filled_area', 'filled_image'])
    assert p['filled_area'] == f.size and p['filled_image'].all()
    p = M.regionprops_more(DIAGONAL_LEAK, ['filled_area', 'filled_image'])
    assert p['filled_area'] == DIAGONAL_LEAK.sum()
    assert np.array_equal(p['filled_image'], DIAGONAL_LEAK)
    # the cross structure would have filled it: the 3x3 structure is what makes the difference
    import scipy.ndimage as ndi
    assert ndi.binary_fill_holes(DIAGONAL_LEAK).sum() == DIAGONAL_LEAK.sum() + 2


def test_crofton_lut_equals_transition_form_and_symmetries():
    rng = np.random.default_rng(5)
    for trial in range(60):
        h, w = int(rng.integers(1, 40)), int(rng.integers(1, 40))
        a = U.rand_masks(rng, 1, h, w, p_empty=0.0)[0]
        if trial % 3 == 0:
            a = rng.random((h, w)) < 0.5
        lut = M.perimeter_crofton4(a)
        assert abs(lut - _crofton_from_transitions(a)) <= 1e-12 * max(1.0, lut), trial
        for b in (a.T, np.rot90(a), np.rot90(a, 2), np.rot90(a, 3)):
            assert abs(M.perimeter_crofton4(b) - lut) <= 1e-12 * max(1.0, lut), trial
    assert abs(M.perimeter_crofton4(np.ones((10, 10), bool)) - 36.8117) < 1e-4


def test_hu_symmetries():
    rng = np.random.default_rng(6)
    for trial in range(30):
        a = U.rand_masks(rng, 1, 31, 23, p_empty=0.0)[0]
        if not a.any():
            continue
        hu = M.regionprops_more(a, ['moments_hu'])['moments_hu']
        ht = M.regionprops_more(a.T, ['moments_hu'])['moments_hu']
        scale = np.abs(hu) + 1e-15
        assert np.all(np.abs(hu[:6] - ht[:6]) <= 1e-9 * scale[:6] + 1e-15), trial
        assert abs(hu[6] + ht[6]) <= 1e-9 * scale[6] + 1e-15, trial


def test_inertia_eigvals_are_the_axis_lengths_behind_major_minor():
    rng = np.random.default_rng(7)
    for trial in range(20):
        a = U.rand_masks(rng, 1, 25, 37, p_empty=0.0)[0]
        if not a.any():
            continue
        l1, l2 = M.regionprops_more(a, ['inertia_tensor_eigvals'])['inertia_tensor_eigvals']
        one = R.regionprops_one(a)
        assert np.isclose(4 * np.sqrt(l1), one['major_axis_length'], rtol=1e-12, atol=1e-12)
        assert np.isclose(4 * np.sqrt(l2), one['minor_axis_length'], rtol=1e-12, atol=1e-9)


def test_coords_image_slice():
    a = np.zeros((6, 8), bool)
    a[2, 3] = a[4, 6] = a[3, 4] = True
    p = M.regionprops_more(a, ['coords', 'image', 'slice', 'convex_image'])
    assert p['slice'] == (slice(2, 5), slice(3, 7))
    assert np.array_equal(p['image'], a[2:5, 3:7])
    assert p['coords'].tolist() == [[2, 3], [3, 4], [4, 6]]
    assert p['convex_image'].shape == (3, 4)
    assert M.regionprops_more(np.zeros((3, 3), bool), ['coords']) == {}


NEW_KEYS = ['moments', 'moments_central', 'moments_normalized', 'moments_hu', 'inertia_tensor',
            'inertia_tensor_eigvals', 'filled_area', 'filled_image', 'perimeter_crofton', 'feret_diameter_max',
            'convex_image', 'image', 'coords', 'slice']


def test_regionprops_more_against_real_skimage():
    sk = pytest.importorskip('skimage.measure', reason='scikit-image is not installed (parity stays unpinned)')
    from oracle import cocomask as rle
    m = U.load('spheroidite_measure.npz')
    masks = U.unpack_strings(m['1_blob'], m['1_off'], m['1_size'])[:30]
    rng = np.random.default_rng(8)
    dense = [rle.decode(mk).astype(bool) for mk in masks] + list(U.rand_masks(rng, 10, 37, 53)) + [DIAGONAL_LEAK]
    for a in dense:
        if not a.any():
            continue
        want = sk.regionprops(a.astype(int))[0]
        got = M.regionprops_more(a, NEW_KEYS)
        for k in NEW_KEYS:
            w, g = want[k], got[k]
            if k == 'slice':
                assert tuple(w) == g
            elif k in ('filled_image', 'convex_image', 'image', 'coords', 'filled_area'):
                assert np.array_equal(np.asarray(w), np.asarray(g)), k
            else:
                assert np.allclose(np.asarray(w, float), np.asarray(g, float), rtol=1e-6, atol=1e-9, equal_nan=True), k
