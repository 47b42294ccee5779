"""CPU tests of the restatement of skimage 0.18.3's intensity region properties (tests/_rprops_intensity_ref.py):
closed forms for constant and linear-ramp images, the zero-sum, negative-sum and NaN rules, the host formation of
the weighted moments from exact integer sums, and -- when scikit-image is installed -- the real
regionprops_table."""
import numpy as np
import pytest

from tests import _rprops_intensity_ref as I
from tests import _rprops_ref as M
from tests import _util as U


def _S(p, n):
    return sum(k ** p for k in range(n))


def _blob(seed=3, h=31, w=23):
    rng = np.random.default_rng(seed)
    a = U.rand_masks(rng, 4, h, w, p_empty=0.0)
    return next(m for m in a if m.sum() > 20)


@pytest.mark.parametrize('k', [1, 7, -3, 0.5])
def test_constant_image_gives_k_times_the_unweighted_moments(k):
    mask = _blob()
    img = np.full(mask.shape, k, dtype=np.float64)
    p = I.regionprops_intensity(mask, img)
    un = M.regionprops_more(mask, ['moments', 'moments_central', 'moments_normalized', 'moments_hu'])
    assert np.allclose(p['weighted_moments'], k * un['moments'], rtol=1e-12, atol=0)
    assert np.allclose(p['weighted_moments_central'], k * un['moments_central'], rtol=1e-9, atol=1e-9)
    sl = I.region_slice(mask)
    r, c = np.nonzero(mask)
    assert np.allclose(p['weighted_centroid'], (r.mean(), c.mean()), rtol=1e-12)
    assert np.allclose(p['weighted_local_centroid'], (r.mean() - sl[0].start, c.mean() - sl[1].start), rtol=1e-12)
    assert p['max_intensity'] == p['min_intensity'] == k and np.isclose(p['mean_intensity'], k)
    if k > 0:      # nu scales by k^(-(p+q)/2): it is not invariant to the weight
        for a in range(4):
            for b in range(4):
                if a + b >= 2:
                    want = un['moments_normalized'][a, b] * k ** (-(a + b) / 2)
                    assert np.isclose(p['weighted_moments_normalized'][a, b], want, rtol=1e-9, atol=1e-12)


def test_linear_ramp_has_polynomial_sums():
    h, w, r0, c0 = 9, 13, 4, 6
    a, b, d = 3, -2, 50
    mask = np.zeros((20, 25), bool)
    mask[r0:r0 + h, c0:c0 + w] = True
    rr, cc = np.mgrid[0:20, 0:25]
    img = (a * rr + b * cc + d).astype(np.int64)
    exact = I.exact_weighted_moments(mask, img)
    p = I.regionprops_intensity(mask, img)
    for pp in range(4):
        for q in range(4):
            want = (a * (_S(pp + 1, h) + r0 * _S(pp, h)) * _S(q, w) + b * _S(pp, h) * (_S(q + 1, w) + c0 * _S(q, w))
                    + d * _S(pp, h) * _S(q, w))
            assert exact[pp][q] == want, (pp, q)
            assert p['weighted_moments'][pp, q] == want, (pp, q)
    assert p['min_intensity'] == img[mask].min() and p['max_intensity'] == img[mask].max()
    assert p['intensity_image'].dtype == np.int64 and p['intensity_image'].shape == (h, w)


def test_zero_sum_rules():
    mask = np.zeros((6, 7), bool)
    mask[1:4, 2:6] = True
    p = I.regionprops_intensity(mask, np.zeros((6, 7), np.uint8))
    assert np.all(np.isnan(p['weighted_local_centroid'])) and np.all(np.isnan(p['weighted_centroid']))
    mu = p['weighted_moments_central']
    assert mu[0, 0] == 0.0 and np.isnan(mu.ravel()[1:]).all()
    assert np.isnan(p['weighted_moments_normalized']).all() and np.isnan(p['weighted_moments_hu']).all()
    img = np.zeros((6, 7), np.int16)
    img[1, 2], img[3, 5] = 5, -5                         # sums to 0, first moments do not: centroid is +-inf
    p = I.regionprops_intensity(mask, img)
    assert np.isinf(p['weighted_local_centroid']).all()
    assert p['weighted_local_centroid'][0] < 0 and p['weighted_local_centroid'][1] < 0
    mu = p['weighted_moments_central']
    assert mu[0, 0] == 0.0 and np.isnan(mu.ravel()[1:]).all()


def test_negative_sum_gives_nan_not_complex():
    mask = _blob(5)
    p = I.regionprops_intensity(mask, np.full(mask.shape, -2, np.int32))
    nu = p['weighted_moments_normalized']
    assert p['weighted_moments_central'][0, 0] == -2 * mask.sum()
    assert np.isfinite(nu[2, 0]) and np.isfinite(nu[1, 1])      # mu00 ** 2
    assert np.isnan(nu[3, 0]) and np.isnan(nu[2, 1])            # mu00 ** 2.5 of a negative float64
    assert nu.dtype == np.float64


def test_nan_inside_and_outside_the_region():
    mask = np.zeros((8, 8), bool)
    mask[2:6, 2:6] = True
    mask[2, 2] = False                                   # in the box, outside the region
    img = np.arange(64, dtype=np.float64).reshape(8, 8)
    inside = img.copy()
    inside[4, 4] = np.nan
    p = I.regionprops_intensity(mask, inside)
    assert np.isnan(p['max_intensity']) and np.isnan(p['min_intensity']) and np.isnan(p['mean_intensity'])
    assert np.isnan(p['weighted_moments']).all()
    outside = img.copy()
    outside[2, 2] = np.nan
    p = I.regionprops_intensity(mask, outside)
    assert p['max_intensity'] == 45.0 and p['min_intensity'] == 19.0
    assert np.isnan(p['weighted_moments']).all() and np.isnan(p['weighted_moments_central']).all()
    far = img.copy()
    far[7, 7] = np.nan                                   # outside the box: no effect
    p = I.regionprops_intensity(mask, far)
    assert np.isfinite(p['weighted_moments']).all()


def test_host_formation_from_exact_sums():
    """structures forms the weighted central, normalized and Hu moments from the exact sums the GPU returns."""
    from ampis_b200 import engine, structures as S
    rng = np.random.default_rng(21)
    for trial in range(12):
        mask = _blob(30 + trial)
        img = rng.integers(-1000 if trial % 2 else 0, 1000, mask.shape).astype(np.int64)
        if trial == 11:
            img = np.full(mask.shape, -7, np.int64)
        want = I.regionprops_intensity(mask, img)
        Mx = I.exact_weighted_moments(mask, img)
        mu = S._exact_central(Mx)
        got = S._moment_props(Mx, mu)
        wlc = (want['weighted_local_centroid'])
        mag = I.weighted_magnitude(mask, img, wlc)
        assert np.all(np.abs(mu - want['weighted_moments_central']) <= 1e-9 * mag), trial
        assert np.allclose(got['moments_normalized'], want['weighted_moments_normalized'], rtol=1e-7, atol=1e-15,
                           equal_nan=True), trial
        assert np.allclose(got['moments_hu'], want['weighted_moments_hu'], rtol=1e-6, atol=1e-15,
                           equal_nan=True), trial
    mu = S._exact_central([[0, 5, 0, 0], [-5, 0, 0, 0], [0, 0, 0, 0], [0, 0, 0, 0]])
    assert mu[0, 0] == 0.0 and np.isnan(mu.ravel()[1:]).all()
    assert np.isinf(S._div(-5, 0)) and np.isnan(S._div(0, 0)) and S._div(1, 3) == 1 / 3
    for v in (0, 1, -1, 2 ** 191 - 1, -2 ** 191, 12345 * 2 ** 130 - 99):
        u = v % (1 << 192)
        assert engine._i192([u & (2 ** 64 - 1), (u >> 64) & (2 ** 64 - 1), u >> 128]) == v


def test_intensity_image_shape_check():
    from ampis_b200 import structures as S
    rle = [{'size': [6, 7], 'counts': b'0'}]
    for bad in (np.zeros((7, 6)), np.zeros((6, 7, 3)), np.zeros(42)):
        with pytest.raises(ValueError, match='Label and intensity image must have the same shape.'):
            S.region_properties(rle, ['max_intensity'], intensity_image=bad)
    with pytest.raises(NotImplementedError, match='intensity_image'):
        S.region_properties(rle, ['mean_intensity'])


KEYS = list(I.KEYS)


def test_restatement_against_real_skimage():
    sk = pytest.importorskip('skimage.measure', reason='scikit-image is not installed (parity stays unpinned)')
    from oracle import cocomask as rle
    m = U.load('spheroidite_measure.npz')
    masks = U.unpack_strings(m['1_blob'], m['1_off'], m['1_size'])[:20]
    rng = np.random.default_rng(8)
    dense = [rle.decode(mk).astype(bool) for mk in masks]
    imgs = [rng.integers(0, 256, dense[0].shape).astype(np.uint8), rng.normal(size=dense[0].shape)]
    small = list(U.rand_masks(rng, 8, 37, 53))
    small_imgs = [rng.integers(-300, 300, (37, 53)).astype(np.int16), rng.random((37, 53)).astype(np.float32)]
    for masks_, imgs_ in ((dense, imgs), (small, small_imgs)):
        for img in imgs_:
            for a in masks_:
                if not a.any():
                    continue
                want = sk.regionprops(a.astype(int), intensity_image=img)[0]
                got = I.regionprops_intensity(a, img)
                for k in KEYS:
                    w, g = want[k], got[k]
                    if k == 'intensity_image':
                        assert np.array_equal(w, g) and w.dtype == g.dtype
                    elif k in ('max_intensity', 'min_intensity'):
                        assert w == g and np.asarray(w).dtype == np.asarray(g).dtype, k
                    else:
                        assert np.allclose(np.asarray(w, float), np.asarray(g, float), rtol=1e-6, atol=1e-9,
                                           equal_nan=True), k
