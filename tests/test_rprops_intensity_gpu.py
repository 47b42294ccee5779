"""GPU tests of the intensity region properties of skimage 0.18.3 (region_properties / compute_rprops with an
intensity_image) against the restatement in tests/_rprops_intensity_ref.py: shipped spheroidite and powder masks,
random masks on odd frames, every supported pixel type, exact integer sums beyond 128 bits, tall frames, and the
zero-sum, NaN and empty-mask rules."""
import os

import numpy as np
import pytest

from tests import _rprops_intensity_ref as I
from tests import _util as U

pytestmark = pytest.mark.gpu

KEYS = list(I.KEYS)
INT_KINDS = 'biu'


@pytest.fixture(scope='module')
def mods():
    import torch
    assert torch.cuda.is_available(), 'these tests need the B200'
    from ampis_b200 import engine, structures
    from oracle import cocomask as rle

    class M:
        pass
    m = M()
    m.E, m.S, m.rle = engine, structures, rle
    return m


def _enc(rle, a):
    return rle.encode(np.asfortranarray(np.asarray(a).transpose(1, 2, 0).astype(np.uint8)))


def _image(rng, dtype, h, w):
    dt = np.dtype(dtype)
    if dt == np.bool_:
        return rng.random((h, w)) < 0.5
    if dt.kind == 'f':
        return (rng.normal(size=(h, w)) * 100).astype(dt)
    info = np.iinfo(dt)
    lo = 2 ** 31 if dt == np.uint32 else int(info.min)              # uint32: all above 2^31
    img = rng.integers(lo, int(info.max), size=(h, w), dtype=dt, endpoint=True)
    if dt.itemsize == 8:                                             # the limits themselves
        img.ravel()[::7] = info.max
        if dt.kind == 'i':
            img.ravel()[3::11] = info.min
    return img


def _same(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.array_equal(np.isnan(a), np.isnan(b))


def _check(got, want, mask, img, tag):
    assert set(got) == set(want), tag
    if not want:
        return
    dt = np.asarray(img).dtype
    for k in KEYS:
        g, w = got[k], want[k]
        if k == 'intensity_image':
            assert g.dtype == w.dtype and np.array_equal(g, w, equal_nan=dt.kind == 'f'), (tag, k)
        elif k in ('max_intensity', 'min_intensity'):
            assert np.asarray(g).dtype == dt, (tag, k)
            assert (np.isnan(w) and np.isnan(g)) if dt.kind == 'f' and np.isnan(w) else g == w, (tag, k, g, w)
        elif k == 'mean_intensity':                      # numpy sums float16 / float32 in their own precision
            eps = 1e-12 if dt.kind in INT_KINDS or dt == np.float64 else 64 * np.finfo(dt).eps
            a = np.abs(np.asarray(img)[mask].astype(np.float64))
            scale = a[np.isfinite(a)].mean() if np.isfinite(a).any() else 0.0
            assert np.allclose(g, w, rtol=0, atol=eps * scale, equal_nan=True), (tag, k, g, w)
        elif k in ('weighted_moments', 'weighted_moments_central'):
            center = (0, 0) if k == 'weighted_moments' else want['weighted_local_centroid']
            assert _same(g, w), (tag, k, g, w)
            ok = ~np.isnan(np.asarray(w, np.float64))
            if np.isfinite(center).all():
                mag = I.weighted_magnitude(mask, img, center)
                assert np.all(np.abs(g - w)[ok] <= 1e-9 * mag[ok] + 1e-12 * np.abs(w[ok])), (tag, k, g, w)
            else:                                        # zero sum: only [0, 0] is a number
                assert np.allclose(g[ok], w[ok], rtol=1e-9, atol=0), (tag, k, g, w)
        elif k in ('weighted_centroid', 'weighted_local_centroid'):
            assert np.allclose(np.asarray(g, float), np.asarray(w, float), rtol=1e-6, atol=1e-12,
                               equal_nan=True), (tag, k, g, w)
        else:                                            # normalized, Hu: cancellation relative to the largest
            w = np.asarray(w, float)
            scale = np.nanmax(np.abs(w)) if not np.isnan(w).all() else 0.0
            assert np.allclose(np.asarray(g, float), w, rtol=1e-6, atol=1e-9 * scale + 1e-15,
                               equal_nan=True), (tag, k, g, w)


def _check_masks(mods, a, img, tag):
    """a: bool[n, h, w]; every intensity key of region_properties against the restatement, and for integer and
    bool images the weighted sums of the measurement step against the exact Python-int sums."""
    enc = _enc(mods.rle, a)
    got = mods.S.region_properties(enc, KEYS, intensity_image=img)
    assert len(got) == len(a)
    for i, d in enumerate(a):
        _check(got[i], I.regionprops_intensity(d, img), d, img, (tag, i))
    if np.asarray(img).dtype.kind in INT_KINDS:
        m = mods.E.region_measurements_for(enc, {'weighted_intensity'}, img)
        for i, d in enumerate(a):
            if d.any():
                assert m['intensity_moments'][i] == I.exact_weighted_moments(d, img), (tag, i)


def test_fixture_masks_uint8(mods):
    m = U.load('spheroidite_measure.npz')
    masks = U.unpack_strings(m['1_blob'], m['1_off'], m['1_size'])[:60]
    _, _, pr = U.powder_match_image(3)
    rng = np.random.default_rng(41)
    for tag, ms in (('spheroidite', masks), ('powder', pr[:25])):
        dense = mods.rle.decode(ms).transpose(2, 0, 1).astype(bool)
        img = rng.integers(0, 256, dense.shape[1:], dtype=np.uint8)
        got = mods.S.region_properties(ms, KEYS, intensity_image=img)
        for i, d in enumerate(dense):
            _check(got[i], I.regionprops_intensity(d, img), d, img, (tag, i))


DTYPES = [np.bool_, np.uint8, np.uint16, np.int16, np.int32, np.uint32, np.int64, np.uint64, np.float16, np.float32,
          np.float64]


@pytest.mark.parametrize('dtype', DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize('seed', range(int(os.environ.get('AMPIS_FUZZ_SEEDS', '2'))))
def test_random_masks_on_odd_frames(mods, dtype, seed):
    rng = np.random.default_rng(9400 + seed)
    for h, w in [(1, 1), (3, 40), (40, 3), (37, 53), (70, 70), (100, 3)]:
        a = U.rand_masks(rng, 8, h, w)
        a[0] = rng.random((h, w)) < 0.5
        a[1] = True
        a[2] = np.eye(h, w, dtype=bool)
        _check_masks(mods, a, _image(rng, dtype, h, w), (np.dtype(dtype).name, seed, h, w))


def test_exact_sums_beyond_128_bits(mods):
    n, v = 4096, 2 ** 62
    rle = mods.rle.encode(np.asfortranarray(np.ones((n, n, 1), np.uint8)))
    img = np.full((n, n), v, np.int64)
    M = mods.E.region_measurements_for(rle, {'weighted_intensity'}, img)['intensity_moments'][0]
    S = [n, n * (n - 1) // 2, (n - 1) * n * (2 * n - 1) // 6, (n * (n - 1) // 2) ** 2]
    for p in range(4):
        for q in range(4):
            assert M[p][q] == v * S[p] * S[q], (p, q)
    assert M[3][3] > 2 ** 153
    p = mods.S.region_properties(rle, ['mean_intensity', 'weighted_local_centroid', 'max_intensity',
                                       'weighted_moments_central'], intensity_image=img)[0]
    assert p['mean_intensity'] == float(v) and p['max_intensity'] == v
    assert p['weighted_local_centroid'] == ((n - 1) / 2, (n - 1) / 2)
    for a in range(4):
        for b in range(4):
            if a % 2 or b % 2:
                assert p['weighted_moments_central'][a, b] == 0.0


def test_tall_frames(mods):
    rng = np.random.default_rng(34)
    h, w = 8200, 9
    a = np.zeros((3, h, w), bool)
    a[0, 3:8190, 1:8] = True
    a[0, 40:8100, 3:6] = False
    a[1] = rng.random((h, w)) < 0.5
    a[2, 100:8150, 4] = True
    for dtype in (np.uint16, np.float64):
        _check_masks(mods, a, _image(rng, dtype, h, w), ('tall', np.dtype(dtype).name))


def test_zero_sums_nan_pixels_and_empty_masks(mods):
    h, w = 12, 14
    a = np.zeros((5, h, w), bool)
    a[0, 1:5, 1:6] = True                        # all-zero intensity
    a[1, 6:9, 2:7] = True                        # signed, sums to zero
    a[2, 2:6, 8:12] = True                       # holds the NaN pixel (3, 9)
    a[3, 1:11, 7:13] = True                      # L shape whose box holds (3, 9) but not the pixel
    a[3, 1:6, 8:13] = False
    a[4] = False                                 # empty
    ints = np.zeros((h, w), np.int16)
    ints[6, 2], ints[8, 6] = 300, -300
    ints[7, 4] = 0
    _check_masks(mods, a, ints, 'int16 zero sums')
    got = mods.S.region_properties(_enc(mods.rle, a), KEYS, intensity_image=ints)
    assert np.isnan(got[0]['weighted_local_centroid']).all()
    assert np.isinf(got[1]['weighted_local_centroid']).all()
    assert got[1]['weighted_moments_central'][0, 0] == 0.0
    assert np.isnan(got[1]['weighted_moments_central'].ravel()[1:]).all()
    assert got[4] == {}
    f = np.random.default_rng(5).random((h, w))
    f[3, 9] = np.nan
    _check_masks(mods, a, f, 'float64 NaN')
    got = mods.S.region_properties(_enc(mods.rle, a), KEYS, intensity_image=f)
    assert np.isnan(got[2]['max_intensity']) and np.isnan(got[2]['mean_intensity'])
    assert np.isfinite(got[3]['max_intensity']) and np.isfinite(got[3]['mean_intensity'])
    assert np.isnan(got[3]['weighted_moments']).all()
    assert np.isfinite(got[0]['weighted_moments']).all()


def _iset(mods, a):
    from ampis_b200.containers import Instances
    n, h, w = a.shape
    return mods.S.InstanceSet(instances=Instances((h, w), masks=mods.S.RLEMasks(_enc(mods.rle, a)),
                                                  boxes=np.zeros((n, 4)), class_idx=np.arange(n)))


def test_input_checks(mods):
    rng = np.random.default_rng(13)
    a = U.rand_masks(rng, 3, 20, 30, p_empty=0.0)
    iset = _iset(mods, a)
    for bad in (np.zeros((30, 20), np.uint8), np.zeros((20, 30, 3), np.uint8), np.zeros((20, 31))):
        with pytest.raises(ValueError, match='Label and intensity image must have the same shape.'):
            iset.compute_rprops(keys=['mean_intensity'], intensity_image=bad)
    with pytest.raises(NotImplementedError, match='intensity_image'):
        iset.compute_rprops(keys=['area', 'max_intensity'])
    with pytest.raises(NotImplementedError):
        iset.compute_rprops(keys=['euler_number'], intensity_image=np.zeros((20, 30)))


def test_compute_rprops_columns(mods):
    S = mods.S
    rng = np.random.default_rng(14)
    a = U.rand_masks(rng, 4, 40, 30, p_empty=0.0)
    a[0] = True
    a[2] = False                                 # empty mask
    img = rng.integers(0, 65536, (40, 30), dtype=np.uint16)
    keys = list(S.InstanceSet.RPROPS_INTENSITY_KEYS) + ['area', 'centroid', 'moments_hu']
    df = _iset(mods, a).compute_rprops(keys=keys, return_df=True, intensity_image=img)
    shapes = {'weighted_centroid': (2,), 'weighted_local_centroid': (2,), 'weighted_moments': (4, 4),
              'weighted_moments_central': (4, 4), 'weighted_moments_normalized': (4, 4), 'weighted_moments_hu': (7,),
              'centroid': (2,), 'moments_hu': (7,)}
    want_cols = []
    for k in keys:
        want_cols += ['-'.join(map(str, (k,) + loc)) for loc in np.ndindex(shapes[k])] if k in shapes else [k]
    assert list(df.columns) == want_cols + ['class_idx']
    for col in want_cols:
        empty = df[col][2]
        assert empty.shape == (0,), col
        assert empty.dtype == (object if col == 'intensity_image' else np.int64 if col == 'area' else np.float64), col
        for i in (0, 1, 3):
            cell = df[col][i]
            assert cell.shape == (1,), (col, i)
            assert cell.dtype == empty.dtype, (col, i)
    want = I.regionprops_intensity(a[1], img)
    assert np.array_equal(df['intensity_image'][1][0], want['intensity_image'])
    assert df['intensity_image'][1][0].dtype == np.uint16
    assert df['max_intensity'][1][0] == float(want['max_intensity'])
    assert df['weighted_moments-2-1'][1][0] == want['weighted_moments'][2, 1]
    assert np.isnan(df['weighted_moments_normalized-0-1'][1][0])
    assert np.isclose(df['weighted_centroid-1'][3][0], I.regionprops_intensity(a[3], img)['weighted_centroid'][1])


def test_only_the_needed_kernels_run(mods, monkeypatch):
    rng = np.random.default_rng(4)
    a = U.rand_masks(rng, 6, 30, 30)
    enc = _enc(mods.rle, a)
    calls, box_scans = [], []
    real = mods.E.N.call

    def spy(name, *args):
        calls.append(name)
        if name == 'ampis_rle_intensity':
            box_scans.append(args[9])           # scan_box: the raw pass reads whole boxes only for weighted keys
        return real(name, *args)
    monkeypatch.setattr(mods.E.N, 'call', spy)
    rprops = {'ampis_crop_convex_area', 'ampis_crop_convex_feret', 'ampis_rle_moments', 'ampis_rle_moments3',
              'ampis_crop_perimeter', 'ampis_crop_unpack_image', 'ampis_crop_fill_holes'}
    mods.S.region_properties(enc, ['max_intensity', 'mean_intensity', 'min_intensity'],
                             intensity_image=rng.integers(0, 256, (30, 30), dtype=np.uint8))
    assert calls.count('ampis_rle_intensity') == 1 and box_scans == [0] and not rprops & set(calls)
    calls.clear()
    box_scans.clear()
    mods.S.region_properties(enc, ['weighted_moments_hu'], intensity_image=rng.random((30, 30)))
    assert calls.count('ampis_rle_intensity') == 2 and not rprops & set(calls)          # raw, then central
    assert box_scans == [1, 0]
    calls.clear()
    box_scans.clear()
    got = mods.S.region_properties(enc, ['max_intensity', 'mean_intensity', 'min_intensity'],
                                   intensity_image=rng.random((30, 30)))
    assert calls.count('ampis_rle_intensity') == 1 and box_scans == [0] and not rprops & set(calls)
    assert all(set(g) == {'max_intensity', 'mean_intensity', 'min_intensity'} for g in got if g)
    calls.clear()
    mods.S.region_properties(enc, ['intensity_image'], intensity_image=rng.random((30, 30)))
    assert 'ampis_rle_intensity' not in calls and 'ampis_crop_unpack_image' in calls
