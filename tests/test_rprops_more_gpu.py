"""GPU tests of the remaining skimage 0.18.3 region properties (moments to order 3, inertia tensor, hole
fill, Crofton perimeter, maximum Feret diameter, convex / box / filled images, coords, slice) against the
restatement in tests/_rprops_ref.py: shipped spheroidite and powder masks, random masks on odd frames, rings, holes,
spirals, tall frames, and a full 2048 x 2048 mask whose exact moments have closed forms."""
import os

import numpy as np
import pytest

from tests import _util as U

pytestmark = pytest.mark.gpu

NEW_KEYS = ['moments', 'moments_central', 'moments_normalized', 'moments_hu', 'inertia_tensor',
            'inertia_tensor_eigvals', 'filled_area', 'filled_image', 'perimeter_crofton', 'feret_diameter_max',
            'convex_image', 'image', 'coords', 'slice']


@pytest.fixture(scope='module')
def mods():
    import torch
    assert torch.cuda.is_available(), 'these tests need the B200'
    from ampis_b200 import engine, structures
    from tests import _rprops_ref as R
    from oracle import cocomask as rle

    class M:
        pass
    m = M()
    m.E, m.S, m.R, m.rle = engine, structures, R, rle
    return m


def _enc(rle, a):
    return rle.encode(np.asfortranarray(np.asarray(a).transpose(1, 2, 0).astype(np.uint8)))


def _check(got, want, img, tag):
    """got / want: dicts of one mask; img: its box image (for the magnitude of cancelling sums)."""
    assert set(got) == set(want), tag
    if not want:
        return
    h, w = img.shape
    r, c = np.nonzero(img)
    for k, wv in want.items():
        gv = got[k]
        if k == 'slice':
            assert gv == wv, (tag, k)
        elif k in ('filled_area', 'filled_image', 'convex_image', 'image', 'coords'):
            assert np.array_equal(np.asarray(gv), np.asarray(wv)), (tag, k)
            if k != 'filled_area':
                assert np.asarray(gv).dtype == np.asarray(wv).dtype, (tag, k)
        elif k == 'feret_diameter_max':
            assert gv == wv, (tag, k, gv, wv)
        elif k == 'moments':
            assert np.allclose(gv, wv, rtol=1e-12, atol=0), (tag, k)
        elif k in ('moments_central', 'inertia_tensor'):
            dr, dc = np.abs(r - r.mean()), np.abs(c - c.mean())
            if k == 'moments_central':
                mag = np.array([[(dr ** p * dc ** q).sum() for q in range(4)] for p in range(4)])
            else:
                mag = np.array([[(dc ** 2).sum(), (dr * dc).sum()], [(dr * dc).sum(), (dr ** 2).sum()]]) / len(r)
            assert np.all(np.abs(np.asarray(gv) - wv) <= 1e-6 * np.abs(wv) + 1e-9 * mag), (tag, k, gv, wv)
        else:                                   # normalized, hu, eigenvalues, crofton
            assert np.allclose(np.asarray(gv, float), np.asarray(wv, float), rtol=1e-6, atol=1e-12,
                               equal_nan=True), (tag, k, gv, wv)


def _check_masks(mods, a, tag, keys=NEW_KEYS):
    """a: bool[n, h, w]; every new key of region_properties(keys) against regionprops_more."""
    got = mods.S.region_properties(_enc(mods.rle, a), keys)
    assert len(got) == len(a)
    for i, d in enumerate(a):
        want = mods.R.regionprops_more(d, keys)
        img = want.get('image') if want else None
        if want and img is None:
            sl = mods.R.regionprops_more(d, ['slice'])['slice']
            img = d[sl]
        _check(got[i], want, img, (tag, i))


def test_fixture_masks(mods):
    m = U.load('spheroidite_measure.npz')
    masks = U.unpack_strings(m['1_blob'], m['1_off'], m['1_size'])[:60]
    _, _, pr = U.powder_match_image(3)
    for tag, ms in (('spheroidite', masks), ('powder', pr[:25])):
        dense = mods.rle.decode(ms).transpose(2, 0, 1).astype(bool)
        got = mods.S.region_properties(ms, NEW_KEYS)
        for i, d in enumerate(dense):
            want = mods.R.regionprops_more(d, NEW_KEYS)
            _check(got[i], want, want.get('image'), (tag, i))


@pytest.mark.parametrize('seed', range(int(os.environ.get('AMPIS_FUZZ_SEEDS', '3'))))
def test_random_masks_on_odd_frames(mods, seed):
    rng = np.random.default_rng(9100 + seed)
    for h, w in [(1, 1), (3, 40), (40, 3), (37, 53), (70, 70), (100, 3)]:
        a = U.rand_masks(rng, 10, h, w)
        a[0] = rng.random((h, w)) < 0.5
        a[1] = True
        a[2] = np.eye(h, w, dtype=bool)
        _check_masks(mods, a, (seed, h, w))


def test_rings_holes_spirals_and_diagonal_leak(mods):
    n = 64
    yy, xx = np.mgrid[0:n, 0:n]
    d2 = (yy - 31.5) ** 2 + (xx - 31.5) ** 2
    ring = (d2 <= 30 ** 2) & (d2 >= 20 ** 2)
    holes = np.ones((n, n), bool)
    for cy, cx in [(10, 10), (10, 50), (40, 20), (50, 50)]:
        holes &= (yy - cy) ** 2 + (xx - cx) ** 2 > 16
    holes[30, 30] = False                      # one-pixel hole
    holes[0, 5] = False                        # border notch: not a hole
    spiral = np.zeros((n, n), bool)            # square spiral wall: the background corridor inside winds inwards
    r0, c0, r1, c1 = 0, 0, n - 1, n - 1
    while r1 - r0 >= 2 and c1 - c0 >= 2:
        spiral[r0, c0:c1 + 1] = True
        spiral[r0:r1 + 1, c1] = True
        spiral[r1, c0:c1 + 1] = True
        spiral[r0 + 2:r1 + 1, c0] = True
        r0, c0, r1, c1 = r0 + 2, c0 + 2, r1 - 2, c1 - 2
    closed_spiral = spiral.copy()
    closed_spiral[1, 0] = True                 # closes the corridor's mouth: the whole corridor is a hole
    leak = np.zeros((n, n), bool)
    leak[10:14, 20:24] = [[1, 1, 1, 0], [1, 0, 1, 0], [1, 1, 0, 1], [0, 0, 1, 1]]
    frame = np.zeros((n, n), bool)
    frame[5:40, 7:60] = True
    frame[8:37, 9:58] = False
    a = np.stack([ring, holes, spiral, closed_spiral, leak, frame, ~ring, ~spiral])
    _check_masks(mods, a, 'shapes')
    got = mods.S.region_properties(_enc(mods.rle, a[[5, 4, 3]]), ['filled_area'])
    assert got[0]['filled_area'] == 35 * 53
    assert got[1]['filled_area'] == 10
    assert got[2]['filled_area'] > closed_spiral.sum()


def test_tall_frames(mods):
    rng = np.random.default_rng(33)
    h, w = 8200, 9
    a = np.zeros((4, h, w), bool)
    a[0, 3:8190, 1:8] = True
    a[0, 40:8100, 3:6] = False                 # a hole 8,060 rows long
    a[1] = rng.random((h, w)) < 0.5
    a[2, 100:8150, 4] = True                   # a vertical line
    a[3, ::7, :] = True
    _check_masks(mods, a, 'tall')


def test_full_frame_moments_are_exact(mods):
    n = 2048
    rle = mods.rle.encode(np.asfortranarray(np.ones((n, n, 1), np.uint8)))
    m = mods.E.region_measurements_for(rle, {'moments3'})['moments3'][0]
    S = [n, n * (n - 1) // 2, (n - 1) * n * (2 * n - 1) // 6, (n * (n - 1) // 2) ** 2]
    for p in range(4):
        for q in range(4):
            assert m[p][q] == S[p] * S[q], (p, q)
    assert S[3] * S[3] > 2 ** 64
    p = mods.S.region_properties(rle, ['moments_central', 'feret_diameter_max', 'filled_area', 'perimeter_crofton'])[0]
    assert p['filled_area'] == n * n
    assert p['feret_diameter_max'] == np.sqrt(n * n + (n - 1) ** 2)
    assert abs(p['perimeter_crofton'] - mods.R.perimeter_crofton4(np.ones((n, n), bool))) < 1e-9 * 4 * n
    for a in range(4):
        for b in range(4):
            if a % 2 or b % 2:
                assert p['moments_central'][a, b] == 0.0


def test_only_the_needed_kernels_run(mods, monkeypatch):
    rng = np.random.default_rng(4)
    a = U.rand_masks(rng, 6, 30, 30)
    calls = []
    real = mods.E.N.call
    monkeypatch.setattr(mods.E.N, 'call', lambda name, *args: (calls.append(name), real(name, *args))[1])
    mods.S.region_properties(_enc(mods.rle, a), ['filled_area'])
    assert 'ampis_crop_fill_holes' in calls
    assert not {'ampis_crop_convex_area', 'ampis_crop_convex_feret', 'ampis_rle_moments', 'ampis_rle_moments3',
                'ampis_crop_perimeter', 'ampis_crop_unpack_image'} & set(calls)


def test_compute_rprops_columns_with_an_empty_mask(mods):
    from ampis_b200.containers import Instances
    S, R = mods.S, mods.R
    rng = np.random.default_rng(12)
    a = U.rand_masks(rng, 5, 40, 30, p_empty=0.0)
    a[0] = True
    a[2] = False                               # empty mask
    enc = _enc(mods.rle, a)
    iset = S.InstanceSet(instances=Instances((40, 30), masks=S.RLEMasks(enc), boxes=np.zeros((5, 4)),
                                             class_idx=np.arange(5)))
    keys = list(S.InstanceSet.RPROPS_GPU_KEYS)
    df = iset.compute_rprops(keys=keys, return_df=True)
    want_cols = []
    shapes = {'bbox': (4,), 'centroid': (2,), 'local_centroid': (2,), 'moments': (4, 4), 'moments_central': (4, 4),
              'moments_normalized': (4, 4), 'moments_hu': (7,), 'inertia_tensor': (2, 2),
              'inertia_tensor_eigvals': (2,)}
    for k in keys:
        if k in shapes:
            want_cols += ['-'.join(map(str, (k,) + loc)) for loc in np.ndindex(shapes[k])]
        else:
            want_cols.append(k)
    assert list(df.columns) == want_cols + ['class_idx']
    ints = {'area', 'bbox-0', 'bbox-1', 'bbox-2', 'bbox-3', 'bbox_area', 'convex_area', 'label', 'filled_area'}
    objs = {'image', 'filled_image', 'convex_image', 'coords', 'slice'}
    for col in want_cols:
        empty = df[col][2]
        assert empty.shape == (0,), col
        assert empty.dtype == (object if col in objs else np.int64 if col in ints else np.float64), col
        for i in (0, 1, 3, 4):
            cell = df[col][i]
            assert cell.shape == (1,), (col, i)
            if col in objs:
                assert cell.dtype == object
    full = R.regionprops_more(a[1], NEW_KEYS)
    assert np.array_equal(df['image'][1][0], full['image'])
    assert np.array_equal(df['coords'][1][0], full['coords'])
    assert df['slice'][1][0] == full['slice']
    assert df['moments-2-1'][1][0] == full['moments'][2, 1]
    assert np.isnan(df['moments_normalized-0-0'][1][0])
    assert df['filled_area'][1].dtype == np.int64
    with pytest.raises(NotImplementedError):
        iset.compute_rprops(keys=['euler_number'])
