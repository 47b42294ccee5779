"""powder.satellite_measurements_sweep / engine.eval_images_sat_sweep (ampis_eval_images_sat_sweep_host, the satellite
staircase and sat_sweep_counts_kernel of csrc/score.cu) on the B200 against tests/_sat_sweep_ref.py, bit for bit:
fixture satellite images with seeded scores, random odd frames, copies of one particle whose winner moves with the
particle cut-off, zero-area masks, images without particles, satellites or any match, scores and match ratios exactly
on a threshold, a native C3 batch, workspaces grown from 4 KB and the particle limit; with no score axes the result
equals powder.satellite_measurements and distributed.satellite_measurements_sharded key for key."""
import os

import numpy as np
import pytest

from tests import _sat_sweep_ref as SR
from tests import _util
from tests.test_sat_sweep_oracle import _dataset
from tests.test_sweep_oracle import _rle

pytestmark = pytest.mark.gpu

P_TH = [0.5, -np.inf, 0.0, 0.25, 0.25, 0.7, 0.95, 1.0]
S_TH = [0.3, -np.inf, 0.6, 0.9, 0.3]
M_TH = [0.5, 0.0, 0.25, 0.75, 0.5, 0.99]


@pytest.fixture(scope='module')
def P():
    import torch
    assert torch.cuda.is_available(), 'these tests need the B200'
    from ampis_b200.applications import powder
    return powder


def _scores(rng, n, dtype=np.float32):
    """Seeded scores on a coarse grid: many equal to a threshold or to each other."""
    return np.round(rng.random(n), 2).astype(dtype)


def _check(P, psi, *args, what='', **kw):
    got = P.satellite_measurements_sweep(psi, *args, **kw)
    SR.assert_same(got, SR.sweep(psi, *args, **kw), what)
    return got


def _fixture_psi(rng=None):
    s = _util.load('powder_satellite.npz')
    out = []
    for k, dt in zip(range(len(s['names'])), (np.float32, np.float64, np.float16, np.float32, np.float64)):
        _, part, sat = _util.powder_satellite_image(k)
        size = tuple(int(v) for v in s['%d_size' % k])
        sc = (None, None) if rng is None else (_scores(rng, len(part), dt), _scores(rng, len(sat), dt))
        out.append(SR.psi_of(part, sat, size, *sc))
    return out


def test_fixture_images(P):
    psi = _fixture_psi(np.random.default_rng(5))
    got = _check(P, psi, P_TH, S_TH, M_TH)
    assert got['n_satellites'].max() > 0 and len(np.unique(got['n_satellited_particels'])) > 5


def test_no_score_axes_equal_satellite_measurements(P):
    """All score axes None, match 0.5: powder.satellite_measurements and its sharded form, key for key."""
    from ampis_b200 import distributed
    psi = _fixture_psi()
    got = _check(P, psi)
    at = P.satellite_measurements_at(got, 0, 0, 0)
    for want in (P.satellite_measurements([p.copy() for p in psi], print_summary=False, output_dict=True),
                 distributed.satellite_measurements_sharded(psi, thresh=0.5)):
        assert set(at) == set(want)
        for key in want:
            assert SR.same_value(at[key], want[key]), key


@pytest.mark.parametrize('seed', range(int(os.environ.get('AMPIS_FUZZ_SEEDS', '3'))))
def test_random_odd_frames(P, seed):
    _check(P, _dataset(100 + seed, 16), P_TH, S_TH, M_TH, what='seed %d' % seed)


def test_winner_moves_with_the_particle_cutoff(P):
    """Exact copies of one particle with different scores: the lowest kept index wins, so the satellites' owner
    moves as the copies fall on either side of a cut-off; a shifted copy that overlaps less takes over when all
    copies are dropped."""
    h, w = 30, 40
    f = np.zeros((h, w), bool)
    f[5:15, 5:20] = True
    sh = np.roll(f, 3, axis=1)
    sats = []
    for y, x in ((4, 6), (14, 18), (10, 4), (8, 19)):           # on the edges: part inside, part outside
        s = np.zeros((h, w), bool)
        s[y:y + 2, x:x + 3] = True
        sats.append(_rle(s))
    parts = [_rle(f), _rle(sh), _rle(f), _rle(f)]
    psi = [SR.psi_of(parts, sats, (h, w), np.asarray([0.3, 0.9, 0.5, 0.7], np.float32),
                     np.asarray([0.9, 0.8, 0.4, 0.6], np.float32))]
    got = _check(P, psi, [0.0, 0.3, 0.35, 0.5, 0.6, 0.7, 0.8], [0.0, 0.5, 0.7], [0.0, 0.3, 0.5, 0.6])
    assert got['n_satellites'].max() == 4


def test_empty_masks_and_images(P):
    """Zero-area satellites and particles; images without particles, without satellites, without any match; a
    satellite score exactly on a threshold and a satellite whose match ratio is exactly a match threshold."""
    h, w = 17, 13
    f = np.zeros((h, w), bool)
    f[2:9, 3:7] = True
    far = np.zeros((h, w), bool)
    far[12:15, 9:12] = True
    half = np.zeros((h, w), bool)
    half[8:10, 4:6] = True                                      # 4 pixels, 2 of them on f: ratio exactly 0.5
    e = _rle(np.zeros((h, w), bool))
    imgs = [([_rle(f), e], [e, _rle(half)]),                    # zero-area particle and satellite
            ([], [_rle(half), _rle(far)]),                      # no particles
            ([_rle(f)], []),                                    # no satellites
            ([_rle(f)], [_rle(far)]),                           # nothing matches anywhere
            ([], []),
            ([e, e], [e])]
    psi = [SR.psi_of(p, s, (h, w), np.asarray([0.5, 0.9][:len(p)] + [0.2] * max(0, len(p) - 2), np.float32),
                     np.asarray([0.5, 0.25][:len(s)], np.float32)) for p, s in imgs]
    got = _check(P, psi, [0.95, 0.5, 0.0, 1.5], [0.5, 0.25, 0.0], [0.5, 0.0, 0.49])
    assert np.isnan(got['sat_frac'][3]).all() and np.isnan(got['mspp']).any()
    _check(P, psi[1:5], None, None, [0.5])
    _check(P, [], [0.5], [0.5], [0.5])


def _c3(n, seed):
    from ampis_b200 import batch
    from oracle import cocomask as rle
    host = batch.synth(batch.CONFIGS['c3_satellites'], n, seed)
    mk = lambda cs: [{'size': [host.h, host.w], 'counts': rle.string_from_counts(c)} for c in cs]
    return [tuple(mk(x) for x in host.image_masks(g)) for g in range(n)]          # (satellites, particles)


def test_native_c3_batch(P):
    rng = np.random.default_rng(9)
    imgs = _c3(2, 21)
    assert len(imgs[0][0]) == 200 and len(imgs[0][1]) == 2000
    psi = [SR.psi_of(p, s, (2048, 2048), _scores(rng, len(p)), _scores(rng, len(s), np.float64)) for s, p in imgs]
    got = _check(P, psi, [0.2, 0.6, 0.6, 0.95], [0.1, 0.5], [0.5, 0.25, 0.75])
    assert got['n_satellites'].max() > 100


def test_workspace_grows_from_4kb(P):
    import torch
    from ampis_b200 import engine
    psi = _dataset(7, 10)
    dev = engine.require_cuda()
    with engine._image_ws_lock:
        engine._image_ws[dev.index] = [torch.empty(4096, dtype=torch.uint8, device=dev),
                                       torch.empty(4096, dtype=torch.uint8, pin_memory=True)]
    _check(P, psi, P_TH, S_TH, M_TH)
    assert engine._image_ws[dev.index][0].numel() > 4096 and engine._image_ws[dev.index][1].numel() > 4096


def test_particle_limit_is_an_error(P):
    e = _rle(np.zeros((2, 2), bool))
    f = _rle(np.ones((2, 2), bool))
    n = 32768
    ok = P.satellite_measurements_sweep([SR.psi_of([e] * (n - 1) + [f], [f], (2, 2))])
    assert ok['n_satellites'][0, 0, 0] == 1 and ok['n_particles'][0] == n
    with pytest.raises(ValueError, match='more than 32768 particles'):
        P.satellite_measurements_sweep([SR.psi_of([e] * n + [f], [f], (2, 2))])
