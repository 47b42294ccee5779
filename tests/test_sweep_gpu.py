"""analyze.det_seg_scores_sweep / engine.eval_images_sweep (ampis_eval_images_sweep_host, the staircase and count
kernels of csrc/score.cu) on the B200 against tests/_sweep_ref.py, bit for bit: fixture images with seeded scores,
random odd frames, ties that change winner with the score level, empty sides and empty masks, a crowded frame, a
native C4 image, a dataset of 1,000 C2 images, workspaces grown from 4 KB, the per-image prediction limit, and
agreement with engine.eval_images and det_seg_scores_batch on the filtered lists."""
import os

import numpy as np
import pytest

from tests import _sweep_ref as S
from tests import _util
from tests.test_sweep_oracle import _dataset, _rle

pytestmark = pytest.mark.gpu

SCORE_TH = [0.5, -np.inf, 0.0, 0.25, 0.25, 0.7, 0.9, 0.95, 1.0]


@pytest.fixture(scope='module')
def A():
    import torch
    assert torch.cuda.is_available(), 'these tests need the B200'
    from ampis_b200 import analyze
    return analyze


def _scores(rng, n, dtype=np.float32):
    """Seeded scores on a coarse grid: many equal to a threshold or to each other."""
    return np.round(rng.random(n), 2).astype(dtype)


def _synth(cfg, n, seed, **over):
    from ampis_b200 import batch
    from oracle import cocomask as rle
    host = batch.synth(dict(batch.CONFIGS[cfg], **over), n, seed)
    mk = lambda cs: [{'size': [host.h, host.w], 'counts': rle.string_from_counts(c)} for c in cs]
    return [tuple(mk(x) for x in host.image_masks(g)) for g in range(n)]


def _check(A, gts, prs, scores, score_th, iou_th=None, what=''):
    from ampis_b200 import batch
    it = batch.COCO_THRESHOLDS if iou_th is None else iou_th
    got = A.det_seg_scores_sweep(gts, prs, score_th, iou_th, scores=scores)
    S.assert_same(got, S.sweep(gts, prs, scores, score_th, it), what)
    return got


def test_fixture_images(A):
    rng = np.random.default_rng(5)
    imgs = [_util.powder_match_image(k)[1:] for k in range(5)]
    gts, prs = [g for g, _ in imgs], [p for _, p in imgs]
    scores = [_scores(rng, len(p), dt) for p, dt in zip(prs, (np.float32, np.float64, np.float16, np.float32, np.float64))]
    got = _check(A, gts, prs, scores, SCORE_TH)
    assert got['totals'][:, :, 0].max() > 0 and len(np.unique(got['det_tp'][0, :, 0])) > 3


@pytest.mark.parametrize('seed', range(int(os.environ.get('AMPIS_FUZZ_SEEDS', '3'))))
def test_random_odd_frames(A, seed):
    gts, prs, scores = _dataset(100 + seed, 24)
    _check(A, gts, prs, scores, SCORE_TH, [0.0, 0.5, 0.25, 0.75, 0.5], 'seed %d' % seed)


def test_ties_change_with_the_level(A):
    """Exact copies of one prediction with equal IoU: the lowest index wins among the kept, so the winner moves as
    the copies' scores fall on either side of a threshold; a shifted copy with a lower IoU takes over when the
    copies are dropped."""
    h, w = 30, 40
    f = np.zeros((h, w), bool)
    f[5:15, 5:20] = True
    g = _rle(f)
    sh = _rle(np.roll(f, 2, axis=1))
    other = np.zeros((h, w), bool)
    other[20:25, 30:35] = True
    gts = [[g, _rle(other)], [g, g]]
    prs = [[_rle(f), sh, _rle(f), _rle(f), _rle(other)], [sh, _rle(f), _rle(f)]]
    scores = [np.asarray([0.3, 0.9, 0.5, 0.7, 0.2], np.float32), np.asarray([0.8, 0.4, 0.6], np.float64)]
    _check(A, gts, prs, scores, [0.0, 0.3, 0.35, 0.5, 0.6, 0.7, 0.8, 0.9], [0.0, 0.5, 0.8, 0.99])


def test_empty_sides_and_masks(A):
    h, w = 17, 13
    f = np.zeros((h, w), bool)
    f[2:9, 3:7] = True
    far = np.zeros((h, w), bool)
    far[12:15, 9:12] = True
    e = _rle(np.zeros((h, w), bool))
    gts = [[], [_rle(f)], [], [_rle(f), e, _rle(far)], [_rle(f), _rle(far)], [e, e]]
    prs = [[_rle(f), e], [], [], [e, _rle(f), _rle(np.ones((h, w), bool))], [_rle(f)], [e]]
    scores = [np.asarray([0.5, np.nan], np.float32), np.zeros(0, np.float32), np.zeros(0, np.float64),
              np.asarray([0.9, 0.2, np.nan], np.float16), np.asarray([0.99], np.float32), np.asarray([0.1], np.float32)]
    got = _check(A, gts, prs, scores, [0.95, 0.5, 0.0, 1.5])
    assert np.isnan(got['det_precision'][3]).all() and got['n_pred'][:, 3].sum() == 0
    # all images empty
    _check(A, [[], []], [[], []], [np.zeros(0, np.float32)] * 2, [0.5])
    _check(A, [], [], [], [0.5])


def test_crowded_frame(A):
    """A dense_overlap frame: the plain entry would send it to the tensor-core contraction; the sweep joins it."""
    rng = np.random.default_rng(8)
    (g, p), = _synth('dense_overlap', 1, 18, median_diam=96.0)        # a third of all box pairs overlap
    from ampis_b200 import engine
    assert engine.eval_images([g], [p], engine.MODE_IOU, crowd_frac=engine.CROWD_PAIR_FRACTION).crowded
    _check(A, [g], [p], [_scores(rng, len(p))], [0.1, 0.5, 0.9])


def test_native_c4_image(A):
    rng = np.random.default_rng(9)
    (g, p), = _synth('c4_spheroidite', 1, 21)
    assert len(g) == 5000 and len(p) == 5000
    _check(A, [g], [p], [_scores(rng, len(p))], [0.2, 0.6, 0.6, 0.95], [0.5, 0.75])


def test_c2_dataset_and_consistency(A):
    """1,000 C2 images: with [-inf] the counts equal engine.eval_images' arg-max rows counted per threshold; every
    cell equals det_seg_scores_batch on the filtered lists; a sample of images equals the reference."""
    from ampis_b200 import batch, distributed, engine
    rng = np.random.default_rng(10)
    imgs = _synth('c2_powder_batch', 1000, 31)
    gts, prs = [g for g, _ in imgs], [p for _, p in imgs]
    scores = [_scores(rng, len(p)) for p in prs]
    th = batch.COCO_THRESHOLDS
    got = A.det_seg_scores_sweep(gts, prs, [-np.inf, 0.5, 0.9], scores=scores)
    plain = distributed._counts_from_rows(engine.eval_images(gts, prs, engine.MODE_IOU), th)
    for c, k in enumerate(('det_tp', 'det_fp', 'det_fn')):
        assert np.array_equal(got[k][:, 0], plain[..., c]), k
    for k, s in enumerate([-np.inf, 0.5, 0.9]):
        kept = [[p[i] for i in np.flatnonzero(sc > s)] for p, sc in zip(prs, scores)]
        for j in (0, 5, 9):
            try:
                ds = A.det_seg_scores_batch(gts, kept, th[j])
            except ZeroDivisionError:          # an image with nothing kept or nothing matched: no cells to compare
                continue
            for key in ('det_tp', 'det_fp', 'det_fn'):
                assert [len(d[key]) for d in ds] == got[key][:, k, j].tolist(), (s, j, key)
            for key in ('seg_tp', 'seg_fp', 'seg_fn'):
                assert [int(d[key].sum()) for d in ds] == got[key][:, k, j].tolist(), (s, j, key)
    sample = rng.choice(1000, 6, replace=False)
    ref = S.sweep([gts[i] for i in sample], [prs[i] for i in sample], [scores[i] for i in sample],
                  [-np.inf, 0.5, 0.9], th)
    for k in ('n_pred', 'det_tp', 'det_fp', 'det_fn', 'seg_tp', 'seg_fp', 'seg_fn'):
        assert np.array_equal(got[k][sample], ref[k]), k
    # the C entry without per-image outputs gives the same totals
    r = engine.eval_images_sweep(gts, prs, A._score_levels(np.concatenate(scores), np.asarray([-np.inf, 0.5, 0.9])),
                                 3, th, per_image=False)
    assert r.counts is None and np.array_equal(r.totals, got['totals']) and np.array_equal(r.seg_totals, got['seg_totals'])


def test_workspace_grows_from_4kb(A):
    import torch
    from ampis_b200 import engine
    gts, prs, scores = _dataset(7, 12)
    imgs = _synth('c2_powder_batch', 3, 41)
    gts += [g for g, _ in imgs]
    prs += [p for _, p in imgs]
    scores += [_scores(np.random.default_rng(3), len(p)) for _, p in imgs]
    dev = engine.require_cuda()
    with engine._image_ws_lock:
        engine._image_ws[dev.index] = [torch.empty(4096, dtype=torch.uint8, device=dev),
                                       torch.empty(4096, dtype=torch.uint8, pin_memory=True)]
    _check(A, gts, prs, scores, SCORE_TH, [0.5, 0.75])
    assert engine._image_ws[dev.index][0].numel() > 4096 and engine._image_ws[dev.index][1].numel() > 4096


def test_prediction_limit_is_an_error(A):
    from ampis_b200 import _native
    e = _rle(np.zeros((2, 2), bool))
    f = _rle(np.ones((2, 2), bool))
    n = 32768
    ok = A.det_seg_scores_sweep([[f]], [[e] * (n - 1) + [f]], [0.5], [0.5], scores=[np.ones(n, np.float32)])
    assert ok['det_tp'][0, 0, 0] == 1 and ok['det_fp'][0, 0, 0] == n - 1
    with pytest.raises(_native.AmpisNativeError, match='more than 32768 predictions in one image'):
        A.det_seg_scores_sweep([[f]], [[e] * n + [f]], [0.5], [0.5], scores=[np.ones(n + 1, np.float32)])
