"""CPU tests of the score x IoU threshold sweep: the numpy reference (tests/_sweep_ref.py) against AMPIS's own
matcher, the host helpers that turn scores into levels and put thresholds in order, the argument checks of
analyze.det_seg_scores_sweep, and distributed.sweep_sharded on a gloo world of two."""
import multiprocessing as mp
import os
import socket

import numpy as np
import pytest

from tests import _sweep_ref as S


def _rle(frame):
    from oracle import cocomask as rle
    return rle.encode(np.asfortranarray(frame[:, :, None].astype(np.uint8)))[0]


def _image(rng, h, w, n_gt, n_pred):
    """Random boxes and blobs on an h x w frame; some predictions are copies or shifted copies of ground truths,
    a few masks are empty."""
    yy, xx = np.mgrid[0:h, 0:w]

    def blob():
        if rng.random() < 0.06:
            return np.zeros((h, w), bool)
        cy, cx = rng.integers(0, h), rng.integers(0, w)
        ry, rx = rng.integers(1, max(h // 3, 2)), rng.integers(1, max(w // 3, 2))
        return ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1.0
    gt = [blob() for _ in range(n_gt)]
    pred = []
    for _ in range(n_pred):
        if gt and rng.random() < 0.5:
            g = gt[int(rng.integers(0, len(gt)))]
            pred.append(np.roll(g, (int(rng.integers(-2, 3)), int(rng.integers(-2, 3))), axis=(0, 1)))
        else:
            pred.append(blob())
    return [_rle(f) for f in gt], [_rle(f) for f in pred]


def _dataset(seed, n_img=8):
    rng = np.random.default_rng(seed)
    imgs = [_image(rng, int(rng.integers(9, 40)), int(rng.integers(9, 40)), int(rng.integers(0, 7)),
                   int(rng.integers(0, 9))) for _ in range(n_img)]
    scores = [np.round(rng.random(len(p)), 1).astype(rng.choice([np.float16, np.float32, np.float64]))
              for _, p in imgs]
    return [g for g, _ in imgs], [p for _, p in imgs], scores


SCORE_TH = [0.55, -np.inf, 0.0, 0.3, 0.3, 0.9, 1.0]
IOU_TH = [0.5, 0.0, 0.25, 0.75, 0.5, 0.95]


def test_reference_equals_ampis_matcher():
    """Every cell of the reference is det_seg_scores (oracle.ampis_ref: the reference's own loop over RLE.iou chunks)
    on the filtered predictions: len(det_tp / det_fp / det_fn), sums of seg_tp / seg_fp / seg_fn -- or, where that
    raises ZeroDivisionError, piecewise_rle_match's counts with no segmentation sums."""
    from oracle import ampis_ref as R
    gts, prs, scores = _dataset(1)
    ref = S.sweep(gts, prs, scores, SCORE_TH, IOU_TH)
    checked = 0
    for i, (g, p, s) in enumerate(zip(gts, prs, scores)):
        for k, st in enumerate(SCORE_TH):
            kept = [p[c] for c in np.flatnonzero(s > st)]
            assert ref['n_pred'][i, k] == len(kept)
            for j, t in enumerate(IOU_TH):
                got = [ref[key][i, k, j] for key in ('det_tp', 'det_fp', 'det_fn', 'seg_tp', 'seg_fp', 'seg_fn')]
                try:
                    d = R.det_seg_scores(g, kept, iou_thresh=t)
                    want = [len(d['det_tp']), len(d['det_fp']), len(d['det_fn']),
                            d['seg_tp'].sum(), d['seg_fp'].sum(), d['seg_fn'].sum()]
                    checked += 1
                except ZeroDivisionError:
                    m = R.piecewise_rle_match(g, kept, t) if len(g) else {'tp': [], 'fp': np.arange(len(kept)), 'fn': []}
                    want = [len(m['tp']), len(m['fp']), len(m['fn']), 0, 0, 0]
                assert got == [int(v) for v in want], (i, st, t)
    assert checked > 100
    assert np.array_equal(ref['totals'], np.stack([ref['det_tp'], ref['det_fp'], ref['det_fn']], -1).sum(0))


def test_score_levels_follow_numpy_comparison():
    """A prediction is kept at caller threshold k iff level > pos[k], for scores exactly on a threshold and one ulp
    either side, NaN and infinite scores, duplicate and unsorted thresholds, thresholds outside float16's range."""
    from ampis_b200 import analyze as A
    th = [0.5, 0.25, 0.5, 1e6, -1e6, -np.inf, np.inf, 0.1, 65519.0, 65520.0, 1 / 3]
    s_sorted, pos = A._sorted_thresholds(th, 'x')
    assert np.all(np.diff(s_sorted) >= 0) and np.array_equal(s_sorted[pos], np.asarray(th))
    for dt in (np.float16, np.float32, np.float64):
        base = np.asarray([0.5, 0.25, 0.1, 1 / 3, 65504, 0.0, 1.0], dt)
        with np.errstate(over="ignore"):
            up, down = np.nextafter(base, dt(np.inf)), np.nextafter(base, dt(-np.inf))
        s = np.concatenate([base, up, down, np.asarray([np.nan, np.inf, -np.inf], dt)])
        lv = A._score_levels(s, s_sorted)
        assert lv.dtype == np.uint16
        for k, t in enumerate(th):
            with np.errstate(over='ignore'):
                want = s > t
            assert np.array_equal(lv > pos[k], want), (dt, t)
    # 0.1 and 1/3 round differently in float32 than in float64: a float32 score of float32(0.1) is not above 0.1
    f = np.asarray([0.1, 1 / 3], np.float32)
    assert not (A._score_levels(f, np.asarray([0.1, 1 / 3])) > [0, 1]).any()


def test_argument_errors(monkeypatch):
    import torch
    from ampis_b200 import analyze as A
    from ampis_b200 import engine
    monkeypatch.setattr(engine, 'require_cuda', lambda: torch.device('cpu'))
    gts, prs, scores = _dataset(2, 3)
    prs[0] = prs[0] or [_rle(np.ones((5, 5), bool))]
    scores[0] = np.ones(len(prs[0]), np.float32)
    with pytest.raises(ValueError, match='scores for'):
        A.det_seg_scores_sweep(gts, prs, [0.5], scores=[s[:-1] if i == 0 else s for i, s in enumerate(scores)])
    with pytest.raises(ValueError, match='score arrays'):
        A.det_seg_scores_sweep(gts, prs, [0.5], scores=scores[:-1])
    with pytest.raises(ValueError, match='NaN'):
        A.det_seg_scores_sweep(gts, prs, [0.5, np.nan], scores=scores)
    with pytest.raises(ValueError, match='NaN'):
        A.det_seg_scores_sweep(gts, prs, [0.5], [0.5, np.nan], scores=scores)
    with pytest.raises(ValueError, match='negative'):
        A.det_seg_scores_sweep(gts, prs, [0.5], [-0.1], scores=scores)
    with pytest.raises(ValueError, match='at least one'):
        A.det_seg_scores_sweep(gts, prs, [], scores=scores)
    with pytest.raises(ValueError, match='scores are needed'):
        A.det_seg_scores_sweep(gts, prs, [0.5])
    with pytest.raises(ValueError, match='ground-truth images'):
        A.det_seg_scores_sweep(gts[:1], prs, [0.5], scores=scores)
    for bad in ([s.astype(np.int32) for s in scores], [list(s) for s in scores],
                [torch.from_numpy(s.astype(np.float32)).to(torch.bfloat16) for s in scores]):
        with pytest.raises(TypeError):
            A.det_seg_scores_sweep(gts, prs, [0.5], scores=bad)
    # masks of two frame sizes in one image
    mixed = [[gts[0][0] if gts[0] else _rle(np.ones((5, 5), bool))] + [_rle(np.ones((3, 4), bool))]]
    with pytest.raises(ValueError, match='different image sizes'):
        A.det_seg_scores_sweep(mixed, [[]], [0.5], scores=[np.zeros(0, np.float32)])


def _ref_fn(g, p, s, st, it):
    return S.sweep(g, p, s, st, it)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from ampis_b200 import distributed as D
    gts, prs, scores = _dataset(3, 7)
    r = D.sweep_sharded(gts, prs, SCORE_TH, IOU_TH, scores=scores, compute_fn=_ref_fn)
    loc = D.sweep_sharded(gts, prs, SCORE_TH, IOU_TH, scores=scores, compute_fn=_ref_fn, gather=False)
    q.put((rank, r, loc))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_sweep_sharded_two_ranks_gloo():
    gts, prs, scores = _dataset(3, 7)
    want = S.sweep(gts, prs, scores, SCORE_TH, IOU_TH)
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    for rank, r, loc in res:
        assert np.array_equal(r['index'], np.arange(rank, 7, 2))
        S.assert_same(r, want, 'rank %d' % rank)
        for k in ('n_pred', 'det_tp', 'seg_fn'):
            assert np.array_equal(loc[k], want[k][rank::2]), k
        assert np.array_equal(loc['totals'], want['totals'])
    # one process, no group: the same dict
    from ampis_b200 import distributed as D
    S.assert_same(D.sweep_sharded(gts, prs, SCORE_TH, IOU_TH, scores=scores, compute_fn=_ref_fn), want)
