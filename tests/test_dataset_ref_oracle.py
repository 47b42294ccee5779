"""tests/_dataset_ref.py -- the numpy / scipy reference the many-image entry is tested against at dataset scale --
pinned to the literal loops of oracle/ampis_ref.py (per-GT loop over 80-prediction chunks of rleIou, per-satellite
merges) on small seeded datasets: both modes, arg-max ties, IoUs exactly on a threshold, empty and full-frame masks,
images without rows, columns or either.  No GPU needed."""
import numpy as np

from oracle import ampis_ref as R
from oracle import cocomask as rle
from tests import _dataset_ref as D
from tests import _util as U

COCO_THRESHOLDS = np.arange(0.5, 1.0, 0.05)        # ampis_b200.batch.COCO_THRESHOLDS, as stored


def _enc(frames):
    return [rle.encode(np.asfortranarray(f.astype(np.uint8))) for f in frames]


def _images():
    rng = np.random.default_rng(20)
    imgs = []
    for h, w, g, p in ((23, 31, 9, 11), (40, 17, 6, 4), (1, 1, 2, 3), (50, 50, 12, 100), (7, 90, 5, 5)):
        rows, cols = _enc(U.rand_masks(rng, g, h, w, 0.2)), _enc(U.rand_masks(rng, p, h, w, 0.2))
        # exact copies: a row among the columns twice, a column duplicated further on, a row duplicated
        cols = cols[:2] + [rows[0]] + cols[2:] + [rows[0], cols[1]]
        rows = rows + [rows[1]]
        imgs.append((rows, cols))
    # IoU exactly k / 20: a 20-pixel ground truth and a k-pixel subset of it, k = 10 ... 20
    gt, pr = [], []
    for k in range(10, 21):
        f = np.zeros((30, 60), bool)
        y, x = 2 * (k % 7), 5 * (k - 10)
        f[y:y + 4, x:x + 5] = True
        gt.append(f.copy())
        sub = np.zeros(20, bool)
        sub[:k] = True
        f[y:y + 4, x:x + 5] = sub.reshape(5, 4).T
        pr.append(f)
    order = rng.permutation(len(pr))
    imgs.append((_enc(gt), _enc([pr[i] for i in order])))
    # a satellite overlapping two particles equally (the larger particle first) and zero-area satellites
    p0, p1, s0, s1 = (np.zeros((16, 16), bool) for _ in range(4))
    p0[:, :6] = True
    p1[:, 6:9] = True
    s0[6:8, 4:8] = True
    s1[1:3, 7:9] = True
    empty, full = np.zeros((16, 16), bool), np.ones((16, 16), bool)
    imgs.append((_enc([s0, empty, s1, empty, full]), _enc([p0, p1, empty])))
    # images without columns, without rows, without either
    imgs.append((imgs[0][0][:3], []))
    imgs.append(([], imgs[0][1][:4]))
    imgs.append(([], []))
    return imgs


def test_reference_equals_the_literal_loops():
    imgs = _images()
    ref = D.dataset([r for r, _ in imgs], [c for _, c in imgs], D.MODE_IOU, COCO_THRESHOLDS)
    sat = D.dataset([r for r, _ in imgs], [c for _, c in imgs], D.MODE_SAT)
    ties = on_threshold = near = 0
    for g, (rows, cols) in enumerate(imgs):
        one, s1 = ref['images'][g], sat['images'][g]
        masks = rows + cols
        assert np.array_equal(one['area'], rle.area(masks).astype(np.uint32) if masks else np.zeros(0, np.uint32))
        bb = np.array([rle.to_bbox(m) for m in masks]).reshape(-1, 4)
        want_bb = np.stack([bb[:, 0], bb[:, 1], bb[:, 0] + bb[:, 2] - 1, bb[:, 1] + bb[:, 3] - 1], axis=1)
        assert np.array_equal(one['bbox'], want_bb.astype(np.int32)) and not one['status'].any()
        # TP / FP / FN at every COCO threshold, as stored (0.6000000000000001 and not 0.6)
        for t, th in enumerate(COCO_THRESHOLDS):
            m = R.piecewise_rle_match(rows, cols, th)
            assert ref['grp_counts'][g, t].tolist() == [len(m['tp']), len(m['fp']), len(m['fn'])], (g, th)
            on_threshold += int((one['best_score'] == th).sum())
            near += int((np.abs(one['best_score'] - th) < 1e-12).sum())
        if rows and cols:
            # the loop's arg-max: a threshold of -1 makes every ground truth a match with its best column
            m = R.piecewise_rle_match(rows, cols, -1.0)
            assert np.array_equal(one['best_col'], m['tp'][:, 1]) and np.array_equal(one['best_score'], m['iou'])
            inter = [rle.merge_area(rows[i], cols[c], intersect=True) if c >= 0 else 0 for i, c in enumerate(one['best_col'])]
            assert one['best_inter'].tolist() == [int(v) for v in inter]
            iou = R.piecewise_iou(rows, cols)
            ties += int(sum(((iou[i] == iou[i].max()) & (iou[i] > 0)).sum() > 1 for i in range(len(rows))))
            # satellites: rows are satellites, columns particles (powder.py:80-86)
            nz = s1['best_score'] == s1['best_score']
            if nz.any():
                ms = R.rle_satellite_match(cols, rows, -1.0)
                assert np.array_equal(ms['satellite_matches'][:, 0], np.flatnonzero(nz))
                assert np.array_equal(s1['best_col'][nz], ms['satellite_matches'][:, 1])
                assert np.array_equal(s1['best_score'][nz], ms['intersection_scores'])
                inter = [rle.merge_area(rows[i], cols[c], intersect=True) for i, c in ms['satellite_matches']]
                assert s1['best_inter'][nz].tolist() == [int(v) for v in inter]
            assert (s1['best_col'][~nz] == 0).all() and (s1['best_inter'][~nz] == 0).all()
            assert (one['area'][:len(rows)][~nz] == 0).all()
        else:
            assert (one['best_col'] == -1).all() and (one['best_score'] == 0).all() and (one['best_inter'] == 0).all()
    assert np.array_equal(ref['totals'], ref['grp_counts'].astype(np.int64).sum(axis=0))
    # the cases the dataset is there for did occur: ties, IoUs equal to the stored 0.5 and 0.55 and a few ulps below
    # 0.6000000000000001 ... 0.9500000000000004
    assert ties >= 3 and on_threshold >= 2 and near >= 10
    eq = sat['images'][6]
    assert eq['best_col'][0] == 0 and ref['images'][6]['best_col'][0] == 1      # SAT: first max of I; IoU: smaller union
    assert np.isnan(eq['best_score'][[1, 3]]).all()
