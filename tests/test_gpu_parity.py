"""GPU parity tests (run on the B200 box with ``-m gpu``): the CUDA path, called through the
public drop-in API and the C ABI, against the CPU oracle and the frozen golden fixtures.
Bit-exact for intersections, matches, counts, areas and boxes; float64 scores are compared
for equality too (they are correctly-rounded divisions of exact integers, SURVEY.md A.6),
with 1e-6 relative as the stated tolerance for derived quantities (d_eq, psd)."""
import os

import numpy as np
import pytest

from tests import _util as U

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def mods():
    import torch
    assert torch.cuda.is_available(), 'these tests need the B200'
    from ampis_b200 import analyze, batch, data_utils, engine, structures
    from ampis_b200.applications import powder
    from oracle import ampis_ref as R
    from oracle import cocomask as rle

    class M:
        pass
    m = M()
    m.torch, m.analyze, m.batch, m.data_utils, m.engine, m.structures = torch, analyze, batch, data_utils, engine, \
        structures
    m.powder, m.R, m.rle = powder, R, rle
    return m


def _enc(rle, a):
    return rle.encode(np.asfortranarray(np.array(a, np.uint8)))


def test_reference_known_answer(mods):
    """analyze.py:702-728 through the GPU path."""
    A, rle = mods.analyze, mods.rle
    m1 = _enc(rle, [[1, 1, 0, 0], [1, 1, 0, 0], [0, 0, 0, 0], [0, 0, 0, 0]])
    m2 = _enc(rle, [[0, 0, 1, 1], [0, 0, 1, 1], [0, 0, 0, 0], [0, 0, 0, 0]])
    m3 = _enc(rle, [[0, 0, 0, 0], [0, 0, 0, 0], [1, 1, 0, 0], [1, 1, 0, 0]])
    m4 = _enc(rle, [[0, 0, 0, 0], [0, 0, 0, 0], [0, 0, 1, 1], [0, 0, 1, 1]])
    gt, pred = [m1, m2, m3, m4], [m3, m2, m4]
    assert np.all(A._piecewise_iou(gt, pred) == np.array([[0, 0, 0], [0, 1, 0], [1, 0, 0], [0, 0, 1]]))
    match = A._piecewise_rle_match(gt, pred)
    assert np.all(match['tp'] == np.array([[1, 1], [2, 0], [3, 2]]))
    assert np.all(match['fn'] == np.array([0]))
    assert np.all(match['fp'] == np.array([]))
    assert np.all(match['iou'] == np.ones(3))
    assert match['tp'].dtype == np.int64 and match['iou'].dtype == np.float64


def test_string_codec_and_measure_on_fixtures(mods):
    E, rle, torch = mods.engine, mods.rle, mods.torch
    m = U.load('spheroidite_measure.npz')
    for k in range(len(m['names'])):
        masks = U.unpack_strings(m['%d_blob' % k], m['%d_off' % k], m['%d_size' % k])
        t = E.table_from_rle(masks)
        # counts decoded on the GPU == oracle rleFrString
        cnt = t.cnt.cpu().numpy().view(np.uint32)
        off = t.cnt_off.cpu().numpy()
        ln = t.cnt_len.cpu().numpy()
        for i in range(0, len(masks), 7):
            assert np.array_equal(cnt[off[i]:off[i] + ln[i]], rle.counts_from_string(masks[i]['counts']))
        assert np.array_equal(t.areas_np(), m['%d_area' % k])
        bb = t.bbox_np()
        ne = m['%d_area' % k] > 0
        assert np.array_equal(bb[ne].astype(np.float64), m['%d_boxes_d2' % k][ne])
        assert (bb[~ne] == [0, 0, -1, -1]).all()
        # GPU re-encode gives back the bytes pycocotools wrote
        s = E.counts_to_strings(t.cnt, t.cnt_off, t.cnt_len, t.n)
        assert s == [x['counts'] for x in masks]


def test_string_decode_of_long_numbers_and_any_alignment(mods):
    """rleFrString on the GPU (both kernels: a warp per mask for small batches, a thread per mask for large ones)
    against the oracle on strings the fixtures do not hold: numbers of one to ten characters (only the first seven reach the low 32 bits), counts up to 2^28 with
    negative deltas, strings of 0 to ~1,000 characters (several steps, carries of an unfinished number and of both
    delta chains), laid back to back so that they start at every byte alignment."""
    E, rle, torch = mods.engine, mods.rle, mods.torch
    rng = np.random.default_rng(77)
    strings = []
    for t in range(1500):
        if t % 2 == 0:
            m = int(rng.integers(0, 260))
            mag = int(rng.choice([4, 40, 1000, 70000, 2 ** 22, 2 ** 28]))
            strings.append(rle.string_from_counts(rng.integers(0, mag, m, dtype=np.int64).astype(np.uint32)))
        else:
            out = bytearray()
            for _ in range(int(rng.integers(0, 120))):
                k = int(rng.integers(1, 11))
                out += bytes((48 + (int(rng.integers(0, 32)) | 0x20)) for _ in range(k - 1))
                out += bytes([48 + int(rng.integers(0, 32))])
            strings.append(bytes(out))
    want_of = [rle.counts_from_string(x) if len(x) else np.zeros(0, np.uint32) for x in strings]
    # 1,500 strings go through the warp-per-mask kernel (small batches), 18,000 through the thread-per-mask one
    for reps in (1, 12):
        _check_string_decode(mods, strings * reps, want_of * reps, leads=range(4) if reps == 1 else (0, 3))


def _check_string_decode(mods, strings, want_of, leads):
    E, torch = mods.engine, mods.torch
    n = len(strings)
    lens = np.array([len(x) for x in strings], np.int64)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    blob = np.frombuffer(b''.join(strings), np.uint8)
    for lead in leads:                                     # every alignment of the first string, too
        d_chars = torch.from_numpy(np.concatenate([np.zeros(lead, np.uint8), blob])).cuda()
        d_off = torch.from_numpy(off + lead).cuda()
        cnt = torch.full((int(off[-1]) + lead + 1,), -1, dtype=torch.int32, device='cuda')
        cnt_len = torch.empty(n, dtype=torch.int32, device='cuda')
        E.N.call('ampis_rle_string_decode', E._p(d_chars), E._p(d_off), n, E._p(cnt), E._p(d_off), E._p(cnt_len),
                 E._stream())
        got, ln = cnt.cpu().numpy().view(np.uint32), cnt_len.cpu().numpy()
        for i in range(n):
            want = want_of[i]
            assert ln[i] == len(want), (lead, i)
            assert np.array_equal(got[off[i] + lead: off[i] + lead + ln[i]], want), (lead, i)


def test_structures_measurements(mods):
    S, R = mods.structures, mods.R
    from ampis_b200.containers import Instances
    m = U.load('spheroidite_measure.npz')
    masks = U.unpack_strings(m['0_blob'], m['0_off'], m['0_size'])
    size = tuple(int(v) for v in m['0_size'])
    areas = S.mask_areas(masks)
    assert areas.dtype == np.uint32 and np.array_equal(areas, m['0_area'])
    assert np.array_equal(S.mask_areas(S.RLEMasks(masks)), m['0_area'])
    n = len(masks)
    iset = S.InstanceSet(instances=Instances(size, masks=S.RLEMasks(masks), boxes=np.zeros((n, 4)),
                                             class_idx=np.zeros(n, np.int64)))
    filt = iset.filter_mask_size(100, 100000)
    assert len(filt) == int(m['0_size_inliers'].sum())
    assert filt.masks.rle == [x for x, b in zip(masks, m['0_size_inliers']) if b]
    df = iset.compute_rprops(keys=['area', 'equivalent_diameter', 'bbox'], return_df=True)
    ne = m['0_area'] > 0
    got = np.array([v[0] for v in df['equivalent_diameter'][ne]])
    assert np.allclose(got, m['0_deq'][ne], rtol=1e-6, atol=0)
    assert [int(v[0]) for v in df['area'][ne]] == m['0_area'][ne].tolist()
    for k in (1, 3):
        i2 = iset.copy()
        i2.remove_edge_instances(k)
        want = R.edge_inliers(masks, size, k)
        assert i2.instances.masks.rle == [x for x, b in zip(masks, want) if b]
    i2 = iset.copy()
    i2.remove_edge_instances(0)          # reference quirk: k=0 removes every non-empty mask
    assert len(i2.instances) == int((m['0_area'] == 0).sum())


def test_bitmask_array_and_extract_boxes(mods):
    S, D, R = mods.structures, mods.data_utils, mods.R
    m = U.load('spheroidite_measure.npz')
    masks = U.unpack_strings(m['1_blob'], m['1_off'], m['1_size'])[:40]
    bm = S.masks_to_bitmask_array(masks)
    want = R.rle_to_bitmask_array(masks)
    assert bm.dtype == np.bool_ and bm.shape == want.shape and (bm == want).all()
    one = S.masks_to_bitmask_array(S.RLEMasks(masks)[3])
    assert one.shape == (1,) + want.shape[1:] and (one[0] == want[3]).all()
    assert np.array_equal(D.extract_boxes(bm), R.extract_boxes(want))
    assert np.array_equal(D.extract_boxes(bm, box_mode='matterport'), R.extract_boxes(want, box_mode='matterport'))
    mp = np.ascontiguousarray(want.transpose(1, 2, 0))
    assert np.array_equal(D.extract_boxes(mp, mask_mode='matterport'), R.extract_boxes(mp, mask_mode='matterport'))
    assert np.array_equal(D.extract_boxes(want[5]), R.extract_boxes(want[5]))
    assert np.array_equal(S.mask_areas(want), want.sum(axis=(1, 2), dtype=np.uint))
    # odd sizes: packed layout is exercised where h is not a multiple of 32
    rng = np.random.default_rng(5)
    for h, w in [(1, 1), (5, 3), (33, 7), (31, 129), (100, 64)]:
        a = U.rand_masks(rng, 6, h, w)
        enc = [mods.rle.encode(np.asfortranarray(x.astype(np.uint8))) for x in a]
        assert (S.masks_to_bitmask_array(enc) == a).all()
        assert np.array_equal(S.mask_areas(enc), a.sum(axis=(1, 2)).astype(np.uint32))
        assert np.array_equal(D.extract_boxes(a), R.extract_boxes(a))


@pytest.mark.parametrize('layout', ['span', 'full', 'crop', 'one_call'])
def test_golden_matching_all_images(mods, layout, monkeypatch):
    A, E = mods.analyze, mods.engine
    # 'one_call': the product default (ampis_eval_image_host per image); the others: the table API in each layout
    monkeypatch.setattr(A, 'FUSED_CALL', layout == 'one_call')
    if layout != 'one_call':
        monkeypatch.setattr(E, 'MATCH_LAYOUT', {'full': E.LAYOUT_FULL, 'span': E.LAYOUT_SPAN, 'crop': E.LAYOUT_CROP}[layout])
    g = U.load('powder_match.npz')
    for k in range(len(g['names'])):
        _, gt, pr = U.powder_match_image(k)
        res = A.det_seg_scores(gt, pr, 0.5)
        for key in ('det_tp', 'det_fn', 'det_fp', 'seg_tp', 'seg_fn', 'seg_fp', 'det_tp_iou', 'seg_precision',
                    'seg_recall'):
            want = g['%d_%s' % (k, key)]
            assert np.asarray(res[key]).dtype == want.dtype, key
            assert np.array_equal(np.asarray(res[key]), want), (k, key)
        assert [res['det_precision'], res['det_recall']] == list(g['%d_det_pr' % k])
        if k < 2:
            iou = A._piecewise_iou(gt, pr)
            nz = np.argwhere(iou > 0)
            assert np.array_equal(nz, g['%d_iou_nz_idx' % k])
            assert np.array_equal(iou[nz[:, 0], nz[:, 1]], g['%d_iou_nz_val' % k])
        for t, want in zip(g['thresholds'][1::3], g['%d_thr_counts' % k][1::3]):
            mt = A.rle_instance_matcher(gt, pr, t)
            assert [len(mt['tp']), len(mt['fp']), len(mt['fn'])] == list(want)


def test_golden_satellites(mods):
    P, S = mods.powder, mods.structures
    from ampis_b200.containers import Instances
    s = U.load('powder_satellite.npz')
    psis = []
    for k in range(len(s['names'])):
        _, part, sat = U.powder_satellite_image(k)
        size = tuple(int(v) for v in s['%d_size' % k])
        res = P._rle_satellite_match(part, sat, 0.5)
        for key in ('satellite_matches', 'satellites_unmatched', 'particles_unmatched', 'intersection_scores'):
            assert np.array_equal(res[key], s['%d_%s' % (k, key)]), (k, key)
            assert res[key].dtype == s['%d_%s' % (k, key)].dtype
        mk = lambda ms: S.InstanceSet(instances=Instances(size, masks=S.RLEMasks(ms),
                                                          boxes=np.zeros((len(ms), 4))))
        psi = P.PowderSatelliteImage(mk(part), mk(sat))
        psi.compute_matches()
        assert psi.matches['match_pairs'] == res['match_pairs']
        met = psi.compute_satellite_metrics()
        assert np.array_equal(met['mask_areas_all'], mods.rle.area(part))
        psis.append(psi)
    got = P.satellite_measurements(psis, print_summary=False, output_dict=True)
    want = mods.R.satellite_measurements([p.matches for p in psis], [len(p.particles.instances) for p in psis],
                                         [len(p.satellites.instances) for p in psis])
    for key in want:
        assert np.array_equal(np.asarray(got[key]), np.asarray(want[key])), key
    # size distribution: same numerics as the oracle on the same areas, within 1e-6
    isets = [p.particles for p in psis]
    for x in isets:
        x.HFW, x.HFW_units = 103.6, 'um'
    out = P.psd(isets, plot=False, return_results=True)
    ref = mods.R.psd_from_areas([mods.rle.area(p.particles.instances.masks.rle) * (103.6 / 1536) ** 2 for p in psis])
    assert np.allclose(out['x'], ref['x'], rtol=1e-6, atol=0) and np.allclose(out['y'], ref['y'], rtol=1e-6, atol=0)
    assert out['x_label'] == 'Equivalent diameter, um'


def test_golden_polygons(mods):
    S = mods.structures
    from ampis_b200.containers import PolygonMasks
    p = U.load('powder_polygons.npz')
    xy, off = p['0_poly_xy'], p['0_poly_off']
    size = tuple(int(v) for v in p['0_size'])
    polys = [[xy[off[i]:off[i + 1]]] for i in range(len(off) - 1)]
    got = S.masks_to_rle(PolygonMasks(polys), size)
    want = U.unpack_strings(p['0_rle_blob'], p['0_rle_off'], size)
    assert [g['counts'] for g in got] == [w['counts'] for w in want]
    assert np.array_equal(S.mask_areas(got), p['0_area'])


def test_polygons_random_vs_oracle(mods):
    S, rle = mods.structures, mods.rle
    from ampis_b200.containers import PolygonMasks
    rng = np.random.default_rng(11)
    for h, w in [(37, 53), (128, 96), (300, 200)]:
        polys = []
        for _ in range(60):
            k = int(rng.integers(3, 30))
            if rng.random() < 0.3:     # integer / half-integer vertices provoke ties and duplicate crossings
                pts = rng.integers(-3, max(h, w) + 3, (k, 2)).astype(np.float64) + rng.choice([0.0, 0.5])
            else:
                ang = np.sort(rng.uniform(0, 2 * np.pi, k))
                r = rng.uniform(0.2, 0.6) * min(h, w) * rng.uniform(0.5, 1.0, k)
                pts = np.stack([w * rng.uniform(0.1, 0.9) + r * np.cos(ang), h * rng.uniform(0.1, 0.9) + r * np.sin(ang)], 1)
            polys.append([pts.ravel()])
        polys.append([np.array([0.0, 0.0, float(w), 0.0, float(w), float(h), 0.0, float(h)])])   # whole frame
        polys.append([np.array([5.0, 5.0, 5.0, 5.0, 5.0, 5.0])])                                    # degenerate
        got = S.masks_to_rle(PolygonMasks(polys), (h, w))
        want = [rle.frPyObjects(q, h, w)[0] for q in polys]
        for i, (a, b) in enumerate(zip(got, want)):
            assert a['counts'] == b['counts'], (h, w, i)


def _counts_to_rle(rle, cnts, h, w):
    return [{'size': [h, w], 'counts': rle.string_from_counts(c)} for c in cnts]


def test_random_masks_match_oracle(mods):
    """Ragged / empty / odd-sized inputs: GPU matcher and satellite assignment == oracle."""
    A, P, R, rle = mods.analyze, mods.powder, mods.R, mods.rle
    rng = np.random.default_rng(3)
    for h, w, G, Pn in [(7, 9, 3, 4), (33, 31, 12, 9), (64, 100, 40, 70), (50, 37, 1, 90), (129, 65, 85, 2)]:
        a = U.rand_masks(rng, G, h, w)
        b = U.rand_masks(rng, Pn, h, w)
        b[: min(G, Pn) // 2] = a[: min(G, Pn) // 2]          # exact duplicates -> IoU 1 and ties
        ea = [rle.encode(np.asfortranarray(x.astype(np.uint8))) for x in a]
        eb = [rle.encode(np.asfortranarray(x.astype(np.uint8))) for x in b]
        assert np.array_equal(A._piecewise_iou(ea, eb), R.piecewise_iou(ea, eb))
        for th in (0.0, 0.3, 0.5, 0.99):
            got, want = A._piecewise_rle_match(ea, eb, th), R.piecewise_rle_match(ea, eb, th)
            for key in want:
                assert np.array_equal(got[key], want[key]) and got[key].shape == want[key].shape, (key, th)
        try:
            want = R.rle_satellite_match(eb, ea, 0.5)
        except IndexError:
            with pytest.raises(IndexError):
                P._rle_satellite_match(eb, ea, 0.5)
        else:
            got = P._rle_satellite_match(eb, ea, 0.5)
            for key in ('satellite_matches', 'satellites_unmatched', 'particles_unmatched', 'intersection_scores'):
                assert np.array_equal(got[key], want[key]), key
            assert got['match_pairs'] == want['match_pairs']
    with pytest.raises(ZeroDivisionError):
        A.det_seg_scores(mods.structures.RLEMasks([]), mods.structures.RLEMasks([]), 0.5)
    with pytest.raises(IndexError):          # masks_to_rle peeks at masks[0] (structures.py:665)
        A.det_seg_scores([], [], 0.5)


def test_empty_and_error_conventions(mods):
    A, S, rle = mods.analyze, mods.structures, mods.rle
    z = _enc(rle, np.zeros((6, 5)))
    o = _enc(rle, np.ones((6, 5)))
    assert A._piecewise_rle_match([z], [z])['tp'].shape == (0,)
    m = A._piecewise_rle_match([o, z], [])
    assert m['fn'].tolist() == [0, 1] and m['fp'].tolist() == [] and m['tp'].shape == (0,)
    m = A._piecewise_rle_match([], [o, z])
    assert m['fp'].tolist() == [0, 1] and m['fn'].tolist() == []
    with pytest.raises(NotImplementedError):
        S.masks_to_rle(np.zeros((2, 3, 3), bool))
    with pytest.raises(NotImplementedError):
        S.mask_areas('nope')
    with pytest.raises(AssertionError):
        from ampis_b200.containers import PolygonMasks
        S.masks_to_rle(PolygonMasks([[np.array([1., 1, 5, 1, 5, 5])]]))
    with pytest.raises(ValueError):
        S.mask_areas([{'size': [6, 5], 'counts': rle.string_from_counts(np.array([3, 3], np.uint32))}])
    # counts that overshoot the frame are flagged in every storage layout (and painted without writing outside
    # the mask's region: the run below would reach far beyond a 45 x 37 frame)
    good = _enc(rle, np.ones((45, 37)))
    bad = [{'size': [45, 37], 'counts': rle.string_from_counts(np.array([3, 5000, 7, 900], np.uint32))}, good, good]
    for lay in (mods.engine.LAYOUT_SPAN, mods.engine.LAYOUT_FULL, mods.engine.LAYOUT_CROP):
        with pytest.raises(ValueError, match='malformed RLE'):
            mods.engine.table_from_rle(bad, layout=lay)
    assert S.mask_areas([good]).tolist() == [45 * 37]


@pytest.mark.parametrize('cfg,n_img', [('c1_powder_example', 2), ('c2_powder_batch', 2)])
@pytest.mark.parametrize('layout,fused', [('span', False), ('full', False), ('span', True), ('full', True),
                                          ('crop', False), ('crop', True)])
def test_batch_pipeline_vs_oracle(mods, cfg, n_img, layout, fused):
    """Synthetic images through the batch pipeline == oracle per image (matches, IoUs, counts at
    the ten COCO thresholds, dense intersections)."""
    B, E, R, rle = mods.batch, mods.engine, mods.R, mods.rle
    host = B.synth(cfg, n_img, 1001)
    dev = B.DeviceBatch(host, dense=True)
    lay = {'full': E.LAYOUT_FULL, 'span': E.LAYOUT_SPAN, 'crop': E.LAYOUT_CROP}[layout]
    arena = None
    if fused:
        arena = mods.torch.empty(4 * B.arena_chunks_needed(dev, lay), dtype=mods.torch.int32, device='cuda')
    res = B.eval_step(dev, layout=lay, check=True, arena=arena)
    G, Pn = host.n_rows, host.n_cols
    best_col = res.rows.best_col.cpu().numpy().reshape(n_img, G)
    best_iou = res.rows.best_score.cpu().numpy().reshape(n_img, G)
    counts = res.counts.cpu().numpy()
    imat = res.rows.imat.cpu().numpy().reshape(n_img, G, Pn)
    tot = np.zeros((len(B.COCO_THRESHOLDS), 3), np.int64)
    for g in range(n_img):
        rows, cols = host.image_masks(g)
        er, ec = _counts_to_rle(rle, rows, host.h, host.w), _counts_to_rle(rle, cols, host.h, host.w)
        iou = R.piecewise_iou(er, ec)
        ar, ac = rle.area(er).astype(np.int64), rle.area(ec).astype(np.int64)
        # dense intersections: invert iou = I/(a+b-I) exactly where iou>0 via the oracle merge on a sample
        nz = np.argwhere(iou > 0)
        assert np.array_equal(np.argwhere(imat[g] > 0), nz)
        for i, j in nz[:: max(1, len(nz) // 200)]:
            assert imat[g, i, j] == int(rle.merge_area(er[i], ec[j]))
        I = imat[g].astype(np.int64)
        with np.errstate(invalid='ignore', divide='ignore'):
            mine = np.where(I > 0, I / (ar[:, None] + ac[None, :] - I), 0.0)
        assert np.array_equal(mine, iou)
        assert (np.diff(counts[g, :, 0]) <= 0).all()
        for ti in (0, 5, 9):
            th = B.COCO_THRESHOLDS[ti]
            m = R.piecewise_rle_match(er, ec, th)
            assert counts[g, ti].tolist() == [len(m['tp']), len(m['fp']), len(m['fn'])]
            tot[ti] += counts[g, ti]
            if ti == 0:
                matched = best_iou[g] > th
                assert np.array_equal(np.nonzero(matched)[0], m['tp'][:, 0])
                assert np.array_equal(best_col[g][matched], m['tp'][:, 1])
                assert np.array_equal(best_iou[g][matched], m['iou'])
    assert np.array_equal(res.totals.cpu().numpy()[[0, 5, 9]], tot[[0, 5, 9]])
    assert np.array_equal(res.totals.cpu().numpy(), counts.sum(axis=0))


def test_batch_satellites_vs_oracle(mods):
    B, E, R, rle = mods.batch, mods.engine, mods.R, mods.rle
    cfg = dict(B.CONFIGS['c3_satellites'], h=512, w=512, n_rows=40, n_cols=300)
    host = B.synth(cfg, 3, 3003)
    dev = B.DeviceBatch(host)
    res = B.eval_step(dev, check=True)
    S, Np = host.n_rows, host.n_cols
    best = res.rows.best_col.cpu().numpy().reshape(3, S)
    score = res.rows.best_score.cpu().numpy().reshape(3, S)
    counts = res.counts.cpu().numpy()
    spp = np.zeros(64, np.int64)
    for g in range(3):
        rows, cols = host.image_masks(g)
        er, ec = _counts_to_rle(rle, rows, host.h, host.w), _counts_to_rle(rle, cols, host.h, host.w)
        want = R.rle_satellite_match(ec, er, 0.5)
        with np.errstate(invalid='ignore'):
            matched = score[g] > 0.5
        assert np.array_equal(np.stack([np.nonzero(matched)[0], best[g][matched]], 1), want['satellite_matches'])
        assert np.array_equal(score[g][matched], want['intersection_scores'])
        assert counts[g].tolist() == [len(want['satellite_matches']), len(want['satellites_unmatched']),
                                      len(want['match_pairs']), Np]
        for v in want['match_pairs'].values():
            spp[min(len(v), 63)] += 1
    assert np.array_equal(res.spp_hist.cpu().numpy(), spp)


@pytest.mark.parametrize('cfg,over,n_img', [
    ('c2_powder_batch', {}, 3),
    ('c4_spheroidite', dict(n_rows=1500, n_cols=1500, h=1024, w=1024), 2),
    ('dense_overlap', {}, 1),
    ('c3_satellites', dict(n_cols=600, h=1024, w=1024), 2),
    ('c2_powder_batch', dict(h=70, w=45, n_rows=9, n_cols=11, median_diam=30.0), 4),      # windows wider than the frame
])
def test_crop_layout_equals_span_layout(mods, cfg, over, n_img):
    """AMPIS_LAYOUT_CROP (bounding-box windows) == AMPIS_LAYOUT_SPAN bit for bit: measurements, dense
    intersections, arg-max, scores, counts -- fused and unfused construction."""
    B, E, torch = mods.batch, mods.engine, mods.torch
    host = B.synth(dict(B.CONFIGS[cfg], **over), n_img, 777)
    dev = B.DeviceBatch(host, dense=True)
    a = B.eval_step(dev, layout=E.LAYOUT_SPAN, check=True)
    b = B.eval_step(dev, layout=E.LAYOUT_CROP, check=True)                       # measure, scan, crop painter
    arena = torch.empty(4 * B.arena_chunks_needed(dev, E.LAYOUT_CROP), dtype=torch.int32, device='cuda')
    c = B.eval_step(dev, layout=E.LAYOUT_CROP, check=True, arena=arena)          # fused measure+paint
    assert B.arena_chunks_needed(dev, E.LAYOUT_CROP) <= B.arena_chunks_needed(dev, E.LAYOUT_SPAN) or host.h < 128
    for o in (b, c):
        assert torch.equal(a.rows.imat, o.rows.imat)
        assert torch.equal(a.rows.best_col, o.rows.best_col) and torch.equal(a.rows.best_inter, o.rows.best_inter)
        assert np.array_equal(a.rows.best_score.cpu().numpy(), o.rows.best_score.cpu().numpy(), equal_nan=True)
        assert torch.equal(a.counts, o.counts)
        assert torch.equal(a.table.area, o.table.area) and torch.equal(a.table.bbox, o.table.bbox)
    assert int(a.rows.imat.max()) > 0


@pytest.mark.parametrize('cfg,over,n_img', [
    ('c2_powder_batch', {}, 3),
    ('c4_spheroidite', dict(n_rows=1500, n_cols=1500, h=1024, w=1024), 2),
    ('c4_spheroidite', dict(n_rows=700, n_cols=900, h=300, w=2000), 2),                    # cells clamp on one axis
    ('dense_overlap', {}, 1),                                                              # boxes over many cells
    ('c3_satellites', dict(n_cols=1200, h=1024, w=1024), 2),
    ('c2_powder_batch', dict(h=70, w=45, n_rows=9, n_cols=11, median_diam=30.0), 4),
    ('c2_powder_batch', dict(h=512, w=512, n_rows=40, n_cols=40, median_diam=150.0), 2),   # large overlaps: warp-wide phase
    ('dense_overlap', dict(h=512, w=512, n_rows=64, n_cols=64, median_diam=220.0), 2),     # ... more than a warp parks
])
@pytest.mark.parametrize('rows_kernel', ['pairs', 'grid'])
def test_grid_pruned_rows_equal_scanned_rows(mods, cfg, over, n_img, rows_kernel, monkeypatch):
    """Crop rows with the box pre-pruning through the uniform grid -- as the three-pass join ('pairs') and as the
    single rows kernel of round 1 ('grid') -- == the kernel that tests every column's box, bit for bit (dense
    matrix, arg-max, scores, counts); the sparse output is exactly the set of non-zero cells of the dense matrix."""
    B, E, torch = mods.batch, mods.engine, mods.torch
    monkeypatch.setattr(E, 'ROWS_KERNEL', rows_kernel)
    host = B.synth(dict(B.CONFIGS[cfg], **over), n_img, 4242)
    dev = B.DeviceBatch(host, dense=True)
    a = B.eval_step(dev, layout=E.LAYOUT_CROP, check=True, kernel='scan')
    sp = E.SparseRows('cuda', dev.groups.imat_size)
    b = B.eval_step(dev, layout=E.LAYOUT_CROP, check=True, kernel='grid', sparse=sp)
    assert b.rows.grid.needed() == b.rows.grid.capacity > 0
    assert torch.equal(a.rows.imat, b.rows.imat)
    assert torch.equal(a.rows.best_col, b.rows.best_col) and torch.equal(a.rows.best_inter, b.rows.best_inter)
    assert np.array_equal(a.rows.best_score.cpu().numpy(), b.rows.best_score.cpu().numpy(), equal_nan=True)
    assert torch.equal(a.counts, b.counts)
    r, c, v = (x.cpu().numpy() for x in sp.triplets())
    G, Pn = host.n_rows, host.n_cols
    I = a.rows.imat.cpu().numpy()[:n_img * G * Pn].reshape(n_img * G, Pn)
    wr, wc = np.nonzero(I)
    assert np.array_equal(r, wr) and np.array_equal(c, wc) and np.array_equal(v, I[wr, wc])
    # no dense matrix at all: same rows
    dev2 = B.DeviceBatch(host, dense=False)
    d = B.eval_step(dev2, layout=E.LAYOUT_CROP, kernel='grid')
    assert torch.equal(a.rows.best_col, d.rows.best_col) and torch.equal(a.counts, d.counts)
    # pre-sized pipeline form (what bench.py runs)
    arena = torch.empty(4 * B.arena_chunks_needed(dev2, E.LAYOUT_CROP), dtype=torch.int32, device='cuda')
    pipe = B.Pipeline(dev2, E.LAYOUT_CROP, arena, kernel='grid', sparse_capacity=sp.capacity)
    pipe.launch()
    pipe.launch()
    assert torch.equal(pipe.rows.best_col[:dev2.groups.n_rows], a.rows.best_col[:dev2.groups.n_rows])
    assert int(pipe.sparse.count.item()) == len(wr)
    assert pipe.grid.needed() == pipe.grid.capacity
    if rows_kernel == 'pairs':
        # the pair list holds every pair with overlapping boxes (at least the non-zero ones), sized exactly by the dry run
        assert pipe.pairs.needed() == pipe.pairs.capacity >= len(wr)
        # a list that is too small is detected, not overrun
        short = E.PairList('cuda', dev2.groups.n_rows, max(pipe.pairs.capacity // 3, 1))
        t = E.MaskTable(pipe.table.device, host.n_masks, dev2.cnt, dev2.cnt_off, dev2.cnt_len, dev2.h, dev2.w,
                        E.LAYOUT_CROP).measure_paint(arena)
        E.intersect_rows(t, dev2.groups, dev2.mode, grid=pipe.grid, pairs=short)
        assert short.needed() == pipe.pairs.capacity > short.capacity


def test_sparse_iou_equals_nonzeros_of_the_dense_matrix(mods):
    """analyze.sparse_iou == the non-zero cells of analyze._piecewise_iou (which the oracle pins), golden
    powder image and a synthetic spheroidite frame; also the empty conventions."""
    A, B, rle = mods.analyze, mods.batch, mods.rle
    _, gt, pr = U.powder_match_image(0)
    host = B.synth(dict(B.CONFIGS['c4_spheroidite'], n_rows=1200, n_cols=1100, h=1024, w=1024), 1, 99)
    rows, cols = host.image_masks(0)
    mk = lambda cs: [{'size': [host.h, host.w], 'counts': rle.string_from_counts(c)} for c in cs]
    for a, b in ((gt, pr), (mk(rows), mk(cols))):
        dense = A._piecewise_iou(a, b)
        sp = A.sparse_iou(a, b)
        wr, wc = np.nonzero(dense)
        assert sp['shape'] == dense.shape and len(wr) > 0
        assert np.array_equal(sp['row'], wr) and np.array_equal(sp['col'], wc)
        assert np.array_equal(sp['iou'], dense[wr, wc])
        assert sp['inter'].dtype == np.uint32 and sp['inter'].min() > 0
    e = A.sparse_iou([], pr)
    assert e['shape'] == (0, len(pr)) and len(e['row']) == 0


@pytest.mark.parametrize('cfg,over,n_img', [
    ('c2_powder_batch', {}, 2),
    ('c4_spheroidite', dict(n_rows=900, n_cols=900, h=1024, w=1024), 2),
    ('c2_powder_batch', dict(h=600, w=500, n_rows=30, n_cols=30, median_diam=170.0), 2),   # > 64 / 128 runs: global run ends, several tiles
    ('c2_powder_batch', dict(h=70, w=45, n_rows=9, n_cols=11, median_diam=30.0), 3),
])
def test_crop_decode_lane_groups_agree(mods, cfg, over, n_img, monkeypatch):
    """The fused crop decode kernel with 8, 16 or 32 lanes per mask (chosen from a runs-per-mask hint) writes the
    same measurements and, through the rows kernel, the same intersections as the unfused measure / scan / paint."""
    B, E, torch = mods.batch, mods.engine, mods.torch
    host = B.synth(dict(B.CONFIGS[cfg], **over), n_img, 31337)
    dev = B.DeviceBatch(host, dense=True)
    ref = B.eval_step(dev, layout=E.LAYOUT_CROP, check=True, fused=False, kernel='scan')
    arena = torch.empty(4 * B.arena_chunks_needed(dev, E.LAYOUT_CROP), dtype=torch.int32, device='cuda')
    # group decode: warp per mask, 8 lanes, 16 lanes; flat decode: 4, 16, 10, 3, 1 masks per warp
    for decode, hint in [('group', 0), ('group', 30), ('group', 100), ('flat', 0), ('flat', 2), ('flat', 30),
                         ('flat', 100), ('flat', 400)]:
        monkeypatch.setattr(E, 'CROP_DECODE', decode)
        monkeypatch.setattr(E, 'PAINT_RUNS_HINT', hint)
        got = B.eval_step(dev, layout=E.LAYOUT_CROP, check=True, arena=arena, kernel='scan')
        n = host.n_masks
        tag = (decode, hint)
        assert torch.equal(got.table.area[:n], ref.table.area[:n]) and torch.equal(got.table.bbox[:4 * n], ref.table.bbox[:4 * n]), tag
        assert torch.equal(got.table.status[:n], ref.table.status[:n]), tag
        assert torch.equal(got.table.span[:2 * n], ref.table.span[:2 * n]) and torch.equal(got.table.reg[:2 * n], ref.table.reg[:2 * n]), tag
        assert int(got.table.cursor.item()) == int(ref.table.bits_off[n].item()), tag      # same arena need
        assert torch.equal(got.rows.imat, ref.rows.imat), tag
        assert torch.equal(got.rows.best_col, ref.rows.best_col) and torch.equal(got.counts, ref.counts), tag


def _csr_table(mods, masks_bool, layout):
    """bool[n,h,w] -> (device MaskTable inputs) through the oracle's encoder."""
    E, rle, torch = mods.engine, mods.rle, mods.torch
    n, h, w = masks_bool.shape
    cnts = [rle.counts_from_string(rle.encode(np.asfortranarray(m.astype(np.uint8)))['counts']) for m in masks_bool]
    lens = np.array([len(c) for c in cnts], np.int32)
    off = np.zeros(n, np.int64)
    off[1:] = np.cumsum(lens[:-1])
    dev = 'cuda'
    cnt = torch.from_numpy(np.concatenate(cnts).astype(np.uint32).view(np.int32)).to(dev)
    return E.MaskTable(torch.device('cuda', torch.cuda.current_device()), n, cnt, torch.from_numpy(off).to(dev),
                       torch.from_numpy(lens).to(dev), torch.full((n,), h, dtype=torch.int32, device=dev),
                       torch.full((n,), w, dtype=torch.int32, device=dev), layout)


def test_flat_decode_clears_the_buffer_it_is_handed(mods, monkeypatch):
    """MaskTable.measure_paint(arena, zero=buf): the flat crop decode also clears buf (the dense matrices of the rows
    that follow), whatever its length -- whole 16-byte chunks by the kernel, a tail by a memset, nothing beyond it --
    and decodes exactly what it decodes without the side job."""
    E, torch = mods.engine, mods.torch
    monkeypatch.setattr(E, 'CROP_DECODE', 'flat')
    rng = np.random.default_rng(3)
    n, h, w = 37, 90, 70
    m = np.zeros((n, h, w), bool)
    for k in range(n):
        y, x, r = rng.integers(5, h - 5), rng.integers(5, w - 5), rng.integers(2, 14)
        yy, xx = np.ogrid[:h, :w]
        m[k] = (yy - y) ** 2 + (xx - x) ** 2 <= r * r
    ref = _csr_table(mods, m, E.LAYOUT_CROP)
    arena = torch.empty(1 << 16, dtype=torch.int32, device='cuda')
    ref.measure_paint(arena).check()
    assert not ref.zeroed
    want_bits = arena[:4 * int(ref.cursor.item())].clone()
    for ints in (1, 3, 4, 5, 1027, 40000, 1 << 20):
        buf = torch.full((ints + 8,), 7, dtype=torch.int32, device='cuda')
        t = _csr_table(mods, m, E.LAYOUT_CROP)
        arena2 = torch.empty(1 << 16, dtype=torch.int32, device='cuda')
        t.measure_paint(arena2, zero=buf[4:4 + ints])            # 16-byte aligned start, any length
        t.check()
        assert t.zeroed
        assert bool((buf[4:4 + ints] == 0).all()) and bool((buf[:4] == 7).all()) and bool((buf[4 + ints:] == 7).all()), ints
        assert torch.equal(t.area[:n], ref.area[:n]) and torch.equal(t.bbox[:4 * n], ref.bbox[:4 * n])
        assert int(t.cursor.item()) == int(ref.cursor.item())
        # same windows (the arena order may differ between launches: compare through the offsets)
        for k in range(n):
            a0, b0 = int(ref.bits_off[k].item()) * 4, int(t.bits_off[k].item()) * 4
            nw = int(ref.reg[2 * k + 1].item()) * 4
            assert torch.equal(want_bits[a0:a0 + nw], arena2[b0:b0 + nw]), (ints, k)
    # an unaligned buffer is declined: the caller clears it
    t = _csr_table(mods, m, E.LAYOUT_CROP)
    buf = torch.full((64,), 7, dtype=torch.int32, device='cuda')
    t.measure_paint(torch.empty(1 << 16, dtype=torch.int32, device='cuda'), zero=buf[1:33])
    assert not t.zeroed and bool((buf == 7).all())


@pytest.mark.parametrize('h,w', [(8200, 24), (16500, 12), (40, 3000), (65536, 6), (70000, 6)])
def test_crop_decode_of_tall_wide_and_busy_masks(mods, h, w, monkeypatch):
    """Frames taller than the shared-memory tile of the crop painter (a box of more than 128 / 256 / 512 32-row
    bands used to overflow the tile: ADVICE r1; the flat decode keeps rows in 16 bits and hands frames of more than
    65,536 rows to its fallback kernel), masks with thousands of runs, full frames and empty masks next to
    small blobs: every fused crop decode (flat with its fallback list, 8 / 16 / 32 lanes per mask) and the unfused
    painter give the measurements and the all-pairs intersections of a dense numpy formulation."""
    B, E, torch = mods.batch, mods.engine, mods.torch
    rng = np.random.default_rng(h * 7 + w)
    n = 14
    m = np.zeros((n, h, w), bool)
    m[0, :, 2:4] = True                                   # full-height thin mask
    m[1, 1:h - 1, w // 2] = True                          # almost full height, one column
    m[2, ::2, : min(w, 40)] = True                        # thousands of short runs
    m[3] = True                                           # the whole frame
    m[5, h // 2: h // 2 + 9, 1:8] = True                  # small blobs around the tall ones
    m[6, 0:5, 0:3] = True
    m[7, h - 4:, w - 3:] = True
    m[8] = rng.random((h, w)) < 0.3                       # noise: runs everywhere
    m[9, 5: h - 5: 3, 1] = True
    m[10, h // 3: h // 3 + 40, : w // 2] = True
    m[11, :, w - 1] = True
    m[12, 100: h - 100, 0: w: 5] = True
    t_ref = _csr_table(mods, m, E.LAYOUT_CROP).measure().paint().check()
    groups = E.Groups(t_ref.device, np.arange(n), np.zeros(n, np.int64), [0], [n], [0], [n], dense=True)
    ref = E.intersect_rows(t_ref, groups, E.MODE_IOU, grid='scan')
    flat = m.reshape(n, -1).astype(np.int64)
    want_I = flat @ flat.T
    assert np.array_equal(ref.imat.cpu().numpy()[:n * n].reshape(n, n), want_I)
    assert np.array_equal(t_ref.areas_np(), m.sum(axis=(1, 2)))
    need = int(t_ref.bits_off[n].item())
    for decode, hint in [('flat', 0), ('flat', 30), ('flat', 5000), ('group', 0), ('group', 30), ('group', 100)]:
        monkeypatch.setattr(E, 'CROP_DECODE', decode)
        monkeypatch.setattr(E, 'PAINT_RUNS_HINT', hint)
        t = _csr_table(mods, m, E.LAYOUT_CROP)
        arena = torch.empty(4 * need, dtype=torch.int32, device='cuda')
        t.measure_paint(arena).check()
        got = E.intersect_rows(t, groups, E.MODE_IOU, grid='scan')
        tag = (decode, hint)
        assert torch.equal(t.area[:n], t_ref.area[:n]) and torch.equal(t.bbox[:4 * n], t_ref.bbox[:4 * n]), tag
        assert int(t.cursor.item()) == need, tag
        assert np.array_equal(got.imat.cpu().numpy()[:n * n].reshape(n, n), want_I), tag
        # arena exhausted: no kernel may touch memory beyond it, the masks that did not fit are left empty
        small = torch.empty(4 * max(need // 3, 1), dtype=torch.int32, device='cuda')
        t2 = _csr_table(mods, m, E.LAYOUT_CROP)
        t2.measure_paint(small)
        with pytest.raises(mods.engine.N.AmpisNativeError, match='arena too small'):
            t2.check()
        E.intersect_rows(t2, groups, E.MODE_IOU, grid='scan')
        torch.cuda.synchronize()


def test_one_call_image_entry_equals_table_api(mods, monkeypatch):
    """engine.eval_image (ampis_eval_image_host: one library call per image) == the table API kernel by kernel:
    both modes, the scanned and the grid-pruned rows kernel, workspace growth on a large image, malformed RLE."""
    A, B, E, P, rle = mods.analyze, mods.batch, mods.engine, mods.powder, mods.rle
    cases = [('c1_powder_example', {}, E.MODE_IOU),                                              # scan (300 columns)
             ('c2_powder_batch', {}, E.MODE_IOU),                                                # grid (500 columns)
             ('c3_satellites', dict(h=1024, w=1024, n_cols=700), E.MODE_SAT),                    # satellites, grid
             ('c4_spheroidite', dict(n_rows=3000, n_cols=3500), E.MODE_IOU),                     # grows the workspaces
             ('c2_powder_batch', dict(h=640, w=480, n_rows=20, n_cols=25, median_diam=200.0), E.MODE_IOU)]
    for cfg, over, mode in cases:
        host = B.synth(dict(B.CONFIGS[cfg], **over), 1, 2024)
        rows, cols = host.image_masks(0)
        mk = lambda cs: [{'size': [host.h, host.w], 'counts': rle.string_from_counts(c)} for c in cs]
        r_, c_ = mk(rows), mk(cols)
        got = E.eval_image(r_, c_, mode)
        table, groups, res = A._rows_vs_cols(r_, c_, mode)
        G = len(r_)
        assert np.array_equal(got.best_col, res.best_col[:G].cpu().numpy()), cfg
        assert np.array_equal(got.best_inter, res.best_inter[:G].cpu().numpy().view(np.uint32)), cfg
        assert np.array_equal(got.best_score, res.best_score[:G].cpu().numpy(), equal_nan=True), cfg
        assert np.array_equal(got.area, table.areas_np()) and np.array_equal(got.bbox, table.bbox_np()), cfg
        assert abs(got.fill() - E.operand_fill(table)) < 1e-12
    bad = [{'size': [45, 37], 'counts': rle.string_from_counts(np.array([3, 5000, 7, 900], np.uint32))}]
    with pytest.raises(ValueError, match='malformed RLE'):
        E.eval_image(bad, bad, E.MODE_IOU)
    # the satellite function end to end, both ways
    host = B.synth(dict(B.CONFIGS['c3_satellites'], h=1024, w=1024, n_cols=500), 1, 7)
    sat, part = host.image_masks(0)
    mk = lambda cs: [{'size': [host.h, host.w], 'counts': rle.string_from_counts(c)} for c in cs]
    a = P._rle_satellite_match(mk(part), mk(sat), 0.5)
    monkeypatch.setattr(A, 'FUSED_CALL', False)
    b = P._rle_satellite_match(mk(part), mk(sat), 0.5)
    assert all(np.array_equal(a[k], b[k]) for k in ('satellite_matches', 'satellites_unmatched', 'particles_unmatched',
                                                    'intersection_scores')) and a['match_pairs'].keys() == b['match_pairs'].keys()


def test_integration_stub_from_the_docs_runs(mods):
    """The ctypes stub printed in INTEGRATION.md (what a maintainer would paste into ampis/analyze.py) is executed
    as it stands against the built library and gives the matcher's result on a golden image."""
    import re
    from ampis_b200 import build as bld
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    md = open(os.path.join(root, 'INTEGRATION.md')).read()
    blocks = re.findall(r"```python\n(.*?)```", md, re.S)
    code = [b for b in blocks if 'ampis_eval_image_host' in b]
    assert len(code) == 1
    src = code[0].replace("ctypes.CDLL('libampis_b200.so')", "ctypes.CDLL(%r)" % bld.LIB)
    ns = {}
    exec(compile(src, 'INTEGRATION.md', 'exec'), ns)
    _, gt, pr = U.powder_match_image(1)
    got = ns['_piecewise_rle_match'](list(gt), list(pr), 0.5)
    want = mods.analyze._piecewise_rle_match(gt, pr, 0.5)
    for k in ('tp', 'fn', 'fp', 'iou'):
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), k


def test_c_caller_of_the_abi(mods, tmp_path):
    """A plain C program (tests/c_abi/eval_image_main.c: cudaMalloc / cudaHostAlloc, no Python, no PyTorch) links
    libampis_b200.so, evaluates one golden image through ampis_eval_image_host -- growing its workspaces when told
    AMPIS_ENOSPC -- and prints what the oracle computes."""
    import subprocess
    from ampis_b200 import build as bld
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / 'eval_image_main')
    cc = subprocess.run(['gcc', '-O2', '-o', exe, os.path.join(root, 'tests', 'c_abi', 'eval_image_main.c'),
                         '-I', os.path.join(root, 'include'), '-I', '/usr/local/cuda/include',
                         '-L', os.path.dirname(bld.LIB), '-lampis_b200', '-L', '/usr/local/cuda/lib64', '-lcudart',
                         '-Wl,-rpath,' + os.path.dirname(bld.LIB) + ',-rpath,/usr/local/cuda/lib64'],
                        capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr
    _, gt, pr = U.powder_match_image(2)
    masks = list(gt) + list(pr)
    off = np.zeros(len(masks) + 1, np.int64)
    np.cumsum([len(m['counts']) for m in masks], out=off[1:])
    h, w = masks[0]['size']
    path = tmp_path / 'image.bin'
    with open(path, 'wb') as f:
        f.write(np.array([len(gt), len(pr), h, w, 0], np.int32).tobytes())
        f.write(off.tobytes())
        f.write(b''.join(m['counts'] for m in masks))
    run = subprocess.run([exe, str(path)], capture_output=True, text=True, timeout=120)
    assert run.returncode == 0, run.stderr
    rows = [l.split() for l in run.stdout.splitlines() if l.startswith('row')]
    ms = [l.split() for l in run.stdout.splitlines() if l.startswith('mask')]
    assert len(rows) == len(gt) and len(ms) == len(masks)
    want = {}
    mods.analyze._piecewise_rle_match(gt, pr, 0.5, _details=want)
    assert [int(r[2]) for r in rows] == want['best_col'].tolist()
    assert [int(r[3]) for r in rows] == want['best_inter'].tolist()
    assert [float(r[4]) for r in rows] == want['best_iou'].tolist()
    assert [int(m_[2]) for m_ in ms] == mods.rle.area(masks).tolist() and all(int(m_[7]) == 0 for m_ in ms)
    # ---- the many-image entry from C: three golden images of different instance counts in ONE call, strings passed
    # as one contiguous blob and as one descriptor per string; per-row results, areas and TP/FP/FN at two thresholds
    exe2 = str(tmp_path / 'eval_images_main')
    cc = subprocess.run(['gcc', '-O2', '-o', exe2, os.path.join(root, 'tests', 'c_abi', 'eval_images_main.c'),
                         '-I', os.path.join(root, 'include'), '-I', '/usr/local/cuda/include',
                         '-L', os.path.dirname(bld.LIB), '-lampis_b200', '-L', '/usr/local/cuda/lib64', '-lcudart',
                         '-Wl,-rpath,' + os.path.dirname(bld.LIB) + ',-rpath,/usr/local/cuda/lib64'],
                        capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr
    imgs = [U.powder_match_image(k)[1:] for k in (0, 2, 4)]
    allm = [m for g_, p_ in imgs for m in list(g_) + list(p_)]
    path2 = tmp_path / 'images.bin'
    with open(path2, 'wb') as f:
        f.write(np.array([len(imgs)], np.int32).tobytes())
        f.write(np.array([len(g_) for g_, _ in imgs], np.int32).tobytes())
        f.write(np.array([len(p_) for _, p_ in imgs], np.int32).tobytes())
        f.write(np.array([g_[0]['size'][0] for g_, _ in imgs], np.int32).tobytes())
        f.write(np.array([g_[0]['size'][1] for g_, _ in imgs], np.int32).tobytes())
        f.write(np.array([len(m['counts']) for m in allm], np.int32).tobytes())
        f.write(b''.join(m['counts'] for m in allm))
    for extra in ([], ['scattered']):
        run = subprocess.run([exe2, str(path2)] + extra, capture_output=True, text=True, timeout=120)
        assert run.returncode == 0, run.stderr
        rows = [l.split() for l in run.stdout.splitlines() if l.startswith('row')]
        cnt = [[int(v) for v in l.split()[2:]] for l in run.stdout.splitlines() if l.startswith('counts')]
        tot = [l.split() for l in run.stdout.splitlines() if l.startswith('totals')][0]
        r0, want_tot = 0, np.zeros(6, np.int64)
        for (g_, p_), c_ in zip(imgs, cnt):
            want = {}
            mods.analyze._piecewise_rle_match(g_, p_, 0.5, _details=want)
            assert [int(r[2]) for r in rows[r0:r0 + len(g_)]] == want['best_col'].tolist()
            assert [float(r[4]) for r in rows[r0:r0 + len(g_)]] == want['best_iou'].tolist()
            r0 += len(g_)
            ref = []
            for th in (0.5, 0.75):
                m_ = mods.R.piecewise_rle_match(g_, p_, th)
                ref += [len(m_['tp']), len(m_['fp']), len(m_['fn'])]
            assert c_ == ref
            want_tot += np.array(ref)
        assert [int(v) for v in tot[1:7]] == want_tot.tolist() and tot[-1] == '0'
        assert [int(l.split()[2]) for l in run.stdout.splitlines() if l.startswith('mask')] == mods.rle.area(allm).tolist()


def test_full_size_properties(mods):
    """BASELINE config sizes (C2 image count reduced): size-independent properties --
    span and full layouts agree bit for bit, I(gt,pred) == I(pred,gt)^T, area == popcount of the
    unpacked mask, counts add up, self-match gives IoU 1 for every non-empty mask."""
    B, E, torch = mods.batch, mods.engine, mods.torch
    host = B.synth('c2_powder_batch', 6, 2002)
    dev = B.DeviceBatch(host, dense=True)
    a = B.eval_step(dev, layout=E.LAYOUT_SPAN, check=True)
    b = B.eval_step(dev, layout=E.LAYOUT_FULL, check=True)
    arena = torch.empty(4 * B.arena_chunks_needed(dev, E.LAYOUT_SPAN), dtype=torch.int32, device='cuda')
    f = B.eval_step(dev, layout=E.LAYOUT_SPAN, check=True, arena=arena)          # fused measure+paint
    for x, y in [(a.rows.best_col, f.rows.best_col), (a.rows.best_score, f.rows.best_score),
                 (a.rows.imat, f.rows.imat), (a.counts, f.counts), (a.table.area, f.table.area),
                 (a.table.bbox, f.table.bbox), (a.table.span, f.table.span)]:
        assert torch.equal(x, y)
    small = torch.empty(4 * 1000, dtype=torch.int32, device='cuda')             # arena overflow is detected
    with pytest.raises(Exception, match='arena too small'):
        B.eval_step(dev, layout=E.LAYOUT_SPAN, check=True, arena=small)
    for x, y in [(a.rows.best_col, b.rows.best_col), (a.rows.best_inter, b.rows.best_inter),
                 (a.rows.best_score, b.rows.best_score), (a.rows.imat, b.rows.imat), (a.counts, b.counts),
                 (a.table.area, b.table.area), (a.table.bbox, b.table.bbox)]:
        assert torch.equal(x, y)
    G, P, n = host.n_rows, host.n_cols, host.n_images
    c = a.counts.cpu().numpy()
    assert (c[:, :, 0] + c[:, :, 2] == G).all() and (c[:, :, 1] <= P).all() and (c[:, :, 0] >= 0).all()
    assert (np.diff(c[:, :, 0], axis=1) <= 0).all()          # TP is monotone in the threshold
    # transpose property: swap the roles of rows and columns
    per = G + P
    idx = np.arange(n * per).reshape(n, per)
    idx = np.concatenate([idx[:, G:], idx[:, :G]], 1).ravel()
    host_t = B.HostCSR(dict(host.cfg, n_rows=P, n_cols=G), n, host.cnt, host.cnt_off[idx], host.cnt_len[idx])
    t = B.eval_step(B.DeviceBatch(host_t, dense=True), check=True)
    assert torch.equal(t.rows.imat.view(n, P, G).transpose(1, 2).contiguous(), a.rows.imat.view(n, G, P))
    # area == popcount of unpacked bits (first image, rows)
    ub = E.unpack_bool(b.table, np.arange(0, 64), host.h, host.w)
    assert torch.equal(ub.sum(dim=(1, 2)).int(), b.table.area[:64])
    # self match: rows vs rows
    idx2 = np.arange(n * per).reshape(n, per)[:, :G]
    idx2 = np.concatenate([idx2, idx2], 1).ravel()
    host_s = B.HostCSR(dict(host.cfg, n_cols=G), n, host.cnt, host.cnt_off[idx2], host.cnt_len[idx2])
    s = B.eval_step(B.DeviceBatch(host_s), check=True)
    area = s.table.area.view(n, 2 * G)[:, :G].reshape(-1)
    sc = s.rows.best_score
    assert bool(((sc == 1.0) | (area == 0)).all())


@pytest.mark.parametrize('cfg,over,n_img', [
    ('c2_powder_batch', dict(h=256, w=256, n_rows=150, n_cols=300, median_diam=14.0), 3),   # ragged single tiles
    ('dense_overlap', dict(n_rows=300, n_cols=520), 2),                                     # 3 x 3 tiles, ragged
    ('c3_satellites', dict(h=512, w=512, n_rows=40, n_cols=300), 2),                         # satellite scores
])
@pytest.mark.parametrize('layout', ['span', 'full'])
def test_tensor_core_contraction_equals_culled_popc(mods, cfg, over, n_img, layout):
    """ampis_intersect_tcgen05 (dense int8 contraction, no pruning) == ampis_intersect_rows (bbox-culled
    AND+popc): dense intersections, arg-max, scores and counts bit for bit; first image also against
    the oracle's run-walk intersections."""
    B, E, R, rle, torch = mods.batch, mods.engine, mods.R, mods.rle, mods.torch
    c = dict(B.CONFIGS[cfg], **over)
    host = B.synth(c, n_img, 4242)
    dev = B.DeviceBatch(host, dense=True)
    lay = E.LAYOUT_FULL if layout == 'full' else E.LAYOUT_SPAN
    t = E.MaskTable(dev.device, host.n_masks, dev.cnt, dev.cnt_off, dev.cnt_len, dev.h, dev.w, lay)
    t.measure().paint().check()
    a = E.intersect_rows(t, dev.groups, dev.mode)
    m = E.intersect_mma(t, dev.groups, dev.mode, pair=False)
    torch.cuda.synchronize()
    assert torch.equal(a.imat, m.imat)
    for sort in (True, False):                       # CTA pairs (cta_group::2, 256 x 256 tiles): the same matrix
        m2 = E.intersect_mma(t, dev.groups, dev.mode, pair=True, sort=sort)
        torch.cuda.synchronize()
        assert torch.equal(a.imat, m2.imat), 'pair kernel, sort=%s' % sort
        assert torch.equal(a.best_col, m2.best_col) and torch.equal(a.best_inter, m2.best_inter)
    assert torch.equal(a.best_col, m.best_col) and torch.equal(a.best_inter, m.best_inter)
    sa, sm = a.best_score.cpu().numpy(), m.best_score.cpu().numpy()
    assert np.array_equal(sa, sm, equal_nan=True)
    if layout == 'full':                             # TMA-staged shared-memory tiled AND+popc (64 x 64 tiles, tensor map)
        tm = E.intersect_tma(t, dev.groups, dev.mode)
        torch.cuda.synchronize()
        assert torch.equal(a.imat, tm.imat), 'TMA tiled kernel'
        assert torch.equal(a.best_col, tm.best_col) and torch.equal(a.best_inter, tm.best_inter)
        assert np.array_equal(sa, tm.best_score.cpu().numpy(), equal_nan=True)
    rows, cols = host.image_masks(0)
    er, ec = _counts_to_rle(rle, rows, host.h, host.w), _counts_to_rle(rle, cols, host.h, host.w)
    imat = m.imat.cpu().numpy()[:host.n_rows * host.n_cols].reshape(host.n_rows, host.n_cols)
    rng = np.random.default_rng(5)
    for i, j in zip(rng.integers(0, host.n_rows, 300), rng.integers(0, host.n_cols, 300)):
        assert imat[i, j] == int(rle.merge_area(er[i], ec[j]))
    assert imat.max() > 0


def test_hist_and_scan(mods):
    E, torch = mods.engine, mods.torch
    rng = np.random.default_rng(0)
    v = rng.integers(0, 50000, 100003).astype(np.uint32)
    d = torch.from_numpy(v.view(np.int32)).cuda()
    hist = E.hist_u32(d, 100, 37, 512).cpu().numpy()
    b = np.clip((v.astype(np.int64) - 100) // 37, 0, 511)
    assert np.array_equal(hist, np.bincount(b, minlength=512))
    from ampis_b200 import _native as N
    for n in (1, 5, 2048, 2049, 300001):
        x = torch.from_numpy(rng.integers(0, 1 << 33, n)).cuda()
        out = torch.empty(n + 1, dtype=torch.int64, device='cuda')
        nb = N.lib().ampis_scan_tmp_bytes(n)
        tmp = torch.empty(nb // 8 + 1, dtype=torch.int64, device='cuda')
        N.call('ampis_exclusive_scan_i64', E._p(x), E._p(out), n, E._p(tmp), nb, E._stream())
        want = np.concatenate([[0], np.cumsum(x.cpu().numpy())])
        assert np.array_equal(out.cpu().numpy(), want)


def test_encode_on_gpu_equals_pycocotools_strings(mods):
    """engine.encode_bool (pack + rleEncode + rleToString on the GPU) reproduces, byte for byte, the
    strings the real pycocotools.encode wrote into the shipped prediction pickles (decode -> encode
    round trip), and the oracle's encode on random masks incl. first-pixel-set and all-ones."""
    E, S, rle = mods.engine, mods.structures, mods.rle
    _, gt, pr = U.powder_match_image(0)
    sample = pr[:60]
    dense = S.masks_to_bitmask_array(sample)
    got = E.encode_bool(dense)
    assert [g['counts'] for g in got] == [m['counts'] for m in sample]
    assert got[0]['size'] == list(sample[0]['size'])
    rng = np.random.default_rng(11)
    for h, w in [(1, 1), (7, 5), (64, 2), (33, 129), (128, 128)]:
        a = U.rand_masks(rng, 9, h, w)
        a[0] = True
        a[1] = False
        a[2, 0, 0] = True
        a[3, -1, -1] = True
        want = rle.encode(np.asfortranarray(a.transpose(1, 2, 0).astype(np.uint8)))
        got = E.encode_bool(a)
        assert [g['counts'] for g in got] == [m['counts'] for m in want], (h, w)


def test_mask_edge_distance_vs_oracle(mods):
    """analyze.mask_edge_distance == reference algorithm (decode, crop, n x m distances), bit for bit,
    on matched pairs of a shipped image and on random blobs with loose / clipped boxes."""
    A, R, D, S, rle = mods.analyze, mods.R, mods.data_utils, mods.structures, mods.rle
    _, gt, pr = U.powder_match_image(1)
    m = A.rle_instance_matcher(gt, pr, 0.5)
    matches = m['tp'][:40]
    gb = D.extract_boxes(S.masks_to_bitmask_array(gt), box_mode='matterport')
    pb = D.extract_boxes(S.masks_to_bitmask_array(pr), box_mode='matterport')
    fp, fn = A.mask_edge_distance(gt, pr, gb, pb, matches)
    wfp, wfn = R.mask_edge_distance(gt, pr, gb, pb, matches)
    assert len(fp) == len(matches)
    for a, b in zip(fp + fn, wfp + wfn):
        assert a.dtype == mods.torch.float64 and np.array_equal(a.numpy(), b)
    assert sum(len(x) for x in fp) > 100 and sum(len(x) for x in fn) > 100
    # RLEMasks input, CUDA output, loose boxes that stick out of the frame
    rng = np.random.default_rng(3)
    h, w = 61, 47
    g = U.rand_masks(rng, 6, h, w, p_empty=0)
    p = g.copy()
    p[:, 1:] |= g[:, :-1]
    p[:, :, :3] = False
    ge = rle.encode(np.asfortranarray(g.transpose(1, 2, 0).astype(np.uint8)))
    pe = rle.encode(np.asfortranarray(p.transpose(1, 2, 0).astype(np.uint8)))
    boxes = np.tile(np.array([0, h + 5, 0, w + 9]), (6, 1))
    mt = np.stack([np.arange(6), np.arange(6)[::-1]], 1)
    fp, fn = A.mask_edge_distance(S.RLEMasks(ge), S.RLEMasks(pe), boxes, boxes, mt, device='cuda')
    wfp, wfn = R.mask_edge_distance(ge, pe, boxes, boxes, mt)
    for a, b in zip(fp + fn, wfp + wfn):
        assert a.is_cuda and np.array_equal(a.cpu().numpy(), b)
    assert A.mask_edge_distance(ge, pe, boxes, boxes, np.zeros((0, 2), int)) == ([], [])
    # the reference's torch.min raises when the other mask has no pixel in the window
    tiny = np.tile(np.array([0, 2, 0, 2]), (6, 1))
    e = np.zeros((1, h, w), np.uint8)
    f = np.zeros((1, h, w), np.uint8)
    f[0, 0, 0] = 1
    ee = rle.encode(np.asfortranarray(e.transpose(1, 2, 0)))
    fe = rle.encode(np.asfortranarray(f.transpose(1, 2, 0)))
    with pytest.raises(RuntimeError):
        A.mask_edge_distance(ee, fe, tiny, tiny, np.array([[0, 0]]))
    a = mods.torch.tensor([[0, 0], [3, 4]])
    assert A._min_euclid(a, mods.torch.tensor([[0, 1], [3, 0]])).tolist() == [1.0, 4.0]


@pytest.mark.parametrize('mode', ['reduced', 'all'])
def test_seg_and_det_perf_isets_vs_oracle(mods, mode):
    A, R, S, rle = mods.analyze, mods.R, mods.structures, mods.rle
    from ampis_b200.containers import Instances
    _, gt, pr = U.powder_match_image(2)
    m = A.rle_instance_matcher(gt, pr, 0.5)
    iset, colors = A.seg_perf_iset(gt, pr, m, mode=mode)
    want = R.seg_perf_masks(gt, pr, m['tp'], mode)
    got = iset.instances.masks.rle
    assert [x['counts'] for x in got] == [x['counts'] for x in want]
    assert len(colors[0]) == len(got) == (4 if mode == 'reduced' else 7)
    assert len(colors[1]) == (4 if mode == 'reduced' else 8)      # the reference lists 8 names for 7 masks
    assert iset.instances.boxes.shape == (len(got), 4)
    iset2, _ = A.seg_perf_iset(S.RLEMasks(gt), S.RLEMasks(pr), None, mode=mode)       # matcher called inside
    assert [x['counts'] for x in iset2.instances.masks.rle] == [x['counts'] for x in want]
    # det_perf_iset: bookkeeping over the matcher's output
    size = tuple(gt[0]['size'])
    mk = lambda ms: S.InstanceSet(instances=Instances(size, masks=S.RLEMasks(ms),
                                                      boxes=np.arange(4 * len(ms), dtype=float).reshape(-1, 4)))
    G, P = mk(gt), mk(pr)
    d, cmap = A.det_perf_iset(G, P)
    n_tp, n_fp, n_fn = len(m['tp']), len(m['fp']), len(m['fn'])
    assert len(d.instances) == n_tp + n_fp + n_fn and set(cmap) == {'TP', 'FP', 'FN'}
    assert [x['counts'] for x in d.instances.masks.rle[:n_tp]] == [pr[i]['counts'] for i in m['tp'][:, 1]]
    assert np.array_equal(d.instances.boxes[n_tp:n_tp + n_fp], P.instances.boxes[m['fp']])
    assert np.array_equal(d.instances.colors[-1], cmap['FN'])
    d2 = A.det_perf_iset(G, P, m, colormap=cmap, tp_gt=True)
    assert [x['counts'] for x in d2.instances.masks.rle[:n_tp]] == [gt[i]['counts'] for i in m['tp'][:, 0]]


def _write_png(path, arr):
    from PIL import Image
    Image.fromarray(arr).save(str(path))


def test_get_ddicts_binary_and_label_images(mods, tmp_path, monkeypatch):
    """data_utils.get_ddicts('binary' / 'label'): connected components, boxes and RLE of the
    reference's own annotation images == oracle (committed fixture), plus random label images
    with gaps in the label values, touching components and frame-filling instances."""
    D, R, E = mods.data_utils, mods.R, mods.engine
    g = U.load('spheroidite_annotations.npz')
    monkeypatch.chdir(tmp_path)
    (tmp_path / 'im').mkdir()
    (tmp_path / 'ann').mkdir()
    for k, name in enumerate(g['names']):
        shape = tuple(int(v) for v in g['%d_shape' % k])
        a = np.unpackbits(g['%d_bits' % k])[:shape[0] * shape[1]].reshape(shape).astype(np.uint8) * 255
        _write_png(tmp_path / 'im' / str(name), a)
        _write_png(tmp_path / 'ann' / str(name), a)
    dd = D.get_ddicts('binary', 'im', 'ann', dataset_class='Training')
    assert len(dd) == 2
    by_name = {os.path.basename(d['file_name']): d for d in dd}
    for k, name in enumerate(g['names']):
        d = by_name[str(name)]
        shape = tuple(int(v) for v in g['%d_shape' % k])
        want = U.unpack_strings(g['%d_blob' % k], g['%d_off' % k], shape)
        assert (d['height'], d['width']) == shape and d['mask_format'] == 'bitmask'
        assert d['num_instances'] == len(want) == len(d['annotations']) and d['dataset_class'] == 'Training'
        assert [x['segmentation']['counts'] for x in d['annotations']] == [m['counts'] for m in want]
        assert np.array_equal(np.stack([x['bbox'] for x in d['annotations']]), g['%d_boxes' % k])
        assert d['annotations'][0]['bbox'].dtype == np.float64 and d['annotations'][0]['category_id'] == 0
    # label images (.npy) with arbitrary values; engine level against the oracle
    rng = np.random.default_rng(8)
    for h, w in [(5, 7), (64, 33), (97, 130)]:
        lab = rng.choice(np.array([0, 0, 0, 3, 4, 9, 500, 70000]), size=(h, w))
        lab[:, 0] = 9                      # a column-filling instance whose runs cross column ends
        for binary in (False, True):
            rles, bb = E.label_image_to_instances(lab, binary=binary)
            want = R.annotations_from_label_image(lab, binary=binary)
            assert len(rles) == len(want)
            assert [m['counts'] for m in rles] == [m['counts'] for _, m in want]
            assert np.array_equal(bb.astype(np.float64), np.stack([b for b, _ in want]))
    full = np.ones((33, 65), np.int64)
    rles, bb = E.label_image_to_instances(full, binary=True)
    assert len(rles) == 1 and bb.tolist() == [[0, 0, 64, 32]]
    assert rles[0]['counts'] == mods.rle.encode(np.asfortranarray(full.astype(np.uint8)))['counts']
    assert E.label_image_to_instances(np.zeros((4, 4), np.uint8), binary=True)[0] == []
    np.save(str(tmp_path / 'ann2.npy'), lab)
    with pytest.raises(ValueError):
        E.label_image_to_instances(-lab, binary=False)


def test_get_ddicts_rle_json_and_compress_pred(mods, tmp_path, monkeypatch):
    import json
    D, R, S, rle = mods.data_utils, mods.R, mods.structures, mods.rle
    _, gt, pr = U.powder_match_image(0)
    sample = pr[:25]
    monkeypatch.chdir(tmp_path)
    data = [{'file_name': 'images/a.png',
             'segmentations': [{'size': list(m['size']), 'counts': m['counts'].decode('utf-8')} for m in sample]}]
    json.dump(data, open('ann.json', 'w'))
    dd = D.get_ddicts('rle', 'ann.json')
    assert len(dd) == 1 and dd[0]['num_instances'] == 25 and dd[0]['file_name'] == 'images/a.png'
    dense = S.masks_to_bitmask_array(sample)
    assert np.array_equal(np.stack([a['bbox'] for a in dd[0]['annotations']]), R.extract_boxes(dense))
    assert [a['segmentation']['counts'] for a in dd[0]['annotations']] == [m['counts'] for m in sample]

    class Pred(object):
        pass
    p = Pred()
    p.pred_masks = mods.torch.from_numpy(dense).cuda()
    p.pred_boxes = mods.torch.arange(100, dtype=mods.torch.float32).reshape(25, 4)
    p.scores = mods.torch.linspace(0, 1, 25)
    p.pred_classes = mods.torch.zeros(25, dtype=mods.torch.int64)
    out = D.format_outputs('a.png', 'Validation', {'instances': p})
    assert out['dataset'] == 'Validation' and out['pred']['instances'] is p
    assert [m['counts'] for m in p.pred_masks] == [m['counts'] for m in sample]
    assert isinstance(p.scores, np.ndarray) and p.pred_boxes.shape == (25, 4) and p.pred_classes.dtype == np.int64


RPROP_KEYS = ['area', 'bbox', 'bbox_area', 'centroid', 'local_centroid', 'convex_area', 'eccentricity',
              'equivalent_diameter', 'extent', 'label', 'major_axis_length', 'minor_axis_length', 'orientation',
              'perimeter', 'solidity']


def _check_rprops(got, want):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert set(g) == set(w), i
        for k in w:
            if k in ('area', 'bbox', 'bbox_area', 'convex_area', 'label'):
                assert g[k] == w[k], (i, k, g[k], w[k])             # integers: exact
            elif k == 'orientation':
                # an axis direction: +pi/2 and -pi/2 are the same line, and which one the float pipeline of
                # skimage lands on for an exactly axis-aligned shape depends on the sign of a ~1e-17 residue
                d = (g[k] - w[k] + np.pi / 2) % np.pi - np.pi / 2
                assert abs(d) < 1e-6, (i, k, g[k], w[k])
            else:                                                   # derived floats: 1e-6 (north_star)
                assert np.allclose(g[k], w[k], rtol=1e-6, atol=1e-6), (i, k, g[k], w[k])


def test_region_properties_vs_skimage_restatement(mods):
    """compute_rprops keys from exact GPU measurements == oracle restatement of skimage 0.18.3
    (moments, inertia eigenvalues, orientation, 4-neighbourhood perimeter, convex hull image) on
    shipped spheroidite predictions, powder predictions and random / degenerate masks."""
    S, R, rle = mods.structures, mods.R, mods.rle
    from ampis_b200.containers import Instances
    m = U.load('spheroidite_measure.npz')
    masks = U.unpack_strings(m['1_blob'], m['1_off'], m['1_size'])[:60]
    _, gt, pr = U.powder_match_image(3)
    for ms in (masks, pr[:25]):
        dense = rle.decode(ms).transpose(2, 0, 1).astype(bool)
        _check_rprops(S.region_properties(ms), [R.regionprops_one(d) for d in dense])
    rng = np.random.default_rng(21)
    for h, w in [(1, 1), (3, 40), (40, 3), (37, 53), (70, 70)]:
        a = U.rand_masks(rng, 12, h, w)
        a[0] = True                                  # whole frame
        a[1] = False
        a[1, h // 2, w // 2] = True                  # single pixel
        a[2] = np.eye(h, w, dtype=bool)              # diagonal line
        a[3] = False
        a[3, 0, :] = True                            # one-pixel-wide line along the frame edge
        a[3, -1, -1] = True                          # + a detached pixel (one region, two components)
        enc = rle.encode(np.asfortranarray(a.transpose(1, 2, 0).astype(np.uint8)))
        _check_rprops(S.region_properties(enc), [R.regionprops_one(d) for d in a])
    # through InstanceSet.compute_rprops: reference default keys, 1-element cells, tuple keys split
    n = len(masks)
    size = tuple(int(v) for v in m['1_size'])
    iset = S.InstanceSet(instances=Instances(size, masks=S.RLEMasks(masks), boxes=np.zeros((n, 4)),
                                             class_idx=np.arange(n)))
    iset.compute_rprops()
    assert list(iset.rprops.columns) == ['area', 'equivalent_diameter', 'major_axis_length', 'perimeter', 'solidity',
                                         'orientation', 'class_idx']
    dense = rle.decode(masks).transpose(2, 0, 1).astype(bool)
    want = [R.regionprops_one(d) for d in dense]
    for i in range(n):
        for k in ('major_axis_length', 'perimeter', 'solidity', 'orientation'):
            cell = iset.rprops[k][i]
            if want[i]:
                assert cell.shape == (1,) and np.allclose(cell[0], want[i][k], rtol=1e-6, atol=1e-6)
            else:
                assert cell.shape == (0,)
    df = iset.compute_rprops(keys=['centroid', 'bbox'], return_df=True)
    assert list(df.columns) == ['centroid-0', 'centroid-1', 'bbox-0', 'bbox-1', 'bbox-2', 'bbox-3', 'class_idx']
    with pytest.raises(NotImplementedError):
        iset.compute_rprops(keys=['euler_number'])


def test_polygon_bitmasks_follow_skimage_rule(mods):
    """masks_to_bitmask_array(PolygonMasks / list of polygons) == polygon2mask restatement, bit for bit
    (shipped VIA polygons and random polygons incl. ones sticking out of the frame); and it is NOT
    the pycocotools rasterisation masks_to_rle uses -- both behaviours are the reference's."""
    S, R = mods.structures, mods.R
    from ampis_b200.containers import PolygonMasks
    p = U.load('powder_polygons.npz')
    xy, off = p['0_poly_xy'], p['0_poly_off']
    size = tuple(int(v) for v in p['0_size'])
    polys = [xy[off[i]:off[i + 1]] for i in range(60)]
    got = S.masks_to_bitmask_array(PolygonMasks([[q] for q in polys]), size)
    want = R.poly2mask(polys, size)
    assert got.dtype == np.bool_ and got.shape == want.shape and np.array_equal(got, want)
    assert np.array_equal(S.masks_to_bitmask_array([list(q) for q in polys[:5]], size), want[:5])
    via_rle = S.masks_to_bitmask_array(S.masks_to_rle(PolygonMasks([[q] for q in polys]), size))
    assert (via_rle != want).any() and abs(int(via_rle.sum()) - int(want.sum())) < 0.02 * want.sum()
    rng = np.random.default_rng(17)
    h, w = 45, 60
    rnd = [np.round(rng.uniform(-10, 70, size=2 * rng.integers(3, 12)) * 2) / 2 for _ in range(40)]
    assert np.array_equal(S.masks_to_bitmask_array(rnd, (h, w)), R.poly2mask(rnd, (h, w)))
    with pytest.raises(AssertionError):
        S.masks_to_bitmask_array(PolygonMasks([[polys[0]]]))


def test_public_api_takes_the_tensor_core_path_on_crowded_images(mods, monkeypatch):
    """A crowded image (operand fill above engine.MMA_FILL_THRESHOLD) is evaluated by the tcgen05
    contraction from the drop-in API; results equal the oracle like on the culled path."""
    A, B, E, R, rle = mods.analyze, mods.batch, mods.engine, mods.R, mods.rle
    cfg = dict(B.CONFIGS['dense_overlap'], h=128, w=128, n_rows=70, n_cols=90, median_diam=70.0)
    host = B.synth(cfg, 1, 5)
    rows, cols = host.image_masks(0)
    gt, pr = _counts_to_rle(rle, rows, host.h, host.w), _counts_to_rle(rle, cols, host.h, host.w)
    used = []
    real = E.intersect
    monkeypatch.setattr(E, 'intersect', lambda t, g, m, out=None, kernel='auto': (used.append(kernel), real(t, g, m, out, kernel))[1])
    got = A.det_seg_scores(gt, pr, 0.5)
    assert used == ['mma']
    want = R.det_seg_scores(gt, pr, 0.5)
    for k in want:
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), k
    assert np.array_equal(A._piecewise_iou(gt, pr), R.piecewise_iou(gt, pr)) and used == ['mma', 'mma']
    _, g2, p2 = U.powder_match_image(0)
    calls = []
    real_eval = E.eval_images
    monkeypatch.setattr(E, 'eval_images', lambda *a, **k: (calls.append(1), real_eval(*a, **k))[1])
    n_before = len(used)
    one_call = A.rle_instance_matcher(g2, p2)                  # ordinary image: ONE library call, no table API
    assert calls == [1] and len(used) == n_before
    monkeypatch.setattr(A, 'FUSED_CALL', False)                # the table API gives the same answer
    by_table = A.rle_instance_matcher(g2, p2)
    assert used[-1] == 'rows' and all(np.array_equal(one_call[k], by_table[k]) for k in by_table)


def _host_csr_from_bool(B, masks_per_image, n_rows, h, w, rle):
    """list of bool[n_rows + n_cols, h, w] stacks -> batch.HostCSR (run counts via the oracle encoder)."""
    cnts = []
    for stack in masks_per_image:
        for m in stack:
            cnts.append(rle.counts_from_string(rle.encode(np.asfortranarray(m.astype(np.uint8)))['counts']))
    lens = np.array([len(c) for c in cnts], np.int32)
    off = np.zeros(len(cnts), np.int64)
    if len(cnts) > 1:
        off[1:] = np.cumsum(lens[:-1])
    n_cols = masks_per_image[0].shape[0] - n_rows
    cfg = dict(h=h, w=w, n_rows=n_rows, n_cols=n_cols, kind=0, mode=0)
    return B.HostCSR(cfg, len(masks_per_image), np.concatenate(cnts).astype(np.uint32), off, lens)


@pytest.mark.parametrize('seed', range(int(os.environ.get('AMPIS_FUZZ_SEEDS', '4'))))      # soak: AMPIS_FUZZ_SEEDS=200
def test_randomised_batches_all_layouts_and_kernels_vs_dense_numpy(mods, seed):
    """Randomised sweep over frame shapes (1x1 .. odd sizes, not multiples of 32 or 128), mask kinds
    (blobs, full frames, empty, single pixels, stripes that wrap column ends, noise) and group shapes:
    every layout (span / full / crop, fused and unfused construction) and both intersection kernels
    against a dense numpy formulation (bool AND + sum), independent of the run-walk oracle."""
    B, E, rle, torch = mods.batch, mods.engine, mods.rle, mods.torch
    rng = np.random.default_rng(1000 + seed)
    for trial in range(6):
        h, w = int(rng.integers(1, 150)), int(rng.integers(1, 150))
        G, Pn, n_img = int(rng.integers(1, 40)), int(rng.integers(1, 70)), int(rng.integers(1, 4))
        stacks = []
        for _ in range(n_img):
            m = U.rand_masks(rng, G + Pn, h, w, p_empty=0.15)
            kind = rng.integers(0, 6, G + Pn)
            for i, k in enumerate(kind):
                if k == 0:
                    m[i] = True
                elif k == 1:
                    m[i] = False
                    m[i, rng.integers(0, h), rng.integers(0, w)] = True
                elif k == 2:
                    m[i] = False
                    m[i, :, rng.integers(0, w):] = True           # full-height stripe: runs wrap column ends
                elif k == 3:
                    m[i] = rng.random((h, w)) < 0.5
            stacks.append(m)
        host = _host_csr_from_bool(B, stacks, G, h, w, rle)
        dev = B.DeviceBatch(host, dense=True)
        want_I = np.stack([(s[:G, None].astype(np.int64) * s[None, G:].astype(np.int64)).sum(axis=(2, 3)) for s in stacks])
        area = np.stack([s.sum(axis=(1, 2)) for s in stacks]).astype(np.int64)
        with np.errstate(invalid='ignore', divide='ignore'):
            iou = np.where(want_I > 0, want_I / (area[:, :G, None] + area[:, None, G:] - want_I), 0.0)
        want_best = np.where(iou.max(axis=2) > 0, iou.argmax(axis=2), -1)
        ref = None
        for layout in (E.LAYOUT_SPAN, E.LAYOUT_FULL, E.LAYOUT_CROP):
            for fused in (False, True):
                arena = None
                if fused:
                    arena = torch.empty(4 * max(B.arena_chunks_needed(dev, layout), 1), dtype=torch.int32, device='cuda')
                kernels = ('rows', 'grid') if layout == E.LAYOUT_CROP else ('rows', 'mma')
                for kernel in kernels:
                    # fused crop decode: the flat kernel (default) and the lane-group kernels of round 1 in turn
                    E.CROP_DECODE = 'group' if (fused and layout == E.LAYOUT_CROP and kernel == 'grid') else 'flat'
                    r = B.eval_step(dev, layout=layout, check=True, arena=arena, kernel=kernel)
                    E.CROP_DECODE = 'flat'
                    I = r.rows.imat.cpu().numpy()[:n_img * G * Pn].reshape(n_img, G, Pn)
                    tag = (trial, h, w, G, Pn, layout, fused, kernel)
                    assert np.array_equal(I, want_I), tag
                    assert np.array_equal(r.rows.best_col.cpu().numpy()[:n_img * G].reshape(n_img, G), want_best), tag
                    assert np.array_equal(r.rows.best_score.cpu().numpy()[:n_img * G].reshape(n_img, G), iou.max(axis=2)), tag
                    assert np.array_equal(r.table.area.cpu().numpy()[:n_img * (G + Pn)].reshape(n_img, -1), area), tag
                    if ref is None:
                        ref = r.counts.cpu().numpy()
                    else:
                        assert np.array_equal(r.counts.cpu().numpy(), ref), tag


@pytest.mark.parametrize('seed', range(int(os.environ.get('AMPIS_FUZZ_SEEDS', '3'))))
def test_randomised_measurement_kernels_vs_oracle(mods, seed):
    """Randomised sweep of the kernels either side of the matching path on odd frame shapes: RLE
    encoder, string codec round trip, connected components / label instances, region properties,
    polygon rasterisers, boundary distances, pixel-class maps."""
    A, E, S, R, D, rle = mods.analyze, mods.engine, mods.structures, mods.R, mods.data_utils, mods.rle
    rng = np.random.default_rng(7000 + seed)
    for trial in range(3):
        h, w, n = int(rng.integers(1, 140)), int(rng.integers(1, 140)), int(rng.integers(2, 24))
        a = U.rand_masks(rng, n, h, w, p_empty=0.1)
        a[0] = rng.random((h, w)) < 0.5
        a[1] = True
        tag = (seed, trial, h, w, n)
        # encoder (both memory layouts) + decoder round trip
        want = rle.encode(np.asfortranarray(a.transpose(1, 2, 0).astype(np.uint8)))
        assert [m['counts'] for m in E.encode_bool(a)] == [m['counts'] for m in want], tag
        y_major = np.asfortranarray(a.transpose(1, 2, 0)).transpose(2, 0, 1)          # the RLE.decode layout
        assert [m['counts'] for m in E.encode_bool(y_major)] == [m['counts'] for m in want], tag
        assert np.array_equal(S.masks_to_bitmask_array(want), a), tag
        assert np.array_equal(D.extract_boxes(y_major), R.extract_boxes(a)), tag
        # label images: connected components of the union and arbitrary label values
        union = a[2:].any(axis=0)
        for binary, img in ((True, union), (False, (rng.integers(0, 5, (h, w)) * rng.integers(1, 300)).astype(np.int64))):
            got, bb = E.label_image_to_instances(img, binary=binary)
            wl = R.annotations_from_label_image(img, binary=binary)
            assert [m['counts'] for m in got] == [m['counts'] for _, m in wl], tag
            if wl:
                assert np.array_equal(bb.astype(np.float64), np.stack([b for b, _ in wl])), tag
        # region properties
        got, wantp = S.region_properties(want), [R.regionprops_one(x) for x in a]
        _check_rprops(got, wantp)
        # polygons: pycocotools rule (RLE) and skimage rule (bitmask)
        polys = [np.round(rng.uniform(-5, max(h, w) + 5, size=2 * rng.integers(3, 9)) * 2) / 2 for _ in range(6)]
        from ampis_b200.containers import PolygonMasks
        assert [m['counts'] for m in S.masks_to_rle(PolygonMasks([[p] for p in polys]), (h, w))] == \
            [m['counts'] for m in R.polygons_to_rle([[p] for p in polys], (h, w))], tag
        assert np.array_equal(S.masks_to_bitmask_array(polys, (h, w)), R.poly2mask(polys, (h, w))), tag
        # boundary distances and pixel classes of "matches" between shifted copies
        b = np.roll(a, 1, axis=2)
        b[:, :, 0] = False
        eb = rle.encode(np.asfortranarray(b.transpose(1, 2, 0).astype(np.uint8)))
        pairs = np.array([[i, i] for i in range(n) if a[i].any() and b[i].any()]).reshape(-1, 2)
        boxes = np.tile(np.array([0, h, 0, w]), (n, 1))
        if len(pairs):
            fp, fn = A.mask_edge_distance(want, eb, boxes, boxes, pairs)
            wfp, wfn = R.mask_edge_distance(want, eb, boxes, boxes, pairs)
            assert all(np.array_equal(x.numpy(), y) for x, y in zip(fp + fn, wfp + wfn)), tag
            for mode in ('reduced', 'all'):
                iset, _ = A.seg_perf_iset(want, eb, {'tp': pairs}, mode=mode)
                assert [m['counts'] for m in iset.instances.masks.rle] == \
                    [m['counts'] for m in R.seg_perf_masks(want, eb, pairs, mode)], tag


def test_det_seg_scores_batch_equals_per_image_calls(mods):
    """The batch form (one table, one launch per kernel for all images) returns exactly the dicts the
    reference-style per-image loop returns -- shipped images of different instance counts."""
    A = mods.analyze
    g = U.load('powder_match.npz')
    images = [U.powder_match_image(k)[1:] for k in range(len(g['names']))]
    got = A.det_seg_scores_batch([x[0] for x in images], [x[1] for x in images], 0.5)
    assert len(got) == len(images)
    for (gt, pr), res in zip(images, got):
        want = A.det_seg_scores(gt, pr, 0.5)
        assert list(res) == list(want)
        for k in want:
            assert np.array_equal(np.asarray(res[k]), np.asarray(want[k])) and np.asarray(res[k]).dtype == np.asarray(want[k]).dtype, k
    assert A.det_seg_scores_batch([], []) == []
    with pytest.raises(ZeroDivisionError):
        A.det_seg_scores_batch([images[0][0], mods.structures.RLEMasks([])], [images[0][1], mods.structures.RLEMasks([])])


def _dicts(mods, host, g=0):
    rows, cols = host.image_masks(g)
    mk = lambda cs: [{'size': [host.h, host.w], 'counts': mods.rle.string_from_counts(c)} for c in cs]
    return mk(rows), mk(cols)


@pytest.mark.parametrize('decode,rows_kernel', [('flat', 'pairs'), ('group', 'grid'), ('flat', 'grid')])
def test_native_size_c4_image_vs_oracle(mods, decode, rows_kernel, monkeypatch):
    """BASELINE.json configs[3] at its NATIVE size -- one 2048 x 2048 frame, 5,000 x 5,000 small instances --
    through the drop-in functions against the oracle (one rleIou call over all 25 M pairs, the reference's matcher
    rules on its matrix, rleMerge on the matched pairs): det_seg_scores at three thresholds, the sparse IoU list
    against the non-zero cells of the oracle's matrix, areas and equivalent diameters.  Crop windows of 13-px blobs,
    the grid at 5,000 columns, the join and both decode kernels are exactly what VERDICT r1 asked to see here."""
    A, B, E, S, rle = mods.analyze, mods.batch, mods.engine, mods.structures, mods.rle
    monkeypatch.setattr(E, 'CROP_DECODE', decode)
    monkeypatch.setattr(E, 'ROWS_KERNEL', rows_kernel)
    if (decode, rows_kernel) != ('flat', 'pairs'):       # the one-call entries always run flat + pairs: the other
        monkeypatch.setattr(A, 'FUSED_CALL', False)      # kernels are reached through the table API
    host = B.synth('c4_spheroidite', 1, 4004)
    assert (host.h, host.w, host.n_rows, host.n_cols) == (2048, 2048, 5000, 5000)
    gt, pr = _dicts(mods, host)
    iou = U.iou_matrix_one_shot(rle, gt, pr)
    for th in (0.1, 0.5, 0.75):
        want = U.det_seg_scores_one_shot(rle, gt, pr, th, iou=iou)
        got = A.det_seg_scores(gt, pr, th)
        assert want.keys() == got.keys()
        for k in want:
            assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), (th, k)
    # 13-px blobs displaced by N(0, 2 px): most pairs overlap, few reach IoU 0.5
    assert len(U.match_from_iou(iou, 0.1)['tp']) > 2000 and len(U.match_from_iou(iou, 0.5)['tp']) > 50
    # through the table API as bench.py drives it (crop layout, sparse triplets)
    dev = B.DeviceBatch(host, dense=False)
    sp = E.SparseRows('cuda', 64 * host.n_rows)
    arena = mods.torch.empty(4 * B.arena_chunks_needed(dev, E.LAYOUT_CROP), dtype=mods.torch.int32, device='cuda')
    res = B.eval_step(dev, layout=E.LAYOUT_CROP, check=True, kernel='grid', sparse=sp, arena=arena)   # fused decode
    r, c, v = (x.cpu().numpy() for x in sp.triplets())
    wr, wc = np.nonzero(iou)
    assert np.array_equal(r, wr) and np.array_equal(c, wc)
    a_g, a_p = rle.area(gt).astype(np.int64), rle.area(pr).astype(np.int64)
    assert np.array_equal(v / (a_g[r] + a_p[c] - v), iou[wr, wc])
    m = U.match_from_iou(iou, 0.5)
    assert res.counts.cpu().numpy()[0, 0].tolist() == [len(m['tp']), len(m['fp']), len(m['fn'])]
    if decode == 'flat' and rows_kernel == 'pairs':
        sp2 = A.sparse_iou(gt, pr)
        assert np.array_equal(sp2['row'], wr) and np.array_equal(sp2['col'], wc) and np.array_equal(sp2['iou'], iou[wr, wc])
        assert np.array_equal(S.mask_areas(gt), rle.area(gt))
        d_eq = np.sqrt(4 * rle.area(pr).astype(np.float64) / np.pi)
        keep = np.nonzero(rle.area(pr))[0][:600]                     # regionprops rows exist for non-empty masks
        iset = S.InstanceSet()
        iset.instances = S.Instances((host.h, host.w), masks=S.RLEMasks([pr[i] for i in keep]),
                                     class_idx=np.zeros(len(keep), int))
        df = iset.compute_rprops(keys=['area', 'equivalent_diameter'], return_df=True)
        got_d = np.array([float(np.asarray(x).ravel()[0]) for x in df['equivalent_diameter']])
        assert np.allclose(got_d, d_eq[keep], rtol=1e-6, atol=0)        # north_star: 1e-6 relative on derived floats
        assert np.array_equal(np.array([int(np.asarray(x).ravel()[0]) for x in df['area']]), rle.area(pr)[keep])


@pytest.mark.parametrize('decode,rows_kernel', [('flat', 'pairs'), ('group', 'grid')])
def test_native_size_c3_image_vs_oracle(mods, decode, rows_kernel, monkeypatch):
    """BASELINE.json configs[2] at its NATIVE size -- 200 satellites x 2,000 particles in a 2048 x 2048 frame --
    _rle_satellite_match and satellite_measurements against the oracle (intersections by rleMerge wherever rleIou is
    non-zero, then the reference's per-satellite arg-max over all particles)."""
    B, E, P, rle = mods.batch, mods.engine, mods.powder, mods.rle
    monkeypatch.setattr(E, 'CROP_DECODE', decode)
    monkeypatch.setattr(E, 'ROWS_KERNEL', rows_kernel)
    if (decode, rows_kernel) != ('flat', 'pairs'):
        monkeypatch.setattr(mods.analyze, 'FUSED_CALL', False)
    host = B.synth('c3_satellites', 2, 3003)
    assert (host.h, host.w, host.n_rows, host.n_cols) == (2048, 2048, 200, 2000)
    for g in range(2):
        sat, part = _dicts(mods, host, g)
        want = U.satellite_match_one_shot(rle, part, sat, 0.5)
        got = P._rle_satellite_match(part, sat, 0.5)
        for k in ('satellite_matches', 'satellites_unmatched', 'particles_unmatched', 'intersection_scores'):
            assert np.array_equal(got[k], want[k]), (g, k)
        assert {a: list(b) for a, b in got['match_pairs'].items()} == {a: list(b) for a, b in want['match_pairs'].items()}
        assert 100 < len(want['satellite_matches']) < 200
    # the batch step on the same two frames: per-image counts
    dev = B.DeviceBatch(host, dense=False)
    arena = mods.torch.empty(4 * B.arena_chunks_needed(dev, E.LAYOUT_CROP), dtype=mods.torch.int32, device='cuda')
    res = B.eval_step(dev, layout=E.LAYOUT_CROP, check=True, arena=arena)
    for g in range(2):
        sat, part = _dicts(mods, host, g)
        want = U.satellite_match_one_shot(rle, part, sat, 0.5)
        assert res.counts.cpu().numpy()[g].tolist() == [len(want['satellite_matches']), len(want['satellites_unmatched']),
                                                        len(want['match_pairs']), host.n_cols]


def test_many_images_one_call_entry(mods, monkeypatch):
    """engine.eval_images (ampis_eval_images_host: string descriptors from the C marshaller, one upload, one launch
    of each kernel, one download for ALL images) == the per-image entry image by image: mixed image sizes and
    instance counts in one call, empty images, str / bytearray counts, both modes; the result cache; the crowd gate."""
    A, B, E, P, rle = mods.analyze, mods.batch, mods.engine, mods.powder, mods.rle
    imgs = []
    for k, (cfg, over) in enumerate([('c1_powder_example', {}), ('c2_powder_batch', {}),
                                     ('c4_spheroidite', dict(n_rows=900, n_cols=1100, h=1024, w=1024)),
                                     ('c2_powder_batch', dict(h=70, w=45, n_rows=9, n_cols=11, median_diam=30.0)),
                                     ('c3_satellites', dict(h=1024, w=1024, n_cols=700))]):
        host = B.synth(dict(B.CONFIGS[cfg], **over), 1, 900 + k)
        imgs.append(_dicts(mods, host))
    imgs.insert(2, ([], imgs[0][1][:5]))                        # no rows
    imgs.insert(4, (imgs[0][0][:7], []))                        # no columns
    imgs[3] = ([dict(m, counts=m['counts'].decode('ascii')) for m in imgs[3][0]],            # str counts
               [dict(m, counts=bytearray(m['counts']), size=tuple(m['size'])) for m in imgs[3][1]])
    for mode in (E.MODE_IOU, E.MODE_SAT):
        r = E.eval_images([x[0] for x in imgs], [x[1] for x in imgs], mode)
        assert not r.crowded and r.pairs_found > 0
        for g, (rows, cols) in enumerate(imgs):
            one = E.eval_image(rows, cols, mode)
            r0, r1, m0, m1 = int(r.row_off[g]), int(r.row_off[g + 1]), int(r.mask_off[g]), int(r.mask_off[g + 1])
            assert np.array_equal(r.area[m0:m1], one.area) and np.array_equal(r.bbox[m0:m1], one.bbox), (mode, g)
            assert np.array_equal(r.span[m0:m1], one.span), (mode, g)
            if len(rows) and len(cols):
                assert np.array_equal(r.best_col[r0:r1], one.best_col), (mode, g)
                assert np.array_equal(r.best_inter[r0:r1], one.best_inter), (mode, g)
                assert np.array_equal(r.best_score[r0:r1], one.best_score, equal_nan=True), (mode, g)
                assert abs(r.fill(g) - one.fill()) < 1e-12
    # errors: mixed sizes inside an image, malformed RLE, wrong types
    with pytest.raises(ValueError, match='different image sizes'):
        E.eval_images([imgs[0][0]], [imgs[1][1]], E.MODE_IOU)
    bad = [{'size': [45, 37], 'counts': rle.string_from_counts(np.array([3, 5000, 7, 900], np.uint32))}]
    with pytest.raises(ValueError, match='malformed RLE'):
        E.eval_images([bad, imgs[0][0]], [bad, imgs[0][1]], E.MODE_IOU)
    with pytest.raises(TypeError):
        E.eval_images([[{'size': [4, 4], 'counts': 7}]], [[]], E.MODE_IOU)
    # the cache: same string objects -> no second evaluation; new objects with the same content -> evaluated again
    calls = []
    real = E.N.lib().ampis_eval_images_host
    gt, pr = imgs[0]
    first = A.det_seg_scores(gt, pr, 0.5)

    class Spy(object):
        def __getattr__(self, name):
            if name == 'ampis_eval_images_host':
                return lambda *a: (calls.append(1), real(*a))[1]
            return getattr(E.N._lib, name)
    lib = E.N.lib()
    monkeypatch.setattr(E.N, 'lib', lambda: Spy())
    for th in (0.5, 0.6, 0.7, 0.95):
        res = A.det_seg_scores(gt, pr, th)
    assert calls == [] and all(np.array_equal(np.asarray(res[k]), np.asarray(mods.R.det_seg_scores(gt, pr, 0.95)[k])) for k in res)
    gt2 = [dict(m, counts=bytes(bytearray(m['counts']))) for m in gt]           # equal content, other objects
    again = A.det_seg_scores(gt2, pr, 0.5)
    assert calls == [1] and all(np.array_equal(np.asarray(again[k]), np.asarray(first[k])) for k in first)
    gt2[0] = dict(gt2[0], counts=gt2[1]['counts'])                                # content changed in place
    changed = A.det_seg_scores(gt2, pr, 0.5)
    assert calls == [1, 1]
    want = mods.R.det_seg_scores(gt2, pr, 0.5)
    assert all(np.array_equal(np.asarray(changed[k]), np.asarray(want[k])) for k in want)
    monkeypatch.setattr(E.N, 'lib', lambda: lib)
    # the crowd gate: a crowded image comes back flagged without its intersections having been computed
    host = B.synth(dict(B.CONFIGS['dense_overlap'], h=128, w=128, n_rows=70, n_cols=90, median_diam=70.0), 1, 5)
    cg, cp = _dicts(mods, host)
    r = E.eval_images([cg], [cp], E.MODE_IOU, crowd_frac=E.CROWD_PAIR_FRACTION)
    assert r.crowded and r.pairs_found > E.CROWD_PAIR_FRACTION * 70 * 90
    full = E.eval_images([cg], [cp], E.MODE_IOU)                                   # gate off: the culled walk does it all
    one = E.eval_image(cg, cp, E.MODE_IOU)
    assert not full.crowded and np.array_equal(full.best_col, one.best_col) and np.array_equal(full.best_score, one.best_score)
    assert np.array_equal(r.area, one.area)                                        # measurements are valid either way
    # batch scoring on a mix that contains a crowded image: still the per-image dicts
    res = A.det_seg_scores_batch([gt, cg], [pr, cp], 0.5)
    for got, (a_, b_) in zip(res, [(gt, pr), (cg, cp)]):
        want = mods.R.det_seg_scores(a_, b_, 0.5)
        assert all(np.array_equal(np.asarray(got[k]), np.asarray(want[k])) for k in want)


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: float64 arrays of the last timed step, equal whatever --steps is (the inputs are
    seeded), under 64 MB; the totals are those of the JSON line and the per-image counts sum to them."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def bench(steps, out):
        cmd = [sys.executable, os.path.join(root, 'bench.py'), '--images', '8', '--steps', str(steps), '--warmup', '1',
               '--no-cpu', '--no-e2e', '--no-span', '--no-c5', '--no-check', '--dump-outputs', str(out)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-800:]
        return json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][-1])

    a, b = bench(2, tmp_path / 'a'), bench(5, tmp_path / 'b')
    assert (a['steps'], b['steps']) == (2, 5)
    names = sorted(os.listdir(tmp_path / 'a'))
    assert names == sorted(os.listdir(tmp_path / 'b'))
    assert {'totals.npy', 'counts.npy', 'area.npy', 'best_col.npy', 'best_inter.npy', 'best_score.npy',
            'imat.npy'} <= set(names)
    nbytes = 0
    for n in names:
        x, y = np.load(tmp_path / 'a' / n), np.load(tmp_path / 'b' / n)
        assert x.dtype == np.float64 and np.array_equal(x, y), n
        nbytes += x.nbytes
    assert nbytes <= 64 << 20
    totals = np.load(tmp_path / 'a' / 'totals.npy')
    assert totals[0].tolist() == a['totals_tp_fp_fn_at_0.50']
    assert np.array_equal(np.load(tmp_path / 'a' / 'counts.npy').sum(axis=0), totals)
