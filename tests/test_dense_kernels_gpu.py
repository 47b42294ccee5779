"""The dense intersection kernels on the B200 -- the int8 tcgen05 contraction on single CTAs
(intersect_mma_kernel) and on CTA pairs (intersect_mma_pair_kernel), the TMA-tiled AND+popc (intersect_tma_kernel)
and the row results read off their matrices (rows_from_imat_kernel) -- and the crowded-image routes of the drop-in
API that lead to them, against the exact sparse reference of tests/_dense_ref.py.  Everything is compared exactly:
intersections and arg-max indices equal, float64 scores equal bit for bit (NaN where NaN).

Covered: launches of several images with 0 .. 300 rows and columns on frames whose pixel count is no multiple of 128
(tile edges, the last two-slab stage past the frame end, spans that start on an odd chunk); ties at columns 127/128
and 255/256 placed so that the span sort puts the later index first; contractions of thousands of ring iterations
(1024² crowded frames, 70000 x 6 and 6 x 9000 frames); intersections between 2^24 and 2^25, where 128·I no longer fits
a signed 32-bit accumulator; and the crowded images of det_seg_scores, _piecewise_iou, _piecewise_rle_match,
det_seg_scores_batch, _rle_satellite_match and PowderSatelliteImage.compute_matches."""
import os

import numpy as np
import pytest

from tests import _dense_ref as D
from tests import _util as U
from tests.test_gpu_parity import _counts_to_rle, _host_csr_from_bool

pytestmark = pytest.mark.gpu

SIDES = (1, 63, 64, 127, 128, 129, 255, 256, 257, 300)
KERNELS = [(False, True), (False, False), (True, True), (True, False)]          # (CTA pair, sorted tiles)


@pytest.fixture(scope='module')
def M():
    import torch
    assert torch.cuda.is_available(), 'these tests need the B200'
    from ampis_b200 import analyze, batch, engine, structures
    from ampis_b200.applications import powder
    from ampis_b200.containers import Instances
    from oracle import ampis_ref as R
    from oracle import cocomask as rle

    class _M:
        pass
    m = _M()
    m.torch, m.analyze, m.batch, m.engine, m.structures, m.powder, m.Instances, m.R, m.rle = \
        torch, analyze, batch, engine, structures, powder, Instances, R, rle
    return m


# ---- launches and their expected results -----------------------------------------------------------------------

class Launch(object):
    """Images of one frame size in one mask table: image g owns rows then columns, masks as run counts (uint32)."""

    def __init__(self, M, host, Gs, Ps):
        self.M, self.host = M, host
        self.Gs, self.Ps = [int(g) for g in Gs], [int(p) for p in Ps]
        self.dev = M.batch.DeviceBatch(host, dense=True)        # the upload; the groups below mix image shapes
        self.groups = M.engine.Groups.interleaved(self.dev.device, self.Gs, self.Ps, dense=True)
        self.want = {}

    def table(self, layout, fused=False):
        E, B, d = self.M.engine, self.M.batch, self.dev
        t = E.MaskTable(d.device, self.host.n_masks, d.cnt, d.cnt_off, d.cnt_len, d.h, d.w, layout)
        if fused:
            n = max(B.arena_chunks_needed(d, layout), 1)
            t.measure_paint(self.M.torch.empty(4 * n, dtype=self.M.torch.int32, device=d.device))
        else:
            t.measure().paint()
        return t.check()

    def expect(self, I_per_image, area):
        """I_per_image: int64 [G, P] per image; area: int64 per mask of the table."""
        self.I = I_per_image
        self.area = np.asarray(area, np.int64)
        start = np.concatenate([[0], np.cumsum(np.add(self.Gs, self.Ps))])
        self.row_area = [self.area[s:s + g] for s, g in zip(start, self.Gs)]
        self.col_area = [self.area[s + g:s + g + p] for s, g, p in zip(start, self.Gs, self.Ps)]
        return self

    def rows_want(self, mode):
        if mode not in self.want:
            out = []
            for I, ar, ac in zip(self.I, self.row_area, self.col_area):
                if mode == self.M.engine.MODE_IOU:
                    out.append(D.rows_iou(I, ar, ac)[:3])
                else:
                    out.append(D.rows_sat(I, ar))
            self.want[mode] = [np.concatenate([o[k] for o in out]) if out else np.zeros(0) for k in range(3)]
        return self.want[mode]

    def check(self, res, mode, tag):
        """res: an engine.RowResult with dense matrices; every cell and every row against the reference.  A mismatch
        names the image, the row and the column."""
        g = self.groups
        imat = res.imat[:g.imat_size].cpu().numpy().astype(np.int64)
        for k, (I, off) in enumerate(zip(self.I, g.h_imat_off)):
            got = imat[off:off + I.size].reshape(I.shape)
            if not np.array_equal(got, I):
                r, c = np.argwhere(got != I)[0]
                raise AssertionError('%s: image %d (G=%d, P=%d), I[%d, %d] = %d, want %d (%d cells differ)'
                                     % (tag, k, I.shape[0], I.shape[1], r, c, got[r, c], I[r, c],
                                        int((got != I).sum())))
        n = g.n_rows
        best = res.best_col[:n].cpu().numpy().astype(np.int64)
        inter = res.best_inter[:n].cpu().numpy().view(np.uint32).astype(np.int64)
        score = res.best_score[:n].cpu().numpy()
        wb, wi, ws = self.rows_want(mode)
        for name, a, b in (('best_col', best, wb), ('best_inter', inter, wi), ('best_score', score, ws)):
            eq = (a == b) | (np.isnan(a) & np.isnan(b)) if a.dtype.kind == 'f' else a == b
            if not eq.all():
                r = int(np.nonzero(~eq)[0][0])
                k = int(np.searchsorted(np.cumsum(self.Gs), r, side='right'))
                raise AssertionError('%s: %s of row %d (image %d, row %d) = %r, want %r'
                                     % (tag, name, r, k, r - int(g.h_row_begin[k]), a[r], b[r]))


def _bool_launch(M, stacks, Gs, Ps):
    """Bool stacks [G + P, h, w] per image (one frame size) -> Launch with its reference."""
    h, w = stacks[0].shape[1:]
    allm = np.concatenate(stacks)
    host = _host_csr_from_bool(M.batch, [allm], 0, h, w, M.rle)       # one flat list of masks; groups come apart
    L = Launch(M, host, Gs, Ps)
    return L.expect([D.intersections(s[:g], s[g:]) for s, g in zip(stacks, Gs)], D.areas(allm))


def _counts_launch(M, h, w, images, reference=True):
    """images: per image (rows, cols) as lists of uint32 run counts -> Launch, with the sparse reference unless
    reference=False (the caller then sets the expected values)."""
    cnts = [c for rows, cols in images for c in list(rows) + list(cols)]
    lens = np.array([len(c) for c in cnts], np.int32)
    off = np.zeros(len(cnts), np.int64)
    off[1:] = np.cumsum(lens[:-1])
    cfg = dict(h=h, w=w, n_rows=0, n_cols=len(cnts), kind=0, mode=0)
    host = M.batch.HostCSR(cfg, 1, np.concatenate(cnts).astype(np.uint32), off, lens)
    L = Launch(M, host, [len(r) for r, _ in images], [len(c) for _, c in images])
    if not reference:
        return L
    return L.expect([D.intersections(list(r), list(c), hw=h * w) for r, c in images], D.areas(cnts, hw=h * w))


def _counts(intervals, hw):
    """Sorted, disjoint, non-touching [start, end) pixel intervals (column-major) -> RLE run counts."""
    out, pos = [], 0
    for s, e in intervals:
        out += [s - pos, e - s]
        pos = e
    if pos < hw:
        out.append(hw - pos)
    return np.asarray(out if out else [hw], np.uint32)


def _run_all(M, L, layouts=None, tma=True):
    """Every dense kernel configuration and the culled rows kernel on every table, both modes."""
    E = M.engine
    layouts = layouts or [(E.LAYOUT_SPAN, False), (E.LAYOUT_SPAN, True), (E.LAYOUT_FULL, False), (E.LAYOUT_FULL, True)]
    for layout, fused in layouts:
        t = L.table(layout, fused)
        for mode in (E.MODE_IOU, E.MODE_SAT):
            tag = lambda k: 'layout %d fused %d mode %d %s' % (layout, fused, mode, k)
            L.check(E.intersect_rows(t, L.groups, mode), mode, tag('rows'))
            for pair, sort in KERNELS:
                L.check(E.intersect_mma(t, L.groups, mode, pair=pair, sort=sort), mode,
                        tag('mma pair=%s sort=%s' % (pair, sort)))
            if tma and layout == E.LAYOUT_FULL and not fused and L.groups.n_rows:
                L.check(E.intersect_tma(t, L.groups, mode), mode, tag('tma'))


# ---- a. tile edges ------------------------------------------------------------------------------------------------

def _edge_masks(rng, n, h, w):
    """n masks of an h x w frame: blobs and the kinds the tile code trips on -- empty, one pixel, full frame, pixels
    in the last 128-pixel chunk only, a run that starts on an odd chunk, column stripes, row stripes, noise."""
    hw = h * w
    m = U.rand_masks(rng, n, h, w, p_empty=0.05)
    flat = np.zeros(hw, bool)
    last = (hw - 1) // 128 * 128
    n_chunks = (hw + 127) // 128
    for i, k in enumerate(rng.integers(0, 12, n)):
        flat[:] = False
        if k == 0:
            m[i] = False
            continue
        if k == 1:
            flat[rng.integers(0, hw)] = True
        elif k == 2:
            flat[:] = True
        elif k == 3:
            flat[last + rng.integers(0, hw - last, 3)] = True
        elif k == 4 and n_chunks > 2:
            c = 2 * int(rng.integers(0, (n_chunks - 1) // 2)) + 1         # an odd chunk: klo & ~1 rounds below it
            s = c * 128 + int(rng.integers(0, 128))
            flat[s:s + int(rng.integers(1, 700))] = True
        elif k == 5:
            c0 = int(rng.integers(0, w))
            m[i] = False
            m[i, :, c0:c0 + int(rng.integers(1, 6))] = True
            continue
        elif k == 6:
            r0 = int(rng.integers(0, h))
            m[i] = False
            m[i, r0:r0 + int(rng.integers(1, 5)), :] = True
            continue
        elif k == 7:
            m[i] = rng.random((h, w)) < 0.3
            continue
        else:
            continue                                                    # blob
        m[i] = flat.reshape(w, h).T                                     # column-major pixel order
    return m


@pytest.mark.parametrize('seed', range(int(os.environ.get('AMPIS_FUZZ_SEEDS', '3'))))
def test_tile_edges_mixed_images_every_dense_kernel(M, seed):
    """Five images per launch with G, P drawn from tile-edge sizes (one without rows, one without columns, one with
    both sides above 256) on an odd frame: intersect_mma single CTA / CTA pair x sorted / unsorted tiles, SPAN and FULL
    tables (fused and unfused decode), IoU and satellite rows, the TMA kernel on unfused FULL tables and the culled
    rows kernel -- every cell and every row equal to the sparse reference."""
    rng = np.random.default_rng(3100 + seed)
    h, w = 2 * int(rng.integers(10, 45)) + 1, 2 * int(rng.integers(10, 45)) + 1      # h·w odd: no multiple of 128
    n_img = 5
    Gs, Ps = rng.choice(SIDES, n_img), rng.choice(SIDES, n_img)
    Gs[0], Ps[0] = rng.choice([257, 300]), rng.choice([257, 300])
    e0, e1 = rng.choice(np.arange(1, n_img), 2, replace=False)
    Gs[e0], Ps[e1] = 0, 0
    stacks = [_edge_masks(rng, int(g + p), h, w) for g, p in zip(Gs, Ps)]
    L = _bool_launch(M, stacks, Gs, Ps)
    _run_all(M, L)


# ---- b. ties across tile and sort boundaries ---------------------------------------------------------------------

def _tie_image(h, w, G, P, rng, identical_at, split_at):
    """One image whose rows 127 / 128 overlap only a pair of tied columns at `identical_at` (two copies of one mask),
    and whose rows 0 / 255 / 256 overlap only a pair at `split_at`: two different masks of equal area with equal
    intersections, the higher index starting one chunk earlier in the frame, so the span sort puts it first."""
    hw = h * w
    L_, E_ = 150, 20

    def region(base):
        R = np.zeros(hw, bool)
        R[base + E_:base + E_ + 2 * L_] = True
        X = np.zeros(hw, bool)
        X[base + E_ + L_:base + 2 * E_ + 2 * L_] = True                  # later in the frame
        Y = np.zeros(hw, bool)
        Y[base:base + E_ + L_] = True                                    # earlier: first chunk before X's
        return R, X, Y
    fr = lambda v: v.reshape(w, h).T
    m = _edge_masks(rng, G + P, h, w)
    free = 800 // h + 1                                                  # the two regions sit in frame columns < free
    m[:, :, :free] = False
    R1, X1, Y1 = region(0)
    R2, X2, Y2 = region(400)
    for r in (127, 128):
        m[r] = fr(R1)
    for r in (0, 255, 256):
        m[r] = fr(R2)
    c0, c1 = identical_at
    m[G + c0] = m[G + c1] = fr(R1)
    c0, c1 = split_at
    m[G + c0], m[G + c1] = fr(X2), fr(Y2)
    return m


def test_ties_across_tile_and_sort_boundaries(M):
    """Tied columns at 127/128 and 255/256 (a 128-column and a 256-column tile edge, lanes 31 / 0 of the row
    reduction), tied rows on both CTAs of a pair tile and in the next tile: the lowest index wins on every kernel."""
    h, w = 61, 67
    rng = np.random.default_rng(77)
    G, P = 300, 300
    a = _tie_image(h, w, G, P, rng, (127, 128), (255, 256))
    b = _tie_image(h, w, G, P, rng, (255, 256), (127, 128))
    L = _bool_launch(M, [a, b], [G, G], [P, P])
    for k, (cid, csplit) in enumerate((((127, 128), (255, 256)), ((255, 256), (127, 128)))):
        I = L.I[k]
        assert I[127, cid[0]] == I[127, cid[1]] > 0 and I[0, csplit[0]] == I[0, csplit[1]] > 0
        best = D.rows_iou(I, L.row_area[k], L.col_area[k])[0]
        assert best[127] == best[128] == cid[0] and best[0] == best[255] == best[256] == csplit[0]
        assert (D.rows_sat(I, L.row_area[k])[0][[0, 127, 128, 255, 256]] == [csplit[0], cid[0], cid[0], csplit[0],
                                                                               csplit[0]]).all()
    _run_all(M, L, layouts=[(M.engine.LAYOUT_SPAN, False), (M.engine.LAYOUT_FULL, False)])


# ---- c. long contractions ----------------------------------------------------------------------------------------

def test_crowded_1024_frame(M):
    """dense_overlap scaled to a 1024² frame (300 x 520 masks of about 256 px): up to 4,096 ring iterations per tile
    (8,192 slabs, two per stage), so every stage parity flips thousands of times."""
    B = M.batch
    host = B.synth(dict(B.CONFIGS['dense_overlap'], h=1024, w=1024, n_rows=300, n_cols=520, median_diam=256.0), 1, 7)
    rows, cols = host.image_masks(0)
    L = _counts_launch(M, 1024, 1024, [(rows, cols)])
    assert (L.I[0] > 0).mean() > 0.1
    _run_all(M, L, layouts=[(M.engine.LAYOUT_SPAN, True)], tma=False)


@pytest.mark.parametrize('h,w', [(70000, 6), (6, 9000)])
def test_tall_and_wide_frames(M, h, w):
    """Crowded stripes on a 70000 x 6 frame (bands across columns: every mask spans most of the frame, 3,282 slabs)
    and a 6 x 9000 frame (column bands), 129 rows x 257 columns: long contractions on odd tile shapes."""
    rng = np.random.default_rng(h + w)
    hw = h * w

    def stripe():
        if h > w:                                        # rows [a, b) in columns [c0, c1): one run per column
            a = int(rng.integers(0, h - 1))
            b = min(h, a + int(rng.integers(h // 8, h // 2)))
            c0 = int(rng.integers(0, w))
            c1 = int(rng.integers(c0 + 1, w + 1))
            if a == 0 and b == h:
                return _counts([(c0 * h, c1 * h)], hw)
            return _counts([(c * h + a, c * h + b) for c in range(c0, c1)], hw)
        a = int(rng.integers(0, w - 1))                  # columns [a, b), all rows: one run
        b = min(w, a + int(rng.integers(w // 8, w // 2)))
        return _counts([(a * h, b * h)], hw)
    G, P = 129, 257
    L = _counts_launch(M, h, w, [([stripe() for _ in range(G)], [stripe() for _ in range(P)])])
    assert (L.I[0] > 0).mean() > 0.2
    _run_all(M, L, layouts=[(M.engine.LAYOUT_SPAN, False), (M.engine.LAYOUT_FULL, False)], tma=False)


# ---- d. the documented accumulator range --------------------------------------------------------------------------

def test_intersections_between_2_24_and_2_25(M):
    """A 4100 x 4100 frame (16,810,000 pixels): intersections from 2^24 - 1 to 16,810,000 < 2^25, where 128·I passes
    the signed 32-bit range of the accumulator (2^31 at I = 2^24) but not the unsigned one.  Expected values in
    closed form (intervals of the column-major pixel order); single CTA and CTA pairs, FULL and SPAN tables."""
    E = M.engine
    h = w = 4100
    hw = h * w
    T = 1 << 24
    rows = [(0, hw), (0, hw), (0, hw // 2), (0, hw - 1000), (0, T - 1), (0, T)]       # two full, one half frame, ...
    cols = [(0, hw), (0, hw), (hw // 2, hw), (500, hw), (hw - T - 3, hw)]
    inter = lambda a, b: max(0, min(a[1], b[1]) - max(a[0], b[0]))
    I = np.array([[inter(a, b) for b in cols] for a in rows], np.int64)
    assert I.max() == hw < 2 * T and (I > T).sum() >= 10 and (I == T - 1).any() and (I == T).any()
    L = _counts_launch(M, h, w, [([_counts([r], hw) for r in rows], [_counts([c], hw) for c in cols])], reference=False)
    L.expect([I], [e - s for s, e in rows + cols])
    for layout in (E.LAYOUT_FULL, E.LAYOUT_SPAN):
        t = L.table(layout)
        for mode in (E.MODE_IOU, E.MODE_SAT):
            for pair in (False, True):
                L.check(E.intersect_mma(t, L.groups, mode, pair=pair, sort=False), mode,
                        'layout %d mode %d pair %s' % (layout, mode, pair))


# ---- e. crowded images through the drop-in API --------------------------------------------------------------------

def _crowded_image(M, seed, n_rows=130, n_cols=260):
    """A 157 x 141 frame of large overlapping instances: operand fill about 0.35 and a third of all pairs with
    overlapping boxes, above both crowd gates, 130 x 260 masks (tile edges on both sides)."""
    B = M.batch
    host = B.synth(dict(B.CONFIGS['dense_overlap'], h=157, w=141, n_rows=n_rows, n_cols=n_cols, median_diam=80.0), 1,
                   seed)
    rows, cols = host.image_masks(0)
    return _counts_to_rle(M.rle, rows, host.h, host.w), _counts_to_rle(M.rle, cols, host.h, host.w)


def _same(got, want, what):
    for k in want:
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k]), equal_nan=np.asarray(want[k]).dtype.kind == 'f'), \
            (what, k)


@pytest.mark.parametrize('fused_call', [True, False])
def test_crowded_images_of_the_drop_in_api(M, monkeypatch, fused_call):
    """det_seg_scores, _piecewise_iou, _piecewise_rle_match at several thresholds, det_seg_scores_batch on crowded and
    sparse images, _rle_satellite_match and PowderSatelliteImage.compute_matches on crowded images (with zero-area
    satellites and duplicate particles) equal the oracle, and the crowded images go to the contraction."""
    A, E, R, rle, P = M.analyze, M.engine, M.R, M.rle, M.powder
    monkeypatch.setattr(A, 'FUSED_CALL', fused_call)
    used = []
    real = E.intersect
    monkeypatch.setattr(E, 'intersect', lambda t, g, m, out=None, kernel='auto': (used.append(kernel), real(t, g, m, out, kernel))[1])
    gt, pr = _crowded_image(M, 11)
    pr = pr[:40] + [dict(pr[7]), dict(pr[7])] + pr[40:]                  # duplicate predictions: IoU ties
    _same(A.det_seg_scores(gt, pr, 0.5), R.det_seg_scores(gt, pr, 0.5), 'det_seg_scores')
    assert used == ['mma']
    assert np.array_equal(A._piecewise_iou(gt, pr), R.piecewise_iou(gt, pr)) and used[-1] == 'mma'
    for th in (0.0, 0.3, 0.5, 0.8):
        used.clear()
        _same(A._piecewise_rle_match(gt, pr, th), R.piecewise_rle_match(gt, pr, th), '_piecewise_rle_match %s' % th)
        assert used == ['mma'], th
    # a batch of crowded and sparse images: the batch goes image by image, each to its kernel
    B = M.batch
    small = B.synth(dict(B.CONFIGS['c2_powder_batch'], h=157, w=141, n_rows=30, n_cols=30, median_diam=14.0), 1, 3)
    sg, sp = (_counts_to_rle(rle, c, small.h, small.w) for c in small.image_masks(0))
    g2, p2 = _crowded_image(M, 12)
    used.clear()
    got = A.det_seg_scores_batch([gt, sg, g2], [pr, sp, p2], 0.5)
    assert used.count('mma') == 2
    for k, (g, p) in enumerate(((gt, pr), (sg, sp), (g2, p2))):
        _same(got[k], R.det_seg_scores(g, p, 0.5), 'det_seg_scores_batch image %d' % k)
    # satellites: rows = satellites (three of them empty), columns = particles (two of them duplicated)
    empty = rle.encode(np.zeros((157, 141, 1), np.uint8, order='F'))[0]
    sats = gt[:50] + [empty] + gt[50:100] + [empty, empty] + gt[100:]
    parts = pr
    for th in (0.2, 0.5, 0.8):
        used.clear()
        _same(P._rle_satellite_match(parts, sats, th), U.satellite_match_one_shot(rle, parts, sats, th),
              '_rle_satellite_match %s' % th)
        assert used == ['mma'], th
    mk = lambda ms: M.structures.InstanceSet(instances=M.Instances((157, 141), masks=M.structures.RLEMasks(ms),
                                                                   boxes=np.zeros((len(ms), 4))))
    psi = P.PowderSatelliteImage(mk(parts), mk(sats))
    used.clear()
    psi.compute_matches(0.5)
    assert used == ['mma']
    _same(psi.matches, U.satellite_match_one_shot(rle, parts, sats, 0.5), 'compute_matches')
