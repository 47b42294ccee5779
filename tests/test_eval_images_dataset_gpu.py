"""The many-image entry (ampis_eval_images_host, engine.eval_images) at dataset scale against tests/_dataset_ref.py,
a numpy / scipy reference that shares none of its code: one seeded dataset of more than 40 images and 20,000 masks
with frame sizes mixed inside the call, empty and full-frame masks, images without rows or columns, exact copies
(arg-max ties), IoUs exactly on a COCO threshold, equal satellite overlaps, zero-area satellites, frame-spanning
diagonals and one crowded frame.  Every output is compared with the reference, floats bit for bit.  Covered: both
modes; the C entry with ten thresholds through every way of passing strings, lengths and outputs; the 16,384-mask
boundary between host-filled and device-expanded bookkeeping; the AMPIS_ENOSPC protocol from 4 KB workspaces and
their reuse; the grid entry list of frames with diagonals; the drop-in and sharded functions on the same data."""
import ctypes as C
import os
import re
import socket

import numpy as np
import pytest

from tests import _dataset_ref as D

pytestmark = pytest.mark.gpu

HOST_FILL_MAX = 16384               # eval_images.cu: EI_HOST_FILL_MAX


# ---- dataset ---------------------------------------------------------------------------------------------------

def _rle_of_pixels(rle, y, x, h, w):
    """Compressed RLE dict of the pixels (y, x) of an h x w frame."""
    idx = np.unique(np.asarray(x, np.int64) * h + np.asarray(y, np.int64))
    if len(idx) == 0:
        cnt = [h * w]
    else:
        br = np.flatnonzero(np.diff(idx) != 1)
        s = idx[np.r_[0, br + 1]]
        e = idx[np.r_[br, len(idx) - 1]] + 1
        cnt = np.empty(2 * len(s) + 1, np.int64)
        cnt[0] = s[0]
        cnt[1::2] = e - s
        cnt[2:-1:2] = s[1:] - e[:-1]
        cnt[-1] = h * w - e[-1]
        cnt = cnt if cnt[-1] else cnt[:-1]
    return {'size': [h, w], 'counts': rle.string_from_counts(np.asarray(cnt, np.uint32))}


def _rle_of_frame(rle, f):
    y, x = np.nonzero(f)
    return _rle_of_pixels(rle, y, x, *f.shape)


def _synth(mods, cfg, n, seed, **over):
    host = mods.batch.synth(dict(mods.batch.CONFIGS[cfg], **over), n, seed)
    mk = lambda cs: [{'size': [host.h, host.w], 'counts': mods.rle.string_from_counts(c)} for c in cs]
    return [tuple(mk(x) for x in host.image_masks(g)) for g in range(n)]


def _diagonal_image(rle, rng, n_rows=100, n_cols=500, n_diag=14, h=1024, w=1024):
    """Columns: n_diag thin lines across the whole frame (3 % of them) among 5-pixel plus signs; the mean box side
    stays at 32 px, so the grid cells are 32 px and every diagonal registers in all 32 x 32 cells.  Rows: plus signs
    (some copied from the columns, some shifted by a pixel) and two diagonals shifted by a pixel."""
    def plus(cy, cx):
        return _rle_of_pixels(rle, [cy, cy - 1, cy + 1, cy, cy], [cx, cx, cx, cx - 1, cx + 1], h, w)

    def diag(k):
        x = np.arange(w)
        y = (x * (h - 1) // (w - 1) + 37 * k) % h if k % 2 == 0 else (h - 1 - x * (h - 1) // (w - 1) + 37 * k) % h
        return _rle_of_pixels(rle, y, x, h, w)
    cen = rng.integers(1, min(h, w) - 2, size=(n_cols + n_rows, 2))
    cols = [plus(*c) for c in cen[:n_cols - n_diag]]
    for k in range(n_diag):
        cols.insert(int(rng.integers(0, len(cols) + 1)), diag(k))
    rows = [diag(0), _rle_of_pixels(rle, (np.arange(w) + 1) % h, np.arange(w), h, w)]    # the second one px off
    for k in range(n_rows - 2):
        rows.append(cols[int(rng.integers(0, n_cols))] if k % 3 == 0 else plus(*(cen[n_cols + k] + (k % 2))))
    return rows, cols


def _with_copies(rng, rows, cols, k=5):
    """Exact copies: rows among the columns, columns duplicated further on, rows duplicated (ties for the arg-max)."""
    cols = list(cols)
    for m in list(rows[::max(len(rows) // k, 1)][:k]) + list(cols[::max(len(cols) // k, 1)][:k]):
        cols.insert(int(rng.integers(0, len(cols) + 1)), dict(m))
    return list(rows) + [dict(m) for m in rows[:k]], cols


def _hand_images(rle, rng):
    imgs = []
    # IoU exactly k / 20 (k = 10 ... 20): 20-pixel ground truths, k-pixel subsets of them as predictions
    gt, pr = [], []
    for k in range(10, 21):
        y, x = 6 * (k % 5), 6 * (k - 10)
        yy, xx = np.mgrid[y:y + 4, x:x + 5]
        gt.append(_rle_of_pixels(rle, yy.T.ravel(), xx.T.ravel(), 64, 80))
        pr.append(_rle_of_pixels(rle, yy.T.ravel()[:k], xx.T.ravel()[:k], 64, 80))
    imgs.append((gt, [pr[i] for i in rng.permutation(len(pr))]))
    # satellites: one overlapping two particles equally (the larger one first), zero-area satellites
    p0, p1, s0, s1, empty = (np.zeros((16, 16), bool) for _ in range(5))
    p0[:, :6] = True
    p1[:, 6:9] = True
    s0[6:8, 4:8] = True
    s1[1:3, 7:9] = True
    imgs.append(([_rle_of_frame(rle, a) for a in (s0, empty, s1, empty)], [_rle_of_frame(rle, a) for a in (p0, p1, empty)]))
    # empty and full-frame masks on an odd frame
    h, w = 37, 23
    yy, xx = np.mgrid[0:h, 0:w]
    blob = lambda cy, cx, r: (yy - cy) ** 2 + (xx - cx) ** 2 <= r * r
    empty, full = np.zeros((h, w), bool), np.ones((h, w), bool)
    rows = [_rle_of_frame(rle, a) for a in (empty, full, blob(10, 10, 4), blob(30, 5, 6), empty, full)]
    cols = [_rle_of_frame(rle, a) for a in (full, empty, blob(10, 10, 4), full, blob(20, 15, 5), empty)]
    imgs.append((rows, cols))
    # a 1 x 1 frame
    one = lambda v: _rle_of_pixels(rle, [0] * v, [0] * v, 1, 1)
    imgs.append(([one(0), one(1)], [one(1), one(0), one(1)]))
    return imgs


class Dataset(object):
    pass


@pytest.fixture(scope='module')
def mods():
    import torch
    assert torch.cuda.is_available(), 'these tests need the B200'
    from ampis_b200 import analyze, batch, distributed, engine
    from oracle import cocomask as rle

    class M:
        pass
    m = M()
    m.torch, m.analyze, m.batch, m.distributed, m.engine, m.rle = torch, analyze, batch, distributed, engine, rle
    return m


@pytest.fixture(scope='module')
def ds(mods):
    rng = np.random.default_rng(2026)
    rle = mods.rle
    imgs = []
    c2 = _synth(mods, 'c2_powder_batch', 18, 11)                                    # 1024 x 1024, 500 x 500
    for k in (2, 9):
        c2[k] = _with_copies(rng, *c2[k])
    imgs += c2
    imgs += _synth(mods, 'c1_powder_example', 4, 12)                                # 768 x 1024
    imgs += _synth(mods, 'c2_powder_batch', 2, 13, h=1024, w=1536, n_rows=400, n_cols=400)
    imgs += _synth(mods, 'c2_powder_batch', 2, 14, h=1001, w=999, n_rows=300, n_cols=300)
    imgs += _synth(mods, 'c2_powder_batch', 2, 15, h=4100, w=40, n_rows=150, n_cols=150, median_diam=12.0)
    imgs += _synth(mods, 'c2_powder_batch', 2, 16, h=40, w=4100, n_rows=150, n_cols=150, median_diam=12.0)
    small = _synth(mods, 'c2_powder_batch', 3, 17, h=256, w=256, n_rows=40, n_cols=40, median_diam=30.0)
    imgs.append(_with_copies(rng, *small[0], k=12))
    imgs += [([], small[1][1]), (small[2][0], []), ([], [])]                          # no rows / no columns / neither
    imgs += _hand_images(rle, rng)
    d = Dataset()
    d.diag = [_diagonal_image(rle, rng) for _ in range(2)]
    imgs += d.diag
    imgs += _synth(mods, 'dense_overlap', 1, 18)                                    # crowded frame, 512 x 512
    order = rng.permutation(len(imgs))                                              # frame sizes mixed in the call
    d.imgs = [imgs[i] for i in order]
    d.rows, d.cols = [list(r) for r, _ in d.imgs], [list(c) for _, c in d.imgs]
    d.n = sum(len(r) + len(c) for r, c in d.imgs)
    d.th = mods.batch.COCO_THRESHOLDS
    d.ref = {mode: D.dataset(d.rows, d.cols, mode, d.th if mode == D.MODE_IOU else None)
             for mode in (D.MODE_IOU, D.MODE_SAT)}
    assert len(d.imgs) >= 40 and d.n >= 20000
    return d


# ---- helpers ---------------------------------------------------------------------------------------------------

def _same_f64(a, b):
    """float64 arrays equal bit for bit (NaN where the other has NaN: the device's 0/0 has another bit pattern)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))


def _check(got, ref, what):
    assert np.array_equal(np.asarray(got['best_col']), ref['best_col']), what
    assert np.array_equal(np.asarray(got['best_inter']).view(np.uint32), ref['best_inter']), what
    assert _same_f64(got['best_score'], ref['best_score']), what
    assert np.array_equal(np.asarray(got['area']).view(np.uint32), ref['area']), what
    if got.get('bbox') is not None:
        assert np.array_equal(np.asarray(got['bbox']).reshape(-1, 4), ref['bbox']), what
    assert np.array_equal(np.asarray(got['status']), ref['status']), what


def _rows_dict(r):
    return dict(best_col=r.best_col, best_inter=r.best_inter, best_score=r.best_score, area=r.area, bbox=r.bbox,
                status=r.status)


class Entry(object):
    """ampis_eval_images_host through ctypes, with caller-owned workspaces grown as AMPIS_ENOSPC asks."""

    def __init__(self, mods, d_bytes=4096, h_bytes=4096):
        self.m = mods
        self.d_ws = mods.torch.empty(d_bytes, dtype=mods.torch.uint8, device='cuda')
        self.h_ws = mods.torch.empty(h_bytes, dtype=mods.torch.uint8, pin_memory=True)
        self.grown, self.messages = [], []

    def run(self, rows, cols, mode, thresholds=None, contiguous=False, pinned_out=False, pinned_len=False,
            blocking=False, no_box=False, crowd_frac=-1.0, max_calls=12):
        m, torch = self.m, self.m.torch
        E = m.engine
        NI = len(rows)
        n_rows = np.array([len(r) for r in rows], np.int32)
        n_cols = np.array([len(c) for c in cols], np.int32)
        n, R = int(n_rows.sum() + n_cols.sum()), int(n_rows.sum())
        lists = [None] * (2 * NI)
        lists[0::2], lists[1::2] = rows, cols
        ptr, ln, hw = np.empty(max(n, 1), np.uint64), np.empty(max(n, 1), np.int32), np.empty((max(n, 1), 2), np.int32)
        refs = []
        assert E.marshal().gather(lists, ptr, ln, hw, refs)[0] == n
        first = np.r_[0, np.cumsum(n_rows + n_cols)[:-1]].astype(np.int64)
        h = np.where(n_rows + n_cols > 0, hw[np.minimum(first, n - 1), 0], 0).astype(np.uint32)
        w = np.where(n_rows + n_cols > 0, hw[np.minimum(first, n - 1), 1], 0).astype(np.uint32)
        keep = [refs]
        if contiguous:                       # one blob in pinned memory; only str_ptr[0] is read
            blob = b''.join(m_['counts'] for l in lists for m_ in l)
            pb = torch.empty(max(len(blob), 1), dtype=torch.uint8, pin_memory=True).numpy()
            pb[:len(blob)] = np.frombuffer(blob, np.uint8)
            keep.append(pb)
            ptr[:] = 0
            ptr[0] = pb.ctypes.data
        if pinned_len:
            pl = torch.empty(max(n, 1), dtype=torch.int32, pin_memory=True).numpy()
            pl[:] = ln
            ln = pl

        def out(shape, dt):
            # uint32 outputs are int32 buffers seen as uint32 (torch has no pinned uint32 allocation of its own)
            store = np.int32 if dt == np.uint32 else dt
            if pinned_out:
                a = torch.from_numpy(np.empty(0, store)).new_empty(shape).pin_memory().numpy()
            else:
                a = np.empty(shape, store)
            a.reshape(-1).view(np.uint8)[:] = 0xA5             # nothing from an earlier call can pass for a result
            return a.view(dt)
        T = 0 if thresholds is None else len(thresholds)
        o = dict(best_col=out(R, np.int32), best_inter=out(R, np.uint32), best_score=out(R, np.float64),
                 area=out(n, np.uint32), bbox=None if no_box else out((n, 4), np.int32),
                 span=None if no_box else out((n, 2), np.uint32), status=out(n, np.int32),
                 grp_counts=out((NI, T, 3), np.int32) if T else None, totals=out((T, 3), np.int64) if T else None)
        th = np.ascontiguousarray(thresholds, np.float64) if T else None
        found, crowded, need = C.c_int64(-7), C.c_int32(-7), C.c_int64(0)
        a = lambda x: None if x is None else x.ctypes.data
        lib = E.N.lib()
        flags = (1 if contiguous else 0) | (2 if blocking else 0)
        for _ in range(max_calls):
            rc = lib.ampis_eval_images_host(
                a(ptr), a(ln), NI, a(n_rows), a(n_cols), a(h), a(w), mode, flags, float(crowd_frac),
                self.d_ws.data_ptr(), self.d_ws.numel(), self.h_ws.data_ptr(), self.h_ws.numel(), a(o['best_col']),
                a(o['best_inter']), a(o['best_score']), a(o['area']), a(o['bbox']), a(o['span']), a(o['status']),
                a(th), T, a(o['grp_counts']), a(o['totals']), C.byref(found), C.byref(crowded), C.byref(need),
                C.c_void_p(torch.cuda.current_stream().cuda_stream))
            if rc != E.N.ENOSPC:
                break
            self.messages.append(lib.ampis_last_error().decode())
            if need.value < 0:               # exactly what was asked for: no margin to hide a wrong request
                self.h_ws = torch.empty(-need.value, dtype=torch.uint8, pin_memory=True)
                self.grown.append(('host', -need.value))
            else:
                torch.cuda.synchronize()
                self.d_ws = None
                self.d_ws = torch.empty(need.value, dtype=torch.uint8, device='cuda')
                self.grown.append(('device', need.value))
        E.N.check(rc, 'ampis_eval_images_host')
        o['pairs_found'], o['crowded'] = found.value, crowded.value
        return o


def _check_counts(o, ref):
    assert np.array_equal(o['grp_counts'], ref['grp_counts'])
    assert np.array_equal(o['totals'], ref['totals'])


def _cut(d, n_masks):
    """The dataset's images in order, the last one cut (columns first, then rows) to exactly n_masks masks."""
    rows, cols, k = [], [], 0
    for r, c in zip(d.rows, d.cols):
        if k + len(r) + len(c) <= n_masks:
            rows.append(r), cols.append(c)
            k += len(r) + len(c)
            continue
        left = n_masks - k
        r_ = r[:left]
        rows.append(r_), cols.append(c[:left - len(r_)])
        break
    assert sum(map(len, rows)) + sum(map(len, cols)) == n_masks
    return rows, cols


def _kernels_run(torch, fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.key_averages():
        words = e.key.split('(')[0].split('<')[0].split()
        if words:
            names.add(words[-1])
    return res, names


# ---- tests -------------------------------------------------------------------------------------------------------

def test_eval_images_both_modes_equal_the_reference(mods, ds):
    E = mods.engine
    for mode in (E.MODE_IOU, E.MODE_SAT):
        r = E.eval_images(ds.rows, ds.cols, mode)
        assert not r.crowded
        _check(_rows_dict(r), ds.ref[mode], mode)
        # the span against the table API (rle_measure on the same strings, nothing shared with the flat decode)
        masks = [m for rr, cc in ds.imgs for m in list(rr) + list(cc)]
        t = E.table_from_rle(masks, layout=E.LAYOUT_CROP, paint=False)
        assert np.array_equal(r.span.view(np.int32).reshape(-1), t.span[:2 * t.n].cpu().numpy()), mode
    # the cases the dataset is there for did occur
    ref = ds.ref[E.MODE_IOU]
    assert (ref['best_score'] == 1.0).sum() > 50 and (ref['best_score'] == 0.5).sum() >= 1
    assert (ref['area'] == 0).sum() >= 8 and np.isnan(ds.ref[E.MODE_SAT]['best_score']).sum() >= 2
    assert sum(1 for r, c in ds.imgs if not r) >= 2 and sum(1 for r, c in ds.imgs if not c) >= 2


def test_c_entry_all_ways_of_calling_give_identical_bytes(mods, ds):
    E = mods.engine
    ref = ds.ref[E.MODE_IOU]
    e = Entry(mods, 1 << 30, 1 << 26)
    variants = [dict(), dict(contiguous=True), dict(pinned_out=True), dict(pinned_len=True),
                dict(contiguous=True, pinned_out=True, pinned_len=True), dict(blocking=True), dict(no_box=True),
                dict(contiguous=True, pinned_out=True, no_box=True, blocking=True)]
    first = None
    for v in variants:
        o = e.run(ds.rows, ds.cols, E.MODE_IOU, ds.th, **v)
        _check(o, ref, v)
        _check_counts(o, ref)
        assert o['crowded'] == 0 and o['pairs_found'] > 0
        if first is None:
            first = o
            span = o['span']
        for k in ('best_col', 'best_inter', 'best_score', 'area', 'status', 'grp_counts', 'totals', 'bbox', 'span'):
            if o[k] is not None:
                assert o[k].tobytes() == first[k].tobytes(), (v, k)
        assert o['pairs_found'] == first['pairs_found']
    assert not e.grown
    # satellite mode through the C entry as well
    o = e.run(ds.rows, ds.cols, E.MODE_SAT, pinned_out=True, contiguous=True)
    _check(o, ds.ref[E.MODE_SAT], 'sat')
    r = E.eval_images(ds.rows, ds.cols, E.MODE_IOU)
    assert np.array_equal(span, r.span)


@pytest.mark.parametrize('n_masks', [HOST_FILL_MAX, HOST_FILL_MAX + 1])
def test_host_filled_and_device_expanded_bookkeeping(mods, ds, n_masks):
    """Up to 16,384 masks the host fills the per-mask arrays; from 16,385 on expand_images_kernel and a scan do, the
    string lengths are uploaded from where they are when pinned and the results land in pinned outputs directly."""
    E = mods.engine
    rows, cols = _cut(ds, n_masks)
    ref = D.dataset(rows, cols, E.MODE_IOU, ds.th)
    ref_sat = D.dataset(rows, cols, E.MODE_SAT)
    e = Entry(mods, 1 << 30, 1 << 26)
    device_side = n_masks > HOST_FILL_MAX
    expanded = []
    for v in (dict(), dict(pinned_out=True, pinned_len=True), dict(contiguous=True, pinned_out=True)):
        o, names = _kernels_run(mods.torch, lambda: e.run(rows, cols, E.MODE_IOU, ds.th, **v))
        expanded.append('expand_images_kernel' in names)
        _check(o, ref, v)
        _check_counts(o, ref)
        o = e.run(rows, cols, E.MODE_SAT, **v)
        _check(o, ref_sat, v)
    # the results above are the reference's on either side; which side ran is checked last
    assert expanded == [device_side] * 3, expanded


def test_enospc_protocol_and_workspace_reuse(mods, ds):
    """From 4 KB workspaces grown exactly as asked, then the grown workspaces reused for a smaller call, a crowded
    call and a larger one: nothing (arena cursor, totals, counts, crowd flag) carries over from one call to the next."""
    E = mods.engine
    ref = ds.ref[E.MODE_IOU]
    e = Entry(mods)
    o = e.run(ds.rows, ds.cols, E.MODE_IOU, ds.th, crowd_frac=E.CROWD_PAIR_FRACTION)
    assert {k for k, _ in e.grown} == {'host', 'device'} and len(e.grown) <= 6, e.grown
    _check(o, ref, 'grown')
    _check_counts(o, ref)
    assert o['crowded'] == 0
    n_grown = len(e.grown)
    sub = slice(0, 10)
    sub_ref = D.dataset(ds.rows[sub], ds.cols[sub], E.MODE_IOU, ds.th)
    o = e.run(ds.rows[sub], ds.cols[sub], E.MODE_IOU, ds.th, pinned_out=True)
    assert len(e.grown) == n_grown
    _check(o, sub_ref, 'smaller')
    _check_counts(o, sub_ref)
    # a crowded call: the flag is raised, the intersections are skipped, the measurements are valid
    crowd = [i for i, (r, c) in enumerate(ds.imgs) if len(r) == 512 and len(c) == 512]
    assert len(crowd) == 1
    rr, cc = [ds.rows[crowd[0]]], [ds.cols[crowd[0]]]
    o = e.run(rr, cc, E.MODE_IOU, ds.th, crowd_frac=0.1)                # a fifth of its pairs have overlapping boxes
    assert o['crowded'] == 1 and o['pairs_found'] > 0.1 * 512 * 512
    assert np.array_equal(o['area'], ds.ref[E.MODE_IOU]['images'][crowd[0]]['area'])
    # a larger call than the first: the dataset and the diagonal images once more
    big_r, big_c = ds.rows + [r for r, _ in ds.diag], ds.cols + [c for _, c in ds.diag]
    big_ref = dict(ref)
    extra = D.dataset([r for r, _ in ds.diag], [c for _, c in ds.diag], E.MODE_IOU, ds.th)
    for k in ('best_col', 'best_inter', 'best_score', 'area', 'bbox', 'status', 'grp_counts'):
        big_ref[k] = np.concatenate([ref[k], extra[k]])
    big_ref['totals'] = ref['totals'] + extra['totals']
    for v in (dict(crowd_frac=E.CROWD_PAIR_FRACTION), dict(pinned_out=True, pinned_len=True)):
        o = e.run(big_r, big_c, E.MODE_IOU, ds.th, **v)
        assert o['crowded'] == 0
        _check(o, big_ref, v)
        _check_counts(o, big_ref)
    o = e.run(ds.rows[sub], ds.cols[sub], E.MODE_IOU, ds.th)
    _check_counts(o, sub_ref)


def test_grid_entry_list_of_frames_with_diagonals(mods, ds):
    """1024 x 1024 frames of 500 columns, 14 of them thin lines across the frame: each line registers in all
    32 x 32 grid cells, more entries than 16 per column + 4,096 per image.  The entries are measured and the call
    asks for a larger workspace (AMPIS_ENOSPC); every function on top of the entry gives the reference's results."""
    E, A, Dist = mods.engine, mods.analyze, mods.distributed
    rows, cols = [r for r, _ in ds.diag], [c for _, c in ds.diag]
    base = 16 * sum(map(len, cols)) + 4096 * len(cols)
    e = Entry(mods, 1 << 22, 1 << 24)
    ref = D.dataset(rows, cols, E.MODE_IOU, ds.th)
    o = e.run(rows, cols, E.MODE_IOU, ds.th)
    entries = [int(x) for m in e.messages for x in re.findall(r'grid entries: (\d+)', m)]
    assert entries and max(entries) > base, (e.messages, base)
    _check(o, ref, 'diagonals')
    _check_counts(o, ref)
    for mode in (E.MODE_IOU, E.MODE_SAT):
        sref = D.dataset(rows, cols, mode)
        _check(_rows_dict(E.eval_images(rows, cols, mode)), sref, mode)
        for g in range(len(rows)):                      # the one-image entry has the same grid
            one = E.eval_image(rows[g], cols[g], mode)
            _check(dict(best_col=one.best_col, best_inter=one.best_inter, best_score=one.best_score, area=one.area,
                        bbox=one.bbox, status=np.zeros(len(one.area), np.int32)), sref['images'][g], (mode, g))
    _check_drop_in_and_sharded(mods, rows, cols, ds.th)


def test_drop_in_and_sharded_functions_on_the_dataset(mods, ds):
    _check_drop_in_and_sharded(mods, ds.rows, ds.cols, ds.th, ds.ref)


def _det_seg_want(img, th):
    G = img['n_rows']
    matched = img['best_score'] > th
    gi = np.flatnonzero(matched)
    pi = img['best_col'][gi].astype(np.int64)
    fp = np.setdiff1d(np.arange(img['n_cols']), pi)
    inter = img['best_inter'][gi].astype(np.int64)
    a_g, a_p = img['area'][gi].astype(np.int64), img['area'][G + pi].astype(np.int64)
    with np.errstate(invalid='ignore', divide='ignore'):
        return {'det_precision': len(gi) / (len(gi) + len(fp)), 'det_recall': len(gi) / G,
                'seg_precision': inter / a_p, 'seg_recall': inter / a_g, 'det_tp': np.stack([gi, pi], axis=1),
                'det_fn': np.flatnonzero(~matched), 'det_fp': fp, 'seg_tp': inter, 'seg_fn': a_g - inter,
                'seg_fp': a_p - inter, 'det_tp_iou': img['best_score'][gi]}


def _check_drop_in_and_sharded(mods, rows, cols, th, refs=None):
    import torch.distributed as dist
    A, Dist, E = mods.analyze, mods.distributed, mods.engine
    ref = refs[E.MODE_IOU] if refs else D.dataset(rows, cols, E.MODE_IOU, th)
    sat = refs[E.MODE_SAT] if refs else D.dataset(rows, cols, E.MODE_SAT)
    both = [g for g in range(len(rows)) if rows[g] and cols[g]]
    for t in (0.5, th[2]):
        got = A.det_seg_scores_batch([rows[g] for g in both], [cols[g] for g in both], t)
        for g, res in zip(both, got):
            want = _det_seg_want(ref['images'][g], t)
            for k in want:
                a_, b_ = np.asarray(res[k]), np.asarray(want[k])
                if k == 'det_tp':
                    a_, b_ = a_.reshape(-1, 2), b_.reshape(-1, 2)
                assert _same_f64(a_, b_) if a_.dtype.kind == 'f' else np.array_equal(a_, b_), (g, t, k)
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=0, world_size=1)
    try:
        r = Dist.evaluate_sharded(rows, cols, th)
        assert np.array_equal(r['per_image'], ref['grp_counts']) and np.array_equal(r['totals'], ref['totals'])
        s_ = Dist.satellites_sharded(cols, rows, 0.5, 64)
        matched = [img['best_score'] > 0.5 for img in sat['images']]
        owners = [np.unique(img['best_col'][m], return_counts=True)[1] for img, m in zip(sat['images'], matched)]
        per = np.concatenate(owners) if owners else np.zeros(0, np.int64)
        assert s_['n_images'] == len(rows) and s_['n_particles'] == sum(map(len, cols))
        assert s_['n_satellites'] == sum(int(m.sum()) for m in matched)
        assert s_['n_satellites_unmatched'] == sum(map(len, rows)) - s_['n_satellites']
        assert s_['n_satellited_particles'] == len(per)
        assert np.array_equal(s_['spp_hist'], np.bincount(np.minimum(per, 63), minlength=64))
    finally:
        dist.destroy_process_group()
