"""Interval windows of the crop step (rle_flat.cu with intervals on; intersect_pairs.cu): a column-convex mask is
stored as one (first row, last row) word per box column and the pairs join intersects such windows in closed form.
Everything the step produces must be the same bit for bit with the form on and off -- on the synthetic configs, and on
hand-made masks that must stay bitmaps or mix the two forms in one pair -- and equal to the oracle.  The C entry
points decode to intervals on their join branches.  A table holding interval windows cannot reach a bitmap reader."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def mods():
    import torch
    assert torch.cuda.is_available(), 'these tests need the B200'
    from ampis_b200 import batch, engine
    from oracle import cocomask as rle

    class M:
        pass
    m = M()
    m.torch, m.batch, m.engine, m.rle = torch, batch, engine, rle
    return m


# ---- running the step ---------------------------------------------------------------------------------------------

def _step(mods, host, intervals, kernel='grid', sparse=None, dense=True):
    """One Pipeline step of a HostCSR on the crop layout; every output as host arrays."""
    B, E, torch = mods.batch, mods.engine, mods.torch
    dev = B.DeviceBatch(host, dense=dense)
    arena = torch.empty(4 * max(B.arena_chunks_needed(dev, E.LAYOUT_CROP), 1), dtype=torch.int32, device='cuda')
    p = B.Pipeline(dev, E.LAYOUT_CROP, arena, kernel=kernel, intervals=intervals, sparse_capacity=sparse)
    assert p.pairs is not None, 'the pairs join'
    p.launch()
    torch.cuda.synchronize()
    t = p.table
    t.check()
    assert t.intervals == intervals
    n, g = t.n, dev.groups
    o = {}
    o['area'] = t.area[:n].cpu().numpy()
    o['bbox'] = t.bbox[:4 * n].cpu().numpy()
    o['status'] = t.status[:n].cpu().numpy()
    o['best_col'] = p.rows.best_col[:g.n_rows].cpu().numpy()
    o['best_inter'] = p.rows.best_inter[:g.n_rows].cpu().numpy()
    o['best_score'] = p.rows.best_score[:g.n_rows].cpu().numpy()
    if dense:
        o['imat'] = p.rows.imat[:g.imat_size].cpu().numpy()
    npairs = int(p.pairs.count.item())
    assert npairs <= p.pairs.capacity
    ab = p.pairs.ab[:2 * npairs].cpu().numpy().reshape(-1, 2).astype(np.int64)
    inter = p.pairs.inter[:npairs].cpu().numpy()
    order = np.lexsort((ab[:, 1], ab[:, 0]))            # the order of the list depends on the warps' timing
    o['pair_ab'], o['pair_inter'] = ab[order], inter[order]
    if dev.mode == E.MODE_IOU:
        o['counts'] = p.counts.cpu().numpy()
        o['totals'] = p.totals.cpu().numpy()
    else:
        o['counts'] = p.counts.cpu().numpy()
        o['spp_hist'] = p.spp_hist.cpu().numpy()
    if sparse is not None:
        o['sparse'] = [x.cpu().numpy() for x in p.sparse.triplets()]
    o['forms'] = t.reg[:2 * n].cpu().numpy().reshape(-1, 2)[:, 0] & 1      # AMPIS_WIN_INTERVALS
    return o


def _same(a, b, tag):
    assert a.keys() == b.keys()
    for k in a:
        if k == 'forms':
            continue
        if k == 'sparse':
            for x, y in zip(a[k], b[k]):
                assert np.array_equal(x, y), (tag, k)
        else:
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), (tag, k)   # floats bit for bit


def _both_forms(mods, host, tag, **kw):
    on, off = _step(mods, host, True, **kw), _step(mods, host, False, **kw)
    assert not off['forms'].any(), tag
    _same(on, off, tag)
    return on


@pytest.mark.parametrize('cfg,n_img,kw', [
    ('c1_powder_example', 1, {}),
    ('c2_powder_batch', 200, dict(kernel='rows')),
    ('c3_satellites', 4, {}),
    ('dense_overlap', 2, {}),
])
def test_same_results_with_and_without_intervals(mods, cfg, n_img, kw):
    host = mods.batch.synth(cfg, n_img, 4242)
    on = _both_forms(mods, host, cfg, **kw)
    assert on['forms'].mean() > 0.9, (cfg, on['forms'].mean())      # the synthetic blobs are column-convex


def test_native_c4_image_with_sparse_output(mods):
    host = mods.batch.synth('c4_spheroidite', 1, 77)
    on = _both_forms(mods, host, 'c4', sparse=400000)
    assert on['forms'].mean() > 0.9
    assert len(on['sparse'][0]) == int((on['imat'] > 0).sum())


# ---- masks that must stay bitmaps, and pairs of mixed forms ---------------------------------------------------------

def _disc(h, w, cy, cx, r):
    y, x = np.ogrid[:h, :w]
    return (y - cy) ** 2 + (x - cx) ** 2 <= r * r


def _mixed_stack(h, w, rng):
    """rows, cols: bool[k, h, w] with interval masks (blobs, lines, a pixel, a full-height column, two blobs with gap
    columns), bitmaps (ring, C shape, full-height bars whose runs cross column ends), empty masks, nested boxes and
    boxes that touch at one column."""
    cy, cx = h // 2, w // 2
    m = []
    m.append(_disc(h, w, cy, cx, 12))                                           # interval
    m.append(_disc(h, w, cy, cx, 12) & ~_disc(h, w, cy, cx, 6))                 # ring: bitmap
    c = _disc(h, w, cy, cx + 4, 10) & ~_disc(h, w, cy, cx + 10, 6)
    m.append(c)                                                                 # C shape: bitmap
    two = _disc(h, w, cy, cx - 14, 5) | _disc(h, w, cy + 3, cx + 14, 6)
    m.append(two)                                                               # gap columns inside the box
    bar = np.zeros((h, w), bool); bar[:, cx - 3:cx + 2] = True
    m.append(bar)                                                               # top to bottom: runs cross columns
    col = np.zeros((h, w), bool); col[:, cx + 5] = True
    m.append(col)                                                               # one full-height column: interval
    px = np.zeros((h, w), bool); px[cy, cx] = True
    m.append(px)
    row = np.zeros((h, w), bool); row[cy + 1, cx - 20:cx + 20] = True
    m.append(row)                                                               # 1 row
    vcol = np.zeros((h, w), bool); vcol[cy - 9:cy + 9, cx - 1] = True
    m.append(vcol)                                                              # 1 column
    m.append(np.zeros((h, w), bool))                                            # empty
    m.append(_disc(h, w, cy, cx, 3))                                            # nested in the disc's box
    t1 = np.zeros((h, w), bool); t1[cy - 4:cy + 4, cx + 12:cx + 18] = True
    m.append(t1)                                                                # touches the disc at column cx + 12
    lo = np.zeros((h, w), bool); lo[h - 5:, 2:9] = True
    m.append(lo)                                                                # last rows
    noise = rng.random((h, w)) < 0.3
    m.append(noise & _disc(h, w, cy, cx, 15))                                   # several runs per column
    rows = np.stack(m)
    # columns: the same kinds shifted by a pixel or two, so that every pair of forms overlaps
    cols = np.stack([np.roll(np.roll(x, 1, axis=0), int(rng.integers(-2, 3)), axis=1) for x in m] + [m[0], m[3], m[1]])
    return rows, cols


def _host(mods, stacks, n_rows, h, w):
    rle, B = mods.rle, mods.batch
    cnts = []
    for s in stacks:
        for x in s:
            cnts.append(rle.counts_from_string(rle.encode(np.asfortranarray(x.astype(np.uint8)))['counts']))
    lens = np.array([len(c) for c in cnts], np.int32)
    off = np.zeros(len(cnts), np.int64)
    off[1:] = np.cumsum(lens[:-1])
    cfg = dict(h=h, w=w, n_rows=n_rows, n_cols=stacks[0].shape[0] - n_rows, kind=0, mode=mods.engine.MODE_IOU)
    return B.HostCSR(cfg, len(stacks), np.concatenate(cnts).astype(np.uint32), off, lens)


def _dense_ref(rows, cols):
    # intersections as a product of the flattened masks, a million pixels at a time (float32 sums of 0 / 1 are exact
    # below 2^24): frames of 70,000 rows stay at ~130 MB
    a, b = rows.reshape(len(rows), -1), cols.reshape(len(cols), -1)
    I = np.zeros((len(rows), len(cols)), np.int64)
    for k in range(0, a.shape[1], 1 << 20):
        I += (a[:, k:k + (1 << 20)].astype(np.float32) @ b[:, k:k + (1 << 20)].astype(np.float32).T).astype(np.int64)
    ar, ac = a.sum(axis=1).astype(np.int64), b.sum(axis=1).astype(np.int64)
    with np.errstate(invalid='ignore', divide='ignore'):
        iou = np.where(I > 0, I / (ar[:, None] + ac[None, :] - I), 0.0)
    best = np.where(iou.max(axis=1) > 0, iou.argmax(axis=1), -1)
    return I, iou, best, np.r_[ar, ac]


def _check_vs_oracle(mods, o, stacks, n_rows, tag):
    rle = mods.rle
    G = n_rows
    P = stacks[0].shape[0] - G
    imat = o['imat'].reshape(len(stacks), G, P)
    for g, s in enumerate(stacks):
        I, iou, best, area = _dense_ref(s[:G], s[G:])
        assert np.array_equal(imat[g], I), (tag, g)
        assert np.array_equal(o['best_col'][g * G:(g + 1) * G], best), (tag, g)
        assert np.array_equal(o['best_score'][g * G:(g + 1) * G], iou.max(axis=1)), (tag, g)
        assert np.array_equal(o['area'][g * (G + P):(g + 1) * (G + P)], area), (tag, g)
        enc = [rle.encode(np.asfortranarray(x.astype(np.uint8))) for x in s]
        for i, j in np.argwhere(I > 0)[::7]:
            assert I[i, j] == int(rle.merge_area(enc[i], enc[G + j])), (tag, g, i, j)


def _pair_forms(o):
    f = o['forms']
    return {(int(f[a]), int(f[b])) for a, b in o['pair_ab']}


@pytest.mark.parametrize('h,w', [(96, 120), (65535, 40), (65536, 40), (70000, 40)])
def test_masks_that_stay_bitmaps_and_mixed_pairs(mods, h, w):
    rng = np.random.default_rng(h)
    hh = min(h, 96)
    rows, cols = _mixed_stack(hh, w, rng)
    if h > hh:   # the same masks at the bottom of a tall frame, plus one at the very last row
        pad = lambda s: np.concatenate([np.zeros((s.shape[0], h - hh, w), bool), s], axis=1)
        rows, cols = pad(rows), pad(cols)
        last = np.zeros((1, h, w), bool); last[0, h - 1, 3:7] = True
        rows, cols = np.concatenate([rows, last]), np.concatenate([cols, last])
    stacks = [np.concatenate([rows, cols])]
    host = _host(mods, stacks, len(rows), h, w)
    on = _both_forms(mods, host, (h, w))
    _check_vs_oracle(mods, on, stacks, len(rows), (h, w))
    forms = on['forms']
    if h <= 65536:
        assert forms[0] == 1 and forms[1] == 0 and forms[2] == 0 and forms[5] == 1
        assert forms[9] == 0                                                     # empty: bitmap
        if h == hh:
            assert forms[4] == 0                                                 # full-height bar: runs cross columns
        assert _pair_forms(on) == {(0, 0), (0, 1), (1, 0), (1, 1)}
    else:
        assert not forms.any()                                                   # taller than 65,536 rows: fallback


def test_window_wider_than_the_tile_stays_a_bitmap(mods):
    """A column-convex mask whose interval window (700 words) is larger than the tile goes to the fallback kernel and
    is a bitmap there: two bands per column, so its bitmap takes twice the chunks its interval window would."""
    h, w = 64, 700
    band = np.zeros((h, w), bool); band[20:40, :] = True
    d = _disc(h, w, 30, 300, 8)
    rows = np.stack([band, d])
    cols = np.stack([d, band, _disc(h, w, 36, 650, 6)])
    stacks = [np.concatenate([rows, cols])]
    on = _both_forms(mods, _host(mods, stacks, 2, h, w), 'wide')
    _check_vs_oracle(mods, on, stacks, 2, 'wide')
    assert on['forms'].tolist() == [0, 1, 1, 0, 1]


def test_interval_against_bitmap_deeper_than_four_bands(mods):
    """Interval x bitmap overlaps of nine bands: the join splits a column into items of four bands (w0 = 0, 4, 8)."""
    h, w = 320, 64
    y, x = np.ogrid[:h, :w]
    ell = lambda cy, cx, ry, rx: ((y - cy) / ry) ** 2 + ((x - cx) / rx) ** 2 <= 1.0
    rng = np.random.default_rng(3)
    tall = ell(160, 32, 140, 20)                                                # interval
    ring = tall & ~ell(160, 32, 60, 8)                                          # two runs per column: bitmap
    noisy = tall & (rng.random((h, w)) < 0.6)                                   # bitmap
    rows = np.stack([tall, ring, noisy])
    cols = np.stack([np.roll(tall, 3, axis=0), np.roll(ring, -2, axis=1), np.roll(noisy, 1, axis=1), tall])
    stacks = [np.concatenate([rows, cols])]
    on = _both_forms(mods, _host(mods, stacks, 3, h, w), 'deep')
    _check_vs_oracle(mods, on, stacks, 3, 'deep')
    assert on['forms'].tolist() == [1, 0, 0, 1, 0, 0, 1]
    assert _pair_forms(on) == {(0, 0), (0, 1), (1, 0), (1, 1)}


# ---- the C entry points ---------------------------------------------------------------------------------------------

def _rle_dicts(mods, s):
    rle = mods.rle
    h, w = s.shape[1:]
    return [{'size': [h, w], 'counts': rle.encode(np.asfortranarray(x.astype(np.uint8)))['counts']} for x in s]


@pytest.mark.parametrize('n_cols', [40, 90])
def test_c_entries_on_mixed_images(mods, n_cols):
    """ampis_eval_image_host: the pairs join (>= 64 columns, interval windows) and the column scan (fewer, bitmaps);
    ampis_eval_images_host: always the join."""
    E = mods.engine
    h, w = 96, 120
    rng = np.random.default_rng(n_cols)
    rows, cols = _mixed_stack(h, w, rng)
    extra = [np.roll(_disc(h, w, int(rng.integers(10, 86)), int(rng.integers(10, 110)), int(rng.integers(2, 9))),
                     0, axis=0) for _ in range(n_cols - len(cols))]
    cols = np.concatenate([cols, np.stack(extra)])[:n_cols]
    I, iou, best, area = _dense_ref(rows, cols)
    rr, cc = _rle_dicts(mods, rows), _rle_dicts(mods, cols)
    one = E.eval_image(rr, cc, E.MODE_IOU, dense_iou=True)
    many = E.eval_images([rr], [cc], E.MODE_IOU)
    for r, tag in ((one, 'image'), (many, 'images')):
        assert np.array_equal(r.best_col.astype(np.int64), best), tag
        assert np.array_equal(r.best_score, iou.max(axis=1)), tag
        got_inter = r.best_inter.astype(np.int64)
        want_inter = np.where(best >= 0, I[np.arange(len(rows)), np.maximum(best, 0)], 0)
        assert np.array_equal(got_inter, want_inter), tag
        assert np.array_equal(r.area.astype(np.int64), area), tag
    assert np.array_equal(one.iou, iou)


def _probe_rles():
    """One 512 x 512 image of large discs with few overlaps: 6 rows, 70 columns (the grid branch of the one-image
    entry), whose bitmap windows take about four times the arena of their interval windows."""
    from oracle import cocomask as rle
    h = w = 512
    rng = np.random.default_rng(11)
    enc = lambda m: {'size': [h, w], 'counts': rle.encode(np.asfortranarray(m.astype(np.uint8)))['counts']}
    disc = lambda: _disc(h, w, int(rng.integers(45, 467)), int(rng.integers(45, 467)), int(rng.integers(30, 41)))
    return [enc(disc()) for _ in range(6)], [enc(disc()) for _ in range(70)]


def _fits(entry, size):
    """True when ampis_eval_image_host (entry 'image') or ampis_eval_images_host ('images') evaluates the probe image
    in a device workspace of `size` bytes without asking for more."""
    import torch
    from ampis_b200 import engine as E
    rr, cc = _probe_rles()
    pair = [torch.empty(size, dtype=torch.uint8, device='cuda'), torch.empty(64 << 20, dtype=torch.uint8, pin_memory=True)]
    mine, old = pair[0], E._workspaces
    E._workspaces = lambda device: pair
    try:
        if entry == 'image':
            E.eval_image(rr, cc, E.MODE_IOU)
        else:
            E.eval_images([rr], [cc], E.MODE_IOU)
    finally:
        E._workspaces = old
    return pair[0] is mine                       # the call grew the workspace when it did not fit


@pytest.mark.parametrize('entry', ['image', 'images'])
def test_c_entries_decode_interval_windows(mods, entry):
    """The arena a C entry uses is the one its decode filled.  The smallest workspace that holds the probe image here
    is too small where every window is a bitmap (AMPIS_PI_FLAT=0, where the join does not read intervals)."""
    if not mods.engine.pairs_read_intervals():
        pytest.skip('the join reads bitmaps only under this AMPIS_PI_FLAT')
    lo, hi = 4096, 64 << 20
    assert not _fits(entry, lo) and _fits(entry, hi)
    while hi - lo > 256:
        mid = (lo + hi) // 2
        lo, hi = (lo, mid) if _fits(entry, mid) else (mid, hi)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, '-c', 'from tests.test_crop_intervals_gpu import _fits; '
                          'print(_fits(%r, %d))' % (entry, hi)], cwd=root, capture_output=True, text=True,
                         env=dict(os.environ, AMPIS_PI_FLAT='0'), timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.split()[-1] == 'False', (hi, out.stdout)


# ---- no bitmap reader gets an interval table --------------------------------------------------------------------------

def test_bitmap_readers_refuse_an_interval_table(mods):
    E, B, torch = mods.engine, mods.batch, mods.torch
    host = B.synth('c1_powder_example', 1, 5)
    dev = B.DeviceBatch(host, dense=True)
    arena = torch.empty(4 * B.arena_chunks_needed(dev, E.LAYOUT_CROP), dtype=torch.int32, device='cuda')
    p = B.Pipeline(dev, E.LAYOUT_CROP, arena, kernel='grid')
    assert p.intervals
    p.launch()
    t = p.table
    assert t.intervals
    with pytest.raises(ValueError, match='interval windows'):
        E.intersect_rows(t, dev.groups, dev.mode, grid='scan')             # the column scan of the crop kernel
    with pytest.raises(ValueError, match='interval windows'):
        E.unpack_bool(t, [0, 1], host.h, host.w)
    # a Pipeline whose table goes elsewhere keeps bitmaps; so does measure_paint by default
    assert not B.Pipeline(dev, E.LAYOUT_CROP, arena, kernel='scan').intervals
    t.measure_paint(arena)
    assert not t.intervals
    torch.cuda.synchronize()
