"""The annotation kernels on the B200 -- union-find labelling and per-label boxes and runs (label.cu), rleFrPoly and
polygon2mask (poly.cu), boundary distances (edge.cu) and the pixel-class projection of seg_perf_iset -- through the
public API, against the exact references of tests/_annot_ref.py and the oracle, at frame scale and at the kernels'
limits.  Everything is compared exactly: RLE strings, boxes and instance order equal; float64 distances equal bit for
bit and in the same order.

Covered: random binary images around the 8-connected percolation point (giant components merged across many
blocks), pixel counts that are no multiple of 256, 1 x n and n x 1 frames, diagonal-only connectivity, 262,144
labels, long rings and a spiral, full-height components whose runs cross column ends, label values up to 2^24 - 1;
polygons of 4096 vertices and of exactly 8192 crossings, and one past each limit, polygons needing the host's second
launch, polygons outside the frame; candidate tiles of 1023, 1024 and 1025 boundary pixels, windows exactly 32767
wide, a 32767 x 32767 frame.  Every input comes from a fixed seed."""
import numpy as np
import pytest

from tests import _annot_ref as A
from tests.test_annot_ref_oracle import _polys

pytestmark = pytest.mark.gpu

EDGE_WORK_LIMIT = 10 ** 9          # queries x boundary candidates of one pair: one CTA does all of it


@pytest.fixture(scope='module')
def M():
    import torch
    assert torch.cuda.is_available(), 'these tests need the B200'
    from ampis_b200 import analyze, data_utils, engine, structures
    from ampis_b200.containers import PolygonMasks
    from oracle import ampis_ref as R
    from oracle import cocomask as rle

    class _M:
        pass
    m = _M()
    m.torch, m.analyze, m.data_utils, m.engine, m.structures, m.PolygonMasks, m.R, m.rle = \
        torch, analyze, data_utils, engine, structures, PolygonMasks, R, rle
    return m


# ---- labelling ----------------------------------------------------------------------------------------------------

def _check_labels(M, img, binary):
    """engine.label_image_to_instances == reference: strings, boxes and order.  Returns the number of instances."""
    h, w = img.shape
    rles, bb = M.engine.label_image_to_instances(img, binary=binary)
    boxes, counts = A.label_instances(img, binary)
    assert len(rles) == len(counts) == len(bb)
    assert all(r['size'] == [h, w] for r in rles)
    assert np.array_equal(np.asarray(bb, np.int64).reshape(-1, 4), boxes)
    assert [r['counts'] for r in rles] == [M.rle.string_from_counts(c) for c in counts]
    return len(counts)


@pytest.mark.parametrize('density', [0.3, 0.41, 0.6])
def test_labels_of_random_images_near_percolation(M, density):
    rng = np.random.default_rng(int(density * 100))
    img = rng.random((2048, 2048)) < density
    n = _check_labels(M, img, True)
    sizes = np.bincount(A.dense_labels(img, True)[0].ravel())[1:]
    assert n > 1000 or density > 0.5
    assert density < 0.4 or sizes.max() > 10 ** 5          # a giant component merged across thousands of blocks


@pytest.mark.parametrize('h,w', [(1000, 3001), (1, 100003), (100003, 1)])
def test_labels_of_odd_frames(M, h, w):
    rng = np.random.default_rng(h + w)
    img = rng.random((h, w)) < 0.45
    img.flat[0] = img.flat[-1] = True
    assert (h * w) % 256
    _check_labels(M, img, True)
    _check_labels(M, img.astype(np.int32) * (1 + (np.arange(h * w).reshape(h, w) % 3)), False)


def test_labels_of_checkerboard_grid_rings_and_spiral(M):
    cb = np.add.outer(np.arange(1024), np.arange(1023)) % 2 == 0          # diagonal neighbours only
    assert _check_labels(M, cb, True) == 1
    grid = np.zeros((1024, 1024), bool)
    grid[::2, ::2] = True                                                  # one label per pixel
    assert _check_labels(M, grid, True) == 512 * 512
    n = 1024
    cheb = np.maximum(np.abs(np.arange(n)[:, None] - n // 2), np.abs(np.arange(n)[None, :] - n // 2))
    rings = cheb % 2 == 0                                                  # one-pixel square rings, one-pixel gaps
    assert _check_labels(M, rings, True) == n // 4 + 1
    spiral = np.zeros((n, n), bool)
    t, b, lo, r = 0, n - 1, 0, n - 1
    while t <= b and lo <= r:
        spiral[t, lo:r + 1] = True
        spiral[t:b + 1, r] = True
        spiral[b, lo:r + 1] = True
        if t + 2 <= b:
            spiral[t + 2:b + 1, lo] = True
            spiral[t + 2, lo:lo + 2] = True
        t, b, lo, r = t + 2, b - 2, lo + 2, r - 2
    assert _check_labels(M, spiral, True) == 1


def test_labels_whose_runs_cross_column_ends(M):
    """Components spanning the full height, with and without the full width: the previous pixel is carried from the
    bottom of one column to the top of the next only then (the gap rule of label_rle_kernel)."""
    h, w = 301, 257
    img = np.zeros((h, w), bool)
    img[:, 3:6] = True                      # full height, not full width: no run boundary between its columns
    img[:, 10] = img[h - 1, 10:13] = img[:, 12] = True      # a U: column 11 holds only the last row
    img[5:h - 5, 20] = True                 # not full height
    img[:, 30] = True
    img[0, 31] = True                       # the last row of column 30 runs into the first row of column 31
    assert _check_labels(M, img, True) == 4
    ring = np.zeros((h, w), bool)           # touches all four borders: full height and full width
    ring[0, :] = ring[-1, :] = ring[:, 0] = ring[:, -1] = True
    ring[100:200, 100:150] = True
    assert _check_labels(M, ring, True) == 2
    rng = np.random.default_rng(5)
    noisy = ring | (rng.random((h, w)) < 0.2)
    _check_labels(M, noisy, True)
    assert _check_labels(M, np.zeros((h, w), bool), True) == 0
    assert _check_labels(M, np.ones((h, w), bool), True) == 1
    lab = np.where(img, 7, 0) + np.where(ring, 9, 0)
    _check_labels(M, lab, False)


def test_label_values_up_to_2_pow_24(M):
    rng = np.random.default_rng(24)
    vals = np.unique(np.r_[rng.integers(1, 1 << 24, 3000), (1 << 24) - 1, 1, 2])
    blocks = rng.choice(vals, (150, 110))
    img = np.kron(blocks, np.ones((10, 10), np.int64))[:1499, :1093]          # runs over several rows and columns
    img[::97, :] = 0
    img[:, 500:520] = vals[-1]                                               # one value in disconnected pieces
    img[700:720, :] = vals[-1]
    n = _check_labels(M, img, False)
    assert n == len(np.unique(img)) - 1
    no_zero = img.copy()
    no_zero[no_zero == 0] = 12345
    assert _check_labels(M, no_zero, False) == len(np.unique(no_zero))
    with pytest.raises(ValueError):
        M.engine.label_image_to_instances(np.full((4, 5), 1 << 24, np.int64), binary=False)


def test_get_ddicts_binary_png_round_trip(M, tmp_path, monkeypatch):
    from PIL import Image
    rng = np.random.default_rng(2048)
    img = rng.random((2048, 2048)) < 0.41
    monkeypatch.chdir(tmp_path)
    for d in ('im', 'ann'):
        (tmp_path / d).mkdir()
        Image.fromarray(img.astype(np.uint8) * 255).save(str(tmp_path / d / 'a.png'))
    dd = M.data_utils.get_ddicts('binary', 'im', 'ann')
    assert len(dd) == 1 and (dd[0]['height'], dd[0]['width']) == (2048, 2048)
    boxes, counts = A.label_instances(img, True)
    ann = dd[0]['annotations']
    assert dd[0]['num_instances'] == len(ann) == len(counts)
    assert [a['segmentation']['counts'] for a in ann] == [M.rle.string_from_counts(c) for c in counts]
    got = np.stack([a['bbox'] for a in ann])
    assert got.dtype == np.float64 and np.array_equal(got, boxes.astype(np.float64))   # extract_boxes' form


# ---- polygons -----------------------------------------------------------------------------------------------------

def _poly_rle(M, polys, h, w):
    return [r['counts'] for r in M.structures.masks_to_rle(M.PolygonMasks([[np.asarray(p)] for p in polys]), (h, w))]


def _oracle_rle(M, polys, h, w):
    return [M.rle.frPyObjects([list(np.asarray(p, np.float64))], h, w)[0]['counts'] for p in polys]


def _star(n_vert, cx, cy, r, amp):
    ang = np.arange(n_vert) * (2 * np.pi / n_vert)
    rad = r + amp * (np.arange(n_vert) % 2)
    return np.stack([cx + rad * np.cos(ang), cy + rad * np.sin(ang)], 1).ravel()


def _comb_up(n_teeth, x0, y_base, y_tip, extra=0):
    """Teeth one column wide and one apart pointing up from a bar: 2 + 4·n_teeth + extra vertices."""
    right = x0 + 2 * n_teeth
    pts = [(x0, y_base + 3)] + [(x0 + (right - x0) * (i + 1) / (extra + 1), y_base + 3) for i in range(extra)]
    pts += [(right, y_base + 3)]
    for i in range(n_teeth - 1, -1, -1):
        a = x0 + 2 * i
        pts += [(a + 1, y_base), (a + 1, y_tip), (a, y_tip), (a, y_base)]
    return np.asarray(pts, np.float64).ravel()


def _comb_side(lengths, x_spine, y0, spine_w, leftwards=False, spine_bottom=None):
    """Teeth two rows high, two apart, off a vertical spine; integer vertices, so every unit of a horizontal edge is
    one crossing: 2·Σlengths + 2·spine_w crossings inside the frame."""
    s = -1 if leftwards else 1
    xa, xb = (x_spine + spine_w, x_spine) if leftwards else (x_spine, x_spine + spine_w)
    bottom = y0 + 4 * len(lengths) + 1 if spine_bottom is None else spine_bottom
    pts = [(xa, y0)]
    for i, L in enumerate(lengths):
        top = y0 + 1 + 4 * i
        pts += [(xb, top), (xb + s * L, top), (xb + s * L, top + 2), (xb, top + 2)]
    pts += [(xb, bottom), (xa, bottom)]
    return np.asarray(pts, np.float64).ravel()


def test_polygons_at_the_vertex_limit(M):
    h, w = 1024, 1536
    star = _star(4096, 768.3, 511.7, 400.0, 1.5)
    assert len(A.poly_crossings(star, h, w)) <= 8192
    comb = _comb_up(1023, 1.0, 1800.0, 40.0, extra=2)
    assert len(comb) == len(star) == 2 * 4096 and len(A.poly_crossings(comb, 2048, 2048)) <= 8192
    assert _poly_rle(M, [star], h, w) == _oracle_rle(M, [star], h, w)
    assert _poly_rle(M, [comb], 2048, 2048) == _oracle_rle(M, [comb], 2048, 2048)
    with pytest.raises(ValueError):
        _poly_rle(M, [_star(4097, 768.3, 511.7, 400.0, 1.5)], h, w)
    with pytest.raises(ValueError):
        _poly_rle(M, [star, _comb_up(1023, 1.0, 1800.0, 40.0, extra=3)], 2048, 2048)


def test_polygons_at_the_crossing_limit(M):
    """Exactly 8192 crossings (per the reference) rasterise; one more is refused.  The odd counts come from a spine
    in the last column reaching below the frame: its crossing at position h·w is dropped."""
    h = w = 2048
    even = _comb_side([1024, 1024, 1023, 1023], 0.0, 10.0, 2.0)
    odd = _comb_side([1024, 1024, 1024, 1023], float(w - 1), 10.0, 1.0, leftwards=True, spine_bottom=h + 7.0)
    over = _comb_side([1024, 1024, 1024, 1024], float(w - 1), 10.0, 1.0, leftwards=True, spine_bottom=h + 7.0)
    assert [len(A.poly_crossings(p, h, w)) for p in (even, odd, over)] == [8192, 8191, 8193]
    want = _oracle_rle(M, [even, odd], h, w)
    assert _poly_rle(M, [even, odd], h, w) == want
    assert [M.rle.string_from_counts(A.poly_counts(p, h, w)) for p in (even, odd)] == want
    with pytest.raises(ValueError):
        _poly_rle(M, [even, over], h, w)


def test_polygons_needing_the_second_launch(M):
    h, w = 1024, 1536
    cap = 2 * (w + 2) + 8
    many = _comb_side([200] * 20, 300.0, 50.0, 3.0)                # every column of the teeth crossed 40 times
    assert len(A.poly_counts(many, h, w)) > cap
    polys = [_star(64, 700.0, 500.0, 300.0, 40.0), many, _comb_side([1500] * 2, 5.0, 900.0, 2.0)]
    assert _poly_rle(M, polys, h, w) == _oracle_rle(M, polys, h, w)


@pytest.mark.parametrize('h,w', [(1024, 1536), (2048, 2048)])
def test_polygons_outside_on_the_edge_and_half_integer(M, h, w):
    rng = np.random.default_rng(h + w)
    polys = _polys(rng, h, w)
    polys += [np.array([-0.5, -0.5, w - 0.5, -0.5, w - 0.5, h - 0.5, -0.5, h - 0.5]),
              np.array([0.0, h / 2, w / 2, 0.0, float(w), h / 2, w / 2, float(h)]),
              np.array([-50.0, -50.0, -10.0, -50.0, -10.0, -10.0]),
              np.array([w - 3.5, h - 3.5, w + 40.0, h - 3.5, w + 40.0, h + 40.0])]
    n_cross = np.array([len(A.poly_crossings(p, h, w)) for p in polys])
    ok = [p for p, n in zip(polys, n_cross) if n <= 8192]
    assert len(ok) > 20
    assert _poly_rle(M, ok, h, w) == _oracle_rle(M, ok, h, w)
    for p in [p for p, n in zip(polys, n_cross) if n > 8192][:2]:
        with pytest.raises(ValueError):
            _poly_rle(M, [p], h, w)


def test_polygon_bitmasks_clipped_by_the_frame(M):
    h, w = 1024, 1536
    rng = np.random.default_rng(1536)
    polys = []
    for cx, cy in [(-60, -40), (w + 50, 300), (700, h + 30), (w - 20, h - 10), (10.5, 500.5), (800, -120)]:
        k = int(rng.integers(150, 320))
        ang = np.sort(rng.uniform(0, 2 * np.pi, k))
        r = rng.uniform(60, 200, k)
        p = np.stack([cx + r * np.cos(ang), cy + r * np.sin(ang)], 1)
        if rng.random() < 0.5:
            p = np.round(p * 2) / 2                               # half-integer vertices: pixel centres on edges
        polys.append(p.ravel())
    got = M.structures.masks_to_bitmask_array(M.PolygonMasks([[p] for p in polys]), (h, w))
    want = M.R.poly2mask(polys, (h, w))
    assert want.sum(axis=(1, 2)).min() > 0
    assert got.dtype == np.bool_ and np.array_equal(got, want)


# ---- boundary distances -------------------------------------------------------------------------------------------

def _tight_box(m):
    rr, cc = np.nonzero(m)
    return [int(rr.min()), int(rr.max()) + 1, int(cc.min()), int(cc.max()) + 1]


def _check_edges(M, g, p, gb, pb, matches):
    """mask_edge_distance, CPU and CUDA outputs, == reference; the work of every pair checked before the launch."""
    c = A.edge_counts(g, p, gb, pb, matches)
    assert (c[:, 0] * c[:, 2] + c[:, 1] * c[:, 3]).max() <= EDGE_WORK_LIMIT
    wfp, wfn = A.edge_distances(g, p, gb, pb, matches)
    assert all(x is not None for x in wfp + wfn)
    enc = lambda ms: [M.rle.encode(np.asfortranarray(m.astype(np.uint8))) for m in ms]
    ge, pe = enc(g), enc(p)
    for device in ('cpu', 'cuda'):
        fp, fn = M.analyze.mask_edge_distance(ge, pe, gb, pb, matches, device=device)
        assert len(fp) == len(fn) == len(matches)
        for a, b in zip(fp + fn, wfp + wfn):
            assert a.dtype == M.torch.float64 and a.is_cuda == (device == 'cuda')
            assert np.array_equal(a.cpu().numpy(), b)
    return c


def test_edge_candidate_tiles(M):
    """The other mask has 1023, 1024, 1025 and thousands of boundary pixels in the window; the last candidate sits
    alone at the end of the raster, nearest to a crowd of queries, so it lands in the next tile."""
    h, w = 1024, 1024
    gs, ps = [], []
    for a, b, extra in [(256, 257, True), (257, 257, False), (257, 257, True)]:
        r = np.zeros((h, w), bool)
        r[100:100 + a, 100:100 + b] = True
        if extra:
            r[640, 641] = True
        block = np.zeros((h, w), bool)
        block[50:651, 60:663] = True                              # window 601 x 603: no multiple of 256
        gs += [r, block]
        ps += [block, r]
    rng = np.random.default_rng(1)
    noise = np.zeros((h, w), bool)
    noise[300:400, 500:600] = rng.random((100, 100)) < 0.5
    block = np.zeros((h, w), bool)
    block[250:451, 450:651] = True
    gs += [noise, block]
    ps += [block, noise]
    boxes_g = np.array([_tight_box(m) for m in gs])
    boxes_p = np.array([_tight_box(m) for m in ps])
    matches = np.stack([np.arange(len(gs)), np.arange(len(ps))], 1)
    c = _check_edges(M, gs, ps, boxes_g, boxes_p, matches)
    assert c[0:6:2, 2].tolist() == [1023, 1024, 1025] and c[1:6:2, 3].tolist() == [1023, 1024, 1025]
    assert c[6, 2] > 3000 and c[7, 3] > 3000
    assert (c[:, 0] + c[:, 1] > 256).all()
    win = (boxes_g[:, 1] - boxes_g[:, 0]) * (boxes_g[:, 3] - boxes_g[:, 2])
    assert (np.maximum(win, 1) % 256 != 0).any()


def _blob(rng, h, w):
    m = np.zeros((h, w), bool)
    while not m.any():
        cy, cx = rng.uniform(0, h), rng.uniform(0, w)
        ry, rx = rng.uniform(3, 90, 2)
        r0, r1 = max(int(cy - ry) - 1, 0), min(int(cy + ry) + 2, h)
        c0, c1 = max(int(cx - rx) - 1, 0), min(int(cx + rx) + 2, w)
        yy, xx = np.ogrid[r0:r1, c0:c1]
        m[r0:r1, c0:c1] = ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1
        if rng.random() < 0.3:
            m[r0:r1, c0:c1] ^= rng.random((r1 - r0, c1 - c0)) < 0.1
    return m


def test_edge_many_pairs_shared_masks_reverse_order(M):
    h, w = 1024, 1536
    rng = np.random.default_rng(77)
    g = [_blob(rng, h, w) for _ in range(40)]
    p = []
    for m in g:
        q = np.roll(m, (int(rng.integers(-6, 7)), int(rng.integers(-6, 7))), axis=(0, 1))
        p.append(q if q.any() else m)
    gb = np.array([_tight_box(m) for m in g])
    pb = np.array([_tight_box(m) for m in p])
    loose = rng.random(len(gb)) < 0.2                                  # loose boxes sticking out of the frame
    gb[loose, 1] += 300
    gb[loose, 3] += 400
    pairs = np.array([(i, i) for i in range(40)] + [(int(a), int(b)) for a, b in rng.integers(0, 40, (80, 2))])
    fp, fn = A.edge_distances(g, p, gb, pb, pairs)
    matches = np.array([q for q, a, b in zip(pairs, fp, fn) if a is not None and b is not None][::-1])
    assert len(matches) > 60
    _check_edges(M, g, p, gb, pb, matches)


def test_edge_windows_at_32767(M):
    rng = np.random.default_rng(32767)
    h, w = 3, 32767
    g = rng.random((h, w)) < 0.01
    g[0, 0] = True
    p = np.roll(g, 5, axis=1)
    p[2, w - 1] = True
    box = np.array([[0, h, 0, w]])
    _check_edges(M, [g], [p], box, box, np.array([[0, 0]]))
    wide = np.zeros((3, 32768), bool)
    wide[1, 7] = True
    enc = [M.rle.encode(np.asfortranarray(wide.astype(np.uint8)))]
    with pytest.raises(ValueError):
        M.analyze.mask_edge_distance(enc, enc, np.array([[0, 3, 0, 32768]]), np.array([[1, 2, 7, 8]]), [[0, 0]])
    with pytest.raises(ValueError):
        M.analyze.mask_edge_distance(enc, enc, np.array([[0, 3, -1, 8]]), np.array([[1, 2, 7, 8]]), [[0, 0]])


def test_edge_corner_to_corner_on_a_32767_frame(M):
    """Single pixels at (0, 0) and (32766, 32766): the window is the whole 1.07 G-pixel frame, scanned by one CTA,
    and the squared distance 2·32766² is the largest the kernel's int arithmetic meets."""
    n = 32767
    hw = n * n
    s = M.rle.string_from_counts
    gt = [{'size': [n, n], 'counts': s(np.array([0, 1, hw - 1], np.uint32))}]
    pr = [{'size': [n, n], 'counts': s(np.array([hw - 1, 1], np.uint32))}]
    d = np.sqrt(np.float64(2 * 32766 ** 2))
    fp, fn = M.analyze.mask_edge_distance(gt, pr, np.array([[0, 1, 0, 1]]), np.array([[n - 1, n, n - 1, n]]), [[0, 0]])
    assert fp[0].tolist() == [d] and fn[0].tolist() == [d]


def test_edge_pair_without_the_other_mask_raises(M):
    h, w = 600, 700
    rng = np.random.default_rng(9)
    g = [_blob(rng, h, w) for _ in range(4)]
    p = [m.copy() for m in g]
    p[3][:] = False
    p[3][500:520, 600:650] = True
    g[3][:] = False
    g[3][10:20, 10:20] = True
    gb = np.array([_tight_box(m) for m in g])
    pb = np.array([_tight_box(m) for m in p])
    gb[3] = pb[3]                                  # the window holds pred pixels only: FP queries, no candidates
    matches = np.array([[0, 0], [1, 1], [3, 3], [2, 2]])
    fp, fn = A.edge_distances(g, p, gb, pb, matches)
    assert fp[2] is None and all(x is not None for x in fp[:2] + fp[3:])
    enc = lambda ms: [M.rle.encode(np.asfortranarray(m.astype(np.uint8))) for m in ms]
    with pytest.raises(RuntimeError):
        M.analyze.mask_edge_distance(enc(g), enc(p), gb, pb, matches)


# ---- pixel-class projection ---------------------------------------------------------------------------------------

@pytest.mark.parametrize('mode', ['reduced', 'all'])
def test_seg_perf_iset_of_crowded_overlapping_pairs(M, mode):
    """~300 matched pairs piled on a 1000 x 1001 frame (h·w no multiple of 32): the projection ORs every pair into
    the same words, and the encoder's last word is partial."""
    h, w = 1000, 1001
    rng = np.random.default_rng(1001)
    g = [_blob(rng, 400, 400) for _ in range(120)]
    g = [np.pad(m, ((300, h - 700), (300, w - 700))) for m in g]
    p = [np.roll(m, (int(rng.integers(-9, 10)), int(rng.integers(-9, 10))), axis=(0, 1)) for m in g]
    g[0][-1, -1] = p[1][-1, -1] = True
    pairs = np.array([(i, i) for i in range(120)] + [(int(a), int(b)) for a, b in rng.integers(0, 120, (180, 2))])
    enc = lambda ms: [M.rle.encode(np.asfortranarray(m.astype(np.uint8))) for m in ms]
    ge, pe = enc(g), enc(p)
    iset, _ = M.analyze.seg_perf_iset(ge, pe, {'tp': pairs}, mode=mode)
    want = M.R.seg_perf_masks(ge, pe, pairs, mode)
    assert [m['counts'] for m in iset.instances.masks.rle] == [m['counts'] for m in want]
