"""The flat crop decode (rle_flat.cu) on hand-made run-count tables laid out against its 8-pair lane slices: mask
boundaries at every slot of a lane and on lane boundaries, masks of one pair, a mask of exactly the 256-pair round
budget, empty tables, and malformed tables (runs past the frame, saturated runs, zero-length runs, totals other than
H * W).  Area, box, span, status, window form and size against the CPU model of the measure pass
(tests/test_flat_round_model.py) and, for well-formed masks, the oracle; windows through the crop step against the
oracle's dense intersections.  Intervals on and off, several masks-per-warp hints."""
import numpy as np
import pytest

from tests.test_crop_intervals_gpu import _check_vs_oracle, _host, _same, _step, mods  # noqa: F401
from tests.test_flat_round_model import CAP, M32, blob_counts, div_by, model_pass32

pytestmark = pytest.mark.gpu

CHUNK_BITS = 128


def _expected(cnt, H, W, intervals):
    """area, bbox, span, status, form and window chunks the decode writes for one table (records of
    rle_flat_crop_kernel from the model's per-mask statistics)"""
    st, _ = model_pass32([cnt], [(H, W)])
    ar, fi, la = st['area'][0], st['first'][0], st['last'][0]
    HW = H * W
    rcp = M32 // H
    bb, sp = (0, 0, -1, -1), (0, 0)
    if ar > 0:
        nchunks = (HW + CHUNK_BITS - 1) // CHUNK_BITS
        sp = (fi // CHUNK_BITS, min((la + CHUNK_BITS - 1) // CHUNK_BITS, nchunks))
        bb = (div_by(fi, H, rcp), st['ymin'][0], div_by(la - 1, H, rcp), 0xffff - st['ymaxi'][0])
    form = int(intervals and ar > 0 and st['convex'][0] == 1)
    if form:
        chunks = (bb[2] - bb[0] + 4) // 4
    else:
        words = 0 if bb[2] < bb[0] else (bb[2] - bb[0] + 1) * ((bb[3] >> 5) - (bb[1] >> 5) + 1)
        chunks = (words + 3) // 4
    return ar, bb, sp, 0 if st['total'][0] == HW else 1, form, chunks


def _tables(rng):
    """(counts, H, W) of every layout, the well-formed ones first (mixed), the 61 malformed ones after.  Windows of
    at most 300 x 32 or 60 x 64 pixels stay inside the tile, so that no table goes to the fallback kernel"""
    H, W = 32, 300
    t = []
    for slot in range(8):                                   # the next mask starts at slot `slot` of a lane
        for n in (8 + slot, 8 * 5 + slot, 1, 7, 9, 33):
            t.append((blob_counts(n, H, W, rng), H, W))
    t += [(blob_counts(1, H, W, rng), H, W) for _ in range(20)]                     # one pair each
    t.append((np.array([H * W], np.int64), H, W))                                   # one 0-run
    t.append((blob_counts(256, 30, 300, rng), 30, 300))                             # exactly the round budget
    t.append((blob_counts(255, 30, 300, rng, tail=True), 30, 300))
    t = [t[i] for i in rng.permutation(len(t))]
    t.append((np.zeros(0, np.int64), H, W))                                         # no counts: total 0
    for k in range(60):                                                             # malformed
        h, w = int(rng.integers(1, 64)), int(rng.integers(1, 60))
        m = int(rng.integers(0, 2 * CAP + 1))
        mag = int(rng.choice([3, 40, h * w + 1, 2 ** 20, 2 ** 31, 2 ** 32 - 1]))
        c = rng.integers(0, mag, m, dtype=np.int64)
        if m and k % 3 == 0:
            c = c % max(h, 1)
            c[-1] = max(h * w - int(c[:-1].sum()), 0)                              # a right total, odd runs
        if m and k % 4 == 1:
            c[rng.integers(0, m, max(1, m // 4))] = 0                               # zero-length runs
        t.append((c, h, w))
    return t


@pytest.mark.parametrize('hint', [-1, 0, 2, 30, 100])
@pytest.mark.parametrize('intervals', [False, True])
def test_flat_decode_of_hand_made_tables(mods, monkeypatch, intervals, hint):
    E, torch = mods.engine, mods.torch
    monkeypatch.setattr(E, 'CROP_DECODE', 'flat')
    monkeypatch.setattr(E, 'PAINT_RUNS_HINT', hint)
    rng = np.random.default_rng(2024)
    tabs = _tables(rng)
    n = len(tabs)
    lens = np.array([len(c) for c, _, _ in tabs], np.int32)
    off = np.zeros(n, np.int64)
    off[1:] = np.cumsum(lens[:-1])
    cnt = np.concatenate([c for c, _, _ in tabs]).astype(np.uint32)
    dev = 'cuda'
    t = E.MaskTable(torch.device('cuda', torch.cuda.current_device()), n,
                    torch.from_numpy(cnt.view(np.int32)).to(dev), torch.from_numpy(off).to(dev),
                    torch.from_numpy(lens).to(dev),
                    torch.tensor([h for _, h, _ in tabs], dtype=torch.int32, device=dev),
                    torch.tensor([w for _, _, w in tabs], dtype=torch.int32, device=dev), E.LAYOUT_CROP)
    arena = torch.empty(4 * 128 * n, dtype=torch.int32, device=dev)                 # a tile per mask: never short
    t.measure_paint(arena, intervals=intervals)
    torch.cuda.synchronize()
    iv = intervals and E.pairs_read_intervals()
    assert t.intervals == iv
    assert int(t.list[0].item()) == 0                                               # nothing for the fallback
    area = t.area[:n].cpu().numpy().view(np.uint32)
    bbox = t.bbox[:4 * n].cpu().numpy().reshape(-1, 4)
    span = t.span[:2 * n].cpu().numpy().view(np.uint32).reshape(-1, 2)
    reg = t.reg[:2 * n].cpu().numpy().view(np.uint32).reshape(-1, 2)
    status = t.status[:n].cpu().numpy()
    for i, (c, h, w) in enumerate(tabs):
        ar, bb, sp, stt, form, chunks = _expected(c, h, w, iv)
        tag = (i, len(c), h, w)
        assert area[i] == ar and tuple(bbox[i]) == bb and tuple(span[i]) == sp and status[i] == stt, tag
        assert tuple(reg[i]) == (form, chunks), tag
    from oracle import cocomask as rle
    for i, (c, h, w) in enumerate(tabs[:-61]):                                      # well-formed: the oracle
        m = np.asarray(rle.decode({'size': [h, w], 'counts': rle.string_from_counts(c.astype(np.uint32))}), bool)
        assert area[i] == m.sum(), i
        if m.any():
            ys, xs = np.nonzero(m)
            assert tuple(bbox[i]) == (xs.min(), ys.min(), xs.max(), ys.max()), i


def _blob_stack(rng, layout, h, w):
    """bool[k, h, w] masks of the given pair counts (one vertical 1-run per column, the last column's reaching the
    frame's end), through the oracle's decoder"""
    from oracle import cocomask as rle
    return np.stack([np.asarray(rle.decode({'size': [h, w], 'counts': rle.string_from_counts(
        blob_counts(n, h, w, rng).astype(np.uint32))}), bool) for n in layout])


def test_crop_step_windows_against_the_oracle(mods):
    """Two images whose masks put mask boundaries at every slot of a lane, masks of one pair and a 256-pair mask;
    the step with intervals on and off gives the same results, equal to the oracle's dense intersections."""
    rng = np.random.default_rng(77)
    h, w = 32, 300
    layout = [8 + s for s in range(8)] + [1] * 6 + [256] + [7, 9, 17, 33, 1, 2]      # 22 rows + 22 columns
    stacks = []
    for img in range(2):
        rows = _blob_stack(rng, layout, h, w)
        cols = _blob_stack(rng, list(reversed(layout)), h, w)
        stacks.append(np.concatenate([rows, cols]))
    n_rows = len(layout)
    host = _host(mods, stacks, n_rows, h, w)
    on, off = _step(mods, host, True), _step(mods, host, False)
    assert not off['forms'].any() and on['forms'].all()                            # every blob is column-convex
    _same(on, off, 'blobs')
    _check_vs_oracle(mods, on, stacks, n_rows, 'blobs')
