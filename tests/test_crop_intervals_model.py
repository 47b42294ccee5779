"""Host model of the column-convex test of the flat crop decode (rle_flat.cu, intervals on).  The kernel decides per
(0-run, 1-run) pair, without a scan: a 1-run that crosses a column end, or one that is not the mask's first and whose
0-run is shorter than its first row (so the 1-run before it ends in the same column), makes the mask a bitmap.  On
canonical RLE this must equal the definition -- at most one 1-run per column and none crossing a column end -- and it
must never call a mask an interval mask that is not one."""
import numpy as np

from oracle import cocomask as rle


def _kernel_rule(counts, h):
    pos = 0
    for k in range(0, len(counts), 2):
        z = int(counts[k])
        o = int(counts[k + 1]) if k + 1 < len(counts) else 0
        start = pos + z
        pos = start + o
        if o == 0:
            continue
        x, ys = divmod(start, h)
        if ys + o - 1 >= h or (k >= 2 and z < ys):
            return False
    return True


def _definition(m):
    h, w = m.shape
    flat = m.T.reshape(-1).astype(np.int8)                  # column-major, as RLE counts it
    d = np.diff(np.r_[0, flat, 0])
    starts, ends = np.flatnonzero(d == 1), np.flatnonzero(d == -1)
    if ((starts // h) != ((ends - 1) // h)).any():          # a run crosses a column end
        return False
    return np.bincount(starts // h, minlength=w).max(initial=0) <= 1


def _masks(rng, n, h, w):
    y, x = np.ogrid[:h, :w]
    for _ in range(n):
        kind = rng.integers(0, 6)
        if kind == 0:                                         # blob
            cy, cx, r = rng.integers(0, h), rng.integers(0, w), rng.integers(1, max(h, w) + 1)
            yield (y - cy) ** 2 + (x - cx) ** 2 <= r * r
        elif kind == 1:                                       # ring
            cy, cx, r = h // 2, w // 2, rng.integers(3, max(h, w) // 2 + 4)
            d = (y - cy) ** 2 + (x - cx) ** 2
            yield (d <= r * r) & (d > (r // 2) ** 2)
        elif kind == 2:                                       # full-height stripes: runs cross column ends
            m = np.zeros((h, w), bool)
            m[:, rng.integers(0, w):rng.integers(0, w) + 1] = True
            yield m
        elif kind == 3:                                       # noise
            yield rng.random((h, w)) < rng.random()
        elif kind == 4:                                       # a run per column at random rows
            m = np.zeros((h, w), bool)
            for c in range(w):
                if rng.random() < 0.7:
                    a = rng.integers(0, h)
                    m[a:rng.integers(a, h) + 1, c] = True
            yield m
        else:                                                 # single pixels, rows, columns, empty
            m = np.zeros((h, w), bool)
            k = rng.integers(0, 4)
            if k == 1:
                m[rng.integers(0, h), rng.integers(0, w)] = True
            elif k == 2:
                m[rng.integers(0, h), :] = True
            elif k == 3:
                m[:, rng.integers(0, w)] = True
            yield m


def test_column_convex_rule_of_the_flat_decode_equals_the_definition():
    rng = np.random.default_rng(7)
    seen = set()
    for h, w in ((1, 1), (1, 9), (7, 1), (5, 6), (32, 33), (40, 17)):
        for m in _masks(rng, 300, h, w):
            cnt = rle.counts_from_string(rle.encode(np.asfortranarray(m.astype(np.uint8)))['counts'])
            got, want = _kernel_rule(cnt, h), _definition(m)
            assert got == want, (h, w, m.astype(int).tolist())
            seen.add(want)
    assert seen == {True, False}


def test_zero_length_runs_make_a_bitmap_never_a_wrong_interval():
    """Non-canonical counts (a zero-length 1-run inside the list) may only turn an interval mask into a bitmap."""
    h = 10
    # column 0 rows 1..2 and 5..6 with a zero-length 1-run between them: two runs in a column, a bitmap
    assert not _kernel_rule([1, 2, 1, 0, 1, 2], h)
    # column 0 rows 2..4, a zero-length 1-run at column 1 row 2, column 1 rows 4..5: an interval mask, which the
    # rule conservatively leaves a bitmap ...
    assert not _kernel_rule([2, 3, 7, 0, 2, 2], h)
    # ... and takes as intervals in canonical form
    assert _kernel_rule([2, 3, 9, 2], h)
