"""CPU model (numpy / Python integers) of the measure pass of rle_flat_crop_kernel (csrc/rle_flat.cu), lane by lane:
the round's pairs staged lane-strided into a swizzled buffer and padded to whole 8-pair slices, lane l owning pairs
8l .. 8l+7, head bits from the mask bytes, pass 1 (saturating end sums from the last start), ONE segmented warp scan
with the head flag in bit 31, pass 2 (records, per-slice statistics, flushes, totals, column-convex rule).

It is checked against the oracle's decoded masks and, pair for pair, against a model of the previous pass (32 pairs
per pass, three segmented scans, ballots, a carry from pass to pass), including malformed run-count tables: runs past
the frame, saturated runs, zero-length runs, totals other than H * W.  The shared buffers keep what earlier rounds left
in them (random words at the start), as they do in the kernel."""
import numpy as np
import pytest

SAT, SPAN, HEAD, M32 = 0x7fffffff, 0x80000000, 0x80000000, 0xffffffff
CAP = 256


def sat_add(a, b):
    return min(a + b, SAT)


def div_by(s, d, rcp):
    q = (s * rcp) >> 32
    if s - q * d >= d:
        q += 1
    return q


def vminu2(a, b):
    return min(a & 0xffff, b & 0xffff) | (min(a >> 16, b >> 16) << 16)


def vcmpne4(a, b):
    return sum((0xff << (8 * i)) for i in range(4) if ((a >> (8 * i)) & 0xff) != ((b >> (8 * i)) & 0xff))


def swz(f):
    return f ^ ((f >> 3) & 6)


def geo_of(cnts, frames):
    return [(H, (M32 // H) if H else 0, (H * W) & M32, len(c)) for c, (H, W) in zip(cnts, frames)]


def record(start, o, H, rcp, z, head):
    """the painter's record, the row-range word and whether the pair breaks column-convexity"""
    x = div_by(start, H, rcp)
    ys = start - x * H
    yl = ys + o - 1
    breaks = yl >= H or (not head and z < ys)
    if yl >= H:
        return (start | SPAN, o), (0xffff - (H - 1)) << 16, breaks
    return (x, ys | (yl << 16)), ys | ((0xffff - yl) << 16), breaks


def fresh_stats(nb):
    return dict(area=[0] * nb, first=[M32] * nb, last=[0] * nb, ymin=[M32] * nb, ymaxi=[M32] * nb, total=[0] * nb,
                convex=[1] * nb)


def model_pass32(cnts, frames):
    """The previous measure pass: 32 pairs per pass, lane = pair, segmented inclusive scans reaching min(lane, p)
    lanes down, a carry from lane 31 to the next pass, ballots for the first / last good lane of a segment."""
    geo = geo_of(cnts, frames)
    npairs = [(len(c) + 1) >> 1 for c in cnts]
    pb = np.concatenate([[0], np.cumsum(npairs)]).astype(np.int64)
    T, nb = int(pb[-1]), len(cnts)
    st = fresh_stats(nb)
    rec, carry = [None] * T, 0
    for f0 in range(0, T, 32):
        ok = [f0 + l < T for l in range(32)]
        j = [int(np.searchsorted(pb, f0 + l, side='right') - 1) if ok[l] else 0 for l in range(32)]
        p = [f0 + l - int(pb[j[l]]) if ok[l] else 0 for l in range(32)]
        z, o = [0] * 32, [0] * 32
        for l in range(32):
            if ok[l]:
                c = cnts[j[l]]
                z[l] = min(int(c[2 * p[l]]), SAT)
                o[l] = min(int(c[2 * p[l] + 1]), SAT) if 2 * p[l] + 1 < len(c) else 0
        end, osum = [sat_add(z[l], o[l]) for l in range(32)], list(o)
        reach = [min(l, p[l]) if ok[l] else 0 for l in range(32)]
        d = 1
        while d < 32:
            te, to = [end[l - d] if l >= d else end[l] for l in range(32)], [osum[l - d] if l >= d else osum[l] for l in range(32)]
            for l in range(32):
                if d <= reach[l]:
                    end[l], osum[l] = sat_add(end[l], te[l]), (osum[l] + to[l]) & M32
            d <<= 1
        for l in range(32):
            if ok[l] and p[l] > l:
                end[l] = sat_add(end[l], carry)
        carry = end[31]
        inb = [ok[l] and end[l] <= geo[j[l]][2] for l in range(32)]
        good = [inb[l] and o[l] > 0 for l in range(32)]
        start = [(end[l] - o[l]) & M32 for l in range(32)]
        ypk = [M32] * 32
        for l in range(32):
            if not ok[l]:
                continue
            rec[f0 + l] = (0, 0x0000ffff)
            if good[l]:
                H, rcp = geo[j[l]][0], geo[j[l]][1]
                rec[f0 + l], ypk[l], breaks = record(start[l], o[l], H, rcp, z[l], p[l] == 0)
                if breaks:
                    st['convex'][j[l]] = 0
        d = 1
        while d < 32:
            t = [ypk[l - d] if l >= d else ypk[l] for l in range(32)]
            ypk = [vminu2(ypk[l], t[l]) if d <= reach[l] else ypk[l] for l in range(32)]
            d <<= 1
        for l in range(32):
            f = f0 + l
            if not ok[l]:
                continue
            seg_end = f + 1 == pb[j[l] + 1]
            if not (seg_end or l == 31):
                continue
            lo = l - reach[l]
            gs = [k for k in range(lo, l + 1) if good[k]]
            ins = [k for k in range(lo, l + 1) if inb[k]]
            if gs:
                jj = j[l]
                st['area'][jj] += osum[ins[-1]]
                st['first'][jj] = min(st['first'][jj], start[gs[0]])
                st['last'][jj] = max(st['last'][jj], end[gs[-1]])
                st['ymin'][jj] = min(st['ymin'][jj], ypk[l] & 0xffff)
                st['ymaxi'][jj] = min(st['ymaxi'][jj], ypk[l] >> 16)
            if seg_end:
                st['total'][j[l]] = end[l]
    return st, rec


class RoundModel:
    """The new pass.  pair / mid are the warp's shared buffers and live from round to round."""

    def __init__(self, rng):
        self.pair = [(int(rng.integers(0, 2 ** 32)), int(rng.integers(0, 2 ** 32))) for _ in range(CAP)]
        self.mid = [int(rng.integers(0, 256)) for _ in range(CAP)]

    def run(self, cnts, frames):
        geo = geo_of(cnts, frames)
        nb = len(cnts)
        npairs = [(len(c) + 1) >> 1 for c in cnts]
        pb = [0] + list(np.cumsum(npairs))
        T = int(pb[-1])
        assert T <= CAP and nb <= 16
        st = fresh_stats(nb)
        pair, mid = self.pair, self.mid
        # staging: lane-strided, padded with (0, 0) pairs of the last mask to a multiple of 8
        Tr = (T + 7) & ~7
        for lane in range(32):
            j, cur, nxt = 0, 0, pb[1]
            for f in range(lane, Tr, 32):
                zo = (0, 0)
                if f < T:
                    while f >= nxt:
                        j += 1
                        cur, nxt = nxt, pb[j + 1]
                    p, c = f - cur, cnts[j]
                    zo = (min(int(c[2 * p]), SAT), min(int(c[2 * p + 1]), SAT) if 2 * p + 1 < geo[j][3] else 0)
                mid[f] = j if f < T else nb - 1
                pair[swz(f)] = zo
        # pass 1
        mm = [(sum(mid[8 * l + i] << (8 * i) for i in range(4)), sum(mid[8 * l + 4 + i] << (8 * i) for i in range(4)))
              for l in range(32)]
        hb, sc = [0] * 32, [0] * 32
        for l in range(32):
            lo, hi = mm[l]
            mprev = (mm[l - 1] if l > 0 else mm[l])[1] >> 24                    # __shfl_up: lane 0 reads itself
            dl = vcmpne4(lo, ((lo << 8) | mprev) & M32)
            dh = vcmpne4(hi, ((hi << 8) | (lo >> 24)) & M32)
            hb[l] = (((dl & 0x01010101) * 0x01020408) & M32) >> 24 | (((dh & 0x01010101) * 0x01020408) & M32) >> 20 \
                | (l == 0)
            assert hb[l] < 256
            sw, s = (l >> 1) & 3, 0
            for q in range(4):
                c0, c1 = pair[8 * l + 2 * (q ^ sw)], pair[8 * l + 2 * (q ^ sw) + 1]
                s = sat_add(0 if (hb[l] >> (2 * q)) & 1 else s, sat_add(c0[0], c0[1]))
                s = sat_add(0 if (hb[l] >> (2 * q + 1)) & 1 else s, sat_add(c1[0], c1[1]))
            sc[l] = s | (HEAD if hb[l] else 0)
        # one segmented scan
        d = 1
        while d < 32:
            t = [sc[l - d] if l >= d else sc[l] for l in range(32)]
            sc = [sc[l] if sc[l] & HEAD else sat_add(t[l] & SAT, sc[l]) | (t[l] & HEAD) for l in range(32)]
            d <<= 1
        # pass 2
        for l in range(32):
            f8 = 8 * l
            e = (sc[l - 1] if l > 0 else sc[l]) & SAT
            if f8 >= T:
                continue
            sw = (l >> 1) & 3
            j = mm[l][0] & 0xff
            acc = dict(ar=0, fi=M32, la=0, ypk=M32)

            def flush(j, ended, e):
                if acc['fi'] != M32:
                    st['area'][j] = (st['area'][j] + acc['ar']) & M32
                    st['first'][j] = min(st['first'][j], acc['fi'])
                    st['last'][j] = max(st['last'][j], acc['la'])
                    st['ymin'][j] = min(st['ymin'][j], acc['ypk'] & 0xffff)
                    st['ymaxi'][j] = min(st['ymaxi'][j], acc['ypk'] >> 16)
                if ended:
                    st['total'][j] = e

            for q in range(4):
                out = []
                for k in (2 * q, 2 * q + 1):
                    z, o = pair[8 * l + 2 * (q ^ sw) + (k & 1)]
                    h = (hb[l] >> k) & 1
                    if k > 0 and h:
                        flush(j, True, e)
                        j = mid[f8 + k]
                        acc = dict(ar=0, fi=M32, la=0, ypk=M32)
                    H, rcp, HW, _ = geo[j]
                    e = sat_add(0 if h else e, sat_add(z, o))
                    pr = (0, 0x0000ffff)
                    if e <= HW:
                        acc['ar'] = (acc['ar'] + o) & M32
                        if o > 0:
                            start = e - o
                            pr, yp, breaks = record(start, o, H, rcp, z, h)
                            if breaks:
                                st['convex'][j] = 0
                            acc['fi'], acc['la'] = min(acc['fi'], start), e
                            acc['ypk'] = vminu2(acc['ypk'], yp)
                    out.append(pr)
                pair[8 * l + 2 * (q ^ sw)], pair[8 * l + 2 * (q ^ sw) + 1] = out
            flush(j, f8 + 8 >= T or mid[f8 + 8] != j, e)
        rec = [pair[swz(f)] for f in range(T)]
        assert [mid[f] for f in range(T)] == [int(np.searchsorted(pb, f, side='right') - 1) for f in range(T)]
        return st, rec


def check_equal_to_pass32(model, cnts, frames, tag):
    st, rec = model.run(cnts, frames)
    st0, rec0 = model_pass32(cnts, frames)
    assert rec == rec0, tag
    for k in st0:
        assert st[k] == st0[k], (tag, k)
    return st, rec


def counts_of(m):
    from oracle import cocomask as rle
    return rle.counts_from_string(rle.encode(np.asfortranarray(m.astype(np.uint8)))['counts']).astype(np.int64)


def random_mask(rng, H, W):
    kind = rng.integers(0, 5)
    m = np.zeros((H, W), bool)
    if kind == 1:
        m = rng.random((H, W)) < rng.random()
    elif kind == 2:
        m[:, int(rng.integers(0, W)):] = True
    elif kind >= 3:
        y, x, r = rng.integers(0, H), rng.integers(0, W), rng.integers(1, 12)
        yy, xx = np.ogrid[:H, :W]
        m = (yy - y) ** 2 + (xx - x) ** 2 <= r * r
    return m


def test_round_model_equals_the_oracle_and_the_previous_pass():
    """Decoded masks of the oracle: area, box, rows, the records painted back, column-convexity."""
    rng = np.random.default_rng(11)
    model = RoundModel(rng)
    done = 0
    for trial in range(60):
        H, W = int(rng.integers(3, 90)), int(rng.integers(3, 90))
        K = int(rng.integers(1, 9))
        masks = [random_mask(rng, H, W) for _ in range(K)]
        cnts = [counts_of(m) for m in masks]
        if sum((len(c) + 1) >> 1 for c in cnts) > CAP:
            continue
        done += 1
        st, rec = check_equal_to_pass32(model, cnts, [(H, W)] * K, trial)
        pb = np.concatenate([[0], np.cumsum([(len(c) + 1) >> 1 for c in cnts])])
        for k, m in enumerate(masks):
            assert st['area'][k] == m.sum() and st['total'][k] == H * W, (trial, k)
            painted = np.zeros((W, H), bool)
            for f in range(int(pb[k]), int(pb[k + 1])):
                x, y = rec[f]
                if x & SPAN:
                    painted.reshape(-1)[(x & ~SPAN):(x & ~SPAN) + y] = True
                elif (y & 0xffff) <= (y >> 16):
                    painted[x, (y & 0xffff):(y >> 16) + 1] = True
            assert np.array_equal(painted.T, m), (trial, k)
            if m.any():
                ys_, xs_ = np.nonzero(m)
                assert st['first'][k] // H == xs_.min() and (st['last'][k] - 1) // H == xs_.max(), (trial, k)
                assert (st['ymin'][k], 0xffff - st['ymaxi'][k]) == (ys_.min(), ys_.max()), (trial, k)
                if st['convex'][k]:                                       # one 1-run per column: really convex
                    assert all(np.diff(np.nonzero(m[:, x])[0]).max(initial=1) == 1 for x in range(W)), (trial, k)
    assert done >= 30


def blob_counts(npairs, H, W, rng, tail=False):
    """a well-formed table of exactly npairs (0-run, 1-run) pairs in an H x W frame (npairs <= W): one vertical 1-run
    in each of npairs columns, the last one ending on the frame's last pixel -- or, with tail, a final 0-run after it
    (one pair more)"""
    cols = np.sort(rng.choice(W - 1, npairs - (not tail), replace=False))
    m = np.zeros((H, W), bool)
    for x in cols:                                          # row 0 stays clear: runs of neighbouring columns never join
        y0 = int(rng.integers(1, H))
        m[y0:int(rng.integers(y0, H)) + 1, x] = True
    if not tail:
        m[int(rng.integers(1, H)):, W - 1] = True
    c = counts_of(m)
    assert (len(c) + 1) >> 1 == npairs + tail
    return c


@pytest.mark.parametrize('slot', range(8))
def test_mask_boundaries_at_every_slot_of_a_lane(slot):
    """The first mask ends so that the next starts at slot `slot` of a lane (slot 0: exactly on a lane boundary),
    followed by masks of 1, 7, 8, 9 and 33 pairs, an empty table and a mask of one pair."""
    rng = np.random.default_rng(100 + slot)
    model = RoundModel(rng)
    H, W = 40, 300
    for first in (8 * 1 + slot, 8 * 4 + slot, 8 * 11 + slot):
        tables = [blob_counts(first, H, W, rng)]
        for n in (1, 7, 8, 9, 33):
            tables.append(blob_counts(n, H, W, rng))
        tables.append(np.zeros(0, np.int64))                              # no run counts: no pairs
        tables.append(np.array([H * W], np.int64))                         # one 0-run: one pair, nothing painted
        tables.append(blob_counts(1, H, W, rng))
        assert sum((len(c) + 1) >> 1 for c in tables) <= CAP
        st, _ = check_equal_to_pass32(model, tables, [(H, W)] * len(tables), (slot, first))
        assert st['total'] == [H * W] * len(tables[:6]) + [0, H * W, H * W]


def test_one_pair_masks_and_a_full_round_of_one_mask():
    rng = np.random.default_rng(5)
    model = RoundModel(rng)
    H, W = 30, 300
    ones = [blob_counts(1, H, W, rng) for _ in range(16)]                   # 16 masks of one pair each
    check_equal_to_pass32(model, ones, [(H, W)] * 16, 'ones')
    big = blob_counts(256, H, W, rng)                                       # exactly the pair budget
    assert (len(big) + 1) >> 1 == 256
    st, rec = check_equal_to_pass32(model, [big], [(H, W)], 'cap')
    assert st['total'] == [H * W] and st['convex'] == [1]
    odd = blob_counts(255, H, W, rng, tail=True)                            # 255 pairs + a final 0-run: 256
    check_equal_to_pass32(model, [odd], [(H, W)], 'cap-odd')


def test_malformed_tables_equal_the_previous_pass():
    """Runs past the frame, saturated runs (>= 2^31), zero-length 1-runs and 0-runs, totals short of or beyond H * W,
    frames of different sizes in one round; mask boundaries anywhere."""
    rng = np.random.default_rng(21)
    model = RoundModel(rng)
    for trial in range(150):
        K = int(rng.integers(1, 17))
        frames, tables = [], []
        budget = CAP
        for k in range(K):
            H, W = int(rng.integers(1, 70)), int(rng.integers(1, 70))
            m = int(rng.integers(0, min(budget, 80) * 2 + 1)) if budget else 0
            if rng.random() < 0.1 and budget >= 128:
                m = 2 * budget - int(rng.integers(0, 2))                    # fill the round up to the last pair
            mag = int(rng.choice([2, 5, 40, H * W + 1, 2 ** 20, 2 ** 31, 2 ** 32 - 1]))
            c = rng.integers(0, mag, m, dtype=np.int64) if mag > 2 else rng.integers(0, 3, m, dtype=np.int64)
            if m and rng.random() < 0.3:                                     # a well-formed total with odd runs
                c = np.abs(c) % max(H, 1)
                c[-1] = max(H * W - int(c[:-1].sum()), 0)
            if m and rng.random() < 0.2:
                c[rng.integers(0, m, max(1, m // 4))] = 0                   # zero-length runs
            budget -= (m + 1) >> 1
            frames.append((H, W))
            tables.append(c.astype(np.int64))
        check_equal_to_pass32(model, tables, frames, trial)


def test_scan_carries_a_mask_over_many_lanes_with_saturation():
    """One mask whose ends saturate in the middle of a lane, then a well-formed one; and a round whose pairs all
    belong to one saturated mask."""
    rng = np.random.default_rng(3)
    model = RoundModel(rng)
    H, W = 64, 64
    sat = np.full(100, 2 ** 30, np.int64)                                  # ends reach 2^31 - 1 after two pairs
    check_equal_to_pass32(model, [sat, blob_counts(20, H, W, rng)], [(H, W)] * 2, 'sat')
    check_equal_to_pass32(model, [np.full(512, 2 ** 32 - 1, np.int64)], [(H, W)], 'sat-all')
