"""Batch (many images per launch) evaluation on one GPU -- the form in which the hot path is
benchmarked and sharded across GPUs.  Not part of the reference API: AMPIS evaluates one image
per Python call (Colab cell 44); this module evaluates a whole shard of images with a handful
of kernel launches and returns device tensors.

Mask table layout of a batch: image by image, ``[rows of image g][columns of image g]`` where
rows are ground-truth masks (or satellites) and columns are predictions (or particles).
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _native as N
from . import engine

COCO_THRESHOLDS = np.arange(0.5, 1.0, 0.05)     # IoU 0.50:0.05:0.95

#: Pipeline: zero the dense matrices of the join on a side stream while the decode kernel runs ('1': fill kernel, '2':
#: device-to-device copies from a block of zeros).  Measured on C2 (profiles/experiments_r02.md): no gain -- the fill
#: kernel takes the SMs it needs from the decode (1.331 vs 1.333 ms per step), the copy engines are slower than the
#: fill (1.505 ms) -- so the default stays in line ('0').
ZERO_AHEAD = os.environ.get('AMPIS_ZERO_AHEAD', '0') != '0'
#: Pipeline: zero the dense matrices on a side stream BESIDE the join's first two passes (load-latency bound)
ZERO_BESIDE_JOIN = os.environ.get('AMPIS_ZERO_BESIDE_JOIN', '1') != '0'
# dense matrices cleared by the decode kernel itself, a share per group of masks (it is bound by instruction issue and
# leaves HBM idle): profiles/experiments_r02.md
ZERO_WITH_DECODE = os.environ.get('AMPIS_ZERO_WITH_DECODE', '1') != '0'
ZERO_BY_COPY = os.environ.get('AMPIS_ZERO_AHEAD', '0') == '2' 

#: synthetic workloads named after BASELINE.json's configs (DESIGN.md "Synthetic data")
CONFIGS = {
    # C1: one 1024x768 powder image, ~300 GT x ~300 predictions
    'c1_powder_example': dict(h=768, w=1024, n_rows=300, n_cols=300, kind=0, median_diam=38.0, sigma_ln=0.45,
                              max_aspect=1.3, sec_median_diam=0.0, mode=engine.MODE_IOU),
    # C2 / C5: 1024x1024, 500 GT x 500 predictions per image
    'c2_powder_batch': dict(h=1024, w=1024, n_rows=500, n_cols=500, kind=0, median_diam=34.0, sigma_ln=0.45,
                            max_aspect=1.3, sec_median_diam=0.0, mode=engine.MODE_IOU),
    # C3: 2048x2048, 200 satellites (rows) x 2000 particles (columns)
    'c3_satellites': dict(h=2048, w=2048, n_rows=200, n_cols=2000, kind=1, median_diam=34.0, sigma_ln=0.45,
                          max_aspect=1.3, sec_median_diam=17.0, mode=engine.MODE_SAT),
    # C4: 2048x2048 spheroidite, 5000 x 5000 small elongated instances
    # (+ the exact area distribution of all instances, one bin per pixel count: equivalent-diameter
    # histograms and the PSD follow from it on the host, d_eq being a function of the area)
    'c4_spheroidite': dict(h=2048, w=2048, n_rows=5000, n_cols=5000, kind=0, median_diam=13.5, sigma_ln=0.6,
                           max_aspect=3.0, sec_median_diam=0.0, mode=engine.MODE_IOU, area_bins=4096,
                           area_bin_width=1),
    # C5: the whole synthetic dataset (10,000 C2 images) split over the ranks of one box -- strong scaling;
    # the all-reduce carries TP/FP/FN and a binned area histogram (size distribution)
    'c5_dataset': dict(h=1024, w=1024, n_rows=500, n_cols=500, kind=0, median_diam=34.0, sigma_ln=0.45,
                       max_aspect=1.3, sec_median_diam=0.0, mode=engine.MODE_IOU, dataset_images=10000,
                       area_bins=4096, area_bin_width=64),
    # crowded frame: 512 x 512 large overlapping instances in 256x256 px (about a quarter of all pairs have
    # overlapping boxes) -- the regime of the tensor-core contraction (engine.intersect_mma), not a
    # BASELINE.json config
    'dense_overlap': dict(h=256, w=256, n_rows=512, n_cols=512, kind=0, median_diam=64.0, sigma_ln=0.3,
                          max_aspect=1.5, sec_median_diam=0.0, mode=engine.MODE_IOU),
}


class HostCSR(object):
    """Run counts of a batch on the host: cnt u32[], cnt_off i64[n], cnt_len i32[n]; every image
    has n_rows + n_cols masks of size (h, w)."""

    def __init__(self, cfg, n_images, cnt, cnt_off, cnt_len):
        self.cfg, self.n_images = cfg, n_images
        self.cnt, self.cnt_off, self.cnt_len = cnt, cnt_off, cnt_len
        self.h, self.w = cfg['h'], cfg['w']
        self.n_rows, self.n_cols = cfg['n_rows'], cfg['n_cols']
        self.per_image = self.n_rows + self.n_cols
        self.n_masks = n_images * self.per_image

    def image_masks(self, g):
        """(rows, cols) of image g as lists of uint32 count arrays."""
        out = []
        for k in range(g * self.per_image, (g + 1) * self.per_image):
            out.append(self.cnt[self.cnt_off[k]:self.cnt_off[k] + self.cnt_len[k]])
        return out[:self.n_rows], out[self.n_rows:]

    def total_runs(self):
        return int(self.cnt_len.sum())

    def slice(self, i0, i1):
        """Images [i0, i1) as a HostCSR of their own (run counts copied out, offsets rebased)."""
        a, b = i0 * self.per_image, i1 * self.per_image
        off, ln = self.cnt_off[a:b], self.cnt_len[a:b]
        if b <= a:
            return HostCSR(self.cfg, 0, np.zeros(0, np.uint32), off.copy(), ln.copy())
        lo, hi = int(off.min()), int((off + ln).max())
        return HostCSR(self.cfg, i1 - i0, self.cnt[lo:hi].copy(), off - lo, ln.copy())


def synth(cfg, n_images, seed, jitter_px=2.0, scale_sigma=0.05, drop_frac=0.08, empty_frac=0.01, n_threads=None):
    """Generate a synthetic batch on the host (synth/synth.cpp -> libampis_synth.so, bench / test data only).  In satellite configs the primaries
    are the particles (columns) and the secondaries the satellites (rows); the generator emits
    primaries first, so the masks are re-ordered to rows-first here."""
    if isinstance(cfg, str):
        cfg = CONFIGS[cfg]
    kind = cfg['kind']
    n_gt, n_sec = (cfg['n_rows'], cfg['n_cols']) if kind == 0 else (cfg['n_cols'], cfg['n_rows'])
    per = n_gt + n_sec
    n = n_images * per
    if n_threads is None:
        n_threads = min(os.cpu_count() or 1, 32)
    cap = max(n * (int(2.5 * cfg['median_diam']) + 8), 1024)
    cnt_off = np.zeros(max(n, 1), np.int64)
    cnt_len = np.zeros(max(n, 1), np.int32)
    while True:
        cnt = np.empty(cap, np.uint32)
        r = N.synth_lib().ampis_synth_batch(int(seed), n_images, cfg['h'], cfg['w'], n_gt, n_sec, kind,
                                      float(cfg['median_diam']), float(cfg['sigma_ln']), float(cfg['max_aspect']),
                                      float(cfg['sec_median_diam']), float(jitter_px), float(scale_sigma),
                                      float(drop_frac), float(empty_frac), int(n_threads),
                                      cnt.ctypes.data_as(C.c_void_p), cap, cnt_off.ctypes.data_as(C.c_void_p),
                                      cnt_len.ctypes.data_as(C.c_void_p))
        if r >= 0:
            cnt = cnt[:r]
            break
        cap = -r
    cnt_off, cnt_len = cnt_off[:n], cnt_len[:n]
    if kind == 1:   # rows (satellites) first
        idx = np.arange(n).reshape(n_images, per)
        idx = np.concatenate([idx[:, n_gt:], idx[:, :n_gt]], axis=1).ravel()
        cnt_off, cnt_len = cnt_off[idx], cnt_len[idx]
    return HostCSR(cfg, n_images, cnt, cnt_off, cnt_len)


class DeviceBatch(object):
    """A HostCSR uploaded once (the "inputs resident in HBM" state of the benchmark)."""

    def __init__(self, host, device=None, dense=False):
        device = device or engine.require_cuda()
        self.host, self.device = host, device
        self.cnt = torch.from_numpy(host.cnt.view(np.int32)).to(device)
        self.cnt_off = torch.from_numpy(host.cnt_off).to(device)
        self.cnt_len = torch.from_numpy(host.cnt_len).to(device)
        self.h = torch.full((max(host.n_masks, 1),), host.h, dtype=torch.int32, device=device)
        self.w = torch.full((max(host.n_masks, 1),), host.w, dtype=torch.int32, device=device)
        self.groups = engine.Groups.interleaved(device, [host.n_rows] * host.n_images,
                                                [host.n_cols] * host.n_images, dense=dense)
        self.mode = host.cfg['mode']


class StepResult(object):
    pass


def eval_step(batch, layout=None, thresholds=COCO_THRESHOLDS, arena=None, rows_out=None,
              sat_thresh=0.5, check=False, fused=None, kernel='rows', sparse=None):
    """One pass of the hot path over a device-resident batch: measure -> paint -> fused
    intersect/arg-max rows -> per-image and total counts.  No host synchronisation when an
    arena is supplied and check is False.  Returns device tensors.  kernel: 'rows' (bbox-culled
    AND+popc; crop tables with many columns per image prune through a grid), 'grid' / 'scan' (crop
    layout: force / forbid the grid), 'mma' (dense tcgen05 contraction).  sparse: an engine.SparseRows
    that receives the non-zero intersections as triplets (crop layout)."""
    layout = engine.DEFAULT_LAYOUT if layout is None else layout
    t = engine.MaskTable(batch.device, batch.host.n_masks, batch.cnt, batch.cnt_off, batch.cnt_len, batch.h,
                         batch.w, layout)
    if fused is None:
        fused = arena is not None
    if fused:
        t.measure_paint(arena)       # one launch: measure + arena allocation + paint
    else:
        t.measure().paint(arena)     # five launches; sizes the arena exactly when none is given
    if kernel in ('mma', 'mma2'):       # 'mma2': CTA pairs (cta_group::2)
        rows = engine.intersect_mma(t, batch.groups, batch.mode, out=rows_out, pair=kernel == 'mma2')
    else:
        assert kernel in ('rows', 'scan', 'mma', 'mma2') or layout == engine.LAYOUT_CROP, 'the grid kernel reads crop tables'
        grid = engine.ColumnGrid(batch.device, batch.groups.n_groups) if kernel == 'grid' else \
            ('scan' if kernel == 'scan' else None)
        rows = engine.intersect_rows(t, batch.groups, batch.mode, out=rows_out, grid=grid, sparse=sparse)
    r = StepResult()
    r.table, r.rows = t, rows
    if batch.mode == engine.MODE_IOU:
        r.counts, r.totals = engine.match_counts(rows, batch.groups, thresholds)
    else:
        r.counts, r.spp_hist = engine.satellite_counts(t, rows, batch.groups, sat_thresh)
    if check:
        t.check()
    return r


class Pipeline(object):
    """The per-batch launch sequence with every buffer allocated up front, so that a step is
    nothing but kernel launches (and can be captured in a CUDA graph):
    fused measure+paint -> intersect rows -> counts."""

    def __init__(self, batch, layout, arena, rows_out=None, thresholds=COCO_THRESHOLDS, totals=None,
                 sat_thresh=0.5, fused=True, kernel='rows', area_hist=None, area_bin_width=64, mma_sort=True,
                 sparse_capacity=None, intervals=True):
        """intervals: when the table goes to the pairs join (and nowhere else), store column-convex masks as one
        interval word per column (engine.MaskTable.measure_paint); False keeps bitmap windows everywhere."""
        dev = batch.device
        self.area_hist, self.area_bin_width = area_hist, area_bin_width     # optional int64 histogram (+=)
        self.batch, self.layout, self.arena, self.fused = batch, layout, arena, fused
        assert kernel in ('rows', 'mma', 'mma2', 'grid', 'scan')
        self.kernel = kernel        # 'rows': bbox-culled AND+popc; 'mma': dense int8 tcgen05 contraction
        # crop layout: candidates through a uniform grid ('grid', or 'rows' with many columns per image)
        # instead of the scan of all columns ('scan'); the entry list is sized once from a dry run
        self.grid, self.sparse, self.pairs = None, None, None
        self.zero_stream = self.zero_done = self.zero_block = None
        if layout == engine.LAYOUT_CROP and (kernel == 'grid' or sparse_capacity is not None or (
                kernel == 'rows' and batch.groups.max_cols >= engine.ROWS_GRID_MIN_COLS)):
            probe = engine.MaskTable(dev, batch.host.n_masks, batch.cnt, batch.cnt_off, batch.cnt_len, batch.h,
                                     batch.w, layout).measure()
            need = engine.ColumnGrid(dev, batch.groups.n_groups).build(probe, batch.groups).capacity
            self.grid = engine.ColumnGrid(dev, batch.groups.n_groups, capacity=need)
            if sparse_capacity is not None:
                self.sparse = engine.SparseRows(dev, sparse_capacity)
            if engine.ROWS_KERNEL == 'pairs':        # the pair list is sized once from a dry run, like the grid
                probe.paint()
                dry = engine.intersect_rows(probe, batch.groups, batch.mode, grid=self.grid)
                self.pairs = engine.PairList(dev, batch.groups.n_rows, dry.pairs.needed())
                del dry
        elif layout == engine.LAYOUT_CROP and kernel == 'scan':
            self.grid = 'scan'
        # the decoded table is read by the join alone (the area histogram and satellite counts read the areas only)
        self.intervals = bool(intervals) and self.pairs is not None and kernel not in ('mma', 'mma2')
        self.mma_sort = mma_sort    # tiles from spatially sorted masks (contracts fewer slabs on large frames)
        if kernel in ('mma', 'mma2'):
            batch.groups.mma_tiles(kernel == 'mma2')
        self.table = engine.MaskTable(dev, batch.host.n_masks, batch.cnt, batch.cnt_off, batch.cnt_len, batch.h,
                                      batch.w, layout)
        g = batch.groups
        nr = max(g.n_rows, 1)
        self.rows = rows_out or engine.RowResult(
            torch.empty(nr, dtype=torch.int32, device=dev), torch.empty(nr, dtype=torch.int32, device=dev),
            torch.empty(nr, dtype=torch.float64, device=dev),
            torch.empty(max(g.imat_size, 1), dtype=torch.int32, device=dev) if g.imat_off is not None else None)
        self.th = torch.from_numpy(np.asarray(thresholds, np.float64)).to(dev)
        self.sat_thresh = sat_thresh
        if batch.mode == engine.MODE_IOU:
            self.counts = torch.empty(max(g.n_groups * self.th.numel() * 3, 1), dtype=torch.int32, device=dev)
            self.totals = totals if totals is not None else torch.zeros(self.th.numel() * 3, dtype=torch.int64,
                                                                       device=dev)
        else:
            self.counts_buf = torch.empty(max(g.n_groups * 4, 1), dtype=torch.int32, device=dev)
            self.counts = None
            self.spp_hist = torch.zeros(64, dtype=torch.int64, device=dev)

    def launch(self, mark=None):
        """Enqueue the kernels on the current stream; `mark(i)` is called between kernel groups."""
        t = self.table
        g = self.batch.groups
        # dense matrices of the join: zeroed on a side stream while the decode kernel (instruction bound, a few % of
        # HBM) runs on the main one -- the rows only patch the non-zero cells afterwards
        zero_ahead = self.pairs is not None and g.imat_off is not None and self.rows.imat is not None and \
            engine.ROWS_KERNEL == 'pairs' and ZERO_AHEAD
        if zero_ahead:
            main = torch.cuda.current_stream()
            if self.zero_stream is None:
                self.zero_stream, self.zero_done = torch.cuda.Stream(device=self.batch.device), torch.cuda.Event()
            self.zero_stream.wait_stream(main)          # whoever used the matrices before is done
            with torch.cuda.stream(self.zero_stream):
                if ZERO_BY_COPY:
                    # device-to-device copies from a block of zeros: work for the copy engines, which idle during the
                    # decode, instead of a fill kernel that competes with it for the SMs
                    if self.zero_block is None:
                        self.zero_block = torch.zeros(16 << 20, dtype=torch.int32, device=self.batch.device)
                    zb = self.zero_block.numel()
                    for o in range(0, g.imat_size, zb):
                        k = min(zb, g.imat_size - o)
                        self.rows.imat[o:o + k].copy_(self.zero_block[:k], non_blocking=True)
                else:
                    self.rows.imat[:g.imat_size].zero_()
                self.zero_done.record()
        if mark: mark(0)
        zeroed = self.zero_done if zero_ahead else None
        if self.fused:
            if mark: mark(1)
            with_decode = ZERO_WITH_DECODE and not zero_ahead and self.pairs is not None and g.imat_off is not None \
                and self.rows.imat is not None and engine.ROWS_KERNEL == 'pairs' and self.kernel not in ('mma', 'mma2')
            t.measure_paint(self.arena, zero=self.rows.imat[:g.imat_size] if with_decode else None,
                            intervals=self.intervals)
            if with_decode and t.zeroed:
                zeroed = True
        else:
            t.measure()
            if mark: mark(1)
            t.paint(self.arena)
        if mark: mark(2)
        if self.kernel in ('mma', 'mma2'):
            engine.intersect_mma(t, self.batch.groups, self.batch.mode, out=self.rows, sort=self.mma_sort,
                                 pair=self.kernel == 'mma2')
        else:
            side = None
            if ZERO_BESIDE_JOIN and zeroed is None and self.pairs is not None and g.imat_off is not None:
                if self.zero_stream is None:
                    self.zero_stream = torch.cuda.Stream(device=self.batch.device)
                side = self.zero_stream
            engine.intersect_rows(t, self.batch.groups, self.batch.mode, out=self.rows, grid=self.grid,
                                  sparse=self.sparse, pairs=self.pairs, zeroed=zeroed,
                                  zero_stream=side)
        if mark: mark(3)
        if self.batch.mode == engine.MODE_IOU:
            engine.match_counts(self.rows, self.batch.groups, self.th, totals=self.totals, counts=self.counts)
        else:
            self.counts, _ = engine.satellite_counts(t, self.rows, self.batch.groups, self.sat_thresh,
                                                     hist=self.spp_hist, counts=self.counts_buf)
        if self.area_hist is not None:
            engine.hist_u32(t.area[:t.n], 0, self.area_bin_width, self.area_hist.numel(), hist=self.area_hist)
        if mark: mark(4)


def arena_chunks_needed(batch, layout):
    """Number of uint4 chunks the packed-mask arena needs for a DeviceBatch: one measurement
    pass on the GPU and a read-back (used to size the workspace before the timed region)."""
    t = engine.MaskTable(batch.device, batch.host.n_masks, batch.cnt, batch.cnt_off, batch.cnt_len, batch.h,
                         batch.w, layout)
    t.measure()
    return int(t.bits_off[t.n].item())
