"""A/B of the interval windows of the crop step (profiles/intervals_r01.md): the batch.Pipeline of a config built with
the form on and off, both replayed from CUDA graphs and alternated over several rounds in one process; then one
torch.profiler pass per form for the per-kernel times; and the exact arena bytes of either form, counted on the host
from the run counts (--count-only needs no GPU).

    python profiles/bench_intervals.py --out DIR [--configs c2,c1,c3,c4] [--rounds 7] [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {  # name -> (config, images per step, sparse output)
    'c2': ('c2_powder_batch', 1000, False),
    'c1': ('c1_powder_example', 1000, False),
    'c3': ('c3_satellites', 1000, False),
    'c4': ('c4_spheroidite', 40, True),
}
KERNELS = ('rle_flat_crop_kernel', 'pairs_from_grid', 'pair_intersect_flat', 'rows_from_pairs')


def interval_stats(host):
    """Masks, masks stored as intervals, and the arena bytes of the bitmap-only and of the mixed form, computed from
    the run counts with the rules of rle_flat.cu (fallback masks and empty masks stay bitmaps)."""
    H, W = host.h, host.w
    ln = host.cnt_len.astype(np.int64)
    n = len(ln)
    first = np.repeat(np.cumsum(ln) - ln, ln)
    k = np.arange(int(ln.sum())) - first                     # index of the count inside its mask
    c = host.cnt[np.repeat(host.cnt_off, ln) + k].astype(np.int64)
    mid = np.repeat(np.arange(n), ln)
    cs = np.cumsum(c)
    end = cs - np.repeat(cs[np.cumsum(ln) - ln] - c[np.cumsum(ln) - ln], ln)   # run end inside the mask
    one = (k % 2 == 1) & (c > 0) & (end <= H * W)
    s = end[one] - c[one]
    x, ys = s // H, s % H
    yl = ys + c[one] - 1
    span = yl >= H
    z = c[np.flatnonzero(one) - 1]
    bad = span | ((k[one] >= 3) & (z < ys))
    m = mid[one]
    area = np.bincount(m, c[one], n)
    x0 = np.full(n, 1 << 40); np.minimum.at(x0, m, x)
    x1 = np.full(n, -1); np.maximum.at(x1, m, (end[one] - 1) // H)
    y0 = np.full(n, 1 << 40); np.minimum.at(y0, m, np.where(span, 0, ys))
    y1 = np.full(n, -1); np.maximum.at(y1, m, np.where(span, H - 1, yl))
    convex = np.bincount(m, bad, n) == 0
    has = area > 0
    width = np.where(has, x1 - x0 + 1, 0)
    bands = np.where(has, y1 // 32 - y0 // 32 + 1, 0)
    bm_words = np.where(has, width * bands, 0)
    bm = (bm_words + 3) // 4
    # the tile test is made on the window the mask gets: an interval window of <= 512 columns fits even where the
    # bitmap would not
    iv = has & convex & ~(((ln + 1) // 2 > 256) | (H > 65536)) & (width <= 512)
    mixed = np.where(iv, (width + 3) // 4, bm)
    return dict(masks=int(n), interval_masks=int(iv.sum()), bitmap_arena_bytes=int(16 * bm.sum()),
                interval_arena_bytes=int(16 * mixed.sum()))


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip()


class Arm(object):
    def __init__(self, dev, intervals, sparse):
        import torch
        from ampis_b200 import batch, engine
        self.arena = torch.empty(4 * max(batch.arena_chunks_needed(dev, engine.LAYOUT_CROP), 1), dtype=torch.int32,
                                 device='cuda')
        self.pipe = batch.Pipeline(dev, engine.LAYOUT_CROP, self.arena, intervals=intervals,
                                   sparse_capacity=32 * dev.groups.n_rows if sparse else None)
        assert self.pipe.intervals == intervals
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                self.launch()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.launch()

    def launch(self):
        p = self.pipe
        if p.batch.mode == 0:
            p.totals.zero_()
        else:
            p.spp_hist.zero_()
        p.launch()

    def time(self, reps):
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.graph.replay()
        e0.record()
        for _ in range(reps):
            self.graph.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def kernels(self, reps=5):
        import torch
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                self.launch()
            torch.cuda.synchronize()
        tot = {}
        for e in prof.events():
            if e.device_type.name != 'CUDA':
                continue
            key = next((k for k in KERNELS if k in e.name), None)
            if key:
                tot[key] = tot.get(key, 0.0) + e.device_time / 1000.0 / reps
        return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--configs', default='c2,c1,c3,c4')
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--count-only', action='store_true', help='arena bytes only (host, no GPU)')
    a = ap.parse_args()
    from ampis_b200 import batch
    res = {}
    if not a.count_only:
        res['gpu'] = gpu_info()
        print('GPU (name, power limit, max SM clock):', res['gpu'], flush=True)
    for name in a.configs.split(','):
        cfg, n_img, sparse = CONFIGS[name]
        host = batch.synth(cfg, n_img, 1)
        r = res[name] = dict(config=cfg, images=n_img, **interval_stats(host))
        print(name, json.dumps({k: v for k, v in r.items()}), flush=True)
        if a.count_only:
            continue
        import torch
        dev = batch.DeviceBatch(host, dense=not sparse)
        on, off = Arm(dev, True, sparse), Arm(dev, False, sparse)
        # the exact chunks the decode reserved, against the host count
        r['gpu_arena_bytes_on'] = 16 * int(on.pipe.table.cursor.item())
        r['gpu_arena_bytes_off'] = 16 * int(off.pipe.table.cursor.item())
        t_on, t_off = [], []
        for _ in range(a.rounds):
            t_off.append(off.time(a.reps))
            t_on.append(on.time(a.reps))
        r['ms_on'], r['ms_off'] = t_on, t_off
        r['kernels_on'], r['kernels_off'] = on.kernels(), off.kernels()
        print(name, 'ms/step off %.4f [%.4f, %.4f]  on %.4f [%.4f, %.4f]  (median, min, max of %d rounds x %d replays)'
              % (np.median(t_off), min(t_off), max(t_off), np.median(t_on), min(t_on), max(t_on), a.rounds, a.reps))
        print(name, 'kernels off', json.dumps(r['kernels_off']))
        print(name, 'kernels on ', json.dumps(r['kernels_on']), flush=True)
        del on, off, dev
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'intervals.json'), 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
