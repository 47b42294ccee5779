#!/usr/bin/env python
"""Timings of analyze.det_seg_scores_sweep (K = 101 score thresholds 0.00:0.01:1.00 x the ten COCO IoU thresholds)
next to one plain engine.eval_images call on the same input and the loop the sweep replaces,
det_seg_scores_batch once per score threshold on the filtered prediction lists.

    python profiles/bench_sweep.py [out.md] [--reps N]

Inputs are synthetic (csrc/synth.cpp): C2 (1,000 images of 500 ground-truth and 500 predicted masks, 1024x1024)
and one C4 image (5,000 x 5,000 masks, 2048x2048).  Scores are seeded and follow the IoU of each prediction's best
match (0.6 IoU + 0.4 uniform noise, float32), so the staircases are not trivial.  Every timing is warm (one call of
each kind first), best of --reps, host clock around calls that end in a stream synchronise; the device span of
the sweep and plain calls is also taken with CUDA events on the current stream.  The two new kernels
(sweep_rows_kernel, sweep_counts_kernel) run inside the library call, where no event can be placed between them;
they are timed from the kernel records of torch.profiler (CUDA activity) in a separate call, and the CUDA-event
spans of the sweep and plain calls bound what the whole sweep adds to one evaluation.  The loop runs
det_seg_scores_batch at IoU 0.5 only, one call per cut-off: covering the ten IoU thresholds of the sweep would take
ten times as many calls, so the loop's time understates the work the sweep replaces.
The card's name and power limit are read in the same run and printed with the numbers."""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = 'unknown'
    return name, limit


def dataset(cfg, n, seed):
    from ampis_b200 import analyze, batch, engine
    from oracle import cocomask as rle
    host = batch.synth(batch.CONFIGS[cfg], n, seed)
    mk = lambda cs: [{'size': [host.h, host.w], 'counts': rle.string_from_counts(c)} for c in cs]
    imgs = [tuple(mk(x) for x in host.image_masks(g)) for g in range(n)]
    gts, prs = [g for g, _ in imgs], [p for _, p in imgs]
    r = engine.eval_images(gts, prs, engine.MODE_IOU)
    rng = np.random.default_rng(seed)
    scores = []
    for g in range(n):
        P = len(prs[g])
        best = np.zeros(P)
        rows = slice(int(r.row_off[g]), int(r.row_off[g + 1]))
        c, s = r.best_col[rows], r.best_score[rows]
        ok = c >= 0
        np.maximum.at(best, c[ok], s[ok])
        scores.append(np.clip(0.6 * best + 0.4 * rng.random(P), 0.0, 1.0).astype(np.float32))
    return gts, prs, scores, analyze


def best_of(fn, reps):
    import torch
    t = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        t.append(time.perf_counter() - t0)
    return min(t)


def device_span(fn, reps):
    import torch
    best = None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        v = a.elapsed_time(b) / 1e3
        best = v if best is None else min(best, v)
    return best


def kernel_times(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and 'sweep_' in e.name:
            k = 'sweep_rows_kernel' if 'sweep_rows' in e.name else 'sweep_counts_kernel'
            out[k] = out.get(k, 0.0) + e.device_time_total / 1e6
    return out


def run(name, cfg, n, seed, reps, loop_reps, lines):
    from ampis_b200 import batch, engine
    gts, prs, scores, A = dataset(cfg, n, seed)
    K = np.round(np.arange(101) * 0.01, 2)
    sweep = lambda: A.det_seg_scores_sweep(gts, prs, K, scores=scores)
    plain = lambda: engine.eval_images(gts, prs, engine.MODE_IOU)

    def loop():
        # images with no prediction above a cut-off cannot be passed to det_seg_scores_batch: they are left out of
        # that cut-off's call (its bookkeeping would raise ZeroDivisionError for them)
        out = []
        for s in K:
            kept = [[p[i] for i in np.flatnonzero(sc > s)] for p, sc in zip(prs, scores)]
            some = [i for i, k in enumerate(kept) if k]
            try:
                out.append(A.det_seg_scores_batch([gts[i] for i in some], [kept[i] for i in some], 0.5) if some else [])
            except ZeroDivisionError:     # an image with no match and nothing unmatched: raised after the evaluation
                out.append(None)
        return out
    sweep(), plain(), loop()
    t_sweep, t_plain = best_of(sweep, reps), best_of(plain, reps)
    d_sweep, d_plain = device_span(sweep, reps), device_span(plain, reps)
    t_loop = best_of(loop, loop_reps)
    kt = kernel_times(sweep)
    res = sweep()
    tp = res['totals'][:, 0, 0]
    lines.append('| %s | %d x %d x %d | %.1f | %.1f | %.1f | %.1f | %.3f | %.3f | %.0f |'
                 % (name, n, len(gts[0]), len(prs[0]), t_sweep * 1e3, t_plain * 1e3, d_sweep * 1e3, d_plain * 1e3,
                    kt.get('sweep_rows_kernel', float('nan')) * 1e3, kt.get('sweep_counts_kernel', float('nan')) * 1e3,
                    t_loop * 1e3))
    print(lines[-1], flush=True)
    print('  TP at IoU 0.5 over score cut-offs 0, 0.5, 1.0: %d %d %d' % (tp[0], tp[50], tp[100]), flush=True)


def main():
    args = sys.argv[1:]
    reps = 5
    if '--reps' in args:
        i = args.index('--reps')
        reps = int(args[i + 1])
        del args[i:i + 2]
    out = args[0] if args else None
    import torch
    name, limit = card()
    lines = ['Measured on %s, power limit %s.' % (name, limit), '',
             'K = 101 score thresholds x T = 10 IoU thresholds.  Times in ms: whole calls (host clock, best of %d), '
             'device span of the call (CUDA events), the two new kernels (torch.profiler, one call), and the loop of '
             '101 det_seg_scores_batch calls at IoU 0.5 on filtered lists (one IoU threshold where the sweep gives ten; '
             'images with nothing kept left out; best of 2).' % reps, '',
             '| input | images x GT x pred | sweep call | eval_images call | sweep device span | eval_images device span '
             '| sweep_rows_kernel | sweep_counts_kernel | batch loop |', '|---|---|---|---|---|---|---|---|---|']
    print(lines[0], flush=True)
    run('C2', 'c2_powder_batch', 1000, 1, reps, 2, lines)
    run('C4', 'c4_spheroidite', 1, 2, reps, 2, lines)
    text = '\n'.join(lines) + '\n'
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, 'w') as f:
            f.write(text)
    print(text)


if __name__ == '__main__':
    main()
