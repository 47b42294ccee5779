#!/usr/bin/env python
"""Timings of powder.satellite_measurements_sweep next to one plain engine.eval_images(..., MODE_SAT) call on the same
input and the loop the sweep replaces, satellite_measurements on the filtered lists of every cell.

    python profiles/bench_sat_sweep.py [out.md] [--reps N]

Input: C3 (200 images of 200 satellites x 2,000 particles, 2048x2048, synthetic, csrc/synth.cpp) with seeded float32
scores on both sides.  Grids: K = L = 21 particle / satellite score thresholds 0.00:0.05:1.00 x T = 10 match thresholds
0.0:0.1:0.9, and a larger one, K = L = 41 (0.000:0.025:1.000) x T = 20 (0.00:0.05:0.95).  Every timing is warm (one
call of each kind first), best of --reps, host clock around calls that end in a stream synchronise; the device span
of the sweep and plain calls is also taken with CUDA events.  The two kernels of the sweep after the join
(sweep_rows_kernel in its satellite form, sat_sweep_counts_kernel) run inside one library call; they are timed from
torch.profiler's kernel records in a separate call.  The loop is what a user runs today per cell: filter the lists,
compute_matches(t) per image (an image with no match raises IndexError in the reference, so it is caught and
counted as such) and satellite_measurements.  It is SUBSAMPLED: a few cells are timed and the time is scaled to the
whole grid.  The card's name and power limit are read in the same run and printed with the numbers."""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from profiles.bench_sweep import best_of, card, device_span  # noqa: E402


def dataset(n, seed):
    from ampis_b200 import batch
    from ampis_b200.applications.powder import PowderSatelliteImage
    from ampis_b200.containers import Instances
    from ampis_b200.structures import InstanceSet, RLEMasks
    from oracle import cocomask as rle
    host = batch.synth(batch.CONFIGS['c3_satellites'], n, seed)
    mk = lambda cs: [{'size': [host.h, host.w], 'counts': rle.string_from_counts(c)} for c in cs]
    rng = np.random.default_rng(seed)
    psi = []
    for g in range(n):
        sats, parts = (mk(x) for x in host.image_masks(g))
        iset = lambda ms: InstanceSet(instances=Instances((host.h, host.w), masks=RLEMasks(ms),
                                                          scores=rng.random(len(ms)).astype(np.float32)))
        psi.append(PowderSatelliteImage(particles=iset(parts), satellites=iset(sats)))
    return psi


def kernel_times(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            k = 'rows' if 'sweep_rows_kernel' in e.name else 'counts' if 'sat_sweep_counts_kernel' in e.name else None
            if k:
                out[k] = out.get(k, 0.0) + e.device_time_total / 1e6
    return out


def loop_cells(psi, cells):
    """satellite_measurements on the filtered lists of each (particle cut-off, satellite cut-off, match threshold)."""
    from ampis_b200.applications import powder
    from ampis_b200.containers import Instances
    from ampis_b200.structures import InstanceSet, RLEMasks
    for ps, ss, mt in cells:
        kept = []
        for im in psi:
            sub = []
            for side, s in ((im.particles, ps), (im.satellites, ss)):
                keep = np.flatnonzero(side.instances.scores > s)
                ms = side.instances.masks.rle
                sub.append(InstanceSet(instances=Instances(side.instances.image_size,
                                                           masks=RLEMasks([ms[i] for i in keep]))))
            p = powder.PowderSatelliteImage(particles=sub[0], satellites=sub[1])
            try:
                p.compute_matches(mt)
                kept.append(p)
            except (IndexError, ValueError):      # the reference raises for an image without a match
                pass
        if kept:
            powder.satellite_measurements(kept, print_summary=False, output_dict=True)


def run(name, psi, pt, st, mt, reps, lines):
    from ampis_b200 import engine
    from ampis_b200.applications import powder
    from ampis_b200.structures import masks_to_rle
    sats = [masks_to_rle(im.satellites.instances) for im in psi]
    parts = [masks_to_rle(im.particles.instances) for im in psi]
    sweep = lambda: powder.satellite_measurements_sweep(psi, pt, st, mt)
    plain = lambda: engine.eval_images(sats, parts, engine.MODE_SAT)
    sweep(), plain()
    t_sweep, t_plain = best_of(sweep, reps), best_of(plain, reps)
    d_sweep, d_plain = device_span(sweep, reps), device_span(plain, reps)
    kt = kernel_times(sweep)
    n_cells = len(pt) * len(st) * len(mt)
    sample = [(pt[len(pt) // 4], st[len(st) // 4], mt[len(mt) // 2]), (pt[len(pt) // 2], st[0], mt[0]),
              (pt[0], st[len(st) // 2], mt[-1])]
    loop_cells(psi, sample[:1])
    t0 = time.perf_counter()
    loop_cells(psi, sample)
    t_loop = (time.perf_counter() - t0) / len(sample) * n_cells
    res = sweep()
    lines.append('| %s | %d x %d x %d | %.1f | %.1f | %.1f | %.1f | %.3f | %.3f | %.0f |'
                 % (name, len(pt), len(st), len(mt), t_sweep * 1e3, t_plain * 1e3, d_sweep * 1e3, d_plain * 1e3,
                    kt.get('rows', float('nan')) * 1e3, kt.get('counts', float('nan')) * 1e3, t_loop))
    print(lines[-1], flush=True)
    print('  sat_frac at the lowest cut-offs, match 0.5: %.4f; matched satellites: %d'
          % (res['sat_frac'][0, 0, len(mt) // 2], res['n_satellites'][0, 0, len(mt) // 2]), flush=True)


def main():
    args = sys.argv[1:]
    reps = 5
    if '--reps' in args:
        i = args.index('--reps')
        reps = int(args[i + 1])
        del args[i:i + 2]
    out = args[0] if args else None
    name, limit = card()
    lines = ['Measured on %s, power limit %s.' % (name, limit), '',
             'C3: 200 images of 200 satellites x 2,000 particles, 2048x2048.  Times in ms: whole calls (host clock, '
             'best of %d), device span of the call (CUDA events), the two kernels after the join (torch.profiler, one '
             'call); the loop of satellite_measurements on filtered lists per cell in s, timed on 3 cells and scaled '
             'to the grid.' % reps, '',
             '| input | K x L x T | sweep call | eval_images call | sweep device span | eval_images device span '
             '| sweep_rows_kernel | sat_sweep_counts_kernel | loop (s, scaled) |', '|---|---|---|---|---|---|---|---|---|']
    print(lines[0], flush=True)
    psi = dataset(200, 3)
    g21, m10 = np.round(np.arange(21) * 0.05, 2), np.round(np.arange(10) * 0.1, 1)
    run('C3', psi, g21, g21, m10, reps, lines)
    g41, m20 = np.round(np.arange(41) * 0.025, 3), np.round(np.arange(20) * 0.05, 2)
    run('C3', psi, g41, g41, m20, reps, lines)
    text = '\n'.join(lines) + '\n'
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, 'w') as f:
            f.write(text)
    print(text)


if __name__ == '__main__':
    main()
