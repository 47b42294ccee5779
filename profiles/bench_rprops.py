#!/usr/bin/env python
"""Timings of InstanceSet.compute_rprops with every supported key (the 15 scalar keys and the 14 added with
moments to order 3, hole fill, Crofton perimeter, Feret diameter and the box images), next to the
numpy/scipy restatement of skimage 0.18.3 (oracle/ampis_ref.py for the fifteen, tests/_rprops_ref.py for
the rest) on the same masks.

    python profiles/bench_rprops.py [out.md]
    python profiles/bench_rprops.py --intensity [out.md]

--intensity times the ten intensity keys instead, with a seeded uint16 intensity image of the frame's size, next
to the numpy restatement of tests/_rprops_intensity_ref.py.  The kernel column times the native entry points only;
the image upload and its transpose on the device (torch) are part of the measurement step, not of that column.

Inputs are synthetic (csrc/synth.cpp): the 100 first predictions of a C1-like image (1024x768, as
profiles/bench_functions.py uses) and one C4-like image of 5,000 masks (2048x2048).  Per input it reports
  * the whole call (warm, best of 3, ends in a device synchronise),
  * every kernel launch timed with CUDA events (sum per kernel, from a separate instrumented call),
  * the measurement step (table + kernels + copies back) and the per-mask host formation of the properties,
  * the oracle on decoded box crops (frames decoded outside the timed region; on the C4 image a sample of
    500 masks, scaled to 5,000).
The card's name and power limit are read in the same run and printed with the numbers."""
import json
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


def main():
    import torch
    from ampis_b200 import batch as B, engine as E, structures as S
    from ampis_b200.containers import Instances
    from oracle import ampis_ref as R
    from oracle import cocomask as rle
    from tests import _rprops_intensity_ref as MI
    from tests import _rprops_ref as M
    rle.build()
    torch.cuda.set_device(0)
    name, limit = card()
    intensity = '--intensity' in sys.argv
    args = [a for a in sys.argv[1:] if a != '--intensity']
    keys = list(S.InstanceSet.RPROPS_INTENSITY_KEYS if intensity else S.InstanceSet.RPROPS_GPU_KEYS)
    new_keys = keys[15:]
    rows = []

    def image(cfg_name, seed):
        host = B.synth(dict(B.CONFIGS[cfg_name]), 1, seed)
        _, c = host.image_masks(0)
        size = [host.h, host.w]
        return [{'size': size, 'counts': rle.string_from_counts(x)} for x in c], (host.h, host.w)

    def kernel_times(masks, img):
        """CUDA-event time of every launch of one region_properties call, summed per entry point (ms)."""
        real = E.N.call
        ev = []

        def timed(nm, *args):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            real(nm, *args)
            b.record()
            ev.append((nm, a, b))
        E.N.call = timed
        try:
            S.region_properties(masks, keys, img)
        finally:
            E.N.call = real
        torch.cuda.synchronize()
        out = {}
        for nm, a, b in ev:
            out[nm] = out.get(nm, 0.0) + a.elapsed_time(b)
        return out

    def best(fn, n=3):
        t = 1e30
        for _ in range(n):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            t = min(t, time.perf_counter() - t0)
        return t

    c1, size1 = image('c1_powder_example', 11)
    c4, size4 = image('c4_spheroidite', 13)
    for label, masks, size, sample in (('C1-like, 100 masks', c1[:100], size1, 100),
                                       ('C4-like, %d masks' % len(c4), c4, size4, 500)):
        n = len(masks)
        img = np.random.default_rng(5).integers(0, 65536, size, dtype=np.uint16) if intensity else None
        iset = S.InstanceSet(instances=Instances(size, masks=S.RLEMasks(masks), boxes=np.zeros((n, 4)),
                                                 class_idx=np.arange(n)))
        iset.compute_rprops(keys=keys, intensity_image=img)  # warm-up: library load, CUDA context
        t_call = best(lambda: iset.compute_rprops(keys=keys, intensity_image=img))
        need = {x for k in keys for x in S._MEASUREMENTS_OF[k]}
        t_meas = best(lambda: E.region_measurements_for(masks, need, img))
        t_props = best(lambda: S.region_properties(masks, keys, img))
        kt = kernel_times(masks, img)
        # oracle on box crops of a sample (decode + crop outside the timed region)
        crops = []
        for mk in masks[:sample]:
            d = rle.decode(mk).astype(bool)
            if d.any():
                r, c = np.nonzero(d)
                sl = (slice(max(r.min() - 1, 0), r.max() + 2), slice(max(c.min() - 1, 0), c.max() + 2))
                crops.append((d[sl], img[sl]) if intensity else
                             np.pad(d[r.min():r.max() + 1, c.min():c.max() + 1], 1))
        t0 = time.perf_counter()
        for d in crops:
            if intensity:
                MI.regionprops_intensity(d[0], d[1], keys)
            else:
                R.regionprops_one(d)
                M.regionprops_more(d, new_keys)
        t_oracle = (time.perf_counter() - t0) * n / sample
        row = {'input': label, 'gpu': name, 'power_limit': limit, 'compute_rprops_ms': 1e3 * t_call,
               'region_properties_ms': 1e3 * t_props, 'measurements_ms': 1e3 * t_meas,
               'host_formation_ms': 1e3 * (t_props - t_meas), 'kernels_ms': kt,
               'kernels_total_ms': sum(kt.values()), 'oracle_ms': 1e3 * t_oracle,
               'oracle_note': 'measured on %d masks, scaled to %d' % (sample, n) if sample != n else 'all masks'}
        rows.append(row)
        print(json.dumps(row), flush=True)
    if args:
        with open(args[0], 'w') as f:
            f.write('# compute_rprops with the ten intensity keys, uint16 image\n\n' if intensity else
                    '# compute_rprops with all %d supported keys\n\n' % len(keys))
            f.write('Measured on %s, power limit %s, by `profiles/bench_rprops.py`. Times in ms. Whole call: warm, '
                    'best of 3. Kernels: CUDA events around every launch of one call, summed per entry point. '
                    'Host formation: `region_properties` minus the measurement step. Oracle: numpy/scipy '
                    'restatement of skimage 0.18.3 on box crops, one run on the host cores of the same machine.\n\n'
                    % (name, limit))
            f.write('| input | compute_rprops | measurements (table, kernels, copies) | kernels (events) | '
                    'host formation | oracle |\n|---|---|---|---|---|---|\n')
            for r in rows:
                f.write('| %s | %.1f | %.1f | %.2f | %.1f | %.0f (%s) |\n'
                        % (r['input'], r['compute_rprops_ms'], r['measurements_ms'], r['kernels_total_ms'],
                           r['host_formation_ms'], r['oracle_ms'], r['oracle_note']))
            f.write('\nKernel time per entry point (ms, CUDA events):\n\n| input | ' +
                    ' | '.join(sorted(rows[0]['kernels_ms'])) + ' |\n|---|' + '---|' * len(rows[0]['kernels_ms']) + '\n')
            for r in rows:
                f.write('| %s | ' % r['input'] + ' | '.join('%.3f' % r['kernels_ms'].get(k, 0.0)
                                                          for k in sorted(rows[0]['kernels_ms'])) + ' |\n')


if __name__ == '__main__':
    main()
