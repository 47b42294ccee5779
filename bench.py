#!/usr/bin/env python
"""bench.py -- throughput of the mask-evaluation hot path on B200 (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--layout crop|span|full] [--config NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...        # the reference's CPU algorithm on the host cores

A step is one pass of the hot path over one batch of synthetic images (BASELINE.json
configs[1]: 1,000 images of 1024x1024 with 500 GT x 500 predicted masks each, per GPU):
RLE run counts resident in HBM -> per-mask measurements -> bit-packed masks -> bbox-pruned
intersections (dense int32 G x P matrix out) + per-GT arg-max IoU -> TP/FP/FN at IoU
0.50:0.05:0.95 per image and in total (+ one NCCL all-reduce of the totals when N > 1).

The headline (`value`, `roofline`, `e2e`) is the PRODUCT path: bounding-box windows (crop layout), flat decode,
candidate-pair join -- what the drop-in functions run.  `full_layout` repeats the step in the canonical two-pass
full-frame layout of SURVEY 8d (its decode kernel is the HBM-saturation proof), `span_layout` in the linear culled
layout; all three give bit-identical totals (asserted).  `e2e` goes through the C ABI from host buffers
(ampis_eval_images_host), `e2e_api` through the Python drop-in signature (dict lists -> det_seg_scores_batch),
`c5_strong` is the 10,000-image dataset of configs[4] split over the ranks.  Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'mask-pair IoUs/sec (GT x pred mask pairs matched and scored, IoU 0.50:0.95)'
UNIT = 'pairs/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='c2_powder_batch')
    ap.add_argument('--images', type=int, default=1000, help='images per GPU per step')
    ap.add_argument('--layout', default='crop', choices=['full', 'span', 'crop'],
                    help='layout of the HEADLINE run: crop = bounding-box windows (the product path, the cropped '
                         'accounting of SURVEY 8d); span = linear culled storage (first..last 1-pixel of each mask); '
                         'full = canonical full-frame packed masks (the two-pass accounting of SURVEY 8d).  The other '
                         'two are measured beside it unless --no-span')
    ap.add_argument('--sub', type=int, default=0, help='images per launch group (0 = auto)')
    ap.add_argument('--kernel', default='rows', choices=['rows', 'mma', 'mma2', 'grid', 'scan'],
                    help='intersection kernel: rows = bbox-culled AND+popc (default; crop layout with >= 384 '
                         'columns per image prunes through a uniform grid); grid / scan = crop layout with the grid '
                         'forced / forbidden; mma = dense int8 tcgen05 contraction (for crowded images, e.g. '
                         '--config dense_overlap)')
    ap.add_argument('--sparse', action='store_true',
                    help='crop layout: no dense G x P matrix, the non-zero intersections come out as triplets '
                         '(bbox-pruned sparse IoU, the C4 form of SURVEY 8d)')
    ap.add_argument('--mma-sort', action='store_true',
                    help='with --kernel mma: cut the tiles from spatially sorted masks (fewer slabs contracted; the '
                         'default contracts the full pixel range so that the tensor roofline counts executed work)')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-api', action='store_true', help='skip the e2e_api leg (Python drop-in signature)')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-c5', action='store_true', help='skip the c5_strong sub-measurement (10,000-image dataset)')
    ap.add_argument('--no-check', action='store_true', help='skip the oracle check of a 2-image sample')
    ap.add_argument('--graph', action='store_true', help='(default for the culled headline run) replay each step from a CUDA graph')
    ap.add_argument('--no-graph', action='store_true', help='launch the kernels of the headline run one by one instead of replaying a captured graph')
    ap.add_argument('--span-sub', type=int, default=0, help='images per launch group of the secondary runs')
    ap.add_argument('--unfused', action='store_true', help='separate measure / scan / paint launches')
    ap.add_argument('--no-span', action='store_true', help='skip the secondary layouts')
    ap.add_argument('--e2e-chunk', type=int, default=0,
                    help='images per C-ABI call of the e2e leg (0 = about 250,000 masks per call, equal calls)')
    ap.add_argument('--api-images', type=int, default=200, help='images per call of the e2e_api leg')
    ap.add_argument('--cpu-images', type=int, default=0)
    ap.add_argument('--cpu-threads', type=int, default=0, help='reference arm: worker processes (0 = all cores)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last step of the headline run computed to '
                         'DIR/<name>.npy (float64; a seeded sample of arrays longer than 2^19 elements), so that two '
                         'builds can be compared output for output on identical inputs')
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def tensor_peak_tops():
    """int8 tensor peak in TOP/s: twice the measured dense bf16 rate (the i8 pipe is 2x bf16 on sm_100;
    nominal 4.5 POP/s).  Burst figure: the contraction draws ~230 W and holds 1965 MHz, it never
    reaches the power cap that defines the sustained bf16 number."""
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return 2.0 * float(d['bf16_tflops']), '2 x measured bf16 burst (MEASURED_PEAKS.json bf16_tflops)'
    return 2.0 * 1590.0, '2 x fallback bf16 burst (B200_PROFILING.md)'


def gpu_local_cpus(index):
    """CPUs NVML reports as local to GPU `index` (its NUMA node), restricted to the ones this process may use;
    None when NVML cannot say."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_words = ((os.cpu_count() or 64) + 63) // 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (int(wd) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        return cpus or None
    except Exception:
        return None


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw'

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(',')]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'note': 'nvidia-smi unavailable'}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 6] or [r for _, r in self.rows if len(r) >= 6]
        if not rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'note': 'no samples'}
        sm = sorted(float(r[0]) for r in rows)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith('active') for r in rows)]
        out = {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(rows[0][1]), 'reasons': reasons, 'samples': len(rows)}
        try:
            out['power_w_max'] = max(float(r[6]) for r in rows)
        except Exception:
            pass
        return out


def cpu_seconds_per_task(cfg_name, cfg):
    """Seconds one (image, threshold) task of the reference port takes on one core (measured), used to bound the
    CPU samples: G x ceil(P / 80) rleIou calls that re-parse 81 strings each grow with G x P."""
    if cfg['mode'] != 0:
        return 2.5
    return max(0.05, 0.75 * (cfg['n_rows'] * cfg['n_cols']) / 250000.0)


def workload_config(args, cfg, images_per_gpu):
    """The `config` object -- the WORKLOAD, identical (keys and values) in both arms; how an arm runs it is in `run`."""
    sat = cfg['mode'] != 0
    return {'workload': '%s: %dx%d px, %d x %d masks per image' % (args.config, cfg['w'], cfg['h'], cfg['n_rows'],
                                                                   cfg['n_cols']),
            'images_per_gpu_per_step': int(images_per_gpu),
            'thresholds': 'satellite overlap > 0.5' if sat else 'IoU 0.50:0.05:0.95',
            'l2': 'every kernel of a step streams its inputs and outputs once (run counts, window arena, dense '
                  'matrices: ~0.3 MB or more per image, hundreds of MB per step), larger than the 126 MB L2; no '
                  'explicit flush'}


# ------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's algorithm (oracle port) on the host cores
# ------------------------------------------------------------------------------------------
def _cpu_task(args):
    gt, pr, th, mode = args
    from oracle import ampis_ref as R
    if mode == 0:
        r = R.det_seg_scores(gt, pr, th)
        return len(r['det_tp']), len(r['det_fp']), len(r['det_fn'])
    r = R.rle_satellite_match(pr, gt, th)
    return len(r['satellite_matches']), 0, len(r['satellites_unmatched'])


def cpu_images(cfg_name, n_img, seed):
    """n_img synthetic images as lists of compressed-RLE dicts (what the reference consumes).  The generator is
    libampis_synth.so; the product library is never loaded in this arm."""
    from ampis_b200 import batch
    from oracle import cocomask as rle
    host = batch.synth(cfg_name, n_img, seed)
    out = []
    for g in range(n_img):
        rows, cols = host.image_masks(g)
        size = [host.h, host.w]
        out.append(([{'size': size, 'counts': rle.string_from_counts(c)} for c in rows],
                    [{'size': size, 'counts': rle.string_from_counts(c)} for c in cols]))
    return host, out


def cpu_run(pool, images, thresholds, mode):
    tasks = [(gt, pr, float(t), mode) for gt, pr in images for t in thresholds]
    t0 = time.perf_counter()
    res = pool.map(_cpu_task, tasks, chunksize=1) if pool is not None else [_cpu_task(t) for t in tasks]
    return time.perf_counter() - t0, res


def reference_arm(args):
    """--impl reference: per step, `n_img` images of the same synthetic workload through the
    reference's loops (analyze.py:149-172 + 315-327 restated in oracle/ampis_ref.py over the C
    restatement of pycocotools), one det_seg_scores call per IoU threshold as a user of the
    reference does, on all host cores (or --cpu-threads).  kind = "port": pycocotools itself is not
    installable here (DESIGN.md)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    from ampis_b200 import batch
    from oracle import cocomask
    cocomask.build()
    cores = args.cpu_threads or (os.cpu_count() or 1)
    cfg = batch.CONFIGS[args.config]
    thresholds = list(batch.COCO_THRESHOLDS) if cfg['mode'] == 0 else [0.5]
    per_task = cpu_seconds_per_task(args.config, cfg)
    budget = min(8.0, 200.0 / max(args.steps + args.warmup, 1))
    n_img = args.cpu_images or max(1, int(cores * budget / (per_task * len(thresholds))))
    host, images = cpu_images(args.config, n_img, 777)
    pairs = n_img * host.n_rows * host.n_cols
    if cores == 1:          # what the reference itself does: one serial loop (analyze.py:149-172)
        for _ in range(args.warmup):
            cpu_run(None, images[:1], thresholds[:1], cfg['mode'])
        t = sum(cpu_run(None, images, thresholds, cfg['mode'])[0] for _ in range(args.steps))
    else:
        with mp.get_context('fork').Pool(cores) as pool:
            for _ in range(args.warmup):
                cpu_run(pool, images[:max(1, min(n_img, cores // len(thresholds)))], thresholds, cfg['mode'])
            t = sum(cpu_run(pool, images, thresholds, cfg['mode'])[0] for _ in range(args.steps))
    value = pairs * args.steps / t
    sample = '%d synthetic %s image(s) per step, one call per IoU threshold (%d calls per image), oracle port of the ' \
             'reference loops, %d process(es)' % (n_img, args.config, len(thresholds), cores)
    strong = 'dataset_images' in cfg
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * t / args.steps, 'higher_is_better': True,
        'scaling': 'strong' if strong else 'weak', 'vs_baseline': None, 'dtype': 'u32', 'data': 'synthetic',
        'images_per_s': n_img * args.steps / t,
        'config': workload_config(args, cfg, cfg['dataset_images'] // max(args.gpus, 1) if strong else args.images),
        'run': {'sample_images_per_step': n_img, 'processes': cores, 'thresholds_per_image': len(thresholds),
                'note': 'a bounded sample of the workload in `config`; the reference evaluates one threshold per '
                        'det_seg_scores call, so the 10-threshold sweep re-matches every image 10 times'},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample,
                         'thresholds_per_image': len(thresholds)},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
KERNELS = ['measure+scan', 'paint', 'rows', 'counts']


class LayoutRun(object):
    """Inputs of one rank resident in HBM + the workspace for one storage layout."""

    def __init__(self, args, dev, hosts, layout, cfg, sparse=False):
        import torch
        from ampis_b200 import batch, engine
        self.layout, self.dev, self.cfg = layout, dev, cfg
        self.sub = max(h.n_images for h in hosts)
        self.n_images = sum(h.n_images for h in hosts)
        self.fused = not args.unfused
        self.subs = [batch.DeviceBatch(h, dev, dense=not (sparse and layout == engine.LAYOUT_CROP)) for h in hosts]
        self.total_runs = sum(b.host.total_runs() for b in self.subs)
        need = [batch.arena_chunks_needed(b, layout) for b in self.subs]
        self.stored_chunks = sum(need)
        self.arena = torch.empty(4 * max(need), dtype=torch.int32, device=dev)
        n_rows = max(b.groups.n_rows for b in self.subs)
        self.rows_out = engine.RowResult(torch.empty(n_rows, dtype=torch.int32, device=dev),
                                         torch.empty(n_rows, dtype=torch.int32, device=dev),
                                         torch.empty(n_rows, dtype=torch.float64, device=dev),
                                         torch.empty(max(max(b.groups.imat_size for b in self.subs), 1),
                                                     dtype=torch.int32, device=dev))
        self.thresholds = batch.COCO_THRESHOLDS
        n_tot = len(self.thresholds) * 3
        bins = cfg.get('area_bins', 0)
        # one int64 payload for the all-reduce: TP/FP/FN x thresholds [+ binned area histogram]
        self.payload = torch.zeros(n_tot + bins, dtype=torch.int64, device=dev)
        self.totals = self.payload[:n_tot]
        self.area_hist = self.payload[n_tot:] if bins else None
        self.kernel = args.kernel
        self.mode = cfg['mode']
        self.pipes = [batch.Pipeline(b, layout, self.arena, self.rows_out, self.thresholds, self.totals,
                                     fused=self.fused, kernel=args.kernel, mma_sort=args.mma_sort,
                                     area_hist=self.area_hist, area_bin_width=cfg.get('area_bin_width', 64),
                                     sparse_capacity=(32 * b.groups.n_rows if sparse and
                                                      layout == engine.LAYOUT_CROP else None)) for b in self.subs]
        if self.mode != 0:
            for p in self.pipes[1:]:
                p.spp_hist = self.pipes[0].spp_hist
        self.graph = None
        self.sparse_pairs = None
        self.kt_passes = 1

    def launch_all(self, record=None):
        import torch
        self.payload.zero_()
        if self.mode != 0:
            self.pipes[0].spp_hist.zero_()
        for p in self.pipes:
            if record is None:
                p.launch()
            else:
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
                p.launch(lambda i, ev=ev: ev[i].record())
                record.append(ev)

    def capture(self):
        """Capture one step's launch sequence in a CUDA graph (launch-bound for small launch groups)."""
        import torch
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.launch_all()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.launch_all()

    def step(self, world, dist, record=None):
        """one pass over the rank's batch; `record` collects the CUDA events around each kernel group"""
        if self.graph is not None and record is None:
            self.graph.replay()
        else:
            self.launch_all(record)
        if world > 1:       # TP/FP/FN x thresholds (or the satellites-per-particle histogram): the only exchange
            dist.all_reduce(self.payload if self.mode == 0 else self.pipes[0].spp_hist)
        return self.totals

    def timed(self, steps, warmup, world, dist, sync):
        import torch
        for _ in range(max(warmup, 3)):
            self.step(world, dist)
        sync()
        record = []
        use_graph = self.graph is not None
        if use_graph:     # per-kernel shares come from an instrumented pass outside the timed region
            for _ in range(2):
                self.launch_all(record)
            sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            self.step(world, dist, None if use_graph else record)
        e1.record()
        sync()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=self.dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        kt = np.zeros(4)
        for ev in record:
            for i in range(4):
                kt[i] += ev[i].elapsed_time(ev[i + 1])
        self.kt_passes = 2 if use_graph else steps
        self.pipes[-1].table.check()      # arena large enough, RLE well-formed (after the timed region)
        if self.pipes[0].sparse is not None:
            cnt = [int(p.sparse.count.item()) for p in self.pipes]
            assert all(c <= p.sparse.capacity for c, p in zip(cnt, self.pipes)), 'sparse triplet list overflowed'
            self.sparse_pairs = sum(cnt)
        for p in self.pipes:
            if getattr(p.grid, 'capacity', None):
                assert p.grid.needed() <= p.grid.capacity, 'grid entry list overflowed'
            if p.pairs is not None:
                assert p.pairs.needed() <= p.pairs.capacity, 'candidate pair list overflowed'
        if self.mode != 0:      # satellites: per-image counts summed over the batch + the global histogram
            c = sum(p.counts.cpu().numpy().sum(axis=0) for p in self.pipes)
            return float(ms.item()), kt, np.concatenate([c, self.pipes[0].spp_hist.cpu().numpy()[:8]]).reshape(1, -1)
        return float(ms.item()), kt, self.totals.cpu().numpy().reshape(-1, 3)

    def kernels_per_sub(self):
        """Kernel launches of one launch group (memset nodes not counted)."""
        from ampis_b200 import engine
        grid = getattr(self.pipes[0].grid, 'capacity', None)
        if self.kernel in ('mma', 'mma2'):
            rows = 2                                    # contraction + rows from the dense matrices
        elif grid and self.pipes[0].pairs is not None:
            rows = 4                                    # grid build, join, AND+popc per pair, per-row arg-max
        elif grid:
            rows = 2                                    # grid build, grid rows kernel
        else:
            rows = 1
        if not self.fused:
            paint = 5                                   # measure, 3 x scan, paint
        elif self.layout == engine.LAYOUT_CROP and engine.CROP_DECODE == 'flat':
            paint = 2                                   # flat decode + its fallback list kernel
        else:
            paint = 1
        return paint + rows + 1 + (1 if self.area_hist is not None else 0)

    def describe(self, args):
        grid = getattr(self.pipes[0].grid, 'capacity', None)
        from ampis_b200 import engine
        kern = args.kernel
        if self.layout == engine.LAYOUT_CROP and kern in ('rows', 'grid'):
            kern = ('pairs (grid + three-pass join)' if self.pipes[0].pairs is not None else 'grid') if grid else 'scan'
        return {'layout': layout_name(self.layout), 'intersection_kernel': kern + ('+sorted tiles' if args.kernel in (
                    'mma', 'mma2') and args.mma_sort else ''),
                'decode_kernel': ('flat' if engine.CROP_DECODE == 'flat' else 'lane groups') if self.layout == engine.LAYOUT_CROP
                else 'fused measure+paint', 'images_per_launch': self.sub, 'sparse_output': bool(self.pipes[0].sparse),
                'cuda_graph': self.graph is not None, 'cuda_graph_error': getattr(self, 'graph_error', None), 'runs_per_mask': self.total_runs / max(self.n_images * (
                    self.cfg['n_rows'] + self.cfg['n_cols']), 1)}


def layout_name(layout):
    from ampis_b200 import engine
    return {engine.LAYOUT_FULL: 'full', engine.LAYOUT_SPAN: 'span', engine.LAYOUT_CROP: 'crop'}[layout]


def roofline_of(args, run, ms, kt, steps):
    """Roofline of the dominant kernel of a layout run -- like for like: the bytes THAT kernel has to move in THAT
    layout over its measured time -- plus the whole step against the accounting of its own layout, and (separately,
    never as a fraction) how many times the canonical two-pass roofline of SURVEY 8d the step runs at."""
    from ampis_b200 import engine
    cfg = run.cfg
    peak, peak_src = peaks()
    n_img = run.n_images
    per_image = cfg['n_rows'] + cfg['n_cols']
    B_m = ((cfg['h'] * cfg['w'] + 127) // 128) * 16
    pairs_img = cfg['n_rows'] * cfg['n_cols']
    stored = run.stored_chunks * 16.0
    dense_out = run.pipes[0].sparse is None
    out_bytes = 4.0 * n_img * pairs_img if dense_out else 24.0 * (run.sparse_pairs or 0)
    lay = layout_name(run.layout)
    # per-kernel algorithmic bytes: decode = 4R in + stored bytes out; intersection = every stored mask read once +
    # the intersections out (full layout: stored = N * B_m, SURVEY 8d's canonical per-kernel figure)
    alg = {'paint': 4.0 * run.total_runs + stored, 'rows': stored + out_bytes}
    # the flat decode kernel also clears the dense matrices (a share per group of masks): those bytes are written by
    # it, not by the rows, which then only patch the non-zero cells
    zero_in_decode = bool(dense_out and getattr(run.pipes[0].table, 'zeroed', False))
    if zero_in_decode:
        alg = {'paint': 4.0 * run.total_runs + stored + out_bytes, 'rows': float(stored)}
    canonical_img = 4.0 * run.total_runs / n_img + 2 * per_image * B_m + 4 * pairs_img + 8 * per_image + 32 * cfg['n_rows']
    own_img = 4.0 * run.total_runs / n_img + 2.0 * stored / n_img + out_bytes / n_img + 8 * per_image + 32 * cfg['n_rows']
    dom = 'paint' if kt[1] >= kt[2] else 'rows'
    launches = len(run.subs)
    dur_ms = kt[KERNELS.index(dom)] / (run.kt_passes * launches)
    achieved = alg[dom] / launches / (dur_ms / 1e3) / 1e9
    traffic, traffic_detail = None, None
    tp = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tp):
        traffic_detail = json.load(open(tp)).get('%s/%s/%s' % (args.config, lay, dom))
        if traffic_detail:
            traffic = traffic_detail['bytes_per_image'] * n_img / launches
    step_s = ms / 1e3 / steps
    share = {k: float(v) for k, v in zip(KERNELS, kt / max(kt.sum(), 1e-30))}
    step = {'accounting': {'full': 'canonical two-pass full-frame (SURVEY 8d)',
                           'crop': 'cropped (SURVEY 8d, C4 form): 4R + 2 x window bytes + output + 8(G+P) + 32G',
                           'span': '4R + 2 x span bytes + output + 8(G+P) + 32G'}[lay],
            'output': 'dense G x P matrix' if dense_out else 'sparse triplets',
            'bytes_per_image': own_img, 'achieved': own_img * n_img / step_s / 1e9, 'unit': 'GB/s',
            'frac': own_img * n_img / step_s / 1e9 / peak}
    canonical = {'bytes_per_image': canonical_img, 'x_canonical_roofline': canonical_img * n_img / step_s / 1e9 / peak,
                 'note': 'images/s of this step over the images/s at which the canonical two-pass full-frame '
                         'accounting would saturate HBM -- a speed-up over that design point, NOT a roofline '
                         'fraction: culled layouts move far fewer bytes'}
    if run.kernel in ('mma', 'mma2') and dom == 'rows':
        tpeak, tsrc = tensor_peak_tops()
        ops = 2.0 * pairs_img * cfg['h'] * cfg['w'] * n_img / launches
        ach = ops / (dur_ms / 1e3) / 1e12
        return {'bound': 'tensor', 'kernel': 'intersect_mma_kernel (+ rows_from_imat_kernel)', 'achieved': ach,
                'peak': tpeak, 'unit': 'TOP/s', 'frac': ach / tpeak, 'traffic': None, 'peak_source': tsrc,
                'algorithmic_ops_per_launch': ops, 'launch_ms': dur_ms, 'step': step, 'canonical': canonical,
                'kernel_share': share}
    pk = 'rle_paint_kernel' if args.unfused else 'rle_measure_paint_kernel'
    rk = 'intersect_rows_kernel'
    if run.layout == engine.LAYOUT_CROP:
        grid = getattr(run.pipes[0].grid, 'capacity', None)
        rk = ('grid_build + pairs_from_grid + pair_intersect + rows_from_pairs kernels' if run.pipes[0].pairs is not None
              else 'grid_build + intersect_rows_grid kernels') if grid else 'intersect_rows_crop_kernel'
        if not args.unfused:
            pk = 'rle_flat_crop_kernel (+ rle_measure_paint_list_kernel)' if engine.CROP_DECODE == 'flat' else \
                'rle_measure_paint_crop_kernel'
    return {'bound': 'hbm', 'kernel': {'paint': pk, 'rows': rk}[dom], 'layout': lay,
            'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic,
            'traffic_detail': traffic_detail, 'peak_source': peak_src,
            'algorithmic_bytes_per_launch': alg[dom] / launches, 'launch_ms': dur_ms,
            'dense_matrices_cleared_by': ('decode kernel' if zero_in_decode else 'rows (fill)') if dense_out else None,
            'bound_note': {'full': 'pure write stream of full frames: HBM-bound; the measured peak is a COPY (half reads, '
                                   'half writes), a write-only stream sustains slightly more, hence frac a little above 1',
                           'span': 'culled storage: the kernels are bound by instruction issue / load latency, not by '
                                   'these bytes',
                           'crop': 'culled storage: the decode kernel is bound by instruction issue (ncu: issue slots '
                                   '~72 % busy, DRAM 35 % of peak with the dense matrices it clears), the join by load latency -- these are the bytes the kernel '
                                   'MUST move; the fraction says how far from bandwidth-bound it is '
                                   '(profiles/kernels_r02.md)'}[lay],
            'step': step, 'canonical': canonical, 'kernel_share': share}


def layout_summary(args, run, ms, kt, steps, job_images):
    cfg = run.cfg
    out = {'value': job_images * cfg['n_rows'] * cfg['n_cols'] * steps / (ms / 1e3), 'unit': UNIT,
           'images_per_s': job_images * steps / (ms / 1e3), 'ms_per_step': ms / steps,
           'stored_bytes_per_image': run.stored_chunks * 16 / run.n_images, 'run': run.describe(args),
           'roofline': roofline_of(args, run, ms, kt, steps)}
    if run.sparse_pairs is not None:
        out['nonzero_pairs_per_image'] = run.sparse_pairs / run.n_images
    return out


def oracle_sample_check(run):
    """After the timed region: the per-image counts the GPU produced for two images of the run against the CPU
    oracle on the same inputs (one rleIou call over all pairs of an image + the reference's matcher rules;
    tests/test_oracle.py pins that form to the literal loops).  Checker only -- nothing here is timed."""
    from oracle import cocomask as rle
    rle.build()
    host = run.subs[0].host
    picks = sorted(set([0, host.n_images - 1]))
    counts = run.pipes[0].counts.cpu().numpy()
    counts = counts.reshape(host.n_images, -1, 3) if run.mode == 0 else counts.reshape(host.n_images, 4)
    for g in picks:
        rows, cols = host.image_masks(g)
        size = [host.h, host.w]
        R_ = [{'size': size, 'counts': rle.string_from_counts(c)} for c in rows]
        C_ = [{'size': size, 'counts': rle.string_from_counts(c)} for c in cols]
        iou = np.ascontiguousarray(rle.iou(C_, R_, np.zeros(len(R_), np.uint8)).T)       # [rows, cols]
        if run.mode == 0:
            best = iou.argmax(axis=1)
            top = iou[np.arange(len(R_)), best]
            for t, th in enumerate(run.thresholds):
                m = top > th
                want = [int(m.sum()), len(C_) - len(np.unique(best[m])), int((~m).sum())]
                assert counts[g, t].tolist() == want, ('oracle check failed', g, float(th), counts[g, t].tolist(), want)
        else:
            inter = np.zeros(iou.shape, np.uint32)
            for s_, p_ in zip(*np.nonzero(iou)):
                inter[s_, p_] = rle.merge_area(R_[s_], C_[p_], intersect=True)
            with np.errstate(invalid='ignore', divide='ignore'):
                score = inter / rle.area(R_).astype(np.uint32)[:, None]
            best = score.argmax(axis=1)
            m = score[np.arange(len(R_)), best] > 0.5
            want = [int(m.sum()), int((~m).sum()), len(np.unique(best[m])), len(C_)]
            assert counts[g].tolist() == want, ('oracle check failed', g, counts[g].tolist(), want)
    return {'images_checked': len(picks), 'against': 'oracle: rleIou over all pairs of the image + the reference\'s '
            'matcher rules, TP/FP/FN at every threshold', 'equal': True}


DUMP_CAP = 1 << 19      # elements kept per dumped array: 4 MB in float64, ten arrays at most


def dump_outputs(run, out_dir):
    """--dump-outputs: what the last timed step of the headline run computed, as its caller receives it from the
    device, one float64 DIR/<name>.npy each: `totals` (TP/FP/FN per threshold) or `spp_hist` (satellites per
    particle), per-image `counts`, per-mask `area`, per-row `best_col` / `best_inter` / `best_score`, and the
    intersections -- `imat` (the dense G x P matrices) or, with --sparse, `sparse_row` / `sparse_col` /
    `sparse_inter` sorted by row and column.  The launch groups of a step share the row and matrix buffers, so the
    per-row arrays and the intersections hold the images of the last group (all images when the step is one launch,
    as for the default C2 batch).  An array of more than DUMP_CAP elements is cut to the elements at DUMP_CAP
    positions drawn with a fixed seed (the same positions for every array of that length)."""
    import torch
    last, g = run.pipes[-1], run.pipes[-1].batch.groups
    u32 = lambda t: t.long() & 0xffffffff                     # uint32 payload in an int32 tensor
    out = {}
    if run.mode == 0:
        n_th = len(run.thresholds)
        out['totals'] = run.totals.view(n_th, 3)
        out['counts'] = torch.cat([p.counts[:p.batch.groups.n_groups * n_th * 3].view(-1, n_th, 3)
                                   for p in run.pipes])
    else:
        out['spp_hist'] = run.pipes[0].spp_hist
        out['counts'] = torch.cat([p.counts for p in run.pipes])
    if run.area_hist is not None:
        out['area_hist'] = run.area_hist
    out['area'] = torch.cat([u32(p.table.area[:p.table.n]) for p in run.pipes])
    out['best_col'] = last.rows.best_col[:g.n_rows]
    out['best_inter'] = u32(last.rows.best_inter[:g.n_rows])
    out['best_score'] = last.rows.best_score[:g.n_rows]
    if last.sparse is not None:
        out['sparse_row'], out['sparse_col'], out['sparse_inter'] = last.sparse.triplets()
    elif last.rows.imat is not None and g.imat_off is not None:
        out['imat'] = last.rows.imat[:g.imat_size]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        if t.numel() > DUMP_CAP:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_CAP, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + '.npy'), t.to(torch.float64).cpu().numpy())


def strings_of(batch_dev):
    """Compressed RLE strings of a DeviceBatch (GPU encoder; setup, untimed): (uint8 blob, int32 lengths)."""
    import torch
    from ampis_b200 import engine
    from ampis_b200 import _native as N
    _p, _s = engine._p, engine._stream
    b = batch_dev
    n = b.host.n_masks
    lens = b.cnt_len.cpu().numpy().astype(np.int64)
    choff = np.zeros(n + 1, np.int64)
    np.cumsum(7 * lens, out=choff[1:])
    d_choff = torch.from_numpy(choff).to(b.device)
    chars = torch.empty(max(int(choff[-1]), 1), dtype=torch.uint8, device=b.device)
    chlen = torch.empty(max(n, 1), dtype=torch.int32, device=b.device)
    N.call('ampis_rle_string_encode', _p(b.cnt), _p(b.cnt_off), _p(b.cnt_len), n, _p(chars), _p(d_choff),
           _p(chlen), _s())
    ln = chlen[:n].cpu().numpy().astype(np.int64)
    buf = chars.cpu().numpy()
    start = np.cumsum(ln) - ln
    keep = np.repeat(choff[:-1] - start, ln) + np.arange(int(ln.sum()))
    return buf[keep], ln.astype(np.int32)


def run_e2e_cabi(args, hosts, dev, cfg, world, dist, sync):
    """The same metric END TO END through the C ABI from HOST buffers: per step, every chunk of images goes through
    ONE ampis_eval_images_host call -- compressed RLE strings lying back to back in pinned host memory (what the
    reference API receives, already serialised), their lengths and the per-image sizes in; H2D, string decode, flat
    decode, grids, join, AND+popc, arg-max, TP/FP/FN at all thresholds on the device; per-row matches, areas and the
    counts back on the host.  Two host threads with a stream and workspaces each keep two calls in flight, so the
    upload of one chunk overlaps the evaluation of the other."""
    import torch
    from ampis_b200 import batch
    from ampis_b200 import _native as N
    lib = N.lib()
    mode = cfg['mode']
    thr = np.ascontiguousarray(batch.COCO_THRESHOLDS.astype(np.float64)) if mode == 0 else np.zeros(0)
    chunks = []
    for hst in hosts:
        # calls of ~250,000 masks but at least 80 images, all of the same size.  Measured (images per call / calls in
        # flight -> ms per step): C2 125/4 6.6, 250/4 1.88, 250/6 1.80, 334/4 1.90, 500/3 1.94, 1000/2 2.31;
        # C4 (10,000 masks per image, 160 images) 23/2 3.84, 80/3 1.98, 160/2 2.27; C3 100/3 0.94, 200/2 1.05
        e2e_chunk = args.e2e_chunk
        if e2e_chunk <= 0:
            want = max(80, 250000 // max(hst.per_image, 1))
            n_calls = max(1, -(-hst.n_images // want))
            e2e_chunk = max(1, -(-hst.n_images // n_calls))
        for s0 in range(0, hst.n_images, e2e_chunk):
            part = hst.slice(s0, min(s0 + e2e_chunk, hst.n_images))
            blob, ln = strings_of(batch.DeviceBatch(part, dev))
            ni = part.n_images
            pin = lambda a: torch.from_numpy(a).pin_memory().numpy()          # page-locked arrays: DMA endpoints
            ch = {'blob': torch.from_numpy(blob).pin_memory(), 'len': pin(ln), 'n_images': ni,
                  'n_rows': np.full(ni, part.n_rows, np.int32), 'n_cols': np.full(ni, part.n_cols, np.int32),
                  'h': np.full(ni, part.h, np.uint32), 'w': np.full(ni, part.w, np.uint32)}
            R, n = ni * part.n_rows, part.n_masks
            # two sets of outputs: the calls of consecutive steps may be in flight together
            ch['out'] = [dict(best_col=pin(np.empty(R, np.int32)), best_inter=pin(np.empty(R, np.uint32)),
                              best_score=pin(np.empty(R)), area=pin(np.empty(n, np.uint32)),
                              status=pin(np.empty(n, np.int32)), counts=np.zeros((ni, max(len(thr), 1), 3), np.int32),
                              totals=np.zeros((max(len(thr), 1), 3), np.int64)) for _ in range(2)]
            ch['ptr'] = (C.c_void_p * 1)(ch['blob'].data_ptr())
            ch['h2d'] = int(blob.nbytes + 4 * n + 32 * ni + 8 * len(thr))
            ch['d2h'] = int(16 * R + 8 * n + 12 * len(thr) * ni + 24 * len(thr))
            chunks.append(ch)
    # calls in flight: three quarters of the calls of two steps (the main thread queues one step ahead).  Measured on
    # C2 (4 calls per step): 4 / 6 / 8 workers = 1.88 / 1.82 / 6.1 ms per step -- with a worker for every queued call
    # the kernels of step i+1 share the GPU with those of step i, whose totals the main thread is waiting for
    # ... and never more spinning threads than this rank's share of the host cores (8 ranks on a 32-core host: 3;
    # with 6 each the 8-rank step took 5.54 ms instead of 5.0, profiles/scaling_r02.md)
    n_workers = int(os.environ.get('AMPIS_E2E_WORKERS', '0')) or \
        max(2, min(6, (3 * 2 * len(chunks)) // 4, (os.cpu_count() or 8) // max(world, 1) - 1))
    # AMPIS_STRINGS_CONTIGUOUS (1) [+ AMPIS_WAIT_BLOCKING (2): measured per box, profiles/scaling_r02.md]
    call_flags = 1 | (2 if os.environ.get('AMPIS_E2E_BLOCKING', '0') == '1' else 0)
    workers = [{'stream': torch.cuda.Stream(device=dev),
                'd_ws': torch.empty(1 << 24, dtype=torch.uint8, device=dev),
                'h_ws': torch.empty(1 << 22, dtype=torch.uint8, pin_memory=True)} for _ in range(n_workers)]
    pa = lambda a: a.ctypes.data_as(C.c_void_p)

    def one(ch, wk, o):
        need, found, crowded = C.c_int64(0), C.c_int64(0), C.c_int32(0)
        for _ in range(8):
            rc = lib.ampis_eval_images_host(ch['ptr'], pa(ch['len']), ch['n_images'], pa(ch['n_rows']), pa(ch['n_cols']),
                                            pa(ch['h']), pa(ch['w']), mode, call_flags, -1.0,
                                            C.c_void_p(wk['d_ws'].data_ptr()), wk['d_ws'].numel(),
                                            C.c_void_p(wk['h_ws'].data_ptr()), wk['h_ws'].numel(),
                                            pa(o['best_col']), pa(o['best_inter']), pa(o['best_score']),
                                            pa(o['area']), None, None, pa(o['status']),
                                            pa(thr) if len(thr) else None, len(thr),
                                            pa(o['counts']) if len(thr) else None,
                                            pa(o['totals']) if len(thr) else None, C.byref(found), C.byref(crowded),
                                            C.byref(need), C.c_void_p(wk['stream'].cuda_stream))
            if rc != N.ENOSPC:
                break
            if need.value < 0:
                wk['h_ws'] = torch.empty(int(-need.value * 5 // 4), dtype=torch.uint8, pin_memory=True)
            else:
                wk['stream'].synchronize()
                wk['d_ws'] = None
                wk['d_ws'] = torch.empty(int(need.value * 5 // 4), dtype=torch.uint8, device=dev)
        N.check(rc, 'ampis_eval_images_host')

    # Every worker owns a stream, its workspaces and a queue of calls; a step is the calls of all its chunks.  The
    # steps are PIPELINED: the calls of step i+1 are already queued while step i is being evaluated, so its upload
    # overlaps that evaluation (as a data loader prefetches the next batch); the main thread collects the totals of a
    # step as soon as its calls have returned (and all-reduces them when N > 1).
    import queue
    jobs = queue.Queue()                      # one queue: whichever worker is free takes the next call

    def worker(w):
        torch.cuda.set_device(dev)
        while True:
            job = jobs.get()
            if job is None:
                return
            ch, o, done = job
            try:
                one(ch, workers[w], o)
                assert not o['status'].any()
                done.put(o['totals'].copy())
            except Exception as ex:          # surface in the main thread
                done.put(ex)

    threads = [threading.Thread(target=worker, args=(w,), daemon=True) for w in range(n_workers)]
    for t_ in threads:
        t_.start()
    red = torch.zeros(max(3 * len(thr), 4), dtype=torch.int64, device=dev)

    parity = [0]

    def submit():
        done = queue.Queue()
        for ch in chunks:
            jobs.put((ch, ch['out'][parity[0]], done))
        parity[0] ^= 1
        return done

    def collect(done):
        tot = 0
        for _ in chunks:
            r = done.get()
            if isinstance(r, Exception):
                raise r
            tot = tot + r
        if world > 1:           # the same exchange as the device-resident step
            red[:tot.size] = torch.from_numpy(np.ascontiguousarray(tot).reshape(-1)).to(dev)
            dist.all_reduce(red)
            return red.cpu().numpy()[:tot.size].reshape(tot.shape)
        return tot

    def run_steps(k):
        pending = [submit()]
        tot = None
        for i in range(k):
            if i + 1 < k:
                pending.append(submit())         # one step ahead
            tot = collect(pending.pop(0))
        return tot

    run_steps(max(args.warmup, 3))             # also sizes the workspaces
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    tot = run_steps(args.steps)
    e1.record()
    sync()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    for _ in threads:
        jobs.put(None)
    for t_ in threads:
        t_.join()
    n_img = sum(c_['n_images'] for c_ in chunks)
    pairs = world * n_img * cfg['n_rows'] * cfg['n_cols']
    return {'value': pairs * args.steps / (ms / 1e3), 'unit': UNIT, 'h2d_bytes_per_step': sum(c_['h2d'] for c_ in chunks),
            'd2h_bytes_per_step': sum(c_['d2h'] for c_ in chunks), 'ms_per_step': ms / args.steps,
            'images_per_s': world * n_img * args.steps / (ms / 1e3), 'wall_ms_per_step': wall_ms / args.steps,
            'calls_per_step': len(chunks), 'images_per_call': max(c_['n_images'] for c_ in chunks), 'calls_in_flight': n_workers,
            'pipelining': 'the calls of step i+1 are queued while step i is evaluated (its upload overlaps that '
                          'evaluation); the totals of every step are read on the host before the step counts as done',
            'entry': 'ampis_eval_images_host (C ABI, include/ampis_b200.h): strings back to back in pinned host memory '
                     '(AMPIS_STRINGS_CONTIGUOUS), one upload / one download / one synchronisation per call; host '
                     'read of the totals every step'}, (tot if len(thr) else None)


def run_e2e_api(args, host, cfg, world, dist, sync, dev):
    """The same metric through the PYTHON drop-in signature: lists of COCO RLE dicts per image (what a user of the
    reference holds, Colab cell 44) -> analyze.det_seg_scores_batch -> the list of eleven-key dicts
    analyze.py:329-339 returns, on the host.  Everything a caller pays is inside the timed region: the C marshaller's
    walk over the dicts, the gather of the strings into pinned memory, H2D, kernels, D2H, the numpy bookkeeping."""
    import torch
    from ampis_b200 import analyze, batch
    from ampis_b200.applications import powder
    n_img = min(args.api_images, host.n_images)
    part = host.slice(0, n_img)
    blob, ln = strings_of(batch.DeviceBatch(part, dev))
    off = np.zeros(len(ln) + 1, np.int64)
    np.cumsum(ln, out=off[1:])
    raw = blob.tobytes()
    # every dict with its own size list and its own int objects, as pycocotools' encode / a json file hand them out
    hs, ws = np.full(len(ln), part.h), np.full(len(ln), part.w)
    masks = [{'size': [int(hs[i]), int(ws[i])], 'counts': raw[off[i]:off[i + 1]]} for i in range(len(ln))]
    per = part.per_image
    rows = [masks[g * per:g * per + part.n_rows] for g in range(n_img)]
    cols = [masks[g * per + part.n_rows:(g + 1) * per] for g in range(n_img)]
    if cfg['mode'] == 0:
        call = lambda: analyze.det_seg_scores_batch(rows, cols, 0.5)
        name = 'analyze.det_seg_scores_batch(list of GT dict lists, list of prediction dict lists, 0.5) -> list of ' \
               '11-key dicts (reference: analyze.py:226-339 in the loop of Colab cell 44)'
    else:
        def call():
            out = []
            for s_, p_ in zip(rows, cols):
                try:
                    out.append(powder._rle_satellite_match(p_, s_, 0.5))
                except IndexError:
                    out.append(None)
            return out
        name = 'powder._rle_satellite_match(particles, satellites, 0.5) per image (reference: powder.py:28-112)'
    for _ in range(2):
        res = call()
    sync()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = call()
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    dt = float(dt.item())
    assert len(res) == n_img
    return {'value': world * n_img * cfg['n_rows'] * cfg['n_cols'] * args.steps / dt, 'unit': UNIT,
            'images_per_s': world * n_img * args.steps / dt, 'ms_per_call': 1e3 * dt / args.steps,
            'images_per_call': n_img, 'call': name,
            'h2d_bytes_per_step': int(blob.nbytes + 4 * len(ln)),
            'timed_with': 'host clock around the call (it takes and returns host objects), max over ranks',
            'note': 'bounded by the host: per call %d dicts are walked by the C marshaller, their strings gathered into '
                    'pinned memory, and %d result dicts are cut from the flat arrays in Python' % (len(ln), n_img)}


def run_c5_strong(args, dev, rank, world, dist, sync):
    """BASELINE.json configs[4]: the 10,000-image dataset split over the ranks (STRONG scaling), crop layout, one
    all-reduce of TP/FP/FN + the 4096-bin area histogram per pass."""
    from ampis_b200 import batch, engine
    cfg = batch.CONFIGS['c5_dataset']
    total = cfg['dataset_images']
    mine = total // world + (1 if rank < total % world else 0)
    by_imat = max(1, int(4e9 // (4 * cfg['n_rows'] * cfg['n_cols'])))
    hosts = [batch.synth('c5_dataset', min(by_imat, mine - s0), 5_000_011 * (rank + 1) + s0)
             for s0 in range(0, mine, by_imat)]
    sub_args = argparse.Namespace(**dict(vars(args), kernel='rows', unfused=False, mma_sort=False))
    run = LayoutRun(sub_args, dev, hosts, engine.LAYOUT_CROP, cfg)
    passes = args.steps
    ms, kt, tot = run.timed(passes, args.warmup, world, dist, sync)
    hist = run.area_hist.cpu().numpy()
    return {'workload': 'c5_dataset: %d images of 1024x1024 px, 500 x 500 masks, split over %d GPU(s)' % (total, world),
            'scaling': 'strong', 'images': total, 'images_per_gpu': mine, 'passes_timed': passes,
            'ms_per_pass': ms / passes, 'images_per_s': total * passes / (ms / 1e3),
            'value': total * cfg['n_rows'] * cfg['n_cols'] * passes / (ms / 1e3), 'unit': UNIT, 'layout': 'crop',
            'all_reduce': 'int64 x %d: TP/FP/FN at 10 thresholds + %d-bin area histogram' % (run.payload.numel(),
                                                                                            cfg['area_bins']),
            'totals_tp_fp_fn_at_0.50': tot[0].tolist(), 'area_histogram_instances': int(hist.sum())}


def main():
    args = parse()
    if args.impl == 'reference':
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    from ampis_b200 import batch, engine
    from ampis_b200 import _native as N

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    # pinned staging buffers should live on the GPU's own NUMA node: run on its CPUs before anything is allocated
    cpus = gpu_local_cpus(local)
    if cpus:
        try:
            os.sched_setaffinity(0, cpus)
        except OSError:
            cpus = None
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    N.lib()

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cfg = batch.CONFIGS[args.config]
    strong = 'dataset_images' in cfg
    if strong:          # a fixed dataset split over the ranks (strong scaling); every rank gets its share
        total_images = cfg['dataset_images']
        args.images = total_images // world + (1 if rank < total_images % world else 0)
    job_images = cfg['dataset_images'] if strong else world * args.images        # images all ranks evaluate per step
    layouts = {'full': engine.LAYOUT_FULL, 'span': engine.LAYOUT_SPAN, 'crop': engine.LAYOUT_CROP}
    layout = layouts[args.layout]
    per_image = cfg['n_rows'] + cfg['n_cols']
    B_m = ((cfg['h'] * cfg['w'] + 127) // 128) * 16

    def auto_sub(lay, forced=0):
        if forced:
            return forced
        by_imat = max(1, int(4e9 // (4 * cfg['n_rows'] * cfg['n_cols'])))          # dense matrices <= 4 GB per launch
        if lay == engine.LAYOUT_FULL:
            return max(1, min(args.images, int(12e9 // (per_image * B_m)), by_imat))       # ~12 GB arena
        if args.sparse and lay == engine.LAYOUT_CROP:
            by_imat = args.images
        # culled layouts: the arena is small, so all images of the step go out in ONE launch of each kernel (bounded by
        # 4 GB of dense matrices) -- at 91 or 250 images per launch the short kernels of this step were mostly ramp and
        # tail (profiles/kernels_r02.md: 2.62 / 1.74 / 1.36 ms per 1,000 C2 images at 91 / 250 / 1,000 per launch)
        return min(args.images, by_imat)

    # ---- synthetic inputs: generated ONCE per rank, cut into launch groups per layout
    t0 = time.time()
    host_all = batch.synth(args.config, args.images, 1_000_003 * (rank + 1))
    t_gen = time.time() - t0

    def hosts_for(sub):
        return [host_all.slice(s0, min(s0 + sub, args.images)) for s0 in range(0, args.images, sub)]

    sampler = ClockSampler(local) if rank == 0 else None       # samples cover warm-up + timed steps
    wall0 = time.time()
    sparse = args.sparse and layout == engine.LAYOUT_CROP
    run = LayoutRun(args, dev, hosts_for(auto_sub(layout, args.sub)), layout, cfg, sparse=sparse)
    # the step is a fixed sequence of ~12 short kernels: replayed from a CUDA graph (batch.Pipeline launches are
    # capturable), which removes ~30 us of launch gaps per step; --no-graph launches them one by one
    if (args.graph or (args.kernel in ('rows', 'grid') and layout == engine.LAYOUT_CROP)) and not args.no_graph:
        try:
            run.capture()
        except Exception as ex:          # fall back to plain launches (and say so in the JSON line)
            if args.graph:
                raise
            run.graph = None
            run.graph_error = repr(ex)[:200]
            torch.cuda.synchronize()
    ms, kt, final_totals = run.timed(args.steps, args.warmup, world, dist, sync)
    wall1 = time.time()
    clocks = sampler.stop(wall0, wall1) if sampler else None
    head = layout_summary(args, run, ms, kt, args.steps, job_images)
    launches = int(args.steps * len(run.subs) * run.kernels_per_sub())
    check = None if (args.no_check or rank != 0) else oracle_sample_check(run)
    if args.dump_outputs and rank == 0:
        dump_outputs(run, args.dump_outputs)

    # ---- end to end: C ABI from host buffers, and the Python drop-in signature
    e2e = e2e_api = None
    culled = args.kernel in ('rows', 'grid')
    if not args.no_e2e and culled:
        e2e, e2e_tot = run_e2e_cabi(args, [b.host for b in run.subs], dev, cfg, world, dist, sync)
        if e2e_tot is not None:
            assert np.array_equal(np.asarray(e2e_tot).reshape(-1, 3), final_totals), 'C-ABI end-to-end totals differ'
        if not args.no_api:
            e2e_api = run_e2e_api(args, run.subs[0].host, cfg, world, dist, sync, dev)

    # ---- the other storage layouts, measured beside the headline one: same inputs, bit-identical totals
    del run.arena, run.rows_out
    run.pipes, run.subs = [], []
    torch.cuda.empty_cache()
    others = {}
    if not args.no_span and culled and not args.sparse:
        for name in ('full', 'span', 'crop'):
            if layouts[name] == layout:
                continue
            orun = LayoutRun(args, dev, hosts_for(auto_sub(layouts[name], args.span_sub)), layouts[name], cfg)
            if args.graph:
                orun.capture()
            oms, okt, otot = orun.timed(args.steps, args.warmup, world, dist, sync)
            assert np.array_equal(otot, final_totals), '%s and %s layouts disagree' % (name, args.layout)
            others[name + '_layout'] = layout_summary(args, orun, oms, okt, args.steps, job_images)
            others[name + '_layout']['note'] = {
                'full': 'same inputs, bit-identical totals; the canonical two-pass full-frame layout of SURVEY 8d -- its '
                        'decode kernel is the HBM-saturation proof (a pure write stream at the copy peak), but 97 % of '
                        'what it writes are zeros: not the layout the drop-in functions use',
                'span': 'same inputs, bit-identical totals; only first..last 1-pixel of each mask is stored',
                'crop': 'same inputs, bit-identical totals; only the bounding-box window of each mask is stored'}[name]
            del orun
            torch.cuda.empty_cache()

    c5 = None
    if not args.no_c5 and args.config == 'c2_powder_batch' and culled and not args.sparse:
        c5 = run_c5_strong(args, dev, rank, world, dist, sync)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    out = {
        'metric': METRIC, 'value': head['value'], 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True,
        'scaling': 'strong' if strong else 'weak', 'vs_baseline': None, 'dtype': 'u32', 'data': 'synthetic',
        'images_per_s': head['images_per_s'],
        'config': workload_config(args, cfg, args.images),
        'run': dict(head['run'], parallelism='images sharded over %d GPU(s); one int64 all-reduce of TP/FP/FN%s per step'
                    % (world, ' + %d-bin area histogram' % cfg['area_bins'] if cfg.get('area_bins') else ''),
                    stored_bytes_per_image=head['stored_bytes_per_image']),
        'roofline': head['roofline'],
        'gpu_launches': launches,
    }
    if 'nonzero_pairs_per_image' in head:
        out['run']['nonzero_pairs_per_image'] = head['nonzero_pairs_per_image']
    if e2e:
        out['e2e'] = e2e
    if e2e_api:
        out['e2e_api'] = e2e_api
    out.update(others)
    if c5:
        out['c5_strong'] = c5
    out[('totals_tp_fp_fn_at_0.50' if cfg['mode'] == 0 else 'sat_matched_unmatched_satellited_particles+spp_hist')] = \
        final_totals[0].tolist()
    out['oracle_check'] = check
    out['clocks'] = clocks
    out['setup_s'] = {'synthesize': t_gen, 'numa': ('process bound to the %d CPUs local to GPU %d before pinned '
                      'allocations' % (len(cpus), local)) if cpus else 'NVML gave no CPU affinity; not bound'}
    if not args.no_cpu:
        out['cpu_baseline'] = cpu_baseline(args)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline(args):
    """The reference's CPU algorithm (oracle port) on bounded samples of the same workload, each in a fresh process
    (no CUDA context is forked): one step of the --impl reference arm on ALL host cores sized to ~15 s, and one on a
    SINGLE thread (what the reference itself does: analyze.py:149-172 is a serial loop) on one image."""
    cores = os.cpu_count() or 1
    from ampis_b200 import batch
    cfg = batch.CONFIGS[args.config]
    n_thr = len(batch.COCO_THRESHOLDS) if cfg['mode'] == 0 else 1
    per_task = cpu_seconds_per_task(args.config, cfg)
    env = dict(os.environ, RANK='0', WORLD_SIZE='1', CUDA_VISIBLE_DEVICES='')
    try:
        os.sched_setaffinity(0, range(cores))        # the CPU arm may use every core again
    except OSError:
        pass

    def arm(n_img, threads):
        r = subprocess.run([sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '1',
                            '--warmup', '0', '--config', args.config, '--cpu-images', str(n_img), '--cpu-threads',
                            str(threads)], env=env, capture_output=True, text=True, timeout=900)
        line = [l for l in r.stdout.splitlines() if l.startswith('{')]
        if r.returncode != 0 or not line:
            return {'value': None, 'unit': UNIT, 'cores': threads or cores, 'kind': 'port',
                    'sample': 'failed: ' + r.stderr[-300:]}
        d = json.loads(line[-1])
        cb = d['cpu_baseline']
        cb['images_per_s'] = d['images_per_s']
        return cb

    allc = arm(args.cpu_images or max(1, int(cores * 15.0 / (per_task * n_thr))), 0)
    # the single-thread figure on one image; where even that takes minutes (C4: 25 M pairs per image) it is skipped
    one = arm(1, 1) if per_task * n_thr <= 60.0 else {'value': None, 'images_per_s': None, 'cores': 1,
                                                        'sample': 'skipped: one image takes ~%d s on one core' % (per_task * n_thr)}
    out = dict(allc)
    out['all_cores'] = {k: allc.get(k) for k in ('value', 'images_per_s', 'cores', 'sample')}
    out['single_thread'] = {k: one.get(k) for k in ('value', 'images_per_s', 'cores', 'sample')}
    out['thresholds_per_image'] = n_thr
    out['note'] = 'the reference answers one IoU threshold per det_seg_scores call, so the CPU arm matches every image ' \
                  '%d times for the 0.50:0.95 sweep; the GPU arm reads all thresholds off one pass.  Divide the CPU ' \
                  'times by %d for a single-threshold comparison.  `value` = all cores (the favourable figure for the ' \
                  'CPU); the reference itself is single-threaded' % (n_thr, n_thr)
    return out


if __name__ == '__main__':
    main()
