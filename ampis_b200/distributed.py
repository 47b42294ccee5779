"""Multi-GPU evaluation: one process per GPU, images sharded across ranks, one small
all-reduce at the end (SURVEY.md section 8e).

Images are independent units of the hot path, so there is no data-path collective: rank r
evaluates images r, r+W, r+2W, ... on its own GPU.  The only exchange is the sum of the
dataset-level counters -- [TP, FP, FN] per IoU threshold, satellite totals, histograms -- an
int64 vector of a few hundred bytes, reduced with torch.distributed (NCCL over NVLink on the
B200 box, gloo in the CPU tests).  Per-image results stay rank-local unless gathered.
"""
import numpy as np
import torch
import torch.distributed as dist

from . import batch, engine


def world_info(group=None):
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def shard_indices(n_items, rank, world):
    """Strided shard: rank r owns items r, r+W, ... (order restored by index on gather)."""
    return np.arange(rank, n_items, world, dtype=np.int64)


def all_reduce_sum_(t, group=None):
    """In-place SUM all-reduce of an int64 tensor (no-op without a process group)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def gather_rows(local_rows, local_index, n_items, group=None):
    """Gather per-image rows (int64 [n_local, k]) of all ranks into [n_items, k] ordered by
    image index; every rank receives the result."""
    rank, world = world_info(group)
    local_rows = np.asarray(local_rows, np.int64).reshape(len(local_index), -1)
    k = local_rows.shape[1]
    out = np.zeros((n_items, k), np.int64)
    if world == 1:
        out[local_index] = local_rows
        return out
    dev = torch.device('cuda', torch.cuda.current_device()) if dist.get_backend(group) == 'nccl' else 'cpu'
    n_max = (n_items + world - 1) // world
    buf = torch.full((n_max, k + 1), -1, dtype=torch.int64, device=dev)
    if len(local_index):
        buf[:len(local_index), 0] = torch.from_numpy(np.asarray(local_index, np.int64)).to(dev)
        buf[:len(local_index), 1:] = torch.from_numpy(local_rows).to(dev)
    parts = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf, group=group)
    for p in parts:
        p = p.cpu().numpy()
        ok = p[:, 0] >= 0
        out[p[ok, 0]] = p[ok, 1:]
    return out


def all_gather_varlen(values, group=None):
    """All-gather of one 1-D int64 array of arbitrary length per rank: the list of every rank's array, in rank
    order, identical on every rank (lengths are exchanged first, payloads travel padded to the longest)."""
    rank, world = world_info(group)
    values = np.ascontiguousarray(np.asarray(values, np.int64).ravel())
    if world == 1:
        return [values]
    dev = torch.device('cuda', torch.cuda.current_device()) if dist.get_backend(group) == 'nccl' else 'cpu'
    n = torch.tensor([len(values)], dtype=torch.int64, device=dev)
    lens = [torch.empty_like(n) for _ in range(world)]
    dist.all_gather(lens, n, group=group)
    lens = [int(x.item()) for x in lens]
    buf = torch.zeros(max(max(lens), 1), dtype=torch.int64, device=dev)
    if len(values):
        buf[:len(values)] = torch.from_numpy(values).to(dev)
    parts = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf, group=group)
    return [p[:k].cpu().numpy() for p, k in zip(parts, lens)]


def _counts_from_rows(r, thresholds):
    """[n_images, T, 3] TP/FP/FN (analyze.py:166-174) from the per-row results of engine.eval_images."""
    n_img, T = len(r.n_rows), len(thresholds)
    G, P = r.n_rows.astype(np.int64), r.n_cols.astype(np.int64)
    img_of_row = np.repeat(np.arange(n_img), G)
    pred_off = np.zeros(n_img + 1, np.int64)
    np.cumsum(P, out=pred_off[1:])
    key = pred_off[img_of_row] + r.best_col.astype(np.int64)
    out = np.zeros((n_img, T, 3), np.int64)
    for t, th in enumerate(thresholds):
        m = r.best_score > th
        tp = np.bincount(img_of_row[m], minlength=n_img)
        claimed = np.unique(key[m])                                   # predictions matched by at least one GT
        n_claimed = np.bincount(np.searchsorted(pred_off, claimed, side='right') - 1, minlength=n_img)
        out[:, t, 0] = tp
        out[:, t, 1] = P - n_claimed
        out[:, t, 2] = G - tp
    return out


def _gpu_match_counts(gt_lists, pred_lists, thresholds):
    """[n_local, T, 3] TP/FP/FN of the local images: ONE library call on this rank's GPU (engine.eval_images), the
    threshold bookkeeping on its flat per-row output."""
    n = len(gt_lists)
    T = len(thresholds)
    if n == 0:
        return np.zeros((0, T, 3), np.int64)
    if sum(map(len, gt_lists)) + sum(map(len, pred_lists)) == 0:
        return np.zeros((n, T, 3), np.int64)
    return _counts_from_rows(engine.eval_images(gt_lists, pred_lists, engine.MODE_IOU), thresholds)


def evaluate_sharded(gt_lists, pred_lists, thresholds=batch.COCO_THRESHOLDS, group=None, gather=True,
                     compute_fn=None):
    """Dataset-level detection counts over all ranks.

    gt_lists / pred_lists: per image, lists of COCO RLE dicts (every rank passes the full
    dataset description; only its shard is touched).  Returns a dict with
      'totals'    int64 [T, 3]  TP/FP/FN summed over the dataset (identical on every rank)
      'per_image' int64 [n_images, T, 3] in image order (if gather) else the local shard
      'index'     the image indices this rank evaluated
    compute_fn(gt_shard, pred_shard, thresholds) -> [n_local, T, 3] overrides the GPU pipeline
    (used by the CPU tests)."""
    rank, world = world_info(group)
    n = len(gt_lists)
    idx = shard_indices(n, rank, world)
    fn = compute_fn or _gpu_match_counts
    local = np.asarray(fn([gt_lists[i] for i in idx], [pred_lists[i] for i in idx], thresholds), np.int64)
    T = len(thresholds)
    local = local.reshape(len(idx), T, 3)
    totals = torch.from_numpy(local.sum(axis=0).reshape(-1).copy())
    use_cuda = world > 1 and dist.get_backend(group) == 'nccl'
    if use_cuda:
        totals = totals.cuda()
    all_reduce_sum_(totals, group)
    out = {'totals': totals.cpu().numpy().reshape(T, 3), 'index': idx}
    if gather:
        out['per_image'] = gather_rows(local.reshape(len(idx), -1), idx, n, group).reshape(n, T, 3)
    else:
        out['per_image'] = local
    return out


_SWEEP_KEYS = ('n_pred', 'det_tp', 'det_fp', 'det_fn', 'seg_tp', 'seg_fp', 'seg_fn')


def _gpu_sweep(gt_lists, pred_lists, scores, score_thresholds, iou_thresholds):
    from . import analyze
    return analyze.det_seg_scores_sweep(gt_lists, pred_lists, score_thresholds, iou_thresholds, scores=scores)


def sweep_sharded(gt_lists, pred_lists, score_thresholds, iou_thresholds=None, scores=None, group=None, gather=True,
                  compute_fn=None):
    """``analyze.det_seg_scores_sweep`` of a dataset whose images are sharded over the ranks: rank r evaluates images
    r, r+W, ... in one library call on its GPU, the int64 totals are summed with ONE all-reduce and the precision /
    recall grids are formed from them on every rank.  Every rank passes the full dataset (and, for RLE lists, the
    full list of per-image score arrays); only its shard is touched.  Returns the keys of det_seg_scores_sweep, the
    per-image arrays [n_images, ...] in image order when gather (else those of the local shard), plus ``index``
    (the images this rank evaluated).  compute_fn(gt_shard, pred_shard, score_shard, score_thresholds,
    iou_thresholds) -> a det_seg_scores_sweep dict overrides the GPU path (CPU tests)."""
    rank, world = world_info(group)
    n = len(gt_lists)
    idx = shard_indices(n, rank, world)
    if iou_thresholds is None:
        iou_thresholds = batch.COCO_THRESHOLDS
    s_th = np.asarray(score_thresholds, np.float64).reshape(-1)
    i_th = np.asarray(iou_thresholds, np.float64).reshape(-1)
    K, T = len(s_th), len(i_th)
    shard = [scores[i] for i in idx] if scores is not None else None
    local = (compute_fn or _gpu_sweep)([gt_lists[i] for i in idx], [pred_lists[i] for i in idx], shard, s_th, i_th)
    sums = torch.from_numpy(np.concatenate([np.asarray(local['totals'], np.int64).ravel(),
                                            np.asarray(local['seg_totals'], np.int64).ravel()]))
    if world > 1 and dist.get_backend(group) == 'nccl':
        sums = sums.cuda()
    all_reduce_sum_(sums, group)
    sums = sums.cpu().numpy()
    totals, seg_totals = sums[:3 * K * T].reshape(K, T, 3), sums[3 * K * T:].reshape(K, T, 3)
    tp, fp, fn = (totals[..., c].astype(np.float64) for c in range(3))
    with np.errstate(invalid='ignore', divide='ignore'):
        out = {'score_thresholds': s_th, 'iou_thresholds': i_th, 'totals': totals, 'seg_totals': seg_totals,
               'det_precision': tp / (tp + fp), 'det_recall': tp / (tp + fn), 'index': idx}
    shapes = {k: (K,) if k == 'n_pred' else (K, T) for k in _SWEEP_KEYS}
    if gather:
        rows = np.concatenate([np.asarray(local[k], np.int64).reshape(len(idx), int(np.prod(shapes[k])))
                               for k in _SWEEP_KEYS], axis=1)
        full = gather_rows(rows, idx, n, group)
        at = 0
        for k in _SWEEP_KEYS:
            w = int(np.prod(shapes[k]))
            out[k] = full[:, at:at + w].reshape((n,) + shapes[k])
            at += w
    else:
        out.update({k: np.asarray(local[k], np.int64) for k in _SWEEP_KEYS})
    return out


def _satellite_rows(part_lists, sat_lists, thresh):
    """Per image of the local shard: (matched, unmatched satellites, satellited particles, particles) and the
    number of satellites of every satellited particle (ascending particle index, powder.py:101-103), from ONE
    library call."""
    n = len(part_lists)
    if n == 0 or sum(map(len, part_lists)) + sum(map(len, sat_lists)) == 0:
        return np.zeros((n, 4), np.int64), [np.zeros(0, np.int64) for _ in range(n)]
    return _satellite_counts_from_rows(engine.eval_images(sat_lists, part_lists, engine.MODE_SAT), thresh)


def _satellite_counts_from_rows(r, thresh):
    """powder.py:85-103 on the flat per-row output of engine.eval_images (rows = satellites, columns = particles)."""
    n = len(r.n_rows)
    S, Np = r.n_rows.astype(np.int64), r.n_cols.astype(np.int64)
    img_of_row = np.repeat(np.arange(n), S)
    part_off = np.zeros(n + 1, np.int64)
    np.cumsum(Np, out=part_off[1:])
    with np.errstate(invalid='ignore'):
        m = r.best_score > thresh                                    # NaN (empty satellite) is never a match
    matched = np.bincount(img_of_row[m], minlength=n)
    owners, per = np.unique(part_off[img_of_row[m]] + r.best_col[m].astype(np.int64), return_counts=True)
    img_of_owner = np.searchsorted(part_off, owners, side='right') - 1
    satellited = np.bincount(img_of_owner, minlength=n)
    counts = np.stack([matched, S - matched, satellited, Np], axis=1).astype(np.int64)
    cut = np.zeros(n + 1, np.int64)
    np.cumsum(satellited, out=cut[1:])
    return counts, [per[cut[g]:cut[g + 1]].astype(np.int64) for g in range(n)]


def _gpu_satellite_counts(part_lists, sat_lists, thresh, n_bins):
    counts, per = _satellite_rows(part_lists, sat_lists, thresh)
    allp = np.concatenate(per) if per else np.zeros(0, np.int64)
    return counts, np.bincount(np.minimum(allp, n_bins - 1), minlength=n_bins).astype(np.int64)


def satellites_sharded(particle_lists, satellite_lists, thresh=0.5, n_bins=64, group=None, compute_fn=None):
    """Dataset-level satellite statistics over all ranks (the sums of powder.py:525-547).

    Returns totals dict {n_images, n_particles, n_satellites, n_satellites_unmatched,
    n_satellited_particles, sat_frac} and the satellites-per-particle histogram (bin b counts
    particles owning b satellites, last bin clamps) -- both identical on every rank."""
    rank, world = world_info(group)
    n = len(particle_lists)
    idx = shard_indices(n, rank, world)
    fn = compute_fn or _gpu_satellite_counts
    counts, hist = fn([particle_lists[i] for i in idx], [satellite_lists[i] for i in idx], thresh, n_bins)
    counts = np.asarray(counts, np.int64).reshape(len(idx), 4)
    payload = torch.from_numpy(np.concatenate([[len(idx)], counts.sum(axis=0), np.asarray(hist, np.int64)]))
    if world > 1 and dist.get_backend(group) == 'nccl':
        payload = payload.cuda()
    all_reduce_sum_(payload, group)
    p = payload.cpu().numpy()
    n_img, matched, unmatched, sat_particles, particles = p[:5]
    return {'n_images': int(n_img), 'n_particles': int(particles), 'n_satellites': int(matched),
            'n_satellites_unmatched': int(unmatched), 'n_satellited_particles': int(sat_particles),
            'sat_frac': sat_particles / particles if particles else float('nan'),
            'spp_hist': p[5:].copy(), 'index': idx}


def area_histogram_sharded(mask_lists, lo, bin_width, n_bins, group=None, compute_fn=None):
    """Binned mask-area histogram of the dataset (size-distribution payload), summed over ranks."""
    rank, world = world_info(group)
    idx = shard_indices(len(mask_lists), rank, world)

    def gpu(shard):
        masks = [m for ml in shard for m in ml]
        if not masks:
            return np.zeros(n_bins, np.int64)
        t = engine.table_from_rle(masks, paint=False)
        return engine.hist_u32(t.area[:t.n], lo, bin_width, n_bins).cpu().numpy()

    hist = torch.from_numpy(np.asarray((compute_fn or gpu)([mask_lists[i] for i in idx]), np.int64).copy())
    if world > 1 and dist.get_backend(group) == 'nccl':
        hist = hist.cuda()
    all_reduce_sum_(hist, group)
    return hist.cpu().numpy()


def _gather_per_image(local_arrays, idx, n_items, group=None):
    """Per-image 1-D int64 arrays of the local shard (image indices idx) -> the list of all n_items arrays in image
    order on every rank."""
    rank, world = world_info(group)
    lens = np.asarray([len(a) for a in local_arrays], np.int64)
    flat = np.concatenate([np.asarray(a, np.int64).ravel() for a in local_arrays]) if len(local_arrays) else \
        np.zeros(0, np.int64)
    got_idx = all_gather_varlen(idx, group)
    got_len = all_gather_varlen(lens, group)
    got_val = all_gather_varlen(flat, group)
    out = [None] * n_items
    for ii, ll, vv in zip(got_idx, got_len, got_val):
        cut = np.zeros(len(ll) + 1, np.int64)
        np.cumsum(ll, out=cut[1:])
        for k, i in enumerate(ii):
            out[int(i)] = vv[cut[k]:cut[k + 1]]
    return out


def psd_sharded(particles, xvals='d_eq', yvals='cvf', c=None, distance='length', group=None, areas_fn=None):
    """``powder.psd(..., return_results=True)`` of a dataset whose images are sharded over the ranks (SURVEY 8e):
    every rank measures the mask areas of ITS images on its GPU, the exact areas are all-gathered (np.unique
    semantics, powder.py:417, are not sum-reducible: a binned histogram would change x and y), and the curve is
    formed by powder.psd's own code on every rank -- the returned dict equals the single-process one bit for bit,
    on every rank.  Every rank passes the full list of InstanceSet / PowderSatelliteImage objects; only its shard
    is measured.  areas_fn(item) -> per-mask areas overrides the GPU measurement (CPU tests)."""
    from .applications import powder
    from .structures import mask_areas
    rank, world = world_info(group)
    measure = areas_fn or mask_areas

    def areas_of(items):
        idx = shard_indices(len(items), rank, world)
        local = [np.asarray(measure(items[int(i)])) for i in idx]
        kinds = set(a.dtype.kind for a in local)
        is_float = int(bool(kinds - {'u', 'i'}))
        flags = all_gather_varlen([is_float], group)
        is_float = any(int(f[0]) for f in flags)
        # exact transport: integers as int64, float64 bit patterns as int64
        wire = [a.astype(np.float64).view(np.int64) if is_float else a.astype(np.int64) for a in local]
        full = _gather_per_image(wire, idx, len(items), group)
        return [a.view(np.float64) if is_float else a.astype(np.uint32) for a in full]

    return powder.psd(particles, xvals=xvals, yvals=yvals, c=c, distance=distance, plot=False, return_results=True,
                      _areas_of=areas_of)


def satellite_measurements_sharded(psi, thresh=0.5, print_summary=False, group=None, match_fn=None):
    """``powder.satellite_measurements(psi, output_dict=True)`` with the images sharded over the ranks: every rank
    matches the satellites of ITS images (one library call for the whole shard), the satellites-per-particle lists
    are all-gathered in image order -- the median ``mspp`` (powder.py:535) and the exact ``unique / counts`` keys
    (powder.py:542-562) are not sum-reducible -- and the summary is formed by powder's own code on every rank: the
    dict equals the single-process one key for key, on every rank, with no histogram clamp.  psi: list of
    PowderSatelliteImage (every rank passes all of them).  match_fn(particles_rle_lists, satellites_rle_lists,
    thresh) -> (counts[n, 4], list of per-particle arrays) overrides the GPU path (CPU tests)."""
    from .applications import powder
    from .structures import masks_to_rle
    rank, world = world_info(group)
    images = [psi] if type(psi) == powder.PowderSatelliteImage else psi
    assert all(type(im) == powder.PowderSatelliteImage for im in images), 'psi must be list of PowderSatelliteImage objects!'
    n = len(images)
    idx = shard_indices(n, rank, world)
    parts = [masks_to_rle(images[int(i)].particles.instances) for i in idx]
    sats = [masks_to_rle(images[int(i)].satellites.instances) for i in idx]
    counts, per = (match_fn or _satellite_rows)(parts, sats, thresh)
    counts = np.asarray(counts, np.int64).reshape(len(idx), 4)
    per_all = _gather_per_image(per, idx, n, group)
    sums = torch.from_numpy(counts.sum(axis=0).copy())
    if world > 1 and dist.get_backend(group) == 'nccl':
        sums = sums.cuda()
    all_reduce_sum_(sums, group)
    matched, unmatched, satellited, particles = (int(v) for v in sums.cpu().numpy())
    per_particle = np.concatenate(per_all) if n else np.zeros(0, np.int64)
    out = powder._satellite_summary(per_particle, n, particles - satellited, unmatched,
                                    sum(len(im.particles.instances) for im in images),
                                    sum(len(im.satellites.instances) for im in images))
    if print_summary and rank == 0:
        powder._print_summary(out)
    return out


def satellite_measurements_sweep_sharded(psi, particle_score_thresholds=None, satellite_score_thresholds=None,
                                         match_thresholds=(0.5,), particle_scores=None, satellite_scores=None,
                                         group=None, compute_fn=None):
    """``powder.satellite_measurements_sweep`` of a dataset whose images are sharded over the ranks: rank r sweeps
    images r, r+W, ... in one library call on its GPU and the totals, the satellites-per-particle histograms and the
    kept counts are summed with ONE int64 all-reduce.  Every quantity, mspp included, is exact after the sum (the
    median is read off the summed histogram), so the dataset keys equal the single-process ones on every rank.  Every
    rank passes the full dataset (and the full per-image score lists); the histogram's length comes from all of it.
    The per-image keys are those of the local shard, ``index`` the images this rank swept.  compute_fn: replaces
    powder.satellite_measurements_sweep (same arguments, CPU tests)."""
    from .applications import powder
    rank, world = world_info(group)
    images = [psi] if type(psi) == powder.PowderSatelliteImage else list(psi)
    assert all(type(im) == powder.PowderSatelliteImage for im in images), 'psi must be list of PowderSatelliteImage objects!'
    n = len(images)
    idx = shard_indices(n, rank, world)
    pick = lambda xs: None if xs is None else [xs[int(i)] for i in idx]
    local = (compute_fn or powder.satellite_measurements_sweep)(
        [images[int(i)] for i in idx], particle_score_thresholds, satellite_score_thresholds, match_thresholds,
        pick(particle_scores), pick(satellite_scores), _n_bins=powder._sweep_bins(images))
    parts = [np.asarray(local[k], np.int64) for k in ('n_particles', 'n_satellite_instances')]
    tot, hist = np.asarray(local['n_satellites'], np.int64), np.asarray(local['spp_hist'], np.int64)
    totals = np.stack([tot, local['n_satellites_unmatched'], local['n_satellited_particels']], axis=-1).astype(np.int64)
    sums = torch.from_numpy(np.concatenate([totals.ravel(), hist.ravel()] + parts))
    if world > 1 and dist.get_backend(group) == 'nccl':
        sums = sums.cuda()
    all_reduce_sum_(sums, group)
    sums = sums.cpu().numpy()
    a, b = totals.size, totals.size + hist.size
    K, L = len(parts[0]), len(parts[1])
    out = {k: local[k] for k in ('particle_score_thresholds', 'satellite_score_thresholds', 'match_thresholds')}
    out.update(powder._sweep_summary(n, sums[b:b + K], sums[b + K:b + K + L], sums[:a].reshape(totals.shape),
                                     sums[a:b].reshape(hist.shape)))
    out.update({k: local[k] for k in ('image_counts', 'image_particles', 'image_satellites')})
    out['index'] = idx
    return out
