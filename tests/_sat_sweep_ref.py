"""Reference of the satellite sweep (powder.satellite_measurements_sweep, ampis_eval_images_sat_sweep_host) in numpy,
sharing none of its code.  Per image, the satellite x particle intersections come from the oracle (rleIou over all
pairs, rleMerge where it is non-zero, as tests/_util.satellite_match_one_shot); then for every cell the particles and
satellites are filtered with numpy's own ``scores > s`` on the caller's arrays and the reference's matcher runs on the
kept sub-matrix: score = I / area(s), first arg-max over the kept particles, matched when strictly above the match
threshold.  Where the reference raises (no kept satellite, no kept particle, nothing matched) the cell holds its counts.
The dataset cell is powder.py:525-562 on the satellites-per-particle lists of all images, with NaN for sat_frac / mspp
where the reference divides by zero or takes the median of nothing."""
import numpy as np

from tests import _util as U


def psi_of(parts, sats, size, part_scores=None, sat_scores=None):
    """A PowderSatelliteImage over RLE lists, with instance scores when given."""
    from ampis_b200.applications.powder import PowderSatelliteImage
    from ampis_b200.containers import Instances
    from ampis_b200.structures import InstanceSet, RLEMasks

    def iset(masks, scores):
        f = {'masks': RLEMasks(list(masks)), 'class_idx': np.zeros(len(masks), int)}
        if scores is not None:
            f['scores'] = scores
        return InstanceSet(instances=Instances(tuple(size), **f))
    return PowderSatelliteImage(particles=iset(parts, part_scores), satellites=iset(sats, sat_scores))


def image_matrix(parts, sats):
    """(intersections uint32 [S, N], satellite areas uint32 [S]) of one image."""
    from oracle import cocomask as rle
    S, N = len(sats), len(parts)
    inter = np.zeros((S, N), np.uint32)
    if S and N:
        iou = U.iou_matrix_one_shot(rle, sats, parts)
        for s, p in zip(*np.nonzero(iou)):
            inter[s, p] = rle.merge_area(sats[s], parts[p], intersect=True)
    area = np.asarray(rle.area(sats), np.uint32).reshape(-1) if S else np.zeros(0, np.uint32)
    return inter, area


def cell(inter, area, keep_p, keep_s, t):
    """(matched, unmatched, satellites of every satellited particle in particle order) of one image and cell."""
    sub = inter[np.ix_(keep_s, keep_p)]
    Sk, Nk = sub.shape
    if Sk == 0 or Nk == 0:
        return 0, Sk, np.zeros(0, np.int64)
    with np.errstate(invalid='ignore', divide='ignore'):
        score = sub / area[keep_s][:, None]
    best = score.argmax(axis=1)
    top = score[np.arange(Sk), best]
    with np.errstate(invalid='ignore'):
        m = top > float(t)
    per = np.bincount(best[m], minlength=Nk)
    return int(m.sum()), Sk - int(m.sum()), per[per > 0].astype(np.int64)


def _keeps(scores, th, n):
    if th is None:
        return [np.arange(n)]
    with np.errstate(over='ignore', invalid='ignore'):
        return [np.flatnonzero(np.asarray(scores) > float(s)) for s in th]


def _scores(inst_scores, given, i):
    return given[i] if given is not None else inst_scores


def summary(per, n_images, n_particles, matched, unmatched):
    """powder.py:525-562 on one cell's satellites-per-particle list, NaN where the reference cannot divide."""
    per = np.asarray(per, np.int64)
    values, freq = np.unique(per, return_counts=True)
    with np.errstate(invalid='ignore', divide='ignore'):
        cum = freq.cumsum() / freq.sum()
    return {'n_images': n_images, 'n_particles': n_particles, 'n_satellites': matched,
            'n_satellites_unmatched': unmatched, 'n_satellited_particels': len(per),
            'sat_frac': len(per) / n_particles if n_particles else float('nan'),
            'mspp': np.median(per) if len(per) else np.float64('nan'),
            'unique_satellites_per_particle': values, 'counts_satellites_per_particle': cum}


def sweep(psi, particle_score_thresholds=None, satellite_score_thresholds=None, match_thresholds=(0.5,),
          particle_scores=None, satellite_scores=None, _n_bins=None):
    """The dict of powder.satellite_measurements_sweep (same arguments), plus ``cells``: the summary dict of every
    (k, l, t)."""
    images = list(psi)
    n = len(images)
    pt, st, mt = particle_score_thresholds, satellite_score_thresholds, list(np.asarray(match_thresholds).reshape(-1))
    K = 1 if pt is None else len(pt)
    L = 1 if st is None else len(st)
    T = len(mt)
    B = (1 + max([len(im.satellites.instances.masks.rle) for im in images], default=0)) if _n_bins is None else _n_bins
    img_counts = np.zeros((n, K, L, T, 3), np.int64)
    img_p, img_s = np.zeros((n, K), np.int64), np.zeros((n, L), np.int64)
    per = [[[[] for _ in range(T)] for _ in range(L)] for _ in range(K)]
    for i, im in enumerate(images):
        parts, sats = im.particles.instances.masks.rle, im.satellites.instances.masks.rle
        inter, area = image_matrix(parts, sats)
        pk = _keeps(None if pt is None else _scores(getattr(im.particles.instances, 'scores', None), particle_scores, i),
                    pt, len(parts))
        sk = _keeps(None if st is None else _scores(getattr(im.satellites.instances, 'scores', None), satellite_scores, i),
                    st, len(sats))
        img_p[i] = [len(x) for x in pk]
        img_s[i] = [len(x) for x in sk]
        for k in range(K):
            for l in range(L):
                for t in range(T):
                    a, b, pp = cell(inter, area, pk[k], sk[l], mt[t])
                    img_counts[i, k, l, t] = [a, b, len(pp)]
                    per[k][l][t].append(pp)
    totals = img_counts.sum(axis=0)
    out = {'particle_score_thresholds': None if pt is None else np.asarray(pt, np.float64),
           'satellite_score_thresholds': None if st is None else np.asarray(st, np.float64),
           'match_thresholds': np.asarray(mt, np.float64), 'n_images': n, 'n_particles': img_p.sum(axis=0),
           'n_satellite_instances': img_s.sum(axis=0), 'n_satellites': totals[..., 0],
           'n_satellites_unmatched': totals[..., 1], 'n_satellited_particels': totals[..., 2],
           'image_counts': img_counts, 'image_particles': img_p, 'image_satellites': img_s}
    hist = np.zeros((K, L, T, B), np.int64)
    sat_frac, mspp = np.zeros((K, L, T)), np.zeros((K, L, T))
    cells = np.empty((K, L, T), object)
    for k in range(K):
        for l in range(L):
            for t in range(T):
                pp = np.concatenate(per[k][l][t]) if n else np.zeros(0, np.int64)
                hist[k, l, t] = np.bincount(pp, minlength=B)
                c = summary(pp, n, int(out['n_particles'][k]), int(totals[k, l, t, 0]), int(totals[k, l, t, 1]))
                cells[k, l, t] = c
                sat_frac[k, l, t], mspp[k, l, t] = c['sat_frac'], c['mspp']
    out.update({'spp_hist': hist, 'sat_frac': sat_frac, 'mspp': mspp, 'cells': cells})
    return out


INT_KEYS = ('n_particles', 'n_satellite_instances', 'n_satellites', 'n_satellites_unmatched', 'n_satellited_particels',
            'spp_hist', 'image_counts', 'image_particles', 'image_satellites')


def same_value(a, b):
    """Equal values, floats bit for bit, NaN where the other has NaN."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape:
        return False
    if a.dtype.kind == 'f' or b.dtype.kind == 'f':
        a, b = a.astype(np.float64), b.astype(np.float64)
        return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)].view(np.uint64),
                                                                           b[~np.isnan(b)].view(np.uint64))
    return np.array_equal(a, b)


def assert_same(got, ref, what=''):
    """Every key of the sweep equal, and satellite_measurements_at equal to the reference summary at every cell."""
    from ampis_b200.applications import powder
    assert got['n_images'] == ref['n_images'], what
    for k in ('particle_score_thresholds', 'satellite_score_thresholds', 'match_thresholds'):
        assert (got[k] is None) == (ref[k] is None) and (got[k] is None or same_value(got[k], ref[k])), (what, k)
    for k in INT_KEYS:
        assert np.asarray(got[k]).dtype == np.int64, (what, k)
        assert same_value(got[k], ref[k]), (what, k)
    for k in ('sat_frac', 'mspp'):
        assert same_value(got[k], ref[k]), (what, k)
    for idx in np.ndindex(*ref['cells'].shape):
        at = powder.satellite_measurements_at(got, *idx)
        want = ref['cells'][idx]
        assert set(at) == set(want), (what, idx)
        for key in want:
            assert same_value(at[key], want[key]), (what, idx, key, at[key], want[key])
