"""Powder characterisation -- drop-in for ``ampis.applications.powder`` (reference
ampis/applications/powder.py) with the satellite/particle overlap assignment and the mask
areas computed on the GPU.  Plotting (matplotlib) is outside the accelerated path: ``psd``
computes and returns the distribution, and draws only if an axis is passed.
"""
import copy

import numpy as np

from .. import analyze, engine
from ..containers import Instances
from ..structures import InstanceSet, mask_areas, masks_to_rle


def _rle_satellite_match(particles, satellites, match_thresh=0.5):
    """Match every satellite to the particle it overlaps most (reference powder.py:28-112).

    score(s, p) = |s AND p| / |s|; satellite s goes to argmax_p (first on ties) if that score is
    strictly above *match_thresh*.  A satellite matches at most one particle, a particle may own
    many satellites.  The reference evaluates all S x N pairs with RLE.merge + RLE.area; the
    fused row kernel visits only pairs whose boxes overlap (the others intersect in 0 pixels,
    which cannot win an arg-max against any positive score and ties resolve to index 0 either way).
    Raises IndexError when no satellite matches, like the reference (powder.py:101)."""
    particles = masks_to_rle(particles)
    satellites = masks_to_rle(satellites)
    S, Np = len(satellites), len(particles)
    if S and Np == 0:
        raise ValueError('attempt to get argmax of an empty sequence')
    if S:
        try:        # the marshaller checks every mask's size on its way (a Python loop over them cost half the call)
            best, score, _, _ = analyze._image_rows(satellites, particles, engine.MODE_SAT)   # NaN score for zero-area
        except ValueError as e:                                                               # satellites, as numpy's 0/0
            if 'different image sizes' in str(e):
                raise ValueError('particle and satellite masks must share one image size') from e
            raise
    else:
        best, score = np.zeros(0, np.int64), np.zeros(0)
    with np.errstate(invalid='ignore'):
        matched = score > match_thresh
    particles_matched_bool = np.zeros(Np, dtype=np.bool_)
    particles_matched_bool[best[matched]] = True
    satellite_matches = np.stack([np.nonzero(matched)[0], best[matched]], axis=1).astype(np.int64) \
        if matched.any() else np.asarray([], np.int64)
    satellites_unmatched = np.nonzero(~matched)[0].astype(np.int64)
    particles_unmatched = np.nonzero(~particles_matched_bool)[0].astype(np.int64)
    intersection_scores = score[matched]

    match_pairs = {x: [] for x in np.unique(satellite_matches[:, 1])}   # IndexError if nothing matched
    for match in satellite_matches:
        match_pairs[match[1]].append(match[0])

    return {'satellite_matches': satellite_matches,
            'satellites_unmatched': satellites_unmatched,
            'particles_unmatched': particles_unmatched,
            'intersection_scores': intersection_scores,
            'match_pairs': match_pairs}


#: legacy name (SURVEY.md F3)
fast_satellite_match = _rle_satellite_match


class PowderSatelliteImage(object):
    """Particle and satellite instances of one image (reference powder.py:115-285)."""

    def __init__(self, particles=None, satellites=None, matches=None):
        self.particles = particles
        self.satellites = satellites
        self.matches = matches

    def compute_matches(self, thresh=0.5):
        self.matches = _rle_satellite_match(self.particles.instances, self.satellites.instances, thresh)

    def compute_satellite_metrics(self):
        """Counts and particle mask areas for size filtering (reference powder.py:221-273)."""
        assert None not in (self.particles, self.satellites, self.matches)
        n_satellites = len(self.satellites.instances)
        matched_particle_idx = list(self.matches['match_pairs'])
        n_particles_matched = len(matched_particle_idx)
        n_particles_all = len(self.particles.instances)
        particle_masks_all = masks_to_rle(self.particles.instances.masks.rle)
        mask_areas_all = mask_areas(particle_masks_all)
        mask_areas_matched = mask_areas_all[matched_particle_idx]
        return {'n_satellites': n_satellites,
                'n_particles_matched': n_particles_matched,
                'n_particles_all': n_particles_all,
                'mask_areas_matched': mask_areas_matched,
                'mask_areas_all': mask_areas_all}

    def copy(self):
        return copy.deepcopy(self)


def _pixel_scale(isets):
    """Length per pixel of every image from its horizontal field width (HFW / image width), and the
    unit string, for psd(distance='length') without an explicit c (reference powder.py:370-388)."""
    if type(isets[0]) != InstanceSet:
        raise ValueError('Cannot infer c from particles (must be list of InstanceSet or PowderSatelliteImage '
                         'objects')
    if isets[0].HFW is None:
        raise ValueError('Cannot infer c because HFW is not defined')
    widths_um = [s.HFW for s in isets]
    assert None not in widths_um, 'all HFW values must be specified if c is not defined'
    units = isets[0].HFW_units
    assert all(s.HFW_units == units for s in isets), 'all HFW values should have same units'
    widths_px = [int(s.instances.image_size[1]) for s in isets]
    return [um / px for um, px in zip(widths_um, widths_px)], units


_PSD_X = {'d_eq': ('Equivalent diameter', ', {}'), 'area': ('Mask area', '- ${}^2$')}
_PSD_Y = {'cvf': 'cumulative volume fraction', 'counts': 'counts (cumulative)'}


def psd(particles, xvals='d_eq', yvals='cvf', c=None, distance='length', ax=None, plot=True, return_results=False,
        _areas_of=None):
    """Cumulative particle size distribution (reference powder.py:288-461).

    Areas come from the GPU measurement pass; they are scaled to length units by *c* (a number, one
    number per image, or ``(c, unit)``; inferred from HFW when omitted), or left in pixels with
    ``distance='pixels'``.  Distinct areas are counted exactly (``np.unique``), mapped to
    ``d_eq = 2 sqrt(A / pi)`` when ``xvals='d_eq'``, weighted by the sphere volume
    ``4/3 pi^(-1/2) A^(3/2)`` when ``yvals='cvf'``, accumulated and normalised to end at 1.  The same
    arguments raise the same ``ValueError``s as the reference.  Nothing is drawn unless an axis is
    passed (matplotlib is not a dependency); ``return_results=True`` returns the curve and labels.
    ``_areas_of`` (internal): replaces the per-image area measurement -- ``distributed.psd_sharded`` passes the
    sharded, all-gathered form, everything after it is this very code on every rank."""
    if _areas_of is None:
        _areas_of = lambda items: [mask_areas(item) for item in items]
    xkey, ykey, how = xvals.lower(), yvals.lower(), distance.lower()
    units = ''
    if type(c) == tuple:
        c, units = c
    if type(particles) in (InstanceSet, PowderSatelliteImage):
        particles = [particles]
    if type(particles[0]) == PowderSatelliteImage:
        particles = [item.particles for item in particles]
    per_image = _areas_of(particles)                              # the reference's list branch is dead (quirk B.6)

    if how == 'length':
        if c is None:
            c, units = _pixel_scale(particles)
        if type(c) in [list, np.ndarray]:
            assert len(c) == len(per_image), 'if c (or c[0] if passed as tuple) is a list or array ' \
                                             'it must have the same length as particles.'
            per_image = [a * k ** 2 for a, k in zip(per_image, c)]
        elif type(c) in [int, float]:                                # numpy scalars are rejected, as in the reference
            per_image = [a * c ** 2 for a in per_image]
        else:
            raise ValueError('c (or c[0] if passed as tuple) must be a list, array, int, or float')
    elif how == 'pixels':
        units = 'px'
        per_image = _areas_of(particles)                             # recomputed, as in the reference (powder.py:410)
    else:
        raise ValueError('distance must be "length" or "pixels"')
    areas = np.concatenate(per_image, axis=0) if type(per_image[0]) in (list, np.ndarray) else per_image

    x, weight = np.unique(areas, return_counts=True)
    if xkey not in _PSD_X:
        raise ValueError('xvals must be "d_eq" or "area"')
    if xkey == 'd_eq':
        x = 2 * np.sqrt(x / np.pi)
    name, unit_fmt = _PSD_X[xkey]
    xlabel = name + (unit_fmt.format(units) if units else '')
    if ykey not in _PSD_Y:
        raise ValueError('yvals must be "cvf" or "counts"')
    if ykey == 'cvf':
        weight = 4 / 3 * np.pi ** (-1 / 2) * x ** (3 / 2) * weight
    ylabel = _PSD_Y[ykey]
    y = weight.cumsum()
    y = y / y[-1]

    if ax is not None:
        ax.grid(axis='both', which='both', color=(0.85, 0.85, 0.85), linewidth=1, linestyle='--')
        ax.plot(x, y, '-.k')
        ax.set_xlabel(xlabel)
        ax.set_ylabel(ylabel)
    if return_results:
        return {'x': x, 'y': y, 'x_label': xlabel, 'y_label': ylabel}


_SUMMARY_ROWS = (('n_images', 'number of images'),
                 ('n_particles', 'number of particles'),
                 ('n_satellites', 'number of matched satellites'),
                 ('n_satellites_unmatched', 'number of unmatched satellites'),
                 ('n_satellited_particels', 'number of satellited particles'),            # key spelled as in the reference
                 ('sat_frac', 'fraction of satellited particles'),
                 ('mspp', 'median number of satellites per\nsatellited particle             '))


def _satellite_summary(per_particle, n_images, n_particles_unmatched, n_satellites_unmatched, n_particle_instances,
                       n_satellite_instances):
    """The dataset-level numbers of powder.py:525-562 from the satellites-per-satellited-particle list and four
    sums (shared by satellite_measurements and distributed.satellite_measurements_sharded, which gathers exactly
    these quantities from all ranks)."""
    per_particle = np.asarray(per_particle)
    out = {'n_images': n_images}
    satellited = len(per_particle)
    out['n_particles'] = satellited + n_particles_unmatched
    out['n_satellites'] = sum(per_particle)
    out['n_satellites_unmatched'] = n_satellites_unmatched
    out['n_satellited_particels'] = satellited
    out['sat_frac'] = satellited / out['n_particles']
    out['mspp'] = np.median(per_particle)
    values, freq = np.unique(per_particle, return_counts=True)
    # consistency with the instance lists themselves (the reference asserts the same three sums)
    assert freq.sum() == satellited
    assert out['n_particles'] == n_particle_instances
    assert out['n_satellites'] + out['n_satellites_unmatched'] == n_satellite_instances
    out['unique_satellites_per_particle'] = values
    out['counts_satellites_per_particle'] = freq.cumsum() / freq.sum()
    return out


def _print_summary(out):
    for key, label in _SUMMARY_ROWS:
        print('{:35}\t{}'.format(label, out[key]))


def satellite_measurements(psi, print_summary=True, output_dict=False):
    """Satellite content of a set of images (reference powder.py:463-569): totals, the fraction of
    particles that carry satellites, the median number of satellites per satellited particle and
    the cumulative distribution of that number.  Images without matches get them computed first.
    The same sums are what ``distributed.satellites_sharded`` all-reduces over GPUs."""
    images = [psi] if type(psi) == PowderSatelliteImage else psi
    assert all(type(im) == PowderSatelliteImage for im in images), 'psi must be list of PowderSatelliteImage objects!'
    if any(im.matches is None for im in images):
        for im in images:
            im.compute_matches()
    found = [im.matches for im in images]

    per_particle = np.asarray([len(sats) for m in found for sats in m['match_pairs'].values()])
    out = _satellite_summary(per_particle, len(images),
                             sum(len(m['particles_unmatched']) for m in found),
                             sum(len(m['satellites_unmatched']) for m in found),
                             sum(len(im.particles.instances) for im in images),
                             sum(len(im.satellites.instances) for im in images))

    if print_summary:
        _print_summary(out)
    if output_dict:
        return out


#: limits of the satellite sweep's grid (include/ampis_b200.h): K x L x T x B histogram cells, and (L + 1) x (T + 1),
#: the per-cell tables the count kernel keeps in shared memory
SAT_SWEEP_MAX_HIST = 1 << 26
SAT_SWEEP_MAX_LT = 4096
SAT_SWEEP_MAX_PARTICLES = 32768


def _sweep_side(thresholds, scores, instances, counts, what):
    """One score axis of the satellite sweep: (thresholds as given or None, position of each in sorted order, level of
    every instance in image order, kept instances int64 [n, K]).  None keeps every instance: one level, no scores."""
    n = len(counts)
    if thresholds is None:
        return None, np.zeros(1, np.int64), np.ones(int(sum(counts)), np.uint16), \
            np.asarray(counts, np.int64).reshape(n, 1)
    th = np.asarray(thresholds, np.float64).reshape(-1)
    sorted_th, pos = analyze._sorted_thresholds(th, what + '_score_thresholds')
    if len(th) > 65535:
        raise ValueError('at most 65,535 %s score thresholds' % what)
    if scores is None:
        scores = [getattr(inst, 'scores', None) if hasattr(inst, 'has') and inst.has('scores') else None
                  for inst in instances]
        if any(s is None for s in scores):
            raise ValueError('%s scores are needed: pass %s_scores or instances with scores' % (what, what))
    if len(scores) != n:
        raise ValueError('%d %s score arrays for %d images' % (len(scores), what, n))
    sc = [analyze._score_array(s) for s in scores]
    for i, (s, c) in enumerate(zip(sc, counts)):
        if len(s) != c:
            raise ValueError('image %d: %d %s scores for %d %ss' % (i, len(s), what, c, what))
    levels, kept = analyze._image_levels(sc, sorted_th)
    return th, pos, levels, kept


def _sweep_summary(n_images, n_particles, n_satellite_instances, totals, spp_hist):
    """The dataset keys of satellite_measurements_sweep from its sum-reducible parts: kept particles [K], kept
    satellites [L], totals [K, L, T, 3] and the satellites-per-particle histogram [K, L, T, B].  sat_frac is NaN where
    no particle is kept, mspp (the median of the histogram, as np.median forms it) where none is satellited."""
    satp = totals[..., 2]
    with np.errstate(invalid='ignore', divide='ignore'):
        sat_frac = satp / n_particles.astype(np.float64)[:, None, None]
    cum = np.cumsum(spp_hist, axis=-1)
    lo = ((cum <= ((satp - 1) // 2)[..., None]).sum(axis=-1)).astype(np.float64)
    hi = ((cum <= (satp // 2)[..., None]).sum(axis=-1)).astype(np.float64)
    mspp = np.where(satp > 0, (lo + hi) / 2, np.nan)
    return {'n_images': n_images, 'n_particles': n_particles, 'n_satellite_instances': n_satellite_instances,
            'n_satellites': totals[..., 0], 'n_satellites_unmatched': totals[..., 1], 'n_satellited_particels': satp,
            'sat_frac': sat_frac, 'mspp': mspp, 'spp_hist': spp_hist}


def _sweep_bins(images):
    """Histogram bins of a sweep over these images: 1 + the most satellites of any image (no particle owns more)."""
    return 1 + max([len(im.satellites.instances) for im in images], default=0)


def satellite_measurements_sweep(psi, particle_score_thresholds=None, satellite_score_thresholds=None,
                                 match_thresholds=(0.5,), particle_scores=None, satellite_scores=None, _n_bins=None):
    """Satellite statistics of a set of images over a grid of particle-score x satellite-score x match thresholds,
    from one evaluation.  Cell (k, l, t) of image i is ``_rle_satellite_match(particles_i[ps_i > P_k],
    satellites_i[ss_i > S_l], match_thresh=T_t)`` reduced to counts (numpy's comparison on the caller's scores: NaN is
    never kept); the dataset cell is ``satellite_measurements(filtered psi, output_dict=True)`` after
    ``compute_matches(T_t)``.  Where the reference raises (nothing matched in an image, satellites without particles,
    no particle at all) the counts are returned instead: sat_frac is NaN when no particle is kept, mspp when none is
    satellited, and the unique / cumulative arrays of satellite_measurements_at are empty.

    psi: a PowderSatelliteImage or a list of them.  A threshold vector of None keeps every instance of that side (the
    axis has length 1 and needs no scores: ground-truth sets).  Scores default to ``instances.scores``;
    particle_scores / satellite_scores (one float16/32/64 numpy or torch array per image) override them.  Thresholds
    may come in any order and repeat; results come back in the caller's order.  match_thresholds must be >= 0.

    Returns a dict: the three threshold vectors as given (float64, None stays None), ``n_images``, ``n_particles``
    int64 [K] and ``n_satellite_instances`` int64 [L] (kept), ``n_satellites`` / ``n_satellites_unmatched`` /
    ``n_satellited_particels`` int64 [K, L, T], ``sat_frac`` / ``mspp`` float64 [K, L, T], ``spp_hist`` int64
    [K, L, T, B] (bin b >= 1: particles owning exactly b satellites; B = 1 + the most satellites of any image),
    ``image_counts`` int64 [n, K, L, T, 3] (matched, unmatched, satellited particles per image), ``image_particles``
    int64 [n, K] and ``image_satellites`` int64 [n, L].  Read one cell with satellite_measurements_at.  One library
    call (engine.eval_images_sat_sweep).  _n_bins (internal): B of the whole dataset when psi is one shard of it."""
    images = [psi] if type(psi) == PowderSatelliteImage else list(psi)
    assert all(type(im) == PowderSatelliteImage for im in images), 'psi must be list of PowderSatelliteImage objects!'
    n = len(images)
    m_th = np.asarray(match_thresholds, np.float64).reshape(-1)
    m_sorted, m_pos = analyze._sorted_thresholds(m_th, 'match_thresholds')
    if m_sorted[0] < 0:
        raise ValueError('match_thresholds must not be negative')
    if len(m_th) > 256:
        raise ValueError('at most 256 match thresholds')
    parts = [masks_to_rle(im.particles.instances) for im in images]
    sats = [masks_to_rle(im.satellites.instances) for im in images]
    n_part, n_sat = [len(p) for p in parts], [len(s) for s in sats]
    if n and max(n_part) > SAT_SWEEP_MAX_PARTICLES:
        raise ValueError('more than %d particles in one image' % SAT_SWEEP_MAX_PARTICLES)
    p_th, p_pos, plevels, p_kept = _sweep_side(particle_score_thresholds, particle_scores,
                                               [im.particles.instances for im in images], n_part, 'particle')
    s_th, s_pos, slevels, s_kept = _sweep_side(satellite_score_thresholds, satellite_scores,
                                               [im.satellites.instances for im in images], n_sat, 'satellite')
    K, L, T = len(p_pos), len(s_pos), len(m_th)
    B = 1 + max(n_sat, default=0) if _n_bins is None else int(_n_bins)
    if K * L * T * B > SAT_SWEEP_MAX_HIST or (L + 1) * (T + 1) > SAT_SWEEP_MAX_LT:
        raise ValueError('satellite sweep grid too large: K x L x T x B = %d x %d x %d x %d (at most 2^26 cells) and '
                         '(L + 1) x (T + 1) = %d (at most %d)' % (K, L, T, B, (L + 1) * (T + 1), SAT_SWEEP_MAX_LT))
    r = engine.eval_images_sat_sweep(sats, parts, plevels, K, slevels, L, m_sorted, B)
    # back to the caller's order of thresholds
    order = lambda a, ax: analyze._reorder(analyze._reorder(analyze._reorder(a, p_pos, ax), s_pos, ax + 1), m_pos, ax + 2)
    n_particles = analyze._reorder(p_kept.sum(axis=0), p_pos, 0)
    n_satellite_instances = analyze._reorder(s_kept.sum(axis=0), s_pos, 0)
    out = {'particle_score_thresholds': p_th, 'satellite_score_thresholds': s_th, 'match_thresholds': m_th}
    out.update(_sweep_summary(n, n_particles, n_satellite_instances, order(r.totals, 0), order(r.spp_hist, 0)))
    out['image_counts'] = order(r.counts, 1).astype(np.int64)
    out['image_particles'] = analyze._reorder(p_kept, p_pos, 1)
    out['image_satellites'] = analyze._reorder(s_kept, s_pos, 1)
    return out


def satellite_measurements_at(result, k, l, t):
    """Cell (k, l, t) of a satellite_measurements_sweep result as the dict of satellite_measurements(output_dict=True):
    the counts, sat_frac and mspp of the cell, and the unique / cumulative satellites-per-particle arrays formed from
    its spp_hist row."""
    h = np.asarray(result['spp_hist'][k, l, t])
    values = np.flatnonzero(h).astype(np.int64)
    freq = h[values]
    with np.errstate(invalid='ignore', divide='ignore'):
        cum = freq.cumsum() / freq.sum()
    return {'n_images': result['n_images'], 'n_particles': int(result['n_particles'][k]),
            'n_satellites': int(result['n_satellites'][k, l, t]),
            'n_satellites_unmatched': int(result['n_satellites_unmatched'][k, l, t]),
            'n_satellited_particels': int(result['n_satellited_particels'][k, l, t]),
            'sat_frac': float(result['sat_frac'][k, l, t]), 'mspp': np.float64(result['mspp'][k, l, t]),
            'unique_satellites_per_particle': values, 'counts_satellites_per_particle': cum}
