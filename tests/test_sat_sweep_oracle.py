"""CPU tests of the satellite sweep: the numpy reference (tests/_sat_sweep_ref.py) against the oracle's literal loops
(rle_satellite_match per kept list, satellite_measurements per cell), the host layer of
powder.satellite_measurements_sweep on a stand-in for the library call (levels, caller order, None axes, the median
read off the histogram), its argument errors and grid cap, and distributed.satellite_measurements_sweep_sharded on a
gloo world of two."""
import multiprocessing as mp
import os

import numpy as np
import pytest

from tests import _sat_sweep_ref as SR
from tests.test_sweep_oracle import _free_port, _rle

P_TH = [0.5, -np.inf, 0.0, 0.3, 0.3, 0.9]
S_TH = [0.2, 0.6, -np.inf, 0.6]
M_TH = [0.5, 0.0, 0.25, 0.75, 0.5]


def _image(rng, h, w, n_part, n_sat):
    """Particles are larger blobs, some of them copies of one another; satellites are small blobs, many on a
    particle's edge, a few empty."""
    yy, xx = np.mgrid[0:h, 0:w]

    def blob(rmax):
        if rng.random() < 0.06:
            return np.zeros((h, w), bool)
        cy, cx = rng.integers(0, h), rng.integers(0, w)
        ry, rx = rng.integers(1, rmax + 1), rng.integers(1, rmax + 1)
        return ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1.0
    parts = []
    for _ in range(n_part):
        parts.append(parts[int(rng.integers(0, len(parts)))] if parts and rng.random() < 0.2
                     else blob(max(min(h, w) // 3, 2)))
    sats = []
    for _ in range(n_sat):
        f = blob(3)
        on = [q for q in parts if q.any()]
        if on and f.any() and rng.random() < 0.6:                  # moved onto a pixel of a particle
            ys, xs = np.nonzero(on[int(rng.integers(0, len(on)))])
            j = int(rng.integers(0, len(ys)))
            cy, cx = np.nonzero(f)
            f = np.roll(f, (ys[j] - int(cy.mean()), xs[j] - int(cx.mean())), axis=(0, 1))
        sats.append(f)
    return [_rle(f) for f in parts], [_rle(f) for f in sats]


def _dataset(seed, n_img=6, least=0):
    """PowderSatelliteImage objects with seeded scores of mixed float dtypes on a coarse grid; least: the fewest
    particles and satellites of an image."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n_img):
        h, w = int(rng.integers(9, 40)), int(rng.integers(9, 40))
        parts, sats = _image(rng, h, w, int(rng.integers(least, 7)), int(rng.integers(2 * least, 12)))
        dt = rng.choice([np.float16, np.float32, np.float64])
        out.append(SR.psi_of(parts, sats, (h, w), np.round(rng.random(len(parts)), 1).astype(dt),
                             np.round(rng.random(len(sats)), 1).astype(dt)))
    return out


def test_reference_equals_oracle_loops():
    """Every image cell is rle_satellite_match (the reference's merge per pair) on the filtered lists -- or, where it
    raises, no match; every dataset cell where no image raises is the oracle's satellite_measurements."""
    from oracle import ampis_ref as R
    psi = _dataset(1, 4, least=3)
    ref = SR.sweep(psi, P_TH, S_TH, M_TH)
    full = 0
    for k, ps in enumerate(P_TH):
        for l, ss in enumerate(S_TH):
            kp = [np.flatnonzero(im.particles.instances.scores > ps) for im in psi]
            ks = [np.flatnonzero(im.satellites.instances.scores > ss) for im in psi]
            for t, mt in enumerate(M_TH):
                matches, raised = [], False
                for i, im in enumerate(psi):
                    parts = [im.particles.instances.masks.rle[c] for c in kp[i]]
                    sats = [im.satellites.instances.masks.rle[c] for c in ks[i]]
                    try:
                        m = R.rle_satellite_match(parts, sats, mt)
                        want = [len(m['satellite_matches']), len(m['satellites_unmatched']), len(m['match_pairs'])]
                        matches.append(m)
                    except (IndexError, ValueError):
                        want, raised = [0, len(sats), 0], True
                    assert ref['image_counts'][i, k, l, t].tolist() == want, (i, k, l, t)
                if not raised:
                    want = R.satellite_measurements(matches, [len(x) for x in kp], [len(x) for x in ks])
                    got = ref['cells'][k, l, t]
                    for key in want:
                        assert SR.same_value(got[key], want[key]), (k, l, t, key)
                    full += 1
    assert full > 0 and ref['n_satellites'].max() > 0


def _fake_engine(sats, parts, plevels, K, slevels, L, m_sorted, B, per_image=True):
    """engine.eval_images_sat_sweep from the reference: particles of level > k and satellites of level > l kept."""
    from ampis_b200.engine import ImagesSatSweep
    n, T = len(sats), len(m_sorted)
    r = ImagesSatSweep()
    r.totals, r.spp_hist = np.zeros((K, L, T, 3), np.int64), np.zeros((K, L, T, B), np.int64)
    r.counts = np.zeros((n, K, L, T, 3), np.int32)
    po = so = 0
    for i, (s, p) in enumerate(zip(sats, parts)):
        inter, area = SR.image_matrix(p, s)
        pl, sl = plevels[po:po + len(p)], slevels[so:so + len(s)]
        po, so = po + len(p), so + len(s)
        for k in range(K):
            for l in range(L):
                for t in range(T):
                    a, b, pp = SR.cell(inter, area, np.flatnonzero(pl > k), np.flatnonzero(sl > l), m_sorted[t])
                    r.counts[i, k, l, t] = [a, b, len(pp)]
                    r.spp_hist[k, l, t] += np.bincount(pp, minlength=B)
    r.totals[:] = r.counts.sum(axis=0)
    r.n_rows, r.n_cols, r.pairs_found = np.asarray([len(s) for s in sats]), np.asarray([len(p) for p in parts]), 0
    return r


@pytest.fixture
def host_only(monkeypatch):
    import torch
    from ampis_b200 import engine
    monkeypatch.setattr(engine, 'require_cuda', lambda: torch.device('cpu'))
    monkeypatch.setattr(engine, 'eval_images_sat_sweep', _fake_engine)


def test_host_layer_against_reference(host_only):
    """Unsorted, repeated thresholds of all three axes, scores from the instances or given explicitly (a torch array
    too), None axes: every key and every cell's satellite_measurements_at equal the reference."""
    import torch
    from ampis_b200.applications import powder
    psi = _dataset(2, 7)
    SR.assert_same(powder.satellite_measurements_sweep(psi, P_TH, S_TH, M_TH), SR.sweep(psi, P_TH, S_TH, M_TH))
    ps = [torch.from_numpy(np.round(np.random.default_rng(i).random(len(im.particles.instances)), 1))
          for i, im in enumerate(psi)]
    got = powder.satellite_measurements_sweep(psi, [0.7, 0.2], None, [0.3], particle_scores=ps)
    SR.assert_same(got, SR.sweep(psi, [0.7, 0.2], None, [0.3], particle_scores=[p.numpy() for p in ps]))
    assert got['satellite_score_thresholds'] is None and got['n_satellite_instances'].shape == (1,)
    one = powder.satellite_measurements_sweep(psi[3])
    SR.assert_same(one, SR.sweep([psi[3]]))


def test_none_axes_need_no_scores(host_only):
    from ampis_b200.applications import powder
    psi = [SR.psi_of(im.particles.instances.masks.rle, im.satellites.instances.masks.rle,
                     im.particles.instances.image_size) for im in _dataset(3, 5)]
    got = powder.satellite_measurements_sweep(psi, match_thresholds=[0.6, 0.1])
    assert got['particle_score_thresholds'] is None and got['spp_hist'].shape[:3] == (1, 1, 2)
    SR.assert_same(got, SR.sweep(psi, None, None, [0.6, 0.1]))
    with pytest.raises(ValueError, match='scores are needed'):
        powder.satellite_measurements_sweep(psi, [0.5])


def test_median_from_histogram():
    """mspp from the summed histogram equals np.median of the list it counts, for odd and even lengths."""
    from ampis_b200.applications import powder
    rng = np.random.default_rng(4)
    lists = [rng.integers(1, 6, int(rng.integers(0, 12))) for _ in range(200)]
    hist = np.stack([np.bincount(x, minlength=8) for x in lists]).reshape(200, 1, 1, 8)
    totals = np.zeros((200, 1, 1, 3), np.int64)
    totals[..., 2] = hist.sum(axis=-1)
    s = powder._sweep_summary(1, np.full(200, 10, np.int64), np.ones(1, np.int64), totals, hist)
    for x, m in zip(lists, s['mspp'][:, 0, 0]):
        assert SR.same_value(m, np.median(x) if len(x) else np.nan)


def test_argument_errors(monkeypatch):
    """Every error is raised before the library call (mixed frame sizes by the marshaller on its way to it)."""
    import torch
    from ampis_b200 import engine
    from ampis_b200.applications import powder
    monkeypatch.setattr(engine, 'require_cuda', lambda: torch.device('cpu'))
    psi = _dataset(5, 3)
    psc = [im.particles.instances.scores for im in psi]
    with pytest.raises(ValueError, match='NaN'):
        powder.satellite_measurements_sweep(psi, [0.5, np.nan])
    with pytest.raises(ValueError, match='NaN'):
        powder.satellite_measurements_sweep(psi, None, [np.nan])
    with pytest.raises(ValueError, match='NaN'):
        powder.satellite_measurements_sweep(psi, match_thresholds=[np.nan])
    with pytest.raises(ValueError, match='negative'):
        powder.satellite_measurements_sweep(psi, match_thresholds=[0.5, -0.1])
    with pytest.raises(ValueError, match='at least one'):
        powder.satellite_measurements_sweep(psi, [])
    with pytest.raises(ValueError, match='particle scores for'):
        powder.satellite_measurements_sweep(psi, [0.5], particle_scores=[np.append(s, 0.5) for s in psc])
    with pytest.raises(ValueError, match='score arrays'):
        powder.satellite_measurements_sweep(psi, [0.5], particle_scores=psc[:-1])
    for bad in ([s.astype(np.int32) for s in psc], [list(s) for s in psc],
                [torch.from_numpy(s.astype(np.float32)).to(torch.bfloat16) for s in psc]):
        with pytest.raises(TypeError):
            powder.satellite_measurements_sweep(psi, [0.5], particle_scores=bad)
    # particles and satellites of two frame sizes in one image
    mixed = SR.psi_of([_rle(np.ones((5, 5), bool))], [_rle(np.ones((3, 4), bool))], (5, 5))
    with pytest.raises(ValueError, match='different image sizes'):
        powder.satellite_measurements_sweep([mixed])
    # the particle limit
    e = _rle(np.zeros((2, 2), bool))
    with pytest.raises(ValueError, match='more than 32768 particles'):
        powder.satellite_measurements_sweep([SR.psi_of([e] * 32769, [e], (2, 2))])


def test_grid_cap(host_only):
    """K x L x T x B above 2^26 or (L + 1) x (T + 1) above 4096 is refused before any work."""
    from ampis_b200.applications import powder
    psi = _dataset(6, 2)
    B = 1 + max(len(im.satellites.instances) for im in psi)
    K = (1 << 26) // (B * 400) + 1                                  # L = T = 20
    assert K <= 65535
    with pytest.raises(ValueError, match='too large'):
        powder.satellite_measurements_sweep(psi, np.linspace(0, 1, K), np.linspace(0, 1, 20), np.linspace(0, 1, 20))
    with pytest.raises(ValueError, match='too large'):
        powder.satellite_measurements_sweep(psi, None, np.linspace(0, 1, 409), np.linspace(0, 1, 10))
    ok = powder.satellite_measurements_sweep(psi, None, np.linspace(0, 1, 408)[:3], np.linspace(0, 1, 10))
    assert ok['spp_hist'].shape == (1, 3, 10, B)


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from ampis_b200 import distributed as D
    psi = _dataset(7, 5)
    r = D.satellite_measurements_sweep_sharded(psi, P_TH, S_TH, M_TH, compute_fn=SR.sweep)
    q.put((rank, {k: v for k, v in r.items() if k != 'cells'}))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_sweep_sharded_two_ranks_gloo():
    from ampis_b200.applications import powder
    psi = _dataset(7, 5)
    want = SR.sweep(psi, P_TH, S_TH, M_TH)
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    for rank, r in res:
        assert np.array_equal(r['index'], np.arange(rank, 5, 2))
        for k in ('n_particles', 'n_satellite_instances', 'n_satellites', 'n_satellites_unmatched',
                  'n_satellited_particels', 'spp_hist', 'sat_frac', 'mspp'):
            assert SR.same_value(r[k], want[k]), (rank, k)
        for k in ('image_counts', 'image_particles', 'image_satellites'):
            assert np.array_equal(r[k], want[k][rank::2]), (rank, k)
        for idx in np.ndindex(*want['cells'].shape):
            at = powder.satellite_measurements_at(r, *idx)
            for key, v in want['cells'][idx].items():
                assert SR.same_value(at[key], v), (rank, idx, key)
