"""Restatement of the ten intensity region properties of scikit-image 0.18.3 for one region (test infrastructure,
not product code), written with numpy on ``oracle.ampis_ref._moments_central``.  It is what the GPU path of these
keys is checked against.

Restated from skimage 0.18.3 measure/_regionprops.py, class RegionProperties:
  intensity_image          = self._intensity_image[self.slice] * self.image
  max_intensity            = np.max(self.intensity_image[self.image])        (min_intensity, mean_intensity alike)
  weighted_moments         = _moments.moments(self.intensity_image, 3)
  weighted_local_centroid  = M[tuple(np.eye(2, dtype=int))] / M[(0, 0)]
  weighted_centroid        = tuple(idx + slc.start for idx, slc in zip(weighted_local_centroid, self.slice))
  weighted_moments_central = _moments.moments_central(self.intensity_image, center=weighted_local_centroid, order=3)
  weighted_moments_normalized = _moments.moments_normalized(weighted_moments_central, 3)
  weighted_moments_hu      = _moments.moments_hu(weighted_moments_normalized)
and measure/_moments.py: moments(image, order) = moments_central(image, (0, 0), order), which sums
image.astype(float) * delta_r^p * delta_c^q with numpy's float64 arithmetic (so nan ** 0 = inf ** 0 = 1, and
0 * inf = nan).  The whole box is weighted: a nan or inf pixel of the box outside the region becomes nan there.

skimage forms those sums with np.dot, and a dot product may skip a zero factor (numpy's small-matrix paths and
reference BLAS do), so 0 * nan can come out as 0 depending on the platform.  Where a non-finite value takes part --
a non-finite pixel in the box, or the nan / inf centroid of a region whose intensities sum to zero -- the sums
here are taken element by element, in plain IEEE arithmetic, which is the rule the GPU path follows."""
import numpy as np

from oracle.ampis_ref import _moments_central
from tests._rprops_ref import moments_hu, moments_normalized

KEYS = ('intensity_image', 'max_intensity', 'mean_intensity', 'min_intensity', 'weighted_centroid',
        'weighted_local_centroid', 'weighted_moments', 'weighted_moments_central', 'weighted_moments_normalized',
        'weighted_moments_hu')


def region_slice(mask):
    rows, cols = np.nonzero(mask)
    return slice(int(rows.min()), int(rows.max()) + 1), slice(int(cols.min()), int(cols.max()) + 1)


def _moments(calc, center):
    """sum calc (r - r0)^p (c - c0)^q for p, q <= 3: skimage's moments_central (oracle.ampis_ref._moments_central)
    when everything is finite, otherwise the same sums element by element (see above)."""
    if np.isfinite(calc).all() and np.isfinite(center).all():
        return _moments_central(calc, center, 3)
    pr = (np.arange(calc.shape[0]) - center[0])[:, None] ** np.arange(4)
    pc = (np.arange(calc.shape[1]) - center[1])[:, None] ** np.arange(4)
    return (calc[:, :, None, None] * pr[:, None, :, None] * pc[None, :, None, :]).sum(axis=(0, 1))


def regionprops_intensity(mask, img, keys=KEYS):
    """The intensity properties `keys` of the single region `mask` over the intensity image `img` (same shape), as
    regionprops computes them; {} for an empty mask."""
    mask = np.asarray(mask, bool)
    img = np.asarray(img)
    if not mask.any():
        return {}
    sl = region_slice(mask)
    image = mask[sl]
    ii = img[sl] * image
    vals = ii[image]
    out = {}
    with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
        M = _moments(ii.astype(np.double), (0, 0))
        wlc = M[1, 0] / M[0, 0], M[0, 1] / M[0, 0]
        mu = _moments(ii.astype(np.double), wlc)
        nu = moments_normalized(mu, 3)
        for k in keys:
            if k == 'intensity_image':
                out[k] = ii
            elif k == 'max_intensity':
                out[k] = np.max(vals)
            elif k == 'min_intensity':
                out[k] = np.min(vals)
            elif k == 'mean_intensity':
                out[k] = np.mean(vals)
            elif k == 'weighted_local_centroid':
                out[k] = wlc
            elif k == 'weighted_centroid':
                out[k] = (wlc[0] + sl[0].start, wlc[1] + sl[1].start)
            elif k == 'weighted_moments':
                out[k] = M
            elif k == 'weighted_moments_central':
                out[k] = mu
            elif k == 'weighted_moments_normalized':
                out[k] = nu
            elif k == 'weighted_moments_hu':
                out[k] = moments_hu(nu)
            else:
                raise KeyError(k)
    return out


def exact_weighted_moments(mask, img):
    """M[p][q] = sum I r^p c^q over the region's pixels, box-local r, c, as exact Python ints (integer and bool
    images)."""
    mask = np.asarray(mask, bool)
    sl = region_slice(mask)
    r, c = np.nonzero(mask[sl])
    vals = [int(v) for v in np.asarray(img)[sl][mask[sl]]]
    r, c = r.tolist(), c.tolist()
    return [[sum(v * rr ** p * cc ** q for v, rr, cc in zip(vals, r, c)) for q in range(4)] for p in range(4)]


def weighted_magnitude(mask, img, center):
    """sum |I| |r - r0|^p |c - c0|^q over the region (float64[4, 4]): the scale of the cancellation in the sums
    about `center`, what the float comparisons are relative to."""
    mask = np.asarray(mask, bool)
    sl = region_slice(mask)
    r, c = np.nonzero(mask[sl])
    a = np.abs(np.asarray(img)[sl][mask[sl]].astype(np.float64))
    dr, dc = np.abs(r - center[0]), np.abs(c - center[1])
    return np.array([[(a * dr ** p * dc ** q).sum() for q in range(4)] for p in range(4)])
