"""Restatement of the scikit-image 0.18.3 region properties beyond the fifteen of
``oracle.ampis_ref.regionprops_one`` (test infrastructure, not product code): moments to order 3,
inertia tensor, hole fill, Crofton perimeter, maximum Feret diameter, convex / box / filled images,
coords and slice, written with numpy / scipy.  It builds on the oracle's ``_moments_central`` and
``_convex_hull_image`` and is what the GPU path of these keys is checked against."""
import numpy as np

from oracle.ampis_ref import _convex_hull_image, _moments_central

# Restated from measure/_regionprops.py, measure/_moments.py, measure/_moments_cy.pyx (moments_hu),
# measure/_regionprops_utils.py (perimeter_crofton) with numpy / scipy; euler_number is not restated.

_CROFTON_COEFS_4 = [0, np.pi / 4 * (1 + 1 / (np.sqrt(2))), np.pi / (4 * np.sqrt(2)), np.pi / (2 * np.sqrt(2)), 0,
                    np.pi / 4 * (1 + 1 / (np.sqrt(2))), 0, np.pi / (4 * np.sqrt(2)), np.pi / 4, np.pi / 2,
                    np.pi / (4 * np.sqrt(2)), np.pi / (4 * np.sqrt(2)), np.pi / 4, np.pi / 2, 0, 0]


def perimeter_crofton4(image):
    """skimage.measure.perimeter_crofton(image, directions=4): 2x2 configuration histogram of the zero-padded
    image, dotted with the 4-direction Crofton coefficients."""
    import scipy.ndimage as ndi
    image = np.pad((np.asarray(image) > 0).astype(np.uint8), pad_width=1, mode='constant')
    XF = ndi.convolve(image, np.array([[0, 0, 0], [0, 1, 4], [0, 2, 8]]), mode='constant', cval=0)
    h = np.bincount(XF.ravel(), minlength=16)
    return float(np.asarray(_CROFTON_COEFS_4) @ h)


def crofton_transitions(image):
    """Pixel pairs of the zero-padded image that differ: along rows, columns, (r+1, c+1), (r+1, c-1)."""
    p = np.pad(np.asarray(image, bool), 1)
    return (int((p[:, 1:] != p[:, :-1]).sum()), int((p[1:, :] != p[:-1, :]).sum()),
            int((p[1:, 1:] != p[:-1, :-1]).sum()), int((p[1:, :-1] != p[:-1, 1:]).sum()))


def moments_hu(nu):
    """skimage.measure._moments_cy.moments_hu, in its order of operations."""
    hu = np.zeros((7,), dtype=np.double)
    t0 = nu[3, 0] + nu[1, 2]
    t1 = nu[2, 1] + nu[0, 3]
    q0 = t0 * t0
    q1 = t1 * t1
    n4 = 4 * nu[1, 1]
    s = nu[2, 0] + nu[0, 2]
    d = nu[2, 0] - nu[0, 2]
    hu[0] = s
    hu[1] = d * d + n4 * nu[1, 1]
    hu[3] = q0 + q1
    hu[5] = d * (q0 - q1) + n4 * t0 * t1
    t0 *= q0 - 3 * q1
    t1 *= 3 * q0 - q1
    q0 = nu[3, 0] - 3 * nu[1, 2]
    q1 = 3 * nu[2, 1] - nu[0, 3]
    hu[2] = q0 * q0 + q1 * q1
    hu[4] = q0 * t0 + q1 * t1
    hu[6] = q1 * t0 - q0 * t1
    return hu


def moments_normalized(mu, order=3):
    nu = np.zeros_like(mu)
    mu0 = mu.ravel()[0]
    for powers in np.ndindex(*(order + 1,) * mu.ndim):
        if sum(powers) < 2:
            nu[powers] = np.nan
        else:
            nu[powers] = mu[powers] / (mu0 ** (sum(powers) / mu.ndim + 1))
    return nu


def inertia_tensor(mu):
    """skimage.measure.inertia_tensor of a 2-D image from its central moments."""
    mu0 = mu[0, 0]
    result = np.zeros((2, 2))
    corners2 = (np.array([2, 0]), np.array([0, 2]))
    d = (np.sum(mu[corners2]) - mu[corners2]) / mu0
    result[0, 0], result[1, 1] = d
    result[0, 1] = result[1, 0] = -mu[1, 1] / mu0
    return result


def contour_midpoints(image):
    """Vertices of find_contours(image, 0.5) on a 0/1 image: the midpoints of the 4-adjacent (inside, outside)
    pixel pairs, (row, col) float."""
    a = np.asarray(image, bool)
    r, c = np.nonzero(a[:, 1:] != a[:, :-1])
    h = np.stack([r.astype(float), c + 0.5], axis=1)
    r, c = np.nonzero(a[1:, :] != a[:-1, :])
    v = np.stack([r + 0.5, c.astype(float)], axis=1)
    return np.concatenate([h, v])


def feret_diameter_max(convex_image):
    """sqrt(max pdist(contour of pad(convex_image, 2) at 0.5, 'sqeuclidean')); the farthest pair lies on the
    convex hull of the contour points, so pdist runs over its vertices."""
    from scipy.spatial import ConvexHull
    from scipy.spatial.distance import pdist
    pts = contour_midpoints(np.pad(np.asarray(convex_image, bool), 2))
    try:
        pts = pts[ConvexHull(pts).vertices]
    except Exception:                   # degenerate (collinear) point sets: all of them
        pass
    return float(np.sqrt(np.max(pdist(pts, 'sqeuclidean'))))


def regionprops_more(mask, keys):
    """The properties `keys` (non-intensity, not euler_number, not the fifteen of regionprops_one) of the single
    region `mask.astype(int)` defines, as regionprops computes them per region; {} for an empty mask."""
    import scipy.ndimage as ndi
    mask = np.asarray(mask, bool)
    if not mask.any():
        return {}
    rows, cols = np.nonzero(mask)
    r0, r1, c0, c1 = rows.min(), rows.max() + 1, cols.min(), cols.max() + 1
    img = mask[r0:r1, c0:c1]
    M = _moments_central(img.astype(np.uint8), (0, 0), 3)
    local_centroid = (M[1, 0] / M[0, 0], M[0, 1] / M[0, 0])
    mu = _moments_central(img.astype(np.uint8), local_centroid, 3)
    out = {}
    for k in keys:
        if k == 'moments':
            out[k] = M
        elif k == 'moments_central':
            out[k] = mu
        elif k == 'moments_normalized':
            out[k] = moments_normalized(mu, 3)
        elif k == 'moments_hu':
            out[k] = moments_hu(moments_normalized(mu, 3))
        elif k == 'inertia_tensor':
            out[k] = inertia_tensor(mu)
        elif k == 'inertia_tensor_eigvals':
            ev = np.linalg.eigvalsh(inertia_tensor(mu))
            ev = np.clip(ev, 0, None, out=ev)
            out[k] = sorted(ev, reverse=True)
        elif k == 'filled_image':
            out[k] = ndi.binary_fill_holes(img, structure=np.ones((3, 3)))
        elif k == 'filled_area':
            out[k] = int(ndi.binary_fill_holes(img, structure=np.ones((3, 3))).sum())
        elif k == 'perimeter_crofton':
            out[k] = perimeter_crofton4(img)
        elif k == 'feret_diameter_max':
            out[k] = feret_diameter_max(_convex_hull_image(img))
        elif k == 'convex_image':
            out[k] = _convex_hull_image(img)
        elif k == 'image':
            out[k] = img
        elif k == 'coords':
            out[k] = np.vstack(np.nonzero(img)).T + np.array([r0, c0])
        elif k == 'slice':
            out[k] = (slice(int(r0), int(r1)), slice(int(c0), int(c1)))
        else:
            raise KeyError(k)
    return out
