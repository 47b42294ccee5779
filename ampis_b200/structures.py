"""Mask containers and converters -- drop-in for ``ampis.structures`` (reference
ampis/structures.py) with the mask arithmetic running on the GPU.

Same names, argument order, defaults, return dtypes and exceptions as the reference; the
dispatch on ``type(x) ==`` (not isinstance) is deliberate, it is what the reference does
(structures.py:57-81, 556-583, 663-690, 736-774).
"""
import colorsys
import copy
from pathlib import Path
from typing import List, Union

import numpy as np
import pandas as pd
import torch

from . import engine
from .containers import BitMasks, Boxes, Instances, PolygonMasks


def random_colors(n, seed, bright=True):
    """n distinguishable RGB colours in a seeded random order (reference ampis/visualize.py:19-56; the
    InstanceSet readers attach them as the ``colors`` field): evenly spaced hues, full saturation,
    value 1.0 (0.7 when not *bright*), shuffled by RandomState(seed)."""
    value = 1.0 if bright else 0.7
    palette = [colorsys.hsv_to_rgb(k / n, 1, value) for k in range(n)]
    np.random.RandomState(seed=seed).shuffle(palette)
    return np.asarray(palette)


def _is_bool_selector(item):
    """Boolean masks in the forms RLEMasks.__getitem__ accepts: torch bool tensor, numpy bool array,
    list whose first element is a bool."""
    if type(item) == torch.BoolTensor or (type(item) == torch.Tensor and item.dtype == torch.bool):
        return True
    if type(item) == np.ndarray:
        return item.dtype == np.bool_
    return type(item) == list and type(item[0]) == bool


class RLEMasks(object):
    """List of COCO RLE dicts that indexes like detectron2's mask containers (reference
    structures.py:24-95): int, slice, boolean mask (same length) or a sequence of indices."""

    def __init__(self, rle):
        super().__init__()
        self.rle = rle

    def __getitem__(self, item: Union[int, slice, List[int], List[bool], torch.BoolTensor, np.ndarray]):
        if type(item) in (int, slice):
            return RLEMasks(self.rle[item])          # an int wraps ONE dict, like the reference (quirk B.13)
        if _is_bool_selector(item):
            if type(item) in (np.ndarray, list):
                assert len(item) == len(self)
            return RLEMasks([m for m, keep in zip(self.rle, item) if keep])
        return RLEMasks([self.rle[k] for k in item])

    def __len__(self):
        return len(self.rle)


def _parse_hfw(value):
    """'103.6 um' -> (103.6, 'um'); a bare number -> (number, None); None -> (None, None); anything else
    is kept as it is (reference structures.py:294-305)."""
    if value is None:
        return None, None
    try:
        return float(value), None
    except ValueError:
        parts = value.split(' ')
        if len(parts) == 2:
            return float(parts[0]), parts[1]
        return value, None


class InstanceSet(object):
    """Everything AMPIS keeps about the instances of one image (reference structures.py:98-533): the
    ``Instances`` (masks, boxes, class_idx, scores, colors), where they came from (``filepath``,
    ``dataset_class``, ``pred_or_gt``, ``mask_format``), the physical scale (``HFW``, ``HFW_units``)
    and the measured ``rprops``."""

    def __init__(self, mask_format=None, bbox_mode=None, filepath=None, annotations=None, instances=None, img=None,
                 dataset_class=None, pred_or_gt=None, HFW=None, HFW_units=None, randomstate=None):
        super().__init__()
        self.mask_format, self.bbox_mode = mask_format, bbox_mode
        self.filepath, self.img = filepath, img
        self.annotations, self.instances = annotations, instances
        self.dataset_class, self.pred_or_gt = dataset_class, pred_or_gt
        self.HFW, self.HFW_units = HFW, HFW_units
        self.rprops = None
        self.colors = None
        self.randomstate = np.random.randint(2 ** 32 - 1) if randomstate is None else randomstate

    def _attach(self, instances):
        self.instances = instances
        self.instances.colors = random_colors(len(instances), self.randomstate)

    def read_from_ddict(self, ddict, inplace=True):
        """Fill the set from a ground-truth data dict (reference structures.py:203-309): RLE dicts
        become RLEMasks, bool arrays BitMasks, coordinate lists PolygonMasks; ``HFW`` strings like
        '103.6 um' are split into value and unit."""
        annos = ddict['annotations']
        self.pred_or_gt, self.filepath, self.mask_format = 'gt', Path(ddict['file_name']), ddict['mask_format']
        segs = [a['segmentation'] for a in annos]
        kind = type(segs[0])
        if kind == dict:
            masks = RLEMasks(segs)
        elif kind == np.ndarray:
            if segs[0].dtype == np.bool_:
                masks = BitMasks(np.stack(segs))
        else:
            masks = PolygonMasks(segs)
        self._attach(Instances((ddict['height'], ddict['width']), masks=masks,
                               boxes=np.stack([a['bbox'] for a in annos]),
                               class_idx=np.asarray([a['category_id'] for a in annos], np.int64)))
        self.dataset_class = ddict.get('dataset_class', None)
        self.HFW, self.HFW_units = _parse_hfw(ddict.get('HFW', None))
        return None if inplace else self

    def read_from_model_out(self, outs, inplace=True):
        """Fill the set from ``data_utils.format_outputs`` output (reference structures.py:312-371).
        A dataset name like 'powder_Validation' yields dataset_class 'Validation'."""
        self.pred_or_gt, self.mask_format, self.filepath = 'pred', 'bitmask', outs['file_name']
        self.dataset_class = outs['dataset'].split('_')[-1]
        pred = outs['pred']['instances']
        self._attach(Instances(pred.image_size, masks=RLEMasks(pred.pred_masks), boxes=pred.pred_boxes,
                               class_idx=pred.pred_classes, scores=pred.scores))
        return None if inplace else self

    def filter_mask_size(self, min_thresh=100, max_thresh=100000, to_rle=False):
        """New ``Instances`` holding the instances with min_thresh < area < max_thresh (both strict,
        ``None`` disables a side); the set itself is not modified (reference structures.py:374-442)."""
        masks = self.instances.masks
        if to_rle:
            masks = RLEMasks(masks_to_rle(masks, self.instances.image_size))
        areas = mask_areas(masks)
        keep = np.ones(areas.shape, np.bool_)
        if min_thresh is not None:
            keep &= areas > min_thresh
        if max_thresh is not None:
            keep &= areas < max_thresh
        if type(masks) == PolygonMasks:
            masks = PolygonMasks([p for p, k in zip(masks.polygons, keep) if k])
        else:
            masks = masks[keep]
        fields = {name: (masks if name == 'masks' else value[keep]) for name, value in self.instances._fields.items()}
        return Instances(self.instances.image_size, **fields)

    def remove_edge_instances(self, k=1):
        """Drop instances that touch the k-pixel image border, in place (reference
        structures.py:445-469).  The reference intersects every mask with an RLE border frame
        (``border[k:-k, k:-k] = 0``); a mask meets that frame iff its tight bounding box does,
        so the GPU measurement pass answers it without any merge.  ``k=0`` keeps the reference
        quirk: the slice is empty, the frame is the whole image and every non-empty mask goes."""
        r, c = self.instances.image_size
        rle = masks_to_rle(self.instances.masks, (r, c))
        area, bb = engine.measure_rle(rle)
        # ``border[k:-k, k:-k] = 0`` zeroes nothing when the slice is empty
        if k <= 0 or r - 2 * k <= 0 or c - 2 * k <= 0:
            touches = area > 0
        else:
            # frame = complement of the zeroed interior [k, r-k) x [k, c-k)
            touches = (area > 0) & ((bb[:, 0] < k) | (bb[:, 2] >= c - k) | (bb[:, 1] < k) | (bb[:, 3] >= r - k))
        inlier_instances = ~touches
        self.instances = self.instances[inlier_instances]

    #: region properties compute_rprops derives from the GPU measurements (skimage names): every non-intensity
    #: property of scikit-image 0.18.3 except euler_number
    RPROPS_GPU_KEYS = ('area', 'bbox', 'bbox_area', 'centroid', 'local_centroid', 'convex_area', 'eccentricity',
                       'equivalent_diameter', 'extent', 'label', 'major_axis_length', 'minor_axis_length',
                       'orientation', 'perimeter', 'solidity', 'moments', 'moments_central', 'moments_normalized',
                       'moments_hu', 'inertia_tensor', 'inertia_tensor_eigvals', 'filled_area', 'filled_image',
                       'perimeter_crofton', 'feret_diameter_max', 'convex_image', 'image', 'coords', 'slice')
    #: the intensity properties of scikit-image 0.18.3; compute_rprops takes them when given an intensity_image
    RPROPS_INTENSITY_KEYS = ('intensity_image', 'max_intensity', 'mean_intensity', 'min_intensity',
                             'weighted_centroid', 'weighted_local_centroid', 'weighted_moments',
                             'weighted_moments_central', 'weighted_moments_normalized', 'weighted_moments_hu')
    #: properties regionprops_table keeps whole, one object cell per region
    RPROPS_OBJECT_KEYS = ('image', 'filled_image', 'convex_image', 'coords', 'slice', 'intensity_image')
    #: shape of the array-valued properties, split into key-i(-j) columns; integer-valued properties
    _RPROPS_SHAPES = {'bbox': (4,), 'centroid': (2,), 'local_centroid': (2,), 'moments': (4, 4),
                      'moments_central': (4, 4), 'moments_normalized': (4, 4), 'moments_hu': (7,),
                      'inertia_tensor': (2, 2), 'inertia_tensor_eigvals': (2,), 'weighted_centroid': (2,),
                      'weighted_local_centroid': (2,), 'weighted_moments': (4, 4), 'weighted_moments_central': (4, 4),
                      'weighted_moments_normalized': (4, 4), 'weighted_moments_hu': (7,)}
    _RPROPS_INT_KEYS = ('area', 'bbox', 'bbox_area', 'convex_area', 'label', 'filled_area')

    def compute_rprops(self, keys=None, return_df=False, intensity_image=None):
        """Region properties per mask (reference structures.py:474-514, which decodes every mask to a
        full int64 frame and runs skimage.measure.regionprops_table on it).  Here the GPU delivers
        exact integer measurements from the run table and the packed bounding-box windows
        (csrc/rprops.cu: raw moments, perimeter histogram, convex hull, hole fill, Crofton transitions,
        Feret diameter, box images) and the properties are formed on the host with skimage 0.18.3's
        formulas.  Default keys are the reference's; cells are 1-element arrays (empty for an empty mask)
        as regionprops_table returns them; tuple- and array-valued properties become ``key-0``, ``key-1``
        ... (``key-0-0`` ... for 2-D arrays) columns, and image, filled_image, convex_image, coords, slice and
        intensity_image one column of 1-element object arrays.

        intensity_image: the grayscale image the masks were found on (2-D, the shape of ``instances.image_size``,
        otherwise ValueError as skimage raises), needed for RPROPS_INTENSITY_KEYS; bool, integer and
        float16/32/64 pixels.  Its min, max and weighted moments are measured on the GPU -- exact integer sums for
        integer and bool images, float64 sums for float images -- and formed here as skimage 0.18.3 does.
        max_intensity, min_intensity and mean_intensity cells are float64, as regionprops_table's are.  One
        deviation: the mean of a float16 / float32 image is taken in float64, where numpy sums in the input
        precision."""
        if keys is None:
            keys = ['area', 'equivalent_diameter', 'major_axis_length', 'perimeter', 'solidity', 'orientation']
        supported = self.RPROPS_GPU_KEYS + self.RPROPS_INTENSITY_KEYS
        unsupported = [k for k in keys if k not in supported]
        if unsupported:
            raise NotImplementedError('region properties %s are not part of the GPU path (supported: %s)'
                                      % (unsupported, list(supported)))
        if intensity_image is not None:
            _check_intensity_shape(intensity_image, [tuple(self.instances.image_size)])
        rle = masks_to_rle(self.instances.masks, self.instances.image_size)
        if type(rle) == dict:
            rle = [rle]
        props = region_properties(rle, keys, intensity_image)
        rows = []
        for p in props:
            row = {}
            for k in keys:
                v = p.get(k)
                if k in self.RPROPS_OBJECT_KEYS:
                    cell = np.empty(1 if v is not None else 0, dtype=object)
                    if v is not None:
                        cell[0] = v
                    row[k] = cell
                elif v is None:            # empty mask: regionprops finds no region
                    empty = np.array([], np.int64 if k in self._RPROPS_INT_KEYS else np.float64)
                    shape = self._RPROPS_SHAPES.get(k)
                    if shape:
                        for loc in np.ndindex(shape):
                            row['-'.join(map(str, (k,) + loc))] = empty
                    else:
                        row[k] = empty
                elif isinstance(v, (tuple, list, np.ndarray)):
                    a = np.asarray(v)
                    for loc in np.ndindex(a.shape):
                        row['-'.join(map(str, (k,) + loc))] = np.array([a[loc].item()])
                elif k in self.RPROPS_INTENSITY_KEYS:     # max / min / mean: float columns in regionprops_table
                    row[k] = np.array([v], np.float64)
                else:
                    row[k] = np.array([v])
            rows.append(row)
        df = pd.DataFrame(rows)
        df['class_idx'] = self.instances.class_idx
        self.rprops = df
        if return_df:
            return self.rprops

    def copy(self):
        return copy.deepcopy(self)


def mask_areas(masks):
    """Area in pixels of each mask (reference structures.py:536-583): ndarray -> uint64 sums,
    PolygonMasks -> shoelace float64, RLE -> uint32 pixel counts (GPU), containers recurse."""
    kind = type(masks)
    if kind == np.ndarray:
        if masks.dtype == np.bool_ and masks.ndim == 3 and masks.size:
            return engine.bool_area_bbox(masks)[0].astype(np.uint)
        return masks.sum(axis=(1, 2), dtype=np.uint)
    if kind == PolygonMasks:
        return np.asarray([_shoelace_area(ring[0][::2], ring[0][1::2]) for ring in masks.polygons])
    if kind == RLEMasks or (kind == list and type(masks[0]) == dict):
        return engine.measure_rle(masks.rle if kind == RLEMasks else masks)[0]
    if kind in (Instances, InstanceSet):
        return mask_areas(masks.masks if kind == Instances else masks.instances)
    if kind == list:
        return [mask_areas(m) for m in masks]
    raise NotImplementedError('Not implemented for type {}'.format(kind))


def _shoelace_area(x, y):
    """Polygon area from vertex coordinates (reference structures.py:586-610)."""
    return 0.5 * np.abs(np.dot(x, np.roll(y, 1)) - np.dot(y, np.roll(x, 1)))


def boxes_to_array(boxes):
    """n x 4 ndarray from an ndarray, a list of 4-sequences or detectron2 ``Boxes`` (reference
    structures.py:613-639); other types give None, as in the reference."""
    if type(boxes) == np.ndarray:
        return boxes
    if type(boxes) == list:
        assert len(boxes[0]) == 4
        return np.asarray(boxes)
    if type(boxes) == Boxes:
        return boxes.tensor.to('cpu').numpy()


def masks_to_rle(masks, size=None):
    """Any supported mask container -> list of COCO RLE dicts (reference structures.py:643-690).
    RLE input is returned as it is.  Polygons need *size* and are rasterised by the GPU restatement of
    pycocotools' rleFrPoly -- the first polygon of each instance only, as ``RLE.frPyObjects(p, *size)[0]``
    does -- and compressed by the GPU string encoder."""
    kind = type(masks)
    if kind == list:
        if type(masks[0]) == dict:
            return masks
        if type(masks[0]) == list:
            raise NotImplementedError('):')
    if kind == RLEMasks:
        return masks.rle
    if kind == PolygonMasks:
        assert size is not None
        h, w = int(size[0]), int(size[1])
        rings = [np.asarray(p[0], np.float64) for p in masks.polygons]
        cnt, cnt_off, cnt_len, _, _ = engine.polygons_to_counts(rings, h, w)
        return [{'size': [h, w], 'counts': c} for c in engine.counts_to_strings(cnt, cnt_off, cnt_len, len(rings))]
    if kind in (Instances, InstanceSet):
        inst = masks if kind == Instances else masks.instances
        return masks_to_rle(inst.masks, inst.image_size)
    raise NotImplementedError('cannot convert mask type {} to RLE'.format(masks))


def _rle_to_bool(rle):
    t = engine.table_from_rle(rle)
    h, w = rle[0]['size']
    for m in rle:
        if list(m['size']) != [h, w]:
            raise ValueError('all masks must share one image size')
    return engine.to_host(engine.unpack_bool(t, np.arange(len(rle)), int(h), int(w)))


def _poly2mask(masks, size):
    """list of [x0,y0,x1,y1,...] polygons -> bool[n, r, c] with skimage.draw.polygon2mask's rule
    (reference structures.py:693-715), rasterised on the GPU (csrc/poly.cu polygon2mask_kernel)."""
    return engine.polygons_to_bool([np.asarray(p, np.float64).ravel() for p in masks], size[0], size[1])


def masks_to_bitmask_array(masks, size=None):
    """Anything -> bool[n_mask, r, c] (reference structures.py:717-774).  RLE input is decoded
    and transposed on the GPU.  Polygon input goes through ``_poly2mask`` like the reference
    (first polygon of every instance, skimage's point-in-polygon rule -- NOT the pycocotools
    rasteriser ``masks_to_rle`` uses; the two differ on boundary pixels, as in the reference)."""
    dtype = type(masks)
    if dtype == np.ndarray:
        assert masks.dtype == np.bool_
        return masks
    elif dtype == PolygonMasks:
        assert size is not None
        return _poly2mask([p[0] for p in masks.polygons], size)
    elif dtype == list:
        if type(masks[0]) == dict:
            return _rle_to_bool(masks)
        elif type(masks[0]) == list or type(masks[0]) == np.ndarray:
            assert size is not None
            return _poly2mask(masks, size)
        else:
            raise NotImplementedError
    elif dtype == RLEMasks:
        if type(masks.rle) == dict:      # RLEMasks[int] wraps one dict (quirk B.13)
            return _rle_to_bool([masks.rle])
        return _rle_to_bool(masks.rle)
    elif dtype == InstanceSet:
        return masks_to_bitmask_array(masks.instances.masks, masks.instances.image_size)
    elif dtype == Instances:
        return masks_to_bitmask_array(masks.masks, masks.image_size)
    else:
        raise NotImplementedError


_PERIMETER_CODES = [5, 7, 15, 17, 25, 27, 21, 33, 13, 23]
_PERIMETER_WEIGHTS = np.zeros(50, dtype=np.double)
_PERIMETER_WEIGHTS[[5, 7, 15, 17, 25, 27]] = 1
_PERIMETER_WEIGHTS[[21, 33]] = np.sqrt(2)
_PERIMETER_WEIGHTS[[13, 23]] = (1 + np.sqrt(2)) / 2

#: the GPU measurements (engine.REGION_MEASUREMENTS) each region property is formed from
_MEASUREMENTS_OF = {
    'area': (), 'bbox': (), 'bbox_area': (), 'equivalent_diameter': (), 'extent': (), 'label': (), 'slice': (),
    'centroid': ('moments',), 'local_centroid': ('moments',), 'eccentricity': ('moments',),
    'major_axis_length': ('moments',), 'minor_axis_length': ('moments',), 'orientation': ('moments',),
    'inertia_tensor': ('moments',), 'inertia_tensor_eigvals': ('moments',),
    'perimeter': ('perimeter_hist',), 'convex_area': ('convex_area',), 'solidity': ('convex_area',),
    'moments': ('moments3',), 'moments_central': ('moments3',), 'moments_normalized': ('moments3',),
    'moments_hu': ('moments3',), 'filled_area': ('filled',), 'filled_image': ('filled_image',),
    'perimeter_crofton': ('crofton',), 'feret_diameter_max': ('convex_feret',), 'convex_image': ('convex_feret',),
    'image': ('image',), 'coords': ('image',), 'intensity_image': ('image',),
    'max_intensity': ('intensity',), 'mean_intensity': ('intensity',), 'min_intensity': ('intensity',),
    'weighted_centroid': ('weighted_intensity',), 'weighted_local_centroid': ('weighted_intensity',),
    'weighted_moments': ('weighted_intensity',), 'weighted_moments_central': ('weighted_intensity',),
    'weighted_moments_normalized': ('weighted_intensity',), 'weighted_moments_hu': ('weighted_intensity',),
}
_DEFAULT_KEYS = ('area', 'bbox', 'bbox_area', 'centroid', 'local_centroid', 'convex_area', 'eccentricity',
                 'equivalent_diameter', 'extent', 'major_axis_length', 'minor_axis_length', 'orientation', 'perimeter',
                 'solidity', 'label')


def _box_props(n, bb):
    x0, y0, x1, y1 = (int(v) for v in bb)
    bbox_area = (y1 - y0 + 1) * (x1 - x0 + 1)
    return {'area': n, 'bbox': (y0, x0, y1 + 1, x1 + 1), 'bbox_area': bbox_area,
            'equivalent_diameter': float(np.sqrt(4 * n / np.pi)), 'extent': n / bbox_area, 'label': 1,
            'slice': (slice(y0, y1 + 1), slice(x0, x1 + 1))}


def _second_order_props(mom, y0, x0):
    """Centroids, inertia tensor and the ellipse properties from the exact order-2 raw moments."""
    N, Sx, Sy, Sxx, Syy, Sxy = (int(v) for v in mom)
    # central second moments times N, exact integers: N*mu20 = N*Syy - Sy^2, ...
    n_rr, n_cc, n_rc = N * Syy - Sy * Sy, N * Sxx - Sx * Sx, N * Sxy - Sx * Sy
    a, c, b = n_cc / (N * N), n_rr / (N * N), -(n_rc / (N * N))    # inertia tensor [[a, b], [b, c]]; -0.0 kept
    half_tr, half_diff = (a + c) / 2, (a - c) / 2
    l1 = half_tr + np.sqrt(half_diff * half_diff + b * b)
    det = (n_cc * n_rr - n_rc * n_rc) / (N ** 4)                    # exact numerator: no cancellation
    l2 = max(det / l1, 0.0) if l1 > 0 else 0.0
    if n_cc == n_rr:
        orientation = -np.pi / 4. if b < 0 else np.pi / 4.
    else:
        orientation = 0.5 * np.arctan2(-2 * b, c - a)
    return {'centroid': (Sy / N, Sx / N), 'local_centroid': ((Sy - N * y0) / N, (Sx - N * x0) / N),
            'eccentricity': 0. if l1 == 0 else float(np.sqrt(1 - l2 / l1)),
            'major_axis_length': float(4 * np.sqrt(l1)), 'minor_axis_length': float(4 * np.sqrt(l2)),
            'orientation': float(orientation), 'inertia_tensor': np.array([[a, b], [b, c]]),
            'inertia_tensor_eigvals': [float(l1), float(l2)]}


_BINOM = [[1], [1, 1], [1, 2, 1], [1, 3, 3, 1]]


def _exact_central(M):
    """Central moments float64[4, 4] from exact box-local raw moments M[p][q] = sum w r^p c^q (Python ints; w = 1
    for a mask, the pixel values for weighted moments, so N = M[0][0] may be zero or negative).  They are expanded
    exactly about the rational centroid -- N^(p+q) mu[p][q] is an integer -- and rounded once.  N = 0 follows
    skimage's float arithmetic: the centroid is nan or +-inf, mu[0][0] = sum w = 0.0 and every other entry nan."""
    N, Sr, Sc = M[0][0], M[1][0], M[0][1]
    if N == 0:
        mu = np.full((4, 4), np.nan)
        mu[0, 0] = 0.0
        return mu
    mu = np.zeros((4, 4))
    for p in range(4):
        for q in range(4):
            num = 0
            for i in range(p + 1):
                for j in range(q + 1):
                    num += _BINOM[p][i] * _BINOM[q][j] * (-Sr) ** (p - i) * (-Sc) ** (q - j) * N ** (i + j) * M[i][j]
            mu[p, q] = num / N ** (p + q)
    return mu


def _moment_props(M, mu):
    """moments, moments_central, moments_normalized, moments_hu (skimage 0.18.3) from the box-local raw moments M
    (4x4 Python ints or float64) and the central moments mu (float64[4, 4]).  mu[0][0] is a numpy float, so a
    weighted mu[0][0] <= 0 gives nan or inf in the normalized moments as in skimage, never a complex number."""
    nu = np.full((4, 4), np.nan)
    with np.errstate(divide='ignore', invalid='ignore'):
        for p in range(4):
            for q in range(4):
                if p + q >= 2:
                    nu[p, q] = mu[p, q] / (mu[0, 0] ** ((p + q) / 2 + 1))
        hu = _hu(nu)
    return {'moments': np.array(M, dtype=np.float64), 'moments_central': mu, 'moments_normalized': nu,
            'moments_hu': hu}


def _check_intensity_shape(img, sizes):
    """skimage's condition on an intensity image: 2-D (one channel, as 0.18.3 has) and of the label image's shape;
    `sizes` are the frame sizes of the masks."""
    shape = np.shape(img)
    if len(shape) != 2 or any(tuple(int(v) for v in sz) != shape for sz in sizes):
        raise ValueError('Label and intensity image must have the same shape.')


def _div(a, b):
    """a / b as skimage's float64 division gives it: correctly rounded, nan or +-inf for b = 0."""
    with np.errstate(divide='ignore', invalid='ignore'):
        return a / b if b else float(np.float64(a) / np.float64(b))


def _intensity_props(m, i, area, y0, x0, box_img, intensity_image):
    """The intensity properties of mask i from the 'intensity' / 'weighted_intensity' measurements taken (and, for
    intensity_image, the 'image' one)."""
    p = {}
    if box_img is not None:
        p['intensity_image'] = np.asarray(intensity_image)[y0:y0 + box_img.shape[0], x0:x0 + box_img.shape[1]] * box_img
    if 'intensity_min' in m:
        p.update({'max_intensity': m['intensity_max'][i], 'min_intensity': m['intensity_min'][i],
                  'mean_intensity': m['intensity_sum'][i] / area})
    if 'intensity_moments' not in m:
        return p
    M = m['intensity_moments'][i]
    if 'intensity_central' in m:                    # float image: float64 sums, central ones from the second pass
        mu = m['intensity_central'][i]
        lr, lc = _div(M[1, 0], M[0, 0]), _div(M[0, 1], M[0, 0])
    else:
        mu = _exact_central(M)
        lr, lc = _div(M[1][0], M[0][0]), _div(M[0][1], M[0][0])
    mom = _moment_props(M, mu)
    p.update({'weighted_local_centroid': (lr, lc), 'weighted_centroid': (lr + y0, lc + x0),
              'weighted_moments': mom['moments'], 'weighted_moments_central': mu,
              'weighted_moments_normalized': mom['moments_normalized'], 'weighted_moments_hu': mom['moments_hu']})
    return p


def _hu(nu):
    """skimage 0.18.3 measure._moments_cy.moments_hu, in its order of operations."""
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


_CROFTON_SCALE = np.pi / 8


def region_properties(rle, keys=None, intensity_image=None):
    """skimage 0.18.3 region properties of every mask of an RLE list (one region per mask, as
    ``regionprops_table(mask.astype(int), intensity_image)`` sees it) from the exact GPU measurements.  Returns one
    dict per mask ({} for an empty mask).  keys=None: the fifteen scalar and tuple properties of
    _DEFAULT_KEYS; otherwise the listed properties of InstanceSet.RPROPS_GPU_KEYS and RPROPS_INTENSITY_KEYS, and
    only the GPU measurements those need are taken.

    intensity_image: 2-D array of the masks' frame size (ValueError otherwise), bool, integer or float16/32/64;
    required by the intensity keys.  max_intensity and min_intensity come in its dtype; weighted moments are exact
    for bool and integer images (frames up to 65,536 pixels a side) and summed in float64 for float images.
    mean_intensity is a float64 -- for float16 / float32 images numpy would sum in the input precision."""
    if intensity_image is not None:
        _check_intensity_shape(intensity_image, {tuple(mk['size']) for mk in rle})
    if keys is None:
        m = engine.region_measurements(rle)
        keys = _DEFAULT_KEYS
    else:
        keys = list(keys)
        unknown = [k for k in keys if k not in _MEASUREMENTS_OF]
        if unknown:
            raise NotImplementedError('region properties %s are not part of the GPU path' % unknown)
        wanted = [k for k in keys if k in InstanceSet.RPROPS_INTENSITY_KEYS]
        if wanted and intensity_image is None:
            raise NotImplementedError('region properties %s need an intensity image: pass intensity_image, a 2-D '
                                      'array of the masks\' frame size' % wanted)
        m = engine.region_measurements_for(rle, {x for k in keys for x in _MEASUREMENTS_OF[k]},
                                           intensity_image if wanted else None)
    out = []
    for i in range(len(rle)):
        n = int(m['area'][i])
        if n == 0:
            out.append({})
            continue
        bb = m['bbox'][i]
        x0, y0 = int(bb[0]), int(bb[1])
        p = _box_props(n, bb)
        if 'moments' in m:
            p.update(_second_order_props(m['moments'][i], y0, x0))
        if 'perimeter_hist' in m:
            hist = np.zeros(50, np.int64)
            hist[_PERIMETER_CODES] = m['perimeter_hist'][i]
            p['perimeter'] = float(hist @ _PERIMETER_WEIGHTS)
        if 'convex_area' in m:
            p['convex_area'] = int(m['convex_area'][i])
            p['solidity'] = n / p['convex_area']
        if 'moments3' in m:
            p.update(_moment_props(m['moments3'][i], _exact_central(m['moments3'][i])))
        if 'filled_area' in m:
            p['filled_area'] = int(m['filled_area'][i])
        if 'filled_image' in m:
            p['filled_image'] = m['filled_image'][i]
        if 'crofton_trans' in m:
            t = m['crofton_trans'][i]
            p['perimeter_crofton'] = float(_CROFTON_SCALE * (int(t[0]) + int(t[1]) + (int(t[2]) + int(t[3])) / np.sqrt(2)))
        if 'feret_d2' in m:
            p['feret_diameter_max'] = float(np.sqrt(float(m['feret_d2'][i]))) / 2
            rg = m['convex_ranges'][i]
            rows = np.arange(int(bb[3]) - y0 + 1)[:, None]
            p['convex_image'] = (rows >= rg[:, 0]) & (rows < rg[:, 1])
        if 'image' in m:
            img = m['image'][i]
            p['image'] = img
            r, c = np.nonzero(img)
            p['coords'] = np.stack([r + y0, c + x0], axis=1).astype(np.int64)
        if 'intensity_min' in m or 'intensity_image' in keys:
            p.update(_intensity_props(m, i, n, y0, x0, p.get('image') if 'intensity_image' in keys else None,
                                      intensity_image))
        out.append({k: p[k] for k in keys})
    return out
