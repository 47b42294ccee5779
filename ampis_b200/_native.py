"""ctypes binding of libampis_b200.so (the C ABI declared in include/ampis_b200.h).

There is no CPU fallback: if the library is missing it is built with nvcc, and if a
kernel entry point is called without a CUDA device the call raises.
"""
import ctypes as C
import os

from . import build as _build

LAYOUT_SPAN, LAYOUT_FULL, LAYOUT_CROP = 0, 1, 2
MODE_IOU, MODE_SAT = 0, 1
ST_BAD_TOTAL = 1
OK, EINVAL, ECUDA, ENOSPC = 0, -1, -2, -3

_p = C.c_void_p
_i32, _i64, _u32, _u64, _f64 = C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_double

# name -> (restype, argtypes); must list every symbol of include/ampis_b200.h
SIGNATURES = {
    'ampis_version': (C.c_int, []),
    'ampis_last_error': (C.c_char_p, []),
    'ampis_sm_count': (C.c_int, []),
    'ampis_rle_string_decode': (C.c_int, [_p, _p, _i32, _p, _p, _p, _p]),
    'ampis_rle_string_encode': (C.c_int, [_p, _p, _p, _i32, _p, _p, _p, _p]),
    'ampis_rle_measure': (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p]),
    'ampis_scan_tmp_bytes': (C.c_size_t, [_i64]),
    'ampis_exclusive_scan_i64': (C.c_int, [_p, _p, _i64, _p, C.c_size_t, _p]),
    'ampis_rle_decode_packed': (C.c_int, [_p, _p, _p, _p, _p, _p, _i32, _p, _i64, _p]),
    'ampis_unpack_bool_nrc': (C.c_int, [_p, _p, _p, _p, _i32, _u32, _u32, _p, _p]),
    'ampis_bool_area_bbox': (C.c_int, [_p, _i32, _u32, _u32, _i32, _p, _p, _p]),
    'ampis_pack_bool_nrc': (C.c_int, [_p, _i32, _u32, _u32, _i32, _p, _p, _p]),
    'ampis_rows_per_block': (C.c_int, []),
    'ampis_intersect_rows': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _i32, _p, _p,
                                       _p, _p, _p]),
    'ampis_rle_measure_paint': (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p,
                                          _i32, _p]),
    'ampis_rle_measure_paint_flat': (C.c_int, [_p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p,
                                               _p, _i32, _i32, _p]),
    'ampis_rle_measure_paint_flat_zero': (C.c_int, [_p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _i64,
                                                    _p, _p, _i32, _p, _i64, _i32, _p]),
    'ampis_intersect_rows_crop': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _i32, _p, _p, _p,
                                            _p, _p]),
    'ampis_grid_cells': (C.c_int, []),
    'ampis_grid_build': (C.c_int, [_p, _p, _p, _i32, _p, _p, _p, _p, _i64, _p, _p]),
    'ampis_intersect_rows_grid': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _i64,
                                            _p, _i32, _p, _i64, _p, _p, _p, _p, _p, _p, _i64, _p, _p]),
    'ampis_pairs_read_intervals': (C.c_int, []),
    'ampis_intersect_rows_pairs': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _p, _p,
                                             _i64, _p, _p, _p, _p, _i32, _p, _i64, _p, _p, _p, _p, _p, _p, _i64, _p,
                                             _p, _p]),
    'ampis_rle_decode_crop': (C.c_int, [_p, _p, _p, _p, _p, _p, _i32, _p, _i64, _p]),
    'ampis_mma_tile_rows': (C.c_int, []),
    'ampis_mma_tile_cols': (C.c_int, []),
    'ampis_intersect_tcgen05': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p]),
    'ampis_eval_image_host': (C.c_int, [_p, _p, _i32, _i32, _u32, _u32, _i32, _i32, _p, _i64, _p, _i64, _p, _p, _p, _p, _p,
                                        _p, _p, _p, _p, _p]),
    'ampis_eval_images_host': (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _i32, _i32, _f64, _p, _i64, _p, _i64, _p, _p, _p, _p, _p,
                                         _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p]),
    'ampis_eval_images_sweep_host': (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _i32, _p, _i32, _p, _i32, _p, _i64, _p,
                                               _i64, _p, _p, _p, _p, _p, _p, _p, _p]),
    'ampis_eval_images_sat_sweep_host': (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _i32, _p, _i32, _p, _i32, _p, _i32,
                                                   _i32, _p, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, _p]),
    'ampis_mma_pair_tile_rows': (C.c_int, []),
    'ampis_mma_pair_tile_cols': (C.c_int, []),
    'ampis_intersect_tcgen05_pair': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p,
                                               _p]),
    'ampis_tma_tile': (C.c_int, []),
    'ampis_intersect_tma': (C.c_int, [_p, _i64, _i32, _p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p]),
    'ampis_rows_from_imat': (C.c_int, [_p, _p, _p, _p, _p, _i32, _p, _p, _p, _i32, _p, _p, _p, _p]),
    'ampis_iou_matrix_f64': (C.c_int, [_p, _p, _p, _i32, _i32, _p, _p]),
    'ampis_match_counts': (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, _p, _i32, _p, _p, _p]),
    'ampis_satellite_counts': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _i32, _i32, _f64, _p, _p, _i32, _p]),
    'ampis_hist_u32': (C.c_int, [_p, _i64, _u32, _u32, _p, _i32, _p]),
    'ampis_bits_to_rle_count': (C.c_int, [_p, _p, _p, _p, _i32, _p, _p]),
    'ampis_bits_to_rle_emit': (C.c_int, [_p, _p, _p, _p, _i32, _p, _p, _p, _p]),
    'ampis_project_pairs': (C.c_int, [_p, _p, _p, _p, _p, _p, _i32, _i64, _i32, _p, _p, _p]),
    'ampis_rle_moments': (C.c_int, [_p, _p, _p, _p, _i32, _p, _p]),
    'ampis_crop_perimeter': (C.c_int, [_p, _p, _p, _i32, _p, _p, _p]),
    'ampis_crop_convex_area': (C.c_int, [_p, _p, _p, _i32, _p, _p, _p, _p]),
    'ampis_rle_moments3': (C.c_int, [_p, _p, _p, _p, _p, _i32, _p, _p]),
    'ampis_crop_fill_holes': (C.c_int, [_p, _p, _p, _i32, _p, _p, _p, _p]),
    'ampis_crop_convex_feret': (C.c_int, [_p, _p, _p, _i32, _p, _p, _p, _p, _p, _p]),
    'ampis_crop_unpack_image': (C.c_int, [_p, _p, _p, _i32, _p, _p, _p]),
    'ampis_rle_intensity': (C.c_int, [_p, _p, _p, _p, _p, _i32, _p, _i32, _p, _i32, _p, _p, _p]),
    'ampis_ccl_label': (C.c_int, [_p, _i32, _i32, _p, _p, _p, _p, C.c_size_t, _p, _p]),
    'ampis_label_values_present': (C.c_int, [_p, _i64, _p, _i32, _p, _p]),
    'ampis_label_dense': (C.c_int, [_p, _p, _i32, _i32, _i32, _p, _p]),
    'ampis_label_bbox': (C.c_int, [_p, _i32, _i32, _i32, _p, _p]),
    'ampis_label_rle_count': (C.c_int, [_p, _i32, _i32, _i32, _p, _p, _p]),
    'ampis_label_rle_emit': (C.c_int, [_p, _i32, _i32, _i32, _p, _p, _p, _p, _p]),
    'ampis_edge_count': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _i32, _p, _p]),
    'ampis_edge_distances': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p,
                                       _p, _p]),
    'ampis_poly_to_rle': (C.c_int, [_p, _p, _p, _p, _i32, _p, _p, _p, _p]),
    'ampis_polygon2mask': (C.c_int, [_p, _p, _i32, _i32, _i32, _p, _p]),
}

#: libampis_synth.so (bench / test data generator, include/ampis_synth.h) -- a separate library on purpose
SYNTH_SIGNATURES = {
    'ampis_synth_batch': (_i64, [_u64, _i32, _u32, _u32, _i32, _i32, _i32, _f64, _f64, _f64, _f64, _f64, _f64,
                                 _f64, _f64, _i32, _p, _i64, _p, _p]),
}

_lib = None
_synth = None
ABI_VERSION = 201       # ampis_version(): bumped whenever a signature of include/ampis_b200.h changes


class AmpisNativeError(RuntimeError):
    pass


def lib():
    """Load (building if necessary) libampis_b200.so."""
    global _lib
    if _lib is None:
        path = _build.LIB
        # (re)build when the library is missing or older than its sources -- unless nvcc is not there (a box that
        # only received the prebuilt library): then a stale or missing library fails loudly below
        nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
        if not os.path.exists(path) or (os.path.exists(nvcc) and _build.needs_build()):
            _build.build()
        l = C.CDLL(path)
        if l.ampis_version() != ABI_VERSION:
            raise AmpisNativeError('libampis_b200.so reports ABI %d, this package expects %d: rebuild with '
                                   '`python -m ampis_b200.build --force`' % (l.ampis_version(), ABI_VERSION))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)     # AttributeError if the .so is stale / incomplete
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def synth_lib():
    """Load (building if necessary) libampis_synth.so, the synthetic-data generator.  Never touches libampis_b200.so."""
    global _synth
    if _synth is None:
        l = C.CDLL(_build.build_synth())
        for name, (res, args) in SYNTH_SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _synth = l
    return _synth


def check(rc, what=''):
    if rc != 0:
        msg = lib().ampis_last_error().decode('utf-8', 'replace')
        raise AmpisNativeError('%s failed (%d): %s' % (what or 'libampis_b200 call', rc, msg))


def call(name, *args):
    """Call an int-returning entry point and raise on a non-zero code."""
    check(getattr(lib(), name)(*args), name)
