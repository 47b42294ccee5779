"""Device-side engine: marshals AMPIS mask containers into the GPU mask table and drives
the kernels of libampis_b200.so.  PyTorch is used only for device memory, streams and
(in ampis_b200.distributed) the NCCL plumbing; every computation on masks is one of the
hand-written sm_100a kernels.  There is no CPU fallback anywhere in this module.
"""
import ctypes as C
import itertools
import os
import threading

import numpy as np
import torch

from . import _native as N

LAYOUT_SPAN, LAYOUT_FULL, LAYOUT_CROP = N.LAYOUT_SPAN, N.LAYOUT_FULL, N.LAYOUT_CROP
MODE_IOU, MODE_SAT = N.MODE_IOU, N.MODE_SAT
DEFAULT_LAYOUT = LAYOUT_SPAN
#: storage the matching / satellite functions of the drop-in API paint (crowded images switch to SPAN + contraction)
MATCH_LAYOUT = LAYOUT_CROP


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError('ampis_b200 runs its mask arithmetic on a CUDA device (B200, sm_100a); '
                           'no device is visible and there is no CPU fallback')
    return torch.device('cuda', torch.cuda.current_device())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


#: host arrays up to this size are staged through a pinned copy (asynchronous upload); larger ones are copied
#: straight from pageable memory -- allocating hundreds of MB of pinned memory per call costs more than it saves
PIN_LIMIT_BYTES = 8 << 20


def _dev(a, dtype, device):
    """numpy array -> device tensor of the given torch dtype."""
    t = torch.from_numpy(np.ascontiguousarray(a))
    if t.dtype != dtype:
        t = t.to(dtype)
    if t.numel() == 0:
        return torch.empty(0, dtype=dtype, device=device)
    if torch.device(device).type != 'cuda':
        return t.clone()
    if t.numel() * t.element_size() > PIN_LIMIT_BYTES:
        return t.to(device)
    return t.pin_memory().to(device, non_blocking=True)


#: runs per mask hinted to the fused crop decode kernel (-1: the table's own average; 0: always a warp per mask)
PAINT_RUNS_HINT = int(os.environ.get('AMPIS_PAINT_RUNS_HINT', -1))


#: fused crop decode: 'flat' = a warp decodes several masks at once over their concatenated runs (rle_flat.cu);
#: 'group' = 8 / 16 / 32 lanes per mask (rle_paint.cu, round 1) -- same results, kept for A/B measurements
CROP_DECODE = os.environ.get('AMPIS_CROP_DECODE', 'flat')


class MaskTable(object):
    """Structure-of-arrays table of n masks on the GPU (see include/ampis_b200.h)."""

    def __init__(self, device, n, cnt, cnt_off, cnt_len, h, w, layout):
        self.device, self.n, self.layout = device, int(n), layout
        self.cnt, self.cnt_off, self.cnt_len, self.h, self.w = cnt, cnt_off, cnt_len, h, w
        i32, i64 = torch.int32, torch.int64
        n1 = max(self.n, 1)
        self.cum = torch.empty(max(cnt.numel(), 1), dtype=i32, device=device)
        self.area = torch.empty(n1, dtype=i32, device=device)          # uint32 payload
        self.bbox = torch.empty(4 * n1, dtype=i32, device=device)
        self.span = torch.empty(2 * n1, dtype=i32, device=device)      # uint32 payload
        self.reg = torch.empty(2 * n1, dtype=i32, device=device)       # uint32 payload
        self.reg_chunks = torch.empty(n1, dtype=i64, device=device)
        self.status = torch.empty(n1, dtype=i32, device=device)
        self.bits_off = torch.empty(n1 + 1, dtype=i64, device=device)
        self.cursor = torch.empty(1, dtype=i64, device=device)   # chunks the arena needed (fused path)
        self.fused = False
        self.list = None        # scratch of the flat crop decode (masks left to its fallback kernel)
        self.zeroed = False     # the last measure_paint also cleared the buffer it was handed
        self.bits = None
        self.bits_capacity = 0
        # the last measure_paint may have stored column-convex masks as interval windows (one word per column), which
        # only the pairs join reads: see measure_paint(intervals=True) and require_bitmaps()
        self.intervals = False

    # -- construction steps ---------------------------------------------------------------
    def measure(self):
        N.call('ampis_rle_measure', _p(self.cnt), _p(self.cnt_off), _p(self.cnt_len), _p(self.h), _p(self.w),
               self.n, self.layout, _p(self.cum), _p(self.area), _p(self.bbox), _p(self.span), _p(self.reg),
               _p(self.reg_chunks), _p(self.status), _stream())
        tmp_bytes = N.lib().ampis_scan_tmp_bytes(self.n)
        tmp = torch.empty(max(tmp_bytes // 8, 1), dtype=torch.int64, device=self.device)
        N.call('ampis_exclusive_scan_i64', _p(self.reg_chunks), _p(self.bits_off), self.n, _p(tmp), tmp_bytes,
               _stream())
        return self

    def paint(self, arena=None):
        """RLE -> packed bits.  Without an arena the needed size is read back (one sync)."""
        if arena is None:
            total = int(self.bits_off[self.n].item()) if self.n else 0
            arena = torch.empty(4 * max(total, 1), dtype=torch.int32, device=self.device)
        self.bits = arena
        self.bits_capacity = arena.numel() // 4
        self.intervals = False
        if self.layout == LAYOUT_CROP:
            N.call('ampis_rle_decode_crop', _p(self.cum), _p(self.cnt_off), _p(self.cnt_len), _p(self.bbox),
                   _p(self.h), _p(self.bits_off), self.n, _p(self.bits), self.bits_capacity, _stream())
        else:
            N.call('ampis_rle_decode_packed', _p(self.cum), _p(self.cnt_off), _p(self.cnt_len), _p(self.span),
                   _p(self.reg), _p(self.bits_off), self.n, _p(self.bits), self.bits_capacity, _stream())
        return self

    def measure_paint(self, arena, zero=None, intervals=False):
        """Fused single-launch form of measure() + paint(arena): arena space is handed out by an
        atomic cursor, so the arena must be supplied (size it with a previous measure() or
        generously) and overflow is detected afterwards by check().  zero: a device tensor the launch also clears
        (the dense matrices of the rows that follow; flat crop decode only -- returns with self.zeroed set when the
        kernel took the job, else the caller clears it).  intervals: store column-convex masks as one interval word
        per column (flat crop decode only; smaller windows, a cheaper decode and join).  Such a table can only go to
        the pairs join (intersect_rows with ROWS_KERNEL 'pairs'); every other reader of the windows raises."""
        self.zeroed = False
        self.intervals = False
        self.bits = arena
        self.bits_capacity = arena.numel() // 4
        self.fused = True
        hint = PAINT_RUNS_HINT if PAINT_RUNS_HINT >= 0 else (self.cnt.numel() // max(self.n, 1))
        if self.layout == LAYOUT_CROP and CROP_DECODE == 'flat':
            if self.list is None:
                self.list = torch.empty(self.n + 1, dtype=torch.int32, device=self.device)
            iv = bool(intervals) and pairs_read_intervals()
            if zero is not None and zero.numel() and zero.data_ptr() % 16 == 0:
                N.call('ampis_rle_measure_paint_flat_zero', _p(self.cnt), _p(self.cnt_off), _p(self.cnt_len),
                       _p(self.h), _p(self.w), self.n, _p(self.cum), _p(self.area), _p(self.bbox), _p(self.span),
                       _p(self.reg), _p(self.bits_off), _p(self.status), _p(self.bits), self.bits_capacity,
                       _p(self.cursor), _p(self.list), hint, _p(zero), zero.numel() * zero.element_size(), int(iv),
                       _stream())
                self.zeroed = True
                self.intervals = iv
                return self
            N.call('ampis_rle_measure_paint_flat', _p(self.cnt), _p(self.cnt_off), _p(self.cnt_len), _p(self.h),
                   _p(self.w), self.n, _p(self.cum), _p(self.area), _p(self.bbox), _p(self.span), _p(self.reg),
                   _p(self.bits_off), _p(self.status), _p(self.bits), self.bits_capacity, _p(self.cursor),
                   _p(self.list), hint, int(iv), _stream())
            self.intervals = iv
            return self
        N.call('ampis_rle_measure_paint', _p(self.cnt), _p(self.cnt_off), _p(self.cnt_len), _p(self.h), _p(self.w),
               self.n, self.layout, _p(self.cum), _p(self.area), _p(self.bbox), _p(self.span), _p(self.reg),
               _p(self.bits_off), _p(self.status), _p(self.bits), self.bits_capacity, _p(self.cursor), hint, _stream())
        return self

    def require_bitmaps(self):
        """Raise unless every window of the table is a bitmap (the form all readers but the pairs join expect)."""
        if self.intervals:
            raise ValueError('this mask table holds interval windows (measure_paint(intervals=True)), which only the '
                             'pairs join reads; decode it with intervals=False for this use')
        return self

    def relayout(self, layout):
        """Switch the storage layout of a measured, not yet painted table (re-derives the stored regions)."""
        assert self.bits is None
        if layout != self.layout:
            self.layout = layout
            self.measure()
        return self

    def check(self):
        """Raise on malformed RLE (sum(counts) != h*w), where pycocotools would hang or mis-decode."""
        if self.n and bool((self.status[:self.n] != 0).any().item()):
            bad = torch.nonzero(self.status[:self.n]).flatten()[:8].tolist()
            raise ValueError('malformed RLE: run counts do not sum to h*w for masks %s' % bad)
        if self.bits is not None and self.n:
            need = int((self.cursor[0] if self.fused else self.bits_off[self.n]).item())
            if need > self.bits_capacity:
                raise N.AmpisNativeError('packed-mask arena too small: %d chunks needed, %d available'
                                         % (need, self.bits_capacity))
        return self

    # -- results ----------------------------------------------------------------------------
    def areas_np(self):
        return self.area[:self.n].cpu().numpy().view(np.uint32).copy()

    def bbox_np(self):
        return self.bbox[:4 * self.n].cpu().numpy().reshape(-1, 4).copy()


def pairs_read_intervals():
    """True when the pairs join reads interval windows (its default intersection pass; not with the A/B variants
    AMPIS_PI_FLAT=0 / 2)."""
    return bool(N.lib().ampis_pairs_read_intervals())


def table_from_counts(cnt, cnt_off, cnt_len, h, w, layout=None, arena=None, check=True):
    """Device-resident CSR run counts -> measured + painted MaskTable."""
    layout = DEFAULT_LAYOUT if layout is None else layout
    device = cnt.device
    t = MaskTable(device, cnt_len.numel(), cnt, cnt_off, cnt_len, h, w, layout)
    t.measure().paint(arena)
    if check:
        t.check()
    return t


def _rle_fields(masks):
    """list of COCO RLE dicts -> (list of bytes, h array, w array); mirrors the input
    handling of pycocotools' _frString (str counts are accepted and encoded)."""
    strings = [m['counts'] for m in masks]
    if set(map(type, strings)) - {bytes}:
        for i, c in enumerate(strings):
            if type(c) == str:
                strings[i] = c.encode('ascii')
            elif isinstance(c, (bytes, bytearray)):
                strings[i] = bytes(c)
            else:
                raise TypeError('RLE counts must be compressed bytes/str, got %s' % type(c))
    n = len(strings)
    try:                                    # [h, w] pairs, flattened without building n small arrays
        hw = np.fromiter(itertools.chain.from_iterable(m['size'] for m in masks), np.int64)
        if hw.size != 2 * n:
            raise ValueError
        hw = hw.reshape(n, 2)
    except (ValueError, TypeError):         # sizes that are not plain pairs of ints
        hw = np.asarray([m['size'] for m in masks], np.int64).reshape(n, -1)
    return strings, hw[:, 0], hw[:, 1]


def _upload(device, *arrays):
    """Several small host arrays -> device tensors through ONE pinned staging buffer and ONE copy
    (each numpy array keeps its dtype; pieces are 16-byte aligned views of the same allocation)."""
    arrays = [np.ascontiguousarray(a) for a in arrays]
    offs, total = [], 0
    for a in arrays:
        offs.append(total)
        total += (a.nbytes + 15) & ~15
    if torch.device(device).type != 'cuda' or total > PIN_LIMIT_BYTES:
        return [_dev(a.view(np.int32) if a.dtype == np.uint32 else a, _TORCH_DTYPE[a.dtype.name], device)
                for a in arrays]
    stage = torch.empty(max(total, 16), dtype=torch.uint8, pin_memory=True)
    host = stage.numpy()
    for a, o in zip(arrays, offs):
        host[o:o + a.nbytes] = a.view(np.uint8).reshape(-1)
    dev = stage.to(device, non_blocking=True)
    out = []
    for a, o in zip(arrays, offs):
        t = dev[o:o + a.nbytes].view(_TORCH_DTYPE[a.dtype.name])
        out.append(t if a.size else torch.empty(0, dtype=t.dtype, device=device))
    return out


_TORCH_DTYPE = {'uint8': torch.uint8, 'int32': torch.int32, 'int64': torch.int64, 'float64': torch.float64,
                'uint32': torch.int32}


def table_from_rle(masks, layout=None, paint=True):
    """Host list of compressed RLE dicts -> MaskTable (string decode happens on the GPU)."""
    layout = DEFAULT_LAYOUT if layout is None else layout
    device = require_cuda()
    strings, hs, ws = _rle_fields(masks)
    n = len(strings)
    lens = np.fromiter(map(len, strings), np.int64, n)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    blob = np.frombuffer(b''.join(strings), np.uint8) if n else np.zeros(0, np.uint8)
    d_off, d_h, d_w, d_chars = _upload(device, off, hs.astype(np.int32), ws.astype(np.int32), blob)
    cnt = torch.empty(max(int(off[-1]), 1), dtype=torch.int32, device=device)
    cnt_len = torch.empty(max(n, 1), dtype=torch.int32, device=device)
    N.call('ampis_rle_string_decode', _p(d_chars), _p(d_off), n, _p(cnt), _p(d_off), _p(cnt_len), _stream())
    t = MaskTable(device, n, cnt, d_off, cnt_len, d_h, d_w, layout)
    t.measure()
    if paint:
        t.paint()
    t.check()
    return t


class ImageRows(object):
    """Result of eval_image(): per-row arg-max results and per-mask measurements of one image (numpy)."""
    __slots__ = ('best_col', 'best_inter', 'best_score', 'area', 'bbox', 'span', 'n_rows', 'n_cols', 'hw', 'iou')

    def fill(self):
        """Operand fill (see operand_fill) from the returned spans."""
        slabs = (self.hw[0] * self.hw[1] + 127) // 128
        n = len(self.area)
        return float((self.span[:, 1].astype(np.int64) - self.span[:, 0]).sum()) / max(slabs * n, 1)


_image_ws = {}          # device index -> [device workspace, pinned host workspace]
_image_ws_lock = threading.Lock()


def _workspaces(device):
    """[device workspace, pinned host workspace] of the one-call entries on `device` (created once, grown on demand;
    call with _image_ws_lock held)."""
    ws = _image_ws.get(device.index)
    if ws is None:
        ws = _image_ws[device.index] = [torch.empty(1 << 22, dtype=torch.uint8, device=device),
                                        torch.empty(1 << 20, dtype=torch.uint8, pin_memory=True)]
    return ws


def eval_image(rows_rle, cols_rle, mode, dense_iou=False):
    """One image, rows x columns, through ampis_eval_image_host -- the per-image work of the reference's
    analyze.py:149-164 (G x ceil(P/80) RLE.iou calls + arg-max), analyze.py:315-321 (merge + area per match),
    powder.py:80-86 (S x N RLE.merge + RLE.area) and, with dense_iou, analyze.py:54-112: ONE library call stages the compressed strings,
    runs string decode -> fused measure + crop decode -> rows kernel and brings the per-row results back with one
    synchronisation (the drop-in matching functions call this once per image).  Raises ValueError when the masks
    do not share one image size and on malformed RLE (like MaskTable.check())."""
    device = require_cuda()
    strings, hs, ws = _rle_fields(list(rows_rle) + list(cols_rle))
    n_rows, n_cols = len(rows_rle), len(cols_rle)
    n = n_rows + n_cols
    if n and ((hs != hs[0]).any() or (ws != ws[0]).any()):
        k = int(np.nonzero((hs != hs[0]) | (ws != ws[0]))[0][0])
        raise ValueError('masks of different image sizes cannot be compared (%s vs %s)'
                         % ((int(hs[0]), int(ws[0])), (int(hs[k]), int(ws[k]))))
    off = np.zeros(n + 1, np.int64)
    np.cumsum(np.fromiter(map(len, strings), np.int64, n), out=off[1:])
    blob = b''.join(strings)
    r = ImageRows()
    r.n_rows, r.n_cols, r.hw = n_rows, n_cols, (int(hs[0]), int(ws[0])) if n else (0, 0)
    r.best_col = np.empty(n_rows, np.int32)
    r.best_inter = np.empty(n_rows, np.uint32)
    r.best_score = np.empty(n_rows, np.float64)
    r.area = np.empty(n, np.uint32)
    r.bbox = np.empty((n, 4), np.int32)
    r.span = np.empty((n, 2), np.uint32)
    status = np.empty(n, np.int32)
    r.iou = np.zeros((n_rows, n_cols)) if dense_iou else None       # float64 IoU matrix of _piecewise_iou
    if n == 0:
        return r
    need = C.c_int64(0)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    lib = N.lib()
    with _image_ws_lock:
        ws_pair = _workspaces(device)
        for _ in range(8):
            d_ws, h_ws = ws_pair
            rc = lib.ampis_eval_image_host(blob, ptr(off), n_rows, n_cols, r.hw[0], r.hw[1], mode, ROWS_GRID_MIN_COLS,
                                           _p(d_ws), d_ws.numel(), _p(h_ws), h_ws.numel(), ptr(r.best_col),
                                           ptr(r.best_inter), ptr(r.best_score), ptr(r.area), ptr(r.bbox), ptr(r.span),
                                           ptr(status), ptr(r.iou) if dense_iou and r.iou.size else None,
                                           C.byref(need), _stream())
            if rc != N.ENOSPC:
                break
            if need.value < 0:          # pinned host workspace too small
                ws_pair[1] = torch.empty(int(-need.value * 3 // 2), dtype=torch.uint8, pin_memory=True)
            else:
                torch.cuda.current_stream().synchronize()
                ws_pair[0] = None
                ws_pair[0] = torch.empty(int(need.value * 3 // 2), dtype=torch.uint8, device=device)
        N.check(rc, 'ampis_eval_image_host')
    if status.any():
        raise ValueError('malformed RLE: run counts do not sum to h*w for masks %s' % np.nonzero(status)[0][:8].tolist())
    return r


class ImagesRows(object):
    """Result of eval_images(): per-row arg-max results and per-mask measurements of a list of images, image after
    image (numpy).  row_off[g] / mask_off[g] = first row / first mask of image g (rows of an image come before its
    columns in the mask arrays)."""
    __slots__ = ('best_col', 'best_inter', 'best_score', 'area', 'bbox', 'span', 'status', 'n_rows', 'n_cols', 'hw',
                 'row_off', 'mask_off', 'pairs_found', 'crowded')

    def fill(self, g=0):
        """Operand fill of image g (see operand_fill) from the returned spans."""
        m0, m1 = int(self.mask_off[g]), int(self.mask_off[g + 1])
        slabs = (int(self.hw[g, 0]) * int(self.hw[g, 1]) + 127) // 128
        sp = self.span[m0:m1]
        return float((sp[:, 1].astype(np.int64) - sp[:, 0]).sum()) / max(slabs * (m1 - m0), 1)


_marshal = None


def marshal():
    """The CPython extension that walks lists of RLE dicts (ampis_b200/cext/pymarshal.c), built on first use."""
    global _marshal
    if _marshal is None:
        from . import build as _build
        _build.build_marshal()
        from . import _pymarshal
        _marshal = _pymarshal
    return _marshal


#: candidate pairs above this fraction of all row x column pairs: the culled walk is skipped on the device and the
#: image goes to the tensor-core contraction (profiles/crossover_r01.md: the kernels cross at fill 0.25, where a
#: fifth of all pairs have overlapping boxes)
CROWD_PAIR_FRACTION = 0.2

def _addr(a):
    """Address of a numpy array's data: 0.7 us through the buffer protocol against 2.8 us for a.ctypes.data /
    __array_interface__ -- a single-image call passes thirteen arrays."""
    try:
        return C.addressof(C.c_char.from_buffer(a))
    except (TypeError, ValueError, BufferError):          # empty, read-only or non-contiguous
        return a.ctypes.data


_images_cache = {}      # mode -> (key, references that keep the strings alive, result)


def _marshal_images(rows_lists, cols_lists, refs):
    """The per-image sizes of a list of images (an ImagesRows with n_rows, n_cols, row_off, mask_off and hw set) and
    the address, length and size of every compressed string, from the C marshaller: (r, ptr, ln, hw, n, R).  refs:
    a list that receives the string objects, or None.  Raises ValueError when the masks of an image do not share one
    size."""
    n_img = len(rows_lists)
    assert len(cols_lists) == n_img
    r = ImagesRows()
    if n_img == 1:
        # one image per call (det_seg_scores, _rle_satellite_match, mask_areas): the bookkeeping in plain Python -- a
        # dozen numpy calls on one-element arrays cost more than the GPU needs for the image
        G1, P1 = len(rows_lists[0]), len(cols_lists[0])
        n, R = G1 + P1, G1
        r.n_rows, r.n_cols = np.array([G1], np.int32), np.array([P1], np.int32)
        r.row_off, r.mask_off = np.array([0, G1], np.int64), np.array([0, n], np.int64)
    else:
        r.n_rows = np.fromiter(map(len, rows_lists), np.int32, n_img)
        r.n_cols = np.fromiter(map(len, cols_lists), np.int32, n_img)
        r.row_off = np.zeros(n_img + 1, np.int64)
        np.cumsum(r.n_rows, out=r.row_off[1:])
        r.mask_off = np.zeros(n_img + 1, np.int64)
        np.cumsum(r.n_rows.astype(np.int64) + r.n_cols, out=r.mask_off[1:])
        n, R = int(r.mask_off[-1]), int(r.row_off[-1])
    n1 = max(n, 1)
    ptr, ln, hw = np.empty(n1, np.uint64), np.empty(n1, np.int32), np.empty((n1, 2), np.int32)
    lists = [None] * (2 * n_img)
    lists[0::2] = rows_lists
    lists[1::2] = cols_lists
    got, mixed = marshal().gather(lists, ptr, ln, hw, refs)
    assert got == n
    # one size per image: the first mask of each image speaks for it.  The marshaller has checked every list on its
    # own (mixed = first list holding two sizes); what is left is rows against columns of the same image
    if n_img == 1 and mixed < 0 and (G1 == 0 or P1 == 0 or (hw[0, 0] == hw[G1, 0] and hw[0, 1] == hw[G1, 1])):
        r.hw = np.array([[int(hw[0, 0]), int(hw[0, 1])] if n else [0, 0]], np.int64)
    else:
        first = np.minimum(r.mask_off[:-1], max(n - 1, 0))
        r.hw = np.where(((r.n_rows + r.n_cols) > 0)[:, None], hw[first], 0).astype(np.int64)
        if n:
            first_col = np.minimum(r.mask_off[:-1] + r.n_rows, n - 1)
            both = (r.n_rows > 0) & (r.n_cols > 0)
            clash = np.nonzero(both & (hw[first_col] != hw[first]).any(axis=1))[0]
            if mixed >= 0 or len(clash):
                g = min(([mixed // 2] if mixed >= 0 else []) + [int(c) for c in clash[:1]])
                m0, m1 = int(r.mask_off[g]), int(r.mask_off[g + 1])
                k = m0 + int(np.nonzero((hw[m0:m1] != hw[m0]).any(axis=1))[0][0])
                raise ValueError('masks of different image sizes cannot be compared (%s vs %s)'
                                 % (tuple(int(v) for v in hw[m0]), tuple(int(v) for v in hw[k])))
    return r, ptr, ln, hw, n, R


def _call_growing(device, name, call):
    """rc = call(d_ws, h_ws, need) of a one-call entry with the shared workspaces of `device`, grown and retried as
    AMPIS_ENOSPC asks; raises on any other error."""
    need = C.c_int64(0)
    with _image_ws_lock:
        ws_pair = _workspaces(device)
        for _ in range(8):
            d_ws, h_ws = ws_pair
            rc = call(d_ws, h_ws, need)
            if rc != N.ENOSPC:
                break
            if need.value < 0:          # pinned host workspace too small
                ws_pair[1] = torch.empty(int(-need.value * 3 // 2), dtype=torch.uint8, pin_memory=True)
            else:
                torch.cuda.current_stream().synchronize()
                ws_pair[0] = None
                ws_pair[0] = torch.empty(int(need.value * 3 // 2), dtype=torch.uint8, device=device)
        N.check(rc, name)


def _check_status(status):
    if status.any():
        raise ValueError('malformed RLE: run counts do not sum to h*w for masks %s' % np.nonzero(status)[0][:8].tolist())


def eval_images(rows_lists, cols_lists, mode, crowd_frac=-1.0, cache=False):
    """Many images, rows x columns each, through ampis_eval_images_host -- the per-image work of the reference's
    analyze.py:149-164 (+ 315-321) or powder.py:80-86 for a whole list of images in ONE library call: the C
    marshaller hands over the address of every compressed string (no join, no per-mask Python work), the library
    gathers them into pinned memory and runs string decode -> flat measure + crop decode -> column grids ->
    candidate-pair join -> AND+popc -> per-row arg-max with one upload, one download and one synchronisation.
    rows_lists[g] / cols_lists[g]: lists of RLE dicts of image g.  Raises ValueError when the masks of an image do
    not share one size and on malformed RLE.  cache=True keeps the last result per mode and returns it when the very
    same string objects come again (a loop over IoU thresholds costs one evaluation)."""
    device = require_cuda()
    n_img = len(rows_lists)
    refs = [] if cache else None            # the string objects themselves: their addresses are the cache key
    r, ptr, ln, hw, n, R = _marshal_images(rows_lists, cols_lists, refs)
    key = None
    if cache:
        key = (mode, float(crowd_frac), ptr[:n].tobytes(), ln[:n].tobytes(), hw[:n].tobytes(), r.n_rows.tobytes())
        hit = _images_cache.get(mode)
        if hit is not None and hit[0] == key:
            return hit[2]
    r.best_col = np.empty(R, np.int32)
    r.best_inter = np.empty(R, np.uint32)
    r.best_score = np.empty(R, np.float64)
    r.area = np.empty(n, np.uint32)
    r.bbox = np.empty((n, 4), np.int32)
    r.span = np.empty((n, 2), np.uint32)
    r.status = np.empty(n, np.int32)
    r.pairs_found, r.crowded = 0, False
    if n:
        found, crowded = C.c_int64(0), C.c_int32(0)
        pa = _addr                                               # plain address (argtypes say c_void_p)
        h32, w32 = np.ascontiguousarray(r.hw[:, 0].astype(np.uint32)), np.ascontiguousarray(r.hw[:, 1].astype(np.uint32))
        lib = N.lib()
        _call_growing(device, 'ampis_eval_images_host', lambda d_ws, h_ws, need: lib.ampis_eval_images_host(
            pa(ptr), pa(ln), n_img, pa(r.n_rows), pa(r.n_cols), pa(h32), pa(w32), mode, 0, float(crowd_frac), _p(d_ws),
            d_ws.numel(), _p(h_ws), h_ws.numel(), pa(r.best_col), pa(r.best_inter), pa(r.best_score), pa(r.area),
            pa(r.bbox), pa(r.span), pa(r.status), None, 0, None, None, C.byref(found), C.byref(crowded),
            C.byref(need), _stream()))
        r.pairs_found, r.crowded = int(found.value), bool(crowded.value)
        _check_status(r.status)
    if cache:
        # the references keep every string object alive, so an address in the key cannot be recycled while the entry lives
        _images_cache[mode] = (key, refs, r)
    return r


class ImagesSweep(object):
    """Result of eval_images_sweep() (numpy), thresholds in the sorted order they were passed in: totals and
    seg_totals int64 [K, T, 3] (TP / FP / FN and seg TP / FP / FN), counts int32 and seg int64 [n_images, K, T, 3]
    (None unless per_image), n_rows / n_cols per image, pairs_found."""
    __slots__ = ('totals', 'seg_totals', 'counts', 'seg', 'n_rows', 'n_cols', 'pairs_found')


def eval_images_sweep(rows_lists, cols_lists, levels, n_levels, iou_sorted, per_image=True):
    """Detection and segmentation counts of many images over a grid of score x IoU thresholds in ONE library call
    (ampis_eval_images_sweep_host): the decode, join and intersections of eval_images once, then the staircase and
    count passes of csrc/score.cu.  rows_lists / cols_lists: ground truth / predictions of every image (RLE dicts).
    levels: uint16 per prediction in image order, the number of the n_levels sorted score thresholds strictly below its
    score (kept at sorted threshold k iff level > k).  iou_sorted: IoU thresholds, ascending, each >= 0.  No identity
    cache: the result depends on the levels as well as on the strings."""
    device = require_cuda()
    n_img = len(rows_lists)
    r, ptr, ln, hw, n, R = _marshal_images(rows_lists, cols_lists, None)
    iou = np.ascontiguousarray(iou_sorted, np.float64)
    K, T = int(n_levels), len(iou)
    lv = np.ascontiguousarray(levels, np.uint16)
    assert len(lv) == int(r.n_cols.astype(np.int64).sum())
    out = ImagesSweep()
    out.n_rows, out.n_cols, out.pairs_found = r.n_rows, r.n_cols, 0
    out.totals = np.zeros((K, T, 3), np.int64)
    out.seg_totals = np.zeros((K, T, 3), np.int64)
    out.counts = np.zeros((n_img, K, T, 3), np.int32) if per_image else None
    out.seg = np.zeros((n_img, K, T, 3), np.int64) if per_image else None
    status = np.empty(max(n, 1), np.int32)
    found = C.c_int64(0)
    pa = _addr
    h32, w32 = np.ascontiguousarray(r.hw[:, 0].astype(np.uint32)), np.ascontiguousarray(r.hw[:, 1].astype(np.uint32))
    lib = N.lib()
    _call_growing(device, 'ampis_eval_images_sweep_host', lambda d_ws, h_ws, need: lib.ampis_eval_images_sweep_host(
        pa(ptr), pa(ln), n_img, pa(r.n_rows), pa(r.n_cols), pa(h32), pa(w32), 0, pa(lv) if len(lv) else None, K,
        pa(iou), T, _p(d_ws), d_ws.numel(), _p(h_ws), h_ws.numel(), pa(status), pa(out.totals), pa(out.seg_totals),
        pa(out.counts) if per_image and out.counts.size else None, pa(out.seg) if per_image and out.seg.size else None,
        C.byref(found), C.byref(need), _stream()))
    out.pairs_found = int(found.value)
    _check_status(status[:n])
    return out


class ImagesSatSweep(object):
    """Result of eval_images_sat_sweep() (numpy), thresholds in sorted order: totals int64 [K, L, T, 3] (matched,
    unmatched, satellited particles), spp_hist int64 [K, L, T, n_bins], counts int32 [n_images, K, L, T, 3] (None
    unless per_image), n_rows (satellites) / n_cols (particles) per image, pairs_found."""
    __slots__ = ('totals', 'spp_hist', 'counts', 'n_rows', 'n_cols', 'pairs_found')


def eval_images_sat_sweep(sat_lists, part_lists, plevels, n_plevels, slevels, n_slevels, match_sorted, n_bins,
                          per_image=True):
    """Satellite statistics of many images over a grid of particle-score x satellite-score x match thresholds in ONE
    library call (ampis_eval_images_sat_sweep_host): the decode, join and intersections of eval_images in MODE_SAT
    once, then the staircase and satellite count passes of csrc/score.cu.  sat_lists / part_lists: satellites (rows)
    and particles (columns) of every image (RLE dicts).  plevels / slevels: uint16 per particle / satellite in image
    order, the number of the n_plevels / n_slevels sorted score thresholds strictly below its score.  match_sorted:
    match thresholds, ascending, each >= 0.  n_bins: 1 + at least the most satellites of any image."""
    device = require_cuda()
    n_img = len(sat_lists)
    r, ptr, ln, hw, n, R = _marshal_images(sat_lists, part_lists, None)
    mt = np.ascontiguousarray(match_sorted, np.float64)
    K, L, T, B = int(n_plevels), int(n_slevels), len(mt), int(n_bins)
    plv, slv = np.ascontiguousarray(plevels, np.uint16), np.ascontiguousarray(slevels, np.uint16)
    assert len(plv) == int(r.n_cols.astype(np.int64).sum()) and len(slv) == R
    out = ImagesSatSweep()
    out.n_rows, out.n_cols, out.pairs_found = r.n_rows, r.n_cols, 0
    out.totals = np.zeros((K, L, T, 3), np.int64)
    out.spp_hist = np.zeros((K, L, T, B), np.int64)
    out.counts = np.zeros((n_img, K, L, T, 3), np.int32) if per_image else None
    status = np.empty(max(n, 1), np.int32)
    found = C.c_int64(0)
    pa = _addr
    h32, w32 = np.ascontiguousarray(r.hw[:, 0].astype(np.uint32)), np.ascontiguousarray(r.hw[:, 1].astype(np.uint32))
    lib = N.lib()
    _call_growing(device, 'ampis_eval_images_sat_sweep_host', lambda d_ws, h_ws, need: lib.ampis_eval_images_sat_sweep_host(
        pa(ptr), pa(ln), n_img, pa(r.n_rows), pa(r.n_cols), pa(h32), pa(w32), 0, pa(plv) if len(plv) else None, K,
        pa(slv) if len(slv) else None, L, pa(mt), T, B, _p(d_ws), d_ws.numel(), _p(h_ws), h_ws.numel(), pa(status),
        pa(out.totals), pa(out.spp_hist), pa(out.counts) if per_image and out.counts.size else None, C.byref(found),
        C.byref(need), _stream()))
    out.pairs_found = int(found.value)
    _check_status(status[:n])
    return out


def measure_rle(masks):
    """(area uint32[n], tight bbox int32[n, 4]) of a list of RLE dicts: rleArea (structures.py:568,571;
    powder.py:264) and the box extract_boxes (data_utils.py:229-239) reads off the decoded mask.  Masks of one image size go through the one-call entry point (no intersection is run); mixed
    sizes through the table API."""
    masks = list(masks)
    if masks:
        try:
            r = eval_images([masks], [[]], MODE_IOU, cache=True)      # repeated measurements of one list: one call
            return r.area.copy(), r.bbox.copy()                          # the cached arrays stay untouched
        except ValueError as e:
            if 'different image sizes' not in str(e):
                raise
    t = table_from_rle(masks, paint=False)
    return t.areas_np(), t.bbox_np()


class Groups(object):
    """Row/column bookkeeping of a batch: group g (an image) owns rows (ground truth or
    satellites) and columns (predictions or particles); all are mask ids of one MaskTable."""

    def __init__(self, device, row_mask, row_grp, grp_row_begin, grp_row_count, grp_col_begin, grp_col_count,
                 dense=False):
        self.device = device
        self.n_rows = int(len(row_mask))
        self.n_groups = int(len(grp_row_begin))
        self.max_cols = int(max(grp_col_count)) if self.n_groups else 0
        self.h_row_count = np.asarray(grp_row_count, np.int64)
        self.h_col_count = np.asarray(grp_col_count, np.int64)
        self.h_row_begin = np.asarray(grp_row_begin, np.int64)
        rpb = N.lib().ampis_rows_per_block()
        nb = (self.h_row_count + rpb - 1) // rpb                    # CTAs per group
        blk_grp = np.repeat(np.arange(self.n_groups, dtype=np.int64), nb)
        first = np.zeros(self.n_groups + 1, np.int64)
        np.cumsum(nb, out=first[1:])
        blk_row0 = self.h_row_begin[blk_grp] + rpb * (np.arange(int(first[-1]), dtype=np.int64) - first[blk_grp])
        self.n_blocks = int(first[-1])
        i32 = np.int32
        (self.row_mask, self.row_grp, self.blk_grp, self.blk_row0, self.grp_row_begin, self.grp_row_count,
         self.grp_col_begin, self.grp_col_count) = _upload(
            device, np.asarray(row_mask, i32), np.asarray(row_grp, i32), blk_grp.astype(i32), blk_row0.astype(i32),
            np.asarray(grp_row_begin, i32), np.asarray(grp_row_count, i32), np.asarray(grp_col_begin, i32),
            np.asarray(grp_col_count, i32))
        self.imat_off = None
        self.h_imat_off = None
        self.imat_size = 0
        if dense:
            sizes = self.h_row_count * self.h_col_count
            off = np.zeros(self.n_groups + 1, np.int64)
            np.cumsum(sizes, out=off[1:])
            self.h_imat_off = off
            self.imat_size = int(off[-1])
            self.imat_off = _dev(off[:-1], torch.int64, device)

    def mma_tiles(self, pair=False):
        """Tile list of the dense kernels: every group's dense matrix cut into tiles of the kernel's size -- 128 x 256
        (tcgen05 contraction, ampis_intersect_tcgen05), 256 x 256 (CTA pairs, pair=True) or the square tile of the
        TMA-staged AND+popc kernel (pair='tma'); built once, cached."""
        cache = getattr(self, '_mma', None)
        if cache is None:
            cache = self._mma = {}
        if pair not in cache:
            assert self.imat_off is not None, 'the dense kernels write dense matrices: Groups(dense=True)'
            lib = N.lib()
            if pair == 'tma':
                tm = tn = lib.ampis_tma_tile()
            else:
                tm, tn = (lib.ampis_mma_pair_tile_rows(), lib.ampis_mma_pair_tile_cols()) if pair else \
                    (lib.ampis_mma_tile_rows(), lib.ampis_mma_tile_cols())
            grp, m0, n0 = [], [], []
            for g in range(self.n_groups):
                G, P = int(self.h_row_count[g]), int(self.h_col_count[g])
                if G == 0 or P == 0:
                    continue
                mm, nn = np.meshgrid(np.arange(0, G, tm), np.arange(0, P, tn), indexing='ij')
                grp.append(np.full(mm.size, g, np.int32))
                m0.append(mm.ravel().astype(np.int32))
                n0.append(nn.ravel().astype(np.int32))
            cat = lambda v: np.concatenate(v) if v else np.zeros(0, np.int32)
            cache[pair] = (len(cat(grp)), _dev(cat(grp), torch.int32, self.device),
                           _dev(cat(m0), torch.int32, self.device), _dev(cat(n0), torch.int32, self.device))
        return cache[pair]

    @staticmethod
    def interleaved(device, n_rows_per_group, n_cols_per_group, dense=False):
        """Mask table laid out image by image as [rows of g][cols of g]."""
        G = np.asarray(n_rows_per_group, np.int64)
        P = np.asarray(n_cols_per_group, np.int64)
        ng = len(G)
        start = np.zeros(ng + 1, np.int64)
        np.cumsum(G + P, out=start[1:])
        row_begin = np.zeros(ng + 1, np.int64)
        np.cumsum(G, out=row_begin[1:])
        row_grp = np.repeat(np.arange(ng, dtype=np.int64), G)
        row_mask = np.arange(int(row_begin[-1]), dtype=np.int64) - row_begin[row_grp] + start[row_grp]
        return Groups(device, row_mask, row_grp, row_begin[:-1], G, start[:-1] + G, P, dense=dense)


class RowResult(object):
    def __init__(self, best_col, best_inter, best_score, imat):
        self.best_col, self.best_inter, self.best_score, self.imat = best_col, best_inter, best_score, imat


#: from this many column masks per image on, the crop rows kernel finds its candidates through a
#: uniform grid over the image (ampis_intersect_rows_grid) instead of scanning every column's box
#: (measured: C2, 500 columns per image, rows kernel 1.25 -> 1.00 ms per 1,000 images; C4, 5,000 columns, 2.4 ->
#: 0.25 ms per 40 images; below a few hundred columns the six small launches that build the grid cost more)
ROWS_GRID_MIN_COLS = int(os.environ.get('AMPIS_ROWS_GRID_MIN_COLS', 64))


class ColumnGrid(object):
    """Uniform 32 x 32 grid over every image of a batch with the column masks binned by bounding box
    (the spatial index of ampis_intersect_rows_grid), built by one kernel launch.  build() needs the measured boxes
    of `table`; without a capacity a sizing launch is made first and the number of entries read back (one sync)."""

    def __init__(self, device, n_groups, capacity=None):
        self.device, self.n_groups = device, int(n_groups)
        cells = N.lib().ampis_grid_cells()
        self.shift = torch.empty(max(self.n_groups, 1), dtype=torch.int32, device=device)
        self.cell_off = torch.empty(max(self.n_groups, 1) * (cells + 1), dtype=torch.int64, device=device)
        self.cursor = torch.zeros(1, dtype=torch.int64, device=device)
        self.entries = self.entry_bbox = None
        self.capacity = None
        if capacity is not None:
            self._alloc(int(capacity))

    def _alloc(self, capacity):
        self.capacity = capacity
        self.entries = torch.empty(max(capacity, 1), dtype=torch.int32, device=self.device)
        self.entry_bbox = torch.empty(4 * max(capacity, 1), dtype=torch.int32, device=self.device)

    def _launch(self, table, groups, capacity):
        N.call('ampis_grid_build', _p(table.bbox), _p(groups.grp_col_begin), _p(groups.grp_col_count),
               groups.n_groups, _p(self.shift), _p(self.cell_off), _p(self.entries), _p(self.entry_bbox), capacity,
               _p(self.cursor), _stream())

    def build(self, table, groups):
        if self.entries is None:
            self._launch(table, groups, 0)          # sizing pass: counts only
            self._alloc(self.needed())
        self._launch(table, groups, self.capacity)
        return self

    def needed(self):
        """Entries the last build() wanted (read-back; compare with .capacity)."""
        return int(self.cursor.item())


#: grid-pruned crop rows: 'pairs' = spatial join in three flat passes (intersect_pairs.cu); 'grid' = one kernel,
#: eight lanes per row (intersect_grid.cu, round 1) -- same results, kept for A/B measurements
ROWS_KERNEL = os.environ.get('AMPIS_ROWS_KERNEL', 'pairs')


class PairList(object):
    """Candidate pairs of ampis_intersect_rows_pairs: (row mask, column mask) ids, their intersections, and the
    range of every row.  `count` may exceed `capacity` (then the results are void and the list must grow)."""

    def __init__(self, device, n_rows, capacity):
        self.capacity = int(capacity)
        c = max(self.capacity, 1)
        self.ab = torch.empty(2 * c, dtype=torch.int32, device=device)
        self.desc = torch.empty(8 * c, dtype=torch.int32, device=device)        # 32-byte overlap descriptors
        self.inter = torch.empty(c, dtype=torch.int32, device=device)          # uint32 payload
        self.row_off = torch.empty(max(n_rows, 1), dtype=torch.int64, device=device)
        self.row_cnt = torch.empty(max(n_rows, 1), dtype=torch.int32, device=device)
        self.count = torch.zeros(1, dtype=torch.int64, device=device)

    def needed(self):
        return int(self.count.item())


class SparseRows(object):
    """Sparse output of ampis_intersect_rows_grid: the non-zero intersections as (row, column-in-group,
    intersection) triplets, unordered; `count` may exceed `capacity` (the excess was dropped)."""

    def __init__(self, device, capacity):
        self.capacity = int(capacity)
        c = max(self.capacity, 1)
        self.row = torch.empty(c, dtype=torch.int32, device=device)
        self.col = torch.empty(c, dtype=torch.int32, device=device)
        self.inter = torch.empty(c, dtype=torch.int32, device=device)      # uint32 payload
        self.count = torch.zeros(1, dtype=torch.int64, device=device)

    def triplets(self):
        """(row, col, inter) as int64 device tensors sorted by (row, col); raises if entries were dropped."""
        n = int(self.count.item())
        if n > self.capacity:
            raise N.AmpisNativeError('sparse intersection list too small: %d triplets, capacity %d'
                                     % (n, self.capacity))
        r, c = self.row[:n].long(), self.col[:n].long()
        order = torch.argsort((r << 32) | c)
        return r[order], c[order], (self.inter[:n].long() & 0xffffffff)[order]


def intersect_rows(table, groups, mode, out=None, grid=None, sparse=None, pairs=None, zeroed=None, zero_stream=None):
    """Run the fused row kernel.  Returns device tensors (no sync).  Crop-layout tables with many
    columns per image (ROWS_GRID_MIN_COLS), or whenever a ColumnGrid / SparseRows is passed, go through
    the grid-pruned kernels; grid='scan' forces the all-columns scan.  The grid-pruned form is the three-pass
    join (ROWS_KERNEL 'pairs'; `pairs` = a pre-sized PairList, else one is sized here with a read-back)
    or the single rows kernel of round 1 ('grid').  zeroed: True = the dense matrices are all zeros already on this stream (MaskTable.measure_paint(zero=...)), or a
    CUDA event after which they are (the caller cleared them on another stream); the join then does not clear them.
    zero_stream: a torch stream on which the join zeroes the dense matrices itself while its first two passes run."""
    dev = table.device
    nr = max(groups.n_rows, 1)
    use_grid = table.layout == LAYOUT_CROP and not isinstance(grid, str) and \
        (grid is not None or sparse is not None or groups.max_cols >= ROWS_GRID_MIN_COLS)
    if not (use_grid and ROWS_KERNEL == 'pairs'):
        table.require_bitmaps()
    if out is None:
        imat = torch.empty(max(groups.imat_size, 1), dtype=torch.int32, device=dev) \
            if groups.imat_off is not None else None
        out = RowResult(torch.empty(nr, dtype=torch.int32, device=dev),
                        torch.empty(nr, dtype=torch.int32, device=dev),
                        torch.empty(nr, dtype=torch.float64, device=dev), imat)
    assert use_grid or sparse is None, 'sparse output comes from the grid kernel (crop layout)'
    if use_grid:
        if grid is None:
            grid = ColumnGrid(dev, groups.n_groups)
        grid.build(table, groups)
        out.grid = grid
        if sparse is not None:
            sparse.count.zero_()
        if ROWS_KERNEL == 'pairs':
            own = pairs is None
            if own:
                pairs = PairList(dev, groups.n_rows, 8 * groups.n_rows + 4096)
            if zeroed is not None and zeroed is not True:
                torch.cuda.current_stream().wait_event(zeroed)
            while True:
                N.call('ampis_intersect_rows_pairs', _p(table.bits), _p(table.bits_off),
                       _p(table.reg) if table.intervals else None, _p(table.bbox),
                       _p(table.area), _p(groups.row_mask), _p(groups.row_grp), groups.n_rows,
                       _p(groups.grp_row_begin), _p(groups.grp_col_begin), _p(groups.grp_col_count), _p(grid.shift),
                       _p(grid.cell_off), _p(grid.entries), _p(grid.entry_bbox), grid.capacity, _p(pairs.ab),
                       _p(pairs.desc), _p(pairs.inter), pairs.capacity, _p(pairs.row_off), _p(pairs.row_cnt), _p(pairs.count),
                       _p(groups.imat_off), mode, _p(out.imat),
                       groups.imat_size if groups.imat_off is not None and out.imat is not None and zeroed is None else 0,
                       _p(out.best_col), _p(out.best_inter), _p(out.best_score),
                       _p(sparse.row) if sparse else None, _p(sparse.col) if sparse else None,
                       _p(sparse.inter) if sparse else None, sparse.capacity if sparse else 0,
                       _p(sparse.count) if sparse else None,
                       C.c_void_p(zero_stream.cuda_stream) if zero_stream is not None else None, _stream())
                if not own or pairs.needed() <= pairs.capacity:
                    break
                pairs = PairList(dev, groups.n_rows, pairs.needed())         # crowded images: grow and repeat
                if sparse is not None:
                    sparse.count.zero_()
            out.pairs = pairs
            return out
        N.call('ampis_intersect_rows_grid', _p(table.bits), _p(table.bits_off), _p(table.bbox), _p(table.area),
               _p(groups.row_mask), _p(groups.blk_grp), _p(groups.blk_row0), groups.n_blocks,
               _p(groups.grp_row_begin), _p(groups.grp_row_count), _p(groups.grp_col_begin),
               _p(groups.grp_col_count), _p(grid.shift), _p(grid.cell_off), _p(grid.entries), _p(grid.entry_bbox),
               grid.capacity, _p(groups.imat_off), mode, _p(out.imat),
               groups.imat_size if groups.imat_off is not None and out.imat is not None else 0,
               _p(out.best_col), _p(out.best_inter), _p(out.best_score),
               _p(sparse.row) if sparse else None, _p(sparse.col) if sparse else None,
               _p(sparse.inter) if sparse else None, sparse.capacity if sparse else 0,
               _p(sparse.count) if sparse else None, _stream())
        return out
    if table.layout == LAYOUT_CROP:
        N.call('ampis_intersect_rows_crop', _p(table.bits), _p(table.bits_off), _p(table.bbox), _p(table.area),
               _p(groups.row_mask), _p(groups.blk_grp), _p(groups.blk_row0), groups.n_blocks,
               _p(groups.grp_row_begin), _p(groups.grp_row_count), _p(groups.grp_col_begin),
               _p(groups.grp_col_count), _p(groups.imat_off), mode, _p(out.imat), _p(out.best_col),
               _p(out.best_inter), _p(out.best_score), _stream())
        return out
    N.call('ampis_intersect_rows', _p(table.bits), _p(table.bits_off), _p(table.reg), _p(table.span),
           _p(table.bbox), _p(table.area), _p(groups.row_mask), _p(groups.blk_grp), _p(groups.blk_row0),
           groups.n_blocks, _p(groups.grp_row_begin), _p(groups.grp_row_count), _p(groups.grp_col_begin),
           _p(groups.grp_col_count), _p(groups.imat_off), mode, _p(out.imat), _p(out.best_col),
           _p(out.best_inter), _p(out.best_score), _stream())
    return out


def _span_orders(table, groups):
    """Per-group orders of the rows and of the columns by first occupied slab (device int32 arrays in
    the index spaces ampis_intersect_tcgen05 expects).  Index plumbing with torch sorts; the masks
    themselves are not touched."""
    n = table.n
    lo = table.span[:2 * n].view(n, 2)[:, 0].to(torch.int64) & 0xffffffff
    if getattr(groups, '_col_grp', None) is None:
        col_grp = np.full(n, -1, np.int64)          # group of every column mask (host bookkeeping, cached)
        cb, cc = groups.grp_col_begin.cpu().numpy(), groups.h_col_count
        for g in range(groups.n_groups):
            col_grp[cb[g]:cb[g] + cc[g]] = g
        groups._col_grp = _dev(col_grp, torch.int64, table.device)
        groups._row_begin_of_row = groups.grp_row_begin.long()[groups.row_grp.long()]
    # rows: sort (group, span start); group blocks stay where they are, subtract the block start
    key_r = (groups.row_grp.long() << 32) | lo[groups.row_mask.long()]
    row_order = (torch.argsort(key_r, stable=True) - groups._row_begin_of_row).to(torch.int32)
    # columns: same over mask ids; non-column masks get the largest key and stay out of every block
    cg = groups._col_grp
    key_c = torch.where(cg >= 0, (cg << 32) | lo, torch.full_like(lo, 1 << 62))
    order_c = torch.argsort(key_c, stable=True)               # sorted position -> mask id, grouped by image
    n_cols = int((cg >= 0).sum().item()) if getattr(groups, '_n_cols', None) is None else groups._n_cols
    groups._n_cols = n_cols
    col_ids = order_c[:n_cols]
    g_of = cg[col_ids]
    begin = groups.grp_col_begin.long()[g_of]
    # position of every sorted column inside its group: columns of a group are consecutive in the sort
    first_of_group = torch.zeros(groups.n_groups + 1, dtype=torch.int64, device=table.device)
    first_of_group[1:] = torch.cumsum(torch.from_numpy(groups.h_col_count).to(table.device), 0)
    pos = torch.arange(n_cols, device=table.device) - first_of_group[g_of]
    col_order = torch.zeros(max(n, 1), dtype=torch.int32, device=table.device)
    col_order[begin + pos] = (col_ids - begin).to(torch.int32)
    return row_order, col_order


#: tensor-core contraction on CTA pairs (tcgen05 cta_group::2, 256 x 256 tiles) instead of single CTAs
#: (128 x 256 tiles): 'auto' = pairs when the tiles contract the full pixel range (sort=False: tensor pipe 90 % vs
#: 78 % busy, 1.15-1.22x), single CTAs when tiles are cut from spatially sorted masks (the smaller tile contracts a
#: shorter slab range: 2.27 vs 3.08 ms on C2 frames, 1.89 vs 2.01 ms on crowded 256 x 256 frames;
#: profiles/mma_pair_r01.md); '0' / '1' force one of them
MMA_PAIR = os.environ.get('AMPIS_MMA_PAIR', 'auto')


def intersect_mma(table, groups, mode, out=None, sort=True, pair=None):
    """Dense intersection matrices by the int8 tcgen05 contraction (no pruning), then the per-row
    arg-max from the matrices.  Same RowResult as intersect_rows(), bit for bit; the choice
    between the two is a cost decision (DESIGN.md).  sort=True cuts the tiles from rows / columns
    ordered by position in the image, which shortens the pixel range each tile contracts."""
    table.require_bitmaps()
    dev = table.device
    assert table.layout != LAYOUT_CROP, 'the contraction reads linear packed masks (span or full layout)'
    nr = max(groups.n_rows, 1)
    if pair is None:
        pair = (not sort) if MMA_PAIR == 'auto' else MMA_PAIR != '0'
    n_tiles, tile_grp, tile_m0, tile_n0 = groups.mma_tiles(pair)
    if out is None:
        out = RowResult(torch.empty(nr, dtype=torch.int32, device=dev),
                        torch.empty(nr, dtype=torch.int32, device=dev),
                        torch.empty(nr, dtype=torch.float64, device=dev),
                        torch.empty(max(groups.imat_size, 1), dtype=torch.int32, device=dev))
    assert out.imat is not None
    row_order, col_order = _span_orders(table, groups) if sort and groups.n_rows else (None, None)
    N.call('ampis_intersect_tcgen05_pair' if pair else 'ampis_intersect_tcgen05', _p(table.bits), _p(table.bits_off), _p(table.reg), _p(table.span),
           _p(groups.row_mask), _p(row_order), _p(col_order), _p(tile_grp), _p(tile_m0), _p(tile_n0), n_tiles,
           _p(groups.grp_row_begin),
           _p(groups.grp_row_count), _p(groups.grp_col_begin), _p(groups.grp_col_count), _p(groups.imat_off),
           _p(out.imat), _stream())
    N.call('ampis_rows_from_imat', _p(out.imat), _p(groups.imat_off), _p(table.area), _p(groups.row_mask),
           _p(groups.row_grp), groups.n_rows, _p(groups.grp_row_begin), _p(groups.grp_col_begin),
           _p(groups.grp_col_count), mode, _p(out.best_col), _p(out.best_inter), _p(out.best_score), _stream())
    return out


def intersect_tma(table, groups, mode, out=None):
    """Dense intersection matrices by the TMA-staged shared-memory tiled AND+popc kernel (ampis_intersect_tma), then
    the per-row arg-max from the matrices.  Same RowResult as intersect_rows() / intersect_mma(), bit for bit.  Needs
    a FULL-layout table painted by the unfused path (frames stored regularly, which is what a tensor map describes)
    whose masks all share one frame size.  A measurement kernel (profiles/crossover_r02.md), not a product path."""
    table.require_bitmaps()
    dev = table.device
    assert table.layout == LAYOUT_FULL and not table.fused, 'regular full frames: MaskTable(..., LAYOUT_FULL).measure().paint()'
    nr = max(groups.n_rows, 1)
    n_tiles, tile_grp, tile_m0, tile_n0 = groups.mma_tiles('tma')
    if out is None:
        out = RowResult(torch.empty(nr, dtype=torch.int32, device=dev),
                        torch.empty(nr, dtype=torch.int32, device=dev),
                        torch.empty(nr, dtype=torch.float64, device=dev),
                        torch.empty(max(groups.imat_size, 1), dtype=torch.int32, device=dev))
    assert out.imat is not None
    frame_chunks = getattr(table, '_frame_chunks', None)
    if frame_chunks is None:            # one frame size for the whole table (read back once)
        hw = (table.h[:table.n].to(torch.int64) * table.w[:table.n].to(torch.int64))
        assert table.n and bool((hw == hw[0]).all().item()), 'all masks must share one frame size'
        frame_chunks = table._frame_chunks = (int(hw[0].item()) + 127) // 128
    N.call('ampis_intersect_tma', _p(table.bits), frame_chunks, table.n, _p(table.span), _p(groups.row_mask),
           _p(tile_grp), _p(tile_m0), _p(tile_n0), n_tiles, _p(groups.grp_row_begin), _p(groups.grp_row_count),
           _p(groups.grp_col_begin), _p(groups.grp_col_count), _p(groups.imat_off), _p(out.imat), _stream())
    N.call('ampis_rows_from_imat', _p(out.imat), _p(groups.imat_off), _p(table.area), _p(groups.row_mask),
           _p(groups.row_grp), groups.n_rows, _p(groups.grp_row_begin), _p(groups.grp_col_begin),
           _p(groups.grp_col_count), mode, _p(out.best_col), _p(out.best_inter), _p(out.best_score), _stream())
    return out


#: operand fill above which the dense tensor-core contraction beats the culled AND+popc walk
#: (measured crossover, profiles/crossover_r01.md)
MMA_FILL_THRESHOLD = 0.25
#: below this many rows / columns a 128 x 256 tile is mostly padding and the contraction cannot win
MMA_MIN_SIDE = 64


def operand_fill(table, groups=None):
    """Fraction of the dense operand volume (masks x 128-pixel slabs of the frame) that lies inside
    the masks' spans -- a device reduction and one 8-byte read-back."""
    n = table.n
    if n == 0:
        return 0.0
    sp = table.span[:2 * n].view(n, 2).to(torch.int64)
    slabs = (table.h[:n].to(torch.int64) * table.w[:n].to(torch.int64) + 127) // 128
    return float(((sp[:, 1] - sp[:, 0]).sum().double() / slabs.sum().double().clamp(min=1)).item())


def choose_kernel(table, groups):
    """'mma' (dense int8 tcgen05 contraction) for crowded images, 'rows' (bbox-culled AND+popc)
    otherwise.  Both give identical results; this is only a cost decision."""
    if groups.imat_off is None or groups.n_rows == 0 or table.layout == LAYOUT_CROP:
        return 'rows'
    return 'mma' if operand_fill(table, groups) >= MMA_FILL_THRESHOLD else 'rows'


def intersect(table, groups, mode, out=None, kernel='auto'):
    """Intersection rows by the kernel named (or chosen by choose_kernel for 'auto')."""
    if kernel == 'auto':
        kernel = choose_kernel(table, groups)
    return (intersect_mma if kernel == 'mma' else intersect_rows)(table, groups, mode, out=out)


def match_counts(rows, groups, thresholds, totals=None, counts=None):
    """TP/FP/FN per group and threshold -> int32[n_groups, n_thresh, 3] (device), totals += .
    `thresholds` may be a host sequence or a float64 device tensor (no copy then)."""
    dev = groups.device
    th = thresholds if isinstance(thresholds, torch.Tensor) else \
        _dev(np.asarray(thresholds, np.float64), torch.float64, dev)
    nt = th.numel()
    if counts is None:
        counts = torch.empty(max(groups.n_groups * nt * 3, 1), dtype=torch.int32, device=dev)
    if totals is None:
        totals = torch.zeros(max(nt * 3, 1), dtype=torch.int64, device=dev)
    N.call('ampis_match_counts', _p(rows.best_col), _p(rows.best_score), _p(groups.grp_row_begin),
           _p(groups.grp_row_count), _p(groups.grp_col_count), groups.n_groups, groups.max_cols, _p(th), nt,
           _p(counts), _p(totals), _stream())
    return counts[:groups.n_groups * nt * 3].view(groups.n_groups, nt, 3), totals[:nt * 3].view(nt, 3)


def satellite_counts(table, rows, groups, thresh, n_bins=64, hist=None, counts=None):
    dev = groups.device
    if counts is None:
        counts = torch.empty(max(groups.n_groups * 4, 1), dtype=torch.int32, device=dev)
    if hist is None:
        hist = torch.zeros(n_bins, dtype=torch.int64, device=dev)
    N.call('ampis_satellite_counts', _p(rows.best_col), _p(rows.best_inter), _p(table.area), _p(groups.row_mask),
           _p(groups.grp_row_begin), _p(groups.grp_row_count), _p(groups.grp_col_count), groups.n_groups,
           groups.max_cols, float(thresh), _p(counts), _p(hist), n_bins, _stream())
    return counts[:groups.n_groups * 4].view(groups.n_groups, 4), hist


def iou_matrix(table, rows, groups, g=0):
    """float64[G, P] IoU matrix of group g from the dense intersections."""
    G, P = int(groups.h_row_count[g]), int(groups.h_col_count[g])
    out = torch.empty(max(G * P, 1), dtype=torch.float64, device=table.device)
    if G * P:
        off = int(groups.h_imat_off[g])
        imat = rows.imat[off:off + G * P]
        r0 = int(groups.h_row_begin[g])
        row_ids = groups.row_mask[r0:r0 + G].long()
        c0 = int(groups.grp_col_begin[g].item())
        ar = table.area[row_ids].contiguous()
        ac = table.area[c0:c0 + P].contiguous()
        N.call('ampis_iou_matrix_f64', _p(imat), _p(ar), _p(ac), G, P, _p(out), _stream())
    return out[:G * P].view(G, P)


def edge_distances(table, gt_ids, pred_ids, windows):
    """Boundary disagreement of matched pairs (analyze.mask_edge_distance): for pair i the masks
    gt_ids[i], pred_ids[i] of `table` inside windows[i] = (r1, r2, c1, c2).  Returns
    (counts int64[n, 4], fp_dist float64 device tensor, fn_dist float64 device tensor, off_fp, off_fn)."""
    table.require_bitmaps()
    assert table.layout != LAYOUT_CROP
    dev = table.device
    n = len(gt_ids)
    d_g = _dev(np.asarray(gt_ids, np.int32), torch.int32, dev)
    d_p = _dev(np.asarray(pred_ids, np.int32), torch.int32, dev)
    d_w = _dev(np.asarray(windows, np.int32).reshape(-1), torch.int32, dev)
    counts = torch.empty(max(4 * n, 1), dtype=torch.int32, device=dev)
    N.call('ampis_edge_count', _p(table.bits), _p(table.bits_off), _p(table.reg), _p(table.span), _p(table.h),
           _p(d_g), _p(d_p), _p(d_w), n, _p(counts), _stream())
    c = counts[:4 * n].cpu().numpy().reshape(n, 4).astype(np.int64)
    off = np.zeros((4, n + 1), np.int64)
    np.cumsum(c.T, axis=1, out=off[:, 1:])
    d_off = [_dev(off[k, :n], torch.int64, dev) for k in range(4)]
    lists = [torch.empty(max(int(off[k, n]), 1), dtype=torch.int32, device=dev) for k in range(4)]
    d_fp = torch.empty(max(int(off[0, n]), 1), dtype=torch.float64, device=dev)
    d_fn = torch.empty(max(int(off[1, n]), 1), dtype=torch.float64, device=dev)
    status = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    N.call('ampis_edge_distances', _p(table.bits), _p(table.bits_off), _p(table.reg), _p(table.span), _p(table.h),
           _p(d_g), _p(d_p), _p(d_w), n, _p(d_off[0]), _p(d_off[1]), _p(d_off[2]), _p(d_off[3]), _p(lists[0]),
           _p(lists[1]), _p(lists[2]), _p(lists[3]), _p(d_fp), _p(d_fn), _p(status), _stream())
    if n and bool(status[:n].any().item()):
        bad = int(torch.nonzero(status[:n]).flatten()[0].item())
        raise RuntimeError('mask_edge_distance: pair %d has disagreement pixels but no pixel of the other mask '
                           'inside the merged box (min over an empty set)' % bad)
    return c, d_fp[:int(off[0, n])], d_fn[:int(off[1, n])], off[0], off[1]


def hist_u32(values, lo, bin_width, n_bins, hist=None):
    if hist is None:
        hist = torch.zeros(n_bins, dtype=torch.int64, device=values.device)
    N.call('ampis_hist_u32', _p(values), values.numel(), int(lo), int(bin_width), _p(hist), n_bins, _stream())
    return hist


def unpack_bool(table, ids, h, w):
    """Packed masks -> bool[n, h, w] device tensor (structures.masks_to_bitmask_array)."""
    table.require_bitmaps()
    dev = table.device
    assert table.layout != LAYOUT_CROP, 'unpack reads linear packed masks (span or full layout)'
    
    n = len(ids)
    out = torch.empty((n, h, w), dtype=torch.uint8, device=dev)
    d_ids = _dev(np.asarray(ids, np.int32), torch.int32, dev)
    step = 32768
    for s in range(0, n, step):
        k = min(step, n - s)
        N.call('ampis_unpack_bool_nrc', _p(table.bits), _p(table.bits_off), _p(table.reg), _p(d_ids[s:]), k, h, w,
               _p(out[s:]), _stream())
    return out.view(torch.bool)


def _stack_memory(a):
    """bool/uint8 [n, h, w] host array -> (flat uint8 memory, y_major).  The two layouts that occur --
    C order, and the transposed view of a Fortran-ordered h x w x n stack that RLE.decode(...)
    .transpose(2, 0, 1) yields (memory [n][w][h]) -- are uploaded as they are; anything else is
    copied to C order first."""
    if a.dtype == np.bool_:
        a = a.view(np.uint8)
    assert a.ndim == 3 and a.dtype == np.uint8
    if a.flags.c_contiguous:
        return a.reshape(-1), 0
    t = a.transpose(0, 2, 1)
    if t.flags.c_contiguous:
        return t.reshape(-1), 1
    return np.ascontiguousarray(a).reshape(-1), 0


def to_host(t):
    """Device tensor -> numpy array.  Large results land in pinned memory (PyTorch caches the
    allocation, so repeated calls pay for it once): a pageable read-back of a few hundred MB runs at a
    fraction of the link rate."""
    if t.numel() * t.element_size() <= PIN_LIMIT_BYTES:
        return t.cpu().numpy()
    view_bool = t.dtype == torch.bool
    src = t.view(torch.uint8) if view_bool else t
    host = torch.empty(src.shape, dtype=src.dtype, pin_memory=True)
    host.copy_(src)
    out = host.numpy()
    return out.view(np.bool_) if view_bool else out


def bool_area_bbox(masks_np):
    """bool[n, h, w] host array -> (uint64 areas, int32 tight boxes x0,y0,x1,y1) on the host."""
    dev = require_cuda()
    flat, y_major = _stack_memory(masks_np)
    n, h, w = masks_np.shape
    d = _dev(flat, torch.uint8, dev)
    area = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    bbox = torch.empty(4 * max(n, 1), dtype=torch.int32, device=dev)
    N.call('ampis_bool_area_bbox', _p(d), n, h, w, y_major, _p(area), _p(bbox), _stream())
    return area[:n].cpu().numpy().view(np.uint64), bbox[:4 * n].cpu().numpy().reshape(-1, 4)


def polygons_to_counts(polys, h, w):
    """list of flat [x0,y0,x1,y1,...] polygons -> (device cnt, cnt_off, cnt_len) via rleFrPoly on the GPU."""
    dev = require_cuda()
    n = len(polys)
    lens = np.fromiter((len(p) for p in polys), np.int64, n)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    xy = np.concatenate([np.asarray(p, np.float64).ravel() for p in polys]) if n else np.zeros(0, np.float64)
    cap = 2 * (int(w) + 2) + 8                      # typical: two crossings per column
    d_xy = _dev(xy, torch.float64, dev)
    d_off = _dev(off, torch.int64, dev)
    d_h = torch.full((max(n, 1),), int(h), dtype=torch.int32, device=dev)
    d_w = torch.full((max(n, 1),), int(w), dtype=torch.int32, device=dev)
    while True:
        coff = np.arange(n + 1, dtype=np.int64) * cap
        d_coff = _dev(coff, torch.int64, dev)
        cnt = torch.empty(max(n * cap, 1), dtype=torch.int32, device=dev)
        clen = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        N.call('ampis_poly_to_rle', _p(d_xy), _p(d_off), _p(d_h), _p(d_w), n, _p(cnt), _p(d_coff), _p(clen),
               _stream())
        lens_out = clen[:n].cpu().numpy()
        if n and lens_out.min() < 0:
            raise ValueError('polygon %d is outside the GPU rasteriser limits (1..4096 vertices, '
                             '<=8192 boundary crossings)' % int(np.argmin(lens_out)))
        if n == 0 or lens_out.max() <= cap:
            return cnt, d_coff, clen, d_h, d_w
        cap = int(lens_out.max())


def counts_to_strings(cnt, cnt_off, cnt_len, n):
    """Device run counts -> list of compressed RLE byte strings (rleToString on the GPU)."""
    if n == 0:
        return []
    dev = cnt.device
    lens = cnt_len[:n].cpu().numpy().astype(np.int64)
    choff = np.zeros(n + 1, np.int64)
    np.cumsum(7 * lens, out=choff[1:])
    d_choff = _dev(choff, torch.int64, dev)
    chars = torch.empty(max(int(choff[-1]), 1), dtype=torch.uint8, device=dev)
    chlen = torch.empty(n, dtype=torch.int32, device=dev)
    N.call('ampis_rle_string_encode', _p(cnt), _p(cnt_off), _p(cnt_len), n, _p(chars), _p(d_choff), _p(chlen),
           _stream())
    buf = chars.cpu().numpy().tobytes()
    ln = chlen.cpu().numpy()
    return [buf[choff[i]:choff[i] + ln[i]] for i in range(n)]


def exclusive_scan(values_i64):
    """Exclusive prefix sum on the device: int64[n] -> int64[n + 1] (last = total)."""
    n = values_i64.numel()
    out = torch.empty(n + 1, dtype=torch.int64, device=values_i64.device)
    tmp_bytes = N.lib().ampis_scan_tmp_bytes(n)
    tmp = torch.empty(max(tmp_bytes // 8, 1), dtype=torch.int64, device=values_i64.device)
    N.call('ampis_exclusive_scan_i64', _p(values_i64), _p(out), n, _p(tmp), tmp_bytes, _stream())
    return out


def frames_to_rle(bits, n, h, w):
    """n consecutive FULL-layout frames of (h, w) in `bits` (int32 device tensor) -> list of COCO RLE
    dicts: rleEncode + rleToString on the GPU (the reference's RLE.encode)."""
    if n == 0:
        return []
    dev = bits.device
    chunks = (int(h) * int(w) + 127) // 128
    d_off = torch.arange(n, dtype=torch.int64, device=dev) * chunks
    d_h = torch.full((n,), int(h), dtype=torch.int32, device=dev)
    d_w = torch.full((n,), int(w), dtype=torch.int32, device=dev)
    n_runs = torch.empty(n, dtype=torch.int64, device=dev)
    N.call('ampis_bits_to_rle_count', _p(bits), _p(d_off), _p(d_h), _p(d_w), n, _p(n_runs), _stream())
    cnt_off = exclusive_scan(n_runs)
    total = int(cnt_off[n].item())
    cnt = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
    cnt_len = torch.empty(n, dtype=torch.int32, device=dev)
    N.call('ampis_bits_to_rle_emit', _p(bits), _p(d_off), _p(d_h), _p(d_w), n, _p(cnt_off), _p(cnt), _p(cnt_len),
           _stream())
    strings = counts_to_strings(cnt, cnt_off, cnt_len, n)
    return [{'size': [int(h), int(w)], 'counts': s} for s in strings]


def encode_bool(masks):
    """bool/uint8 [n, h, w] host array OR CUDA tensor -> list of COCO RLE dicts (RLE.encode of the
    Fortran-ordered h x w x n stack, data_utils.py:275,423): pack, run-length encode and string-encode
    on the GPU.  A CUDA tensor (model output) is encoded where it is -- no round trip through the host."""
    dev = require_cuda()
    y_major = 0
    if isinstance(masks, torch.Tensor):
        assert masks.dim() == 3 and masks.dtype in (torch.bool, torch.uint8)
        n, h, w = (int(v) for v in masks.shape)
        if n == 0:
            return []
        d = masks.to(dev).contiguous().view(torch.uint8).reshape(-1)
    else:
        n, h, w = masks.shape
        if n == 0:
            return []
        flat, y_major = _stack_memory(np.asarray(masks))
        d = _dev(flat, torch.uint8, dev)
    chunks = (h * w + 127) // 128
    bits = torch.empty(4 * n * chunks, dtype=torch.int32, device=dev)
    d_off = torch.arange(n, dtype=torch.int64, device=dev) * chunks
    N.call('ampis_pack_bool_nrc', _p(d), n, h, w, y_major, _p(bits), _p(d_off), _stream())
    return frames_to_rle(bits, n, h, w)


def project_pairs(table, gt_ids, pred_ids, h, w, mode):
    """Pixel-class frames of analyze.seg_perf_iset as RLE dicts: mode 'reduced' -> 4, 'all' -> 7."""
    table.require_bitmaps()
    assert table.layout != LAYOUT_CROP
    dev = table.device
    chunks = (int(h) * int(w) + 127) // 128
    n_out = 4 if mode == 'reduced' else 7
    d_g = _dev(np.asarray(gt_ids, np.int32), torch.int32, dev)
    d_p = _dev(np.asarray(pred_ids, np.int32), torch.int32, dev)
    tmp = torch.empty(4 * 3 * chunks, dtype=torch.int32, device=dev)
    out = torch.empty(4 * n_out * chunks, dtype=torch.int32, device=dev)
    N.call('ampis_project_pairs', _p(table.bits), _p(table.bits_off), _p(table.reg), _p(table.span), _p(d_g),
           _p(d_p), len(gt_ids), chunks, 0 if mode == 'reduced' else 1, _p(tmp), _p(out), _stream())
    return frames_to_rle(out, n_out, h, w)


MAX_LABEL_VALUE = 1 << 24     # 'label' annotation images: values are ranked through a flag table of this size


def label_image_to_instances(ann, binary):
    """Annotation image (H x W host array) -> (list of RLE dicts, int32 tight boxes x0,y0,x1,y1), one
    per instance in the reference's order (data_utils.py:408-424): `binary` -> connected components
    (8-connectivity, raster order), otherwise ascending label value with a leading 0 skipped."""
    dev = require_cuda()
    a = np.asarray(ann)
    if a.ndim != 2:
        raise ValueError('annotation images must be 2-D, got shape %s' % (a.shape,))
    h, w = a.shape
    n = h * w
    dense_t = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    if binary:
        img = _dev(np.ascontiguousarray(a.astype(np.bool_)).view(np.uint8).reshape(-1), torch.uint8, dev)
        work = torch.empty(n, dtype=torch.int32, device=dev)
        flags = torch.empty(n, dtype=torch.int64, device=dev)
        rank = torch.empty(n + 1, dtype=torch.int64, device=dev)
        tmp_bytes = N.lib().ampis_scan_tmp_bytes(n)
        tmp = torch.empty(max(tmp_bytes // 8, 1), dtype=torch.int64, device=dev)
        N.call('ampis_ccl_label', _p(img), h, w, _p(work), _p(flags), _p(rank), _p(tmp), tmp_bytes, _p(dense_t),
               _stream())
        n_labels = int(rank[n].item())
    else:
        if not np.issubdtype(a.dtype, np.integer) and not a.dtype == np.bool_:
            raise ValueError('label images must hold integers, got %s' % a.dtype)
        lo, hi = (int(a.min()), int(a.max())) if n else (0, 0)
        if lo < 0 or hi >= MAX_LABEL_VALUE:
            raise ValueError('label values must lie in [0, %d)' % MAX_LABEL_VALUE)
        n_values = hi + 1                                       # size of the flag table
        d_ann = _dev(np.ascontiguousarray(a).astype(np.int64).reshape(-1), torch.int32, dev)
        present = torch.zeros(n_values, dtype=torch.int64, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        N.call('ampis_label_values_present', _p(d_ann), n, _p(present), n_values, _p(bad), _stream())
        rank = exclusive_scan(present)
        zero_present = int(present[0].item())
        n_labels = int(rank[n_values].item()) - zero_present
        N.call('ampis_label_dense', _p(d_ann), _p(rank), zero_present, h, w, _p(dense_t), _stream())
    if n_labels == 0:
        return [], np.zeros((0, 4), np.int32)
    big = np.iinfo(np.int32).max
    bbox = torch.tensor([big, big, -1, -1], dtype=torch.int32, device=dev).repeat(n_labels).contiguous()
    N.call('ampis_label_bbox', _p(dense_t), h, w, n_labels, _p(bbox), _stream())
    n_runs = torch.empty(n_labels, dtype=torch.int64, device=dev)
    N.call('ampis_label_rle_count', _p(dense_t), h, w, n_labels, _p(bbox), _p(n_runs), _stream())
    cnt_off = exclusive_scan(n_runs)
    cnt = torch.empty(max(int(cnt_off[n_labels].item()), 1), dtype=torch.int32, device=dev)
    cnt_len = torch.empty(n_labels, dtype=torch.int32, device=dev)
    N.call('ampis_label_rle_emit', _p(dense_t), h, w, n_labels, _p(bbox), _p(cnt_off), _p(cnt), _p(cnt_len),
           _stream())
    strings = counts_to_strings(cnt, cnt_off, cnt_len, n_labels)
    rles = [{'size': [int(h), int(w)], 'counts': s} for s in strings]
    return rles, bbox.cpu().numpy().reshape(-1, 4)


def region_measurements(masks):
    """Per-mask raw measurements behind compute_rprops, all exact integers: dict of numpy arrays
    area[n], bbox[n,4] (x0,y0,x1,y1), moments[n,6] (N, Sx, Sy, Sxx, Syy, Sxy as Python-int-safe uint64),
    perimeter_hist[n,10], convex_area[n].  One CROP-layout table, four small launches."""
    t = table_from_rle(masks, layout=LAYOUT_CROP)
    dev, n = t.device, t.n
    mom = torch.empty(max(6 * n, 1), dtype=torch.int64, device=dev)
    N.call('ampis_rle_moments', _p(t.cum), _p(t.cnt_off), _p(t.cnt_len), _p(t.h), n, _p(mom), _stream())
    border = torch.empty_like(t.bits)
    hist = torch.empty(max(10 * n, 1), dtype=torch.int32, device=dev)
    N.call('ampis_crop_perimeter', _p(t.bits), _p(t.bits_off), _p(t.bbox), n, _p(border), _p(hist), _stream())
    bb = t.bbox_np()
    bw = np.maximum(bb[:, 2] - bb[:, 0] + 1, 0).astype(np.int64)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(10 * bw + 4, out=off[1:])
    scratch = torch.empty(max(int(off[n]), 1), dtype=torch.int32, device=dev)
    convex = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    d_off = _dev(off[:n], torch.int64, dev)          # named: a temporary would be recycled before the launch
    N.call('ampis_crop_convex_area', _p(t.bits), _p(t.bits_off), _p(t.bbox), n, _p(d_off), _p(scratch), _p(convex),
           _stream())
    return {'area': t.areas_np().astype(np.int64), 'bbox': bb,
            'moments': mom[:6 * n].cpu().numpy().view(np.uint64).reshape(n, 6),
            'perimeter_hist': hist[:10 * n].cpu().numpy().reshape(n, 10).astype(np.int64),
            'convex_area': convex[:n].cpu().numpy().astype(np.int64)}


#: measurements region_measurements_for can take, each one kernel (or pair of kernels) over one CROP table
REGION_MEASUREMENTS = ('moments', 'perimeter_hist', 'convex_area', 'moments3', 'filled', 'crofton', 'convex_feret',
                       'image', 'filled_image', 'intensity', 'weighted_intensity')
#: ampis_rle_moments3 and ampis_rle_intensity are exact while both sides of the frame stay below this
MOMENTS3_MAX_SIDE = 65536
#: pixel type codes of ampis_rle_intensity (AMPIS_PIX_* of include/ampis_b200.h) by numpy dtype
INTENSITY_PIX = {np.dtype(t): code for t, code in
                 ((np.bool_, 0), (np.uint8, 0), (np.int8, 1), (np.uint16, 2), (np.int16, 3), (np.uint32, 4),
                  (np.int32, 5), (np.uint64, 6), (np.int64, 7), (np.float16, 8), (np.float32, 9), (np.float64, 10))}
_SAME_WIDTH_TORCH = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}


def _i192(limbs):
    """Three 64-bit limbs (low first, as Python ints) -> the signed 192-bit integer they hold."""
    v = limbs[0] | (limbs[1] << 64) | (limbs[2] << 128)
    return v - (1 << 192) if v >> 191 else v


def _intensity_measurements(t, intensity_image, weighted):
    """ampis_rle_intensity over the masks of table t (see region_measurements_for, 'intensity' and
    'weighted_intensity').  The image is uploaded once, as raw pixels of its own width, and transposed to
    column-major order on the device.  Without `weighted`, a float image takes one pass and no box scan."""
    dev, n = t.device, t.n
    a = np.asarray(intensity_image)
    dt = a.dtype.newbyteorder('=')
    if dt not in INTENSITY_PIX:
        raise TypeError('intensity images of dtype %s are not supported (%s)'
                        % (a.dtype, ', '.join(sorted({str(d) for d in INTENSITY_PIX}))))
    if n and max(int(t.h[:n].max().item()), int(t.w[:n].max().item())) > MOMENTS3_MAX_SIDE:
        raise ValueError('moments to order 3 are exact for frames up to %d pixels a side' % MOMENTS3_MAX_SIDE)
    raw = np.ascontiguousarray(a, dtype=dt)
    img = _dev(raw.view(np.dtype('u1') if dt.itemsize == 1 else np.dtype('i%d' % dt.itemsize)),
               _SAME_WIDTH_TORCH[dt.itemsize], dev).reshape(raw.shape).t().contiguous()
    pix, flt = INTENSITY_PIX[dt], dt.kind == 'f'
    stats = torch.empty(max(4 * n, 1), dtype=torch.int64, device=dev)
    mom = torch.empty(max((16 if flt else 48) * n, 1), dtype=torch.float64 if flt else torch.int64, device=dev)
    N.call('ampis_rle_intensity', _p(t.cum), _p(t.cnt_off), _p(t.cnt_len), _p(t.h), _p(t.bbox), n, _p(img), pix,
           None, int(flt and weighted), _p(mom), _p(stats), _stream())
    st = stats[:4 * n].cpu().numpy().reshape(n, 4)
    wide = np.float64 if flt else np.int64 if dt.kind == 'i' else np.uint64
    out = {'intensity_min': np.ascontiguousarray(st[:, 0]).view(wide).astype(dt),
           'intensity_max': np.ascontiguousarray(st[:, 1]).view(wide).astype(dt)}
    if not flt:
        limbs = mom[:48 * n].cpu().numpy().view(np.uint64).reshape(n, 16, 3).tolist()
        out['intensity_sum'] = [_i192(row[0]) for row in limbs]
        if weighted:
            out['intensity_moments'] = [[[_i192(row[4 * p + q]) for q in range(4)] for p in range(4)] for row in limbs]
        return out
    if not weighted:
        out['intensity_sum'] = mom[:16 * n].view(n, 16)[:, 0].cpu().numpy()
        return out
    # float pixels: the central sums in a second pass about the weighted centroid, formed on the device
    m = mom[:16 * n].view(n, 16)
    center = torch.stack([m[:, 4] / m[:, 0], m[:, 1] / m[:, 0]], dim=1).contiguous()
    central = torch.empty(max(16 * n, 1), dtype=torch.float64, device=dev)
    N.call('ampis_rle_intensity', _p(t.cum), _p(t.cnt_off), _p(t.cnt_len), _p(t.h), _p(t.bbox), n, _p(img), pix,
           _p(center), 0, _p(central), None, _stream())
    raw_m, cen_m = m.cpu().numpy().reshape(n, 4, 4), central[:16 * n].cpu().numpy().reshape(n, 4, 4)
    # skimage weighs the whole box, img[slice] * image: a NaN or inf of the box outside the mask gives NaN * 0
    out['intensity_sum'] = raw_m[:, 0, 0].copy()             # of the mask's pixels, for the mean
    outside = st[:, 3] > st[:, 2]
    raw_m[outside] = np.nan
    cen_m[outside] = np.nan
    out['intensity_moments'], out['intensity_central'] = raw_m, cen_m
    return out


def _ragged_u8(flat, off, shapes):
    return [flat[off[i]:off[i + 1]].reshape(shapes[i]).view(np.bool_) for i in range(len(shapes))]


def region_measurements_for(masks, need, intensity_image=None):
    """Per-mask raw measurements behind compute_rprops for the measurement names in `need` only (see
    REGION_MEASUREMENTS): one CROP-layout table, then only the launches those names require.  Always present:
    area[n], bbox[n,4] (x0,y0,x1,y1).  Optional, all exact integers but the sums of float intensity images:
      moments[n,6], perimeter_hist[n,10], convex_area[n]   as region_measurements;
      moments3: list of n 4x4 nested lists of Python ints, M[p][q] = sum r^p c^q in box-local coordinates;
      filled: filled_area[n] (binary_fill_holes with an all-ones 3x3 structure);
      filled_image: list of n bool box images of the filled masks (implies filled);
      crofton: crofton_trans[n,4], differing pixel pairs along rows, columns, diagonal, anti-diagonal;
      convex_feret: convex_ranges (list of n int32[box_w, 2] box-local row ranges [lo, hi) of
        convex_hull_image) and feret_d2[n] = (2 * feret_diameter_max)^2;
      image: list of n bool box images;
      intensity (needs `intensity_image`, a 2-D array of the masks' frame size, bool / integer / float16-64):
        intensity_min[n], intensity_max[n] in the image's dtype (NaN when a float mask holds a NaN pixel) and
        intensity_sum[n], the sum of the mask's pixels (exact Python ints for integer and bool images);
      weighted_intensity (implies intensity, needs the image as well): intensity_moments, M[p][q] = sum I r^p c^q in box-local coordinates -- for integer and bool images a list
        of n 4x4 nested lists of exact Python ints; for float images float64[n,4,4] summed in float64, with
        intensity_central[n,4,4], the sums about the weighted centroid (M[1][0] / M[0][0], M[0][1] / M[0][0]).
        A NaN or inf in a mask's box but outside the mask makes both NaN, as skimage's img[slice] * image does."""
    need = set(need)
    bad = need - set(REGION_MEASUREMENTS)
    if bad:
        raise ValueError('unknown region measurements %s' % sorted(bad))
    if 'weighted_intensity' in need:
        need.add('intensity')
    if 'intensity' in need and intensity_image is None:
        raise ValueError('the intensity measurements need an intensity image')
    if 'filled_image' in need:
        need.add('filled')
    t = table_from_rle(masks, layout=LAYOUT_CROP)
    dev, n = t.device, t.n
    bb = t.bbox_np()
    out = {'area': t.areas_np().astype(np.int64), 'bbox': bb}
    bw = np.maximum(bb[:, 2] - bb[:, 0] + 1, 0).astype(np.int64)
    bh = np.where(bw > 0, bb[:, 3] - bb[:, 1] + 1, 0).astype(np.int64)
    if 'moments' in need:
        mom = torch.empty(max(6 * n, 1), dtype=torch.int64, device=dev)
        N.call('ampis_rle_moments', _p(t.cum), _p(t.cnt_off), _p(t.cnt_len), _p(t.h), n, _p(mom), _stream())
        out['moments'] = mom[:6 * n].cpu().numpy().view(np.uint64).reshape(n, 6)
    if 'moments3' in need:
        if n and max(int(t.h[:n].max().item()), int(t.w[:n].max().item())) > MOMENTS3_MAX_SIDE:
            raise ValueError('moments to order 3 are exact for frames up to %d pixels a side' % MOMENTS3_MAX_SIDE)
        m3 = torch.empty(max(32 * n, 1), dtype=torch.int64, device=dev)
        N.call('ampis_rle_moments3', _p(t.cum), _p(t.cnt_off), _p(t.cnt_len), _p(t.h), _p(t.bbox), n, _p(m3),
               _stream())
        halves = m3[:32 * n].cpu().numpy().view(np.uint64).reshape(n, 16, 2).tolist()
        out['moments3'] = [[[lo | (hi << 64) for lo, hi in row[4 * p:4 * p + 4]] for p in range(4)] for row in halves]
    if 'perimeter_hist' in need:
        border = torch.empty_like(t.bits)
        hist = torch.empty(max(10 * n, 1), dtype=torch.int32, device=dev)
        N.call('ampis_crop_perimeter', _p(t.bits), _p(t.bits_off), _p(t.bbox), n, _p(border), _p(hist), _stream())
        out['perimeter_hist'] = hist[:10 * n].cpu().numpy().reshape(n, 10).astype(np.int64)
    if 'filled' in need or 'crofton' in need:
        filled = torch.zeros_like(t.bits) if 'filled' in need else None
        farea = torch.empty(max(n, 1), dtype=torch.int64, device=dev) if 'filled' in need else None
        trans = torch.empty(max(4 * n, 1), dtype=torch.int64, device=dev) if 'crofton' in need else None
        N.call('ampis_crop_fill_holes', _p(t.bits), _p(t.bits_off), _p(t.bbox), n, _p(filled), _p(farea), _p(trans),
               _stream())
        if filled is not None:
            out['filled_area'] = farea[:n].cpu().numpy()
        if trans is not None:
            out['crofton_trans'] = trans[:4 * n].cpu().numpy().reshape(n, 4)
    if 'convex_area' in need or 'convex_feret' in need:
        off = np.zeros(n + 1, np.int64)
        np.cumsum(10 * bw + 4, out=off[1:])
        scratch = torch.empty(max(int(off[n]), 1), dtype=torch.int32, device=dev)
        d_off = _dev(off[:n], torch.int64, dev)          # named: a temporary would be recycled before the launch
        if 'convex_area' in need:
            convex = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
            N.call('ampis_crop_convex_area', _p(t.bits), _p(t.bits_off), _p(t.bbox), n, _p(d_off), _p(scratch),
                   _p(convex), _stream())
            out['convex_area'] = convex[:n].cpu().numpy().astype(np.int64)
        if 'convex_feret' in need:
            col_off = np.zeros(n + 1, np.int64)
            np.cumsum(bw, out=col_off[1:])
            d_col = _dev(col_off[:n], torch.int64, dev)
            ranges = torch.empty(max(2 * int(col_off[n]), 1), dtype=torch.int32, device=dev)
            d2 = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
            N.call('ampis_crop_convex_feret', _p(t.bits), _p(t.bits_off), _p(t.bbox), n, _p(d_off), _p(scratch),
                   _p(d_col), _p(ranges), _p(d2), _stream())
            rg = ranges[:2 * int(col_off[n])].cpu().numpy().reshape(-1, 2)
            out['convex_ranges'] = [rg[col_off[i]:col_off[i + 1]] for i in range(n)]
            out['feret_d2'] = d2[:n].cpu().numpy()
    if 'image' in need or 'filled_image' in need:
        img_off = np.zeros(n + 1, np.int64)
        np.cumsum(bh * bw, out=img_off[1:])
        d_img_off = _dev(img_off[:n], torch.int64, dev)
        shapes = list(zip(bh.tolist(), bw.tolist()))
        for key, src in (('image', t.bits), ('filled_image', filled if 'filled_image' in need else None)):
            if key not in need:
                continue
            img = torch.empty(max(int(img_off[n]), 1), dtype=torch.uint8, device=dev)
            N.call('ampis_crop_unpack_image', _p(src), _p(t.bits_off), _p(t.bbox), n, _p(d_img_off), _p(img),
                   _stream())
            out[key] = _ragged_u8(to_host(img[:int(img_off[n])]), img_off, shapes)
    if 'intensity' in need:
        out.update(_intensity_measurements(t, intensity_image, 'weighted_intensity' in need))
    return out


def polygons_to_bool(polys, h, w):
    """list of flat [x0,y0,x1,y1,...] polygons -> bool[n, h, w] host array by skimage's polygon2mask
    rule (structures._poly2mask), rasterised on the GPU."""
    dev = require_cuda()
    n = len(polys)
    if n == 0:
        return np.zeros((0, int(h), int(w)), bool)
    lens = np.fromiter((len(p) for p in polys), np.int64, n)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    xy = np.concatenate([np.asarray(p, np.float64).ravel() for p in polys])
    out = torch.empty((n, int(h), int(w)), dtype=torch.uint8, device=dev)
    d_xy, d_off = _dev(xy, torch.float64, dev), _dev(off, torch.int64, dev)      # keep both alive for the launch
    N.call('ampis_polygon2mask', _p(d_xy), _p(d_off), n, int(h), int(w), _p(out), _stream())
    return out.cpu().numpy().view(np.bool_)
