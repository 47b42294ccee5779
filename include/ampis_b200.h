/*
 * ampis_b200.h -- C ABI of libampis_b200.so: the B200 (sm_100a) kernels behind
 * AMPIS's mask-evaluation hot path.
 *
 * The reference (rccohn/AMPIS, pure Python) has no FFI of its own: every
 * number on this path comes from pycocotools' C routines called through
 * `pycocotools.mask` (SURVEY.md F2).  Each entry point below names the
 * reference call site(s) it replaces.  All pointers prefixed d_ are DEVICE
 * pointers owned by the caller (PyTorch allocates them); `stream` is a
 * cudaStream_t passed as void*.  Nothing here allocates device memory, throws,
 * or synchronises unless stated.  Return value: 0 on success, a negative
 * AMPIS_E* code otherwise (ampis_last_error() gives the text).
 *
 * Device data model ("mask table", structure of arrays, n masks):
 *   cnt      u32[]   run-length counts of all masks, COCO order: column-major pixels
 *                    (index = x*h + y), first run counts zeros
 *   cnt_off  i64[n]  first count of mask i inside cnt
 *   cnt_len  i32[n]  number of runs of mask i
 *   h, w     u32[n]  image size of mask i
 *   cum      u32[]   inclusive prefix sums of cnt (same indexing) = run end positions
 *   area     u32[n]  number of 1-pixels (rleArea)
 *   bbox     i32[4n] tight box x0,y0,x1,y1 (inclusive); empty mask = 0,0,-1,-1
 *   span     u32[2n] [lo,hi) in 128-bit chunks of the linear bit vector that holds all 1s
 *   reg      u32[2n] [lo,hi) chunk region actually stored for mask i
 *                    (layout SPAN: = span; layout FULL: 0..ceil(h*w/128))
 *   bits_off i64[n+1] first uint4 of mask i's region inside the `bits` arena
 *   bits     uint4[] packed masks: bit k of a mask = pixel k in column-major order,
 *                    little-endian inside 32-bit words
 */
#ifndef AMPIS_B200_H
#define AMPIS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AMPIS_OK            0
#define AMPIS_EINVAL       -1   /* bad argument */
#define AMPIS_ECUDA        -2   /* CUDA runtime error (see ampis_last_error) */
#define AMPIS_ENOSPC       -3   /* caller-provided buffer too small */

#define AMPIS_LAYOUT_SPAN   0   /* store only [first 1, last 1] of each mask (culled) */
#define AMPIS_LAYOUT_FULL   1   /* store the full h*w frame of each mask (canonical) */
#define AMPIS_LAYOUT_CROP   2   /* store only the bounding-box window of each mask: for every column
                                   x0..x1 the 32-row words (y0>>5)..(y1>>5) of that column, column after
                                   column (SURVEY 8d "cropped accounting"); reg = [0, ceil(words/4)) */

#define AMPIS_MODE_IOU      0   /* score = I / (a_row + a_col - I), analyze.py:158 */
#define AMPIS_MODE_SAT      1   /* score = I / a_row,               powder.py:82-83 */

/* bit flags written to status[i] by ampis_rle_measure */
#define AMPIS_ST_BAD_TOTAL  1   /* sum(counts) != h*w (pycocotools would hang or mis-decode) */

int         ampis_version(void);
const char *ampis_last_error(void);
/* number of SMs of the current device (grid sizing); <0 on error */
int         ampis_sm_count(void);

/* ---- RLE string codec -------------------------------------------------------
 * Replaces pycocotools rleFrString as invoked by every RLE.iou / merge / area /
 * decode call in the reference (analyze.py:108,158,315-321; powder.py:82-83,264;
 * structures.py:467,568,571,752,761).  d_chars holds the n compressed strings back
 * to back, d_chr_off[n+1] their byte offsets.  Counts of mask i are written at
 * d_cnt + d_cnt_off[i] (a string of L bytes yields at most L counts, so
 * cnt_off = chr_off is always large enough); d_cnt_len[i] receives the run count.
 * The kernel reads d_chars as aligned 32-bit words (only words that hold a character of a string): the allocation
 * behind d_chars must cover whole words, as every cudaMalloc / torch allocation does.  One thread per string. */
int ampis_rle_string_decode(const uint8_t *d_chars, const int64_t *d_chr_off, int32_t n,
                            uint32_t *d_cnt, const int64_t *d_cnt_off, int32_t *d_cnt_len,
                            void *stream);

/* Inverse (pycocotools rleToString; data_utils.py:275, structures.py:465 via RLE.encode).
 * d_chars needs 7 bytes per count at d_chr_off[i] (= 7*cnt_off[i] is always enough);
 * d_chr_len[i] receives the string length. */
int ampis_rle_string_encode(const uint32_t *d_cnt, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                            int32_t n, uint8_t *d_chars, const int64_t *d_chr_off, int32_t *d_chr_len,
                            void *stream);

/* ---- per-mask measurements ---------------------------------------------------
 * One pass over the run counts: rleArea (structures.py:568,571; analyze.py:320-321;
 * powder.py:264), the tight bounding box that extract_boxes (data_utils.py:180-252)
 * reads off the decoded mask, the storage span/region, and the prefix sums the
 * decoder needs.  d_reg_chunks[i] = reg_hi - reg_lo (input of the offset scan). */
int ampis_rle_measure(const uint32_t *d_cnt, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                      const uint32_t *d_h, const uint32_t *d_w, int32_t n, int32_t layout,
                      uint32_t *d_cum, uint32_t *d_area, int32_t *d_bbox, uint32_t *d_span,
                      uint32_t *d_reg, int64_t *d_reg_chunks, int32_t *d_status, void *stream);

/* Exclusive prefix sum of n int64 values into d_out[n+1] (d_out[n] = total).
 * d_tmp needs ampis_scan_tmp_bytes(n) bytes. */
size_t ampis_scan_tmp_bytes(int64_t n);
int    ampis_exclusive_scan_i64(const int64_t *d_in, int64_t *d_out, int64_t n,
                                void *d_tmp, size_t tmp_bytes, void *stream);

/* ---- RLE -> bit-packed masks ---------------------------------------------------
 * Replaces pycocotools rleDecode (structures.py:752,761; analyze.py:472-473) as the
 * producer of the mask representation every later kernel reads.  Writes exactly the
 * region [reg_lo,reg_hi) of every mask, 128 bits per store.  bits_capacity = number of
 * uint4 in d_bits; masks that would not fit are skipped and AMPIS_ENOSPC is NOT
 * detected here (the caller sized the arena from d_bits_off[n]). */
int ampis_rle_decode_packed(const uint32_t *d_cum, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                            const uint32_t *d_span, const uint32_t *d_reg, const int64_t *d_bits_off,
                            int32_t n, void *d_bits, int64_t bits_capacity, void *stream);

/* Same for AMPIS_LAYOUT_CROP tables (needs the tight boxes and image heights of the masks). */
int ampis_rle_decode_crop(const uint32_t *d_cum, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                          const int32_t *d_bbox, const uint32_t *d_h, const int64_t *d_bits_off, int32_t n,
                          void *d_bits, int64_t bits_capacity, void *stream);

/* Fused form of ampis_rle_measure + scan + ampis_rle_decode_packed in ONE launch: every CTA
 * measures its masks, reserves arena space with one atomicAdd on *d_cursor (zeroed by this call)
 * and paints.  Arena order is arbitrary (d_bits_off[i] is still written per mask; there is no
 * d_bits_off[n]).  After the stream has completed, *d_cursor = uint4 chunks needed; if it exceeds
 * bits_capacity some masks were not painted and the caller must retry with a larger arena.
 * d_cum is only touched for masks with more runs than fit in shared memory.
 * runs_hint: typical number of runs per mask (0 = unknown).  CROP layout only: small masks (<= 40 / <= 112 runs)
 * are handled by 8 / 16 lanes each instead of a warp; results do not depend on it. */
int ampis_rle_measure_paint(const uint32_t *d_cnt, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                            const uint32_t *d_h, const uint32_t *d_w, int32_t n, int32_t layout,
                            uint32_t *d_cum, uint32_t *d_area, int32_t *d_bbox, uint32_t *d_span,
                            uint32_t *d_reg, int64_t *d_bits_off, int32_t *d_status, void *d_bits,
                            int64_t bits_capacity, uint64_t *d_cursor, int32_t runs_hint, void *stream);

/* AMPIS_LAYOUT_CROP form of ampis_rle_measure_paint, third generation ("flat"): a warp decodes several masks at
 * once with its lanes spread over their concatenated (0-run, 1-run) pairs -- one segmented scan per 32 pairs, one
 * record-forming lane per mask, one arena reservation and one contiguous copy-out per warp (csrc/rle_flat.cu).
 * Same outputs as ampis_rle_measure_paint(layout = AMPIS_LAYOUT_CROP), bit for bit; arena order differs.
 * d_list: int32[n + 1] scratch; masks outside the per-warp budgets (more than 512 runs, window larger than 2 KB,
 * frame of 2^31 pixels or more or taller than 65,536 rows) are listed there and worked off by a second launch (a warp per mask, any size). */
int ampis_rle_measure_paint_flat(const uint32_t *d_cnt, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                                 const uint32_t *d_h, const uint32_t *d_w, int32_t n, uint32_t *d_cum,
                                 uint32_t *d_area, int32_t *d_bbox, uint32_t *d_span, uint32_t *d_reg,
                                 int64_t *d_bits_off, int32_t *d_status, void *d_bits, int64_t bits_capacity,
                                 uint64_t *d_cursor, int32_t *d_list, int32_t runs_hint, void *stream);

/* The same launch with a side job: the kernel also ZEROES d_zero[0 .. zero_bytes) (16-byte aligned; NULL = nothing), a
 * share per group of masks.  The decode is bound by instruction issue and leaves HBM idle, so the dense matrices the
 * row pass will patch (analyze.py:149-158: one G x P matrix per image, 1 GB per 1,000 C2 images) are cleared here for
 * ~1 % more instructions instead of by a separate fill.  Pass imat_ints = 0 to ampis_intersect_rows_pairs afterwards. */
int ampis_rle_measure_paint_flat_zero(const uint32_t *d_cnt, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                                      const uint32_t *d_h, const uint32_t *d_w, int32_t n, uint32_t *d_cum,
                                      uint32_t *d_area, int32_t *d_bbox, uint32_t *d_span, uint32_t *d_reg,
                                      int64_t *d_bits_off, int32_t *d_status, void *d_bits, int64_t bits_capacity,
                                      uint64_t *d_cursor, int32_t *d_list, int32_t runs_hint, void *d_zero,
                                      int64_t zero_bytes, void *stream);

/* bits -> bool[n][h][w] row-major bytes (RLE.decode(...).astype(bool).transpose(2,0,1),
 * structures.py:752,765).  All n masks must share (h,w). d_mask_ids selects masks. */
int ampis_unpack_bool_nrc(const void *d_bits, const int64_t *d_bits_off, const uint32_t *d_reg,
                          const int32_t *d_mask_ids, int32_t n, uint32_t h, uint32_t w,
                          uint8_t *d_out, void *stream);

/* bool[n][h][w] -> area (u64) and tight bbox (mask_areas on ndarray, structures.py:558-560;
 * extract_boxes, data_utils.py:229-239).  y_major != 0: the memory is [n][w][h] (row index fastest),
 * the layout behind RLE.decode(...).transpose(2,0,1) -- accepted as it is, no host-side re-layout. */
int ampis_bool_area_bbox(const uint8_t *d_masks, int32_t n, uint32_t h, uint32_t w, int32_t y_major,
                         uint64_t *d_area, int32_t *d_bbox, void *stream);

/* bool[n][h][w] (row-major) -> packed FULL-layout bits (RLE.encode producer side,
 * data_utils.py:275,423): region of mask i is chunk 0..ceil(h*w/128) at d_bits_off[i]. */
int ampis_pack_bool_nrc(const uint8_t *d_masks, int32_t n, uint32_t h, uint32_t w, int32_t y_major,
                        void *d_bits, const int64_t *d_bits_off, void *stream);

/* ---- intersection / IoU rows ----------------------------------------------------
 * The fused hot kernel.  For every row mask r (a ground-truth mask, or a satellite) it
 * visits the column masks of its group (the predictions, or the particles, of the same
 * image), prunes by bounding box exactly as rleIou's bbIou pre-pass does, computes
 * I = popcount(row AND col) over the overlap of the two spans, and keeps the first
 * arg-max of the score.  Replaces the G x ceil(P/80) RLE.iou calls of
 * analyze.py:149-164 and the S x N RLE.merge+RLE.area calls of powder.py:80-86.
 *   row_mask[r]                    mask id of row r (rows of a group are contiguous)
 *   blk_grp[b], blk_row0[b]        CTA b handles rows blk_row0[b] .. +ampis_rows_per_block()-1
 *                                  (clipped to the group) of group blk_grp[b]
 *   grp_row_begin[g], grp_row_count[g]   rows of group g
 *   grp_col_begin[g], grp_col_count[g]   column masks of group g (contiguous mask ids)
 *   grp_imat_off[g]                offset (in int32) of group g's dense G x P intersection
 *                                  matrix inside d_imat, or -1 / d_imat NULL for none
 * Outputs per row: best_col (index inside the group, IOU mode: -1 if every IoU is 0;
 * SAT mode: 0 if every intersection is 0), best_inter, best_score (double). */
int ampis_rows_per_block(void);
int ampis_intersect_rows(const void *d_bits, const int64_t *d_bits_off, const uint32_t *d_reg,
                         const uint32_t *d_span, const int32_t *d_bbox, const uint32_t *d_area,
                         const int32_t *d_row_mask, const int32_t *d_blk_grp, const int32_t *d_blk_row0,
                         int32_t n_blocks, const int32_t *d_grp_row_begin, const int32_t *d_grp_row_count,
                         const int32_t *d_grp_col_begin, const int32_t *d_grp_col_count,
                         const int64_t *d_grp_imat_off, int32_t mode, int32_t *d_imat,
                         int32_t *d_best_col, uint32_t *d_best_inter, double *d_best_score,
                         void *stream);

/* The same kernel over AMPIS_LAYOUT_CROP tables: AND+popc only over the overlap of the two
 * bounding-box windows (words of the same column and the same 32-row band line up without
 * shifts because bands are absolute).  Same outputs, bit for bit.  The column metadata is staged
 * by TMA bulk copies: d_bbox, d_area and d_bits_off must be 16-byte aligned. */
int ampis_intersect_rows_crop(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox,
                              const uint32_t *d_area, const int32_t *d_row_mask, const int32_t *d_blk_grp,
                              const int32_t *d_blk_row0, int32_t n_blocks, const int32_t *d_grp_row_begin,
                              const int32_t *d_grp_row_count, const int32_t *d_grp_col_begin,
                              const int32_t *d_grp_col_count, const int64_t *d_grp_imat_off, int32_t mode,
                              int32_t *d_imat, int32_t *d_best_col, uint32_t *d_best_inter,
                              double *d_best_score, void *stream);

/* The crop rows kernel with the bbox pre-pruning (rleIou's bbIou pass, analyze.py:108,158) done through a
 * uniform grid instead of a scan of all G x P boxes -- for images with thousands of instances
 * (spheroidite, satellites vs 2,000 particles).  The column masks of every group are binned into
 * ampis_grid_cells() = 32 x 32 square cells of side 2^grp_shift[g] pixels by ampis_grid_build (one CTA per
 * group: counts and their scan in shared memory, one atomicAdd on *d_cursor -- zeroed by the call -- per group):
 *   d_grp_shift[g]                       log2 of the cell side (>= mean box side of the group's columns)
 *   d_cell_off i64[n_groups * (cells+1)] absolute position of every cell's first entry (+ one end marker per group)
 *   d_entries i32[capacity], d_entry_bbox i32[4 * capacity]   column index (inside the group) and box, cell by cell
 * After the stream has completed *d_cursor = entries needed; beyond `capacity` nothing is written (call with
 * capacity 0 to size the lists).  ampis_intersect_rows_grid then gives the same per-row outputs (and dense rows,
 * if asked: the first imat_ints values of d_imat are zeroed by a memset node, the kernel patches the non-zero
 * cells) as ampis_intersect_rows_crop, bit for bit.  Eight lanes per row, four rows per warp.  Optional sparse
 * output: the non-zero intersections as (row, column-in-group, intersection) triplets in no particular order;
 * *d_coo_count (zeroed by the caller) counts them and may exceed coo_capacity, in which case the excess was
 * dropped. */
int ampis_grid_cells(void);
int ampis_grid_build(const int32_t *d_bbox, const int32_t *d_grp_col_begin, const int32_t *d_grp_col_count,
                     int32_t n_groups, int32_t *d_grp_shift, int64_t *d_cell_off, int32_t *d_entries,
                     int32_t *d_entry_bbox, int64_t capacity, uint64_t *d_cursor, void *stream);
int ampis_intersect_rows_grid(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox,
                              const uint32_t *d_area, const int32_t *d_row_mask, const int32_t *d_blk_grp,
                              const int32_t *d_blk_row0, int32_t n_blocks, const int32_t *d_grp_row_begin,
                              const int32_t *d_grp_row_count, const int32_t *d_grp_col_begin,
                              const int32_t *d_grp_col_count, const int32_t *d_grp_shift,
                              const int64_t *d_cell_off, const int32_t *d_entries,
                              const int32_t *d_entry_bbox, int64_t capacity,
                              const int64_t *d_grp_imat_off, int32_t mode, int32_t *d_imat, int64_t imat_ints,
                              int32_t *d_best_col, uint32_t *d_best_inter, double *d_best_score,
                              int32_t *d_coo_row, int32_t *d_coo_col, uint32_t *d_coo_inter,
                              int64_t coo_capacity, uint64_t *d_coo_count, void *stream);

/* The grid-pruned crop rows as a spatial JOIN in three flat passes (csrc/intersect_pairs.cu), same outputs as
 * ampis_intersect_rows_grid bit for bit (same grid from ampis_grid_build):
 *   1. one thread per row walks the grid cells of its box and appends the (row mask, column mask) pairs whose
 *      boxes overlap -- rleIou's bbIou pre-pass (analyze.py:108,158) -- to d_pair_ab (int32[2 * pair_capacity],
 *      8-byte aligned) and the geometry of the overlap of their windows to d_pair_desc (32 bytes per pair,
 *      16-byte aligned); the pairs of row r are d_row_pair_cnt[r] consecutive entries from d_row_pair_off[r];
 *   2. eight lanes per pair: d_pair_inter[q] = popcount(A & B) over the overlap of the two windows;
 *   3. one thread per row: score and first arg-max over its pairs, dense cells / sparse triplets.
 * d_row_grp[r] = group of row r.  *d_pair_count (zeroed by the call) = pairs found; when it exceeds pair_capacity
 * nothing useful was computed and the caller retries with a larger list.  zero_stream (may be NULL): a second
 * stream on which the dense matrices are zeroed while passes 1 and 2 run on `stream` (fork / join by events inside
 * the call); NULL = zeroed in line. */
int ampis_intersect_rows_pairs(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox,
                               const uint32_t *d_area, const int32_t *d_row_mask, const int32_t *d_row_grp,
                               int32_t n_rows, const int32_t *d_grp_row_begin, const int32_t *d_grp_col_begin,
                               const int32_t *d_grp_col_count, const int32_t *d_grp_shift,
                               const int64_t *d_cell_off, const int32_t *d_entries, const int32_t *d_entry_bbox,
                               int64_t grid_capacity, int32_t *d_pair_ab, void *d_pair_desc,
                               uint32_t *d_pair_inter, int64_t pair_capacity, int64_t *d_row_pair_off, int32_t *d_row_pair_cnt,
                               uint64_t *d_pair_count, const int64_t *d_grp_imat_off, int32_t mode, int32_t *d_imat,
                               int64_t imat_ints, int32_t *d_best_col, uint32_t *d_best_inter, double *d_best_score,
                               int32_t *d_coo_row, int32_t *d_coo_col, uint32_t *d_coo_inter, int64_t coo_capacity,
                               uint64_t *d_coo_count, void *zero_stream, void *stream);

/* ---- one image, one call (host entry point) ---------------------------------------------------------
 * The per-image work of analyze.py:149-164 (rle_instance_matcher / det_seg_scores: G x ceil(P/80) RLE.iou calls +
 * arg-max) and powder.py:80-86 (_rle_satellite_match) from HOST buffers: the n_rows + n_cols compressed strings
 * (rows first; all masks of size h x w) are staged through h_ws (pinned host memory), uploaded with one copy,
 * decoded, measured and painted as bounding-box windows, intersected (all-columns scan below grid_min_cols
 * columns, grid-pruned from there on) and the results come back with one copy and ONE stream synchronisation:
 * per row best_col / best_inter / best_score as ampis_intersect_rows, per mask area, bbox, span and status
 * (AMPIS_ST_BAD_TOTAL marks malformed RLE); iou_out, when not NULL, receives the full float64 n_rows x n_cols IoU
 * matrix of analyze._piecewise_iou (analyze.py:54-112).  Nothing is allocated: d_ws (256-byte aligned device memory) and
 * h_ws are the caller's; when one is too small the call returns AMPIS_ENOSPC with *need_bytes = device bytes
 * wanted (> 0) or minus the host bytes wanted (< 0).  The column grid's entry list takes the larger of 16 entries per
 * column + 4,096 and a 32nd of d_ws (20 bytes per entry); boxes far larger than the image's mean box (a thin diagonal
 * across a frame of small blobs registers in all 32 x 32 cells) can need more, which is reported the same way:
 * AMPIS_ENOSPC and a device size whose 32nd holds the measured entries. */
int ampis_eval_image_host(const uint8_t *chars, const int64_t *chr_off, int32_t n_rows, int32_t n_cols,
                          uint32_t h, uint32_t w, int32_t mode, int32_t grid_min_cols,
                          void *d_ws, int64_t d_ws_bytes, void *h_ws, int64_t h_ws_bytes,
                          int32_t *best_col, uint32_t *best_inter, double *best_score, uint32_t *area,
                          int32_t *bbox, uint32_t *span, int32_t *status, double *iou_out, int64_t *need_bytes,
                          void *stream);

/* ---- many images, one call (host entry point) -------------------------------------------------------
 * The loop a user of the reference writes around det_seg_scores / _rle_satellite_match (Colab cell 44 ->
 * analyze.py:226-339; cell 62 -> powder.py:138 -> powder.py:28-112), i.e. per image analyze.py:149-164 or
 * powder.py:80-86, for n_images images in ONE call from HOST string descriptors: str_ptr[k] / str_len[k] = address
 * and length of the k-th compressed RLE string, image after image, rows (ground truth / satellites) of an image
 * before its columns (predictions / particles); n_rows[g], n_cols[g], h[g], w[g] per image.  The strings are
 * gathered into h_ws (pinned), uploaded with one copy, decoded (rleFrString), measured and painted as windows (flat
 * decode), the columns binned into per-image grids, candidate pairs joined, intersected and reduced to per-row
 * results; one download, ONE stream synchronisation.  Outputs: best_col / best_inter / best_score for all rows
 * (concatenated in image order; best_col counts inside the image), area / bbox / span / status for all masks.
 * *pairs_found = candidate pairs (overlapping boxes).  crowd_frac in [0, 1): when the candidate pairs exceed that
 * fraction of all row x column pairs the AND+popc pass is skipped ON THE DEVICE and *crowded = 1 is returned (the
 * per-row outputs are void; measurements are valid) -- such batches belong to ampis_intersect_tcgen05; pass a
 * negative value to disable.  flags & AMPIS_STRINGS_CONTIGUOUS: the caller's strings already lie back to back
 * starting at str_ptr[0] (e.g. a blob in pinned memory): they are uploaded from where they are, nothing is gathered.
 * bbox and span may be NULL (not downloaded).  n_thresh > 0 (AMPIS_MODE_IOU): TP / FP / FN of the matcher
 * (analyze.py:166-174) at every IoU threshold, grp_counts int32[n_images][n_thresh][3] and totals int64[n_thresh][3],
 * counted on the device (ampis_match_counts) before the download.  Batches of more than 16,384 masks form their per-mask bookkeeping
 * on the device (expand_images_kernel + offset scan), so the host work per call is O(n_images) plus the gather.
 * For such batches, str_len and the output arrays are used as DMA endpoints directly when they are page-locked
 * (cudaHostAlloc / cudaHostRegister): no staging copy on either side.
 * Workspaces and AMPIS_ENOSPC protocol as ampis_eval_image_host (grid entry list: the larger of 16 entries per column
 * + 4,096 per image and a 32nd of d_ws).  Nothing carries over from one call to the next: a workspace grown for one
 * batch may be reused for any other. */
#define AMPIS_STRINGS_CONTIGUOUS 1   /* flags: the strings lie back to back from str_ptr[0] (only that pointer is read) */
#define AMPIS_WAIT_BLOCKING      2   /* flags: wait for the results on a blocking event instead of spinning */
int ampis_eval_images_host(const uint8_t *const *str_ptr, const int32_t *str_len, int32_t n_images,
                           const int32_t *n_rows, const int32_t *n_cols, const uint32_t *h, const uint32_t *w,
                           int32_t mode, int32_t flags, double crowd_frac, void *d_ws, int64_t d_ws_bytes, void *h_ws,
                           int64_t h_ws_bytes, int32_t *best_col, uint32_t *best_inter, double *best_score,
                           uint32_t *area, int32_t *bbox, uint32_t *span, int32_t *status,
                           const double *thresholds, int32_t n_thresh, int32_t *grp_counts, int64_t *totals,
                           int64_t *pairs_found, int32_t *crowded, int64_t *need_bytes, void *stream);

/* ---- many images, detection and segmentation counts over score x IoU thresholds, one call ------------------------
 * What ampis_eval_images_host followed by analyze.py:166-174 + 300-339 gives for every cut-off of the predictions'
 * confidence scores, from one decode, one join and one intersection per candidate pair.  Strings, sizes, flags and
 * workspaces as ampis_eval_images_host (rows = ground truth, columns = predictions; IoU matching; no crowd gate: a
 * crowded image only makes more candidate pairs).  levels[p], one per prediction in image order: the number of
 * (sorted) score thresholds strictly below its score, 0 for a NaN score; prediction p is kept at sorted score
 * threshold k iff levels[p] > k (levels[p] <= n_levels).  iou_thresh[0 .. n_iou): sorted ascending, each in
 * [0, inf).  For score level k and IoU threshold j, each cell equals det_seg_scores on the kept predictions: TP /
 * FP / FN = matched rows, kept predictions no matched row claims, unmatched rows; seg TP / FP / FN = sums over the
 * matched rows of intersection, prediction area - intersection, GT area - intersection.  Outputs: totals and
 * seg_totals int64[n_levels][n_iou][3] (required); counts int32[n_images][n_levels][n_iou][3] and seg_sums
 * int64[n_images][n_levels][n_iou][3] (NULL: not formed, their device space is not needed); status int32 per mask as
 * ampis_eval_images_host.  The per-image arrays are copied after the one wait for the results (blocking copies when
 * they are pageable).  An image may hold at most AMPIS_SWEEP_MAX_PREDS predictions (AMPIS_EINVAL otherwise);
 * 1 <= n_levels <= 65535, 1 <= n_iou <= AMPIS_SWEEP_MAX_IOU. */
#define AMPIS_SWEEP_MAX_PREDS 32768
#define AMPIS_SWEEP_MAX_IOU   256
int ampis_eval_images_sweep_host(const uint8_t *const *str_ptr, const int32_t *str_len, int32_t n_images,
                                 const int32_t *n_rows, const int32_t *n_cols, const uint32_t *h, const uint32_t *w,
                                 int32_t flags, const uint16_t *levels, int32_t n_levels, const double *iou_thresh,
                                 int32_t n_iou, void *d_ws, int64_t d_ws_bytes, void *h_ws, int64_t h_ws_bytes,
                                 int32_t *status, int64_t *totals, int64_t *seg_totals, int32_t *counts,
                                 int64_t *seg_sums, int64_t *pairs_found, int64_t *need_bytes, void *stream);

/* ---- dense intersection matrices on the tensor cores (tcgen05, int8 contraction) -----------
 * Same quantity as the dense output of ampis_intersect_rows -- I[r][c] = popcount(row AND col),
 * what rleIou's run walk accumulates per pair (analyze.py:108,158; powder.py:82) -- computed for
 * EVERY pair of a group as I = A * B^T over pixels with u8 operands expanded from the packed
 * bits in shared memory and an int32 accumulator in tensor memory.  No pruning: cost grows with
 * G*P*(pixel range), so this is the path for images with heavily overlapping instances; the
 * culled AND+popc kernel is the one for sparse images (DESIGN.md, "choice of intersection kernel").
 * A tile is ampis_mma_tile_rows() x ampis_mma_tile_cols() cells of one group's matrix:
 *   tile_grp[t], tile_m0[t], tile_n0[t]   group and first row / first column of tile t
 * Every group with at least one tile must have a dense matrix (grp_imat_off[g] >= 0).
 * Optional d_row_order / d_col_order (NULL = identity): tiles are cut from per-group SORTED lists --
 * row_order[grp_row_begin[g] + pos] = row index inside group g, col_order[grp_col_begin[g] + pos] =
 * column index inside group g.  Sorting by span start makes the masks of a tile neighbours in the image,
 * so the slab range a tile has to contract (rows' range AND columns' range) shrinks; results are
 * written at the unsorted indices. */
int ampis_mma_tile_rows(void);
int ampis_mma_tile_cols(void);
int ampis_intersect_tcgen05(const void *d_bits, const int64_t *d_bits_off, const uint32_t *d_reg,
                            const uint32_t *d_span, const int32_t *d_row_mask,
                            const int32_t *d_row_order, const int32_t *d_col_order,
                            const int32_t *d_tile_grp, const int32_t *d_tile_m0, const int32_t *d_tile_n0,
                            int32_t n_tiles, const int32_t *d_grp_row_begin, const int32_t *d_grp_row_count,
                            const int32_t *d_grp_col_begin, const int32_t *d_grp_col_count,
                            const int64_t *d_grp_imat_off, int32_t *d_imat, void *stream);

/* The same contraction on CTA pairs (tcgen05 cta_group::2, clusters of two CTAs on one TPC): one
 * M256 N256 K32 instruction per step over a 256 x 256 tile, each CTA expanding only its own 128 rows and
 * 128 columns.  Tiles are ampis_mma_pair_tile_rows() x ampis_mma_pair_tile_cols(); otherwise the same
 * arguments and the same output, bit for bit. */
int ampis_mma_pair_tile_rows(void);
int ampis_mma_pair_tile_cols(void);
int ampis_intersect_tcgen05_pair(const void *d_bits, const int64_t *d_bits_off, const uint32_t *d_reg,
                            const uint32_t *d_span, const int32_t *d_row_mask,
                            const int32_t *d_row_order, const int32_t *d_col_order,
                            const int32_t *d_tile_grp, const int32_t *d_tile_m0, const int32_t *d_tile_n0,
                            int32_t n_tiles, const int32_t *d_grp_row_begin, const int32_t *d_grp_row_count,
                            const int32_t *d_grp_col_begin, const int32_t *d_grp_col_count,
                            const int64_t *d_grp_imat_off, int32_t *d_imat, void *stream);

/* The same dense matrices by the TMA-staged, shared-memory tiled AND+popc kernel north_star names (no tensor cores,
 * no pruning beyond the K range a tile's spans share): operands are FULL-layout frames stored REGULARLY -- mask i
 * at d_bits + i * frame_chunks uint4, i.e. the arena of ampis_rle_measure + scan + ampis_rle_decode_packed -- and are
 * described to the TMA unit by one 2-D tensor map (cuTensorMapEncodeTiled, 128-byte swizzle); every CTA computes an
 * ampis_tma_tile() x ampis_tma_tile() tile through a 4-stage cp.async.bulk.tensor / mbarrier ring.  The rows of a
 * group must be consecutive masks (row_mask[r0 + k] = row_mask[r0] + k).  Built to be measured against the culled
 * kernels and the tensor-core contraction (profiles/crossover_r02.md): it is bound by the POPC pipe. */
int ampis_tma_tile(void);
int ampis_intersect_tma(const void *d_bits, int64_t frame_chunks, int32_t n_masks, const uint32_t *d_span,
                        const int32_t *d_row_mask, const int32_t *d_tile_grp, const int32_t *d_tile_m0,
                        const int32_t *d_tile_n0, int32_t n_tiles, const int32_t *d_grp_row_begin,
                        const int32_t *d_grp_row_count, const int32_t *d_grp_col_begin,
                        const int32_t *d_grp_col_count, const int64_t *d_grp_imat_off, int32_t *d_imat, void *stream);

/* Per-row results (same outputs and tie rules as ampis_intersect_rows) from dense matrices:
 * row_grp[r] = group of row r. */
int ampis_rows_from_imat(const int32_t *d_imat, const int64_t *d_grp_imat_off, const uint32_t *d_area,
                         const int32_t *d_row_mask, const int32_t *d_row_grp, int32_t n_rows,
                         const int32_t *d_grp_row_begin, const int32_t *d_grp_col_begin,
                         const int32_t *d_grp_col_count, int32_t mode, int32_t *d_best_col,
                         uint32_t *d_best_inter, double *d_best_score, void *stream);

/* Full IoU matrix of one group as float64[G][P] from the dense intersections
 * (analyze._piecewise_iou, analyze.py:54-112): I>0 ? I/(a_g+a_p-I) : 0.0 */
int ampis_iou_matrix_f64(const int32_t *d_imat, const uint32_t *d_area_rows, const uint32_t *d_area_cols,
                         int32_t G, int32_t P, double *d_out, void *stream);

/* ---- matching / scoring ------------------------------------------------------------
 * Per group (image): TP/FP/FN of AMPIS's per-GT arg-max matcher (analyze.py:166-174) at
 * n_thresh IoU thresholds from ONE row pass (the arg-max does not depend on the threshold).
 * d_grp_counts[g][t] = (tp, fp, fn) int32; d_totals[t] = (tp, fp, fn) int64, accumulated
 * (+=) over groups: the all-reduce payload of a dataset evaluation. */
int ampis_match_counts(const int32_t *d_best_col, const double *d_best_score,
                       const int32_t *d_grp_row_begin, const int32_t *d_grp_row_count,
                       const int32_t *d_grp_col_count, int32_t n_groups, int32_t max_cols,
                       const double *d_thresh, int32_t n_thresh,
                       int32_t *d_grp_counts, int64_t *d_totals, void *stream);

/* Satellite assignment summary (powder.py:88-96, 525-547): per group
 * (n_sat_matched, n_sat_unmatched, n_particles_matched, n_particles) int32, and a global
 * histogram (+=) of satellites per satellited particle, bins 0..n_bins-1 (last bin clamps). */
int ampis_satellite_counts(const int32_t *d_best_col, const uint32_t *d_best_inter,
                           const uint32_t *d_area, const int32_t *d_row_mask,
                           const int32_t *d_grp_row_begin, const int32_t *d_grp_row_count,
                           const int32_t *d_grp_col_count, int32_t n_groups, int32_t max_cols,
                           double thresh, int32_t *d_grp_counts, int64_t *d_spp_hist, int32_t n_bins,
                           void *stream);

/* Histogram (+=) of n uint32 values (mask areas) into n_bins uniform bins of `bin_width`
 * starting at `lo`; values outside are clamped into the first/last bin (size
 * distributions, powder.py:417 binned form used for multi-GPU reduction). */
int ampis_hist_u32(const uint32_t *d_values, int64_t n, uint32_t lo, uint32_t bin_width,
                   int64_t *d_hist, int32_t n_bins, void *stream);

/* ---- packed masks -> RLE (pycocotools rleEncode; RLE.encode at analyze.py:692, data_utils.py:275,423,
 * structures.py:465, powder.py:209).  Masks are FULL-layout frames (ceil(h*w/128) chunks at
 * d_bits_off[i], bits beyond h*w zero).  ampis_bits_to_rle_count gives the number of runs of each
 * mask; after an exclusive scan of those (ampis_exclusive_scan_i64 -> d_cnt_off),
 * ampis_bits_to_rle_emit writes the counts (first run counts zeros and may be 0) and d_cnt_len. */
int ampis_bits_to_rle_count(const void *d_bits, const int64_t *d_bits_off, const uint32_t *d_h,
                            const uint32_t *d_w, int32_t n, int64_t *d_n_runs, void *stream);
int ampis_bits_to_rle_emit(const void *d_bits, const int64_t *d_bits_off, const uint32_t *d_h,
                           const uint32_t *d_w, int32_t n, const int64_t *d_cnt_off, uint32_t *d_cnt,
                           int32_t *d_cnt_len, void *stream);

/* Pixel classes of matched pairs projected onto the frame (analyze.seg_perf_iset, analyze.py:637-690):
 * TP = OR(g & p), FN = OR(g & ~p), FP = OR(~g & p) over the pairs, then class bitmaps written as
 * consecutive FULL-layout frames into d_out_bits: mode 0 ('reduced') 4 frames [TP only, FN only,
 * FP only, two or more]; mode 1 ('all') 7 frames for codes 1..7 of TP + 2 FN + 4 FP.
 * d_tmp3 = scratch of 3 frames (zeroed here). */
int ampis_project_pairs(const void *d_bits, const int64_t *d_bits_off, const uint32_t *d_reg,
                        const uint32_t *d_span, const int32_t *d_pair_gt, const int32_t *d_pair_pr,
                        int32_t n_pairs, int64_t frame_chunks, int32_t mode, void *d_tmp3, void *d_out_bits,
                        void *stream);

/* ---- region properties (InstanceSet.compute_rprops -> skimage.measure.regionprops_table,
 * structures.py:505-508) -------------------------------------------------------------------------
 * ampis_rle_moments: exact raw moments of every mask from its run table (d_cum = run end positions
 *   from ampis_rle_measure): d_out[i] = { N, sum x, sum y, sum x^2, sum y^2, sum x*y } (x column, y row).
 * ampis_crop_perimeter (AMPIS_LAYOUT_CROP table): skimage.measure.perimeter(neighbourhood=4) as the
 *   ten weighted bins of its 50-bin histogram, order 5,7,15,17,25,27 (weight 1), 21,33 (sqrt 2),
 *   13,23 ((1+sqrt 2)/2); d_border_scratch has the size of the bits arena.
 * ampis_crop_convex_area: number of pixels of skimage's convex_hull_image (hull of the pixel-edge
 *   midpoints, crossing-number test of the pixel centres); scratch of 10*box_width+4 ints per mask
 *   at d_scratch_off[i]. */
int ampis_rle_moments(const uint32_t *d_cum, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                      const uint32_t *d_h, int32_t n, uint64_t *d_out, void *stream);
int ampis_crop_perimeter(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox, int32_t n,
                         void *d_border_scratch, uint32_t *d_hist10, void *stream);
int ampis_crop_convex_area(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox, int32_t n,
                           const int64_t *d_scratch_off, int32_t *d_scratch, uint64_t *d_convex_area,
                           void *stream);

/* The remaining non-intensity region properties (all but euler_number), same tables:
 * ampis_rle_moments3: skimage's `moments` to order 3 in box-local coordinates, exact: d_out[32*i + 2*k],
 *   [32*i + 2*k + 1] = low / high 64 bits of M[p][q] = sum r^p c^q, k = 4p + q, r = row - y0,
 *   c = column - x0 (d_bbox of ampis_rle_measure).  Exact while both frame sides are <= 65536.
 * ampis_crop_fill_holes (AMPIS_LAYOUT_CROP table): d_filled (size of the bits arena, same offsets and layout;
 *   may be null together with d_filled_area) = scipy.ndimage.binary_fill_holes(box image,
 *   structure=ones((3,3))), d_filled_area[i] its pixel count; d_trans (may be null) = 4 counts per mask of
 *   pixel pairs that differ, outside the box = 0: along rows, along columns, along (r+1, c+1), along (r+1, c-1)
 *   -- perimeter_crofton(directions=4) = pi/8 * (t0 + t1 + (t2 + t3) / sqrt 2).
 * ampis_crop_convex_feret: convex_hull_image as row ranges [lo, hi) (box-local; lo == hi for an empty
 *   column) at d_ranges[2 * (d_col_off[i] + c)], and d_feret_d2[i] = (2 * feret_diameter_max)^2 as an exact
 *   integer; scratch as for ampis_crop_convex_area.
 * ampis_crop_unpack_image: the box image of every mask as row-major 0/1 bytes at d_img + d_img_off[i]
 *   (box_h * box_w bytes; pass the filled arena of ampis_crop_fill_holes as d_bits for filled_image). */
int ampis_rle_moments3(const uint32_t *d_cum, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                       const uint32_t *d_h, const int32_t *d_bbox, int32_t n, uint64_t *d_out, void *stream);
int ampis_crop_fill_holes(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox, int32_t n,
                          void *d_filled, uint64_t *d_filled_area, uint64_t *d_trans, void *stream);
int ampis_crop_convex_feret(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox, int32_t n,
                            const int64_t *d_scratch_off, int32_t *d_scratch, const int64_t *d_col_off,
                            int32_t *d_ranges, uint64_t *d_feret_d2, void *stream);
int ampis_crop_unpack_image(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox, int32_t n,
                            const int64_t *d_img_off, uint8_t *d_img, void *stream);

/* The intensity properties (regionprops with an intensity image), same run tables as ampis_rle_moments3:
 * ampis_rle_intensity: d_img = the intensity image, COLUMN-major (pixel (row y, column x) at x * h + y, the order
 *   of the run positions), of the pixel type `pix` (AMPIS_PIX_*; bool as AMPIS_PIX_U8).  Per mask:
 *   - integer pixels: d_moments[48*i + 3*k + {0,1,2}] = the 64-bit limbs, low first, of the signed 192-bit
 *     M[p][q] = sum I r^p c^q, k = 4p + q, box-local r, c as in ampis_rle_moments3; exact while both frame
 *     sides are <= 65536.  d_center must be null.
 *   - float pixels: d_center null: d_moments[16*i + k] = M[p][q] summed in float64.  d_center[2*i], [2*i+1] =
 *     (r0, c0) box-local: d_moments[16*i + k] = sum I (r - r0)^p (c - c0)^q, the central sums.
 *   d_stats (written when d_center is null, which requires it): 4 x 8 bytes per mask = min and max pixel of the
 *   mask (int64 for signed, uint64 for unsigned, float64 for float pixels; NaN when the mask holds a NaN), then
 *   the number of non-finite pixels of the mask and, when scan_box is non-zero, of its bounding box (both 0 for
 *   integer pixels; the box scan reads every pixel of the box, so ask for it only where the weighted moments are
 *   needed). */
#define AMPIS_PIX_U8    0
#define AMPIS_PIX_I8    1
#define AMPIS_PIX_U16   2
#define AMPIS_PIX_I16   3
#define AMPIS_PIX_U32   4
#define AMPIS_PIX_I32   5
#define AMPIS_PIX_U64   6
#define AMPIS_PIX_I64   7
#define AMPIS_PIX_F16   8
#define AMPIS_PIX_F32   9
#define AMPIS_PIX_F64  10
int ampis_rle_intensity(const uint32_t *d_cum, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                        const uint32_t *d_h, const int32_t *d_bbox, int32_t n, const void *d_img, int32_t pix,
                        const double *d_center, int32_t scan_box, void *d_moments, uint64_t *d_stats, void *stream);

/* ---- annotation images -> instances (data_utils.get_ddicts 'binary' / 'label', data_utils.py:394-433) ----
 * ampis_ccl_label: skimage.measure.label of a binary image (row-major u8[h][w], non-zero = foreground,
 *   full 8-connectivity, labels 1..n in raster order of each component's first pixel).  d_work i32[h*w],
 *   d_flags i64[h*w], d_rank i64[h*w+1] (d_rank[h*w] = number of labels afterwards), scan scratch as for
 *   ampis_exclusive_scan_i64.  Output d_dense_t: labels in COLUMN-major order (index x*h + y).
 * ampis_label_values_present / ampis_label_dense: the 'label' format -- arbitrary non-negative label
 *   values < n_values are ranked in ascending order (np.unique), 0 = background when present.
 * ampis_label_bbox: tight box of every label 1..n_labels (d_bbox pre-filled with INT_MAX,INT_MAX,-1,-1).
 * ampis_label_rle_count / _emit: RLE.encode(ann == u) for every label, from the label's box window
 *   only; counts at d_cnt + d_cnt_off[u-1]. */
int ampis_ccl_label(const uint8_t *d_img, int32_t h, int32_t w, int32_t *d_work, int64_t *d_flags,
                    int64_t *d_rank, void *d_scan_tmp, size_t scan_tmp_bytes, int32_t *d_dense_t, void *stream);
int ampis_label_values_present(const int32_t *d_ann, int64_t n, int64_t *d_present, int32_t n_values,
                               int32_t *d_bad, void *stream);
int ampis_label_dense(const int32_t *d_ann, const int64_t *d_rank, int32_t zero_present, int32_t h, int32_t w,
                      int32_t *d_dense_t, void *stream);
int ampis_label_bbox(const int32_t *d_dense_t, int32_t h, int32_t w, int32_t n_labels, int32_t *d_bbox,
                     void *stream);
int ampis_label_rle_count(const int32_t *d_dense_t, int32_t h, int32_t w, int32_t n_labels,
                          const int32_t *d_bbox, int64_t *d_n_runs, void *stream);
int ampis_label_rle_emit(const int32_t *d_dense_t, int32_t h, int32_t w, int32_t n_labels,
                         const int32_t *d_bbox, const int64_t *d_cnt_off, uint32_t *d_cnt, int32_t *d_cnt_len,
                         void *stream);

/* ---- boundary disagreement of matched pairs (analyze.mask_edge_distance, analyze.py:416-499) ------
 * For pair i: masks pair_gt[i], pair_pr[i] (SPAN or FULL layout table) and the window
 * win[i] = (r1, r2, c1, c2), half open, inside the frame (the merged box of analyze.py:466).
 * ampis_edge_count   -> counts[i] = (#false-positive px, #false-negative px, #gt boundary px,
 *                       #pred boundary px) inside the window.
 * ampis_edge_distances, given exclusive offsets of those counts (off_*[i], int64) and scratch
 * lists of matching sizes, writes for every false-positive pixel (row-major order inside the
 * window, np.where order) the distance to the nearest gt pixel, and for every false-negative
 * pixel the distance to the nearest predicted pixel, as float64 = sqrt(exact integer);
 * status[i] = 1 when a pair has false-positive (negative) pixels but no gt (pred) pixel in the
 * window (the reference's torch.min raises there). Window sides must be <= 32767. */
int ampis_edge_count(const void *d_bits, const int64_t *d_bits_off, const uint32_t *d_reg,
                     const uint32_t *d_span, const uint32_t *d_h, const int32_t *d_pair_gt,
                     const int32_t *d_pair_pr, const int32_t *d_win, int32_t n_pairs, int32_t *d_counts,
                     void *stream);
int ampis_edge_distances(const void *d_bits, const int64_t *d_bits_off, const uint32_t *d_reg,
                         const uint32_t *d_span, const uint32_t *d_h, const int32_t *d_pair_gt,
                         const int32_t *d_pair_pr, const int32_t *d_win, int32_t n_pairs,
                         const int64_t *d_off_fp, const int64_t *d_off_fn, const int64_t *d_off_gb,
                         const int64_t *d_off_pb, uint32_t *d_list_fp, uint32_t *d_list_fn,
                         uint32_t *d_list_gb, uint32_t *d_list_pb, double *d_dist_fp, double *d_dist_fn,
                         int32_t *d_status, void *stream);

/* ---- polygon -> RLE (pycocotools rleFrPoly via RLE.frPyObjects, structures.py:677) -----
 * d_xy: vertex coordinates x0,y0,x1,y1,... of all polygons, d_xy_off[n+1] offsets in doubles.
 * Crossing positions (sorted, zero-length runs merged) are written as run counts at
 * d_cnt + d_cnt_off[i]; capacity per polygon is d_cnt_off[i+1]-d_cnt_off[i], the number
 * actually needed is returned in d_cnt_len[i] (> capacity means it did not fit). */
int ampis_poly_to_rle(const double *d_xy, const int64_t *d_xy_off, const uint32_t *d_h,
                      const uint32_t *d_w, int32_t n, uint32_t *d_cnt, const int64_t *d_cnt_off,
                      int32_t *d_cnt_len, void *stream);

/* skimage.draw.polygon2mask as used by structures._poly2mask (structures.py:693-715, reached from
 * masks_to_bitmask_array(PolygonMasks), structures.py:743-747): pixel (r, c) is set when the
 * crossing-number test of skimage's _pnpoly.pxd holds for (x = c, y = r).  d_xy holds x0,y0,x1,y1,...
 * of all polygons (the same layout as ampis_poly_to_rle).  d_out: u8[n][h][w], zeroed here. */
int ampis_polygon2mask(const double *d_xy, const int64_t *d_xy_off, int32_t n, int32_t h, int32_t w,
                       uint8_t *d_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* AMPIS_B200_H */
