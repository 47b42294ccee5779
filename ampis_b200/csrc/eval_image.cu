// One image through the whole matching path in ONE library call (host-side orchestration only; every
// computation is one of the kernels of this library):
//
//   compressed RLE strings (host) -> pinned staging -> one H2D copy -> rleFrString on the GPU -> fused measure +
//   crop decode -> rows kernel (all-columns scan, or grid-pruned from `grid_min_cols` columns on) -> one D2H copy
//   of the per-row results and per-mask measurements -> one stream synchronisation.
//
// This is what analyze.py:149-164 (G x ceil(P/80) RLE.iou calls + arg-max) and powder.py:80-86 (S x N RLE.merge +
// RLE.area) cost per image in the reference.  The drop-in functions evaluate one image per Python call; driving the
// ten kernels from Python costs ~1 ms of interpreter, allocator and launch overhead per call for ~0.1 ms of GPU
// work, which is what this entry point removes.  It allocates nothing: the caller passes a device workspace and a
// pinned host workspace and is told how much is needed when they are too small.
#include <string.h>

#include "common.cuh"

static inline int64_t al256(int64_t x) { return (x + 255) & ~(int64_t)255; }

struct Carve {
    int64_t off = 0;
    int64_t take(int64_t bytes) { const int64_t o = off; off = al256(off + bytes); return o; }
};

extern "C" int ampis_eval_image_host(const uint8_t *chars, const int64_t *chr_off, int32_t n_rows, int32_t n_cols,
                                     uint32_t h, uint32_t w, int32_t mode, int32_t grid_min_cols,
                                     void *d_ws, int64_t d_ws_bytes, void *h_ws, int64_t h_ws_bytes,
                                     int32_t *best_col, uint32_t *best_inter, double *best_score, uint32_t *area,
                                     int32_t *bbox, uint32_t *span, int32_t *status, double *iou_out, int64_t *need_bytes,
                                     void *stream)
{
    AMPIS_REQUIRE(n_rows >= 0 && n_cols >= 0, "negative size");
    AMPIS_REQUIRE(mode == AMPIS_MODE_IOU || mode == AMPIS_MODE_SAT, "bad mode");
    AMPIS_REQUIRE(chr_off && d_ws && h_ws && best_col && best_inter && best_score && area && bbox && span && status && need_bytes,
                  "null pointer");
    AMPIS_REQUIRE(((uintptr_t)d_ws & 255u) == 0, "device workspace must be 256-byte aligned");
    const int64_t n = (int64_t)n_rows + n_cols;
    if (n == 0) return AMPIS_OK;
    const int64_t n_chars = chr_off[n] - chr_off[0];
    AMPIS_REQUIRE(chr_off[0] == 0 && n_chars >= 0 && (chars || n_chars == 0), "bad string offsets");
    const int32_t nb = (n_rows + ampis_rows_per_block() - 1) / ampis_rows_per_block();
    const bool use_grid = n_cols >= grid_min_cols && n_rows > 0;
    const int cells = ampis_grid_cells();
    const int64_t grid_base = use_grid ? 16 * (int64_t)n_cols + 4096 : 0;
    const int64_t grid_cap = use_grid ? ampis_grid_capacity(grid_base, d_ws_bytes) : 0;

    // ---- layout: [upload block][download block][device-only][arena] ---------------------------------------
    Carve c;
    const int64_t u_chars = c.take(n_chars), u_off = c.take(8 * (n + 1)), u_h = c.take(4 * n), u_w = c.take(4 * n);
    const int64_t u_rowmask = c.take(4 * (int64_t)n_rows), u_blkgrp = c.take(4 * (int64_t)nb), u_blkrow = c.take(4 * (int64_t)nb);
    const int64_t u_grb = c.take(4), u_grc = c.take(4), u_gcb = c.take(4), u_gcc = c.take(4);
    const int64_t upload_bytes = c.off;
    const int64_t dl0 = c.off;
    const int64_t o_col = c.take(4 * (int64_t)n_rows), o_inter = c.take(4 * (int64_t)n_rows), o_score = c.take(8 * (int64_t)n_rows);
    const int64_t o_area = c.take(4 * n), o_bbox = c.take(16 * n), o_span = c.take(8 * n), o_status = c.take(4 * n), o_cursor = c.take(8);
    const int64_t o_gridtot = c.take(8), o_pairtot = c.take(8);
    const int64_t download_bytes = c.off - dl0;
    const int64_t host_bytes = c.off;
    const int64_t d_cnt = c.take(4 * n_chars), d_cum = c.take(4 * n_chars), d_cntlen = c.take(4 * n);
    const int64_t d_reg = c.take(8 * n), d_bitsoff = c.take(8 * (n + 1)), d_list = c.take(4 * (n + 1));
    int64_t g_shift = 0, g_off = 0, g_ent = 0, g_entbb = 0, p_off = 0, p_cnt = 0, p_grp = 0;
    if (use_grid) {
        g_shift = c.take(4); g_off = c.take(8 * ((int64_t)cells + 1)); g_ent = c.take(4 * grid_cap);
        g_entbb = c.take(16 * grid_cap);
        p_off = c.take(8 * (int64_t)n_rows); p_cnt = c.take(4 * (int64_t)n_rows); p_grp = c.take(4 * (int64_t)n_rows);
    }
    // optional dense output: int32 intersections and the float64 IoU matrix of _piecewise_iou (analyze.py:54-112)
    const bool dense = iou_out && n_rows > 0 && n_cols > 0;
    const int64_t gp = (int64_t)n_rows * n_cols;
    const int64_t x_imat = dense ? c.take(4 * gp) : 0, x_iou = dense ? c.take(8 * gp) : 0, x_imoff = dense ? c.take(8) : 0;
    const int64_t fixed0 = c.off;
    // the grid entry list is the part of fixed0 that grows with d_ws (common.cuh)
    const int64_t grid_bytes = AMPIS_GRID_ENTRY_BYTES * grid_cap;
    auto need_for = [&](int64_t rest, int64_t entries) {
        return use_grid ? ampis_ws_need_with_grid(rest, grid_base, entries) : rest;
    };
    // what is left: a quarter for the candidate-pair list of the join (44 bytes per pair), the rest for the arena
    // (at least a window of 64 bytes per mask to start with)
    if (h_ws_bytes < host_bytes || d_ws_bytes < fixed0 + 128 * n + 8192) {
        *need_bytes = need_for(fixed0 - grid_bytes + 4096 * n + 131072, 0);
        if (h_ws_bytes < host_bytes) *need_bytes = -(host_bytes);      // negative: the HOST workspace is the short one
        ampis_set_error("%s workspace too small", h_ws_bytes < host_bytes ? "host" : "device");
        return AMPIS_ENOSPC;
    }
    const int64_t pair_cap = use_grid ? ((d_ws_bytes - fixed0) / 4 - 1024) / 44 : 0;
    const int64_t p_ab = c.take(8 * pair_cap), p_desc = c.take(32 * pair_cap), p_inter = c.take(4 * pair_cap);
    const int64_t arena0 = c.off;
    const int64_t arena_chunks = (d_ws_bytes - arena0) / 16;
    uint8_t *H = (uint8_t *)h_ws, *D = (uint8_t *)d_ws;
    cudaStream_t st = as_stream(stream);

    // ---- fill the upload block ---------------------------------------------------------------------------
    if (n_chars) memcpy(H + u_chars, chars, (size_t)n_chars);
    memcpy(H + u_off, chr_off, (size_t)(8 * (n + 1)));
    uint32_t *ph = (uint32_t *)(H + u_h), *pw = (uint32_t *)(H + u_w);
    for (int64_t i = 0; i < n; i++) { ph[i] = h; pw[i] = w; }
    int32_t *prm = (int32_t *)(H + u_rowmask), *pbg = (int32_t *)(H + u_blkgrp), *pbr = (int32_t *)(H + u_blkrow);
    for (int32_t i = 0; i < n_rows; i++) prm[i] = i;
    for (int32_t b = 0; b < nb; b++) { pbg[b] = 0; pbr[b] = b * ampis_rows_per_block(); }
    *(int32_t *)(H + u_grb) = 0; *(int32_t *)(H + u_grc) = n_rows;
    *(int32_t *)(H + u_gcb) = n_rows; *(int32_t *)(H + u_gcc) = n_cols;
    cudaError_t e = cudaMemcpyAsync(D, H, (size_t)upload_bytes, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) { ampis_set_error("upload: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }

    // ---- kernels --------------------------------------------------------------------------------------------
    int rc;
#define STEP(call) do { rc = (call); if (rc != AMPIS_OK) return rc; } while (0)
    // interval windows for the pairs join; the column scan of narrow images (ampis_intersect_rows_crop) reads bitmaps
    const int32_t iv = use_grid && ampis_pairs_read_intervals() ? 1 : 0;
    STEP(ampis_rle_string_decode(D + u_chars, (const int64_t *)(D + u_off), (int32_t)n, (uint32_t *)(D + d_cnt),
                                 (const int64_t *)(D + u_off), (int32_t *)(D + d_cntlen), stream));
    STEP(ampis_rle_measure_paint_flat((const uint32_t *)(D + d_cnt), (const int64_t *)(D + u_off), (const int32_t *)(D + d_cntlen),
                                      (const uint32_t *)(D + u_h), (const uint32_t *)(D + u_w), (int32_t)n,
                                      (uint32_t *)(D + d_cum), (uint32_t *)(D + o_area), (int32_t *)(D + o_bbox),
                                      (uint32_t *)(D + o_span), (uint32_t *)(D + d_reg), (int64_t *)(D + d_bitsoff),
                                      (int32_t *)(D + o_status), D + arena0, arena_chunks, (uint64_t *)(D + o_cursor),
                                      (int32_t *)(D + d_list), (int32_t)(n_chars / n), iv, stream));
    if (dense) {
        e = cudaMemsetAsync(D + x_imoff, 0, 8, st);                 // the image's matrix starts at offset 0
        if (e != cudaSuccess) { ampis_set_error("imat offset: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }
    }
    if (n_rows > 0 && n_cols > 0) {
        if (use_grid) {
            STEP(ampis_grid_build((const int32_t *)(D + o_bbox), (const int32_t *)(D + u_gcb), (const int32_t *)(D + u_gcc), 1,
                                  (int32_t *)(D + g_shift), (int64_t *)(D + g_off), (int32_t *)(D + g_ent),
                                  (int32_t *)(D + g_entbb), grid_cap, (uint64_t *)(D + o_gridtot), stream));
            e = cudaMemsetAsync(D + p_grp, 0, (size_t)(4 * (int64_t)n_rows), st);          // every row belongs to group 0
            if (e != cudaSuccess) { ampis_set_error("row groups: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }
            STEP(ampis_intersect_rows_pairs(D + arena0, (const int64_t *)(D + d_bitsoff),
                                            iv ? (const uint32_t *)(D + d_reg) : nullptr, (const int32_t *)(D + o_bbox),
                                            (const uint32_t *)(D + o_area), (const int32_t *)(D + u_rowmask),
                                            (const int32_t *)(D + p_grp), n_rows, (const int32_t *)(D + u_grb),
                                            (const int32_t *)(D + u_gcb), (const int32_t *)(D + u_gcc),
                                            (const int32_t *)(D + g_shift), (const int64_t *)(D + g_off),
                                            (const int32_t *)(D + g_ent), (const int32_t *)(D + g_entbb), grid_cap,
                                            (int32_t *)(D + p_ab), D + p_desc, (uint32_t *)(D + p_inter), pair_cap,
                                            (int64_t *)(D + p_off), (int32_t *)(D + p_cnt), (uint64_t *)(D + o_pairtot),
                                            dense ? (const int64_t *)(D + x_imoff) : nullptr, mode,
                                            dense ? (int32_t *)(D + x_imat) : nullptr, dense ? gp : 0, (int32_t *)(D + o_col),
                                            (uint32_t *)(D + o_inter), (double *)(D + o_score), nullptr, nullptr, nullptr,
                                            0, nullptr, nullptr, stream));
        } else {
            STEP(ampis_intersect_rows_crop(D + arena0, (const int64_t *)(D + d_bitsoff), (const int32_t *)(D + o_bbox),
                                           (const uint32_t *)(D + o_area), (const int32_t *)(D + u_rowmask),
                                           (const int32_t *)(D + u_blkgrp), (const int32_t *)(D + u_blkrow), nb,
                                           (const int32_t *)(D + u_grb), (const int32_t *)(D + u_grc),
                                           (const int32_t *)(D + u_gcb), (const int32_t *)(D + u_gcc),
                                           dense ? (const int64_t *)(D + x_imoff) : nullptr, mode,
                                           dense ? (int32_t *)(D + x_imat) : nullptr, (int32_t *)(D + o_col), (uint32_t *)(D + o_inter), (double *)(D + o_score), stream));
        }
    }
    if (dense) {
        STEP(ampis_iou_matrix_f64((const int32_t *)(D + x_imat), (const uint32_t *)(D + o_area),
                                  (const uint32_t *)(D + o_area) + n_rows, n_rows, n_cols, (double *)(D + x_iou), stream));
        e = cudaMemcpyAsync(iou_out, D + x_iou, (size_t)(8 * gp), cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) { ampis_set_error("iou download: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }
    }
#undef STEP
    e = cudaMemcpyAsync(H + dl0, D + dl0, (size_t)download_bytes, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { ampis_set_error("download: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }

    // ---- did everything fit? ------------------------------------------------------------------------------------
    const uint64_t used = *(const uint64_t *)(H + o_cursor);
    const int64_t pairs_found = use_grid && n_rows > 0 && n_cols > 0 ? *(const int64_t *)(H + o_pairtot) : 0;
    const int64_t entries = use_grid && n_cols > 0 ? *(const int64_t *)(H + o_gridtot) : 0;
    const bool short_ws = (int64_t)used > arena_chunks || pairs_found > pair_cap;
    if (short_ws || entries > grid_cap) {
        // the free part is split 1 : 3 between the pair list and the arena (when the grid list overflowed, the join
        // missed candidates: a later call may still ask for more pair room)
        int64_t rest = d_ws_bytes - grid_bytes;
        if (short_ws) {
            const int64_t by_arena = (16 * (int64_t)used + 65536) * 4 / 3, by_pairs = (44 * pairs_found + 4096) * 4;
            rest = fixed0 - grid_bytes + (by_arena > by_pairs ? by_arena : by_pairs) + 65536;
        }
        *need_bytes = need_for(rest, entries);
        ampis_set_error("device workspace too small (%lld bytes; grid entries: %lld)", (long long)d_ws_bytes,
                        (long long)entries);
        return AMPIS_ENOSPC;
    }
    if (n_rows > 0 && n_cols > 0) {
        memcpy(best_col, H + o_col, (size_t)(4 * (int64_t)n_rows));
        memcpy(best_inter, H + o_inter, (size_t)(4 * (int64_t)n_rows));
        memcpy(best_score, H + o_score, (size_t)(8 * (int64_t)n_rows));
    }
    memcpy(area, H + o_area, (size_t)(4 * n));
    memcpy(bbox, H + o_bbox, (size_t)(16 * n));
    memcpy(span, H + o_span, (size_t)(8 * n));
    memcpy(status, H + o_status, (size_t)(4 * n));
    return AMPIS_OK;
}
