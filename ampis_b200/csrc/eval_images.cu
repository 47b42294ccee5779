// MANY images through the whole matching path in ONE library call, from host string descriptors: the loop a user of
// the reference writes around det_seg_scores / _rle_satellite_match (Colab cell 44 -> analyze.py:226; cell 62 ->
// powder.py:138), i.e. per image analyze.py:149-164 / powder.py:80-86.  Host-side orchestration only; every
// computation is one of the kernels of this library:
//
//   (pointer, length) of every compressed RLE string (rows of image 0, columns of image 0, rows of image 1, ...)
//   -> strings gathered into pinned staging together with the bookkeeping arrays -> ONE H2D copy -> rleFrString on
//   the GPU -> flat measure + crop decode -> column grid -> candidate-pair join -> AND+popc per pair -> per-row
//   arg-max -> ONE D2H copy of the per-row results and per-mask measurements -> ONE stream synchronisation.
//
// No per-image launch, copy or synchronisation; nothing is allocated (caller's workspaces, sizes reported when too
// small, as ampis_eval_image_host).  A batch whose candidate pairs exceed `crowd_frac` of all row x column pairs is
// CROWDED: the intersections are skipped on the device (no host round trip is needed to decide) and the call returns
// with *crowded = 1, so that the caller can send it to the tensor-core contraction without having paid for the
// culled walk first.
#include <string.h>
#include <thread>
#include <vector>

#include "common.cuh"

static inline int64_t al256(int64_t x) { return (x + 255) & ~(int64_t)255; }

namespace {
struct Carve {
    int64_t off = 0;
    int64_t take(int64_t bytes) { const int64_t o = off; off = al256(off + bytes); return o; }
};
}

// Records the number of candidate pairs and raises the crowd flag when it exceeds the limit (the join was given the
// limit as its capacity, so the AND+popc pass has already returned without doing anything).  One thread.
__global__ void crowd_gate_kernel(unsigned long long *pair_count, unsigned long long *found, long long limit, int *flag)
{
    const unsigned long long n = *pair_count;
    *found = n;
    if (limit >= 0 && (long long)n > limit) { *flag = 1; } else { *flag = 0; }
}

extern "C" int ampis_intersect_rows_pairs(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox,
                                          const uint32_t *d_area, const int32_t *d_row_mask, const int32_t *d_row_grp,
                                          int32_t n_rows, const int32_t *d_grp_row_begin,
                                          const int32_t *d_grp_col_begin, const int32_t *d_grp_col_count,
                                          const int32_t *d_grp_shift, const int64_t *d_cell_off,
                                          const int32_t *d_entries, const int32_t *d_entry_bbox, int64_t grid_capacity,
                                          int32_t *d_pair_ab, void *d_pair_desc, uint32_t *d_pair_inter,
                                          int64_t pair_capacity, int64_t *d_row_pair_off, int32_t *d_row_pair_cnt,
                                          uint64_t *d_pair_count, const int64_t *d_grp_imat_off, int32_t mode,
                                          int32_t *d_imat, int64_t imat_ints, int32_t *d_best_col,
                                          uint32_t *d_best_inter, double *d_best_score, int32_t *d_coo_row,
                                          int32_t *d_coo_col, uint32_t *d_coo_inter, int64_t coo_capacity,
                                          uint64_t *d_coo_count, void *zero_stream, void *stream);

// Per-mask bookkeeping of a large batch formed ON THE DEVICE from the per-image arrays (a host loop over a million
// masks costs more than the GPU needs for the whole evaluation): one CTA per image writes the image size of each of
// its masks, the string lengths as int64 (input of the offset scan) and the row -> mask / row -> image maps.
__global__ void __launch_bounds__(256)
expand_images_kernel(const int *__restrict__ n_rows, const int *__restrict__ n_cols, const u32 *__restrict__ h,
                     const u32 *__restrict__ w, const i64 *__restrict__ mask_off, const i64 *__restrict__ row_off,
                     const int *__restrict__ str_len, u32 *__restrict__ mh, u32 *__restrict__ mw,
                     i64 *__restrict__ len64, int *__restrict__ row_mask, int *__restrict__ row_grp,
                     int *__restrict__ grp_row_begin, int *__restrict__ grp_row_count, int *__restrict__ grp_col_begin,
                     int *__restrict__ grp_col_count)
{
    const int g = blockIdx.x;
    const i64 m0 = mask_off[g], r0 = row_off[g];
    const int nr = n_rows[g], nc = n_cols[g];
    const u32 hh = h[g], ww = w[g];
    for (int k = threadIdx.x; k < nr + nc; k += blockDim.x) {
        mh[m0 + k] = hh;
        mw[m0 + k] = ww;
        len64[m0 + k] = (i64)str_len[m0 + k];
    }
    for (int k = threadIdx.x; k < nr; k += blockDim.x) {
        row_mask[r0 + k] = (int)(m0 + k);
        row_grp[r0 + k] = g;
    }
    if (threadIdx.x == 0) {
        grp_row_begin[g] = (int)r0;
        grp_row_count[g] = nr;
        grp_col_begin[g] = (int)(m0 + nr);
        grp_col_count[g] = nc;
    }
}

#define EI_HOST_FILL_MAX 16384          // up to this many masks the host fills the per-mask arrays itself

// page-locked host memory (cudaHostAlloc / cudaHostRegister)?  Such buffers are DMA targets themselves: large batches
// skip the staging copy for them
static bool is_pinned(const void *p)
{
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// The compressed strings of a call lie wherever Python keeps them: gathering them into the pinned upload block is one
// cache miss (or two) per string -- 4 ms for the 200,000 strings of 200 C2 images on one core, a quarter of such a
// call.  Plain memory, no interpreter state: done by a few threads, each over a contiguous range of masks.
static void gather_strings(uint8_t *dst, const uint8_t *const *str_ptr, const int32_t *str_len, int64_t n, int64_t n_chars)
{
    const unsigned hw = std::thread::hardware_concurrency();
    int64_t T = n_chars >= (4 << 20) ? (hw >= 16 ? 6 : hw >= 8 ? 4 : hw >= 4 ? 2 : 1) : 1;
    if (T > n) T = 1;
    auto part = [=](int64_t k0, int64_t k1, int64_t pos) {
        for (int64_t k = k0; k < k1; k++) {
            if (str_len[k]) memcpy(dst + pos, str_ptr[k], (size_t)str_len[k]);
            pos += str_len[k];
        }
    };
    if (T <= 1) { part(0, n, 0); return; }
    std::vector<std::thread> th;
    int64_t k0 = 0, pos = 0;
    for (int64_t t = 0; t < T; t++) {
        const int64_t k1 = t + 1 == T ? n : n * (t + 1) / T;
        if (t + 1 < T) th.emplace_back(part, k0, k1, pos);
        else part(k0, k1, pos);                     // the last range on the calling thread
        for (int64_t k = k0; k < k1 && t + 1 < T; k++) pos += str_len[k];
        k0 = k1;
    }
    for (auto &x : th) x.join();
}

namespace {
// The inputs of a many-image call that the shared front and back halves read
struct ImagesIn {
    const uint8_t *const *str_ptr;
    const int32_t *str_len;
    int32_t n_images;
    const int32_t *n_rows, *n_cols;
    const uint32_t *h, *w;
    int32_t mode, flags;
    void *d_ws;
    int64_t d_ws_bytes;
    void *h_ws;
    int64_t h_ws_bytes;
    bool rows_out;                  // per-row results and per-mask measurements wanted (else the mask status only)
    int32_t *best_col;
    uint32_t *best_inter;
    double *best_score;
    uint32_t *area;
    int32_t *bbox, *status;
    uint32_t *span;
    int64_t *need_bytes;
    void *stream;
};

// The caller's own parts of the workspaces: up to two host arrays uploaded with the strings, a block downloaded with
// the counters, and device-only space.  images_front places them and returns their offsets.
struct ImagesExtra {
    const void *up[2] = {nullptr, nullptr};
    int64_t up_bytes[2] = {0, 0};
    int64_t dl_bytes = 0, dev_bytes = 0;
    int64_t up_off[2] = {0, 0}, dl_off = 0, dev_off = 0;
};

// Where everything lies after images_front (offsets into both workspaces), and the sizes of the call
struct ImagesRun {
    uint8_t *H, *D;
    cudaStream_t st;
    int64_t n, R, NI, all_pairs;
    int32_t max_cols;
    bool have_rows, out_direct;
    int64_t x_rowmask, x_rowgrp, x_grb, x_grc, x_gcb, x_gcc;
    int64_t o_col, o_inter, o_score, o_area, o_status, o_bbox, o_span;
    int64_t o_cursor, o_gridtot, o_pairfound, o_crowd;
    int64_t p_ab, p_desc, p_inter, p_off, p_cnt, pair_cap;
    int64_t dl0, download_bytes, fixed0, grid_bytes, grid_base, grid_cap, arena_chunks;
};
}

// The part both many-image entries share: sizes and checks, workspace layout, the upload, string decode, flat measure
// + crop decode, column grids, candidate-pair join, AND+popc and per-row arg-max, and the crowd gate (crowd_frac as
// ampis_eval_images_host).
// r.n == 0: no mask at all, nothing was launched.
static int images_front(const ImagesIn &in, ImagesExtra &x, double crowd_frac, ImagesRun &r)
{
    const int32_t n_images = in.n_images;
    const int32_t *n_rows = in.n_rows, *n_cols = in.n_cols;
    const uint32_t *h = in.h, *w = in.w;
    const uint8_t *const *str_ptr = in.str_ptr;
    const int32_t *str_len = in.str_len;
    const int64_t d_ws_bytes = in.d_ws_bytes, h_ws_bytes = in.h_ws_bytes;
    AMPIS_REQUIRE(n_rows && n_cols && h && w, "null pointer");
    int64_t n = 0, R = 0, all_pairs = 0;
    int32_t max_cols = 0;
    for (int32_t g = 0; g < n_images; g++) {
        AMPIS_REQUIRE(n_rows[g] >= 0 && n_cols[g] >= 0, "negative size");
        n += (int64_t)n_rows[g] + n_cols[g];
        R += n_rows[g];
        all_pairs += (int64_t)n_rows[g] * n_cols[g];
        if (n_cols[g] > max_cols) max_cols = n_cols[g];
    }
    AMPIS_REQUIRE(n <= 0x7fffffff, "more than 2^31 masks in one call");
    r.n = n; r.R = R; r.NI = n_images; r.all_pairs = all_pairs; r.max_cols = max_cols;
    r.have_rows = R > 0 && all_pairs > 0;
    if (n == 0) return AMPIS_OK;
    AMPIS_REQUIRE(str_ptr && str_len && in.status && (!in.rows_out || (in.best_col && in.best_inter && in.best_score && in.area)),
                  "null pointer");
    const bool contiguous = (in.flags & AMPIS_STRINGS_CONTIGUOUS) != 0;
    const bool on_device = n > EI_HOST_FILL_MAX;          // per-mask bookkeeping by expand_images_kernel + a scan
    int64_t n_chars = 0;
    int32_t any_negative = 0;
    for (int64_t i = 0; i < n; i++) { n_chars += str_len[i]; any_negative |= str_len[i]; }
    AMPIS_REQUIRE(any_negative >= 0, "negative string length");
    if (!contiguous)
        for (int64_t i = 0; i < n; i++) AMPIS_REQUIRE(str_ptr[i] || str_len[i] == 0, "bad string descriptor");
    AMPIS_REQUIRE(str_ptr[0] || n_chars == 0, "bad string descriptor");
    const int cells = ampis_grid_cells();
    const int64_t grid_base = 16 * (n - R) + 4096 * (int64_t)n_images;
    const int64_t grid_cap = ampis_grid_capacity(grid_base, d_ws_bytes);
    const int64_t scan_tmp = on_device ? (int64_t)ampis_scan_tmp_bytes(n) : 0;
    const int64_t NI = n_images;

    // ---- layout: [upload block][download block][device-only][pair list][arena] -----------------------------------
    // upload: the strings (unless they are uploaded from where they are), their lengths or offsets, and either the
    // per-mask arrays (small batches: filled by the host) or the per-image arrays they are expanded from
    Carve c;
    const int64_t u_chars = contiguous ? 0 : c.take(n_chars);
    const int64_t u_off = on_device ? 0 : c.take(8 * (n + 1));
    const int64_t u_h = on_device ? 0 : c.take(4 * n), u_w = on_device ? 0 : c.take(4 * n);
    const int64_t u_rowmask = on_device ? 0 : c.take(4 * R), u_rowgrp = on_device ? 0 : c.take(4 * R);
    const int64_t u_grb = on_device ? 0 : c.take(4 * NI), u_grc = on_device ? 0 : c.take(4 * NI),
                  u_gcb = on_device ? 0 : c.take(4 * NI), u_gcc = on_device ? 0 : c.take(4 * NI);
    for (int k = 0; k < 2; k++) x.up_off[k] = c.take(x.up_bytes[k]);
    const int64_t i_nr = on_device ? c.take(4 * NI) : 0, i_nc = on_device ? c.take(4 * NI) : 0,
                  i_h = on_device ? c.take(4 * NI) : 0, i_w = on_device ? c.take(4 * NI) : 0,
                  i_moff = on_device ? c.take(8 * NI) : 0, i_roff = on_device ? c.take(8 * NI) : 0;
    // the string lengths last: when the caller keeps them in pinned memory they are uploaded from where they are
    const bool len_direct = on_device && is_pinned(str_len);
    const int64_t staged_upload = c.off;
    const int64_t u_len = on_device ? c.take(4 * n) : 0;
    const int64_t upload_bytes = len_direct ? staged_upload : c.off;
    // download: the caller's block and the counters first (always through the staging buffer), then the status and
    // (when asked for) the per-mask and per-row results -- straight into the caller's arrays when those are pinned,
    // else through the staging buffer too
    const int64_t dl0 = c.off;
    x.dl_off = c.take(x.dl_bytes);
    const int64_t o_cursor = c.take(8), o_gridtot = c.take(8), o_pairtot = c.take(8), o_pairfound = c.take(8),
                  o_crowd = c.take(8);
    const int64_t dl_small = c.off - dl0;
    const int64_t o_status = c.take(4 * n);
    const int64_t dl_status = c.off - dl0;
    const int64_t o_area = c.take(4 * n), o_col = c.take(4 * R), o_inter = c.take(4 * R), o_score = c.take(8 * R);
    const int64_t dl_short = c.off - dl0;
    const int64_t o_bbox = c.take(16 * n), o_span = c.take(8 * n);
    const bool rows_out = in.rows_out;
    const bool out_direct = rows_out && n > EI_HOST_FILL_MAX && is_pinned(in.best_col) && is_pinned(in.best_inter) &&
                            is_pinned(in.best_score) && is_pinned(in.area) && is_pinned(in.status) &&
                            (!in.bbox || is_pinned(in.bbox)) && (!in.span || is_pinned(in.span));
    const int64_t download_bytes = out_direct ? dl_small : !rows_out ? dl_status
                                   : ((in.bbox || in.span) ? c.off - dl0 : dl_short);
    const int64_t host_bytes = dl0 + download_bytes;
    // device only
    const int64_t x_chars = contiguous ? c.take(n_chars) : u_chars;
    const int64_t x_off = on_device ? c.take(8 * (n + 1)) : u_off;
    const int64_t x_len64 = on_device ? c.take(8 * n) : 0, x_scan = on_device ? c.take(scan_tmp) : 0;
    const int64_t x_h = on_device ? c.take(4 * n) : u_h, x_w = on_device ? c.take(4 * n) : u_w;
    const int64_t x_rowmask = on_device ? c.take(4 * R) : u_rowmask, x_rowgrp = on_device ? c.take(4 * R) : u_rowgrp;
    const int64_t x_grb = on_device ? c.take(4 * NI) : u_grb, x_grc = on_device ? c.take(4 * NI) : u_grc,
                  x_gcb = on_device ? c.take(4 * NI) : u_gcb, x_gcc = on_device ? c.take(4 * NI) : u_gcc;
    const int64_t d_cnt = c.take(4 * n_chars), d_cum = c.take(4 * n_chars), d_cntlen = c.take(4 * n);
    const int64_t d_reg = c.take(8 * n), d_bitsoff = c.take(8 * (n + 1)), d_list = c.take(4 * (n + 1));
    const int64_t g_shift = c.take(4 * NI), g_off = c.take(8 * ((int64_t)cells + 1) * NI),
                  g_ent = c.take(4 * grid_cap), g_entbb = c.take(16 * grid_cap);
    const int64_t p_off = c.take(8 * R), p_cnt = c.take(4 * R);
    x.dev_off = c.take(x.dev_bytes);
    const int64_t fixed0 = c.off;
    const int64_t grid_bytes = AMPIS_GRID_ENTRY_BYTES * grid_cap;        // the part of fixed0 that grows with d_ws
    if (h_ws_bytes < host_bytes || d_ws_bytes < fixed0 + 128 * n + 8192) {
        *in.need_bytes = ampis_ws_need_with_grid(fixed0 - grid_bytes + 4096 * n + 131072, grid_base, 0);
        if (h_ws_bytes < host_bytes) *in.need_bytes = -(host_bytes);      // negative: the HOST workspace is the short one
        ampis_set_error("%s workspace too small", h_ws_bytes < host_bytes ? "host" : "device");
        return AMPIS_ENOSPC;
    }
    // what is left: a quarter for the candidate pairs of the join (44 bytes each), the rest for the window arena
    const int64_t pair_cap = R > 0 ? ((d_ws_bytes - fixed0) / 4 - 1024) / 44 : 0;
    const int64_t p_ab = c.take(8 * pair_cap), p_desc = c.take(32 * pair_cap), p_inter = c.take(4 * pair_cap);
    const int64_t arena0 = c.off;
    const int64_t arena_chunks = (d_ws_bytes - arena0) / 16;
    uint8_t *H = (uint8_t *)in.h_ws, *D = (uint8_t *)in.d_ws;
    cudaStream_t st = as_stream(in.stream);
    cudaError_t e;
    r.H = H; r.D = D; r.st = st; r.out_direct = out_direct;
    r.x_rowmask = x_rowmask; r.x_rowgrp = x_rowgrp; r.x_grb = x_grb; r.x_grc = x_grc; r.x_gcb = x_gcb; r.x_gcc = x_gcc;
    r.o_col = o_col; r.o_inter = o_inter; r.o_score = o_score; r.o_area = o_area; r.o_status = o_status;
    r.o_bbox = o_bbox; r.o_span = o_span;
    r.o_cursor = o_cursor; r.o_gridtot = o_gridtot; r.o_pairfound = o_pairfound; r.o_crowd = o_crowd;
    r.p_ab = p_ab; r.p_desc = p_desc; r.p_inter = p_inter; r.p_off = p_off; r.p_cnt = p_cnt; r.pair_cap = pair_cap;
    r.dl0 = dl0; r.download_bytes = download_bytes; r.fixed0 = fixed0; r.grid_bytes = grid_bytes;
    r.grid_base = grid_base; r.grid_cap = grid_cap; r.arena_chunks = arena_chunks;

    // ---- fill the upload block ------------------------------------------------------------------------------------
    for (int k = 0; k < 2; k++)
        if (x.up_bytes[k]) memcpy(H + x.up_off[k], x.up[k], (size_t)x.up_bytes[k]);
    if (on_device) {
        if (!len_direct) memcpy(H + u_len, str_len, (size_t)(4 * n));
        memcpy(H + i_nr, n_rows, (size_t)(4 * NI));
        memcpy(H + i_nc, n_cols, (size_t)(4 * NI));
        memcpy(H + i_h, h, (size_t)(4 * NI));
        memcpy(H + i_w, w, (size_t)(4 * NI));
        int64_t *pm = (int64_t *)(H + i_moff), *pr = (int64_t *)(H + i_roff);
        int64_t i = 0, rr = 0;
        for (int32_t g = 0; g < n_images; g++) { pm[g] = i; pr[g] = rr; i += (int64_t)n_rows[g] + n_cols[g]; rr += n_rows[g]; }
        if (!contiguous) gather_strings(H + u_chars, str_ptr, str_len, n, n_chars);
    } else {
        int64_t *po = (int64_t *)(H + u_off);
        uint32_t *ph = (uint32_t *)(H + u_h), *pw = (uint32_t *)(H + u_w);
        int32_t *prm = (int32_t *)(H + u_rowmask), *prg = (int32_t *)(H + u_rowgrp);
        int32_t *pgrb = (int32_t *)(H + u_grb), *pgrc = (int32_t *)(H + u_grc), *pgcb = (int32_t *)(H + u_gcb),
                *pgcc = (int32_t *)(H + u_gcc);
        uint8_t *pc = contiguous ? nullptr : H + u_chars;
        int64_t i = 0, rr = 0, pos = 0;
        for (int32_t g = 0; g < n_images; g++) {
            pgrb[g] = (int32_t)rr;
            pgrc[g] = n_rows[g];
            pgcb[g] = (int32_t)(i + n_rows[g]);
            pgcc[g] = n_cols[g];
            for (int32_t k = 0; k < n_rows[g]; k++) { prm[rr] = (int32_t)(i + k); prg[rr] = g; rr++; }
            const int64_t end = i + n_rows[g] + n_cols[g];
            for (; i < end; i++) {
                po[i] = pos;
                ph[i] = h[g];
                pw[i] = w[g];
                if (pc && str_len[i]) memcpy(pc + pos, str_ptr[i], (size_t)str_len[i]);
                pos += str_len[i];
            }
        }
        po[n] = pos;
    }
    e = cudaMemcpyAsync(D, H, (size_t)upload_bytes, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && len_direct)
        e = cudaMemcpyAsync(D + u_len, str_len, (size_t)(4 * n), cudaMemcpyHostToDevice, st);
    // strings that already lie back to back (ideally in pinned memory) are uploaded from where they are
    if (e == cudaSuccess && contiguous && n_chars)
        e = cudaMemcpyAsync(D + x_chars, str_ptr[0], (size_t)n_chars, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) { ampis_set_error("upload: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }

    // ---- kernels --------------------------------------------------------------------------------------------------
    int rc;
#define STEP(call) do { rc = (call); if (rc != AMPIS_OK) return rc; } while (0)
    if (on_device) {
        expand_images_kernel<<<n_images, 256, 0, st>>>(
            (const int *)(D + i_nr), (const int *)(D + i_nc), (const u32 *)(D + i_h), (const u32 *)(D + i_w),
            (const i64 *)(D + i_moff), (const i64 *)(D + i_roff), (const int *)(D + u_len), (u32 *)(D + x_h),
            (u32 *)(D + x_w), (i64 *)(D + x_len64), (int *)(D + x_rowmask), (int *)(D + x_rowgrp), (int *)(D + x_grb),
            (int *)(D + x_grc), (int *)(D + x_gcb), (int *)(D + x_gcc));
        AMPIS_CHECK_LAUNCH("expand_images_kernel");
        STEP(ampis_exclusive_scan_i64((const int64_t *)(D + x_len64), (int64_t *)(D + x_off), n, D + x_scan,
                                      (size_t)scan_tmp, in.stream));
    }
    STEP(ampis_rle_string_decode(D + x_chars, (const int64_t *)(D + x_off), (int32_t)n, (uint32_t *)(D + d_cnt),
                                 (const int64_t *)(D + x_off), (int32_t *)(D + d_cntlen), in.stream));
    STEP(ampis_rle_measure_paint_flat((const uint32_t *)(D + d_cnt), (const int64_t *)(D + x_off),
                                      (const int32_t *)(D + d_cntlen), (const uint32_t *)(D + x_h),
                                      (const uint32_t *)(D + x_w), (int32_t)n, (uint32_t *)(D + d_cum),
                                      (uint32_t *)(D + o_area), (int32_t *)(D + o_bbox), (uint32_t *)(D + o_span),
                                      (uint32_t *)(D + d_reg), (int64_t *)(D + d_bitsoff), (int32_t *)(D + o_status),
                                      D + arena0, arena_chunks, (uint64_t *)(D + o_cursor), (int32_t *)(D + d_list),
                                      (int32_t)(n_chars / n), in.stream));
    e = cudaMemsetAsync(D + o_gridtot, 0, (size_t)(o_crowd + 8 - o_gridtot), st);      // grid total, pair total, pairs found, crowd flag
    if (e != cudaSuccess) { ampis_set_error("memset: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }
    if (r.have_rows) {
        STEP(ampis_grid_build((const int32_t *)(D + o_bbox), (const int32_t *)(D + x_gcb), (const int32_t *)(D + x_gcc),
                              n_images, (int32_t *)(D + g_shift), (int64_t *)(D + g_off), (int32_t *)(D + g_ent),
                              (int32_t *)(D + g_entbb), grid_cap, (uint64_t *)(D + o_gridtot), in.stream));
        // crowd gate: more candidate pairs than crowd_frac of all pairs -> the intersections are not computed
        const long long limit = crowd_frac >= 0.0 && crowd_frac < 1.0 ? (long long)(crowd_frac * (double)all_pairs) : -1;
        const int64_t cap = limit >= 0 && limit < pair_cap ? limit : pair_cap;
        STEP(ampis_intersect_rows_pairs(D + arena0, (const int64_t *)(D + d_bitsoff), (const int32_t *)(D + o_bbox),
                                        (const uint32_t *)(D + o_area), (const int32_t *)(D + x_rowmask),
                                        (const int32_t *)(D + x_rowgrp), (int32_t)R, (const int32_t *)(D + x_grb),
                                        (const int32_t *)(D + x_gcb), (const int32_t *)(D + x_gcc),
                                        (const int32_t *)(D + g_shift), (const int64_t *)(D + g_off),
                                        (const int32_t *)(D + g_ent), (const int32_t *)(D + g_entbb), grid_cap,
                                        (int32_t *)(D + p_ab), D + p_desc, (uint32_t *)(D + p_inter), cap,
                                        (int64_t *)(D + p_off), (int32_t *)(D + p_cnt), (uint64_t *)(D + o_pairtot),
                                        nullptr, in.mode, nullptr, 0, (int32_t *)(D + o_col), (uint32_t *)(D + o_inter),
                                        (double *)(D + o_score), nullptr, nullptr, nullptr, 0, nullptr, nullptr,
                                        in.stream));
        crowd_gate_kernel<<<1, 1, 0, st>>>((unsigned long long *)(D + o_pairtot), (unsigned long long *)(D + o_pairfound),
                                           limit, (int *)(D + o_crowd));
        AMPIS_CHECK_LAUNCH("crowd_gate_kernel");
    }
#undef STEP
    return AMPIS_OK;
}

// The other half both entries share: one download (plus the per-row arrays straight into pinned outputs), one wait,
// and the check that the arena, the pair list and the grid entry list were large enough (AMPIS_ENOSPC otherwise,
// with *need_bytes).  The caller has queued its own kernels and copies on r.st before.
static int images_back(const ImagesIn &in, const ImagesRun &r, int64_t *pairs_found, int32_t *crowded)
{
    uint8_t *H = r.H, *D = r.D;
    const cudaStream_t st = r.st;
    const int64_t n = r.n, R = r.R;
    cudaError_t e = cudaMemcpyAsync(H + r.dl0, D + r.dl0, (size_t)r.download_bytes, cudaMemcpyDeviceToHost, st);
    if (r.out_direct) {
#define DL(dst, off, bytes) if (e == cudaSuccess && (bytes) > 0) e = cudaMemcpyAsync(dst, D + (off), (size_t)(bytes), cudaMemcpyDeviceToHost, st)
        if (r.have_rows) { DL(in.best_col, r.o_col, 4 * R); DL(in.best_inter, r.o_inter, 4 * R); DL(in.best_score, r.o_score, 8 * R); }
        DL(in.area, r.o_area, 4 * n);
        DL(in.status, r.o_status, 4 * n);
        if (in.bbox) DL(in.bbox, r.o_bbox, 16 * n);
        if (in.span) DL(in.span, r.o_span, 8 * n);
#undef DL
    }
    if (e == cudaSuccess) {
        if (in.flags & AMPIS_WAIT_BLOCKING) {
            // wait on a BLOCKING event instead of spinning in cudaStreamSynchronize: the cores stay free for the other
            // calls in flight (several host threads per GPU, several ranks per host) at the price of a slower wake-up
            // (one rank alone: 2.75 vs 2.25 ms per C2 step, profiles/scaling_r02.md)
            cudaEvent_t ev;
            e = cudaEventCreateWithFlags(&ev, cudaEventBlockingSync | cudaEventDisableTiming);
            if (e == cudaSuccess) {
                e = cudaEventRecord(ev, st);
                if (e == cudaSuccess) e = cudaEventSynchronize(ev);
                cudaEventDestroy(ev);
            }
        } else {
            e = cudaStreamSynchronize(st);
        }
    }
    if (e != cudaSuccess) { ampis_set_error("download: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }

    // ---- did everything fit? -------------------------------------------------------------------------------------
    const uint64_t used = *(const uint64_t *)(H + r.o_cursor);
    const int64_t found = *(const int64_t *)(H + r.o_pairfound);
    const int64_t entries = *(const int64_t *)(H + r.o_gridtot);
    *pairs_found = found;
    *crowded = *(const int32_t *)(H + r.o_crowd);
    const bool short_ws = (int64_t)used > r.arena_chunks || (!*crowded && found > r.pair_cap);
    if (short_ws || entries > r.grid_cap) {
        // (when the grid list overflowed, the join missed candidates: a later call may still ask for more pair room)
        int64_t rest = in.d_ws_bytes - r.grid_bytes;
        if (short_ws) {
            const int64_t by_arena = (16 * (int64_t)used + 65536) * 4 / 3, by_pairs = (44 * found + 4096) * 4;
            rest = r.fixed0 - r.grid_bytes + (by_arena > by_pairs ? by_arena : by_pairs) + 65536;
        }
        *in.need_bytes = ampis_ws_need_with_grid(rest, r.grid_base, entries);
        ampis_set_error("device workspace too small (%lld bytes; grid entries: %lld)", (long long)in.d_ws_bytes,
                        (long long)entries);
        return AMPIS_ENOSPC;
    }
    if (!r.out_direct) memcpy(in.status, H + r.o_status, (size_t)(4 * n));
    return AMPIS_OK;
}

extern "C" int ampis_eval_images_host(const uint8_t *const *str_ptr, const int32_t *str_len, int32_t n_images,
                                      const int32_t *n_rows, const int32_t *n_cols, const uint32_t *h,
                                      const uint32_t *w, int32_t mode, int32_t flags, double crowd_frac,
                                      void *d_ws, int64_t d_ws_bytes, void *h_ws, int64_t h_ws_bytes,
                                      int32_t *best_col, uint32_t *best_inter, double *best_score, uint32_t *area,
                                      int32_t *bbox, uint32_t *span, int32_t *status, const double *thresholds,
                                      int32_t n_thresh, int32_t *grp_counts, int64_t *totals, int64_t *pairs_found,
                                      int32_t *crowded, int64_t *need_bytes, void *stream)
{
    AMPIS_REQUIRE(n_images >= 0, "negative size");
    AMPIS_REQUIRE(n_thresh >= 0 && (n_thresh == 0 || (thresholds && grp_counts && totals && mode == AMPIS_MODE_IOU)),
                  "threshold counts need thresholds, grp_counts, totals and AMPIS_MODE_IOU");
    AMPIS_REQUIRE(mode == AMPIS_MODE_IOU || mode == AMPIS_MODE_SAT, "bad mode");
    AMPIS_REQUIRE(d_ws && h_ws && need_bytes && pairs_found && crowded, "null pointer");
    AMPIS_REQUIRE(((uintptr_t)d_ws & 255u) == 0, "device workspace must be 256-byte aligned");
    *pairs_found = 0;
    *crowded = 0;
    for (int32_t t = 0; t < 3 * n_thresh; t++) totals[t] = 0;
    if (n_images == 0) return AMPIS_OK;
    for (int64_t t = 0; t < 3 * (int64_t)n_thresh * n_images; t++) grp_counts[t] = 0;
    const ImagesIn in{str_ptr, str_len, n_images, n_rows, n_cols, h, w, mode, flags, d_ws, d_ws_bytes, h_ws,
                      h_ws_bytes, true, best_col, best_inter, best_score, area, bbox, status, span, need_bytes, stream};
    const int64_t NI = n_images;
    ImagesExtra x;
    x.up[0] = thresholds;
    x.up_bytes[0] = 8 * (int64_t)n_thresh;
    x.dl_bytes = 12 * (int64_t)n_thresh * NI + 24 * (int64_t)n_thresh;        // counts, then totals
    ImagesRun r;
    int rc = images_front(in, x, crowd_frac, r);
    if (rc != AMPIS_OK || r.n == 0) return rc;
    uint8_t *H = r.H, *D = r.D;
    const int64_t o_counts = x.dl_off, o_totals = x.dl_off + 12 * (int64_t)n_thresh * NI, R = r.R, n = r.n;
    if (n_thresh && r.have_rows) {       // TP / FP / FN per image and threshold + totals (analyze.py:166-174), still on the device
        const cudaError_t e = cudaMemsetAsync(D + o_totals, 0, (size_t)(24 * (int64_t)n_thresh), r.st);
        if (e != cudaSuccess) { ampis_set_error("memset: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }
        rc = ampis_match_counts((const int32_t *)(D + r.o_col), (const double *)(D + r.o_score),
                                (const int32_t *)(D + r.x_grb), (const int32_t *)(D + r.x_grc),
                                (const int32_t *)(D + r.x_gcc), n_images, r.max_cols, (const double *)(D + x.up_off[0]),
                                n_thresh, (int32_t *)(D + o_counts), (int64_t *)(D + o_totals), stream);
        if (rc != AMPIS_OK) return rc;
    }
    rc = images_back(in, r, pairs_found, crowded);
    if (rc != AMPIS_OK) return rc;
    if (r.have_rows) {
        if (!r.out_direct) {
            memcpy(best_col, H + r.o_col, (size_t)(4 * R));
            memcpy(best_inter, H + r.o_inter, (size_t)(4 * R));
            memcpy(best_score, H + r.o_score, (size_t)(8 * R));
        }
    } else {
        for (int64_t k = 0; k < R; k++) { best_col[k] = -1; best_inter[k] = 0; best_score[k] = 0.0; }
    }
    if (n_thresh && r.have_rows) {
        memcpy(grp_counts, H + o_counts, (size_t)(12 * (int64_t)n_thresh * NI));
        memcpy(totals, H + o_totals, (size_t)(24 * (int64_t)n_thresh));
    } else if (n_thresh) {        // no pairs at all: every ground-truth mask is a false negative, every prediction a false positive
        for (int32_t g = 0; g < n_images; g++)
            for (int32_t t = 0; t < n_thresh; t++) {
                grp_counts[((int64_t)g * n_thresh + t) * 3 + 1] = n_cols[g];
                grp_counts[((int64_t)g * n_thresh + t) * 3 + 2] = n_rows[g];
                totals[3 * t + 1] += n_cols[g];
                totals[3 * t + 2] += n_rows[g];
            }
    }
    if (!r.out_direct) {
        memcpy(area, H + r.o_area, (size_t)(4 * n));
        if (bbox) memcpy(bbox, H + r.o_bbox, (size_t)(16 * n));
        if (span) memcpy(span, H + r.o_span, (size_t)(8 * n));
    }
    return AMPIS_OK;
}

int ampis_sweep_counts(const uint32_t *d_area, const int32_t *d_row_mask, const int32_t *d_row_grp, int32_t n_rows,
                       const int32_t *d_grp_row_begin, const int32_t *d_grp_row_count, const int32_t *d_grp_col_begin,
                       const int32_t *d_grp_col_count, int32_t n_groups, int32_t max_cols, const int32_t *d_pair_ab,
                       const uint32_t *d_pair_inter, const int64_t *d_row_pair_off, const int32_t *d_row_pair_cnt,
                       const uint16_t *d_levels, int32_t n_levels, const double *d_iou_thresh, int32_t n_iou,
                       void *d_stair, int32_t *d_counts, int64_t *d_seg, int64_t *d_totals, int64_t *d_seg_totals,
                       void *stream);

extern "C" int ampis_eval_images_sweep_host(const uint8_t *const *str_ptr, const int32_t *str_len, int32_t n_images,
                                            const int32_t *n_rows, const int32_t *n_cols, const uint32_t *h,
                                            const uint32_t *w, int32_t flags, const uint16_t *levels,
                                            int32_t n_levels, const double *iou_thresh, int32_t n_iou, void *d_ws,
                                            int64_t d_ws_bytes, void *h_ws, int64_t h_ws_bytes, int32_t *status,
                                            int64_t *totals, int64_t *seg_totals, int32_t *counts, int64_t *seg_sums,
                                            int64_t *pairs_found, int64_t *need_bytes, void *stream)
{
    AMPIS_REQUIRE(n_images >= 0, "negative size");
    AMPIS_REQUIRE(n_levels >= 1 && n_levels <= 65535, "the number of score levels must be in [1, 65535]");
    AMPIS_REQUIRE(n_iou >= 1 && n_iou <= AMPIS_SWEEP_MAX_IOU, "the number of IoU thresholds must be in [1, 256]");
    AMPIS_REQUIRE(d_ws && h_ws && need_bytes && pairs_found && totals && seg_totals && iou_thresh, "null pointer");
    AMPIS_REQUIRE(((uintptr_t)d_ws & 255u) == 0, "device workspace must be 256-byte aligned");
    for (int32_t j = 0; j < n_iou; j++)
        AMPIS_REQUIRE(iou_thresh[j] >= 0.0 && (j == 0 || iou_thresh[j] >= iou_thresh[j - 1]),
                      "IoU thresholds must be sorted ascending and not negative or NaN");
    const int64_t KT3 = 3 * (int64_t)n_levels * n_iou, NI = n_images;
    *pairs_found = 0;
    for (int64_t t = 0; t < KT3; t++) totals[t] = seg_totals[t] = 0;
    if (n_images == 0) return AMPIS_OK;
    AMPIS_REQUIRE(n_rows && n_cols, "null pointer");
    int64_t n_pred = 0;
    for (int32_t g = 0; g < n_images; g++) {
        AMPIS_REQUIRE(n_cols[g] <= AMPIS_SWEEP_MAX_PREDS, "more than 32768 predictions in one image");
        n_pred += n_cols[g] > 0 ? n_cols[g] : 0;
    }
    AMPIS_REQUIRE(levels || n_pred == 0, "null pointer");
    for (int64_t p = 0; p < n_pred; p++) AMPIS_REQUIRE(levels[p] <= n_levels, "prediction level above n_levels");
    if (counts) for (int64_t t = 0; t < KT3 * NI; t++) counts[t] = 0;
    if (seg_sums) for (int64_t t = 0; t < KT3 * NI; t++) seg_sums[t] = 0;
    const ImagesIn in{str_ptr, str_len, n_images, n_rows, n_cols, h, w, AMPIS_MODE_IOU, flags, d_ws, d_ws_bytes, h_ws,
                      h_ws_bytes, false, nullptr, nullptr, nullptr, nullptr, nullptr, status, nullptr, need_bytes, stream};
    ImagesExtra x;
    x.up[0] = iou_thresh;
    x.up_bytes[0] = 8 * (int64_t)n_iou;
    x.up[1] = levels;
    x.up_bytes[1] = 2 * n_pred;
    x.dl_bytes = 16 * KT3;                                                     // totals, then seg totals
    const int64_t counts_bytes = counts ? 4 * KT3 * NI : 0, seg_bytes = seg_sums ? 8 * KT3 * NI : 0;
    x.dev_bytes = seg_bytes + 256 + counts_bytes;
    ImagesRun r;
    int rc = images_front(in, x, -1.0, r);
    if (rc != AMPIS_OK || r.n == 0) return rc;
    uint8_t *H = r.H, *D = r.D;
    const int64_t o_totals = x.dl_off, o_segtot = x.dl_off + 8 * KT3;
    const int64_t d_seg = x.dev_off, d_counts = x.dev_off + ((seg_bytes + 255) & ~(int64_t)255);
    cudaError_t e = cudaMemsetAsync(D + o_totals, 0, (size_t)(16 * KT3), r.st);
    // rows without candidate pairs: when the join did not run, no row has any
    if (e == cudaSuccess && !r.have_rows && r.R > 0) e = cudaMemsetAsync(D + r.p_cnt, 0, (size_t)(4 * r.R), r.st);
    if (e != cudaSuccess) { ampis_set_error("memset: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }
    rc = ampis_sweep_counts((const uint32_t *)(D + r.o_area), (const int32_t *)(D + r.x_rowmask),
                            (const int32_t *)(D + r.x_rowgrp), r.have_rows ? (int32_t)r.R : 0,
                            (const int32_t *)(D + r.x_grb), (const int32_t *)(D + r.x_grc),
                            (const int32_t *)(D + r.x_gcb), (const int32_t *)(D + r.x_gcc), n_images, r.max_cols,
                            (const int32_t *)(D + r.p_ab), (const uint32_t *)(D + r.p_inter),
                            (const int64_t *)(D + r.p_off), (const int32_t *)(D + r.p_cnt),
                            (const uint16_t *)(D + x.up_off[1]), n_levels, (const double *)(D + x.up_off[0]), n_iou,
                            D + r.p_desc, counts ? (int32_t *)(D + d_counts) : nullptr,
                            seg_sums ? (int64_t *)(D + d_seg) : nullptr, (int64_t *)(D + o_totals),
                            (int64_t *)(D + o_segtot), stream);
    if (rc != AMPIS_OK) return rc;
    int32_t crowded = 0;
    rc = images_back(in, r, pairs_found, &crowded);
    if (rc != AMPIS_OK) return rc;
    // the per-image cells go straight into the caller's arrays once everything is known to have fit: they can be
    // hundreds of MB, too much to stage in the pinned workspace (pageable destinations make these copies blocking)
    if (counts) e = cudaMemcpyAsync(counts, D + d_counts, (size_t)counts_bytes, cudaMemcpyDeviceToHost, r.st);
    if (e == cudaSuccess && seg_sums) e = cudaMemcpyAsync(seg_sums, D + d_seg, (size_t)seg_bytes, cudaMemcpyDeviceToHost, r.st);
    if (e == cudaSuccess && (counts || seg_sums)) e = cudaStreamSynchronize(r.st);
    if (e != cudaSuccess) { ampis_set_error("download: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }
    memcpy(totals, H + o_totals, (size_t)(8 * KT3));
    memcpy(seg_totals, H + o_segtot, (size_t)(8 * KT3));
    return AMPIS_OK;
}
