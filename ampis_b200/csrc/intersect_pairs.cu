// Intersection rows over AMPIS_LAYOUT_CROP tables as a spatial JOIN in three flat passes (same outputs as
// intersect_rows_grid_kernel / intersect_rows_crop_kernel: analyze.py:149-164 / powder.py:80-86 semantics, see
// intersect.cu), instead of one kernel that walks cells, entries, candidates and window words row by row.
//
// Why: ncu on the grid rows kernel (profiles/kernels_r01p.md) showed 30 M warp instructions per 91 C2 images for
// ~90 k candidate pairs -- a hundred times the AND+popc work itself -- at 34 % issue utilisation: every row ran the
// dependent chain row -> cells -> entries -> window offsets -> window words on its own eight lanes, with half of the
// lanes of a warp idle on average.  Here each link of the chain is its own pass over a flat array, so every pass
// is short straight-line code at full occupancy:
//
//   pairs_from_grid_kernel   one THREAD per row mask: walks the grid cells of the row's box (the grid of the image's
//       column masks, built by grid_build_kernel), tests the boxes stored with the entries -- rleIou's bbIou
//       pre-pass -- and appends the candidate pairs (row mask id, column mask id).  The pairs of a row are contiguous:
//       counts are scanned over the warp and the warp reserves its range with one atomicAdd.
//   pair_intersect_flat_kernel   a warp per eight consecutive pairs, lanes over their concatenated overlap columns:
//       popcount(A & B) per column, per-pair sums by a segmented warp scan.  (pair_intersect_kernel, eight lanes per
//       pair and the whole warp for large overlaps, is the first form of the pass: AMPIS_PI_FLAT=0.)
//   rows_from_pairs_kernel   one thread per row: IoU / overlap score of its pairs, first arg-max (ties broken on the
//       column index, so the order of a row's pairs does not matter), dense matrix cells and sparse triplets.
//
// Either side of a pair may be an INTERVAL window (one word per column, AMPIS_WIN_INTERVALS; rle_flat.cu).  Its
// descriptor side then reads PD_IV | first band of the overlap instead of the words per column, and its word offset
// points at the first overlap column.  An interval x interval column is two loads and a closed form; an interval x
// bitmap column turns the interval into bands on the fly.  Only pair_intersect_flat_kernel reads interval windows.
#include <algorithm>
#include <cstdlib>
#include "common.cuh"

#define PJ_GR_N 32                       // cells per axis of the column grid (= GR_N of intersect_grid.cu)
#define PJ_GR_CELLS (PJ_GR_N * PJ_GR_N)
#define PJ_THREADS 128
#define PJ_KEEP 6                        // candidates of a row kept in registers between counting and writing
#define PI_BIG 1024u                     // overlap words from which a pair gets the whole warp

__device__ __forceinline__ int pj_cell_of(int v, int shift) { return min(v >> shift, PJ_GR_N - 1); }

// everything pair_intersect_kernel needs to know about a candidate pair, formed once by the thread that found it:
// the first word of the overlap in either window (word offsets into the arena), the words per column of either
// window, and the size of the overlap (columns x 32-row bands)
struct __align__(16) PairDesc {
    i64 a_word, b_word;
    u32 rn, cn, nw, ncols;
};
#define PD_IV 0x80000000u                // rn / cn flag: that side is an interval window; the low bits = first band

// the descriptor of the pair (row mask rm with box rb at word a_base, column mask cm with box cbx): overlap of the two
// windows (crop_common.cuh: overlap_of) as word offsets.  ia / ib: the side is an interval window
__device__ __forceinline__ PairDesc pair_desc_of(i64 a_base, int4 rb, bool ia, i64 b_base, int4 cbx, bool ib)
{
    const u32 xa = (u32)max(rb.x, cbx.x), xb = (u32)min(rb.z, cbx.z);
    const u32 rw0 = (u32)rb.y >> 5, rw1 = (u32)rb.w >> 5, cw0 = (u32)cbx.y >> 5, cw1 = (u32)cbx.w >> 5;
    const u32 wa = max(rw0, cw0), wb = min(rw1, cw1);
    PairDesc d;
    d.rn = ia ? PD_IV | wa : rw1 - rw0 + 1u;
    d.cn = ib ? PD_IV | wa : cw1 - cw0 + 1u;
    d.nw = wb - wa + 1u;
    d.ncols = xb - xa + 1u;
    d.a_word = a_base + (ia ? (i64)(xa - (u32)rb.x) : (i64)(xa - (u32)rb.x) * d.rn + (wa - rw0));
    d.b_word = b_base + (ib ? (i64)(xa - (u32)cbx.x) : (i64)(xa - (u32)cbx.x) * d.cn + (wa - cw0));
    return d;
}

struct PairJoinArgs {
    const i64 *bits_off;
    const uint2 *reg;                    // NULL: every window is a bitmap
    PairDesc *pair_desc;
    const int4 *bbox;
    const u32 *area;
    const int *row_mask, *row_grp;
    int n_rows;
    const int *grp_col_begin, *grp_col_count;
    const int *grp_shift;
    const i64 *cell_off;
    const int *entries;
    const int4 *entry_bbox;
    i64 grid_capacity;
    int2 *pair_ab;
    i64 pair_capacity;
    i64 *row_pair_off;
    int *row_pair_cnt;
    unsigned long long *pair_count;
};

// walks the candidates of one row: emit(k) for every column k (index inside the group) whose box overlaps rb
template <class F>
__device__ __forceinline__ void pj_walk(const PairJoinArgs &p, int g, const int4 rb, F emit)
{
    const int s = p.grp_shift[g];
    const i64 *off = p.cell_off + (i64)g * (PJ_GR_CELLS + 1);
    const int cx0 = pj_cell_of(rb.x, s), cx1 = pj_cell_of(rb.z, s), cy0 = pj_cell_of(rb.y, s), cy1 = pj_cell_of(rb.w, s);
    for (int cy = cy0; cy <= cy1; cy++) {
        // the cells of one grid row are consecutive: one entry range per grid row of the box
        const i64 e0 = off[cy * PJ_GR_N + cx0], e1 = off[cy * PJ_GR_N + cx1 + 1];
        for (i64 e = e0; e < e1 && e < p.grid_capacity; e++) {
            const int4 b = __ldg(p.entry_bbox + e);
            if (b.x > rb.z || b.z < rb.x || b.y > rb.w || b.w < rb.y) continue;
            // a column registered in several cells is taken once: in the cell that holds the top-left corner of
            // the overlap of the two boxes, i.e. grid row max(cy0, cell(b.y)) and, inside it, the entry that
            // lies in the range of cell max(cx0, cell(b.x))
            if (max(cy0, pj_cell_of(b.y, s)) != cy) continue;
            const int bx = max(cx0, pj_cell_of(b.x, s));
            if (e < off[cy * PJ_GR_N + bx] || e >= off[cy * PJ_GR_N + bx + 1]) continue;
            emit(__ldg(p.entries + e), b);
        }
    }
}

__global__ void __launch_bounds__(PJ_THREADS)
pairs_from_grid_kernel(const PairJoinArgs p)
{
    const int r = blockIdx.x * PJ_THREADS + threadIdx.x;
    const u32 lane = lane_id();
    const bool valid = r < p.n_rows;
    int g = 0, rm = 0, cb = 0;
    int4 rb = make_int4(0, 0, -1, -1);
    bool active = false;
    if (valid) {
        rm = p.row_mask[r];
        g = p.row_grp[r];
        rb = p.bbox[rm];
        cb = p.grp_col_begin[g];
        active = rb.z >= rb.x && p.area[rm] != 0u && p.grp_col_count[g] > 0;
    }
    int cnt = 0;
    int keep[PJ_KEEP];
#pragma unroll
    for (int i = 0; i < PJ_KEEP; i++) keep[i] = 0;
    if (active)
        pj_walk(p, g, rb, [&](int k, const int4) {
#pragma unroll
            for (int i = 0; i < PJ_KEEP; i++)
                if (cnt == i) keep[i] = k;
            cnt++;
        });
    // the warp's pairs are one contiguous range, row after row
    u32 incl = (u32)cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, incl, d);
        if ((int)lane >= d) incl += t;
    }
    const u32 total = __shfl_sync(0xffffffffu, incl, 31);
    unsigned long long base = 0;
    if (lane == 0 && total) base = atomicAdd(p.pair_count, (unsigned long long)total);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (!valid) return;
    const i64 first = (i64)base + (incl - (u32)cnt);
    const bool room = first + cnt <= p.pair_capacity;        // otherwise the caller retries with a larger list
    p.row_pair_off[r] = first;
    p.row_pair_cnt[r] = room ? cnt : 0;
    if (!room || cnt == 0) return;
    const i64 a_base = p.bits_off[rm] * 4;
    const bool ia = p.reg && (p.reg[rm].x & AMPIS_WIN_INTERVALS);
    auto put = [&](i64 q, int k, const int4 cbx) {
        const int cm = cb + k;
        p.pair_ab[q] = make_int2(rm, cm);
        p.pair_desc[q] = pair_desc_of(a_base, rb, ia, __ldg(p.bits_off + cm) * 4, cbx,
                                      p.reg && (__ldg(&p.reg[cm].x) & AMPIS_WIN_INTERVALS));
    };
    if (cnt <= PJ_KEEP) {
#pragma unroll
        for (int i = 0; i < PJ_KEEP; i++)
            if (i < cnt) put(first + i, keep[i], __ldg(p.bbox + cb + keep[i]));
    } else {
        int w = 0;
        pj_walk(p, g, rb, [&](int k, const int4 b) { put(first + w, k, b); w++; });
    }
}

// The same pass with EIGHT lanes per row (four rows per warp): the lanes test the entries of the row's cells eight at
// a time, so a row's walk is a few load latencies instead of one per entry, and the descriptors of its candidates are
// formed by different lanes at once.  (A row's pairs come out in no particular order: the row pass breaks ties on the
// column index.)
#define PJ8_ROWS (PJ_THREADS / 8)
#define PJ8_KEEP 2

template <class F>
__device__ __forceinline__ void pj_walk8(const PairJoinArgs &p, int g, const int4 rb, u32 t, F emit)
{
    const int s = p.grp_shift[g];
    const i64 *off = p.cell_off + (i64)g * (PJ_GR_CELLS + 1);
    const int cx0 = pj_cell_of(rb.x, s), cx1 = pj_cell_of(rb.z, s), cy0 = pj_cell_of(rb.y, s), cy1 = pj_cell_of(rb.w, s);
    for (int cy = cy0; cy <= cy1; cy++) {
        const i64 e0 = off[cy * PJ_GR_N + cx0], e1 = min(off[cy * PJ_GR_N + cx1 + 1], p.grid_capacity);
        for (i64 e = e0 + t; e < e1; e += 8) {
            const int4 b = __ldg(p.entry_bbox + e);
            if (b.x > rb.z || b.z < rb.x || b.y > rb.w || b.w < rb.y) continue;
            if (max(cy0, pj_cell_of(b.y, s)) != cy) continue;          // taken once: see pj_walk
            const int bx = max(cx0, pj_cell_of(b.x, s));
            if (e < off[cy * PJ_GR_N + bx] || e >= off[cy * PJ_GR_N + bx + 1]) continue;
            emit(__ldg(p.entries + e), b);
        }
    }
}

__global__ void __launch_bounds__(PJ_THREADS)
pairs_from_grid8_kernel(const PairJoinArgs p)
{
    const u32 lane = lane_id(), t = lane & 7u, tile = lane >> 3;
    const int r = blockIdx.x * PJ8_ROWS + (int)(threadIdx.x >> 3);
    const bool valid = r < p.n_rows;
    int g = 0, rm = 0, cb = 0;
    int4 rb = make_int4(0, 0, -1, -1);
    bool active = false;
    if (valid) {
        rm = p.row_mask[r];
        g = p.row_grp[r];
        rb = p.bbox[rm];
        cb = p.grp_col_begin[g];
        active = rb.z >= rb.x && p.area[rm] != 0u && p.grp_col_count[g] > 0;
    }
    int cnt = 0, k0 = 0, k1 = 0;                      // my candidates of the row (the first two kept)
    if (active)
        pj_walk8(p, g, rb, t, [&](int k, const int4) {
            if (cnt == 0) k0 = k;
            else if (cnt == 1) k1 = k;
            cnt++;
        });
    u32 incl = (u32)cnt;                              // prefix over the lanes of the row
#pragma unroll
    for (int d = 1; d < 8; d <<= 1) {
        const u32 v = __shfl_up_sync(0xffffffffu, incl, d, 8);
        if ((int)t >= d) incl += v;
    }
    const u32 row_cnt = __shfl_sync(0xffffffffu, incl, 7, 8);
    // the warp's pairs are one contiguous range, row after row
    const u32 c0 = __shfl_sync(0xffffffffu, row_cnt, 0), c1 = __shfl_sync(0xffffffffu, row_cnt, 8),
              c2 = __shfl_sync(0xffffffffu, row_cnt, 16), c3 = __shfl_sync(0xffffffffu, row_cnt, 24);
    const u32 total = c0 + c1 + c2 + c3;
    const u32 before = (tile > 0u ? c0 : 0u) + (tile > 1u ? c1 : 0u) + (tile > 2u ? c2 : 0u);
    unsigned long long base = 0;
    if (lane == 0 && total) base = atomicAdd(p.pair_count, (unsigned long long)total);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (!valid) return;
    const i64 first = (i64)base + before;
    const bool room = first + row_cnt <= p.pair_capacity;      // otherwise the caller retries with a larger list
    if (t == 0u) {
        p.row_pair_off[r] = first;
        p.row_pair_cnt[r] = room ? (int)row_cnt : 0;
    }
    if (!room || cnt == 0) return;
    const i64 mine = first + (incl - (u32)cnt);
    const i64 a_base = p.bits_off[rm] * 4;
    const bool ia = p.reg && (p.reg[rm].x & AMPIS_WIN_INTERVALS);
    auto put = [&](i64 q, int k, const int4 cbx) {
        const int cm = cb + k;
        p.pair_ab[q] = make_int2(rm, cm);
        p.pair_desc[q] = pair_desc_of(a_base, rb, ia, __ldg(p.bits_off + cm) * 4, cbx,
                                      p.reg && (__ldg(&p.reg[cm].x) & AMPIS_WIN_INTERVALS));
    };
    if (cnt <= PJ8_KEEP) {
        put(mine, k0, __ldg(p.bbox + cb + k0));
        if (cnt == 2) put(mine + 1, k1, __ldg(p.bbox + cb + k1));
    } else {
        int w = 0;
        pj_walk8(p, g, rb, t, [&](int k, const int4 b) { put(mine + w, k, b); w++; });
    }
}

// popcount(A & B) over an overlap of ncols columns x nw bands, by `n_lanes` lanes (lane index t): lanes take
// columns (and walk the few bands of a column) unless the overlap is taller than wide in words, then they take bands
__device__ __forceinline__ u32 desc_popc(const u32 *__restrict__ words, const PairDesc &d, u32 t, u32 n_lanes)
{
    const u32 *A = words + d.a_word, *B = words + d.b_word;
    u32 acc = 0;
    if (d.nw <= d.ncols) {
        // two columns of a lane at a time, all their loads issued before the first popcount: the kernel is bound by
        // the latency of these loads, not by lanes
        for (u32 dx = t; dx < d.ncols; dx += 2 * n_lanes) {
            const u32 dx2 = dx + n_lanes;
            const bool two = dx2 < d.ncols;
            const u32 *a0 = A + dx * d.rn, *b0 = B + dx * d.cn;
            const u32 *a1 = two ? A + dx2 * d.rn : a0, *b1 = two ? B + dx2 * d.cn : b0;
#pragma unroll 2
            for (u32 dw = 0; dw < d.nw; dw++) {
                const u32 x0 = __ldg(a0 + dw), y0 = __ldg(b0 + dw), x1 = __ldg(a1 + dw), y1 = __ldg(b1 + dw);
                acc += __popc(x0 & y0) + (two ? __popc(x1 & y1) : 0u);
            }
        }
    } else {
        for (u32 dx = 0; dx < d.ncols; dx++) {
            const u32 *a = A + dx * d.rn, *b = B + dx * d.cn;
#pragma unroll 4
            for (u32 dw = t; dw < d.nw; dw += n_lanes) acc += __popc(__ldg(a + dw) & __ldg(b + dw));
        }
    }
    return acc;
}

__global__ void __launch_bounds__(256, 6)
pair_intersect_kernel(const u32 *__restrict__ words, const PairDesc *__restrict__ pair_desc,
                      u32 *__restrict__ pair_inter, const unsigned long long *__restrict__ pair_count,
                      i64 pair_capacity)
{
    const u32 lane = lane_id(), sub = lane >> 3, t = lane & 7u;
    const i64 n = (i64)*pair_count;
    if (n > pair_capacity) return;          // the list overflowed (rows without room wrote nothing): the caller retries
    const i64 stride = (i64)gridDim.x * (blockDim.x >> 5) * 4;
    for (i64 q0 = ((i64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 4; q0 < n; q0 += stride) {
        const i64 q = q0 + sub;
        const bool have = q < n;
        PairDesc d;
        d.nw = d.ncols = 0;
        if (have) {
            const uint4 *src = reinterpret_cast<const uint4 *>(pair_desc + q);
            const uint4 lo = __ldg(src), hi = __ldg(src + 1);
            d.a_word = (i64)(((u64)lo.y << 32) | lo.x);
            d.b_word = (i64)(((u64)lo.w << 32) | lo.z);
            d.rn = hi.x; d.cn = hi.y; d.nw = hi.z; d.ncols = hi.w;
        }
        const bool big = have && (u64)d.nw * d.ncols >= PI_BIG;
        u32 v = (have && !big) ? desc_popc(words, d, t, 8) : 0u;
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        u32 bigs = __ballot_sync(0xffffffffu, big && t == 0u);
        while (bigs) {                                        // large overlaps: all 32 lanes on one pair at a time
            const int src = __ffs(bigs) - 1;
            bigs &= bigs - 1u;
            PairDesc b;
            b.a_word = __shfl_sync(0xffffffffu, d.a_word, src);
            b.b_word = __shfl_sync(0xffffffffu, d.b_word, src);
            b.rn = __shfl_sync(0xffffffffu, d.rn, src);
            b.cn = __shfl_sync(0xffffffffu, d.cn, src);
            b.nw = __shfl_sync(0xffffffffu, d.nw, src);
            b.ncols = __shfl_sync(0xffffffffu, d.ncols, src);
            const u32 vb = warp_sum(desc_popc(words, b, lane, 32));
            if ((int)sub == (src >> 3)) v = vb;
        }
        if (have && t == 0u) pair_inter[q] = v;
    }
}

// The same pass FLAT: a warp takes eight consecutive pairs and spreads its lanes over their concatenated overlap columns
// (a column of more than four bands is several items), so every lane has a column whatever the sizes of the eight
// overlaps are, and the per-pair sums are one segmented warp scan per 32 items.  With eight lanes per pair the four
// pairs of a warp ran in lockstep to the trip count of the largest, 2/3 of the lanes busy on average.
#define PF_PAIRS 8
#define PF_WORDS 4u
// interval x interval: columns per item (four loads of a lane in flight; four columns spill at 40 registers)
#define PF_IV_COLS 2u

struct __align__(16) PfWarp {
    uint4 lo[PF_PAIRS], hi[PF_PAIRS];       // the descriptors of the batch
    u32 start[PF_PAIRS + 1];                // first item of every pair
    u32 nsub[PF_PAIRS];                     // items per overlap column (0: PF_IV_COLS columns per item)
    u32 acc[PF_PAIRS];
};

// U = passes of 32 items a warp has in flight (their loads are issued before the first popcount).  Only U = 1 (the
// default) reads interval windows: with them the two-pass form spills (72 bytes) at the 40 registers of 6 CTAs per SM
template <int U>
__global__ void __launch_bounds__(256, 6)
pair_intersect_flat_kernel(const u32 *__restrict__ words, const PairDesc *__restrict__ pair_desc,
                           u32 *__restrict__ pair_inter, const unsigned long long *__restrict__ pair_count,
                           i64 pair_capacity)
{
    __shared__ PfWarp s_w[8];
    PfWarp &S = s_w[threadIdx.x >> 5];
    const u32 lane = lane_id();
    const i64 n = (i64)*pair_count;
    if (n > pair_capacity) return;          // the list overflowed (rows without room wrote nothing): the caller retries
    const i64 stride = (i64)gridDim.x * (blockDim.x >> 5) * PF_PAIRS;
    // batches are taken from the END of the list: the windows of the last images were written last by the decode and
    // are the ones still in L2
    const i64 n_batches = (n + PF_PAIRS - 1) / PF_PAIRS;
    for (i64 bi = (i64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); bi < n_batches; bi += stride / PF_PAIRS) {
        const i64 q0 = (n_batches - 1 - bi) * PF_PAIRS;
        u32 items = 0;
        if (lane < PF_PAIRS) {
            uint4 lo = make_uint4(0u, 0u, 0u, 0u), hi = make_uint4(0u, 0u, 0u, 0u);
            u32 ns = 1u;
            if (q0 + lane < n) {
                const uint4 *src = reinterpret_cast<const uint4 *>(pair_desc + q0 + lane);
                lo = __ldg(src);
                hi = __ldg(src + 1);
                // interval x interval: PF_IV_COLS columns per item whatever the height
                const bool ii = U == 1 && (hi.x & hi.y & PD_IV);
                ns = ii ? 0u : max((hi.z + PF_WORDS - 1u) / PF_WORDS, 1u);
                items = hi.z ? (ii ? (hi.w + PF_IV_COLS - 1u) / PF_IV_COLS : hi.w * ns) : 0u;
            }
            S.lo[lane] = lo; S.hi[lane] = hi; S.nsub[lane] = ns; S.acc[lane] = 0u;
        }
        u32 incl = items;
#pragma unroll
        for (int d = 1; d < PF_PAIRS; d <<= 1) {
            const u32 t = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)lane >= d) incl += t;
        }
        if (lane < PF_PAIRS) S.start[lane] = incl - items;
        if (lane == PF_PAIRS - 1) S.start[PF_PAIRS] = incl;
        __syncwarp();
        const u32 T = S.start[PF_PAIRS];
        const u32 s1 = S.start[1], s2 = S.start[2], s3 = S.start[3], s4 = S.start[4], s5 = S.start[5], s6 = S.start[6],
                  s7 = S.start[7];
        for (u32 c0 = 0; c0 < T; c0 += 32 * U) {
            u32 v[U], j[U], it[U], x0[U], x1[U], wa[U], wb[U], iv[U];
            const u32 *pa[U], *pb[U];
            bool ok[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const u32 c = c0 + 32u * u + lane;
                ok[u] = c < T;
                v[u] = 0u; j[u] = 0u; it[u] = 0u; x0[u] = 0u; x1[u] = 0u; wa[u] = 0u; wb[u] = 0u; iv[u] = 0u;
                pa[u] = pb[u] = words;
                if (ok[u]) {
                    j[u] = (u32)(c >= s1) + (u32)(c >= s2) + (u32)(c >= s3) + (u32)(c >= s4) + (u32)(c >= s5) +
                           (u32)(c >= s6) + (u32)(c >= s7);
                    it[u] = c - S.start[j[u]];
                    const uint4 lo = S.lo[j[u]], hi = S.hi[j[u]];
                    const u32 ns = S.nsub[j[u]];
                    u32 dx = it[u], w0 = 0u, w1 = hi.z;
                    if (ns > 1u) {
                        dx = it[u] / ns;
                        w0 = (it[u] - dx * ns) * PF_WORDS;
                        w1 = min(hi.z, w0 + PF_WORDS);
                    } else if (ns == 0u) {
                        dx = it[u] * PF_IV_COLS;
                    }
                    const bool ia = U == 1 && (hi.x & PD_IV), ib = U == 1 && (hi.y & PD_IV);
                    pa[u] = words + (i64)(((u64)lo.y << 32) | lo.x) + (ia ? (i64)dx : (i64)dx * hi.x + w0);
                    pb[u] = words + (i64)(((u64)lo.w << 32) | lo.z) + (ib ? (i64)dx : (i64)dx * hi.y + w0);
                    wa[u] = w0; wb[u] = w1;
                    if (!(ia | ib)) {
                        // the first two bands of the column (most overlaps have one or two): all loads of all passes
                        // in flight
                        x0[u] = __ldg(pa[u]) & __ldg(pb[u]);
                        if (w0 + 1u < w1) x1[u] = __ldg(pa[u] + 1) & __ldg(pb[u] + 1);
                    } else if (ia & ib) {
                        const u32 left = hi.w - dx;
                        u32 qa[PF_IV_COLS], qb[PF_IV_COLS];
#pragma unroll
                        for (u32 k = 0; k < PF_IV_COLS; k++) {
                            qa[k] = k < left ? __ldg(pa[u] + k) : 0u;         // a zero word is an empty column
                            qb[k] = k < left ? __ldg(pb[u] + k) : 0u;
                        }
#pragma unroll
                        for (u32 k = 0; k < PF_IV_COLS; k++) iv[u] += interval_overlap(qa[k], qb[k]);
                        wb[u] = w0;
                    } else {
                        // interval x bitmap: the interval word as bands (wa..) of the overlap, ANDed with the bitmap's
                        const u32 v = __ldg(ia ? pa[u] : pb[u]), y0 = ((ia ? hi.x : hi.y) & ~PD_IV) * 32u;
                        const u32 *bm = ia ? pb[u] : pa[u];
                        for (u32 w = w0; w < w1; w++)
                            iv[u] += __popc(interval_band(v, y0 + 32u * w) & __ldg(bm + (w - w0)));
                        wb[u] = w0;
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                v[u] = __popc(x0[u]) + __popc(x1[u]) + iv[u];
                for (u32 w = wa[u] + 2u; w < wb[u]; w++) v[u] += __popc(__ldg(pa[u] + (w - wa[u])) & __ldg(pb[u] + (w - wa[u])));
                // sums per pair: the lanes of a pair are contiguous
                const u32 reach = ok[u] ? min(lane, it[u]) : 0u;
#pragma unroll
                for (u32 d = 1; d < 32; d <<= 1) {
                    const u32 t = __shfl_up_sync(0xffffffffu, v[u], d);
                    if (d <= reach) v[u] += t;
                }
                const u32 c = c0 + 32u * u + lane;
                if (ok[u] && (lane == 31u || c + 1u == S.start[j[u] + 1])) atomicAdd(&S.acc[j[u]], v[u]);
            }
        }
        __syncwarp();
        if (lane < PF_PAIRS && q0 + lane < n) pair_inter[q0 + lane] = S.acc[lane];
        __syncwarp();
    }
}

struct PairRowArgs {
    const u32 *area;
    const int *row_mask, *row_grp;
    int n_rows;
    const int *grp_row_begin, *grp_col_begin, *grp_col_count;
    const int2 *pair_ab;
    const u32 *pair_inter;
    const i64 *row_pair_off;
    const int *row_pair_cnt;
    const i64 *grp_imat_off;
    int *imat;
    int *best_col;
    u32 *best_inter;
    double *best_score;
    int *coo_row, *coo_col;
    u32 *coo_inter;
    i64 coo_capacity;
    unsigned long long *coo_count;
};

template <int MODE>
__global__ void __launch_bounds__(PJ_THREADS)
rows_from_pairs_kernel(const PairRowArgs p)
{
    const int r = blockIdx.x * PJ_THREADS + threadIdx.x;
    if (r >= p.n_rows) return;
    const int g = p.row_grp[r];
    const int cb = p.grp_col_begin[g], P = p.grp_col_count[g];
    const u32 ra = p.area[p.row_mask[r]];
    const i64 first = p.row_pair_off[r];
    const int cnt = p.row_pair_cnt[r];
    int *irow = nullptr;
    if (p.imat && p.grp_imat_off && p.grp_imat_off[g] >= 0)
        irow = p.imat + p.grp_imat_off[g] + (i64)(r - p.grp_row_begin[g]) * P;
    double best_s = 0.0;
    u32 best_i = 0;
    int best_c = MODE == AMPIS_MODE_IOU ? -1 : (P > 0 ? 0 : -1);
    // four pairs at a time: their intersections, column ids and column areas are requested before any is looked at
    // (the loop was one dependent chain of three loads per pair)
    for (int i0 = 0; i0 < cnt; i0 += 4) {
        u32 in4[4], ca4[4];
        int cm4[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const bool on = i0 + u < cnt;
            in4[u] = on ? __ldg(p.pair_inter + first + i0 + u) : 0u;
            cm4[u] = on ? __ldg(p.pair_ab + first + i0 + u).y : cb;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) ca4[u] = (MODE == AMPIS_MODE_IOU && in4[u]) ? __ldg(p.area + cm4[u]) : 0u;
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const u32 inter = in4[u];
            if (!inter) continue;
            const int k = cm4[u] - cb;
            if (irow) irow[k] = (int)inter;
            if (p.coo_count) {
                const unsigned long long pos = atomicAdd(p.coo_count, 1ull);
                if ((i64)pos < p.coo_capacity) { p.coo_row[pos] = r; p.coo_col[pos] = k; p.coo_inter[pos] = inter; }
            }
            if (MODE == AMPIS_MODE_IOU) {
                const double s = pair_iou(inter, ra, ca4[u]);
                if (score_beats(s, k, best_s, best_c)) { best_s = s; best_i = inter; best_c = k; }
            } else {
                if (inter > best_i || (inter == best_i && (unsigned)k < (unsigned)best_c)) { best_i = inter; best_c = k; }
            }
        }
    }
    if (MODE == AMPIS_MODE_SAT) best_s = (double)best_i / (double)ra;   // 0/0 = NaN like numpy
    p.best_col[r] = best_c;
    p.best_inter[r] = best_i;
    p.best_score[r] = best_s;
}

// AMPIS_PI_FLAT: 1 (default) = lanes over the concatenated columns of eight pairs, 2 = the same with two passes in
// flight, 0 = eight lanes per pair (profiles/experiments_r02.md: 0.395 / 0.387 / 0.383 ms of rows per C2 step)
static int pi_flat()
{
    static const int flat = [] { const char *v = getenv("AMPIS_PI_FLAT"); return v ? atoi(v) : 1; }();
    return flat;
}

extern "C" int ampis_pairs_read_intervals(void) { return pi_flat() == 1; }

extern "C" int ampis_intersect_rows_pairs(const void *d_bits, const int64_t *d_bits_off, const uint32_t *d_reg,
                                          const int32_t *d_bbox,
                                          const uint32_t *d_area, const int32_t *d_row_mask, const int32_t *d_row_grp,
                                          int32_t n_rows, const int32_t *d_grp_row_begin,
                                          const int32_t *d_grp_col_begin, const int32_t *d_grp_col_count,
                                          const int32_t *d_grp_shift, const int64_t *d_cell_off,
                                          const int32_t *d_entries, const int32_t *d_entry_bbox, int64_t grid_capacity,
                                          int32_t *d_pair_ab, void *d_pair_desc, uint32_t *d_pair_inter,
                                          int64_t pair_capacity,
                                          int64_t *d_row_pair_off, int32_t *d_row_pair_cnt, uint64_t *d_pair_count,
                                          const int64_t *d_grp_imat_off, int32_t mode, int32_t *d_imat,
                                          int64_t imat_ints, int32_t *d_best_col, uint32_t *d_best_inter,
                                          double *d_best_score, int32_t *d_coo_row, int32_t *d_coo_col,
                                          uint32_t *d_coo_inter, int64_t coo_capacity, uint64_t *d_coo_count,
                                          void *zero_stream, void *stream)
{
    AMPIS_REQUIRE(n_rows >= 0 && pair_capacity >= 0 && grid_capacity >= 0 && imat_ints >= 0, "negative size");
    AMPIS_REQUIRE(mode == AMPIS_MODE_IOU || mode == AMPIS_MODE_SAT, "bad mode");
    AMPIS_REQUIRE(!d_reg || ampis_pairs_read_intervals(), "interval windows need the default pair pass (AMPIS_PI_FLAT=1)");
    if (n_rows == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_bits_off && d_bbox && d_area && d_row_mask && d_row_grp && d_grp_row_begin && d_grp_col_begin &&
                      d_grp_col_count && d_grp_shift && d_cell_off && d_row_pair_off && d_row_pair_cnt &&
                      d_pair_count && d_best_col && d_best_inter && d_best_score, "null pointer");
    AMPIS_REQUIRE((d_entries && d_entry_bbox) || grid_capacity == 0, "entries missing");
    AMPIS_REQUIRE((d_pair_ab && d_pair_desc && d_pair_inter) || pair_capacity == 0, "pair list missing");
    AMPIS_REQUIRE(((uintptr_t)d_pair_ab & 7u) == 0 && ((uintptr_t)d_pair_desc & 15u) == 0,
                  "pair list must be 8-byte aligned, pair descriptors 16-byte aligned");
    AMPIS_REQUIRE(!d_coo_count || (d_coo_row && d_coo_col && d_coo_inter && coo_capacity >= 0) || coo_capacity == 0,
                  "sparse output arrays missing");
    cudaStream_t st = as_stream(stream), zs = as_stream(zero_stream);
    cudaError_t e = cudaMemsetAsync(d_pair_count, 0, sizeof(uint64_t), st);
    // dense rows: zeros first, the row pass patches the non-zero cells.  With a zero_stream the fill runs beside the
    // join and the AND+popc pass (both bound by load latency, not by bandwidth) and the row pass waits for it
    const bool dense = d_imat && d_grp_imat_off && imat_ints > 0;
    const bool side = dense && zero_stream && zs != st;
    static thread_local cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    if (e == cudaSuccess && side) {
        if (!ev_fork) {
            e = cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaEventRecord(ev_fork, st);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(zs, ev_fork, 0);
        if (e == cudaSuccess) e = cudaMemsetAsync(d_imat, 0, (size_t)imat_ints * 4, zs);
        if (e == cudaSuccess) e = cudaEventRecord(ev_join, zs);
    } else if (e == cudaSuccess && dense) {
        e = cudaMemsetAsync(d_imat, 0, (size_t)imat_ints * 4, st);
    }
    if (e != cudaSuccess) { ampis_set_error("cudaMemsetAsync: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }
    PairJoinArgs j;
    j.bits_off = d_bits_off; j.reg = (const uint2 *)d_reg; j.pair_desc = (PairDesc *)d_pair_desc;
    j.bbox = (const int4 *)d_bbox; j.area = d_area; j.row_mask = d_row_mask; j.row_grp = d_row_grp; j.n_rows = n_rows;
    j.grp_col_begin = d_grp_col_begin; j.grp_col_count = d_grp_col_count; j.grp_shift = d_grp_shift;
    j.cell_off = d_cell_off; j.entries = d_entries; j.entry_bbox = (const int4 *)d_entry_bbox;
    j.grid_capacity = grid_capacity; j.pair_ab = (int2 *)d_pair_ab; j.pair_capacity = pair_capacity;
    j.row_pair_off = d_row_pair_off; j.row_pair_cnt = d_row_pair_cnt; j.pair_count = (unsigned long long *)d_pair_count;
    const unsigned row_blocks = (unsigned)((n_rows + PJ_THREADS - 1) / PJ_THREADS);
    // Lanes per row in the candidate walk.  A thread per row (default) is the cheaper form in instructions: C2 with
    // 500,000 rows per launch 0.385 against 0.418 ms of rows with eight lanes.  Eight lanes per row (AMPIS_PJ_LANES=8)
    // make the shorter chain of dependent loads: device-resident C3 (40,000 rows) 0.114 -> 0.087 ms -- but end to end,
    // with several calls in flight, the same C3 step went from 0.95 to 1.16 ms (eight times the threads compete with
    // the other calls' kernels), so it is not chosen automatically.
    static const int pj_lanes = [] { const char *v = getenv("AMPIS_PJ_LANES"); return v ? atoi(v) : 1; }();
    if (pj_lanes == 8)
        pairs_from_grid8_kernel<<<(unsigned)((n_rows + PJ8_ROWS - 1) / PJ8_ROWS), PJ_THREADS, 0, st>>>(j);
    else
        pairs_from_grid_kernel<<<row_blocks, PJ_THREADS, 0, st>>>(j);
    AMPIS_CHECK_LAUNCH("pairs_from_grid_kernel");
    if (pair_capacity > 0) {
        // the number of pairs is only known on the device: a grid that covers the capacity, at most ~8 waves
        i64 want = (pair_capacity + 31) / 32;                      // 8 warps x 4 pairs per CTA and trip
        const i64 cap = 148 * 8 * 8;
        if (want > cap) want = cap;
        const int flat = pi_flat();
        if (flat == 1)
            pair_intersect_flat_kernel<1><<<(unsigned)std::min<i64>((pair_capacity + 63) / 64, cap), 256, 0, st>>>(
                (const u32 *)d_bits, (const PairDesc *)d_pair_desc, d_pair_inter, (const unsigned long long *)d_pair_count,
                pair_capacity);
        else if (flat == 2)
            pair_intersect_flat_kernel<2><<<(unsigned)std::min<i64>((pair_capacity + 63) / 64, cap), 256, 0, st>>>(
                (const u32 *)d_bits, (const PairDesc *)d_pair_desc, d_pair_inter, (const unsigned long long *)d_pair_count,
                pair_capacity);
        else
            pair_intersect_kernel<<<(unsigned)want, 256, 0, st>>>((const u32 *)d_bits, (const PairDesc *)d_pair_desc,
                                                              d_pair_inter, (const unsigned long long *)d_pair_count,
                                                              pair_capacity);
        AMPIS_CHECK_LAUNCH("pair_intersect_kernel");
    }
    if (side) {
        e = cudaStreamWaitEvent(st, ev_join, 0);
        if (e != cudaSuccess) { ampis_set_error("cudaStreamWaitEvent: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }
    }
    PairRowArgs a;
    a.area = d_area; a.row_mask = d_row_mask; a.row_grp = d_row_grp; a.n_rows = n_rows;
    a.grp_row_begin = d_grp_row_begin; a.grp_col_begin = d_grp_col_begin; a.grp_col_count = d_grp_col_count;
    a.pair_ab = (const int2 *)d_pair_ab; a.pair_inter = d_pair_inter; a.row_pair_off = d_row_pair_off;
    a.row_pair_cnt = d_row_pair_cnt; a.grp_imat_off = d_grp_imat_off; a.imat = d_imat;
    a.best_col = d_best_col; a.best_inter = d_best_inter; a.best_score = d_best_score;
    a.coo_row = d_coo_row; a.coo_col = d_coo_col; a.coo_inter = d_coo_inter; a.coo_capacity = coo_capacity;
    a.coo_count = (unsigned long long *)d_coo_count;
    if (mode == AMPIS_MODE_IOU)
        rows_from_pairs_kernel<AMPIS_MODE_IOU><<<row_blocks, PJ_THREADS, 0, st>>>(a);
    else
        rows_from_pairs_kernel<AMPIS_MODE_SAT><<<row_blocks, PJ_THREADS, 0, st>>>(a);
    AMPIS_CHECK_LAUNCH("rows_from_pairs_kernel");
    return AMPIS_OK;
}
