// RLE -> bounding-box windows (AMPIS_LAYOUT_CROP), third generation: a warp decodes SEVERAL masks at once with
// its lanes spread over the concatenated run lists ("flat"), instead of a group of 8 / 16 / 32 lanes per mask.
//
// Same role and same outputs as rle_measure_paint_crop_kernel (rle_paint.cu): rleArea (structures.py:568,571;
// analyze.py:320-321; powder.py:264), the tight box extract_boxes reads off the decoded mask (data_utils.py:229-239)
// and rleDecode (structures.py:752,761) restricted to that box -- what every RLE.iou / RLE.merge call of
// analyze.py:158,315 and powder.py:82 decodes again and again in the reference.
//
// Why: ncu on the group-per-mask kernel (profiles/kernels_r01p.md) showed it bound by instruction issue at ~740
// warp instructions per mask.  Most of them were per-MASK fixed costs executed by a whole group (five shuffle
// reductions, the 60-instruction record store, arena reservation, tile zero-fill / copy-out loops with 1-2 trips)
// and passes in which half of the lanes had no run left (75 runs on 2 x 64 slots).  Here
//   * the unit of work is a PAIR (0-run, 1-run); the K masks a warp owns are laid end to end and taken in rounds of
//     at most FL_PAIR_CAP = 256 pairs = 32 lanes x 8;
//   * a round is measured in ONE pass: its pairs are staged in shared memory by coalesced lane-strided loads, then
//     every lane walks its own slice of 8 consecutive pairs in registers.  Run end positions come from a sequential
//     walk inside the slice and ONE segmented warp scan across the slices (segments = masks; 32-bit saturating
//     arithmetic, the "a mask starts here" flag in bit 31); area, first / last 1-pixel and row range are kept per
//     slice segment in registers and added to the mask with shared-memory atomics once per slice it touches.
//     (Before: one pair per lane, passes of 32 pairs, three segmented scans, ballots and a carry per pass -- about
//     half of the kernel's instructions.  Earlier still, a REDUX reduction per mask and pass.)
//   * the measure pass leaves, per pair, what the painter needs -- column and first / last row of the 1-run in one
//     64-bit word (runs that cross a column boundary keep start and length and take a slower path) -- and the
//     per-mask constants of the painter are ONE 128-bit word: no division, no box clipping in the paint loop;
//   * the per-mask records (area, box, span, region, status, arena offset) are formed by ONE lane per mask, all
//     masks of the warp in parallel, and the warp reserves arena space for all of them with a single atomicAdd;
//   * the windows of all K masks are assembled in one shared-memory tile that is contiguous in the arena, so the
//     copy-out is a straight run of 128-bit stores;
//   * the grid is one wave and every warp strides over the groups of K masks (persistent warps).
// Masks that do not fit the per-warp budgets (more than FL_PAIR_CAP pairs, window larger than the tile, frame of
// 2^31 pixels or more or taller than 65,536 rows) are appended to a list that rle_measure_paint_list_kernel (a warp
// per mask, any size; rle_paint.cu) works off in a second launch.
//
// Interval windows (IV = true; asked for by callers whose table only goes to the pairs join, intersect_pairs.cu):
// a COLUMN-CONVEX mask -- every 1-run inside one column, no column with two 1-runs, as every particle blob of the
// synthetic data and most real particles are -- is stored as ONE word per box column, (first row ^ 0xffff) | last
// row << 16, so that a zero word is an empty column (AMPIS_WIN_INTERVALS in reg.x; common.cuh).  The measure pass
// tests the property per pair, without a scan: a pair after the first of its mask whose 0-run is shorter than the
// first row of its 1-run has the previous 1-run in the same column.  The painter then stores one word per 1-run
// instead of OR-ing bands.
#include <algorithm>
#include "common.cuh"
#include "rle_measure.cuh"

#define FL_WARPS 8
#define FL_CTAS_PER_SM 5
#define FL_KMAX 16              // masks per warp and round
#define FL_PAIR_CAP 256         // (0-run, 1-run) pairs per warp and round
#define FL_TILE_WORDS 512       // window words per warp and round
#define FL_SAT 0x7fffffffu      // positions saturate here; frames must be smaller
#define FL_HMAX 65536u          // rows of a column are kept in 16 bits; taller frames go to the fallback kernel
#define FL_SPAN 0x80000000u     // pair.x flag: the 1-run crosses a column boundary, pair = (start | FL_SPAN, length)
#define FL_HEAD 0x80000000u     // flag of a measure-scan value: a mask starts in the lane's slice

// What the measure pass leaves for the painter, one per (0-run, 1-run) pair:
//   1-run inside one column (every run of a blob):  x = column,           y = first row | last row << 16
//   1-run over several columns:                     x = start | FL_SPAN,  y = length
//   nothing to paint:                               x = 0,                y = 0x0000ffff (first row > last row)
#define FL_EMPTY make_uint2(0u, 0x0000ffffu)

struct __align__(16) FlatWarp {
    uint2 pair[FL_PAIR_CAP];
    u32 tile[FL_TILE_WORDS];
    uint4 geo[FL_KMAX];             // per mask of the warp: image height H, 2^32 / H, H * W, number of run counts
    uint4 win[FL_KMAX];             // per mask of the round: H, 2^32 / H, tile word of (column 0, band 0), bands per column
    const u32 *src[FL_KMAX];        // per mask of the warp: its first run count
    u32 pb[FL_KMAX + 1];            // first pair of every mask of the round
    u32 area[FL_KMAX], first[FL_KMAX], last[FL_KMAX], ymin[FL_KMAX], ymaxi[FL_KMAX], total[FL_KMAX];
    u32 convex[FL_KMAX];            // per mask of the round: column-convex so far (IV only)
    __align__(8) uint8_t mid[FL_PAIR_CAP];  // mask (index inside the round) of every pair: 8 per lane in one load
};

__device__ __forceinline__ u32 sat_add(u32 a, u32 b) { return min(a + b, FL_SAT); }

// where pair f of a round is kept in S.pair: bits 1-2 flipped by bits 4-5, so that the 16-byte chunks eight lanes
// read of their own 8-pair slices fall on distinct banks; 16 consecutive pairs stay a permutation of themselves
__device__ __forceinline__ u32 fl_swz(u32 f) { return f ^ ((f >> 3) & 6u); }

__device__ __forceinline__ u32 warp_incl_scan(u32 v, u32 lane)
{
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, v, d);
        if ((int)lane >= d) v += t;
    }
    return v;
}

__device__ __forceinline__ u32 div_by(u32 s, u32 d, u32 rcp)
{
    u32 q = __umulhi(s, rcp);
    if (s - q * d >= d) q++;
    return q;
}

// rows ys..yl (inclusive) of one window column whose band 0 is tile word idx (idx may have wrapped below zero: the
// sum with the band index is taken modulo 2^32)
__device__ __forceinline__ void paint_rows(u32 *tile, u32 idx, u32 ys, u32 yl)
{
    const u32 w0 = ys >> 5, w1 = yl >> 5;
    const u32 m0 = 0xffffffffu << (ys & 31u), m1 = 0xffffffffu >> (31u - (yl & 31u));
    if (w0 == w1) {
        atomicOr(&tile[idx + w0], m0 & m1);
    } else {
        atomicOr(&tile[idx + w0], m0);
#pragma unroll 1
        for (u32 w = w0 + 1u; w < w1; w++) tile[idx + w] = 0xffffffffu;
        atomicOr(&tile[idx + w1], m1);
    }
}

// Persistent: the grid is one wave (FL_CTAS_PER_SM CTAs per SM) and every warp strides over the groups of K masks,
// so no SM waits for the slowest warp of a CTA before it is given new work.
template <bool ZERO, bool IV>
__global__ void __launch_bounds__(FL_WARPS * 32, FL_CTAS_PER_SM)
rle_flat_crop_kernel(const u32 *__restrict__ cnt, const i64 *__restrict__ cnt_off, const int *__restrict__ cnt_len,
                     const u32 *__restrict__ hh, const u32 *__restrict__ ww, int n, int K,
                     u32 *__restrict__ area, int *__restrict__ bbox, u32 *__restrict__ span, u32 *__restrict__ reg,
                     i64 *__restrict__ bits_off, int *__restrict__ status, uint4 *__restrict__ bits, i64 capacity,
                     unsigned long long *__restrict__ cursor, int *__restrict__ big,
                     uint4 *__restrict__ zero, u32 zero_chunks, u32 zero_per_group)
{
    __shared__ FlatWarp s_warp[FL_WARPS];
    FlatWarp &S = s_warp[threadIdx.x >> 5];
    const u32 lane = lane_id();
    // 32-bit group counter (gw < n < 2^31, one wave of warps added): a 64-bit one spills in the interval variant
    const u32 nwarps = gridDim.x * FL_WARPS;
    for (u32 gw = blockIdx.x * FL_WARPS + (threadIdx.x >> 5); (i64)gw * K < n; gw += nwarps) {
        const int i0 = (int)gw * K;                     // < n < 2^31 (loop condition); 64 bits would cost a register
        const int nm = min(K, n - i0);

        // ---- side job: this group's share of a buffer the caller wants zeroed (the dense matrices of the rows that
        // follow).  The decode is bound by instruction issue and leaves HBM idle; these few fire-and-forget stores per
        // group replace a separate 1 GB fill per 1,000 C2 images
        if (ZERO) {
            const u32 z0 = (u32)gw * zero_per_group, z1 = min(z0 + zero_per_group, zero_chunks);     // no overflow: see the launch
            // streaming stores: the zeros must not push the windows written below out of L2 (the join reads them next)
            for (u32 k = z0 + lane; k < z1; k += 32) __stcs(zero + k, make_uint4(0u, 0u, 0u, 0u));
        }

        // ---- the warp's masks: one lane each
        u32 my_pairs = 0;
        bool my_big = false;
        if ((int)lane < nm) {
            const i64 i = i0 + lane;
            const int len = cnt_len[i];
            const u32 H = hh[i];
            const u64 HW = (u64)H * ww[i];
            S.geo[lane] = make_uint4(H, H ? 0xffffffffu / H : 0u, (u32)HW, (u32)len);
            S.src[lane] = cnt + cnt_off[i];
            my_pairs = (u32)(len + 1) >> 1;
            my_big = len < 0 || H == 0 || H > FL_HMAX || HW >= (u64)FL_SAT || my_pairs > FL_PAIR_CAP;
        }
        __syncwarp();

        int a = 0;                                       // first mask of the round (index inside the warp's masks)
        while (a < nm) {
            // ---- round = longest prefix of the remaining masks whose pairs fit (a single small mask always does)
            const bool mine = (int)lane >= a && (int)lane < nm;
            const u32 v = (mine && !my_big) ? my_pairs : 0u;
            const u32 incl = warp_incl_scan(v, lane);
            const bool in_round = mine && incl <= FL_PAIR_CAP;
            const int nb = __popc(__ballot_sync(0xffffffffu, in_round));
            const u32 T = __shfl_sync(0xffffffffu, incl, a + nb - 1);
            const int j_me = (int)lane - a;               // my mask's index inside the round
            if (in_round) {
                S.pb[j_me] = incl - v;
                if (j_me == nb - 1) S.pb[nb] = T;
                S.area[j_me] = 0u; S.first[j_me] = 0xffffffffu; S.last[j_me] = 0u;
                S.ymin[j_me] = 0xffffffffu; S.ymaxi[j_me] = 0xffffffffu; S.total[j_me] = 0u;
                if (IV) S.convex[j_me] = 1u;
                if (my_big) big[1 + atomicAdd(&big[0], 1)] = (int)(i0 + lane);
            }
            __syncwarp();

            // ---- staging: the round's raw pairs, lane-strided (coalesced reads of the run counts), and the mask of
            // every pair.  The round is padded to whole slices of 8 with (0, 0) pairs of its last mask: they move no
            // end, add no pixel and paint nothing.
            const u32 Tr = (T + 7u) & ~7u;
            {
                int j = 0;
                u32 cur = 0, nxt = S.pb[1];              // my mask's first pair and the next mask's: only grow
                for (u32 f = lane; f < Tr; f += 32) {
                    uint2 zo = make_uint2(0u, 0u);
                    if (f < T) {
                        while (f >= nxt) { j++; cur = nxt; nxt = S.pb[j + 1]; }
                        const u32 p = f - cur;
                        const u32 *c = S.src[a + j] + 2 * p;
                        zo.x = min(__ldcs(c), FL_SAT);                      // read once: evict first
                        if ((int)(2 * p + 1) < (int)S.geo[a + j].w) zo.y = min(__ldcs(c + 1), FL_SAT);
                    }
                    S.mid[f] = (uint8_t)(f < T ? j : nb - 1);
                    S.pair[fl_swz(f)] = zo;
                }
            }
            __syncwarp();

            // ---- measure pass: lane l owns pairs 8l .. 8l+7 of the round.  Pass 1 sums (saturating) the run ends
            // from the last mask start in the slice; ONE segmented warp scan of these sums (segments = masks) gives
            // every lane the end position before its first pair; pass 2 walks the slice again, forms the painter's
            // records and keeps each mask's statistics in registers, which it adds to the mask once per slice.
            const u32 f8 = lane * 8u;
            const uint2 mm = *reinterpret_cast<const uint2 *>(&S.mid[f8]);     // masks of my 8 pairs, a byte each
            const u32 mprev = __shfl_up_sync(0xffffffffu, mm.y >> 24, 1);
            // bit k: a mask starts at my pair k (pair 0 of the round always starts one, so lane 0 heads every scan)
            u32 hb;
            {
                const u32 dl = __vcmpne4(mm.x, (mm.x << 8) | mprev), dh = __vcmpne4(mm.y, __funnelshift_l(mm.x, mm.y, 8));
                hb = ((dl & 0x01010101u) * 0x01020408u) >> 24 | ((dh & 0x01010101u) * 0x01020408u) >> 20 | (lane == 0u);
            }
            // my slice in 16-byte chunks, chunk q at q ^ sw (fl_swz)
            uint4 *slice = reinterpret_cast<uint4 *>(S.pair) + 4u * lane;
            const u32 sw = (lane >> 1) & 3u;
            u32 sum = 0;                                  // run ends summed (saturating) from the last start
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint4 c = slice[q ^ sw];
                sum = sat_add((hb >> (2 * q)) & 1u ? 0u : sum, sat_add(c.x, c.y));
                sum = sat_add((hb >> (2 * q + 1)) & 1u ? 0u : sum, sat_add(c.z, c.w));
            }
            u32 sc = sum | (hb ? FL_HEAD : 0u);
            // sat_add is associative on operands <= FL_SAT, so the scan saturates as the sequential walk does.  No
            // lane test: lane 0 is flagged, so a lane below d has a flag by step d and takes nothing from above
#pragma unroll
            for (u32 d = 1; d < 32; d <<= 1) {
                const u32 t = __shfl_up_sync(0xffffffffu, sc, d);
                if (!(sc & FL_HEAD)) sc = sat_add(t & FL_SAT, sc) | (t & FL_HEAD);
            }
            u32 e = __shfl_up_sync(0xffffffffu, sc, 1) & FL_SAT;    // end of the pair before my slice
            if (f8 < T) {
                u32 j = mm.x & 0xffu;
                uint4 g = S.geo[a + j];                   // H, 2^32 / H, H * W
                u32 ar = 0, fi = 0xffffffffu, la = 0, ypk = 0xffffffffu;   // area, first / last pixel, row range
                auto flush = [&](bool ended) {
                    if (fi != 0xffffffffu) {
                        atomicAdd(&S.area[j], ar);
                        atomicMin(&S.first[j], fi);
                        atomicMax(&S.last[j], la);
                        atomicMin(&S.ymin[j], ypk & 0xffffu);
                        atomicMin(&S.ymaxi[j], ypk >> 16);
                    }
                    if (ended) S.total[j] = e;
                };
                auto step = [&](u32 k, u32 z, u32 o) {
                    const bool h = (hb >> k) & 1u;
                    if (k > 0u && h) {                    // the previous mask ended at pair k - 1
                        flush(true);
                        j = S.mid[f8 + k];
                        g = S.geo[a + j];
                        ar = 0u; fi = 0xffffffffu; la = 0u; ypk = 0xffffffffu;
                    }
                    e = sat_add(h ? 0u : e, sat_add(z, o));
                    uint2 pr = FL_EMPTY;
                    if (e <= g.z) {                       // H * W < FL_SAT: nothing saturated up to here
                        ar += o;
                        if (o > 0u) {
                            const u32 H = g.x, start = e - o;
                            const u32 x = div_by(start, H, g.y);
                            const u32 ys = start - x * H, yl = ys + o - 1u;
                            // column-convex test (IV): a 1-run over several columns, or one whose 0-run starts in its
                            // own column behind an earlier pair of the mask -- the 1-run before it ends in this column,
                            // or (a zero-length 1-run in between; conservative) the gap only looks so -- makes the
                            // mask a bitmap
                            if (IV && (yl >= H || (!h && z < ys))) S.convex[j] = 0u;
                            fi = min(fi, start); la = e;
                            if (yl >= H) { pr = make_uint2(start | FL_SPAN, o); ypk = __vminu2(ypk, (0xffffu - (H - 1u)) << 16); }
                            else { pr = make_uint2(x, ys | (yl << 16)); ypk = __vminu2(ypk, ys | ((0xffffu - yl) << 16)); }
                        }
                    }
                    return pr;
                };
                // the painter's records replace the staged pairs
#pragma unroll 1
                for (u32 q = 0; q < 4u; q++) {
                    const uint4 c = slice[q ^ sw];
                    const uint2 r0 = step(2u * q, c.x, c.y), r1 = step(2u * q + 1u, c.z, c.w);
                    slice[q ^ sw] = make_uint4(r0.x, r0.y, r1.x, r1.y);
                }
                flush(f8 + 8u >= T || S.mid[f8 + 8u] != j);
            }
            __syncwarp();

            // ---- records: one lane per mask; window sizes -> tile offsets
            u32 chunks = 0;
            int4 bb = make_int4(0, 0, -1, -1);
            const bool rec = in_round && !my_big;
            uint4 geo = make_uint4(1u, 0u, 0u, 0u);
            if (rec) {
                geo = S.geo[lane];
                const u32 H = geo.x, HW = geo.z;
                const u32 ar = S.area[j_me], fi = S.first[j_me], la = S.last[j_me];
                const u32 nchunks = (HW + AMPIS_CHUNK_BITS - 1u) / AMPIS_CHUNK_BITS;
                uint2 sp = make_uint2(0u, 0u);
                if (ar > 0u) {
                    sp = make_uint2(fi / AMPIS_CHUNK_BITS, min((la + AMPIS_CHUNK_BITS - 1u) / AMPIS_CHUNK_BITS, nchunks));
                    bb = make_int4((int)div_by(fi, H, geo.y), (int)S.ymin[j_me], (int)div_by(la - 1u, H, geo.y),
                                   (int)(0xffffu - S.ymaxi[j_me]));
                }
                // an interval window is never larger than the bitmap window: the arena sizes of measure() still hold
                // (S.convex[j_me] says from here on whether the mask is stored as intervals: no register for it)
                if (IV && ar == 0u) S.convex[j_me] = 0u;
                chunks = IV && S.convex[j_me] ? ((u32)(bb.z - bb.x) + 4u) / 4u : (crop_words(bb) + 3u) / 4u;
                const i64 i = i0 + lane;
                area[i] = ar;
                reinterpret_cast<int4 *>(bbox)[i] = bb;
                reinterpret_cast<uint2 *>(span)[i] = sp;
                // a bitmap until painted below: a window larger than the tile goes to the fallback kernel as a bitmap
                reinterpret_cast<uint2 *>(reg)[i] = make_uint2(0u, chunks);
                status[i] = S.total[j_me] == HW ? 0 : AMPIS_ST_BAD_TOTAL;
            }
            const u32 cincl = warp_incl_scan(chunks, lane);

            // ---- windows: the round's masks are painted in groups that fit the tile (usually all of them at once).
            // Per group: ONE arena reservation, the tile is zeroed, every lane sets the bits of its 1-runs, and the
            // tile -- contiguous in the arena -- is copied out with 128-bit stores.
            int lo = a;                                       // first mask (lane) of the round not yet painted
            const int hi = a + nb;
            while (lo < hi) {
                const u32 before = lo > 0 ? __shfl_sync(0xffffffffu, cincl, lo - 1) : 0u;
                const u32 rel = cincl - before;                // chunks of the masks lo..me
                const bool here = (int)lane >= lo && (int)lane < hi && rel * 4u <= FL_TILE_WORDS;   // a prefix of lo..hi-1
                const u32 here_m = __ballot_sync(0xffffffffu, here);
                if (!((here_m >> lo) & 1u)) {                 // this window alone is larger than the tile: fallback kernel
                    if ((int)lane == lo) big[1 + atomicAdd(&big[0], 1)] = (int)(i0 + lane);
                    lo++;
                    continue;
                }
                const int last = 31 - __clz(here_m);
                const u32 fit = __shfl_sync(0xffffffffu, rel, last);
                unsigned long long base = 0;
                if (lane == 0 && fit) base = atomicAdd(cursor, (unsigned long long)fit);
                base = __shfl_sync(0xffffffffu, base, 0);
                const bool room = (i64)(base + fit) <= capacity;
                if (here && rec) {
                    const i64 i = i0 + lane;
                    if (room) {
                        bits_off[i] = (i64)base + (rel - chunks);
                        if (IV && S.convex[j_me]) {
                            // one word per column; 0 bands per column tells the painter
                            reinterpret_cast<uint2 *>(reg)[i] = make_uint2(AMPIS_WIN_INTERVALS, chunks);
                            S.win[j_me] = make_uint4(geo.x, geo.y, (rel - chunks) * 4u - (u32)bb.x, 0u);
                        } else {
                            const u32 wy0 = (u32)bb.y >> 5, nwy = ((u32)bb.w >> 5) - wy0 + 1u;
                            S.win[j_me] = make_uint4(geo.x, geo.y, (rel - chunks) * 4u - (u32)bb.x * nwy - wy0, nwy);
                        }
                    } else {
                        // arena exhausted: the caller sees *cursor > capacity and retries; until then the mask is empty
                        // for every later kernel (the crop rows kernels size their reads from the box)
                        bits_off[i] = 0;
                        reinterpret_cast<int4 *>(bbox)[i] = make_int4(0, 0, -1, -1);
                        reinterpret_cast<uint2 *>(span)[i] = make_uint2(0u, 0u);
                        reinterpret_cast<uint2 *>(reg)[i] = make_uint2(0u, 0u);
                    }
                }
                if (fit && room) {
                    uint4 *tile4 = reinterpret_cast<uint4 *>(S.tile);
                    for (u32 k = lane; k < fit; k += 32) tile4[k] = make_uint4(0u, 0u, 0u, 0u);
                    __syncwarp();
                    // every 1-run lies inside its mask's box: the box was formed from the same runs
                    const u32 f_end = S.pb[last - a + 1];
                    for (u32 f = S.pb[lo - a] + lane; f < f_end; f += 32) {
                        const uint2 pr = S.pair[fl_swz(f)];
                        if (!(pr.x & FL_SPAN)) {
                            const u32 ys = pr.y & 0xffffu, yl = pr.y >> 16;
                            if (ys > yl) continue;
                            const uint4 d = S.win[S.mid[f]];
                            // interval window: the column's only 1-run; a word left zero is an empty column
                            if (IV && d.w == 0u) S.tile[d.z + pr.x] = pr.y ^ 0xffffu;
                            else paint_rows(S.tile, d.z + pr.x * d.w, ys, yl);
                        } else {
                            const uint4 d = S.win[S.mid[f]];
                            const u32 s = pr.x & ~FL_SPAN;
                            const u32 x = div_by(s, d.x, d.y);
                            u32 ys = s - x * d.x, left = pr.y, idx = d.z + x * d.w;
                            while (left) {
                                const u32 take = min(left, d.x - ys);
                                paint_rows(S.tile, idx, ys, ys + take - 1u);
                                left -= take; ys = 0u; idx += d.w;
                            }
                        }
                    }
                    __syncwarp();
                    uint4 *out = bits + base;
                    for (u32 k = lane; k < fit; k += 32) out[k] = tile4[k];
                }
                __syncwarp();
                lo = last + 1;
            }
            a += nb;
        }
    }
}

// masks per warp for a typical number of runs per mask: fill ~4/5 of the pair budget (a warp whose masks exceed
// it simply works in two rounds)
static int flat_masks_per_warp(int runs_hint)
{
    if (runs_hint <= 0) return 4;
    const int pairs = runs_hint / 2 + 1;
    int k = (FL_PAIR_CAP * 4 / 5) / pairs;
    if (k < 1) k = 1;
    if (k > FL_KMAX) k = FL_KMAX;
    return k;
}

int ampis_launch_measure_paint_list(const uint32_t *d_cnt, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                                    const uint32_t *d_h, const uint32_t *d_w, const int32_t *d_list, int32_t max_n,
                                    uint32_t *d_cum, uint32_t *d_area, int32_t *d_bbox, uint32_t *d_span,
                                    uint32_t *d_reg, int64_t *d_bits_off, int32_t *d_status, void *d_bits,
                                    int64_t bits_capacity, uint64_t *d_cursor, cudaStream_t st);

extern "C" int ampis_rle_measure_paint_flat_zero(const uint32_t *d_cnt, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                                                 const uint32_t *d_h, const uint32_t *d_w, int32_t n, uint32_t *d_cum,
                                                 uint32_t *d_area, int32_t *d_bbox, uint32_t *d_span, uint32_t *d_reg,
                                                 int64_t *d_bits_off, int32_t *d_status, void *d_bits,
                                                 int64_t bits_capacity, uint64_t *d_cursor, int32_t *d_list,
                                                 int32_t runs_hint, void *d_zero, int64_t zero_bytes,
                                                 int32_t intervals, void *stream)
{
    AMPIS_REQUIRE(n >= 0 && zero_bytes >= 0, "n < 0 or zero_bytes < 0");
    cudaStream_t st = as_stream(stream);
    if (n == 0) {
        if (d_zero && zero_bytes > 0 && cudaMemsetAsync(d_zero, 0, (size_t)zero_bytes, st) != cudaSuccess) {
            ampis_set_error("memset: %s", cudaGetErrorString(cudaGetLastError()));
            return AMPIS_ECUDA;
        }
        return AMPIS_OK;
    }
    AMPIS_REQUIRE(d_cnt && d_cnt_off && d_cnt_len && d_h && d_w && d_cum && d_area && d_bbox && d_span && d_reg &&
                      d_bits_off && d_status && d_bits && d_cursor && d_list, "null pointer");
    AMPIS_REQUIRE(((uintptr_t)d_bits & 15u) == 0, "bits arena must be 16-byte aligned");
    AMPIS_REQUIRE(!d_zero || ((uintptr_t)d_zero & 15u) == 0, "buffer to zero must be 16-byte aligned");
    cudaError_t e = cudaMemsetAsync(d_cursor, 0, sizeof(uint64_t), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_list, 0, sizeof(int32_t), st);
    const int K = flat_masks_per_warp(runs_hint);
    const int64_t warps = ((int64_t)n + K - 1) / K;
    // the kernel zeroes whole 16-byte chunks with 32-bit indices: at most 2^32 - 2^24 of them over at most 2^24 groups
    // (84 million masks per launch), so that group x share stays below 2^32; what is left is cleared here
    const int64_t zero_chunks = (d_zero && warps <= (1 << 24)) ? std::min<int64_t>(zero_bytes / 16, 0xff000000ll) : 0;
    if (e == cudaSuccess && d_zero && zero_bytes > zero_chunks * 16)
        e = cudaMemsetAsync((char *)d_zero + zero_chunks * 16, 0, (size_t)(zero_bytes - zero_chunks * 16), st);
    if (e != cudaSuccess) { ampis_set_error("cursor memset: %s", cudaGetErrorString(e)); return AMPIS_ECUDA; }
    static thread_local int wave = 0;                 // one wave of CTAs; every warp strides over the groups
    if (!wave) {
        int dev = 0, sms = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0)
            wave = sms * FL_CTAS_PER_SM;
        else
            wave = 148 * FL_CTAS_PER_SM;
    }
    const unsigned grid = (unsigned)std::min<int64_t>((warps + FL_WARPS - 1) / FL_WARPS, wave);
    // (groups - 1) x share < chunks + groups <= 2^32
    const uint32_t per = zero_chunks > 0 ? (uint32_t)((zero_chunks + warps - 1) / warps) : 0u;
    auto kernel = zero_chunks > 0 ? (intervals ? rle_flat_crop_kernel<true, true> : rle_flat_crop_kernel<true, false>)
                                  : (intervals ? rle_flat_crop_kernel<false, true> : rle_flat_crop_kernel<false, false>);
    kernel<<<grid, FL_WARPS * 32, 0, st>>>(d_cnt, d_cnt_off, d_cnt_len, d_h, d_w, n, K, d_area, d_bbox, d_span, d_reg,
                                           d_bits_off, d_status, (uint4 *)d_bits, bits_capacity,
                                           (unsigned long long *)d_cursor, d_list,
                                           zero_chunks > 0 ? (uint4 *)d_zero : nullptr, (uint32_t)zero_chunks, per);
    AMPIS_CHECK_LAUNCH("rle_flat_crop_kernel");
    return ampis_launch_measure_paint_list(d_cnt, d_cnt_off, d_cnt_len, d_h, d_w, d_list, n, d_cum, d_area, d_bbox,
                                           d_span, d_reg, d_bits_off, d_status, d_bits, bits_capacity, d_cursor, st);
}

extern "C" int ampis_rle_measure_paint_flat(const uint32_t *d_cnt, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                                            const uint32_t *d_h, const uint32_t *d_w, int32_t n, uint32_t *d_cum,
                                            uint32_t *d_area, int32_t *d_bbox, uint32_t *d_span, uint32_t *d_reg,
                                            int64_t *d_bits_off, int32_t *d_status, void *d_bits,
                                            int64_t bits_capacity, uint64_t *d_cursor, int32_t *d_list,
                                            int32_t runs_hint, int32_t intervals, void *stream)
{
    return ampis_rle_measure_paint_flat_zero(d_cnt, d_cnt_off, d_cnt_len, d_h, d_w, n, d_cum, d_area, d_bbox, d_span,
                                             d_reg, d_bits_off, d_status, d_bits, bits_capacity, d_cursor, d_list,
                                             runs_hint, nullptr, 0, intervals, stream);
}
