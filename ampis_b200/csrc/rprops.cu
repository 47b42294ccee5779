// Region properties of instance masks (InstanceSet.compute_rprops, structures.py:474-514: the
// reference decodes every mask to a full int64 frame and calls skimage.measure.regionprops_table on
// it, "~30 s" for 2,300 masks).  Nothing is decoded here:
//   * raw moments up to order 2 come straight from the run table (a 1-run is a vertical segment
//     x, [a,b): its contributions are closed-form integer sums) -> centroid, inertia tensor,
//     major/minor axis length, orientation, eccentricity on the host from EXACT integer sums;
//   * the perimeter (skimage.measure.perimeter, 4-neighbourhood: border = mask minus its erosion,
//     each border pixel weighted by how many border pixels touch it by edge / by corner) is
//     bit-sliced arithmetic on the CROP-layout window words;
//   * the convex area (skimage convex_hull_image: hull of the four edge midpoints of every pixel,
//     then a crossing-number point-in-polygon test of the pixel centres) is exact integer geometry:
//     only the top and bottom pixel of every column can touch the hull, two monotone chains in
//     doubled coordinates, and per column the number of pixel centres in [top, bottom).
// The remaining non-intensity properties (below, after the C entries of the above): moments to order 3 as
// exact 128-bit sums from the runs; hole fill and Crofton transition counts on the CROP windows; the convex
// image as per-column row ranges plus the maximum Feret diameter as an exact integer; box images unpacked
// from the windows for image / coords / filled_image.  The intensity properties (last section): min, max and the
// weighted moments of an intensity image over every mask, from the run table -- exact for integer pixels.
#include <cuda_fp16.h>
#include <math_constants.h>

#include <climits>
#include <type_traits>

#include "common.cuh"

// ---- moments from runs: warp per mask ---------------------------------------------------------
// out[i] = { N, sum x, sum y, sum x^2, sum y^2, sum x*y }  (x = column, y = row), exact u64
__global__ void __launch_bounds__(256)
rle_moments_kernel(const u32 *__restrict__ cum, const i64 *__restrict__ cnt_off,
                   const int *__restrict__ cnt_len, const u32 *__restrict__ hh, int n,
                   unsigned long long *__restrict__ out)
{
    const int i = (int)((blockIdx.x * (u32)blockDim.x + threadIdx.x) >> 5);
    if (i >= n) return;
    const u32 lane = lane_id();
    const u32 *C = cum + cnt_off[i];
    const int m = cnt_len[i];
    const u64 H = hh[i];
    unsigned long long s[6] = {0, 0, 0, 0, 0, 0};
    for (int r = 1 + 2 * (int)lane; r < m; r += 64) {            // odd runs are the 1-runs
        u64 p = C[r - 1];
        const u64 e = C[r];
        while (p < e) {
            const u64 x = p / H, cs = x * H;
            const long long a = (long long)(p - cs), b = (long long)(min(e, cs + H) - cs);   // rows [a,b)
            const unsigned long long cnt = (unsigned long long)(b - a);
            const unsigned long long sy = (unsigned long long)((a + b - 1) * (b - a) / 2);
            const long long fb = (b - 1) * b * (2 * b - 1) / 6, fa = (a - 1) * a * (2 * a - 1) / 6;
            s[0] += cnt;
            s[1] += cnt * x;
            s[2] += sy;
            s[3] += cnt * x * x;
            s[4] += (unsigned long long)(fb - fa);
            s[5] += sy * x;
            p = cs + H;
        }
    }
#pragma unroll
    for (int k = 0; k < 6; k++) {
#pragma unroll
        for (int d = 16; d; d >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], d);
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 6; k++) out[6 * (i64)i + k] = s[k];
    }
}

extern "C" int ampis_rle_moments(const uint32_t *d_cum, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                                 const uint32_t *d_h, int32_t n, uint64_t *d_out, void *stream)
{
    AMPIS_REQUIRE(n >= 0, "n < 0");
    if (n == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_cum && d_cnt_off && d_cnt_len && d_h && d_out, "null pointer");
    rle_moments_kernel<<<(unsigned)(((i64)n * 32 + 255) / 256), 256, 0, as_stream(stream)>>>(
        d_cum, d_cnt_off, d_cnt_len, d_h, n, (unsigned long long *)d_out);
    AMPIS_CHECK_LAUNCH("rle_moments_kernel");
    return AMPIS_OK;
}

// ---- CROP window access -------------------------------------------------------------------------
struct Win {
    const u32 *W;
    int x0, x1;        // columns (inclusive)
    u32 wy0, nwy;      // absolute 32-row bands
    __device__ __forceinline__ u32 word(int x, int wy) const     // wy relative to wy0; zero outside
    {
        if (x < x0 || x > x1 || wy < 0 || wy >= (int)nwy) return 0u;
        return W[(u32)(x - x0) * nwy + (u32)wy];
    }
};

__device__ __forceinline__ Win win_of(const u32 *bits, const i64 *bits_off, const int4 *bbox, int i)
{
    const int4 bb = bbox[i];
    Win w;
    w.W = bits + bits_off[i] * 4;
    w.x0 = bb.x; w.x1 = bb.z;
    w.wy0 = (u32)bb.y >> 5;
    w.nwy = bb.z < bb.x ? 0u : ((u32)bb.w >> 5) - w.wy0 + 1u;
    return w;
}

// neighbours of every pixel of word (x, wy): the pixel one row down (y+1) / up (y-1)
__device__ __forceinline__ u32 shift_next_row(const Win &w, int x, int wy)   // bit j <- pixel y+1
{
    return (w.word(x, wy) >> 1) | (w.word(x, wy + 1) << 31);
}
__device__ __forceinline__ u32 shift_prev_row(const Win &w, int x, int wy)   // bit j <- pixel y-1
{
    return (w.word(x, wy) << 1) | (w.word(x, wy - 1) >> 31);
}

// pass 1: border = mask & ~erosion by the 4-neighbourhood cross (outside the box = background)
__global__ void __launch_bounds__(256)
crop_border_kernel(const u32 *__restrict__ bits, const i64 *__restrict__ bits_off, const int4 *__restrict__ bbox,
                   int n, u32 *__restrict__ border)
{
    const int i = (int)((blockIdx.x * (u32)blockDim.x + threadIdx.x) >> 5);
    if (i >= n) return;
    const Win w = win_of(bits, bits_off, bbox, i);
    if (!w.nwy) return;
    u32 *B = border + bits_off[i] * 4;
    const u32 total = (u32)(w.x1 - w.x0 + 1) * w.nwy;
    for (u32 idx = lane_id(); idx < total; idx += 32) {
        const int x = w.x0 + (int)(idx / w.nwy), wy = (int)(idx % w.nwy);
        const u32 cur = w.word(x, wy);
        const u32 er = cur & shift_next_row(w, x, wy) & shift_prev_row(w, x, wy) & w.word(x - 1, wy) & w.word(x + 1, wy);
        B[idx] = cur & ~er;
    }
}

// pass 2: every border pixel gets the code 1 + 2*(edge-adjacent border pixels) + 10*(corner-adjacent
// border pixels) -- the value skimage's 3x3 convolution [[10,2,10],[2,1,2],[10,2,10]] yields -- and
// the ten codes that carry a weight are counted: order 5,7,15,17,25,27 (weight 1), 21,33 (sqrt 2),
// 13,23 ((1+sqrt 2)/2).
__constant__ int c_code_e[10] = {2, 3, 2, 3, 2, 3, 0, 1, 1, 1};
__constant__ int c_code_d[10] = {0, 0, 1, 1, 2, 2, 2, 3, 1, 2};

__device__ __forceinline__ void count4(u32 a, u32 b, u32 c, u32 d, u32 &p0, u32 &p1, u32 &p2)
{
    const u32 s1 = a ^ b, c1 = a & b, s2 = c ^ d, c2 = c & d, t = s1 & s2;
    p0 = s1 ^ s2; p1 = c1 ^ c2 ^ t; p2 = c1 & c2;
}
__device__ __forceinline__ u32 equals_k(u32 p0, u32 p1, u32 p2, int k)
{
    return ((k & 1) ? p0 : ~p0) & ((k & 2) ? p1 : ~p1) & ((k & 4) ? p2 : ~p2);
}

__global__ void __launch_bounds__(256)
crop_perimeter_kernel(const u32 *__restrict__ border, const i64 *__restrict__ bits_off,
                      const int4 *__restrict__ bbox, int n, u32 *__restrict__ hist10)
{
    const int i = (int)((blockIdx.x * (u32)blockDim.x + threadIdx.x) >> 5);
    if (i >= n) return;
    const Win w = win_of(border, bits_off, bbox, i);
    u32 h[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    const u32 total = w.nwy ? (u32)(w.x1 - w.x0 + 1) * w.nwy : 0u;
    for (u32 idx = lane_id(); idx < total; idx += 32) {
        const int x = w.x0 + (int)(idx / w.nwy), wy = (int)(idx % w.nwy);
        const u32 bc = w.word(x, wy);
        if (!bc) continue;
        u32 e0, e1, e2, d0, d1, d2;
        count4(shift_next_row(w, x, wy), shift_prev_row(w, x, wy), w.word(x - 1, wy), w.word(x + 1, wy), e0, e1, e2);
        count4(shift_next_row(w, x - 1, wy), shift_prev_row(w, x - 1, wy), shift_next_row(w, x + 1, wy),
               shift_prev_row(w, x + 1, wy), d0, d1, d2);
#pragma unroll
        for (int k = 0; k < 10; k++)
            h[k] += __popc(bc & equals_k(e0, e1, e2, c_code_e[k]) & equals_k(d0, d1, d2, c_code_d[k]));
    }
#pragma unroll
    for (int k = 0; k < 10; k++) {
        const u32 v = warp_sum(h[k]);
        if (lane_id() == 0) hist10[10 * (i64)i + k] = v;
    }
}

// ---- convex area: thread per mask -----------------------------------------------------------------
// Doubled coordinates X = 2*column, Y = 2*row.  Candidates of the lower chain (smallest row per X) and
// of the upper chain (largest row per X) come from the top / bottom pixel of every column:
//   even X = 2x   : top(x)*2 - 1            / bottom(x)*2 + 1
//   odd  X = 2x+1 : min top of x, x+1 (*2)  / max bottom of x, x+1 (*2)
__device__ __forceinline__ i64 ceil_div(i64 a, i64 b)      // b > 0
{
    return a >= 0 ? (a + b - 1) / b : -((-a) / b);
}

// Monotone chains of points arriving in increasing X: the lower chain keeps turning left (slopes increase),
// the upper chain keeps turning right (slopes decrease).
struct Chains {
    int *LX, *LY, *UX, *UY;
    int nl, nu;
};

__device__ __forceinline__ void chains_push(int *LX, int *LY, int *UX, int *UY, int &nl, int &nu, int X, int yl, int yu)
{
    while (nl >= 2 && (i64)(LX[nl - 1] - LX[nl - 2]) * (yl - LY[nl - 2]) -
                          (i64)(LY[nl - 1] - LY[nl - 2]) * (X - LX[nl - 2]) <= 0) nl--;
    LX[nl] = X; LY[nl] = yl; nl++;
    while (nu >= 2 && (i64)(UX[nu - 1] - UX[nu - 2]) * (yu - UY[nu - 2]) -
                          (i64)(UY[nu - 1] - UY[nu - 2]) * (X - UX[nu - 2]) >= 0) nu--;
    UX[nu] = X; UY[nu] = yu; nu++;
}

// Hull of the pixel-edge midpoints of a CROP window (scratch of 10*bw+4 ints: top[bw], bot[bw], then the two
// chains of at most 2*bw+1 points each).  Returns false for an empty window.
__device__ __forceinline__ bool hull_of_window(const Win &w, int *scr, Chains &h)
{
    if (!w.nwy) return false;
    const int bw = w.x1 - w.x0 + 1;
    int *top = scr, *bot = top + bw;
    int *LX = bot + bw, *LY = LX + (2 * bw + 1), *UX = LY + (2 * bw + 1), *UY = UX + (2 * bw + 1);
    for (int c = 0; c < bw; c++) {
        int t = -1, b = -1;
        for (u32 k = 0; k < w.nwy; k++) {
            const u32 v = w.W[(u32)c * w.nwy + k];
            if (v) { t = (int)((w.wy0 + k) * 32u) + __ffs(v) - 1; break; }
        }
        for (int k = (int)w.nwy - 1; k >= 0 && t >= 0; k--) {
            const u32 v = w.W[(u32)c * w.nwy + (u32)k];
            if (v) { b = (int)((w.wy0 + (u32)k) * 32u) + 31 - __clz(v); break; }
        }
        top[c] = t; bot[c] = b;
    }
    int nl = 0, nu = 0;
    for (int X = -1; X <= 2 * bw - 1; X++) {               // X relative to 2*x0
        int yl, yu;
        if (X & 1) {                                        // between columns c = (X-1)/2 and c+1
            const int c = (X - 1) >> 1;                     // floor for X = -1 gives -1
            const int t0 = (c >= 0 && top[c] >= 0) ? top[c] : 0x3fffffff;
            const int t1 = (c + 1 < bw && top[c + 1] >= 0) ? top[c + 1] : 0x3fffffff;
            const int b0 = (c >= 0 && top[c] >= 0) ? bot[c] : -1;
            const int b1 = (c + 1 < bw && top[c + 1] >= 0) ? bot[c + 1] : -1;
            if (min(t0, t1) == 0x3fffffff) continue;
            yl = 2 * min(t0, t1); yu = 2 * max(b0, b1);
        } else {
            const int c = X >> 1;
            if (top[c] < 0) continue;
            yl = 2 * top[c] - 1; yu = 2 * bot[c] + 1;
        }
        chains_push(LX, LY, UX, UY, nl, nu, X, yl, yu);
    }
    h.LX = LX; h.LY = LY; h.UX = UX; h.UY = UY; h.nl = nl; h.nu = nu;
    return true;
}

// Pixel centres inside the hull in column c (X = 2c): rows lo <= r < hi (crossing-number rule).  Columns are
// visited in increasing order; il / iu are the chain cursors, starting at 0.  False when the column lies
// outside the hull (cannot happen for a column of the box).
__device__ __forceinline__ bool hull_column(const Chains &h, int c, int &il, int &iu, i64 &lo, i64 &hi)
{
    const int *LX = h.LX, *LY = h.LY, *UX = h.UX, *UY = h.UY;
    const int X = 2 * c;
    while (il + 2 < h.nl && LX[il + 1] <= X) il++;
    while (iu + 2 < h.nu && UX[iu + 1] <= X) iu++;
    if (X < LX[0] || X > LX[h.nl - 1]) return false;
    {
        const i64 D = LX[il + 1] - LX[il];
        const i64 num = (i64)LY[il] * D + (i64)(LY[il + 1] - LY[il]) * (X - LX[il]);    // = Y * D, row = Y / 2
        lo = ceil_div(num, 2 * D);
    }
    {
        const i64 D = UX[iu + 1] - UX[iu];
        const i64 num = (i64)UY[iu] * D + (i64)(UY[iu + 1] - UY[iu]) * (X - UX[iu]);
        hi = ceil_div(num, 2 * D);
    }
    return true;
}

__global__ void __launch_bounds__(128)
crop_convex_area_kernel(const u32 *__restrict__ bits, const i64 *__restrict__ bits_off,
                        const int4 *__restrict__ bbox, int n, const i64 *__restrict__ scr_off,
                        int *__restrict__ scratch, unsigned long long *__restrict__ convex_area)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Win w = win_of(bits, bits_off, bbox, i);
    Chains h;
    if (!hull_of_window(w, scratch + scr_off[i], h)) { convex_area[i] = 0; return; }
    const int bw = w.x1 - w.x0 + 1;
    unsigned long long area = 0;
    int il = 0, iu = 0;
    for (int c = 0; c < bw; c++) {
        i64 lo, hi;
        if (hull_column(h, c, il, iu, lo, hi) && hi > lo) area += (unsigned long long)(hi - lo);
    }
    convex_area[i] = area;
}

extern "C" int ampis_crop_perimeter(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox,
                                    int32_t n, void *d_border_scratch, uint32_t *d_hist10, void *stream)
{
    AMPIS_REQUIRE(n >= 0, "n < 0");
    if (n == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_bits && d_bits_off && d_bbox && d_border_scratch && d_hist10, "null pointer");
    const unsigned blocks = (unsigned)(((i64)n * 32 + 255) / 256);
    crop_border_kernel<<<blocks, 256, 0, as_stream(stream)>>>((const u32 *)d_bits, d_bits_off, (const int4 *)d_bbox, n,
                                                              (u32 *)d_border_scratch);
    AMPIS_CHECK_LAUNCH("crop_border_kernel");
    crop_perimeter_kernel<<<blocks, 256, 0, as_stream(stream)>>>((const u32 *)d_border_scratch, d_bits_off,
                                                                 (const int4 *)d_bbox, n, d_hist10);
    AMPIS_CHECK_LAUNCH("crop_perimeter_kernel");
    return AMPIS_OK;
}

extern "C" int ampis_crop_convex_area(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox,
                                      int32_t n, const int64_t *d_scratch_off, int32_t *d_scratch,
                                      uint64_t *d_convex_area, void *stream)
{
    AMPIS_REQUIRE(n >= 0, "n < 0");
    if (n == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_bits && d_bits_off && d_bbox && d_scratch_off && d_scratch && d_convex_area, "null pointer");
    crop_convex_area_kernel<<<(unsigned)((n + 127) / 128), 128, 0, as_stream(stream)>>>(
        (const u32 *)d_bits, d_bits_off, (const int4 *)d_bbox, n, d_scratch_off, d_scratch,
        (unsigned long long *)d_convex_area);
    AMPIS_CHECK_LAUNCH("crop_convex_area_kernel");
    return AMPIS_OK;
}

// ==== the remaining non-intensity properties of skimage 0.18.3 ======================================

// ---- moments to order 3 in box-local coordinates: warp per mask, exact 128-bit sums ----------------
typedef unsigned __int128 u128;

// sum_{k<m} k^p for p = 0..3 (m < 2^32)
__device__ __forceinline__ void power_sums(u64 m, u128 s[4])
{
    const u64 a = m * (m - 1) / 2;                          // m (m-1) < 2^64
    const u64 t = 2 * m - 1;
    s[0] = m;
    s[1] = a;
    s[2] = (a % 3 == 0) ? (u128)(a / 3) * t : (u128)a * (t / 3);     // a (2m-1) / 3, one factor divides
    s[3] = (u128)a * a;
}

__device__ __forceinline__ u128 shfl_xor_u128(u128 v, int d)
{
    const u64 lo = __shfl_xor_sync(0xffffffffu, (u64)v, d), hi = __shfl_xor_sync(0xffffffffu, (u64)(v >> 64), d);
    return ((u128)hi << 64) | lo;
}

// out[i] = 16 pairs (low, high 64-bit halves) of M[p][q] = sum r^p c^q, p, q = 0..3, row-major in (p, q),
// r = row - y0, c = column - x0 of the mask's box.  Exact while the frame's sides are <= 65536.
__global__ void __launch_bounds__(256)
rle_moments3_kernel(const u32 *__restrict__ cum, const i64 *__restrict__ cnt_off, const int *__restrict__ cnt_len,
                    const u32 *__restrict__ hh, const int4 *__restrict__ bbox, int n, unsigned long long *__restrict__ out)
{
    const int i = (int)((blockIdx.x * (u32)blockDim.x + threadIdx.x) >> 5);
    if (i >= n) return;
    const u32 lane = lane_id();
    const u32 *C = cum + cnt_off[i];
    const int m = cnt_len[i];
    const u64 H = hh[i];
    const int4 bb = bbox[i];
    u128 s[16];
#pragma unroll
    for (int k = 0; k < 16; k++) s[k] = 0;
    for (int r = 1 + 2 * (int)lane; r < m; r += 64) {            // odd runs are the 1-runs
        u64 p = C[r - 1];
        const u64 e = C[r];
        while (p < e) {
            const u64 x = p / H, cs = x * H;
            const u64 a = p - cs - (u64)bb.y, b = min(e, cs + H) - cs - (u64)bb.y;   // local rows [a, b)
            u128 sa[4], sb[4];
            power_sums(a, sa);
            power_sums(b, sb);
            const u128 c = x - (u64)bb.x;
            const u128 cq[4] = {1, c, c * c, c * c * c};
#pragma unroll
            for (int pp = 0; pp < 4; pp++) {
                const u128 rp = sb[pp] - sa[pp];
#pragma unroll
                for (int q = 0; q < 4; q++) s[4 * pp + q] += rp * cq[q];
            }
            p = cs + H;
        }
    }
#pragma unroll
    for (int k = 0; k < 16; k++) {
#pragma unroll
        for (int d = 16; d; d >>= 1) s[k] += shfl_xor_u128(s[k], d);
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            out[32 * (i64)i + 2 * k] = (unsigned long long)s[k];
            out[32 * (i64)i + 2 * k + 1] = (unsigned long long)(s[k] >> 64);
        }
    }
}

extern "C" int ampis_rle_moments3(const uint32_t *d_cum, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                                  const uint32_t *d_h, const int32_t *d_bbox, int32_t n, uint64_t *d_out, void *stream)
{
    AMPIS_REQUIRE(n >= 0, "n < 0");
    if (n == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_cum && d_cnt_off && d_cnt_len && d_h && d_bbox && d_out, "null pointer");
    rle_moments3_kernel<<<(unsigned)(((i64)n * 32 + 255) / 256), 256, 0, as_stream(stream)>>>(
        d_cum, d_cnt_off, d_cnt_len, d_h, (const int4 *)d_bbox, n, (unsigned long long *)d_out);
    AMPIS_CHECK_LAUNCH("rle_moments3_kernel");
    return AMPIS_OK;
}

// ---- hole fill (8-connected background) and Crofton transition counts: warp per mask -------------
// Bits of band wy (relative) that lie on rows y0..y1 of the box.
__device__ __forceinline__ u32 box_rows(const Win &w, int wy, int y0, int y1)
{
    const int base = (int)((w.wy0 + (u32)wy) * 32u);
    const int lo = max(y0 - base, 0), hi = min(y1 - base, 31);        // bits lo..hi
    if (hi < lo) return 0u;
    return (0xffffffffu >> (31 - hi)) & (0xffffffffu << lo);
}

// Bits of the background B reached from the seeds S moving towards higher bits inside runs of B (carry trick);
// bit 31 of the result set = the reach leaves the word at the top.
__device__ __forceinline__ u32 reach_up(u32 S, u32 B)
{
    S &= B;
    return (((B + S) ^ B) & B) | S;
}
__device__ __forceinline__ u32 reach_down(u32 S, u32 B)
{
    return __brev(reach_up(__brev(S), __brev(B)));
}

// Reached-background word of column x, band wy; everything outside the window is reached.
__device__ __forceinline__ u32 reached(const u32 *R, const Win &w, int x, int wy)
{
    if (x < w.x0 || x > w.x1 || wy < 0 || wy >= (int)w.nwy) return 0xffffffffu;
    return R[(u32)(x - w.x0) * w.nwy + (u32)wy];
}

// filled (same CROP layout and offsets as bits, may be null): binary_fill_holes(image, structure=ones((3,3))) of
// the box image -- the background 8-connected to the outside of the box is propagated to a fixed point, whole
// runs at a time: lanes own bands and sweep the columns left-right and right-left (rows and diagonals), then
// lanes own columns and sweep their bands up and down (columns), until a round changes nothing.  A round
// costs O(box words) and the number of rounds follows the turns of the longest background corridor.
// filled_area[i] = its pixel count.  trans (may be null): 4 counts per mask of 4-/8-adjacent pixel pairs
// that differ (outside the box = 0) along rows, columns, the diagonal (r+1, c+1) and the anti-diagonal.
__global__ void __launch_bounds__(256)
crop_fill_trans_kernel(const u32 *__restrict__ bits, const i64 *__restrict__ bits_off, const int4 *__restrict__ bbox,
                       int n, u32 *filled, unsigned long long *__restrict__ filled_area,
                       unsigned long long *__restrict__ trans)
{
    const int i = (int)((blockIdx.x * (u32)blockDim.x + threadIdx.x) >> 5);
    if (i >= n) return;
    const u32 lane = lane_id();
    const Win w = win_of(bits, bits_off, bbox, i);
    const u32 total = w.nwy ? (u32)(w.x1 - w.x0 + 1) * w.nwy : 0u;
    if (trans) {
        unsigned long long t[4] = {0, 0, 0, 0};
        for (u32 idx = lane; idx < total; idx += 32) {
            const int x = w.x0 + (int)(idx / w.nwy), wy = (int)(idx % w.nwy);
            const u32 cur = w.word(x, wy);
            if (!cur) continue;
            // every differing pair has exactly one pixel inside: count the outside neighbours of inside pixels
            t[0] += __popc(cur & ~w.word(x - 1, wy)) + __popc(cur & ~w.word(x + 1, wy));
            t[1] += __popc(cur & ~shift_next_row(w, x, wy)) + __popc(cur & ~shift_prev_row(w, x, wy));
            t[2] += __popc(cur & ~shift_next_row(w, x + 1, wy)) + __popc(cur & ~shift_prev_row(w, x - 1, wy));
            t[3] += __popc(cur & ~shift_next_row(w, x - 1, wy)) + __popc(cur & ~shift_prev_row(w, x + 1, wy));
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
#pragma unroll
            for (int d = 16; d; d >>= 1) t[k] += __shfl_xor_sync(0xffffffffu, t[k], d);
            if (lane == 0) trans[4 * (i64)i + k] = t[k];
        }
    }
    if (!filled) return;
    if (!total) {
        if (lane == 0) filled_area[i] = 0;
        return;
    }
    const int4 bb = bbox[i];
    const int bw = w.x1 - w.x0 + 1, nwy = (int)w.nwy;
    u32 *R = filled + bits_off[i] * 4;                          // reached background while propagating
    for (u32 idx = lane; idx < total; idx += 32) R[idx] = ~box_rows(w, (int)(idx % w.nwy), bb.y, bb.w);
    __syncwarp();
    for (;;) {
        bool changed = false;
        for (int dir = 1; dir >= -1; dir -= 2) {                // rows and diagonals: lanes own bands
            for (int s = 0; s < bw; s++) {
                const int x = dir > 0 ? w.x0 + s : w.x1 - s, xp = x - dir;
                for (int wy = (int)lane; wy < nwy; wy += 32) {
                    const u32 B = ~w.word(x, wy);
                    const u32 np = reached(R, w, xp, wy);
                    const u32 dil = np | (np << 1) | (reached(R, w, xp, wy - 1) >> 31) | (np >> 1) |
                                    (reached(R, w, xp, wy + 1) << 31);
                    u32 *p = R + (u32)(x - w.x0) * w.nwy + (u32)wy;
                    const u32 old = *p;
                    u32 v = old | (dil & B);
                    v = reach_up(v, B) | reach_down(v, B);
                    if (v != old) { *p = v; changed = true; }
                }
                __syncwarp();
            }
        }
        for (int c = (int)lane; c < bw; c += 32) {              // columns: lanes own columns
            u32 *col = R + (u32)c * w.nwy;
            u32 carry = 1u;                                     // the row below the window is outside
            for (int wy = 0; wy < nwy; wy++) {
                const u32 B = ~w.W[(u32)c * w.nwy + (u32)wy], old = col[wy];
                const u32 v = old | reach_up(old | (carry & B), B);
                carry = v >> 31;
                if (v != old) { col[wy] = v; changed = true; }
            }
            carry = 1u;
            for (int wy = nwy - 1; wy >= 0; wy--) {
                const u32 B = ~w.W[(u32)c * w.nwy + (u32)wy], old = col[wy];
                const u32 v = old | reach_down(old | ((carry << 31) & B), B);
                carry = v & 1u;
                if (v != old) { col[wy] = v; changed = true; }
            }
        }
        __syncwarp();
        if (!__any_sync(0xffffffffu, changed)) break;
    }
    unsigned long long area = 0;
    for (u32 idx = lane; idx < total; idx += 32) {
        const u32 f = ~R[idx] & box_rows(w, (int)(idx % w.nwy), bb.y, bb.w);
        R[idx] = f;
        area += __popc(f);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) area += __shfl_xor_sync(0xffffffffu, area, d);
    if (lane == 0) filled_area[i] = area;
}

extern "C" int ampis_crop_fill_holes(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox, int32_t n,
                                     void *d_filled, uint64_t *d_filled_area, uint64_t *d_trans, void *stream)
{
    AMPIS_REQUIRE(n >= 0, "n < 0");
    if (n == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_bits && d_bits_off && d_bbox, "null pointer");
    AMPIS_REQUIRE(!d_filled == !d_filled_area, "d_filled and d_filled_area go together");
    AMPIS_REQUIRE(d_filled || d_trans, "nothing to compute");
    crop_fill_trans_kernel<<<(unsigned)(((i64)n * 32 + 255) / 256), 256, 0, as_stream(stream)>>>(
        (const u32 *)d_bits, d_bits_off, (const int4 *)d_bbox, n, (u32 *)d_filled,
        (unsigned long long *)d_filled_area, (unsigned long long *)d_trans);
    AMPIS_CHECK_LAUNCH("crop_fill_trans_kernel");
    return AMPIS_OK;
}

// ---- convex image column ranges and maximum Feret diameter: thread per mask -----------------------
// Extreme rows of the symmetric difference of the row intervals [la, ha) and [lb, hb) (empty when h <= l).
__device__ __forceinline__ bool symdiff_extremes(int la, int ha, int lb, int hb, int &mn, int &mx)
{
    const bool ea = ha <= la, eb = hb <= lb;
    if (ea && eb) return false;
    if (ea) { mn = lb; mx = hb - 1; return true; }
    if (eb) { mn = la; mx = ha - 1; return true; }
    if (la == lb && ha == hb) return false;
    mn = la != lb ? min(la, lb) : min(ha, hb);
    mx = ha != hb ? max(ha, hb) - 1 : max(la, lb) - 1;
    return true;
}

// ranges[2 * (col_off[i] + c) + {0, 1}] = rows [lo, hi) (box-local, lo == hi when empty) of column c of
// convex_hull_image -- the pixels crop_convex_area_kernel counts.  feret_d2[i] = 4 * feret_diameter_max^2: the
// contour of the padded convex image at level 0.5 passes through the midpoints of its 4-adjacent
// (inside, outside) pixel pairs; in doubled coordinates (X = 2 col, Y = 2 row) only the smallest and largest Y
// of each X can be hull vertices, the chains of those are the hull, and the farthest pair is two of its
// vertices.  Same scratch as crop_convex_area_kernel (reused for the second hull).
__global__ void __launch_bounds__(128)
crop_convex_feret_kernel(const u32 *__restrict__ bits, const i64 *__restrict__ bits_off,
                         const int4 *__restrict__ bbox, int n, const i64 *__restrict__ scr_off,
                         int *__restrict__ scratch, const i64 *__restrict__ col_off, int *__restrict__ ranges,
                         unsigned long long *__restrict__ feret_d2)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Win w = win_of(bits, bits_off, bbox, i);
    Chains h;
    if (!hull_of_window(w, scratch + scr_off[i], h)) { feret_d2[i] = 0; return; }
    const int bw = w.x1 - w.x0 + 1, y0 = bbox[i].y;
    int *rg = ranges + 2 * col_off[i];
    int il = 0, iu = 0;
    for (int c = 0; c < bw; c++) {
        i64 lo = 0, hi = 0;
        if (!hull_column(h, c, il, iu, lo, hi) || hi < lo) hi = lo;
        rg[2 * c] = (int)(lo - y0);
        rg[2 * c + 1] = (int)(hi - y0);
    }
    Chains f = h;                                               // second hull in the same scratch
    int nl = 0, nu = 0;
    for (int X = -1; X <= 2 * bw - 1; X++) {
        int mn, mx;
        if (X & 1) {
            const int c = (X - 1) >> 1;
            const int la = c >= 0 ? rg[2 * c] : 0, ha = c >= 0 ? rg[2 * c + 1] : 0;
            const int lb = c + 1 < bw ? rg[2 * c + 2] : 0, hb = c + 1 < bw ? rg[2 * c + 3] : 0;
            if (!symdiff_extremes(la, ha, lb, hb, mn, mx)) continue;
            mn *= 2; mx *= 2;
        } else {
            const int lo = rg[X], hi = rg[X + 1];
            if (hi <= lo) continue;
            mn = 2 * lo - 1; mx = 2 * hi - 1;
        }
        chains_push(f.LX, f.LY, f.UX, f.UY, nl, nu, X, mn, mx);
    }
    f.nl = nl; f.nu = nu;
    unsigned long long best = 0;
    for (int a = 0; a < f.nl + f.nu; a++) {
        const i64 ax = a < f.nl ? f.LX[a] : f.UX[a - f.nl], ay = a < f.nl ? f.LY[a] : f.UY[a - f.nl];
        for (int b = a + 1; b < f.nl + f.nu; b++) {
            const i64 dx = (b < f.nl ? f.LX[b] : f.UX[b - f.nl]) - ax, dy = (b < f.nl ? f.LY[b] : f.UY[b - f.nl]) - ay;
            best = max(best, (unsigned long long)(dx * dx + dy * dy));
        }
    }
    feret_d2[i] = best;
}

extern "C" int ampis_crop_convex_feret(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox,
                                       int32_t n, const int64_t *d_scratch_off, int32_t *d_scratch,
                                       const int64_t *d_col_off, int32_t *d_ranges, uint64_t *d_feret_d2,
                                       void *stream)
{
    AMPIS_REQUIRE(n >= 0, "n < 0");
    if (n == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_bits && d_bits_off && d_bbox && d_scratch_off && d_scratch && d_col_off && d_ranges && d_feret_d2,
                  "null pointer");
    crop_convex_feret_kernel<<<(unsigned)((n + 127) / 128), 128, 0, as_stream(stream)>>>(
        (const u32 *)d_bits, d_bits_off, (const int4 *)d_bbox, n, d_scratch_off, d_scratch, d_col_off, d_ranges,
        (unsigned long long *)d_feret_d2);
    AMPIS_CHECK_LAUNCH("crop_convex_feret_kernel");
    return AMPIS_OK;
}

// ---- CROP window -> row-major bool box image: block per mask ---------------------------------------
// img[img_off[i] + r * bw + c] = pixel (y0 + r, x0 + c), 0 / 1 bytes, bh * bw bytes per mask.
__global__ void __launch_bounds__(256)
crop_unpack_image_kernel(const u32 *__restrict__ bits, const i64 *__restrict__ bits_off, const int4 *__restrict__ bbox,
                         const i64 *__restrict__ img_off, uint8_t *__restrict__ img)
{
    const int i = blockIdx.x;
    const Win w = win_of(bits, bits_off, bbox, i);
    if (!w.nwy) return;
    const int4 bb = bbox[i];
    const u32 bw = (u32)(bb.z - bb.x + 1);
    const i64 total = (i64)(bb.w - bb.y + 1) * bw;
    uint8_t *out = img + img_off[i];
    for (i64 idx = threadIdx.x; idx < total; idx += blockDim.x) {
        const u32 r = (u32)(idx / bw), c = (u32)(idx - (i64)r * bw);
        const u32 y = (u32)bb.y + r;
        out[idx] = (uint8_t)((__ldg(w.W + c * w.nwy + ((y >> 5) - w.wy0)) >> (y & 31u)) & 1u);
    }
}

extern "C" int ampis_crop_unpack_image(const void *d_bits, const int64_t *d_bits_off, const int32_t *d_bbox,
                                       int32_t n, const int64_t *d_img_off, uint8_t *d_img, void *stream)
{
    AMPIS_REQUIRE(n >= 0, "n < 0");
    if (n == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_bits && d_bits_off && d_bbox && d_img_off && d_img, "null pointer");
    crop_unpack_image_kernel<<<(unsigned)n, 256, 0, as_stream(stream)>>>((const u32 *)d_bits, d_bits_off,
                                                                         (const int4 *)d_bbox, d_img_off, d_img);
    AMPIS_CHECK_LAUNCH("crop_unpack_image_kernel");
    return AMPIS_OK;
}

// ==== intensity properties (regionprops with intensity_image) ==========================================
// Warp per mask over its run table: the lanes walk the 1-runs together, cut at column boundaries into vertical
// segments, and read the pixels of a segment side by side -- coalesced, because the image is column-major on the
// device (pixel (row y, column x) at x * h + y, the order of the run positions).  Per column every lane keeps
// P[p] = sum I r^p of its pixels; when the column changes, P is folded into S[p][q] += P[p] c^q.
//   integer pixels: exact.  A lane may read any subset of the rows of a column (a column of many short segments
//     restarts every segment at lane 0), so its P[p] is bounded by the whole column: |P[3]| <= 2^64 sum_{r<2^16} r^3
//     < 2^126, inside the signed 128-bit P and i192_add_prod's mag < 2^127.  S[p][q] < 2^64 (sum_r r^3) (sum_c c^3)
//     < 2^188 is kept as a signed 192-bit integer.  8- and 16-bit pixels take their products I r^p in 64 bits.
//   float pixels: float64 sums, about a given centre (the second, central pass) or about (0, 0).
typedef __int128 i128;

template <typename T> struct PixFloat {
    static constexpr bool value = std::is_floating_point<T>::value || std::is_same<T, __half>::value;
};
template <typename T> __device__ __forceinline__ double pix_f64(T v) { return (double)v; }
template <> __device__ __forceinline__ double pix_f64<__half>(__half v) { return (double)__half2float(v); }

// signed 192-bit integer in two's complement: lo = bits 0..127, hi = bits 128..191
struct I192 {
    u128 lo;
    u64 hi;
};

// s += (neg ? -1 : 1) * mag * m  (mag < 2^127, m < 2^64)
__device__ __forceinline__ void i192_add_prod(I192 &s, u128 mag, u64 m, bool neg)
{
    const u128 a = (u128)(u64)mag * m, b = (u128)(u64)(mag >> 64) * m;      // mag * m = a + b 2^64
    const u128 lo = a + (b << 64);
    const u64 hi = (u64)(b >> 64) + (lo < a ? 1u : 0u);
    if (neg) {
        const u128 t = s.lo - lo;
        s.hi -= hi + (t > s.lo ? 1u : 0u);
        s.lo = t;
    } else {
        const u128 t = s.lo + lo;
        s.hi += hi + (t < s.lo ? 1u : 0u);
        s.lo = t;
    }
}

__device__ __forceinline__ void i192_shfl_add(I192 &s, int d)
{
    const u128 olo = shfl_xor_u128(s.lo, d);
    const u64 ohi = __shfl_xor_sync(0xffffffffu, s.hi, d);
    const u128 t = s.lo + olo;
    s.hi += ohi + (t < s.lo ? 1u : 0u);
    s.lo = t;
}

// I * rp exactly (rp < 2^48)
template <typename T> __device__ __forceinline__ i128 pix_mul(T v, u64 rp)
{
    if constexpr (sizeof(T) <= 2) {
        if constexpr (std::is_signed<T>::value) return (i128)((i64)v * (i64)rp);      // |I rp| < 2^63
        else return (i128)((u64)v * rp);                                              // I rp < 2^64
    } else if constexpr (std::is_signed<T>::value) {
        const u64 mag = v < 0 ? (u64)0 - (u64)(i64)v : (u64)(i64)v;
        const i128 p = (i128)((u128)mag * rp);
        return v < 0 ? -p : p;
    } else {
        return (i128)((u128)(u64)v * rp);
    }
}

template <typename T, bool FLT = PixFloat<T>::value, bool SIGNED = std::is_signed<T>::value>
struct PixStats;                                    // min / max in the widest type of the pixel's kind
template <typename T, bool SIGNED> struct PixStats<T, true, SIGNED> {
    typedef double W;
    static __device__ __forceinline__ W lo() { return -CUDART_INF; }
    static __device__ __forceinline__ W hi() { return CUDART_INF; }
};
template <typename T> struct PixStats<T, false, true> {
    typedef long long W;
    static __device__ __forceinline__ W lo() { return LLONG_MIN; }
    static __device__ __forceinline__ W hi() { return LLONG_MAX; }
};
template <typename T> struct PixStats<T, false, false> {
    typedef unsigned long long W;
    static __device__ __forceinline__ W lo() { return 0; }
    static __device__ __forceinline__ W hi() { return ULLONG_MAX; }
};

// moments: integer pixels 48 u64 per mask (M[p][q] as 3 limbs, low first, k = 4p + q), float pixels 16 f64.
// stats (raw pass only; 4 x 8 bytes per mask): min, max (long long / unsigned long long / double; NaN when the
// mask holds a NaN pixel), non-finite pixels of the mask, non-finite pixels of the box (0 unless scan_box).
template <typename T>
__global__ void __launch_bounds__(256)
rle_intensity_kernel(const u32 *__restrict__ cum, const i64 *__restrict__ cnt_off, const int *__restrict__ cnt_len,
                     const u32 *__restrict__ hh, const int4 *__restrict__ bbox, int n, const T *__restrict__ img,
                     const double *__restrict__ center, int scan_box, void *__restrict__ moments,
                     unsigned long long *__restrict__ stats)
{
    constexpr bool FLT = PixFloat<T>::value;
    typedef typename PixStats<T>::W W;
    typedef typename std::conditional<FLT, double, i128>::type Part;
    typedef typename std::conditional<FLT, double, I192>::type Sum;
    const int i = (int)((blockIdx.x * (u32)blockDim.x + threadIdx.x) >> 5);
    if (i >= n) return;
    const u32 lane = lane_id();
    const u32 *C = cum + cnt_off[i];
    const int m = cnt_len[i];
    const u64 H = hh[i];
    const int4 bb = bbox[i];
    const double cr = center ? center[2 * (i64)i] : 0.0, cc = center ? center[2 * (i64)i + 1] : 0.0;
    Part P[4];
    Sum S[16];
#pragma unroll
    for (int k = 0; k < 4; k++) P[k] = Part();
#pragma unroll
    for (int k = 0; k < 16; k++) S[k] = Sum();
    W mn = PixStats<T>::hi(), mx = PixStats<T>::lo();
    bool nan = false;
    unsigned long long nf_mask = 0, nf_box = 0;

    auto fold = [&](int x) {                       // S[p][q] += P[p] c^q, P = 0
        if constexpr (FLT) {
            const double c = (double)(x - bb.x) - cc, c2 = c * c;
            const double cq[4] = {1.0, c, c2, c2 * c};
#pragma unroll
            for (int p = 0; p < 4; p++) {
#pragma unroll
                for (int q = 0; q < 4; q++) S[4 * p + q] += q ? P[p] * cq[q] : P[p];
                P[p] = 0.0;
            }
        } else {
            const u64 c = (u64)(x - bb.x);
            const u64 cq[4] = {1, c, c * c, c * c * c};
#pragma unroll
            for (int p = 0; p < 4; p++) {
                const bool neg = P[p] < 0;
                const u128 mag = neg ? (u128)0 - (u128)P[p] : (u128)P[p];
#pragma unroll
                for (int q = 0; q < 4; q++) i192_add_prod(S[4 * p + q], mag, cq[q], neg);
                P[p] = 0;
            }
        }
    };

    int col = -1;
    for (int r = 1; r < m; r += 2) {                               // odd runs are the 1-runs; warp-uniform
        u64 p = C[r - 1];
        const u64 e = C[r];
        while (p < e) {
            const u64 x = p / H, cs = x * H;
            const u64 b = min(e, cs + H) - cs;                     // rows [p - cs, b) of column x
            if ((int)x != col) {
                if (col >= 0) fold(col);
                col = (int)x;
            }
            for (u64 y = p - cs + lane; y < b; y += 32) {
                const T v = img[cs + y];
                const u32 rl = (u32)y - (u32)bb.y;
                if constexpr (FLT) {
                    const double w = pix_f64(v);
                    if (!center) {
                        if (isnan(w)) nan = true;
                        if (!isfinite(w)) nf_mask++;
                        mn = fmin(mn, w);
                        mx = fmax(mx, w);
                    }
                    const double d = (double)rl - cr, d2 = d * d;
                    P[0] += w;
                    P[1] += w * d;
                    P[2] += w * d2;
                    P[3] += w * (d2 * d);
                } else {
                    const W w = (W)v;
                    mn = min(mn, w);
                    mx = max(mx, w);
                    const u64 r2 = (u64)rl * rl;
                    P[0] += pix_mul(v, 1);
                    P[1] += pix_mul(v, rl);
                    P[2] += pix_mul(v, r2);
                    P[3] += pix_mul(v, r2 * rl);
                }
            }
            p = cs + H;
        }
    }
    if (col >= 0) fold(col);
    if constexpr (FLT) {
        if (!center && scan_box) {                                 // skimage multiplies the whole box by the mask:
            for (int x = bb.x; x <= bb.z; x++) {                   // a NaN or inf outside the mask turns into NaN
                for (u32 y = (u32)bb.y + lane; y <= (u32)bb.w; y += 32)
                    if (!isfinite(pix_f64(img[(u64)x * H + y]))) nf_box++;
            }
        }
    }

#pragma unroll
    for (int k = 0; k < 16; k++) {
#pragma unroll
        for (int d = 16; d; d >>= 1) {
            if constexpr (FLT) S[k] += __shfl_xor_sync(0xffffffffu, S[k], d);
            else i192_shfl_add(S[k], d);
        }
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        const W omn = __shfl_xor_sync(0xffffffffu, mn, d), omx = __shfl_xor_sync(0xffffffffu, mx, d);
        if constexpr (FLT) { mn = fmin(mn, omn); mx = fmax(mx, omx); }
        else { mn = min(mn, omn); mx = max(mx, omx); }
        nf_mask += __shfl_xor_sync(0xffffffffu, nf_mask, d);
        nf_box += __shfl_xor_sync(0xffffffffu, nf_box, d);
    }
    nan = __any_sync(0xffffffffu, nan);
    if (lane != 0) return;
    if constexpr (FLT) {
        double *M = (double *)moments + 16 * (i64)i;
#pragma unroll
        for (int k = 0; k < 16; k++) M[k] = S[k];
        if (nan) mn = mx = CUDART_NAN;
    } else {
        unsigned long long *M = (unsigned long long *)moments + 48 * (i64)i;
#pragma unroll
        for (int k = 0; k < 16; k++) {
            M[3 * k] = (unsigned long long)S[k].lo;
            M[3 * k + 1] = (unsigned long long)(S[k].lo >> 64);
            M[3 * k + 2] = S[k].hi;
        }
    }
    if (stats) {
        unsigned long long *st = stats + 4 * (i64)i;
        memcpy(&st[0], &mn, 8);
        memcpy(&st[1], &mx, 8);
        st[2] = nf_mask;
        st[3] = nf_box;
    }
}

template <typename T>
static int launch_intensity(const uint32_t *d_cum, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                            const uint32_t *d_h, const int32_t *d_bbox, int32_t n, const void *d_img,
                            const double *d_center, int32_t scan_box, void *d_moments, uint64_t *d_stats,
                            void *stream)
{
    rle_intensity_kernel<T><<<(unsigned)(((i64)n * 32 + 255) / 256), 256, 0, as_stream(stream)>>>(
        d_cum, d_cnt_off, d_cnt_len, d_h, (const int4 *)d_bbox, n, (const T *)d_img, d_center, scan_box, d_moments,
        (unsigned long long *)d_stats);
    AMPIS_CHECK_LAUNCH("rle_intensity_kernel");
    return AMPIS_OK;
}

extern "C" int ampis_rle_intensity(const uint32_t *d_cum, const int64_t *d_cnt_off, const int32_t *d_cnt_len,
                                   const uint32_t *d_h, const int32_t *d_bbox, int32_t n, const void *d_img,
                                   int32_t pix, const double *d_center, int32_t scan_box, void *d_moments,
                                   uint64_t *d_stats,
                                   void *stream)
{
    AMPIS_REQUIRE(n >= 0, "n < 0");
    AMPIS_REQUIRE(pix >= AMPIS_PIX_U8 && pix <= AMPIS_PIX_F64, "unknown pixel type");
    AMPIS_REQUIRE(!d_center || pix >= AMPIS_PIX_F16, "central sums are for float pixels only");
    AMPIS_REQUIRE(d_center || d_stats, "the raw pass writes the statistics");
    if (n == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_cum && d_cnt_off && d_cnt_len && d_h && d_bbox && d_img && d_moments, "null pointer");
    switch (pix) {
    case AMPIS_PIX_U8: return launch_intensity<uint8_t>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    case AMPIS_PIX_I8: return launch_intensity<int8_t>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    case AMPIS_PIX_U16: return launch_intensity<uint16_t>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    case AMPIS_PIX_I16: return launch_intensity<int16_t>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    case AMPIS_PIX_U32: return launch_intensity<uint32_t>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    case AMPIS_PIX_I32: return launch_intensity<int32_t>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    case AMPIS_PIX_U64: return launch_intensity<uint64_t>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    case AMPIS_PIX_I64: return launch_intensity<int64_t>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    case AMPIS_PIX_F16: return launch_intensity<__half>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    case AMPIS_PIX_F32: return launch_intensity<float>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    default: return launch_intensity<double>(d_cum, d_cnt_off, d_cnt_len, d_h, d_bbox, n, d_img, d_center, scan_box, d_moments, d_stats, stream);
    }
}
