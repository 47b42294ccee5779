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
// from the windows for image / coords / filled_image.
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
