// Shared helpers for the sm_100a kernels of libampis_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/ampis_b200.h"

typedef uint32_t u32;
typedef uint64_t u64;
typedef int64_t i64;

// rows of a group one CTA of the rows kernels handles (blk_grp / blk_row0 lists are shared by all of them;
// ampis_rows_per_block() reports it to the host)
#define AMPIS_ROWS_PER_CTA 8

#define AMPIS_CHUNK_BITS 128u   // one uint4 = 128 pixels of the column-major bit vector

void ampis_set_error(const char *fmt, ...);

#define AMPIS_CHECK_LAUNCH(name)                                              \
    do {                                                                      \
        cudaError_t e__ = cudaGetLastError();                                 \
        if (e__ != cudaSuccess) {                                             \
            ampis_set_error("%s: %s", name, cudaGetErrorString(e__));         \
            return AMPIS_ECUDA;                                               \
        }                                                                     \
    } while (0)

#define AMPIS_REQUIRE(cond, msg)                                              \
    do {                                                                      \
        if (!(cond)) { ampis_set_error("%s: %s", __func__, msg); return AMPIS_EINVAL; } \
    } while (0)

static inline cudaStream_t as_stream(void *s) { return (cudaStream_t)s; }

// Column-grid entry list of the one-call entries (ampis_eval_image_host / ampis_eval_images_host), 20 bytes per entry
// (column index + box).  It holds `base` entries (16 per column + 4,096 per image: enough unless some boxes are much
// larger than the image's mean box) or a 32nd of the device workspace, whichever is more.  A grid that needs more --
// a thin diagonal across a 1024 x 1024 frame of small blobs registers in all 32 x 32 cells -- is reported as
// AMPIS_ENOSPC with a workspace whose 32nd holds it.
#define AMPIS_GRID_ENTRY_BYTES 20
static inline int64_t ampis_grid_capacity(int64_t base, int64_t d_ws_bytes)
{
    const int64_t share = d_ws_bytes / (32 * AMPIS_GRID_ENTRY_BYTES);
    return share > base ? share : base;
}
// Device workspace that leaves `rest` bytes beside the entry list and gives the list room for `entries` entries.  When
// the workspace's 32nd exceeds base, the list takes that 32nd, so `rest` must fit in the other 31 parts; 512 bytes
// cover the two 256-byte alignments of the list.
static inline int64_t ampis_ws_need_with_grid(int64_t rest, int64_t base, int64_t entries)
{
    int64_t need = rest + AMPIS_GRID_ENTRY_BYTES * base + 512;
    const int64_t shared = (rest + 512) * 32 / 31 + 32 * AMPIS_GRID_ENTRY_BYTES;
    if (shared > need) need = shared;
    const int64_t by_entries = 32 * AMPIS_GRID_ENTRY_BYTES * (entries + 1);
    if (entries > base && by_entries > need) need = by_entries;
    return need;
}

// IoU of a (row, column) pair from its intersection and the two areas, as rleIou forms it: the union in uint32 with
// wrap-around, the quotient in float64.  Every kernel that ranks a row's pairs by IoU uses this one expression, so
// their arg-maxes agree bit for bit.
__device__ __forceinline__ double pair_iou(u32 inter, u32 row_area, u32 col_area)
{
    return (double)inter / (double)(row_area + col_area - inter);
}
// AMPIS's per-row arg-max order: a higher score wins, equal scores go to the lower column index (best_c = -1: none yet)
__device__ __forceinline__ bool score_beats(double s, int k, double best_s, int best_c)
{
    return s > best_s || (s == best_s && (unsigned)k < (unsigned)best_c);
}

__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31u; }

__device__ __forceinline__ u32 warp_sum(u32 v)
{
#pragma unroll
    for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}
__device__ __forceinline__ u32 warp_min(u32 v)
{
#pragma unroll
    for (int d = 16; d; d >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, d));
    return v;
}
__device__ __forceinline__ u32 warp_max(u32 v)
{
#pragma unroll
    for (int d = 16; d; d >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, d));
    return v;
}

// Sub-warp groups of L = 8 / 16 / 32 consecutive lanes (one small mask per group): lane mask of the caller's group
// and reductions that stay inside it.
template <int L>
__device__ __forceinline__ u32 group_mask()
{
    return L == 32 ? 0xffffffffu : (((1u << (L & 31)) - 1u) << (lane_id() & ~(u32)(L - 1)));
}
template <int L>
__device__ __forceinline__ u32 group_sum(u32 v, u32 gm)
{
#pragma unroll
    for (int d = L / 2; d; d >>= 1) v += __shfl_xor_sync(gm, v, d);
    return v;
}
template <int L>
__device__ __forceinline__ u32 group_min(u32 v, u32 gm)
{
#pragma unroll
    for (int d = L / 2; d; d >>= 1) v = min(v, __shfl_xor_sync(gm, v, d));
    return v;
}
template <int L>
__device__ __forceinline__ u32 group_max(u32 v, u32 gm)
{
#pragma unroll
    for (int d = L / 2; d; d >>= 1) v = max(v, __shfl_xor_sync(gm, v, d));
    return v;
}

// Division of 32-bit positions by a per-mask constant (the image height: position -> column) without the
// ~20-instruction IDIV sequence: q = umulhi(s, floor((2^32-1)/d)) is floor(s/d) or one less.
struct FastDiv {
    u32 d, m;
};
__device__ __forceinline__ FastDiv fastdiv_make(u32 d)
{
    FastDiv f;
    f.d = d;
    f.m = 0xffffffffu / d;
    return f;
}
__device__ __forceinline__ u32 fastdiv(u32 s, const FastDiv f)
{
    u32 q = __umulhi(s, f.m);
    if (s - q * f.d >= f.d) q++;
    return q;
}

// streaming 128-bit store / load (data is written once and read by a later kernel)
__device__ __forceinline__ void st_v4_stream(uint4 *p, uint4 v)
{
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ uint4 ld_v4_nc(const uint4 *p)
{
    uint4 v;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ u32 popc_and(uint4 a, uint4 b)
{
    return __popc(a.x & b.x) + __popc(a.y & b.y) + __popc(a.z & b.z) + __popc(a.w & b.w);
}
