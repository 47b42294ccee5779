// Matching summaries and histograms: the small reductions that follow the row kernel.
#include <algorithm>

#include "common.cuh"

// One CTA per group (image).  AMPIS's matcher (analyze.py:166-174): a GT is a true positive
// when its best IoU is strictly above the threshold, otherwise a false negative; predictions
// never chosen by a true-positive GT are false positives (several GTs may share a prediction).
// The arg-max is threshold independent, so all thresholds are served by one row pass.
__global__ void __launch_bounds__(256)
match_counts_kernel(const int *__restrict__ best_col, const double *__restrict__ best_score,
                    const int *__restrict__ grp_row_begin, const int *__restrict__ grp_row_count,
                    const int *__restrict__ grp_col_count, const double *__restrict__ thresh, int n_thresh,
                    int *__restrict__ grp_counts, unsigned long long *__restrict__ totals)
{
    extern __shared__ u32 taken[];   // bitmap over the group's predictions
    __shared__ int s_tp, s_used;
    const int g = blockIdx.x;
    const int r0 = grp_row_begin[g], G = grp_row_count[g], P = grp_col_count[g];
    const int words = (P + 31) / 32;
    for (int t = 0; t < n_thresh; t++) {
        const double th = thresh[t];
        for (int k = threadIdx.x; k < words; k += blockDim.x) taken[k] = 0u;
        if (threadIdx.x == 0) { s_tp = 0; s_used = 0; }
        __syncthreads();
        int tp = 0;
        for (int k = threadIdx.x; k < G; k += blockDim.x) {
            const int c = best_col[r0 + k];
            if (best_score[r0 + k] > th && c >= 0) {
                tp++;
                atomicOr(&taken[c >> 5], 1u << (c & 31));
            }
        }
        tp = (int)warp_sum((u32)tp);
        if (lane_id() == 0 && tp) atomicAdd(&s_tp, tp);
        __syncthreads();
        int used = 0;
        for (int k = threadIdx.x; k < words; k += blockDim.x) used += __popc(taken[k]);
        used = (int)warp_sum((u32)used);
        if (lane_id() == 0 && used) atomicAdd(&s_used, used);
        __syncthreads();
        if (threadIdx.x == 0) {
            const int TP = s_tp, FP = P - s_used, FN = G - s_tp;
            int *o = grp_counts + ((i64)g * n_thresh + t) * 3;
            o[0] = TP; o[1] = FP; o[2] = FN;
            if (totals) {
                atomicAdd(totals + 3 * t + 0, (unsigned long long)TP);
                atomicAdd(totals + 3 * t + 1, (unsigned long long)FP);
                atomicAdd(totals + 3 * t + 2, (unsigned long long)FN);
            }
        }
        __syncthreads();
    }
}

extern "C" int ampis_match_counts(const int32_t *d_best_col, const double *d_best_score,
                                  const int32_t *d_grp_row_begin, const int32_t *d_grp_row_count,
                                  const int32_t *d_grp_col_count, int32_t n_groups, int32_t max_cols,
                                  const double *d_thresh, int32_t n_thresh, int32_t *d_grp_counts,
                                  int64_t *d_totals, void *stream)
{
    AMPIS_REQUIRE(n_groups >= 0 && n_thresh >= 0 && max_cols >= 0, "negative size");
    if (n_groups == 0 || n_thresh == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_best_col && d_best_score && d_grp_row_begin && d_grp_row_count && d_grp_col_count &&
                      d_thresh && d_grp_counts, "null pointer");
    const size_t smem = (size_t)((max_cols + 31) / 32 + 1) * sizeof(u32);
    AMPIS_REQUIRE(smem <= 200 * 1024, "too many columns per group for the shared bitmap");
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(match_counts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    match_counts_kernel<<<n_groups, 256, smem, as_stream(stream)>>>(
        d_best_col, d_best_score, d_grp_row_begin, d_grp_row_count, d_grp_col_count, d_thresh, n_thresh,
        d_grp_counts, (unsigned long long *)d_totals);
    AMPIS_CHECK_LAUNCH("match_counts_kernel");
    return AMPIS_OK;
}

// ---- score-threshold sweep -----------------------------------------------------------------------------------------
// A prediction's LEVEL is the number of (sorted) score thresholds strictly below its score: it is kept at sorted
// threshold k iff level > k.  Dropping predictions only changes which of a row's candidate pairs wins, so the whole
// (score threshold x IoU threshold) grid is read off the pairs of one join.
//
// sweep_rows_kernel, one thread per row: the row's STAIRCASE, the points where its best kept prediction changes.
// Entry 0 is the best pair among all kept ones (level >= 1); it stays the best for every k < its level.  Entry i+1 is
// the best pair among those of a higher level than entry i, and so on.  Levels strictly increase along the staircase,
// so the entry active at k is the first one whose level exceeds k.  A row has at most as many entries as pairs: the
// staircase lies at the row's offset of the pair list, in the descriptor array the AND+popc pass no longer needs, and
// a zero entry ends it when it is shorter.  Entry: (level | IoU level << 16, prediction index in the image,
// intersection, prediction area); the IoU level is the number of IoU thresholds strictly below the pair's IoU.
// Each entry costs one walk over the row's pairs, so a row costs cnt x S pair visits with S <= min(cnt, K) entries.
// Rows have a few pairs; S stays small when scores rise with IoU, and only reaches cnt when every higher-scored
// prediction of the row overlaps it less -- on a crowded frame with many score levels that is quadratic in cnt.
__global__ void __launch_bounds__(128)
sweep_rows_kernel(const u32 *__restrict__ area, const int *__restrict__ row_mask, const int *__restrict__ row_grp,
                  int n_rows, const int *__restrict__ grp_row_begin, const int *__restrict__ grp_row_count,
                  const int *__restrict__ grp_col_begin, const int2 *__restrict__ pair_ab,
                  const u32 *__restrict__ pair_inter, const i64 *__restrict__ row_pair_off,
                  const int *__restrict__ row_pair_cnt, const unsigned short *__restrict__ levels,
                  const double *__restrict__ iou_thresh, int n_iou, uint4 *__restrict__ stair)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int cnt = row_pair_cnt[r];
    if (cnt == 0) return;
    const int g = row_grp[r];
    const int cb = grp_col_begin[g];
    const i64 pred0 = (i64)cb - grp_row_begin[g] - grp_row_count[g];       // first prediction of the image
    const u32 ra = area[row_mask[r]];
    const i64 first = row_pair_off[r];
    int out = 0;
    for (u32 lo = 0;;) {
        double best_s = 0.0;
        int best_c = -1;
        u32 best_i = 0, best_a = 0, best_lv = 0;
        for (int i = 0; i < cnt; i++) {
            const u32 inter = __ldg(pair_inter + first + i);
            if (!inter) continue;
            const int cm = __ldg(pair_ab + first + i).y;
            const int k = cm - cb;
            const u32 lv = __ldg(levels + pred0 + k);
            if (lv <= lo) continue;
            const u32 ca = __ldg(area + cm);
            const double s = pair_iou(inter, ra, ca);
            if (score_beats(s, k, best_s, best_c)) { best_s = s; best_c = k; best_i = inter; best_a = ca; best_lv = lv; }
        }
        if (best_c < 0) break;
        u32 il = 0;
        for (int j = 0; j < n_iou; j++) il += __ldg(iou_thresh + j) < best_s;
        stair[first + out++] = make_uint4(best_lv | (il << 16), (u32)best_c, best_i, best_a);
        lo = best_lv;
    }
    if (out < cnt) stair[first + out] = make_uint4(0u, 0u, 0u, 0u);
}

// Warp-aggregated add of (1, a, b, c) into bin L of shared histograms (L = 0: nothing).  Rows of one warp mostly share
// a few bins: one shared atomic per distinct bin instead of 32 on one address.  The 32-bit values are summed as two
// 16-bit halves, which cannot overflow over 32 lanes.
__device__ __forceinline__ void sweep_bin_add(u32 L, u32 a, u32 b, u32 c, u32 *h_n, unsigned long long *h_a,
                                              unsigned long long *h_b, unsigned long long *h_c)
{
    u32 todo = __ballot_sync(0xffffffffu, L != 0u);
    while (todo) {
        const u32 Lc = __shfl_sync(0xffffffffu, L, __ffs(todo) - 1);
        const bool mine = L == Lc;
        const u32 m = __ballot_sync(0xffffffffu, mine);
        todo &= ~m;
        if (!h_a) {
            if (lane_id() == (u32)(__ffs(m) - 1)) atomicAdd(h_n + Lc, (u32)__popc(m));
            continue;
        }
        const u32 alo = __reduce_add_sync(0xffffffffu, mine ? a & 0xffffu : 0u),
                  ahi = __reduce_add_sync(0xffffffffu, mine ? a >> 16 : 0u),
                  blo = __reduce_add_sync(0xffffffffu, mine ? b & 0xffffu : 0u),
                  bhi = __reduce_add_sync(0xffffffffu, mine ? b >> 16 : 0u),
                  clo = __reduce_add_sync(0xffffffffu, mine ? c & 0xffffu : 0u),
                  chi = __reduce_add_sync(0xffffffffu, mine ? c >> 16 : 0u);
        if (lane_id() == (u32)(__ffs(m) - 1)) {
            atomicAdd(h_n + Lc, (u32)__popc(m));
            atomicAdd(h_a + Lc, ((unsigned long long)ahi << 16) + alo);
            atomicAdd(h_b + Lc, ((unsigned long long)bhi << 16) + blo);
            atomicAdd(h_c + Lc, ((unsigned long long)chi << 16) + clo);
        }
    }
}

// sweep_counts_kernel, one CTA per (image, chunk of score levels).  Per level k: every row takes its active staircase
// entry and adds it into shared histograms over IoU levels (true positives, sums of intersection, GT area and
// prediction area); every claimed prediction records the highest IoU level it is claimed at.  A pass over the
// predictions histograms those and counts the kept ones.  Suffix sums over the bins give, per IoU threshold j, the
// rows and predictions above it: TP, FP = kept - claimed, FN = G - TP and the three segmentation sums.  Per-image
// cells go to counts / seg (when given), the dataset totals are added atomically.
__global__ void __launch_bounds__(256)
sweep_counts_kernel(const uint4 *__restrict__ stair, const i64 *__restrict__ row_pair_off,
                    const int *__restrict__ row_pair_cnt, const u32 *__restrict__ area, const int *__restrict__ row_mask,
                    const int *__restrict__ grp_row_begin, const int *__restrict__ grp_row_count,
                    const int *__restrict__ grp_col_begin, const int *__restrict__ grp_col_count,
                    const unsigned short *__restrict__ levels, int n_levels, int n_iou, int levels_per_cta,
                    int *__restrict__ counts, long long *__restrict__ seg, unsigned long long *__restrict__ totals,
                    unsigned long long *__restrict__ seg_totals)
{
    extern __shared__ unsigned long long sw_smem[];
    const int B = n_iou + 1;                                          // bins: IoU levels 0 .. T
    unsigned long long *h_inter = sw_smem, *h_agt = h_inter + B, *h_apr = h_agt + B;
    u32 *h_tp = (u32 *)(h_apr + B), *h_cl = h_tp + B, *s_kept = h_cl + B, *max_l = s_kept + 1;
    const int g = blockIdx.x;
    const int r0 = grp_row_begin[g], G = grp_row_count[g], P = grp_col_count[g];
    const i64 pred0 = (i64)grp_col_begin[g] - r0 - G;
    const int k0 = blockIdx.y * levels_per_cta, k1 = min(n_levels, k0 + levels_per_cta);
    for (int i = threadIdx.x; i < B; i += blockDim.x) { h_inter[i] = h_agt[i] = h_apr[i] = 0ull; h_tp[i] = h_cl[i] = 0u; }
    for (int i = threadIdx.x; i < P; i += blockDim.x) max_l[i] = 0u;
    if (threadIdx.x == 0) *s_kept = 0u;
    __syncthreads();
    const int G32 = (G + 31) & ~31, P32 = (P + 31) & ~31;
    for (int k = k0; k < k1; k++) {
        for (int i = threadIdx.x; i < G32; i += blockDim.x) {
            u32 L = 0, inter = 0, agt = 0, apr = 0;
            const int cnt = i < G ? row_pair_cnt[r0 + i] : 0;
            if (cnt) {
                const uint4 *e = stair + row_pair_off[r0 + i];
                for (int j = 0; j < cnt; j++) {
                    const uint4 v = e[j];
                    const u32 lv = v.x & 0xffffu;
                    if (lv == 0u) break;                              // end of a short staircase
                    if (lv > (u32)k) {
                        L = v.x >> 16;
                        if (L) {
                            inter = v.z;
                            apr = v.w;
                            agt = area[row_mask[r0 + i]];
                            atomicMax(max_l + v.y, L);
                        }
                        break;
                    }
                }
            }
            sweep_bin_add(L, inter, agt, apr, h_tp, h_inter, h_agt, h_apr);
        }
        __syncthreads();
        for (int i = threadIdx.x; i < P32; i += blockDim.x) {
            u32 Lm = 0;
            bool kept = false;
            if (i < P) {
                Lm = max_l[i];
                max_l[i] = 0u;
                kept = levels[pred0 + i] > (u32)k;
            }
            const u32 nk = __popc(__ballot_sync(0xffffffffu, kept));
            if (lane_id() == 0 && nk) atomicAdd(s_kept, nk);
            sweep_bin_add(Lm, 0u, 0u, 0u, h_cl, nullptr, nullptr, nullptr);
        }
        __syncthreads();
        for (int j = threadIdx.x; j < n_iou; j += blockDim.x) {
            u32 tp = 0, cl = 0;
            unsigned long long si = 0, sg = 0, sp = 0;
            for (int L = j + 1; L < B; L++) { tp += h_tp[L]; cl += h_cl[L]; si += h_inter[L]; sg += h_agt[L]; sp += h_apr[L]; }
            const u32 fp = *s_kept - cl, fn = (u32)G - tp;
            const unsigned long long sfp = sp - si, sfn = sg - si;
            const i64 cell = ((i64)g * n_levels + k) * n_iou + j, tcell = (i64)k * n_iou + j;
            if (counts) { counts[3 * cell] = (int)tp; counts[3 * cell + 1] = (int)fp; counts[3 * cell + 2] = (int)fn; }
            if (seg) { seg[3 * cell] = (long long)si; seg[3 * cell + 1] = (long long)sfp; seg[3 * cell + 2] = (long long)sfn; }
            if (tp) atomicAdd(totals + 3 * tcell, (unsigned long long)tp);
            if (fp) atomicAdd(totals + 3 * tcell + 1, (unsigned long long)fp);
            if (fn) atomicAdd(totals + 3 * tcell + 2, (unsigned long long)fn);
            if (si) atomicAdd(seg_totals + 3 * tcell, si);
            if (sfp) atomicAdd(seg_totals + 3 * tcell + 1, sfp);
            if (sfn) atomicAdd(seg_totals + 3 * tcell + 2, sfn);
        }
        __syncthreads();
        for (int i = threadIdx.x; i < B; i += blockDim.x) { h_inter[i] = h_agt[i] = h_apr[i] = 0ull; h_tp[i] = h_cl[i] = 0u; }
        if (threadIdx.x == 0) *s_kept = 0u;
        __syncthreads();
    }
}

// (not part of the C ABI: the step of ampis_eval_images_sweep_host after the join)
int ampis_sweep_counts(const uint32_t *d_area, const int32_t *d_row_mask, const int32_t *d_row_grp,
                                  int32_t n_rows, const int32_t *d_grp_row_begin, const int32_t *d_grp_row_count,
                                  const int32_t *d_grp_col_begin, const int32_t *d_grp_col_count, int32_t n_groups,
                                  int32_t max_cols, const int32_t *d_pair_ab, const uint32_t *d_pair_inter,
                                  const int64_t *d_row_pair_off, const int32_t *d_row_pair_cnt,
                                  const uint16_t *d_levels, int32_t n_levels, const double *d_iou_thresh,
                                  int32_t n_iou, void *d_stair, int32_t *d_counts, int64_t *d_seg,
                                  int64_t *d_totals, int64_t *d_seg_totals, void *stream)
{
    AMPIS_REQUIRE(n_rows >= 0 && n_groups >= 0 && max_cols >= 0, "negative size");
    AMPIS_REQUIRE(n_levels >= 1 && n_levels <= 65535 && n_iou >= 1 && n_iou <= AMPIS_SWEEP_MAX_IOU, "bad threshold count");
    AMPIS_REQUIRE(max_cols <= AMPIS_SWEEP_MAX_PREDS, "too many predictions in one image for the shared claim table");
    if (n_groups == 0) return AMPIS_OK;
    cudaStream_t st = as_stream(stream);
    if (n_rows > 0) {
        sweep_rows_kernel<<<(unsigned)((n_rows + 127) / 128), 128, 0, st>>>(
            d_area, d_row_mask, d_row_grp, n_rows, d_grp_row_begin, d_grp_row_count, d_grp_col_begin,
            (const int2 *)d_pair_ab, d_pair_inter, d_row_pair_off, d_row_pair_cnt, (const unsigned short *)d_levels,
            d_iou_thresh, n_iou, (uint4 *)d_stair);
        AMPIS_CHECK_LAUNCH("sweep_rows_kernel");
    }
    const size_t smem = (size_t)(n_iou + 1) * 32 + 4 + (size_t)max_cols * 4;
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(sweep_counts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   (int)smem);
        if (e != cudaSuccess) {
            ampis_set_error("sweep_counts_kernel: %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
            return AMPIS_ECUDA;
        }
    }
    // enough CTAs for a few per SM: small batches split the score levels into chunks (each re-reads its staircases)
    const int sms = ampis_sm_count();
    if (sms <= 0) return AMPIS_ECUDA;
    int chunks = (int)std::min<int64_t>(n_levels, std::max<int64_t>(1, (8 * (int64_t)sms + n_groups - 1) / n_groups));
    const int per = (n_levels + chunks - 1) / chunks;
    chunks = (n_levels + per - 1) / per;
    sweep_counts_kernel<<<dim3((unsigned)n_groups, (unsigned)chunks), 256, smem, st>>>(
        (const uint4 *)d_stair, d_row_pair_off, d_row_pair_cnt, d_area, d_row_mask, d_grp_row_begin, d_grp_row_count,
        d_grp_col_begin, d_grp_col_count, (const unsigned short *)d_levels, n_levels, n_iou, per, d_counts,
        (long long *)d_seg, (unsigned long long *)d_totals, (unsigned long long *)d_seg_totals);
    AMPIS_CHECK_LAUNCH("sweep_counts_kernel");
    return AMPIS_OK;
}

// Satellite assignment (powder.py:85-96): satellite s goes to particle argmax when
// I/area(s) > thresh (NaN when area(s)==0 => unmatched).  Per particle the number of owned
// satellites feeds the satellites-per-particle histogram (powder.py:529-542).
__global__ void __launch_bounds__(256)
satellite_counts_kernel(const int *__restrict__ best_col, const u32 *__restrict__ best_inter,
                        const u32 *__restrict__ area, const int *__restrict__ row_mask,
                        const int *__restrict__ grp_row_begin, const int *__restrict__ grp_row_count,
                        const int *__restrict__ grp_col_count, double thresh, int *__restrict__ grp_counts,
                        unsigned long long *__restrict__ spp_hist, int n_bins)
{
    extern __shared__ u32 owned[];   // satellites per particle of this group
    __shared__ int s_matched, s_particles;
    const int g = blockIdx.x;
    const int r0 = grp_row_begin[g], S = grp_row_count[g], P = grp_col_count[g];
    for (int k = threadIdx.x; k < P; k += blockDim.x) owned[k] = 0u;
    if (threadIdx.x == 0) { s_matched = 0; s_particles = 0; }
    __syncthreads();
    int matched = 0;
    for (int k = threadIdx.x; k < S; k += blockDim.x) {
        const u32 a = area[row_mask[r0 + k]];
        const int c = best_col[r0 + k];
        const double score = (double)best_inter[r0 + k] / (double)a;
        if (score > thresh && c >= 0) {
            matched++;
            atomicAdd(&owned[c], 1u);
        }
    }
    matched = (int)warp_sum((u32)matched);
    if (lane_id() == 0 && matched) atomicAdd(&s_matched, matched);
    __syncthreads();
    int np = 0;
    for (int k = threadIdx.x; k < P; k += blockDim.x) {
        const u32 o = owned[k];
        if (o) {
            np++;
            if (spp_hist && n_bins > 0) atomicAdd(spp_hist + min((int)o, n_bins - 1), 1ull);
        }
    }
    np = (int)warp_sum((u32)np);
    if (lane_id() == 0 && np) atomicAdd(&s_particles, np);
    __syncthreads();
    if (threadIdx.x == 0) {
        int *o = grp_counts + (i64)g * 4;
        o[0] = s_matched; o[1] = S - s_matched; o[2] = s_particles; o[3] = P;
    }
}

extern "C" int ampis_satellite_counts(const int32_t *d_best_col, const uint32_t *d_best_inter,
                                      const uint32_t *d_area, const int32_t *d_row_mask,
                                      const int32_t *d_grp_row_begin, const int32_t *d_grp_row_count,
                                      const int32_t *d_grp_col_count, int32_t n_groups, int32_t max_cols,
                                      double thresh, int32_t *d_grp_counts, int64_t *d_spp_hist, int32_t n_bins,
                                      void *stream)
{
    AMPIS_REQUIRE(n_groups >= 0 && max_cols >= 0, "negative size");
    if (n_groups == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_best_col && d_best_inter && d_area && d_row_mask && d_grp_row_begin && d_grp_row_count &&
                      d_grp_col_count && d_grp_counts, "null pointer");
    const size_t smem = (size_t)(max_cols + 1) * sizeof(u32);
    AMPIS_REQUIRE(smem <= 200 * 1024, "too many particles per image for the shared counters");
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(satellite_counts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    satellite_counts_kernel<<<n_groups, 256, smem, as_stream(stream)>>>(
        d_best_col, d_best_inter, d_area, d_row_mask, d_grp_row_begin, d_grp_row_count, d_grp_col_count, thresh,
        d_grp_counts, (unsigned long long *)d_spp_hist, n_bins);
    AMPIS_CHECK_LAUNCH("satellite_counts_kernel");
    return AMPIS_OK;
}

// Uniform-bin histogram with per-CTA shared-memory privatisation.
__global__ void __launch_bounds__(256)
hist_u32_kernel(const u32 *__restrict__ v, i64 n, u32 lo, u32 bw, unsigned long long *__restrict__ hist,
                int n_bins)
{
    extern __shared__ u32 h[];
    for (int k = threadIdx.x; k < n_bins; k += blockDim.x) h[k] = 0u;
    __syncthreads();
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        const u32 x = v[i];
        int b = x <= lo ? 0 : (int)min((u64)(x - lo) / bw, (u64)(n_bins - 1));
        atomicAdd(&h[b], 1u);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < n_bins; k += blockDim.x)
        if (h[k]) atomicAdd(hist + k, (unsigned long long)h[k]);
}

extern "C" int ampis_hist_u32(const uint32_t *d_values, int64_t n, uint32_t lo, uint32_t bin_width,
                              int64_t *d_hist, int32_t n_bins, void *stream)
{
    AMPIS_REQUIRE(n >= 0 && n_bins > 0 && bin_width > 0, "bad size");
    AMPIS_REQUIRE(n_bins <= 12288, "at most 12288 bins");
    if (n == 0) return AMPIS_OK;
    AMPIS_REQUIRE(d_values && d_hist, "null pointer");
    int sms = ampis_sm_count();
    if (sms <= 0) return AMPIS_ECUDA;
    i64 blocks = (n + 256 * 16 - 1) / (256 * 16);
    if (blocks > (i64)sms * 8) blocks = (i64)sms * 8;
    hist_u32_kernel<<<(unsigned)blocks, 256, (size_t)n_bins * sizeof(u32), as_stream(stream)>>>(
        d_values, n, lo, bin_width, (unsigned long long *)d_hist, n_bins);
    AMPIS_CHECK_LAUNCH("hist_u32_kernel");
    return AMPIS_OK;
}
