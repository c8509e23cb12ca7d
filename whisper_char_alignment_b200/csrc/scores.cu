// Head scoring, top-k selection and aggregation (north-star kernel 3).
// Replaces the reference's filter_attention (timing.py:13-43, a Python loop with one
// blocking .item() per head), coverage_penalty (metrics.py:99-111) and the aggregation
// branches of force_align (timing.py:84-97).  Everything stays on the device: scores ->
// ranks -> selected list -> (N, F) matrix, no host round trip in between.  Also the
// std-normalisation + mean over the alignment heads of the stock-Whisper baseline
// (default_find_alignment, timing.py:156-163).
#include "common.cuh"

namespace wca {

// Deterministic block sum (fixed shuffle tree + fixed warp order); result valid on thread 0.
__device__ __forceinline__ float block_sum_256(float v, float *scratch /* >= 8 floats */) {
    v = warp_sum(v);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    float total = 0.f;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) total += scratch[w];
    return total;
}

// grid (n_heads, n_utts), block 256 = 8 warps.  ONE pass over the (T, F) tile in chunks of 256 columns: warp w
// streams rows w, w+8, ... (two per iteration) with 128-byte coalesced loads; lane l keeps the partial column
// statistics of columns l, l+32, ... of the chunk in registers (8 of them), so a row contributes to its own norm
// (warp shuffle tree) and to the column sums at the same time.  The 8 warps' column partials are combined in a fixed
// order through shared memory at the end of every chunk (deterministic).  Rows longer than one chunk (F > 256:
// LibriSpeech-shaped utterances) accumulate their sum of squares per row in shared memory across chunks - a row always
// belongs to the same warp - so the register footprint does not grow with F (the earlier 16/32/48-column
// instantiations ran one CTA per SM at F > 1024 and reached 1.2 TB/s).
constexpr int kScoreCols = 8;                      // columns per lane and chunk
constexpr int kScoreChunk = kScoreCols * kWarp;    // 256 columns
constexpr int kScoreMaxRows = 1024;                // rows whose partial norms fit the shared buffer (Whisper caps T at 448)
__global__ void __launch_bounds__(256) head_scores_kernel(const float *__restrict__ ws,
                                                          const wca_utt_t *__restrict__ utts, float w_col,
                                                          float w_row, float w_cov, float *__restrict__ scores) {
    constexpr int kCols = kScoreCols;
    __shared__ float col_part[2 * 8 * kScoreChunk];  // [2][8 warps][256]: sum of squares, plain sum
    __shared__ float row_ss[kScoreMaxRows];
    __shared__ float scratch[8];
    const wca_utt_t u = utts[blockIdx.y];
    const int T = u.n_tokens, F = u.n_frames;
    const float *a = ws + u.ws_off + (int64_t)blockIdx.x * T * F;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    const bool need_cols = w_col > 0.f || w_cov > 0.f;
    const int n_chunks = (F + kScoreChunk - 1) / kScoreChunk;
    if (n_chunks > 1) {
        if (T > kScoreMaxRows) __trap();  // surfaces as a launch failure: never a silently wrong score
        for (int t = threadIdx.x; t < T; t += blockDim.x) row_ss[t] = 0.f;
        __syncthreads();
    }

    float row_part = 0.f;      // sum_t ||a[t,:]||_2        (timing.py:24)
    float col_part_sum = 0.f;  // sum_f ||a[:,f]||_2        (timing.py:21)
    float cov_part = 0.f;      // sum_f max(sum_t a[t,f], .5) (metrics.py:104-109)
    for (int ch = 0; ch < n_chunks; ++ch) {
        const int fbase = ch * kScoreChunk;
        float css[kCols], cs[kCols];
#pragma unroll
        for (int k = 0; k < kCols; ++k) css[k] = cs[k] = 0.f;
        constexpr int kRowsPerIter = 2;  // twice the loads in flight per lane
        for (int t0 = warp; t0 < T; t0 += warps * kRowsPerIter) {
            float p[kRowsPerIter][kCols];
#pragma unroll
            for (int i = 0; i < kRowsPerIter; ++i) {
                const int t = t0 + i * warps;
                const float *r = a + (int64_t)t * F + fbase;
#pragma unroll
                for (int k = 0; k < kCols; ++k) {
                    const int f = lane + k * kWarp;
                    p[i][k] = (t < T && fbase + f < F) ? ld_stream(r + f) : 0.f;
                }
            }
#pragma unroll
            for (int i = 0; i < kRowsPerIter; ++i) {
                float ss = 0.f;
#pragma unroll
                for (int k = 0; k < kCols; ++k) {
                    ss = fmaf(p[i][k], p[i][k], ss);
                    css[k] = fmaf(p[i][k], p[i][k], css[k]);
                    cs[k] += p[i][k];
                }
                ss = warp_sum(ss);
                const int t = t0 + i * warps;
                if (lane == 0 && t < T) {
                    if (n_chunks == 1) row_part += sqrtf(ss);
                    else row_ss[t] += ss;  // rows t = warp (mod 8) are this warp's: no other writer
                }
            }
        }
        if (need_cols) {
            float *pss = col_part, *ps = col_part + 8 * kScoreChunk;
#pragma unroll
            for (int k = 0; k < kCols; ++k) {
                pss[(warp * kCols + k) * kWarp + lane] = css[k];
                ps[(warp * kCols + k) * kWarp + lane] = cs[k];
            }
            __syncthreads();
            const int f = threadIdx.x;  // one column of the chunk per thread
            if (fbase + f < F) {
                const int k = f >> 5, l = f & 31;
                float ss = 0.f, s1 = 0.f;
                for (int w = 0; w < warps; ++w) {  // fixed order
                    ss += pss[(w * kCols + k) * kWarp + l];
                    s1 += ps[(w * kCols + k) * kWarp + l];
                }
                col_part_sum += sqrtf(ss);
                cov_part += s1 < 0.5f ? 0.5f : s1;  // a NaN column sum stays NaN, as in torch.maximum (fmaxf drops it)
            }
            if (ch + 1 < n_chunks) __syncthreads();  // the partials are overwritten by the next chunk
        }
    }
    if (n_chunks > 1) {
        __syncthreads();
        for (int t = threadIdx.x; t < T; t += blockDim.x) row_part += sqrtf(row_ss[t]);
    }
    const float row_sum = block_sum_256(row_part, scratch);
    const float col_sum = block_sum_256(col_part_sum, scratch);
    const float cov_sum = block_sum_256(cov_part, scratch);
    if (threadIdx.x == 0) {
        float score = 0.f;
        if (w_col > 0.f) score += w_col * col_sum;
        if (w_row > 0.f) score += w_row * row_sum;
        if (w_cov > 0.f) score -= w_cov * (cov_sum - (float)F * 0.5f);
        scores[u.score_off + blockIdx.x] = score;
    }
}

// Head scores from the partials the capture kernel leaves behind (wca_capture_attention with d_partials): per
// (utterance, head, block of 128 tokens, group of 32 token rows) the row term sum_t ||p[t,:]||_2 and the F column sums of
// squares.  One warp per (utterance, head): sum_f sqrt(sum over row groups) in a fixed order -- no second read of the maps.
// grid (ceil(n_heads / 4), n_utts), block 128.
__global__ void __launch_bounds__(128) scores_from_partials_kernel(const float *__restrict__ partials,
                                                                   const wca_utt_t *__restrict__ utts, int n_heads,
                                                                   float w_col, float w_row, float *__restrict__ scores) {
    const wca_utt_t u = utts[blockIdx.y];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int head = blockIdx.x * 4 + warp;
    if (head >= n_heads) return;
    const int T = u.n_tokens, F = u.n_frames, tbu = (T + 127) / 128;
    const int groups = (T + 31) / 32;  // groups of 32 token rows that exist: group g lives in token block g / 4, slot g % 4
    const float *row_part = partials + u.part_off + (int64_t)head * tbu * 4;
    const float *col_ss = partials + u.part_off + (int64_t)n_heads * tbu * 4 + (int64_t)head * tbu * 4 * F;
    float col = 0.f;
    if (w_col > 0.f)
        for (int f = lane; f < F; f += kWarp) {
            float ss = 0.f;
            for (int g = 0; g < groups; ++g) ss += col_ss[(int64_t)g * F + f];  // slots of one head are contiguous: [tb][4][F]
            col += sqrtf(ss);
        }
    col = warp_sum(col);
    if (lane == 0) {
        float score = 0.f;
        if (w_col > 0.f) score += w_col * col;
        if (w_row > 0.f) {
            float row = 0.f;
            for (int g = 0; g < groups; ++g) row += row_part[g];
            score += w_row * row;
        }
        scores[u.score_off + head] = score;
    }
}

// Ranking key of a score: an integer ordered like the float, with -0.0 == +0.0 and every NaN (any sign or payload)
// strictly below -inf.
__device__ __forceinline__ int32_t topk_key(float v) {
    if (v != v) return INT32_MIN;
    const int32_t b = __float_as_int(v == 0.f ? 0.f : v);
    return b >= 0 ? b : b ^ 0x7fffffff;  // negatives: larger magnitude, smaller key; -inf gives INT32_MIN + 2^23 - 1 > NaN's
}

// grid (n_utts), block 256, dynamic smem n_heads keys.  Rank by counting with the
// reference's tuple order (score, layer, head): ties go to the smaller head index.  The order must be TOTAL so that
// every output slot is written exactly once: a NaN score (non-finite logits upstream) compares false both ways and
// would give several heads the same rank, leaving `sel` slots uninitialised for aggregate_heads_kernel to
// dereference.  NaN ranks below every number, -inf included, and NaNs among themselves by head index (the reference's
// sorted() leaves NaN order unspecified).
__global__ void __launch_bounds__(256) topk_heads_kernel(const float *__restrict__ scores,
                                                         const wca_utt_t *__restrict__ utts, int n_heads,
                                                         int32_t *__restrict__ sel, float *__restrict__ sel_scores) {
    extern __shared__ int32_t s_key[];
    const wca_utt_t u = utts[blockIdx.x];
    for (int i = threadIdx.x; i < n_heads; i += blockDim.x)
        s_key[i] = topk_key(scores[u.score_off + i]);  // the reported score stays the original value
    __syncthreads();
    const int n_sel = u.n_sel < n_heads ? u.n_sel : n_heads;
    const int first = n_heads - n_sel;
    for (int i = threadIdx.x; i < n_heads; i += blockDim.x) {
        const int32_t ki = s_key[i];
        int rank = 0;
        for (int j = 0; j < n_heads; ++j) {
            const int32_t kj = s_key[j];
            rank += (kj < ki) || (kj == ki && j < i);
        }
        if (rank >= first) {
            sel[u.sel_off + rank - first] = i;
            if (sel_scores) sel_scores[u.sel_off + rank - first] = scores[u.score_off + i];
        }
    }
}

// grid (ceil(max_frames/32), n_utts), block 256 = 8 warps x 32 columns, dynamic smem
// T*32 floats of accumulators.  Lane <-> frame (128-byte coalesced rows), warp <-> rows.
template <int kGroup>
__global__ void __launch_bounds__(256) aggregate_heads_kernel(const float *__restrict__ ws,
                                                              const int32_t *__restrict__ sel,
                                                              const wca_utt_t *__restrict__ utts,
                                                              float *__restrict__ matrix) {
    extern __shared__ float acc_s[];  // [T][32]
    // Heads are taken kGroup at a time: their loads are in flight together and the block meets once per group instead of
    // once per head (mean aggregation walks all 384 / 640 heads: one head per barrier was a chain of ~1 us round trips,
    // 6 % of the HBM rate).  The heads of a group are still added in selection order, so the sums are unchanged bit for bit.
    // kGroup = 1 serves launches of single-head aggregations (the probe sweep: thousands of small blocks, where the 48
    // registers of the grouped code cost more in occupancy than they save).
    __shared__ float part[2][kGroup][8][kWarp];
    const wca_utt_t u = utts[blockIdx.y];
    const int T = u.n_tokens, F = u.n_frames;
    const int f0 = blockIdx.x * kWarp;
    if (f0 >= F) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    const int f = f0 + lane;
    const bool live = f < F;

    for (int t = warp; t < T; t += warps) acc_s[t * kWarp + lane] = 0.f;

    int buf = 0;
    for (int i0 = 0; i0 < u.n_sel; i0 += kGroup, buf ^= 1) {
        const float *a[kGroup];
        float ss[kGroup];
#pragma unroll
        for (int g = 0; g < kGroup; ++g) {
            const int i = min(i0 + g, u.n_sel - 1);  // past the end: a valid pointer that is never loaded from
            a[g] = ws + u.ws_off + (int64_t)sel[u.sel_off + i] * T * F + f;
            ss[g] = 0.f;
        }
        const int ng = min(kGroup, u.n_sel - i0);  // single-head aggregations (the probe sweep) must not load four times
        if (live)
            for (int t = warp; t < T; t += warps) {
                float p[kGroup];
#pragma unroll
                for (int g = 0; g < kGroup; ++g) p[g] = g < ng ? a[g][(int64_t)t * F] : 0.f;
#pragma unroll
                for (int g = 0; g < kGroup; ++g) ss[g] = fmaf(p[g], p[g], ss[g]);
            }
#pragma unroll
        for (int g = 0; g < kGroup; ++g)
            if (g < ng) part[buf][g][warp][lane] = ss[g];
        __syncthreads();
        float cn[kGroup];
#pragma unroll
        for (int g = 0; g < kGroup; ++g) {
            cn[g] = 1.f;
            if (g < ng) {  // (block-uniform)
                float tot = 0.f;
#pragma unroll
                for (int w = 0; w < 8; ++w) tot += (w < warps) ? part[buf][g][w][lane] : 0.f;
                cn[g] = sqrtf(tot);  // ||a_i[:, f]||_2 over all T rows (timing.py:86 / :96)
            }
        }
        if (live)
            for (int t = warp; t < T; t += warps) {
                float p[kGroup];
#pragma unroll
                for (int g = 0; g < kGroup; ++g) p[g] = g < ng ? a[g][(int64_t)t * F] : 0.f;
                float acc = acc_s[t * kWarp + lane];
#pragma unroll
                for (int g = 0; g < kGroup; ++g)
                    if (g < ng) acc += p[g] / cn[g];
                acc_s[t * kWarp + lane] = acc;
            }
    }

    // rows are accumulated by warp (t % warps) but written out by warp ((t - row_begin) % warps)
    __syncthreads();
    const float count = (float)u.n_sel;  // torch.mean = sum / count
    if (live)
        for (int t = u.row_begin + warp; t < u.row_end; t += warps)
            matrix[u.matrix_off + (int64_t)(t - u.row_begin) * F + f] = acc_s[t * kWarp + lane] / count;
}

// Std-normalisation of the alignment heads + mean over heads: the stock-Whisper baseline (timing.py:156-163).
// grid (ceil(max_frames/32), n_utts), block 256 = 8 warps x 32 columns, dynamic smem T*32 floats of accumulators.
// Heads are taken 8 at a time.  Statistics: warp g owns head i0 + g and its lanes walk their whole column (lane <-> frame,
// 128-byte coalesced rows) twice, first for the mean, then for the squared deviations from it; each pass keeps 8
// partial sums (rows t mod 8, independent add chains) combined in a fixed order, so the result depends on nothing but
// the column.  The mean is taken of the shifted values a[t,f] - a[0,f]: exact for a constant column (sd = 0, so 0/0
// gives NaN as in torch) and free of the cancellation of a large mean over a small spread.  Normalisation: warps walk
// the rows of the group's columns (re-reads come from L1/L2) and add the group's heads, in list order, into the
// shared accumulators.
constexpr int kNormGroup = 8;             // heads whose statistics one round computes (one per warp)
constexpr int kNormMaxTokens = 448;       // Whisper's n_text_ctx: 56 KB of accumulators
__global__ void __launch_bounds__(256) normalize_heads_kernel(const float *__restrict__ ws,
                                                              const int32_t *__restrict__ sel,
                                                              const wca_utt_t *__restrict__ utts, int max_tokens,
                                                              float *__restrict__ weights,
                                                              const int64_t *__restrict__ weights_off,
                                                              float *__restrict__ matrix) {
    extern __shared__ float acc_s[];  // [T][32]
    __shared__ float stat[2][2][kNormGroup][kWarp];  // [buffer][mean, sd][head of the group][lane]
    const wca_utt_t u = utts[blockIdx.y];
    const int T = u.n_tokens, F = u.n_frames;
    // a descriptor the accumulators cannot hold, or with no head / a row range outside [0, T): a launch failure,
    // never a silently wrong matrix
    if (T < 1 || T > max_tokens || u.n_sel < 1 || u.row_begin < 0 || u.row_end < u.row_begin || u.row_end > T) __trap();
    const int f0 = blockIdx.x * kWarp;
    if (f0 >= F) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    const int f = f0 + lane;
    const bool live = f < F;
    const int64_t plane = (int64_t)T * F;
    float *w_out = weights ? weights + weights_off[blockIdx.y] : nullptr;

    for (int t = warp; t < T; t += warps) acc_s[t * kWarp + lane] = 0.f;

    int buf = 0;
    for (int i0 = 0; i0 < u.n_sel; i0 += kNormGroup, buf ^= 1) {
        const int ng = min(kNormGroup, u.n_sel - i0);
        if (warp < ng && live) {
            const float *a = ws + u.ws_off + (int64_t)sel[u.sel_off + i0 + warp] * plane + f;
            const float a0 = a[0];
            float s[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) s[j] = 0.f;
            int t = 0;
            for (; t + 8 <= T; t += 8) {
                float p[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) p[j] = a[(int64_t)(t + j) * F];
#pragma unroll
                for (int j = 0; j < 8; ++j) s[j] += p[j] - a0;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (t + j < T) s[j] += a[(int64_t)(t + j) * F] - a0;
            const float mean = a0 + (((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]))) / (float)T;
#pragma unroll
            for (int j = 0; j < 8; ++j) s[j] = 0.f;
            for (t = 0; t + 8 <= T; t += 8) {
                float p[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) p[j] = a[(int64_t)(t + j) * F] - mean;
#pragma unroll
                for (int j = 0; j < 8; ++j) s[j] = fmaf(p[j], p[j], s[j]);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (t + j < T) {
                    const float d = a[(int64_t)(t + j) * F] - mean;
                    s[j] = fmaf(d, d, s[j]);
                }
            const float var = (((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]))) / (float)T;
            stat[buf][0][warp][lane] = mean;
            stat[buf][1][warp][lane] = sqrtf(var);  // population std (unbiased=False, timing.py:160)
        }
        __syncthreads();  // the statistics of this group; the other buffer is still read by no one
        if (live) {
            const float *a[kNormGroup];
            float mu[kNormGroup], sd[kNormGroup];
#pragma unroll
            for (int g = 0; g < kNormGroup; ++g) {
                const int i = min(i0 + g, u.n_sel - 1);  // past the end: a valid pointer that is never loaded from
                a[g] = ws + u.ws_off + (int64_t)sel[u.sel_off + i] * plane + f;
                mu[g] = stat[buf][0][g][lane];
                sd[g] = stat[buf][1][g][lane];
            }
            for (int t = warp; t < T; t += warps) {
                float acc = acc_s[t * kWarp + lane];
#pragma unroll
                for (int g = 0; g < kNormGroup; ++g)
                    if (g < ng) {
                        const float w = (a[g][(int64_t)t * F] - mu[g]) / sd[g];  // true division: 0/0 is NaN (timing.py:161)
                        if (w_out) w_out[(int64_t)(i0 + g) * plane + (int64_t)t * F + f] = w;
                        acc += w;
                    }
                acc_s[t * kWarp + lane] = acc;
            }
        }
        // the next group writes the other statistics buffer, so one barrier per group suffices: a warp that reaches
        // the next group's barrier has finished reading this group's buffer, and buffer `buf` is only written again
        // after that barrier
    }

    // rows are accumulated by warp (t % warps) but written out by warp ((t - row_begin) % warps)
    __syncthreads();
    const float count = (float)u.n_sel;  // torch.mean = sum / count (timing.py:163)
    if (live)
        for (int t = u.row_begin + warp; t < u.row_end; t += warps)
            matrix[u.matrix_off + (int64_t)(t - u.row_begin) * F + f] = acc_s[t * kWarp + lane] / count;
}

int launch_head_scores(const float *d_ws, const wca_utt_t *d_utts, int n_utts, int n_heads, int max_frames, float w_col,
                       float w_row, float w_cov, float *d_scores, cudaStream_t stream) {
    (void)max_frames;  // any row length: the kernel walks it in chunks of 256 columns
    head_scores_kernel<<<dim3(n_heads, n_utts), 256, 0, stream>>>(d_ws, d_utts, w_col, w_row, w_cov, d_scores);
    WCA_LAUNCH_CHECK("head_scores_kernel");
    return WCA_OK;
}

int launch_scores_from_partials(const float *d_partials, const wca_utt_t *d_utts, int n_utts, int n_heads, float w_col,
                                float w_row, float *d_scores, cudaStream_t stream) {
    scores_from_partials_kernel<<<dim3((n_heads + 3) / 4, n_utts), 128, 0, stream>>>(d_partials, d_utts, n_heads, w_col,
                                                                                      w_row, d_scores);
    WCA_LAUNCH_CHECK("scores_from_partials_kernel");
    return WCA_OK;
}

int launch_topk_heads(const float *d_scores, const wca_utt_t *d_utts, int n_utts, int n_heads, int32_t *d_sel,
                      float *d_sel_scores, cudaStream_t stream) {
    topk_heads_kernel<<<n_utts, 256, n_heads * sizeof(int32_t), stream>>>(d_scores, d_utts, n_heads, d_sel,
                                                                           d_sel_scores);
    WCA_LAUNCH_CHECK("topk_heads_kernel");
    return WCA_OK;
}

int launch_aggregate_heads(const float *d_ws, const int32_t *d_sel, const wca_utt_t *d_utts, int n_utts,
                           int max_tokens, int max_frames, int max_sel, float *d_matrix, cudaStream_t stream) {
    const size_t smem = (size_t)max_tokens * kWarp * sizeof(float);
    if (smem > 200u * 1024u) {
        set_error("wca_aggregate_heads: max_tokens=%d exceeds the shared-memory accumulator", max_tokens);
        return WCA_ERR_UNSUPPORTED;
    }
    // the 48 KB a kernel gets without opting in cover static + dynamic shared memory: this kernel has 2 KB of static
    // partials, so 369-384 token rows (46-48 KB of accumulators) already need the attribute
    // (8 KB of static partials in the grouped instantiation)
    const dim3 grid((max_frames + kWarp - 1) / kWarp, n_utts);
    if (max_sel <= 1) {
        if (smem > 40u * 1024u)
            WCA_CUDA(cudaFuncSetAttribute(aggregate_heads_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        aggregate_heads_kernel<1><<<grid, 256, smem, stream>>>(d_ws, d_sel, d_utts, d_matrix);
    } else {
        if (smem > 32u * 1024u)
            WCA_CUDA(cudaFuncSetAttribute(aggregate_heads_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        aggregate_heads_kernel<4><<<grid, 256, smem, stream>>>(d_ws, d_sel, d_utts, d_matrix);
    }
    {
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) {
            set_error("aggregate_heads_kernel: %s (grid %u x %u, %zu bytes of shared memory, max_tokens %d, max_frames %d)",
                      cudaGetErrorString(e), grid.x, grid.y, smem, max_tokens, max_frames);
            return WCA_ERR_CUDA;
        }
        count_launch();
    }
    return WCA_OK;
}

int launch_normalize_heads(const float *d_ws, const int32_t *d_sel, const wca_utt_t *d_utts, int n_utts, int max_tokens,
                           int max_frames, float *d_weights, const int64_t *d_weights_off, float *d_matrix,
                           cudaStream_t stream) {
    if (max_tokens > kNormMaxTokens) {
        set_error("wca_normalize_heads: max_tokens=%d exceeds the %d token rows of the shared-memory accumulator",
                  max_tokens, kNormMaxTokens);
        return WCA_ERR_UNSUPPORTED;
    }
    const size_t smem = (size_t)max_tokens * kWarp * sizeof(float);
    // 4 KB of static statistics: from 353 token rows on, the accumulators need the opt-in beyond 48 KB
    if (smem > 44u * 1024u)
        WCA_CUDA(cudaFuncSetAttribute(normalize_heads_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const dim3 grid((max_frames + kWarp - 1) / kWarp, n_utts);
    normalize_heads_kernel<<<grid, 256, smem, stream>>>(d_ws, d_sel, d_utts, max_tokens, d_weights, d_weights_off, d_matrix);
    WCA_LAUNCH_CHECK("normalize_heads_kernel");
    return WCA_OK;
}

}  // namespace wca
