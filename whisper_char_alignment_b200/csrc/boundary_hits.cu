// Word-boundary hits of many alignments against their reference boundaries: the reference's scoring,
//     metrics.py:22-43  eval_n1(y, y_hat, tolerance)                                  (WCA_HITS_PLAIN)
//     metrics.py:45-72  eval_n1_strict(y, y_hat, words, words_hat, tolerance)          (WCA_HITS_STRICT)
// reduced to the hit count (n_pred = len(y_hat) and n_ref = len(y) are known to the caller in both modes).
//
// One warp per problem, kWarpsPerCta problems per CTA.  y_hat of problem p is the float64 end times wca_dtw_align wrote
// at d_end_times + utts[p].word_off (utts[p].n_words of them), read in place; y is reference list utt_of[p].
//   plain:  lane 0 runs the reference's greedy in-order two-pointer loop in double; a NaN, which orders neither way,
//           stops it, as in metrics.eval_n1.
//   strict: for each predicted word in order the warp scans the reference in 32-wide chunks; lane l of chunk c tests
//           j = 32 c + l (not taken, same word id, |y[j] - y_hat[i]| <= tolerance; NaN never matches) and the lowest
//           qualifying j of the first chunk that has one is taken, which is the first j of the reference's loop.  Lane
//           l keeps bit c of the taken set for j = 32 c + l in a register, so a reference of up to 32 * 32 words needs
//           no shared memory; O(W_hyp * ceil(W_ref / 32)) per problem.
// A problem's result depends on its own inputs only, never on the batch.
#include <math.h>

#include "common.cuh"

namespace wca {

constexpr int kHitsWarpsPerCta = 8;
constexpr int kHitsMaxStrictRef = WCA_HITS_MAX_STRICT_REF_WORDS;
static_assert(kHitsMaxStrictRef == 32 * kWarp, "one 32-bit taken register per lane");

__device__ __forceinline__ bool within(double a, double b, double tol) { return fabs(a - b) <= tol; }

__global__ void __launch_bounds__(kHitsWarpsPerCta * kWarp)
    boundary_hits_kernel(const double *__restrict__ end_times, const wca_utt_t *__restrict__ utts,
                         const int32_t *__restrict__ utt_of, int n_problems, const double *__restrict__ ref_times,
                         const int64_t *__restrict__ ref_off, const int32_t *__restrict__ ref_ids,
                         const int32_t *__restrict__ hyp_ids, const int64_t *__restrict__ hyp_off, double tol, int strict,
                         int32_t *__restrict__ hits) {
    const int lane = threadIdx.x & (kWarp - 1);
    const int p = blockIdx.x * kHitsWarpsPerCta + (threadIdx.x >> 5);
    if (p >= n_problems) return;
    const int u = utt_of[p];
    const int n_hyp = max(utts[p].n_words, 0);
    const double *yh = end_times + utts[p].word_off;
    const int64_t r0 = ref_off[u];
    const int n_ref = (int)(ref_off[u + 1] - r0);
    const double *y = ref_times + r0;

    if (!strict) {
        if (lane != 0) return;
        int h = 0, i = 0, j = 0;
        while (i < n_ref && j < n_hyp) {
            const double a = y[i], b = yh[j];
            if (within(a, b, tol)) {
                ++h;
                ++i;
                ++j;
            } else if (a < b) {
                ++i;
            } else if (a > b) {
                ++j;
            } else {
                break;  // NaN orders neither way: metrics.eval_n1 stops
            }
        }
        hits[p] = h;
        return;
    }

    if (n_ref > kHitsMaxStrictRef) {  // callers check this on the host (the binding refuses it before the launch)
        if (lane == 0) hits[p] = -1;
        return;
    }
    const int32_t *rid = ref_ids + r0;
    const int32_t *hid = hyp_ids + hyp_off[u];
    const int n_chunks = (n_ref + kWarp - 1) / kWarp;
    uint32_t taken = 0;  // bit c: j = 32 c + lane is taken
    int h = 0;
    for (int i = 0; i < n_hyp; ++i) {
        const double b = yh[i];
        const int32_t w = hid[i];
        for (int c = 0; c < n_chunks; ++c) {
            const int j = c * kWarp + lane;
            const bool ok = j < n_ref && !((taken >> c) & 1u) && rid[j] == w && within(y[j], b, tol);
            const uint32_t m = __ballot_sync(0xffffffffu, ok);
            if (m) {
                if (lane == __ffs(m) - 1) taken |= 1u << c;
                ++h;
                break;
            }
        }
    }
    if (lane == 0) hits[p] = h;
}

int launch_boundary_hits(const double *d_end_times, const wca_utt_t *d_utts, const int32_t *d_utt_of, int n_problems,
                         const double *d_ref_times, const int64_t *d_ref_off, const int32_t *d_ref_ids,
                         const int32_t *d_hyp_ids, const int64_t *d_hyp_off, double tolerance, int strict, int32_t *d_hits,
                         cudaStream_t stream) {
    const int blocks = (n_problems + kHitsWarpsPerCta - 1) / kHitsWarpsPerCta;
    boundary_hits_kernel<<<blocks, kHitsWarpsPerCta * kWarp, 0, stream>>>(d_end_times, d_utts, d_utt_of, n_problems,
                                                                         d_ref_times, d_ref_off, d_ref_ids, d_hyp_ids,
                                                                         d_hyp_off, tolerance, strict, d_hits);
    WCA_LAUNCH_CHECK("boundary_hits_kernel");
    return WCA_OK;
}

}  // namespace wca
