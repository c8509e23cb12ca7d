// Probability of one given token per row under a softmax over the row's first n_cols logits -- the word confidence of
// upstream whisper.timing.find_alignment:
//     sampled_logits = logits[len(tokenizer.sot_sequence):, : tokenizer.eot]
//     token_probs = sampled_logits.softmax(dim=-1)
//     text_token_probs = token_probs[np.arange(len(text_tokens)), text_tokens].tolist()
// p[r] = exp(x[r, t_r] - M_r) / sum_c exp(x[r, c] - M_r),  M_r = max_c x[r, c],  c < n_cols.
//
// One CTA per row streams the row once: a scalar head up to the first 16-byte boundary, float4 loads (four in flight
// per thread) and a scalar tail.  Each thread keeps a running (max, sum of exp) over groups of 16 values that share one
// rescale, then the block merges the 256 pairs in a fixed order (warp butterflies, then warps 0..7 in order): the bits
// of a row depend on its address modulo 16 and on n_cols only, never on the batch.  The row is read in place, so a
// row of a (T, V_pad) logits tensor is not copied; columns at or past n_cols are never read.  HBM-bound: 4 * n_cols
// bytes per row.
//
// torch semantics: a NaN anywhere gives NaN (its exp enters the sum), a +inf gives NaN (exp(inf - inf)), an all -inf
// row gives NaN (0/0), a -inf target in a finite row gives exactly 0.  A -inf logit contributes exactly 0 to the sum
// even where a thread's own maximum is still -inf.
#include <math.h>

#include "common.cuh"

namespace wca {

constexpr int kTpThreads = 256;
constexpr int kTpUnroll = 4;  // float4 loads in flight per thread

struct MaxSum {
    float m, s;
};

// exp(x - m), with a -inf logit contributing 0 whatever m is (exp(-inf - -inf) would be NaN)
__device__ __forceinline__ float exp_term(float x, float m) { return x == -INFINITY ? 0.f : expf(x - m); }

// (m, s) of a thread after folding in a group whose maximum is gm and whose terms are added by the caller
__device__ __forceinline__ void rescale_to(MaxSum &a, float gm) {
    const float mn = fmaxf(a.m, gm);  // fmaxf drops NaN: NaN reaches the sum through its exp term
    if (mn > a.m) {
        a.s = a.m == -INFINITY ? a.s : a.s * expf(a.m - mn);
        a.m = mn;
    }
}

__device__ __forceinline__ MaxSum merge(MaxSum a, MaxSum b) {
    const float mn = fmaxf(a.m, b.m);
    if (mn == -INFINITY) return {mn, a.s + b.s};  // both still empty of finite values (NaN sums stay NaN)
    const float sa = a.m == -INFINITY ? a.s * 0.f : a.s * expf(a.m - mn);  // 0, or NaN if a saw a NaN
    const float sb = b.m == -INFINITY ? b.s * 0.f : b.s * expf(b.m - mn);
    return {mn, sa + sb};
}

__device__ __forceinline__ void add_scalar(MaxSum &a, float x) {
    rescale_to(a, x);
    a.s += exp_term(x, a.m);
}

__global__ void __launch_bounds__(kTpThreads) token_probs_kernel(const float *const *__restrict__ rows,
                                                                 const int32_t *__restrict__ targets, int n_cols,
                                                                 float *__restrict__ probs) {
    const int r = blockIdx.x;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const float *row = rows[r];
    const int head = min((int)(((16u - ((uint32_t)(uintptr_t)row & 15u)) & 15u) >> 2), n_cols);
    const int n_vec = (n_cols - head) >> 2;
    const int tail0 = head + 4 * n_vec;

    MaxSum a{-INFINITY, 0.f};
    if (t < head) add_scalar(a, ld_stream(row + t));
    const float4 *vec = reinterpret_cast<const float4 *>(row + head);
    int i = t;
    for (; i + (kTpUnroll - 1) * kTpThreads < n_vec; i += kTpUnroll * kTpThreads) {
        float4 v[kTpUnroll];
#pragma unroll
        for (int u = 0; u < kTpUnroll; ++u) v[u] = ld_stream4(vec + i + u * kTpThreads);
        float gm = -INFINITY;
#pragma unroll
        for (int u = 0; u < kTpUnroll; ++u) gm = fmaxf(gm, fmaxf(fmaxf(v[u].x, v[u].y), fmaxf(v[u].z, v[u].w)));
        rescale_to(a, gm);
        float e[kTpUnroll];
#pragma unroll
        for (int u = 0; u < kTpUnroll; ++u)
            e[u] = (exp_term(v[u].x, a.m) + exp_term(v[u].y, a.m)) + (exp_term(v[u].z, a.m) + exp_term(v[u].w, a.m));
        a.s += (e[0] + e[1]) + (e[2] + e[3]);
    }
    for (; i < n_vec; i += kTpThreads) {
        const float4 v = ld_stream4(vec + i);
        rescale_to(a, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
        a.s += (exp_term(v.x, a.m) + exp_term(v.y, a.m)) + (exp_term(v.z, a.m) + exp_term(v.w, a.m));
    }
    if (t < n_cols - tail0) add_scalar(a, ld_stream(row + tail0 + t));

#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        MaxSum b{__shfl_xor_sync(0xffffffffu, a.m, o), __shfl_xor_sync(0xffffffffu, a.s, o)};
        a = merge(a, b);
    }
    __shared__ MaxSum s_warp[kTpThreads / kWarp];
    if (lane == 0) s_warp[warp] = a;
    __syncthreads();
    if (t != 0) return;
    MaxSum tot = s_warp[0];
#pragma unroll
    for (int w = 1; w < kTpThreads / kWarp; ++w) tot = merge(tot, s_warp[w]);

    const int tgt = targets[r];
    if (tgt < 0 || tgt >= n_cols) {  // callers validate the targets; the row is never read outside [0, n_cols)
        probs[r] = __int_as_float(0x7fc00000);
        return;
    }
    const float x = row[tgt];
    // exp(x - M) with the rounding error of the subtraction folded back in (TwoSum, exact without FMA contraction):
    // for logits of magnitude ~100, x - M is otherwise off by up to 64 ulps of the result
    const float d = x - tot.m;
    float num = exp_term(x, tot.m);
    if (isfinite(d)) {
        const float bp = d - x;
        const float err = (x - (d - bp)) + (-tot.m - bp);
        num += num * err;
    }
    probs[r] = num / tot.s;
}

int launch_token_probs(const float *const *d_rows, const int32_t *d_targets, int n_rows, int n_cols, float *d_probs,
                       cudaStream_t stream) {
    token_probs_kernel<<<n_rows, kTpThreads, 0, stream>>>(d_rows, d_targets, n_cols, d_probs);
    WCA_LAUNCH_CHECK("token_probs_kernel");
    return WCA_OK;
}

}  // namespace wca
