// Single-query attention of one greedy decode step (upstream whisper/model.py MultiHeadAttention.qkv_attention with a
// kv_cache): one query row per batch item against n_kv cached keys, every key visible --
//     out[b, h*64:(h+1)*64] = softmax_j(q[b,h,:] . k[b,j,h,:] / 8) . v[b,j,h,:],   j < n_kv
// It serves the decoder's self-attention over the positions cached so far (n_kv <= 448) and its cross-attention over the
// 1500 encoder rows.  Each key and value is read once and used for 64 multiply-adds, so the step is bound by HBM reads:
// fp32 on the CUDA cores, no tensor cores.
//
// Split over keys: CTA (c, h, b) reduces the keys [64 c, 64 c + 64) of head h of item b to a partial (m, l, o[64]) --
// chunk maximum, sum of exp(s - m), un-normalised output -- in the caller's workspace, so that B * H small problems still
// fill the SMs.  A second kernel merges the chunks of each (b, h) in chunk order.  The chunk length is a constant and the
// number of chunks depends on n_kv only: a row gives the same bits alone and inside any batch.  Keys at or past n_kv are
// never read.
#include "common.cuh"

namespace wca {

constexpr int kDecodeChunk = 64;     // keys per CTA
constexpr int kDecodeThreads = 128;  // 4 warps x 16 keys for the scores; 2 halves x 64 dims for P.V
constexpr int kPartialFloats = 68;   // m, l, 2 pad, o[64]: o stays 16-byte aligned

static int decode_chunks(int n_kv) { return (n_kv + kDecodeChunk - 1) / kDecodeChunk; }

__global__ void __launch_bounds__(kDecodeThreads) decode_attention_kernel(
    const float *__restrict__ q, const float *__restrict__ k, const float *__restrict__ v, int n_kv, int64_t ld_q,
    int64_t ld_k, int64_t ld_v, int64_t bs_k, int64_t bs_v, float *__restrict__ part) {
    const int c = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int j0 = c * kDecodeChunk;
    const float *kb = k + (int64_t)b * bs_k + (int64_t)h * kHeadDim;
    const float *vb = v + (int64_t)b * bs_v + (int64_t)h * kHeadDim;
    __shared__ float s_p[kDecodeChunk];
    __shared__ float s_o[kHeadDim];

    // P.V operands first, so that they are in flight while the scores are computed: thread (half, d) owns dimension d
    // of the keys [32 half, 32 half + 32) of the chunk (a warp reads 128 contiguous bytes per key)
    const int d = t & 63, half = t >> 6;
    float vv[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        const int j = j0 + half * 32 + i;
        vv[i] = j < n_kv ? ld_stream(vb + (int64_t)j * ld_v + d) : 0.f;
    }

    // scores: 8 lanes per key, lane g holds dims [4g, 4g+4) and [32+4g, 32+4g+4) (two 128-byte segments per key);
    // warp w takes keys 16 w + 4 pass + (lane >> 3)
    const int g = lane & 7, sub = lane >> 3;
    const float4 *q4 = reinterpret_cast<const float4 *>(q + (int64_t)b * ld_q + (int64_t)h * kHeadDim);
    const float4 qa = q4[g], qb = q4[8 + g];
    float4 ka[4], kb4[4];
#pragma unroll
    for (int pass = 0; pass < 4; ++pass) {
        const int j = j0 + warp * 16 + pass * 4 + sub;
        if (j < n_kv) {
            const float4 *kr = reinterpret_cast<const float4 *>(kb + (int64_t)j * ld_k);
            ka[pass] = ld_stream4(kr + g);
            kb4[pass] = ld_stream4(kr + 8 + g);
        } else {
            ka[pass] = kb4[pass] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
#pragma unroll
    for (int pass = 0; pass < 4; ++pass) {
        float s = qa.x * ka[pass].x;
        s = fmaf(qa.y, ka[pass].y, s);
        s = fmaf(qa.z, ka[pass].z, s);
        s = fmaf(qa.w, ka[pass].w, s);
        s = fmaf(qb.x, kb4[pass].x, s);
        s = fmaf(qb.y, kb4[pass].y, s);
        s = fmaf(qb.z, kb4[pass].z, s);
        s = fmaf(qb.w, kb4[pass].w, s);
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        const int jl = warp * 16 + pass * 4 + sub;
        if (g == 0) s_p[jl] = j0 + jl < n_kv ? s * 0.125f : -INFINITY;  // / sqrt(64), exact
    }
    __syncthreads();

    // chunk maximum and sum (every warp computes the same values: no second barrier); the chunk holds >= 1 live key
    const float a0 = s_p[lane], a1 = s_p[lane + 32];
    const float m = warp_max(fmaxf(a0, a1));
    const float p0 = expf(a0 - m), p1 = expf(a1 - m);
    const float l = warp_sum(p0 + p1);
    __syncthreads();  // every warp has read the scores
    if (warp == 0) {
        s_p[lane] = p0;
        s_p[lane + 32] = p1;
    }
    __syncthreads();

    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) acc = fmaf(s_p[half * 32 + i], vv[i], acc);
    if (half == 1) s_o[d] = acc;
    __syncthreads();
    float *pp = part + (((int64_t)b * gridDim.y + h) * gridDim.x + c) * kPartialFloats;
    if (half == 0) {
        pp[4 + d] = acc + s_o[d];
        if (d == 0) {
            pp[0] = m;
            pp[1] = l;
        }
    }
}

// out[b, h*64 + d] = sum_c e^(m_c - M) o_c[d] / sum_c e^(m_c - M) l_c, chunks in order; one CTA of 64 threads per (h, b)
__global__ void __launch_bounds__(kHeadDim) decode_combine_kernel(const float *__restrict__ part, int n_chunks,
                                                                  float *__restrict__ out, int64_t ld_out) {
    const int h = blockIdx.x, b = blockIdx.y, d = threadIdx.x;
    const float *pp = part + ((int64_t)b * gridDim.x + h) * n_chunks * kPartialFloats;
    float M = -INFINITY;
    for (int c = 0; c < n_chunks; ++c) M = fmaxf(M, pp[c * kPartialFloats]);
    float L = 0.f, O = 0.f;
    for (int c = 0; c < n_chunks; ++c) {
        const float *pc = pp + c * kPartialFloats;
        const float w = expf(pc[0] - M);
        L = fmaf(w, pc[1], L);
        O = fmaf(w, pc[4 + d], O);
    }
    out[(int64_t)b * ld_out + (int64_t)h * kHeadDim + d] = O / L;
}

int64_t decode_attention_workspace_bytes(int n_batch, int n_heads, int n_kv) {
    return (int64_t)n_batch * n_heads * decode_chunks(n_kv) * kPartialFloats * (int64_t)sizeof(float);
}

int launch_decode_attention(const float *q, const float *k, const float *v, float *out, int n_batch, int n_kv, int n_heads,
                            int64_t ld_q, int64_t ld_k, int64_t ld_v, int64_t ld_out, int64_t bs_k, int64_t bs_v,
                            float *ws, cudaStream_t stream) {
    const int n_chunks = decode_chunks(n_kv);
    decode_attention_kernel<<<dim3(n_chunks, n_heads, n_batch), kDecodeThreads, 0, stream>>>(q, k, v, n_kv, ld_q, ld_k, ld_v,
                                                                                             bs_k, bs_v, ws);
    WCA_LAUNCH_CHECK("decode_attention_kernel");
    decode_combine_kernel<<<dim3(n_heads, n_batch), kHeadDim, 0, stream>>>(ws, n_chunks, out, ld_out);
    WCA_LAUNCH_CHECK("decode_combine_kernel");
    return WCA_OK;
}

}  // namespace wca
