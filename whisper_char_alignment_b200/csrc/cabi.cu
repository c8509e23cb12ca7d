// extern "C" surface of libwca_b200.so -- see include/wca_b200.h for the contract of
// every entry point and the reference lines each one replaces.  Argument validation
// happens here; the kernels live in the sibling translation units.
#include <cstdarg>
#include <cstdio>

#include "common.cuh"

namespace wca {

static thread_local char g_err[512] = "";
static thread_local uint64_t g_launches = 0;

void count_launch() { ++g_launches; }

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what) {
    set_error("%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
    return WCA_ERR_CUDA;
}

static int device_sm_count(int *sms, int *cc) {
    int dev = 0;
    WCA_CUDA(cudaGetDevice(&dev));
    int n = 0, major = 0, minor = 0;
    WCA_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    WCA_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    WCA_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
    if (sms) *sms = n;
    if (cc) *cc = major * 10 + minor;
    return WCA_OK;
}

// kernels (defined in the other translation units)
int launch_capture_logits_simt(const float *const *, const float *const *, int, int, int64_t, int64_t,
                               const wca_utt_t *, int, int, float *, cudaStream_t);
int launch_capture_tc(const float *const *, const float *const *, int, int, int64_t, int64_t, int64_t, int64_t,
                      const wca_utt_t *, int, int, int, int, float, float *, float *, unsigned, int, cudaStream_t);
int launch_scores_from_partials(const float *, const wca_utt_t *, int, int, float, float, float *, cudaStream_t);
bool capture_tc_supported(int max_tokens, int max_frames, int medfilt_width);
int read_capture_trace(long long *, int);
int launch_medfilt_softmax_rows(const float *, int64_t, int64_t, int, int, float, float *, int, cudaStream_t);
int launch_medfilt_softmax_batched(float *, const wca_utt_t *, int, int, int, int, int, float, int, cudaStream_t);
int launch_head_scores(const float *, const wca_utt_t *, int, int, int, float, float, float, float *, cudaStream_t);
int launch_topk_heads(const float *, const wca_utt_t *, int, int, int32_t *, float *, cudaStream_t);
int launch_aggregate_heads(const float *, const int32_t *, const wca_utt_t *, int, int, int, int, float *, cudaStream_t);
int launch_normalize_heads(const float *, const int32_t *, const wca_utt_t *, int, int, int, float *, const int64_t *, float *,
                           cudaStream_t);
int launch_token_probs(const float *const *, const int32_t *, int, int, float *, cudaStream_t);
int launch_boundary_hits(const double *, const wca_utt_t *, const int32_t *, int, const double *, const int64_t *,
                         const int32_t *, const int32_t *, const int64_t *, double, int, int32_t *, cudaStream_t);
int64_t dtw_workspace_bytes(int, int, int);
int launch_dtw_align(const float *, const wca_utt_t *, int, int, int, int, int32_t *, int32_t *, int32_t *, int32_t *,
                     const int32_t *, double *, double *, void *, int64_t, cudaStream_t);

int launch_full_attention(const float *, const float *, const float *, float *, int, int, int, int, int64_t, int64_t, int64_t,
                          int64_t, int, cudaStream_t);

int64_t decode_attention_workspace_bytes(int, int, int);
int launch_decode_attention(const float *, const float *, const float *, float *, int, int, int, int64_t, int64_t, int64_t,
                            int64_t, int64_t, int64_t, float *, cudaStream_t);

void set_enc_attn_debug_buffer(float *);
int launch_add_layernorm(const float *, const float *, const float *, const float *, float *, float *, int64_t, int, float,
                         cudaStream_t);

static bool odd_width_ok(int w) { return w >= 1 && w <= WCA_MAX_MEDFILT && (w & 1) == 1; }

}  // namespace wca

using namespace wca;

extern "C" {

int wca_abi_version(void) { return WCA_ABI_VERSION; }

const char *wca_last_error(void) { return g_err; }

uint64_t wca_launch_count(void) { return g_launches; }

int wca_device_info(int *sm_count, int *compute_capability) { return device_sm_count(sm_count, compute_capability); }

int wca_capture_attention(const float *const *h_q_layers, const float *const *h_k_layers, int n_layers,
                          int n_heads_per_layer, int head_dim, int64_t ld_q, int64_t ld_k, int64_t q_rows,
                          int64_t k_rows, const wca_utt_t *d_utts, int n_utts, int max_tokens, int max_frames, int medfilt_width, float qk_scale, float *d_ws,
                          float *d_partials, unsigned flags, wca_stream_t stream) {
    WCA_CHECK_ARG(h_q_layers && h_k_layers && d_utts && d_ws, "wca_capture_attention: null pointer");
    WCA_CHECK_ARG(n_layers >= 1 && n_layers <= WCA_MAX_LAYERS, "wca_capture_attention: n_layers=%d not in [1,%d]",
                  n_layers, WCA_MAX_LAYERS);
    WCA_CHECK_ARG(n_heads_per_layer >= 1 && (int64_t)n_layers * n_heads_per_layer <= 65535,
                  "wca_capture_attention: bad head count %d", n_heads_per_layer);
    if (head_dim != kHeadDim) {
        set_error("wca_capture_attention: head_dim=%d unsupported (every Whisper size uses 64)", head_dim);
        return WCA_ERR_UNSUPPORTED;
    }
    WCA_CHECK_ARG(ld_q >= (int64_t)n_heads_per_layer * head_dim && ld_k >= (int64_t)n_heads_per_layer * head_dim &&
                      ld_q % 4 == 0 && ld_k % 4 == 0,
                  "wca_capture_attention: leading dimensions (%lld, %lld) must cover H*Dh and be multiples of 4",
                  (long long)ld_q, (long long)ld_k);
    WCA_CHECK_ARG(q_rows >= 1 && k_rows >= 1 && q_rows < (1ll << 31) && k_rows < (1ll << 31),
                  "wca_capture_attention: row counts (%lld, %lld) out of range", (long long)q_rows, (long long)k_rows);
    WCA_CHECK_ARG(n_utts >= 0 && n_utts <= 65535 && max_tokens >= 1 && max_frames >= 1,
                  "wca_capture_attention: bad batch geometry (%d utts, %d tokens, %d frames)", n_utts, max_tokens,
                  max_frames);
    const bool raw = (flags & WCA_CAPTURE_RAW_LOGITS) != 0;
    WCA_CHECK_ARG(raw || odd_width_ok(medfilt_width), "wca_capture_attention: medfilt_width=%d must be odd, 1..%d",
                  medfilt_width, WCA_MAX_MEDFILT);
    for (int l = 0; l < n_layers; ++l)
        WCA_CHECK_ARG(h_q_layers[l] && h_k_layers[l] && ((uintptr_t)h_q_layers[l] % 16 == 0) &&
                          ((uintptr_t)h_k_layers[l] % 16 == 0),
                      "wca_capture_attention: layer %d Q/K pointer null or not 16-byte aligned", l);
    if (n_utts == 0) return WCA_OK;
    int sms = 0, cc = 0;
    int rc = device_sm_count(&sms, &cc);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    const bool want_tc = !(flags & WCA_CAPTURE_FORCE_SIMT) && capture_tc_supported(max_tokens, max_frames, medfilt_width);
    if (want_tc) {
        if (cc < 100) {
            set_error("wca_capture_attention: tcgen05 path needs compute capability 10.x, device is %d", cc);
            return WCA_ERR_NO_DEVICE;
        }
        return launch_capture_tc(h_q_layers, h_k_layers, n_layers, n_heads_per_layer, ld_q, ld_k, q_rows, k_rows, d_utts, n_utts,
                                 max_tokens, max_frames, medfilt_width, qk_scale, d_ws, d_partials, flags, sms, st);
    }
    if (d_partials != nullptr) {
        set_error("wca_capture_attention: head-score partials are only produced by the tcgen05 kernel "
                  "(ask wca_capture_writes_partials first)");
        return WCA_ERR_UNSUPPORTED;
    }
    rc = launch_capture_logits_simt(h_q_layers, h_k_layers, n_layers, n_heads_per_layer, ld_q, ld_k, d_utts, n_utts,
                                    max_tokens, d_ws, st);
    if (rc || raw) return rc;
    return launch_medfilt_softmax_batched(d_ws, d_utts, n_utts, n_layers * n_heads_per_layer, max_tokens, max_frames,
                                          medfilt_width, qk_scale, sms, st);
}

static int attention_entry(const char *who, const float *d_q, const float *d_k, const float *d_v, float *d_out, int n_batch,
                           int n_q, int n_kv, int n_heads, int head_dim, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                           int64_t ld_out, int causal, wca_stream_t stream) {
    WCA_CHECK_ARG(d_q && d_k && d_v && d_out, "%s: null pointer", who);
    if (head_dim != kHeadDim) {
        set_error("%s: head_dim=%d unsupported (every Whisper size uses 64)", who, head_dim);
        return WCA_ERR_UNSUPPORTED;
    }
    WCA_CHECK_ARG(n_batch >= 0 && n_batch <= 65535 && n_heads >= 1 && n_heads <= 65535 && n_q >= 1 && n_q < (1 << 24) &&
                      n_kv >= 1 && n_kv < (1 << 24),
                  "%s: bad geometry (batch %d, n_q %d, n_kv %d, heads %d)", who, n_batch, n_q, n_kv, n_heads);
    const int64_t width = (int64_t)n_heads * head_dim;
    WCA_CHECK_ARG(ld_q >= width && ld_k >= width && ld_v >= width && ld_out >= width && ld_q % 4 == 0 && ld_k % 4 == 0 &&
                      ld_v % 4 == 0 && ld_out % 4 == 0,
                  "%s: leading dimensions must cover H*Dh=%lld and be multiples of 4", who, (long long)width);
    WCA_CHECK_ARG(((uintptr_t)d_q | (uintptr_t)d_k | (uintptr_t)d_v | (uintptr_t)d_out) % 16 == 0,
                  "%s: pointers must be 16-byte aligned", who);
    if (n_batch == 0) return WCA_OK;
    int cc = 0;
    int rc = device_sm_count(nullptr, &cc);
    if (rc) return rc;
    if (cc < 100) {
        set_error("%s: needs compute capability 10.x (tcgen05), device is %d", who, cc);
        return WCA_ERR_NO_DEVICE;
    }
    return launch_full_attention(d_q, d_k, d_v, d_out, n_batch, n_q, n_kv, n_heads, ld_q, ld_k, ld_v, ld_out, causal,
                                 static_cast<cudaStream_t>(stream));
}

int wca_full_attention(const float *d_q, const float *d_k, const float *d_v, float *d_out, int n_batch, int n_q, int n_kv,
                       int n_heads, int head_dim, int64_t ld_q, int64_t ld_k, int64_t ld_v, int64_t ld_out,
                       wca_stream_t stream) {
    return attention_entry("wca_full_attention", d_q, d_k, d_v, d_out, n_batch, n_q, n_kv, n_heads, head_dim, ld_q, ld_k, ld_v,
                           ld_out, 0, stream);
}

int wca_causal_attention(const float *d_q, const float *d_k, const float *d_v, float *d_out, int n_batch, int n_q, int n_kv,
                         int n_heads, int head_dim, int64_t ld_q, int64_t ld_k, int64_t ld_v, int64_t ld_out,
                         wca_stream_t stream) {
    return attention_entry("wca_causal_attention", d_q, d_k, d_v, d_out, n_batch, n_q, n_kv, n_heads, head_dim, ld_q, ld_k,
                           ld_v, ld_out, 1, stream);
}

int64_t wca_decode_attention_workspace_bytes(int n_batch, int n_heads, int n_kv) {
    if (n_batch < 1 || n_heads < 1 || n_kv < 1) return 0;
    return decode_attention_workspace_bytes(n_batch, n_heads, n_kv);
}

int wca_decode_attention(const float *d_q, const float *d_k, const float *d_v, float *d_out, int n_batch, int n_kv,
                         int n_heads, int head_dim, int64_t ld_q, int64_t ld_k, int64_t ld_v, int64_t ld_out,
                         int64_t batch_stride_k, int64_t batch_stride_v, void *d_workspace, int64_t workspace_bytes,
                         wca_stream_t stream) {
    const char *who = "wca_decode_attention";
    WCA_CHECK_ARG(d_q && d_k && d_v && d_out && d_workspace, "%s: null pointer", who);
    if (head_dim != kHeadDim) {
        set_error("%s: head_dim=%d unsupported (every Whisper size uses 64)", who, head_dim);
        return WCA_ERR_UNSUPPORTED;
    }
    WCA_CHECK_ARG(n_batch >= 1 && n_batch <= 65535 && n_heads >= 1 && n_heads <= 65535 && n_kv >= 1 && n_kv < (1 << 24),
                  "%s: bad geometry (batch %d, n_kv %d, heads %d)", who, n_batch, n_kv, n_heads);
    const int64_t width = (int64_t)n_heads * head_dim;
    WCA_CHECK_ARG(ld_q >= width && ld_k >= width && ld_v >= width && ld_out >= width && ld_q % 4 == 0 && ld_k % 4 == 0 &&
                      ld_v % 4 == 0 && ld_out % 4 == 0,
                  "%s: leading dimensions must cover H*Dh=%lld and be multiples of 4", who, (long long)width);
    WCA_CHECK_ARG(batch_stride_k >= 0 && batch_stride_v >= 0 && batch_stride_k % 4 == 0 && batch_stride_v % 4 == 0,
                  "%s: batch strides (%lld, %lld) must be non-negative multiples of 4", who, (long long)batch_stride_k,
                  (long long)batch_stride_v);
    WCA_CHECK_ARG(((uintptr_t)d_q | (uintptr_t)d_k | (uintptr_t)d_v | (uintptr_t)d_out | (uintptr_t)d_workspace) % 16 == 0,
                  "%s: pointers must be 16-byte aligned", who);
    const int64_t need = decode_attention_workspace_bytes(n_batch, n_heads, n_kv);
    WCA_CHECK_ARG(workspace_bytes >= need, "%s: workspace of %lld bytes, %lld needed (wca_decode_attention_workspace_bytes)",
                  who, (long long)workspace_bytes, (long long)need);
    return launch_decode_attention(d_q, d_k, d_v, d_out, n_batch, n_kv, n_heads, ld_q, ld_k, ld_v, ld_out, batch_stride_k,
                                   batch_stride_v, static_cast<float *>(d_workspace), static_cast<cudaStream_t>(stream));
}

int wca_add_layernorm(const float *d_x, const float *d_h, const float *d_gamma, const float *d_beta, float *d_y, float *d_n,
                      int64_t n_rows, int width, float eps, wca_stream_t stream) {
    WCA_CHECK_ARG(d_x && d_gamma && d_beta && d_n, "wca_add_layernorm: null pointer");
    WCA_CHECK_ARG(n_rows >= 0 && n_rows < (1ll << 31) * 8, "wca_add_layernorm: n_rows=%lld", (long long)n_rows);
    WCA_CHECK_ARG(width > 0 && width % 128 == 0, "wca_add_layernorm: width=%d must be a multiple of 128", width);
    WCA_CHECK_ARG(((uintptr_t)d_x | (uintptr_t)d_h | (uintptr_t)d_gamma | (uintptr_t)d_beta | (uintptr_t)d_y | (uintptr_t)d_n) % 16 == 0,
                  "wca_add_layernorm: pointers must be 16-byte aligned");
    if (n_rows == 0) return WCA_OK;
    return launch_add_layernorm(d_x, d_h, d_gamma, d_beta, d_y, d_n, n_rows, width, eps, static_cast<cudaStream_t>(stream));
}

int wca_capture_writes_partials(int max_frames, int medfilt_width, unsigned flags) {
    return !(flags & (WCA_CAPTURE_FORCE_SIMT | WCA_CAPTURE_RAW_LOGITS)) && capture_tc_supported(0, max_frames, medfilt_width) ? 1 : 0;
}

int64_t wca_capture_partials_floats(int n_heads, int n_tokens, int n_frames) {
    if (n_heads <= 0 || n_tokens <= 0 || n_frames <= 0) return 0;
    const int64_t token_blocks = (n_tokens + 127) / 128;
    return (int64_t)n_heads * token_blocks * 4 * (1 + (int64_t)n_frames);
}

int wca_head_scores_from_partials(const float *d_partials, const wca_utt_t *d_utts, int n_utts, int n_heads, float w_colnorm,
                                  float w_rownorm, float *d_scores, wca_stream_t stream) {
    WCA_CHECK_ARG(d_partials && d_utts && d_scores, "wca_head_scores_from_partials: null pointer");
    WCA_CHECK_ARG(n_heads >= 1 && n_heads <= 65535 * 4 && n_utts >= 0 && n_utts <= 65535,
                  "wca_head_scores_from_partials: bad geometry (%d heads, %d utts)", n_heads, n_utts);
    if (n_utts == 0) return WCA_OK;
    return launch_scores_from_partials(d_partials, d_utts, n_utts, n_heads, w_colnorm, w_rownorm, d_scores,
                                       static_cast<cudaStream_t>(stream));
}

void wca_debug_enc_attn_buffer(float *d_buf) { set_enc_attn_debug_buffer(d_buf); }

int wca_debug_capture_trace(long long *h_out, int capacity) {
    WCA_CHECK_ARG(h_out && capacity > 0, "wca_debug_capture_trace: bad buffer");
    return read_capture_trace(h_out, capacity);
}

int wca_medfilt_softmax(const float *d_in, int64_t n_rows, int64_t ld_in, int n_frames, int medfilt_width,
                        float qk_scale, float *d_out, wca_stream_t stream) {
    WCA_CHECK_ARG(d_in && d_out, "wca_medfilt_softmax: null pointer");
    WCA_CHECK_ARG(n_rows >= 0 && n_frames >= 1 && ld_in >= n_frames, "wca_medfilt_softmax: bad shape (%lld x %d, ld %lld)",
                  (long long)n_rows, n_frames, (long long)ld_in);
    WCA_CHECK_ARG(odd_width_ok(medfilt_width), "wca_medfilt_softmax: medfilt_width=%d must be odd, 1..%d",
                  medfilt_width, WCA_MAX_MEDFILT);
    WCA_CHECK_ARG(d_in != d_out || ld_in == n_frames, "wca_medfilt_softmax: in-place use needs ld_in == n_frames");
    if (n_rows == 0) return WCA_OK;
    int sms = 0;
    int rc = device_sm_count(&sms, nullptr);
    if (rc) return rc;
    return launch_medfilt_softmax_rows(d_in, n_rows, ld_in, n_frames, medfilt_width, qk_scale, d_out, sms,
                                       static_cast<cudaStream_t>(stream));
}

int wca_head_scores(const float *d_ws, const wca_utt_t *d_utts, int n_utts, int n_heads, int max_tokens,
                    int max_frames, float w_colnorm, float w_rownorm, float w_coverage, float *d_scores,
                    wca_stream_t stream) {
    WCA_CHECK_ARG(d_ws && d_utts && d_scores, "wca_head_scores: null pointer");
    WCA_CHECK_ARG(max_frames >= 1, "wca_head_scores: max_frames=%d", max_frames);
    // rows longer than one 256-column chunk keep their partial norms in a 1024-entry shared buffer
    WCA_CHECK_ARG(max_frames <= 256 || max_tokens <= 1024,
                  "wca_head_scores: max_tokens=%d with max_frames=%d (more than 1024 token rows need max_frames <= 256)",
                  max_tokens, max_frames);
    WCA_CHECK_ARG(n_heads >= 1 && n_heads <= 65535 * 32 && n_utts >= 0 && n_utts <= 65535,
                  "wca_head_scores: bad geometry (%d heads, %d utts)", n_heads, n_utts);
    if (n_utts == 0) return WCA_OK;
    return launch_head_scores(d_ws, d_utts, n_utts, n_heads, max_frames, w_colnorm, w_rownorm, w_coverage, d_scores,
                              static_cast<cudaStream_t>(stream));
}

int wca_topk_heads(const float *d_scores, const wca_utt_t *d_utts, int n_utts, int n_heads, int32_t *d_sel,
                   float *d_sel_scores, wca_stream_t stream) {
    WCA_CHECK_ARG(d_scores && d_utts && d_sel, "wca_topk_heads: null pointer");
    WCA_CHECK_ARG(n_heads >= 1 && n_heads <= 8192, "wca_topk_heads: n_heads=%d not in [1,8192]", n_heads);
    WCA_CHECK_ARG(n_utts >= 0, "wca_topk_heads: n_utts < 0");
    if (n_utts == 0) return WCA_OK;
    return launch_topk_heads(d_scores, d_utts, n_utts, n_heads, d_sel, d_sel_scores, static_cast<cudaStream_t>(stream));
}

int wca_aggregate_heads(const float *d_ws, const int32_t *d_sel, const wca_utt_t *d_utts, int n_utts, int max_tokens,
                        int max_frames, int max_sel, float *d_matrix, wca_stream_t stream) {
    WCA_CHECK_ARG(d_ws && d_sel && d_utts && d_matrix, "wca_aggregate_heads: null pointer");
    WCA_CHECK_ARG(n_utts >= 0 && n_utts <= 65535 && max_tokens >= 1 && max_frames >= 1 && max_sel >= 1,
                  "wca_aggregate_heads: bad geometry");
    if (n_utts == 0) return WCA_OK;
    return launch_aggregate_heads(d_ws, d_sel, d_utts, n_utts, max_tokens, max_frames, max_sel, d_matrix,
                                  static_cast<cudaStream_t>(stream));
}

int wca_normalize_heads(const float *d_ws, const int32_t *d_sel, const wca_utt_t *d_utts, int n_utts, int max_tokens,
                        int max_frames, float *d_weights, const int64_t *d_weights_off, float *d_matrix,
                        wca_stream_t stream) {
    WCA_CHECK_ARG(d_ws && d_sel && d_utts && d_matrix, "wca_normalize_heads: null pointer");
    WCA_CHECK_ARG((d_weights == nullptr) == (d_weights_off == nullptr),
                  "wca_normalize_heads: give d_weights and d_weights_off together or neither");
    WCA_CHECK_ARG(n_utts >= 0 && n_utts <= 65535 && max_tokens >= 1 && max_frames >= 1 && max_frames <= 65535 * 32,
                  "wca_normalize_heads: bad geometry (%d utts, max_tokens %d, max_frames %d)", n_utts, max_tokens,
                  max_frames);
    if (n_utts == 0) return WCA_OK;
    return launch_normalize_heads(d_ws, d_sel, d_utts, n_utts, max_tokens, max_frames, d_weights, d_weights_off, d_matrix,
                                  static_cast<cudaStream_t>(stream));
}

int wca_token_probs(const float *const *d_rows, const int32_t *d_targets, int n_rows, int n_cols, float *d_probs,
                    wca_stream_t stream) {
    WCA_CHECK_ARG(d_rows && d_targets && d_probs, "wca_token_probs: null pointer");
    WCA_CHECK_ARG(n_rows >= 0 && n_cols >= 1, "wca_token_probs: bad shape (%d rows, %d columns)", n_rows, n_cols);
    if (n_rows == 0) return WCA_OK;
    return launch_token_probs(d_rows, d_targets, n_rows, n_cols, d_probs, static_cast<cudaStream_t>(stream));
}

int wca_boundary_hits(const double *d_end_times, const wca_utt_t *d_utts, const int32_t *d_utt_of, int n_problems,
                      const double *d_ref_times, const int64_t *d_ref_off, const int32_t *d_ref_ids,
                      const int32_t *d_hyp_ids, const int64_t *d_hyp_off, double tolerance, int mode, int32_t *d_hits,
                      wca_stream_t stream) {
    WCA_CHECK_ARG(d_end_times && d_utts && d_utt_of && d_ref_times && d_ref_off && d_hits,
                  "wca_boundary_hits: null pointer");
    WCA_CHECK_ARG(mode == WCA_HITS_PLAIN || mode == WCA_HITS_STRICT, "wca_boundary_hits: unknown mode %d", mode);
    WCA_CHECK_ARG(mode == WCA_HITS_PLAIN || (d_ref_ids && d_hyp_ids && d_hyp_off),
                  "wca_boundary_hits: null pointer (the strict mode needs the word ids)");
    WCA_CHECK_ARG(n_problems >= 0, "wca_boundary_hits: n_problems=%d", n_problems);
    WCA_CHECK_ARG(tolerance >= 0.0, "wca_boundary_hits: tolerance %g must be a non-negative number", tolerance);
    if (n_problems == 0) return WCA_OK;
    return launch_boundary_hits(d_end_times, d_utts, d_utt_of, n_problems, d_ref_times, d_ref_off, d_ref_ids, d_hyp_ids,
                                d_hyp_off, tolerance, mode == WCA_HITS_STRICT, d_hits, static_cast<cudaStream_t>(stream));
}

int64_t wca_dtw_workspace_bytes(int n_utts, int max_rows, int max_frames) {
    if (n_utts <= 0 || max_rows <= 0 || max_frames <= 0) return 0;
    return dtw_workspace_bytes(n_utts, max_rows, max_frames);
}

int wca_dtw_align(const float *d_matrix, const wca_utt_t *d_utts, int n_utts, int max_rows, int max_frames,
                  int negate, int32_t *d_path_text, int32_t *d_path_time, int32_t *d_path_len, int32_t *d_jump_frames,
                  const int32_t *d_word_bounds, double *d_start_times, double *d_end_times, void *d_trace_ws,
                  int64_t trace_ws_bytes, wca_stream_t stream) {
    WCA_CHECK_ARG(d_matrix && d_utts, "wca_dtw_align: null pointer");
    WCA_CHECK_ARG((d_path_text == nullptr) == (d_path_time == nullptr), "wca_dtw_align: give both path buffers or none");
    WCA_CHECK_ARG(n_utts >= 0 && max_rows >= 0 && max_frames >= 0, "wca_dtw_align: negative size");
    if (n_utts == 0) return WCA_OK;
    return launch_dtw_align(d_matrix, d_utts, n_utts, max_rows, max_frames, negate, d_path_text, d_path_time,
                            d_path_len, d_jump_frames, d_word_bounds, d_start_times, d_end_times, d_trace_ws,
                            trace_ws_bytes, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
