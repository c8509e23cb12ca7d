/* wca_b200.h -- C ABI of the B200 (sm_100a) alignment hot path.
 *
 * Drop-in boundary for `timing.get_attentions` + `timing.force_align` of
 * 30stomercury/whisper-char-alignment.  The reference is pure Python and has no FFI of
 * its own; each entry point below replaces the reference lines it cites (paths are
 * relative to the reference checkout).  INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer named `d_*` is DEVICE memory owned by the caller; the library never
 *     allocates, frees, or keeps state between calls, and never synchronises the stream;
 *   - `h_*` pointers are HOST memory read during the call only;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*);
 *   - every function returns WCA_OK (0) or a negative wca_status; wca_last_error() gives
 *     a thread-local human-readable message for the last failure on the calling thread;
 *   - a batch is described by an array of wca_utt_t living in DEVICE memory; per-batch
 *     maxima needed for the launch geometry are passed by value.
 *
 * Shapes: L decoder layers, H heads, Dh = 64 head width, T tokens, F frames (max_frames),
 * N = row_end - row_begin DTW rows (T - len(sot_sequence) - 1), W words.
 */
#ifndef WCA_B200_H
#define WCA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WCA_ABI_VERSION 5
#define WCA_MAX_LAYERS 32      /* decoder layers of the largest published Whisper (large-v3) */
#define WCA_MAX_MEDFILT 31     /* odd widths 1..31 */
#define WCA_TOKENS_PER_SECOND 50.0 /* whisper.audio.TOKENS_PER_SECOND, timing.py:10,111 */

typedef void *wca_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define WCA_API __attribute__((visibility("default")))
#else
#define WCA_API
#endif

typedef enum wca_status {
    WCA_OK = 0,
    WCA_ERR_INVALID = -1,     /* bad argument (null pointer, size out of range, even width ...) */
    WCA_ERR_UNSUPPORTED = -2, /* legal request this build cannot serve (e.g. Dh != 64) */
    WCA_ERR_CUDA = -3,        /* a CUDA runtime / driver call failed */
    WCA_ERR_NO_DEVICE = -4    /* no sm_100 device visible */
} wca_status;

/* One utterance of a batch.  Offsets are in ELEMENTS of the buffer they index. */
typedef struct wca_utt {
    int32_t n_tokens;   /* T: teacher-forced tokens = len(sot_sequence)+1+n_text+1 (infer_ali.py:69-76) */
    int32_t n_frames;   /* F: max_frames = n_samples // 320 (infer_ali.py:78)                            */
    int32_t row_begin;  /* first matrix row kept for DTW = len(tokenizer.sot_sequence) (timing.py:102)   */
    int32_t row_end;    /* one past the last kept row = T-1 (timing.py:102)                              */
    int32_t n_words;    /* W: words incl. the trailing EOT word minus one (timing.py:108,112-113)        */
    int32_t n_sel;      /* heads to aggregate for this utterance (topk clipped to n_heads, or preset)    */
    int64_t q_row0;     /* first row of this utterance in every layer's Q matrix                          */
    int64_t k_row0;     /* first row of this utterance in every layer's K matrix                          */
    int64_t ws_off;     /* float offset of the (n_heads, T, F) attention block                            */
    int64_t score_off;  /* float offset of the n_heads scores                                             */
    int64_t sel_off;    /* int32 offset of the selected-head list (n_sel entries, ascending score)        */
    int64_t matrix_off; /* float offset of the (N, F) aggregated matrix                                   */
    int64_t path_off;   /* int32 offset of the path buffers, capacity N+F each                            */
    int64_t jump_off;   /* int32 offset of the N jump frames                                              */
    int64_t word_off;   /* offset of word_boundaries (W+1 int32) and of start/end times (W float64)       */
    int64_t part_off;   /* float offset of the head-score partials (wca_capture_attention d_partials)      */
} wca_utt_t;

WCA_API int wca_abi_version(void);
WCA_API const char *wca_last_error(void);
/* Kernels launched so far by the calling thread through this library (diagnostic counter;
 * bench.py reports its increase over the timed region as gpu_launches). */
WCA_API uint64_t wca_launch_count(void);
/* Number of SMs and compute capability (major*10+minor) of the current device. */
WCA_API int wca_device_info(int *sm_count, int *compute_capability);

/* (1) Cross-attention capture.  Replaces timing.py:50-66 together with the upstream
 * `qkv_attention` it hooks: for every (utterance, layer, head)
 *     logit[t,f] = sum_c (q[t,c] * Dh^-1/4) * (k[f,c] * Dh^-1/4),   f < n_frames
 * then (unless WCA_CAPTURE_RAW_LOGITS) median filter of odd `medfilt_width` along f with
 * reflect padding inside [0, n_frames), times `qk_scale`, softmax over f.
 * h_q_layers / h_k_layers: HOST arrays of L device pointers; layer l's Q is a row-major
 * matrix of q_rows rows with leading dimension ld_q floats whose row (q_row0 + t) holds
 * token t, columns [h*Dh, (h+1)*Dh) belong to head h; likewise K with k_rows, ld_k and
 * frame rows (the row counts bound the TMA tensor maps: rows past them read as zero).
 * Output: d_ws + ws_off, layout (L, H, T, F) fp32, exactly what get_attentions returns.
 * d_partials (may be NULL): head-score partials for wca_head_scores_from_partials, so that scoring the heads
 * (timing.py:17-34) does not read the maps a second time.  Per utterance, at d_partials + part_off, with
 * B = ceil(T / 128) token blocks of 4 groups of 32 rows: [L*H][B][4] floats sum_t ||p[t,:]||_2 over the rows of the
 * group, then [L*H][B][4][F] floats sum_t p[t,f]^2 over the rows of the group (wca_capture_partials_floats floats in
 * all; groups past the last token row are not written).
 * Only the tcgen05 kernel writes them: wca_capture_writes_partials tells for a launch geometry; passing a
 * non-NULL d_partials when it answers 0 is an error. */
#define WCA_CAPTURE_RAW_LOGITS 1u
#define WCA_CAPTURE_FORCE_SIMT 2u /* use the CUDA-core kernel instead of tcgen05 (test cross-check) */
#define WCA_CAPTURE_TRACE 4u      /* debug: CTA 0 records a clock64 timeline, see wca_debug_capture_trace */
WCA_API int wca_capture_attention(const float *const *h_q_layers, const float *const *h_k_layers, int n_layers,
                          int n_heads_per_layer, int head_dim, int64_t ld_q, int64_t ld_k,
                          int64_t q_rows, int64_t k_rows, const wca_utt_t *d_utts, int n_utts, int max_tokens, int max_frames,
                          int medfilt_width, float qk_scale, float *d_ws, float *d_partials, unsigned flags,
                          wca_stream_t stream);
WCA_API int wca_capture_writes_partials(int max_frames, int medfilt_width, unsigned flags);
WCA_API int64_t wca_capture_partials_floats(int n_heads, int n_tokens, int n_frames);

/* Debug only: copies the timeline recorded by the last WCA_CAPTURE_TRACE launch (synchronises
 * the device).  Returns the number of int64 entries written (tiles x events) or a status < 0. */
WCA_API int wca_debug_capture_trace(long long *h_out, int capacity);

/* (1b) Unmasked attention of the teacher-forced forward (timing.py:57-58 `model(mel, tokens)`;
 * upstream whisper/model.py MultiHeadAttention.qkv_attention): the audio encoder's self-attention
 * (n_q = n_kv = 1500) and the OUTPUT of the decoder's cross-attention (n_q = tokens, n_kv = 1500):
 *     out = softmax(q k^T * Dh^-1/2) v   per (batch, head), no mask,
 * fp32 in and out, fp32-grade arithmetic on the tensor cores (3 x tf32 error-compensated products
 * for both contractions).  d_q / d_out are row-major matrices of n_batch * n_q rows, d_k / d_v of
 * n_batch * n_kv rows; row (b * n + t) holds position t of batch item b, columns [h*Dh, (h+1)*Dh)
 * belong to head h; ld_* are the leading dimensions in floats (multiples of 4, pointers 16-byte
 * aligned).  The cross-attention MAPS are not produced here (that is wca_capture_attention). */
WCA_API int wca_full_attention(const float *d_q, const float *d_k, const float *d_v, float *d_out, int n_batch, int n_q,
                       int n_kv, int n_heads, int head_dim, int64_t ld_q, int64_t ld_k, int64_t ld_v, int64_t ld_out,
                       wca_stream_t stream);

/* (1b') The same kernel with the causal mask of the decoder's self-attention (upstream whisper/model.py
 * TextDecoder: `mask = triu(-inf, 1)`, qkv_attention(..., mask)): key j is visible to query i only for j <= i.
 * Same layout and arithmetic as wca_full_attention; key blocks past a tile's last query row are not visited. */
WCA_API int wca_causal_attention(const float *d_q, const float *d_k, const float *d_v, float *d_out, int n_batch, int n_q,
                         int n_kv, int n_heads, int head_dim, int64_t ld_q, int64_t ld_k, int64_t ld_v, int64_t ld_out,
                         wca_stream_t stream);

/* (1b'') Single-query attention of one greedy decode step (upstream whisper/model.py
 * MultiHeadAttention.qkv_attention with a kv_cache): one query row per batch item, every key visible,
 *     out[b, h*Dh:(h+1)*Dh] = softmax_j(q[b,h,:] . k[b,j,h,:] * Dh^-1/2) . v[b,j,h,:],   j < n_kv,
 * fp32 on the CUDA cores.  It serves the decoder's self-attention over its cache of positions 0..p (n_kv = p + 1) and
 * its cross-attention over the encoder rows.  Row b of q / out is at d_q + b*ld_q / d_out + b*ld_out; key j of item b
 * at d_k + b*batch_stride_k + j*ld_k, value j at d_v + b*batch_stride_v + j*ld_v (a preallocated cache of which n_kv
 * rows are live, or one layer's column slice of a grouped K/V projection, is read in place); columns [h*Dh, (h+1)*Dh)
 * belong to head h.  ld_* and the batch strides are multiples of 4 floats, pointers 16-byte aligned; rows at or past
 * n_kv are never read.  The keys are split into chunks whose partial results go to d_workspace (at least
 * wca_decode_attention_workspace_bytes(n_batch, n_heads, n_kv) bytes) and are merged in chunk order: the chunks depend
 * on n_kv only, so a row gives the same bits alone and inside any batch. */
WCA_API int64_t wca_decode_attention_workspace_bytes(int n_batch, int n_heads, int n_kv);
WCA_API int wca_decode_attention(const float *d_q, const float *d_k, const float *d_v, float *d_out,
                                 int n_batch, int n_kv, int n_heads, int head_dim,
                                 int64_t ld_q, int64_t ld_k, int64_t ld_v, int64_t ld_out,
                                 int64_t batch_stride_k, int64_t batch_stride_v,
                                 void *d_workspace, int64_t workspace_bytes, wca_stream_t stream);

/* (1c) Residual add + LayerNorm of the same forward (upstream ResidualAttentionBlock: `x = x + f(ln(x))`,
 * whisper/model.py LayerNorm = fp32 torch layer_norm): y = x + h (skipped when d_h is NULL; written when d_y is
 * not NULL), n = (y - mean(y)) / sqrt(var(y) + eps) * gamma + beta per row, biased variance, fp32.  All
 * matrices are row-major n_rows x width with leading dimension width; width is a multiple of 128. */
WCA_API int wca_add_layernorm(const float *d_x, const float *d_h, const float *d_gamma, const float *d_beta, float *d_y,
                      float *d_n, int64_t n_rows, int width, float eps, wca_stream_t stream);

/* Debug only: while a non-null device buffer of >= 20000 floats is registered, CTA (0,0,0) of
 * wca_full_attention dumps its first logit block, its un-normalised output rows and the
 * softmax statistics there (tools/debug_enc_attn.py).  Pass NULL to stop. */
WCA_API void wca_debug_enc_attn_buffer(float *d_buf);

/* (2) Median filter -> *qk_scale -> softmax over already materialised logits.
 * Replaces timing.py:64-66 (`weights[..., :max_frames]`, whisper.timing.median_filter,
 * `(weights * qk_scale).softmax(-1)`).  d_in holds n_rows rows of ld_in floats of which
 * the first n_frames are used; d_out holds n_rows rows of n_frames floats.  In-place use
 * (d_out == d_in) is allowed when ld_in == n_frames.  If n_frames <= medfilt_width/2 the
 * filter is the identity, as upstream. */
WCA_API int wca_medfilt_softmax(const float *d_in, int64_t n_rows, int64_t ld_in, int n_frames, int medfilt_width,
                        float qk_scale, float *d_out, wca_stream_t stream);

/* (3a) Head scores.  Replaces timing.py:17-34 (filter_attention) and metrics.py:99-111:
 *   score[head] = w_col * sum_f ||a[:,f]||_2 + w_row * sum_t ||a[t,:]||_2
 *                 - w_cov * (sum_f max(sum_t a[t,f], 0.5) - 0.5 F)
 * Terms with a weight <= 0 are skipped exactly as the reference does.  Output
 * d_scores + score_off, n_heads floats per utterance.  Any n_frames; more than 1024 token
 * rows are only accepted with max_frames <= 256 (Whisper caps n_tokens at 448). */
WCA_API int wca_head_scores(const float *d_ws, const wca_utt_t *d_utts, int n_utts, int n_heads, int max_tokens,
                    int max_frames, float w_colnorm, float w_rownorm, float w_coverage, float *d_scores,
                    wca_stream_t stream);

/* (3a') The same scores from the partials of wca_capture_attention (no coverage term: callers with
 * w_coverage > 0 use wca_head_scores).  n_heads = L*H. */
WCA_API int wca_head_scores_from_partials(const float *d_partials, const wca_utt_t *d_utts, int n_utts, int n_heads,
                                  float w_colnorm, float w_rownorm, float *d_scores, wca_stream_t stream);

/* (3b) Top-k head selection.  Replaces timing.py:36 `sorted(scores)[-topk:]`: ascending
 * by (score, layer, head); the last min(topk, n_heads) survive, still ascending.  -0.0 and +0.0
 * tie; NaN scores rank below every number, -inf included, and among themselves by index.  Writes
 * head indices (layer*H + head) to d_sel + sel_off and their scores to d_sel_scores +
 * sel_off (n_sel entries per utterance, n_sel taken from the descriptor). */
WCA_API int wca_topk_heads(const float *d_scores, const wca_utt_t *d_utts, int n_utts, int n_heads, int32_t *d_sel,
                   float *d_sel_scores, wca_stream_t stream);

/* (3c) Aggregation.  Replaces timing.py:86-89 ("mean") and timing.py:95-97 ("topk"):
 *   matrix[t,f] = (1/n_sel) * sum_{i<n_sel} a_i[t,f] / ||a_i[:,f]||_2 ,  heads taken in list order,
 * the column norm running over ALL T rows; rows [row_begin,row_end) are written to
 * d_matrix + matrix_off as (N, F) fp32 (timing.py:102).  max_sel >= 1 is an upper bound of the descriptors' n_sel (a
 * performance hint: launches of single-head aggregations, probe_oracle.py:82-90, get a leaner kernel; the result does
 * not depend on it). */
WCA_API int wca_aggregate_heads(const float *d_ws, const int32_t *d_sel, const wca_utt_t *d_utts, int n_utts,
                        int max_tokens, int max_frames, int max_sel, float *d_matrix, wca_stream_t stream);

/* (3d) Std-normalisation of a head list + mean over it: the stock-Whisper baseline, default_find_alignment
 * (timing.py:156-163).  For every utterance and every i < n_sel of its list d_sel + sel_off, with
 * a = d_ws + ws_off + d_sel[sel_off + i] * T * F of shape (T, F):
 *   mu[f] = (1/T) sum_t a[t,f],   sd[f] = sqrt((1/T) sum_t (a[t,f] - mu[f])^2)   over ALL T rows (unbiased=False, :160)
 *   w_i[t,f] = (a[t,f] - mu[f]) / sd[f]                                            true division: 0/0 is NaN (:161)
 *   matrix[t - row_begin, f] = (1/n_sel) sum_i w_i[t,f]    heads in list order, rows [row_begin, row_end) (:163, :165)
 * The mean and the spread are two passes over the column (no one-pass sum of squares), in a fixed order: the result
 * depends neither on the batch nor on the launch.  w_i goes to d_weights + d_weights_off[u] + i*T*F, laid out
 * (n_sel, T, F) per utterance (the `weights` default_find_alignment returns); d_weights == NULL (then also
 * d_weights_off == NULL) skips it and leaves the matrix bit for bit the same.  d_weights_off: n_utts int64 in DEVICE
 * memory.  Several utterances may share one list (equal sel_off).  n_tokens <= max_tokens <= 448 (Whisper's text
 * context; a larger max_tokens is WCA_ERR_UNSUPPORTED); a descriptor with n_tokens outside [1, max_tokens], n_sel < 1
 * or a row range outside [0, n_tokens] fails the launch. */
WCA_API int wca_normalize_heads(const float *d_ws, const int32_t *d_sel, const wca_utt_t *d_utts, int n_utts,
                        int max_tokens, int max_frames, float *d_weights, const int64_t *d_weights_off, float *d_matrix,
                        wca_stream_t stream);

/* (3e) Token probabilities: the word confidence of upstream whisper.timing.find_alignment,
 *     sampled_logits = logits[len(tokenizer.sot_sequence):, : tokenizer.eot]
 *     token_probs = sampled_logits.softmax(dim=-1)
 *     text_token_probs = token_probs[np.arange(len(text_tokens)), text_tokens].tolist()
 * p[r] = softmax(row_r[0 : n_cols])[target_r] for r < n_rows  (logits[len(sot):, :eot].softmax(-1)[arange, text_tokens]).
 * Rows are read in place: d_rows[r] is the DEVICE address of row r's first logit (any 4-byte alignment, any pitch);
 * columns >= n_cols are never read.  d_rows (n_rows pointers), d_targets (n_rows int32) and d_probs (n_rows floats) are
 * DEVICE memory.  One CTA per row, fixed-order reductions: a row gives the same bits alone, inside any batch and on a
 * repeated launch.
 * torch semantics: any NaN in the row gives NaN; a +inf gives NaN (exp(inf - inf)); an all -inf row gives NaN (0/0);
 * a -inf target in a finite row gives exactly 0.
 * Targets live on the device, so the library cannot check them without synchronising: the caller checks
 * 0 <= target < n_cols on the host before the launch (upstream would raise an IndexError), as the Python binding
 * (_cabi.token_probs) does.  An out-of-range target that reaches the kernel gives NaN for its row, never a read
 * outside the row.  WCA_ERR_INVALID for a null pointer, n_rows < 0 or n_cols < 1; n_rows == 0 does nothing. */
WCA_API int wca_token_probs(const float *const *d_rows, const int32_t *d_targets, int n_rows, int n_cols,
                            float *d_probs, wca_stream_t stream);

/* (3f) Word-boundary hits of many alignments: the hit count of the reference's scoring, metrics.py:22-43 (eval_n1)
 * and metrics.py:45-72 (eval_n1_strict), one count per problem p < n_problems.
 *   y_hat = d_end_times[word_off .. word_off + n_words) of d_utts[p] (float64 seconds, read in place where
 *           wca_dtw_align wrote them with the same descriptors);
 *   y     = d_ref_times[d_ref_off[u] .. d_ref_off[u + 1]) of the reference list u = d_utt_of[p] (float64).
 * WCA_HITS_PLAIN  : eval_n1(y, y_hat, tolerance): greedy in-order two-pointer match, |y[i] - y_hat[j]| <= tolerance
 *                   in double; a pair that orders neither way (NaN) stops the match; an empty y_hat gives 0.
 * WCA_HITS_STRICT : eval_n1_strict's true positives: for each predicted word i in order, the first unused reference
 *                   index j with d_ref_ids[d_ref_off[u] + j] == d_hyp_ids[d_hyp_off[u] + i] and
 *                   |y[j] - y_hat[i]| <= tolerance is taken; NaN never matches.  The ids are the caller's integer
 *                   codes of the normalised words (w.lower().strip(string.punctuation)); hypothesis ids are per
 *                   reference list u, since every problem of one utterance has the same words.  A reference list of
 *                   more than WCA_HITS_MAX_STRICT_REF_WORDS words gives -1 (the caller checks that on the host).
 * n_pred = n_words and n_ref = d_ref_off[u + 1] - d_ref_off[u] in both modes (eval_n1_strict's tp + fp, tp + fn).
 * Every array is DEVICE memory: d_utt_of (n_problems int32), d_ref_off (int64, one past the largest u used),
 * d_hits (n_problems int32); d_ref_ids, d_hyp_ids, d_hyp_off may be NULL in the plain mode.  One warp per problem:
 * a problem gives the same count alone and inside any batch.  Nothing outside d_hits[0 : n_problems) is written.
 * WCA_ERR_INVALID for a null pointer, n_problems < 0, a negative or NaN tolerance or an unknown mode. */
#define WCA_HITS_PLAIN 0
#define WCA_HITS_STRICT 1
#define WCA_HITS_MAX_STRICT_REF_WORDS 1024
WCA_API int wca_boundary_hits(const double *d_end_times, const wca_utt_t *d_utts, const int32_t *d_utt_of, int n_problems,
                              const double *d_ref_times, const int64_t *d_ref_off, const int32_t *d_ref_ids,
                              const int32_t *d_hyp_ids, const int64_t *d_hyp_off, double tolerance, int mode,
                              int32_t *d_hits, wca_stream_t stream);

/* (4) Batched DTW + backtrace + boundary extraction.  Replaces timing.py:103
 * `dtw(-matrix)` (upstream dtw_cpu + backtrace), timing.py:110-111 (jump frames) and
 * timing.py:111-113 (start/end times).  One problem per utterance: cost = -matrix
 * (negate != 0) or +matrix, (N, F) fp32 at d_matrix + matrix_off.  Bit-exact with the
 * CPU recurrence: fp32 round-to-nearest adds, ties and NaN resolve to the time step.
 * Outputs (any of the three groups may be NULL to skip it):
 *   d_path_text/d_path_time + path_off : the path, forward order, occupying the LAST
 *       d_path_len[u] entries of the N+F capacity;
 *   d_jump_frames + jump_off           : N frames, first path point of every text row;
 *   d_word_bounds (in) + word_off      : W+1 int32 token boundaries (timing.py:108),
 *   d_start_times/d_end_times + word_off : W float64 seconds = frame / 50.
 * d_trace_ws: scratch of trace_ws_bytes, only needed when a problem's 2-bit trace does
 * not fit in shared memory (wca_dtw_workspace_bytes tells; 0 for every legal Whisper
 * shape T<=448, F<=1500). */
WCA_API int64_t wca_dtw_workspace_bytes(int n_utts, int max_rows, int max_frames);
WCA_API int wca_dtw_align(const float *d_matrix, const wca_utt_t *d_utts, int n_utts, int max_rows, int max_frames,
                  int negate, int32_t *d_path_text, int32_t *d_path_time, int32_t *d_path_len,
                  int32_t *d_jump_frames, const int32_t *d_word_bounds, double *d_start_times,
                  double *d_end_times, void *d_trace_ws, int64_t trace_ws_bytes, wca_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* WCA_B200_H */
