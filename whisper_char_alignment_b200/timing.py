"""B200-native `timing` module: same entry points, arguments, return conventions and
error behaviour as the reference's timing.py, with the arithmetic on sm_100a kernels.

    get_attentions(mel, tokens, model, tokenizer, max_frames, medfilt_width=7, qk_scale=1.0)
        reference timing.py:45-67
    filter_attention(attns, topk=20, w_colnorm=1, w_rownorm=1, w_coverage=0)
        reference timing.py:13-43
    force_align(ws, tokens, tokenizer, aligned_unit_type='subword', aggregation="mean", topk=-1,
                w_colnorm=1.0, w_rownorm=1.0, w_coverage=0.0)
        reference timing.py:69-114
    word_probabilities_batch(logits_list, text_tokens_list, tokenizer, aligned_unit_type='subword')
        the word confidence of upstream whisper.timing.find_alignment, which the reference drops
    head_boundary_counts_batch(ws_list, tokens_list, tokenizer, ref_ends_list, ...)
        every head's word-boundary hits on its own (reference metrics.py eval_n1 / eval_n1_strict), to find a
        checkpoint's alignment heads
    get_attentions_widths_batch(mels, tokens_list, model, tokenizer, max_frames_list, widths, ...)
        the maps of several median-filter widths from one forward
    alignment_config_counts_batch(maps_by_width, tokens_list, tokenizer, ref_ends_list, configs, ...)
        the word-boundary counts of many (width, aggregation, top-k, score weights) configurations in one pass, to tune
        a checkpoint's alignment settings

plus `*_batch` variants that push many utterances through one launch of each kernel
(the reference is strictly one utterance at a time, infer_ali.py:48,57).

How it differs underneath (results identical, see DESIGN.md):
  * the model runs with SDPA on; instead of hooking `cross_attn` for a materialised
    (1,H,T,1500) `qk`, the outputs of `cross_attn.query` / `cross_attn.key` are tapped and
    the capture kernel writes the trimmed, filtered, soft-maxed (L,H,T,F) maps directly;
  * head scoring, top-k, aggregation, DTW, backtrace and boundary extraction run
    back-to-back on the device; one device->host copy at the end replaces the reference's
    L*H `.item()` syncs and the `.cpu()` before DTW.

There is no CPU path here: tensors must be CUDA tensors and the extension must be built.
"""
from __future__ import annotations

import os
import string
from typing import NamedTuple, Sequence

import numpy as np
import torch

from . import _cabi
from .retokenize import split_tokens_on_spaces

TOKENS_PER_SECOND = 50  # whisper.audio: SAMPLE_RATE // (HOP_LENGTH * 2)

__all__ = [
    "get_attentions", "get_attentions_batch", "filter_attention", "force_align", "force_align_batch",
    "dtw", "dtw_batch", "median_filter_softmax", "default_find_alignment", "default_find_alignment_batch",
    "probe_heads_batch", "word_probabilities_batch", "head_boundary_counts_batch", "strict_word_ids",
    "get_attentions_widths_batch", "alignment_config_counts_batch",
]


# ---------------------------------------------------------------------------------
# get_attentions
# ---------------------------------------------------------------------------------
class _CrossAttentionTap:
    """Forward hooks on every decoder block's cross_attn.query / cross_attn.key."""

    def __init__(self, model):
        self.blocks = list(model.decoder.blocks)
        self.q = [None] * len(self.blocks)
        self.k = [None] * len(self.blocks)
        self._handles = []

    def __enter__(self):
        for idx, blk in enumerate(self.blocks):
            ca = blk.cross_attn
            self._handles.append(ca.query.register_forward_hook(lambda _m, _i, out, idx=idx: self.q.__setitem__(idx, out)))
            self._handles.append(ca.key.register_forward_hook(lambda _m, _i, out, idx=idx: self.k.__setitem__(idx, out)))
        return self

    def __exit__(self, *exc):
        for h in self._handles:
            h.remove()
        self._handles = []
        return False


_FRAMES_PER_CTA = 224  # csrc/capture_tc.cu: kMaxOwn

#: Head-score partials from the capture epilogue: "1" (default) always, "0" never, "auto" only for batches whose
#: utterances all fit one CTA along the frames (<= 224 frames).  The partials cost the epilogue warps ~15 % more
#: instructions and save the second read of the maps.  Measured on one B200 inside bench.py (capture + scoring):
#: TIMIT-shaped batch of 32: 0.378 + 0.026 ms with, 0.363 + 0.137 ms without; LibriSpeech-shaped drain of 800 utterances:
#: 251.9 + 3.5 ms with, 233.7 + 51.2 ms without.
SCORE_PARTIALS = os.environ.get("WCA_SCORE_PARTIALS", "1")


def _cluster_bucket(n_frames: int) -> int:
    """Cluster size (1-6 or 8 CTAs along frames, 224 frames each) the capture kernel uses for this utterance; the same
    rule as launch_capture_tc (csrc/capture_tc.cu), which derives it from the longest utterance of a launch."""
    size = max(1, -(-n_frames // _FRAMES_PER_CTA))
    return 8 if size >= 7 else size


def _as_f32_rows(t: torch.Tensor) -> torch.Tensor:
    """fp32 rows with unit stride along the width; evenly strided rows are kept as they are (the product model hands
    over column slices of its fused projections), anything else is made contiguous."""
    t = t.detach()
    if t.dtype != torch.float32:
        t = t.float()
    if t.stride(-1) == 1 and all(t.shape[d] == 1 or t.stride(d) == t.stride(d + 1) * t.shape[d + 1] for d in range(t.dim() - 2)):
        return t
    return t.contiguous()


class _ScorePartials:
    """Head-score partials of one utterance's maps, attached to the tensor get_attentions returns.  Valid only for
    that very tensor object as long as nobody has written to it (the version counter is checked): a view, a copy or a
    modified tensor is scored by reading the maps, like any other input."""

    __slots__ = ("buffer", "offset", "version", "data_ptr", "shape")

    def __init__(self, buffer, offset, maps):
        self.buffer, self.offset = buffer, offset
        self.version, self.data_ptr, self.shape = maps._version, maps.data_ptr(), tuple(maps.shape)

    @staticmethod
    def of(maps):
        p = getattr(maps, "_wca_score_partials", None)
        if p is None or p.version != maps._version or p.data_ptr != maps.data_ptr() or p.shape != tuple(maps.shape):
            return None
        return p


def get_attentions_batch(mels, tokens_list: Sequence[torch.Tensor], model, tokenizer, max_frames_list,
                         medfilt_width: int = 7, qk_scale: float = 1.0, *, raw_logits: bool = False,
                         force_simt: bool = False, audio_features=None):
    """Batched get_attentions.  mels: (B, n_mels, n_frames_in) tensor or list of (n_mels, n_frames_in);
    tokens_list: B 1-D int64 tensors; max_frames_list: B ints.  audio_features: the encoder output of the batch,
    (B, n_audio_ctx, d), when it has already been computed (e.g. by the transcription step): the encoder is skipped and
    `mels` may be None.
    Returns ([weights_b (L,H,T_b,F_b) fp32], [logits_b (T_b, V) fp32])."""
    fwd = _cross_qk_forward(mels, tokens_list, model, max_frames_list, audio_features)
    flags = (_cabi.WCA_CAPTURE_RAW_LOGITS if raw_logits else 0) | (_cabi.WCA_CAPTURE_FORCE_SIMT if force_simt else 0)
    return _capture(fwd, model.dims.n_text_head, medfilt_width, qk_scale, flags)


def get_attentions_widths_batch(mels, tokens_list: Sequence[torch.Tensor], model, tokenizer, max_frames_list, widths,
                                qk_scale: float = 1.0, *, audio_features=None):
    """get_attentions_batch for several median-filter widths from ONE forward: the teacher-forced forward runs once and
    the capture kernel runs once per width on the same Q/K.  Arguments as get_attentions_batch; widths: odd ints.
    Returns {width: (weights, logits)} in the order of `widths` (a repeated width is captured once), each value what
    get_attentions_batch(..., medfilt_width=width, qk_scale=qk_scale) returns bit for bit, head-score partials
    included; the logits are the same tensors for every width."""
    widths = list(dict.fromkeys(int(w) for w in widths))
    if not widths:
        raise ValueError("get_attentions_widths_batch: no median-filter width given")
    fwd = _cross_qk_forward(mels, tokens_list, model, max_frames_list, audio_features)
    return {w: _capture(fwd, model.dims.n_text_head, w, qk_scale, 0) for w in widths}


class _CrossQK(NamedTuple):
    """The forward half of get_attentions_batch: every decoder layer's cross-attention Q (B*t_max rows) and K, the
    logits, the token and frame counts of the batch."""

    q_layers: list
    k_layers: list
    logits: torch.Tensor
    lens: list
    frames: list
    t_max: int


def _cross_qk_forward(mels, tokens_list, model, max_frames_list, audio_features) -> _CrossQK:
    if audio_features is None:
        if isinstance(mels, (list, tuple)):
            mels = torch.stack(list(mels))
        B = mels.shape[0]
        device = mels.device
    else:
        B = audio_features.shape[0]
        device = audio_features.device
    if device.type != "cuda":
        raise _cabi.WcaError("get_attentions: tensors must be on a CUDA device (no CPU fallback exists)")
    n_ctx = model.dims.n_audio_ctx
    lens = [int(t.shape[0]) for t in tokens_list]
    frames = [int(f) for f in max_frames_list]
    if len(lens) != B or len(frames) != B:
        raise ValueError("mels, tokens and max_frames must have the same batch length")
    for f in frames:
        if not 1 <= f <= n_ctx:
            raise ValueError(f"max_frames={f} outside [1, {n_ctx}]")
    t_max = max(lens)
    # right-pad with each sequence's own last token: causal masking hides the padding
    tok = torch.stack([
        torch.cat([t.to(device), t[-1:].to(device).expand(t_max - t.shape[0])]) if t.shape[0] < t_max else t.to(device)
        for t in tokens_list
    ])

    if hasattr(model, "forward_with_cross_qk"):
        # the product model hands the projections over itself (its cross-attention K of all layers comes from ONE GEMM,
        # so there is no per-layer `key` module call to hook)
        with torch.no_grad():
            out_logits, qs, ks = model.forward_with_cross_qk(mels, tok, audio_features=audio_features)
    else:
        with torch.no_grad(), _CrossAttentionTap(model) as tap:
            out_logits = model(mels, tok) if audio_features is None else model.decoder(tok, audio_features)
        qs, ks = tap.q, tap.k
    return _CrossQK([_as_f32_rows(q) for q in qs], [_as_f32_rows(k) for k in ks], out_logits, lens, frames, t_max)


def _capture(fwd: _CrossQK, n_heads, medfilt_width, qk_scale, flags):
    """The capture half of get_attentions_batch: the maps of one median-filter width from the forward's Q/K."""
    q_layers, k_layers, out_logits, lens, frames, t_max = fwd
    B, n_layers, device = len(lens), len(q_layers), q_layers[0].device
    # head-score partials: the capture epilogue holds every map value anyway, so it also leaves sum_t ||p[t,:]||_2 and
    # the column sums of squares behind; force_align / filter_attention then score the heads without reading the maps
    with_partials = SCORE_PARTIALS != "0" and _cabi.capture_writes_partials(max(frames), int(medfilt_width), flags)
    if SCORE_PARTIALS == "auto" and max(frames) > _FRAMES_PER_CTA:
        with_partials = False  # see SCORE_PARTIALS
    recs = np.zeros(B, dtype=_cabi.UTT_DTYPE)
    off = part_off = 0
    for b in range(B):
        recs[b]["n_tokens"], recs[b]["n_frames"] = lens[b], frames[b]
        recs[b]["q_row0"], recs[b]["k_row0"] = b * t_max, b * k_layers[0].shape[1]
        recs[b]["ws_off"] = off
        recs[b]["part_off"] = part_off
        off += n_layers * n_heads * lens[b] * frames[b]
        part_off += _cabi.capture_partials_floats(n_layers * n_heads, lens[b], frames[b]) if with_partials else 0
    ws = torch.empty(off, dtype=torch.float32, device=device)
    partials = torch.empty(part_off, dtype=torch.float32, device=device) if with_partials else None
    # One launch per frame-count bucket: the capture kernel spreads an utterance's frames over a
    # cluster of 1-6 or 8 CTAs (224 frames each) and the cluster size is a launch parameter, so
    # short utterances must not share a launch with 30 s ones.
    buckets = {}
    for b in range(B):
        buckets.setdefault(_cluster_bucket(frames[b]), []).append(b)
    for _, members in sorted(buckets.items()):
        sub = recs[members]
        d_utts = _cabi.upload_utts(sub, device)
        _cabi.capture_attention(q_layers, k_layers, n_heads, None, None, d_utts, len(members),
                                int(sub["n_tokens"].max()), int(sub["n_frames"].max()), int(medfilt_width),
                                float(qk_scale), ws, flags, partials)
    weights, logits = [], []
    for b in range(B):
        n = n_layers * n_heads * lens[b] * frames[b]
        w = ws[recs[b]["ws_off"]: recs[b]["ws_off"] + n].view(n_layers, n_heads, lens[b], frames[b])
        if with_partials:
            w._wca_score_partials = _ScorePartials(partials, int(recs[b]["part_off"]), w)
        weights.append(w)
        logits.append(out_logits[b, : lens[b]])
    return weights, logits


def get_attentions(mel, tokens, model, tokenizer, max_frames, medfilt_width=7, qk_scale=1.0):
    """Drop-in for reference timing.py:45-67.  `tokenizer` is accepted and unused, as there."""
    weights, logits = get_attentions_batch(mel.unsqueeze(0), [tokens], model, tokenizer, [int(max_frames)],
                                           medfilt_width, qk_scale)
    return weights[0], logits[0]


def median_filter_softmax(logits: torch.Tensor, max_frames: int, medfilt_width: int = 7, qk_scale: float = 1.0):
    """timing.py:64-66 on already materialised logits (..., n_ctx): trim, median filter,
    scale, softmax.  For callers that captured `qk` themselves (e.g. a stock upstream hook)."""
    if logits.device.type != "cuda":
        raise _cabi.WcaError("median_filter_softmax: CUDA tensor required")
    x = _as_f32_rows(logits)
    ld = x.shape[-1]
    rows = x.numel() // ld
    out = torch.empty(*x.shape[:-1], int(max_frames), dtype=torch.float32, device=x.device)
    _cabi.medfilt_softmax(x, rows, ld, int(max_frames), int(medfilt_width), float(qk_scale), out)
    return out


# ---------------------------------------------------------------------------------
# device-side plan shared by filter_attention / force_align
# ---------------------------------------------------------------------------------
class _Plan:
    """Offsets of one batch inside the flat work buffers + the uploaded descriptors."""

    def __init__(self, ws_list, row_begin, n_sel_list, word_counts=None, *, shared_sel=False):
        self.B = B = len(ws_list)
        # head-score partials left by the capture kernel: usable when every utterance carries valid ones in ONE buffer
        parts = [_ScorePartials.of(w) for w in ws_list]
        self.partials = None
        if all(p is not None for p in parts) and all(p.buffer is parts[0].buffer for p in parts):
            self.partials = parts[0].buffer
        self.device = ws_list[0].device
        self.base_ptr = ws_list[0].data_ptr()
        for w in ws_list:
            if w.device != self.device or w.dtype != torch.float32 or not w.is_contiguous():
                raise _cabi.WcaError("attention maps must be contiguous fp32 CUDA tensors on one device")
        shapes = np.array([w.shape for w in ws_list], dtype=np.int64).reshape(B, 4)
        heads = shapes[:, 0] * shapes[:, 1]
        if (heads != heads[0]).any():
            raise ValueError("all utterances of a batch must have the same number of heads")
        self.n_heads = int(heads[0])
        T, F = shapes[:, 2], shapes[:, 3]
        delta = np.array([w.data_ptr() for w in ws_list], dtype=np.int64) - self.base_ptr
        assert (delta % 4 == 0).all()
        n_sel = np.asarray(n_sel_list, dtype=np.int64)
        n_words = np.zeros(B, dtype=np.int64) if word_counts is None else np.asarray(word_counts, dtype=np.int64)
        row_end = np.maximum(T - 1, row_begin)
        n_rows = row_end - row_begin

        def starts(sizes):  # exclusive prefix sum
            return np.concatenate([[0], np.cumsum(sizes)[:-1]]) if B else np.zeros(0, dtype=np.int64)

        recs = np.zeros(B, dtype=_cabi.UTT_DTYPE)
        recs["n_tokens"], recs["n_frames"] = T, F
        recs["row_begin"], recs["row_end"] = row_begin, row_end
        recs["n_sel"], recs["n_words"] = n_sel, n_words
        recs["ws_off"] = delta // 4
        recs["score_off"] = starts(heads)
        recs["sel_off"] = 0 if shared_sel else starts(n_sel)  # shared_sel: every utterance reads the same head list
        recs["matrix_off"] = starts(n_rows * F)
        recs["path_off"] = starts(n_rows + F)
        recs["jump_off"] = starts(n_rows)
        recs["word_off"] = starts(n_words + 1)
        if self.partials is not None:
            recs["part_off"] = [p.offset for p in parts]
        self.recs = recs
        self.totals = dict(score=int(heads.sum()), sel=int(n_sel.sum()), matrix=int((n_rows * F).sum()),
                           path=int((n_rows + F).sum()), jump=int(n_rows.sum()), word=int((n_words + 1).sum()))
        self.max_tokens = int(T.max())
        self.max_frames = int(F.max())
        self.max_rows = int(n_rows.max())
        self.d_utts = _cabi.upload_utts(recs, self.device)


def _score_and_select(plan: _Plan, w_colnorm, w_rownorm, w_coverage):
    dev = plan.device
    scores = torch.empty(plan.totals["score"], dtype=torch.float32, device=dev)
    sel = torch.empty(max(plan.totals["sel"], 1), dtype=torch.int32, device=dev)
    sel_scores = torch.empty(max(plan.totals["sel"], 1), dtype=torch.float32, device=dev)
    if plan.partials is not None and not w_coverage > 0:
        # the capture kernel already reduced the maps: finish the sums instead of reading the maps again
        _cabi.head_scores_from_partials(plan.partials, plan.d_utts, plan.B, plan.n_heads, w_colnorm, w_rownorm, scores)
    else:
        _cabi.head_scores(plan.base_ptr, plan.d_utts, plan.B, plan.n_heads, plan.max_tokens, plan.max_frames,
                          w_colnorm, w_rownorm, w_coverage, scores)
    _cabi.topk_heads(scores, plan.d_utts, plan.B, plan.n_heads, sel, sel_scores)
    return scores, sel, sel_scores


def _score_table(sel_host, score_host, n_heads_per_layer):
    return [
        (float(s), (int(i) // n_heads_per_layer, int(i) % n_heads_per_layer),
         f"sample_layer{int(i) // n_heads_per_layer}_head{int(i) % n_heads_per_layer}")
        for i, s in zip(sel_host, score_host)
    ]


def filter_attention(attns, topk=20, w_colnorm=1, w_rownorm=1, w_coverage=0):
    """Drop-in for reference timing.py:13-43.  attns: (layers, heads, tokens, frames).
    Returns ([attns[l,h].unsqueeze(0) ...] ascending by score, [(score, (l,h), name) ...])."""
    attns = attns if attns.is_contiguous() else attns.contiguous()
    n_heads = attns.shape[0] * attns.shape[1]
    # python slicing semantics of `sorted(scores)[-topk:]`
    if topk > 0:
        k = min(int(topk), n_heads)
    elif topk == 0:
        k = n_heads
    else:
        k = max(n_heads + int(topk), 0)
    plan = _Plan([attns], 0, [k])
    _, sel, sel_scores = _score_and_select(plan, w_colnorm, w_rownorm, w_coverage)
    sel_h = sel[:k].cpu().numpy()
    score_h = sel_scores[:k].cpu().numpy()
    H = attns.shape[1]
    table = _score_table(sel_h, score_h, H)
    return [attns[l, h].unsqueeze(0) for _, (l, h), _ in table], table


# ---------------------------------------------------------------------------------
# force_align
# ---------------------------------------------------------------------------------
_SENTINEL = lambda: [[], [], [], [], None]  # noqa: E731  (what the reference returns on EOT-only input)


def force_align_batch(ws_list, tokens_list, tokenizer, aligned_unit_type="subword", aggregation="mean", topk=-1,
                      w_colnorm=1.0, w_rownorm=1.0, w_coverage=0.0, *, return_matrix=True):
    """Batched force_align: one launch per stage for the whole list, one sync at the end.
    Returns a list with, per utterance, what reference force_align returns.  `return_matrix=False` leaves the
    aggregated matrices on the device (the tuple carries None): the head sweep of probe_oracle.py reads only the
    words and the end times of each of its 360 alignments per utterance."""
    B = len(ws_list)
    if B == 0:
        return []
    if aggregation not in ("mean", "topk", "grad_norm"):
        # the reference falls through to `matrix[...]` with `matrix` never bound (timing.py:102)
        raise UnboundLocalError("cannot access local variable 'matrix' where it is not associated with a value")
    if aggregation == "topk":
        assert topk > 0
    sot_len = len(tokenizer.sot_sequence)

    # host side: word grouping defines the boundaries the device gathers (timing.py:105-108)
    words_all, wb_all, seen = [], [], {}
    for toks in tokens_list:
        hit = seen.get(id(toks))  # the probe sweep passes the same list once per head
        if hit is None:
            words, word_tokens = split_tokens_on_spaces(list(toks) + [tokenizer.eot], tokenizer, aligned_unit_type)
            hit = ((words, word_tokens), np.pad(np.cumsum([len(t) for t in word_tokens[:-1]]), (1, 0)).astype(np.int32))
            seen[id(toks)] = hit
        words_all.append(hit[0])
        wb_all.append(hit[1])
    word_counts = [max(len(wt) - 1, 0) for _, wt in words_all]

    if aggregation == "grad_norm":
        maps = [w.reshape(1, 1, *w.shape[-2:]) for w in ws_list]  # caller-provided (T, F) matrices
        maps = [m if m.is_contiguous() else m.contiguous() for m in maps]
    else:
        maps = [w if w.is_contiguous() else w.contiguous() for w in ws_list]
    L = [m.shape[0] for m in maps]
    H = [m.shape[1] for m in maps]
    if aggregation == "topk":
        n_sel = [min(int(topk), l * h) for l, h in zip(L, H)]
    else:
        n_sel = [(l - l // 2) * h for l, h in zip(L, H)]  # "mean": layers L//2 .. L-1 (timing.py:87-88)
    plan = _Plan(maps, sot_len, n_sel, word_counts)
    dev = plan.device

    sel_scores = None
    if aggregation == "topk":
        _, sel, sel_scores = _score_and_select(plan, w_colnorm, w_rownorm, w_coverage)
    else:
        sel_host = np.concatenate([np.arange((l // 2) * h, l * h, dtype=np.int32) for l, h in zip(L, H)])
        sel = torch.from_numpy(sel_host).to(dev, non_blocking=True)

    matrix = torch.empty(max(plan.totals["matrix"], 1), dtype=torch.float32, device=dev)
    if aggregation == "grad_norm":
        for b, m in enumerate(maps):  # matrix = ws[sot_len:-1] (timing.py:99-102)
            r = plan.recs[b]
            n = int(r["row_end"] - r["row_begin"]) * int(r["n_frames"])
            matrix[int(r["matrix_off"]): int(r["matrix_off"]) + n].copy_(m[0, 0, int(r["row_begin"]): int(r["row_end"])].reshape(-1))
    else:
        _cabi.aggregate_heads(plan.base_ptr, sel, plan.d_utts, B, plan.max_tokens, plan.max_frames, matrix,
                              max_sel=int(plan.recs["n_sel"].max()))

    wb_flat = np.concatenate([
        np.pad(wb, (0, wc + 1 - len(wb))) if len(wb) < wc + 1 else wb[: wc + 1] for wb, wc in zip(wb_all, word_counts)
    ]).astype(np.int32)
    d_wb = torch.from_numpy(wb_flat).to(dev, non_blocking=True)
    times = torch.empty(2, plan.totals["word"], dtype=torch.float64, device=dev)
    trace_bytes = _cabi.dtw_workspace_bytes(B, plan.max_rows, plan.max_frames)
    trace_ws = torch.empty(trace_bytes, dtype=torch.uint8, device=dev) if trace_bytes else None
    _cabi.dtw_align(matrix.data_ptr(), plan.d_utts, B, plan.max_rows, plan.max_frames, True, word_bounds=d_wb,
                    start_times=times[0], end_times=times[1], trace_ws=trace_ws)

    # the only device->host traffic of the call: matrix (returned to the caller, as the
    # reference does at timing.py:102), W start/end times, k selected heads
    matrix_h = matrix.cpu() if return_matrix else None
    times_h = times.cpu().numpy()
    if sel_scores is not None:
        sel_h = sel.cpu().numpy()
        sel_scores_h = sel_scores.cpu().numpy()

    results = []
    for b in range(B):
        r = plan.recs[b]
        words, word_tokens = words_all[b]
        if len(word_tokens) <= 1:
            results.append(_SENTINEL())
            continue
        n_rows, F = int(r["row_end"] - r["row_begin"]), int(r["n_frames"])
        mo, wo, W = int(r["matrix_off"]), int(r["word_off"]), word_counts[b]
        scores = None
        if sel_scores is not None:
            so, k = int(r["sel_off"]), int(r["n_sel"])
            scores = _score_table(sel_h[so: so + k], sel_scores_h[so: so + k], H[b])
        results.append((words, times_h[0, wo: wo + W].copy(), times_h[1, wo: wo + W].copy(),
                        matrix_h[mo: mo + n_rows * F].view(n_rows, F) if return_matrix else None, scores))
    return results


def force_align(ws, tokens, tokenizer, aligned_unit_type="subword", aggregation="mean", topk=-1,
                w_colnorm=1.0, w_rownorm=1.0, w_coverage=0.0):
    """Drop-in for reference timing.py:69-114.
    ws: (layers, heads, tokens, frames) attention weights ((T, F) for aggregation='grad_norm');
    tokens: python list of the text tokens only.
    Returns (words, start_times, end_times, matrix, scores) or the list [[], [], [], [], None]
    when only EOT remains."""
    return force_align_batch([ws], [tokens], tokenizer, aligned_unit_type, aggregation, topk, w_colnorm, w_rownorm,
                             w_coverage)[0]


def probe_heads_batch(ws_list, tokens_list, tokenizer, aligned_unit_type="subword", n_heads=360, w_colnorm=1.0,
                      w_rownorm=1.0, w_coverage=0.0, *, return_matrix=False):
    """The head sweep of reference probe_oracle.py:82-90 for a batch of utterances: rank the heads
    (`filter_attention(w, topk=n_heads)`, :83), then align EVERY kept head on its own
    (`force_align(w.unsqueeze(0), ..., aggregation="mean", topk=1)`, :89-90 -- with a single head the "mean" branch is
    that head L2-normalised over tokens).  The reference does this with n_heads sequential force_align calls per
    utterance; here all utterances' scores come from one launch and all B * n_heads single-head DTW problems from one
    launch per stage.  Returns, per utterance, (outs, scores): scores as filter_attention returns them (ascending),
    outs[i] what force_align returns for the head of scores[i]."""
    B = len(ws_list)
    if B == 0:
        return []
    ws_list = [w if w.is_contiguous() else w.contiguous() for w in ws_list]
    total = [w.shape[0] * w.shape[1] for w in ws_list]
    k = [min(int(n_heads), t) if n_heads > 0 else (t if n_heads == 0 else max(t + int(n_heads), 0)) for t in total]
    plan = _Plan(ws_list, 0, k)
    _, sel, sel_scores = _score_and_select(plan, w_colnorm, w_rownorm, w_coverage)
    sel_h, score_h = sel.cpu().numpy(), sel_scores.cpu().numpy()
    tables, head_lists = [], []
    for b, w in enumerate(ws_list):
        so = int(plan.recs[b]["sel_off"])
        tables.append(_score_table(sel_h[so: so + k[b]], score_h[so: so + k[b]], w.shape[1]))
        head_lists.append(sel_h[so: so + k[b]].astype(np.int64))
    outs = _align_single_heads(ws_list, head_lists, tokens_list, tokenizer, aligned_unit_type, return_matrix)
    return [(outs[b], tables[b]) for b in range(B)]


def _align_single_heads(ws_list, head_lists, tokens_list, tokenizer, aligned_unit_type, return_matrix):
    """force_align(w[l, h][None, None], tokens, aggregation="mean", topk=1) for every listed head of every utterance
    (probe_oracle.py:89-90), as ONE aggregation launch and ONE DTW launch (_launch_single_heads).  Returns, per
    utterance, the list of what force_align returns per head."""
    B = len(ws_list)
    if sum(len(h) for h in head_lists) == 0:
        return [[] for _ in range(B)]
    sh = _launch_single_heads(ws_list, head_lists, tokens_list, tokenizer, aligned_unit_type)
    matrix_h = sh.matrix.cpu() if return_matrix else None
    times_h = sh.times.cpu().numpy()
    out, p = [], 0
    word_off, matrix_off = sh.recs["word_off"], sh.recs["matrix_off"]
    for b in range(B):
        words, word_tokens = sh.words_all[b]
        W, per_head = int(sh.n_words[b]), []
        for _ in range(len(head_lists[b])):
            if len(word_tokens) <= 1:
                per_head.append(_SENTINEL())
            else:
                wo = int(word_off[p])
                m = None
                if return_matrix:
                    mo, nr, nf = int(matrix_off[p]), int(sh.n_rows[p]), int(sh.recs["n_frames"][p])
                    m = matrix_h[mo: mo + nr * nf].view(nr, nf)
                per_head.append((words, times_h[0, wo: wo + W], times_h[1, wo: wo + W], m, None))
            p += 1
        out.append(per_head)
    return out


class _Problems(NamedTuple):
    """What _launch_problems leaves on the device and on the host: `times` (2, sum of W+1) float64 start / end times
    at each problem's word_off, `matrix` the aggregated matrices, `recs` / `d_utts` the P problems' descriptors,
    `utt_of` the utterance of every problem, `words_all` per utterance the (words, word_tokens) grouping, `n_words` per
    utterance, `n_rows` per problem."""

    times: torch.Tensor
    matrix: torch.Tensor
    recs: np.ndarray
    d_utts: torch.Tensor
    words_all: list
    n_words: np.ndarray
    utt_of: np.ndarray
    n_rows: np.ndarray


def _launch_single_heads(ws_list, head_lists, tokens_list, tokenizer, aligned_unit_type):
    """The single-head alignments of _align_single_heads, left on the device: ONE aggregation launch and ONE DTW launch
    for the P = sum_b len(head_lists[b]) >= 1 problems, no copy back.  Utterance b's heads are problems
    sum(len(head_lists[:b])) .. in list order.  The descriptors are built with numpy from the utterances' base offsets
    (no per-head tensor views: a sweep of 32 utterances is 12 288 problems)."""
    B = len(ws_list)
    base_ptr = ws_list[0].data_ptr()
    n_heads = np.array([len(h) for h in head_lists], dtype=np.int64)
    utt_of = np.repeat(np.arange(B), n_heads)
    shapes = np.array([w.shape[2:] for w in ws_list], dtype=np.int64).reshape(B, 2)
    off = (np.array([w.data_ptr() for w in ws_list], dtype=np.int64) - base_ptr) // 4
    head = np.concatenate(head_lists).astype(np.int64)
    ws_off = off[utt_of] + head * (shapes[:, 0] * shapes[:, 1])[utt_of]  # the block of that head: its head list is [0]
    P = len(utt_of)
    sel = torch.zeros(P, dtype=torch.int32, device=ws_list[0].device)
    return _launch_problems(shapes, [(ws_list, sel, utt_of, ws_off, np.arange(P), np.ones(P, dtype=np.int64))],
                            tokens_list, tokenizer, aligned_unit_type)


def _launch_problems(shapes, groups, tokens_list, tokenizer, aligned_unit_type):
    """force_align_batch's aggregation and DTW for P >= 1 alignment problems over B utterances, left on the device, no
    copy back.  Every problem aggregates a list of heads of one utterance's maps (rows len(sot_sequence) .. T-2, the
    utterance's words); several problems may share an utterance.
    shapes: (B, 2) ints, (T, F) of every utterance's maps.
    groups: runs of consecutive problems whose maps and head lists live in the same buffers, one aggregation launch
    each: (ws_list, sel, utt_of, ws_off, sel_off, n_sel) with ws_list the maps of the run (ws_list[0] the base that the
    float offsets ws_off count from), sel the int32 device buffer of the head lists, and per problem of the run its
    utterance, the offset of its maps, the offset and the length of its head list in sel.
    ONE DTW launch for all P problems."""
    B = len(tokens_list)
    dev = groups[0][1].device
    sot_len = len(tokenizer.sot_sequence)
    words_all, wb_all, n_words = [], [], np.zeros(B, dtype=np.int64)
    for b, toks in enumerate(tokens_list):  # the word grouping is a property of the utterance, not of the problem
        words, word_tokens = split_tokens_on_spaces(list(toks) + [tokenizer.eot], tokenizer, aligned_unit_type)
        words_all.append((words, word_tokens))
        n_words[b] = max(len(word_tokens) - 1, 0)
        wb = np.pad(np.cumsum([len(t) for t in word_tokens[:-1]]), (1, 0)).astype(np.int32)
        wb_all.append(np.pad(wb, (0, int(n_words[b]) + 1 - len(wb))) if len(wb) < n_words[b] + 1 else wb[: int(n_words[b]) + 1])
    T, F = shapes[:, 0], shapes[:, 1]
    utt_of = np.concatenate([g[2] for g in groups]).astype(np.int64)
    P = len(utt_of)
    row_end = np.maximum(T - 1, sot_len)
    n_rows = (row_end - sot_len)[utt_of]
    Fp, Wp = F[utt_of], n_words[utt_of]

    def starts(sizes):  # exclusive prefix sum
        return np.concatenate([[0], np.cumsum(sizes)[:-1]])

    recs = np.zeros(P, dtype=_cabi.UTT_DTYPE)
    recs["n_tokens"], recs["n_frames"] = T[utt_of], Fp
    recs["row_begin"], recs["row_end"] = sot_len, row_end[utt_of]
    recs["n_words"] = Wp
    for k, field in ((3, "ws_off"), (4, "sel_off"), (5, "n_sel")):
        recs[field] = np.concatenate([g[k] for g in groups])
    recs["matrix_off"] = starts(n_rows * Fp)
    recs["path_off"] = starts(n_rows + Fp)
    recs["jump_off"] = starts(n_rows)
    recs["word_off"] = starts(Wp + 1)
    d_utts = _cabi.upload_utts(recs, dev)
    matrix = torch.empty(max(int((n_rows * Fp).sum()), 1), dtype=torch.float32, device=dev)
    max_tokens, max_frames, max_rows = int(T.max()), int(F.max()), int(n_rows.max())
    size, p = _cabi.UTT_DTYPE.itemsize, 0
    for ws_list, sel, u, _, _, n_sel in groups:
        if len(u):
            _cabi.aggregate_heads(ws_list[0].data_ptr(), sel, d_utts[p * size: (p + len(u)) * size], len(u), max_tokens,
                                  max_frames, matrix, max_sel=int(np.max(n_sel)))
        p += len(u)
    # every problem's W+1 word bounds at its word_off: gathered from its utterance's bounds
    wb_cat = np.concatenate(wb_all)
    wb_start = starts(n_words + 1)
    idx = np.repeat(wb_start[utt_of] - recs["word_off"], Wp + 1) + np.arange(int((Wp + 1).sum()))
    d_wb = torch.from_numpy(wb_cat[idx].astype(np.int32)).to(dev, non_blocking=True)
    times = torch.empty(2, int((Wp + 1).sum()), dtype=torch.float64, device=dev)
    trace_bytes = _cabi.dtw_workspace_bytes(P, max_rows, max_frames)
    trace_ws = torch.empty(trace_bytes, dtype=torch.uint8, device=dev) if trace_bytes else None
    _cabi.dtw_align(matrix.data_ptr(), d_utts, P, max_rows, max_frames, True, word_bounds=d_wb, start_times=times[0],
                    end_times=times[1], trace_ws=trace_ws)
    return _Problems(times=times, matrix=matrix, recs=recs, d_utts=d_utts, words_all=words_all, n_words=n_words,
                     utt_of=utt_of, n_rows=n_rows)


def strict_word_ids(word_lists):
    """Per list, int32 ids of its words under eval_n1_strict's normalisation (metrics.py:34-35,
    `w.lower().strip(string.punctuation)`): two words get the same id exactly when eval_n1_strict compares them equal.
    Ids are shared by all the lists of one call."""
    table = {}
    return [np.array([table.setdefault(w.lower().strip(string.punctuation), len(table)) for w in words], dtype=np.int32)
            for words in word_lists]


def head_boundary_counts_batch(ws_list, tokens_list, tokenizer, ref_ends_list, *, aligned_unit_type="subword",
                               tolerance=0.02, ref_words_list=None):
    """Every head's word-boundary accuracy on a batch of utterances: the measurement upstream Whisper chose its
    alignment heads by.  For head (l, h) of utterance b the alignment is force_align(ws_list[b][l, h][None, None],
    tokens_list[b], tokenizer, aligned_unit_type, aggregation="mean") (what probe_heads_batch aligns per head; no head
    scoring is run), scored against ref_ends_list[b] as infer_ali scores it:
        plain  (ref_words_list None): hits = metrics.eval_n1(ref_ends, end_times, tolerance)[0]
        strict (ref_words_list[b] the reference words): hits = tp of metrics.eval_n1_strict(ref_ends, end_times,
               ref_words, " ".join(words[:-1]).split(), tolerance)
    with n_pred = len(end_times) and n_ref = len(ref_ends).  An EOT-only utterance counts (0, 0, len(ref_ends)).
    Returns, per utterance, an int64 array (L, H, 3) of (hits, n_pred, n_ref).
    Strict mode raises IndexError, as eval_n1_strict would index past a list, for an utterance with at least one
    reference boundary and at least one predicted boundary when it has fewer hypothesis words than predicted boundaries
    or fewer reference words than reference boundaries.  The check is made once per utterance, before any head is
    scored, so it is slightly stricter than the reference's loop: that loop reads a missing word only while some
    reference boundary is still unmatched, so a head whose earlier words already matched every reference boundary
    escapes it there.
    All L*H*B alignments take one aggregation and one DTW launch, their scoring one wca_boundary_hits launch that reads
    the end times where the DTW wrote them; the hits are the only device->host copy."""
    B = len(ws_list)
    if len(tokens_list) != B or len(ref_ends_list) != B or (ref_words_list is not None and len(ref_words_list) != B):
        raise ValueError("ws_list, tokens_list, ref_ends_list (and ref_words_list) must have the same batch length")
    if B == 0:
        return []
    for w in ws_list:
        if not w.is_cuda:
            raise _cabi.WcaError("head_boundary_counts: attention maps must be CUDA tensors (no CPU fallback exists)")
    ws_list = [w if w.is_contiguous() else w.contiguous() for w in ws_list]
    L, H = int(ws_list[0].shape[0]), int(ws_list[0].shape[1])
    if any(tuple(w.shape[:2]) != (L, H) for w in ws_list):
        raise ValueError("all utterances of a batch must have the same (layers, heads)")
    sh = _launch_single_heads(ws_list, [np.arange(L * H)] * B, tokens_list, tokenizer, aligned_unit_type)
    return [c.reshape(L, H, 3) for c in _boundary_counts(sh, ref_ends_list, tolerance, ref_words_list)]


def alignment_config_counts_batch(maps_by_width, tokens_list, tokenizer, ref_ends_list, configs, *,
                                  aligned_unit_type="subword", tolerance=0.02, ref_words_list=None):
    """Word-boundary counts of every alignment configuration on a batch of utterances, in one pass over the maps.
    maps_by_width: {medfilt_width: per utterance its (L, H, T, F) maps} (get_attentions_widths_batch's maps);
    configs: (medfilt_width, aggr, topk, w_colnorm, w_rownorm, w_coverage) tuples (tuning.Config), aggr "mean" or
    "topk".  Config c's alignment of utterance b is
        force_align_batch(maps_by_width[c.medfilt_width], tokens_list, tokenizer, aligned_unit_type, c.aggr, c.topk,
                          c.w_colnorm, c.w_rownorm, c.w_coverage)[b]
    scored as infer_ali scores it (eval_n1, or eval_n1_strict with ref_words_list; see head_boundary_counts_batch).
    Returns, per utterance, an int64 array (len(configs), 3) of (hits, n_pred, n_ref).
    As in force_align_batch, topk is capped at L*H and topk <= 0 with aggr "topk" raises AssertionError.  An EOT-only
    utterance counts (0, 0, len(ref_ends)) for every config.  Strict mode raises IndexError as
    head_boundary_counts_batch does; CPU maps raise WcaError.
    Device work: per width, one head-scoring and one top-k launch per weighting of its top-k configs (scores from the
    capture's partials when it left them and w_coverage is not > 0, as _score_and_select chooses) and one aggregation
    launch for all its (utterance, config) problems.  A top-k list for k is the last k entries of the list for the
    largest k of the weighting (the ranking is ascending), so every k reads one ranking.  Configs that align the same
    way (mean configs of one width whatever their weights, top-k configs whose capped k and weights agree) share one
    problem.  Then one DTW launch for every problem of every width, one wca_boundary_hits launch, and the hits are the
    only device->host copy."""
    configs = [tuple(c) for c in configs]
    B = len(tokens_list)
    if len(ref_ends_list) != B or (ref_words_list is not None and len(ref_words_list) != B):
        raise ValueError("tokens_list, ref_ends_list (and ref_words_list) must have the same batch length")
    if not configs:
        raise ValueError("alignment_config_counts_batch: no configuration given")
    for width, aggr, topk, *_ in configs:
        if aggr not in ("mean", "topk"):
            raise ValueError(f"aggregation {aggr!r}: the sweep aligns with 'mean' or 'topk'")
        if aggr == "topk" and not topk > 0:
            raise AssertionError(f"topk={topk}: aggregation 'topk' needs topk > 0 (as force_align)")
        if width not in maps_by_width:
            raise ValueError(f"no maps for median-filter width {width}")
    if B == 0:
        return []
    widths = list(dict.fromkeys(c[0] for c in configs))
    maps = {}
    for width in widths:
        ms = list(maps_by_width[width])
        if len(ms) != B:
            raise ValueError(f"width {width}: {len(ms)} maps for {B} utterances")
        for m in ms:
            if not m.is_cuda:
                raise _cabi.WcaError("alignment_config_counts: attention maps must be CUDA tensors (no CPU fallback exists)")
        maps[width] = [m if m.is_contiguous() else m.contiguous() for m in ms]
    shapes = np.array([m.shape for m in maps[widths[0]]], dtype=np.int64).reshape(B, 4)
    L, H = int(shapes[0, 0]), int(shapes[0, 1])
    for width in widths:
        if not np.array_equal(np.array([m.shape for m in maps[width]], dtype=np.int64).reshape(B, 4), shapes):
            raise ValueError("every width's maps must have the shapes of the first width's")
    if (shapes[:, :2] != (L, H)).any():
        raise ValueError("all utterances of a batch must have the same (layers, heads)")

    # one problem per distinct alignment: (width, "mean") or (width, "topk", weights, k capped at L*H)
    slot_of, slots = [], {}
    for width, aggr, topk, wc, wr, wv in configs:
        key = (width, "mean") if aggr == "mean" else (width, "topk", (wc, wr, wv), min(int(topk), L * H))
        slot_of.append(slots.setdefault(key, len(slots)))
    # problems slot-major, utterances within a slot; slots grouped by width
    keys = sorted(slots, key=lambda k: (widths.index(k[0]), slots[k]))
    renumber = {slots[k]: i for i, k in enumerate(keys)}
    slot_of = np.array([renumber[s] for s in slot_of], dtype=np.int64)

    sot_len = len(tokenizer.sot_sequence)
    n_mean = (L - L // 2) * H  # "mean": layers L//2 .. L-1 (timing.py:87-88)
    groups = []
    for width in widths:
        ms = maps[width]
        dev = ms[0].device
        wkeys = [k for k in keys if k[0] == width]
        weightings = list(dict.fromkeys(k[2] for k in wkeys if k[1] == "topk"))
        k_max = max([k[3] for k in wkeys if k[1] == "topk"], default=0)
        parts, list_off = [], {}
        if any(k[1] == "mean" for k in wkeys):
            parts.append(torch.from_numpy(np.arange(L * H - n_mean, L * H, dtype=np.int32)).to(dev, non_blocking=True))
            list_off["mean"] = 0
        if weightings:
            plan = _Plan(ms, sot_len, [k_max] * B)  # utterance b's ranking at b * k_max
            for wt in weightings:
                _, sel, _ = _score_and_select(plan, *wt)
                list_off[wt] = sum(int(p.numel()) for p in parts)
                parts.append(sel[: B * k_max])
        sel = torch.cat(parts) if len(parts) > 1 else parts[0]
        off = (np.array([m.data_ptr() for m in ms], dtype=np.int64) - ms[0].data_ptr()) // 4
        utt, sel_off, n_sel = [], [], []
        for k in wkeys:
            utt.append(np.arange(B))
            if k[1] == "mean":
                sel_off.append(np.zeros(B, dtype=np.int64))  # every utterance reads the same list
                n_sel.append(np.full(B, n_mean, dtype=np.int64))
            else:
                sel_off.append(list_off[k[2]] + np.arange(B) * k_max + (k_max - k[3]))
                n_sel.append(np.full(B, k[3], dtype=np.int64))
        utt = np.concatenate(utt)
        groups.append((ms, sel, utt, off[utt], np.concatenate(sel_off), np.concatenate(n_sel)))
    sh = _launch_problems(shapes[:, 2:], groups, tokens_list, tokenizer, aligned_unit_type)
    return [c[slot_of] for c in _boundary_counts(sh, ref_ends_list, tolerance, ref_words_list)]


def _boundary_counts(sh, ref_ends_list, tolerance, ref_words_list):
    """The scoring half of head_boundary_counts_batch on the alignments `sh` (_launch_problems) left on the device: per
    utterance b, an int64 (n_b, 3) array of (hits, n_pred, n_ref), one row per problem of b in problem order.  One
    wca_boundary_hits launch, one copy back."""
    B = len(sh.words_all)
    ref_ends = [np.asarray(r, dtype=np.float64).reshape(-1) for r in ref_ends_list]
    ref_ids = hyp_ids = None
    if ref_words_list is not None:
        hyp_words = []
        for b, (words, _) in enumerate(sh.words_all):
            W = int(sh.n_words[b])
            hyp = " ".join(words[:-1]).split()[:W]  # as the CLIs build them (infer_ali.py _align_batch)
            # eval_n1_strict reads hyp_words[i] / ref_words[j] only inside its loop over the reference boundaries
            if W and len(ref_ends[b]) and len(hyp) < W:
                raise IndexError(f"list index out of range: {len(hyp)} hypothesis words for {W} end times (utterance {b})")
            if W and len(ref_words_list[b]) < len(ref_ends[b]):
                raise IndexError(f"list index out of range: {len(ref_words_list[b])} reference words for "
                                 f"{len(ref_ends[b])} reference boundaries (utterance {b})")
            hyp_words.append(hyp + [""] * (W - len(hyp)))  # only without reference boundaries: never compared
        ids = strict_word_ids([list(r)[: len(e)] for r, e in zip(ref_words_list, ref_ends)] + hyp_words)
        # a reference shorter than its boundaries only gets here without predictions: its missing ids match nothing
        ref_ids = [np.pad(i, (0, len(e) - len(i)), constant_values=-1) for i, e in zip(ids[:B], ref_ends)]
        hyp_ids = ids[B:]
    hits = torch.empty(max(len(sh.utt_of), 1), dtype=torch.int32, device=sh.times.device)
    _cabi.boundary_hits(sh.times[1], sh.d_utts, sh.utt_of, ref_ends, tolerance, hits,
                        ref_ids=ref_ids, hyp_ids=hyp_ids, n_pred=sh.recs["n_words"])
    hits_h = hits.cpu().numpy().astype(np.int64)  # the only device->host copy of the call
    order = np.argsort(sh.utt_of, kind="stable")  # problems by utterance, in problem order within one
    bounds = np.concatenate([[0], np.cumsum(np.bincount(sh.utt_of, minlength=B))])
    out = []
    for b in range(B):
        mine = order[bounds[b]: bounds[b + 1]]
        c = np.empty((len(mine), 3), dtype=np.int64)
        c[:, 0] = hits_h[mine]
        c[:, 1] = sh.n_words[b]
        c[:, 2] = len(ref_ends[b])
        out.append(c)
    return out


def word_probabilities_batch(logits_list, text_tokens_list, tokenizer, aligned_unit_type="subword"):
    """Per-word probabilities of upstream whisper.timing.find_alignment for a batch of utterances:
        token_probs = logits[len(sot_sequence):, :eot].softmax(-1)[arange(len(text_tokens)), text_tokens]
        word_probabilities = [mean(token_probs[i:j]) for each word's token range [i, j)]
    logits_list: per utterance the (T_b, V) fp32 CUDA logits of its teacher-forced tokens
    [*sot_sequence, no_timestamps, *text_tokens, eot], as get_attentions_batch returns them (read in place, never
    copied); text_tokens_list: the text tokens.  Words are grouped as force_align groups them
    (split_tokens_on_spaces(tokens + [eot], tokenizer, aligned_unit_type)), so word i is force_align's words[i]; the
    EOT word gets no probability.
    Returns, per utterance, (token_probs float32 (n_text,), word_probs float64 (W,)), the word probabilities the float64
    mean of their tokens' in token order (np.mean, as upstream).  One wca_token_probs launch and one device->host copy
    for the whole batch."""
    B = len(logits_list)
    if len(text_tokens_list) != B:
        raise ValueError("logits_list and text_tokens_list must have the same batch length")
    if B == 0:
        return []
    for lg in logits_list:
        if not lg.is_cuda:
            raise _cabi.WcaError("word_probabilities: logits must be CUDA tensors (no CPU fallback exists)")
        if lg.dtype != torch.float32 or lg.dim() != 2 or lg.stride(-1) != 1:
            raise _cabi.WcaError("word_probabilities: logits must be fp32 (T, V) with unit stride along the vocabulary")
    sot_len = len(tokenizer.sot_sequence)
    n_cols = int(tokenizer.eot)  # the text vocabulary, logits[..., :eot]
    texts = [np.asarray(list(t), dtype=np.int64) for t in text_tokens_list]
    for lg, t in zip(logits_list, texts):
        if lg.shape[0] < sot_len + len(t) or lg.shape[1] < n_cols:
            raise ValueError(f"logits of shape {tuple(lg.shape)} do not cover {len(t)} text tokens after the "
                             f"{sot_len}-token SOT sequence and {n_cols} text-vocabulary columns")
    # device address of row sot_len + i of every utterance
    addrs = np.concatenate([lg.data_ptr() + 4 * lg.stride(0) * (sot_len + np.arange(len(t), dtype=np.int64))
                            for lg, t in zip(logits_list, texts)])
    n_rows = len(addrs)
    probs = torch.empty(max(n_rows, 1), dtype=torch.float32, device=logits_list[0].device)
    _cabi.token_probs(addrs, np.concatenate(texts), n_cols, probs)
    probs_h = probs[:n_rows].cpu().numpy()  # the only device->host copy of the call

    out, off = [], 0
    for toks in texts:
        tp = probs_h[off: off + len(toks)]
        off += len(toks)
        _, word_tokens = split_tokens_on_spaces(toks.tolist() + [tokenizer.eot], tokenizer, aligned_unit_type)
        wb = np.pad(np.cumsum([len(t) for t in word_tokens[:-1]]), (1, 0))
        tp64 = tp.astype(np.float64)  # upstream averages the Python floats of .tolist()
        out.append((tp.copy(), np.array([np.mean(tp64[i:j]) for i, j in zip(wb[:-1], wb[1:])], dtype=np.float64)))
    return out


def default_find_alignment_batch(model, tokenizer, text_tokens_list, mels, max_frames_list, *, medfilt_width=7,
                                 qk_scale=1.0, audio_features=None, word_probabilities=False):
    """The stock-Whisper baseline behind `--default_whisper_timing` (reference timing.py:116-186) for a batch of
    utterances: only `model.alignment_heads` (:156), std/mean normalisation over tokens (:160-161), mean over heads
    (:163), DTW (:165), words grouped on spaces.  text_tokens_list: B lists of text tokens; mels: (B, n_mels, n_frames_in)
    tensor or list of (n_mels, n_frames_in); max_frames_list: B ints; audio_features: as get_attentions_batch takes it
    (mels may then be None).
    Returns, per utterance, what default_find_alignment returns: (words, start_times, end_times,
    weights (n_align, T, F) on the device, None), or [[], [], [], [], None] when only EOT remains.  With
    word_probabilities=True the fifth element is the float64 word-probability array of word_probabilities_batch (words
    grouped with "subword"), where upstream find_alignment carries it; words and times are the same bit for bit.

    One capture (get_attentions_batch), one normalisation launch (wca_normalize_heads) and one DTW launch for the
    whole batch; one device->host copy of the times at the end (plus one wca_token_probs launch and its copy with
    word_probabilities=True)."""
    B = len(text_tokens_list)
    if B == 0:
        return []
    if audio_features is None and isinstance(mels, (list, tuple)):
        mels = torch.stack(list(mels))
    device = mels.device if audio_features is None else audio_features.device
    n_heads = model.dims.n_text_head
    picked = model.alignment_heads.indices().T  # (n, 2) of (layer, head) in the reference's stack order, timing.py:156
    n_align = int(picked.shape[0])
    if n_align == 0:
        raise ValueError("default_find_alignment: the model has no alignment heads")
    sel = (picked[:, 0] * n_heads + picked[:, 1]).to(device=device, dtype=torch.int32)
    tokens = [torch.tensor([*tokenizer.sot_sequence, tokenizer.no_timestamps, *t, tokenizer.eot], device=device)
              for t in text_tokens_list]
    maps, logits = get_attentions_batch(mels, tokens, model, tokenizer, max_frames_list, medfilt_width, qk_scale,
                                        audio_features=audio_features)
    word_probs = None
    if word_probabilities:
        word_probs = [wp for _, wp in word_probabilities_batch(logits, text_tokens_list, tokenizer, "subword")]

    # host side: word grouping defines the boundaries the device gathers (timing.py:167-169)
    words_all, wb_all = [], []
    for toks in text_tokens_list:
        words, word_tokens = split_tokens_on_spaces(list(toks) + [tokenizer.eot], tokenizer, "subword")
        words_all.append((words, word_tokens))
        wb_all.append(np.pad(np.cumsum([len(t) for t in word_tokens[:-1]]), (1, 0)).astype(np.int32))
    word_counts = [max(len(wt) - 1, 0) for _, wt in words_all]

    sot_len = len(tokenizer.sot_sequence)
    plan = _Plan(maps, sot_len, [n_align] * B, word_counts, shared_sel=True)  # rows sot_len .. T-2, timing.py:165
    T = plan.recs["n_tokens"].astype(np.int64)
    F = plan.recs["n_frames"].astype(np.int64)
    w_sizes = n_align * T * F
    w_off = np.concatenate([[0], np.cumsum(w_sizes)[:-1]]).astype(np.int64)
    weights = torch.empty(int(w_sizes.sum()), dtype=torch.float32, device=device)
    d_w_off = torch.from_numpy(w_off).to(device, non_blocking=True)
    matrix = torch.empty(max(plan.totals["matrix"], 1), dtype=torch.float32, device=device)
    _cabi.normalize_heads(plan.base_ptr, sel, plan.d_utts, B, plan.max_tokens, plan.max_frames, matrix, weights, d_w_off)

    wb_flat = np.concatenate([
        np.pad(wb, (0, wc + 1 - len(wb))) if len(wb) < wc + 1 else wb[: wc + 1] for wb, wc in zip(wb_all, word_counts)
    ]).astype(np.int32)
    d_wb = torch.from_numpy(wb_flat).to(device, non_blocking=True)
    times = torch.empty(2, plan.totals["word"], dtype=torch.float64, device=device)
    trace_bytes = _cabi.dtw_workspace_bytes(B, plan.max_rows, plan.max_frames)
    trace_ws = torch.empty(trace_bytes, dtype=torch.uint8, device=device) if trace_bytes else None
    _cabi.dtw_align(matrix.data_ptr(), plan.d_utts, B, plan.max_rows, plan.max_frames, True, word_bounds=d_wb,
                    start_times=times[0], end_times=times[1], trace_ws=trace_ws)
    times_h = times.cpu().numpy()  # the only device->host copy of the call

    results = []
    for b in range(B):
        words, word_tokens = words_all[b]
        if len(word_tokens) <= 1:
            results.append(_SENTINEL())
            continue
        wo, W = int(plan.recs[b]["word_off"]), word_counts[b]
        w = weights[int(w_off[b]): int(w_off[b] + w_sizes[b])].view(n_align, int(T[b]), int(F[b]))
        results.append((words, times_h[0, wo: wo + W].copy(), times_h[1, wo: wo + W].copy(), w,
                        None if word_probs is None else word_probs[b]))
    return results


def default_find_alignment(model, tokenizer, text_tokens, mel, max_frames, *, medfilt_width=7, qk_scale=1.0,
                           word_probabilities=False):
    """Drop-in for reference timing.py:116-186 (the stock-Whisper baseline behind
    `--default_whisper_timing`): only `model.alignment_heads`, std/mean normalisation over
    tokens, mean over heads, DTW, words grouped on spaces.
    Returns (words, start_times, end_times, weights (heads, T, F) on the device, None), the fifth element the word
    probabilities with word_probabilities=True.  A batch of one of default_find_alignment_batch."""
    return default_find_alignment_batch(model, tokenizer, [text_tokens], mel.unsqueeze(0), [max_frames],
                                        medfilt_width=medfilt_width, qk_scale=qk_scale,
                                        word_probabilities=word_probabilities)[0]


# ---------------------------------------------------------------------------------
# dtw (whisper.timing.dtw as the reference calls it at timing.py:103)
# ---------------------------------------------------------------------------------
def dtw_batch(costs: Sequence[torch.Tensor]):
    """costs: list of (N_b, M_b) fp32 CUDA tensors.  Returns [(text_indices, time_indices)] int64 numpy,
    bit-identical to upstream dtw_cpu on the same matrix."""
    B = len(costs)
    xs = [c.detach().float().contiguous() for c in costs]
    dev = xs[0].device
    if dev.type != "cuda":
        raise _cabi.WcaError("dtw: CUDA tensor required (no CPU fallback exists)")
    base = xs[0].data_ptr()
    recs = np.zeros(B, dtype=_cabi.UTT_DTYPE)
    path_off = 0
    for b, x in enumerate(xs):
        n, m = int(x.shape[0]), int(x.shape[1])
        r = recs[b]
        r["n_tokens"], r["n_frames"], r["row_begin"], r["row_end"] = n, m, 0, n
        r["matrix_off"] = (x.data_ptr() - base) // 4
        r["path_off"] = path_off
        r["jump_off"] = 0
        path_off += n + m
    d_utts = _cabi.upload_utts(recs, dev)
    max_rows = int(recs["row_end"].max())
    max_frames = int(recs["n_frames"].max())
    p_text = torch.empty(max(path_off, 1), dtype=torch.int32, device=dev)
    p_time = torch.empty(max(path_off, 1), dtype=torch.int32, device=dev)
    p_len = torch.zeros(B, dtype=torch.int32, device=dev)
    trace_bytes = _cabi.dtw_workspace_bytes(B, max_rows, max_frames)
    trace_ws = torch.empty(trace_bytes, dtype=torch.uint8, device=dev) if trace_bytes else None
    _cabi.dtw_align(base, d_utts, B, max_rows, max_frames, False, path_text=p_text, path_time=p_time, path_len=p_len,
                    trace_ws=trace_ws)
    pt, pj, pl = p_text.cpu().numpy(), p_time.cpu().numpy(), p_len.cpu().numpy()
    out = []
    for b in range(B):
        end = int(recs[b]["path_off"]) + int(recs[b]["row_end"]) + int(recs[b]["n_frames"])
        out.append((pt[end - pl[b]: end].astype(np.int64), pj[end - pl[b]: end].astype(np.int64)))
    return out


def dtw(x: torch.Tensor):
    """(text_indices, time_indices) of the min-cost monotone path through cost matrix x (N, M)."""
    return dtw_batch([x])[0]
