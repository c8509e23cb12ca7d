"""ctypes binding of libwca_b200.so (C ABI declared in include/wca_b200.h).

There is deliberately NO fallback: if the sm_100a library is missing or a call
fails, the product path raises.  PyTorch only supplies device memory and the
current stream; every signature below is plain pointers and sizes.
"""
from __future__ import annotations

import ctypes
import os
from typing import Sequence

import numpy as np
import torch

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libwca_b200.so")

WCA_CAPTURE_RAW_LOGITS = 1
WCA_CAPTURE_FORCE_SIMT = 2
WCA_CAPTURE_TRACE = 4
WCA_MAX_LAYERS = 32
ABI_VERSION = 5

EXPORTS = (
    "wca_abi_version", "wca_last_error", "wca_launch_count", "wca_device_info", "wca_capture_attention", "wca_full_attention", "wca_causal_attention", "wca_decode_attention_workspace_bytes", "wca_decode_attention",
    "wca_add_layernorm", "wca_debug_enc_attn_buffer", "wca_debug_capture_trace", "wca_medfilt_softmax",
    "wca_head_scores", "wca_head_scores_from_partials", "wca_capture_writes_partials", "wca_capture_partials_floats", "wca_topk_heads", "wca_aggregate_heads", "wca_normalize_heads", "wca_token_probs", "wca_dtw_workspace_bytes", "wca_dtw_align",
)


class WcaError(RuntimeError):
    """A libwca_b200 entry point returned a non-zero status."""


class UttDesc(ctypes.Structure):
    """Mirror of `wca_utt_t` (include/wca_b200.h)."""

    _fields_ = [
        ("n_tokens", ctypes.c_int32), ("n_frames", ctypes.c_int32), ("row_begin", ctypes.c_int32),
        ("row_end", ctypes.c_int32), ("n_words", ctypes.c_int32), ("n_sel", ctypes.c_int32),
        ("q_row0", ctypes.c_int64), ("k_row0", ctypes.c_int64), ("ws_off", ctypes.c_int64),
        ("score_off", ctypes.c_int64), ("sel_off", ctypes.c_int64), ("matrix_off", ctypes.c_int64),
        ("path_off", ctypes.c_int64), ("jump_off", ctypes.c_int64), ("word_off", ctypes.c_int64),
        ("part_off", ctypes.c_int64),
    ]


UTT_DTYPE = np.dtype(
    [(name, np.int32 if ct is ctypes.c_int32 else np.int64) for name, ct in UttDesc._fields_], align=True
)
assert UTT_DTYPE.itemsize == ctypes.sizeof(UttDesc) == 104

_lib = None


def load() -> ctypes.CDLL:
    """Load the library once; raise loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the sm_100a extension has not been built "
            "(run `python -m whisper_char_alignment_b200.build`). There is no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise ImportError(f"{LIB_PATH} does not export {name}")
    vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float
    lib.wca_abi_version.restype = i32
    lib.wca_last_error.restype = ctypes.c_char_p
    lib.wca_launch_count.restype = ctypes.c_uint64
    lib.wca_device_info.argtypes = [ctypes.POINTER(i32), ctypes.POINTER(i32)]
    lib.wca_capture_attention.argtypes = [vp, vp, i32, i32, i32, i64, i64, i64, i64, vp, i32, i32, i32, i32, f32, vp, vp,
                                          ctypes.c_uint, vp]
    lib.wca_capture_writes_partials.argtypes = [i32, i32, ctypes.c_uint]
    lib.wca_capture_partials_floats.restype = i64
    lib.wca_capture_partials_floats.argtypes = [i32, i32, i32]
    lib.wca_head_scores_from_partials.argtypes = [vp, vp, i32, i32, f32, f32, vp, vp]
    lib.wca_full_attention.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, i64, i64, i64, i64, vp]
    lib.wca_causal_attention.argtypes = lib.wca_full_attention.argtypes
    lib.wca_decode_attention_workspace_bytes.restype = i64
    lib.wca_decode_attention_workspace_bytes.argtypes = [i32, i32, i32]
    lib.wca_decode_attention.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i64, i64, i64, i64, i64, i64, vp, i64, vp]
    lib.wca_add_layernorm.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, f32, vp]
    lib.wca_medfilt_softmax.argtypes = [vp, i64, i64, i32, i32, f32, vp, vp]
    lib.wca_head_scores.argtypes = [vp, vp, i32, i32, i32, i32, f32, f32, f32, vp, vp]
    lib.wca_topk_heads.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    lib.wca_aggregate_heads.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, vp]
    lib.wca_normalize_heads.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, vp, vp]
    lib.wca_token_probs.argtypes = [vp, vp, i32, i32, vp, vp]
    lib.wca_dtw_workspace_bytes.restype = i64
    lib.wca_dtw_workspace_bytes.argtypes = [i32, i32, i32]
    lib.wca_dtw_align.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]
    if lib.wca_abi_version() != ABI_VERSION:
        raise ImportError(f"{LIB_PATH}: ABI version {lib.wca_abi_version()} != {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


_timer = None


def launch_count() -> int:
    """Kernels launched so far by this thread through the library."""
    return int(load().wca_launch_count())


class KernelTimer:
    """Brackets every library call with CUDA events on the launching stream while active:

        with _cabi.KernelTimer() as kt: ...work...
        kt.summary() -> {entry point: (calls, total_ms)}

    Used by bench.py for the roofline figures; inactive (zero overhead) otherwise."""

    def __init__(self):
        self.records = []

    def __enter__(self):
        global _timer
        self._prev, _timer = _timer, self
        return self

    def __exit__(self, *exc):
        global _timer
        _timer = self._prev
        return False

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, a, b in self.records:
            calls, ms = out.get(name, (0, 0.0))
            out[name] = (calls + 1, ms + a.elapsed_time(b))
        return out


def _check(rc: int, what: str):
    if rc != 0:
        msg = load().wca_last_error().decode("utf-8", "replace")
        raise WcaError(f"{what} failed with status {rc}: {msg}")


class _timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if _timer is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if _timer is not None and exc[0] is None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            _timer.records.append((self.name, self.a, b))
        return False


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dev_ptr(t: torch.Tensor | None, dtype=None, name="tensor") -> int | None:
    if t is None:
        return None
    if not t.is_cuda:
        raise WcaError(f"{name} must live on a CUDA device (no CPU fallback exists)")
    if dtype is not None and t.dtype != dtype:
        raise WcaError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise WcaError(f"{name} must be contiguous")
    return t.data_ptr()


def capture_trace():
    """(tiles, events) int64 clock64 stamps of the last WCA_CAPTURE_TRACE launch (debug)."""
    buf = (ctypes.c_longlong * 4096)()
    n = load().wca_debug_capture_trace(buf, 4096)
    if n < 0:
        _check(n, "wca_debug_capture_trace")
    return np.frombuffer(buf, dtype=np.int64, count=n).copy()


def device_info():
    sm, cc = ctypes.c_int(0), ctypes.c_int(0)
    _check(load().wca_device_info(ctypes.byref(sm), ctypes.byref(cc)), "wca_device_info")
    return sm.value, cc.value


def upload_utts(records: np.ndarray, device) -> torch.Tensor:
    """records: structured array of UTT_DTYPE -> uint8 device tensor (one async H2D copy)."""
    assert records.dtype == UTT_DTYPE
    host = torch.from_numpy(records.view(np.uint8).reshape(-1).copy())
    if torch.cuda.is_available():
        host = host.pin_memory()
    return host.to(device, non_blocking=True)


# ---------------------------------------------------------------------------------
# thin wrappers: tensors in, status checked, nothing else
# ---------------------------------------------------------------------------------
def _rows_and_pitch(t: torch.Tensor, name: str):
    """(rows, floats between rows) of an fp32 (..., rows, width) tensor whose rows are evenly strided -- a contiguous
    tensor or a column slice of a wider one (e.g. one layer's K inside the all-layer K/V projection)."""
    if not t.is_cuda:
        raise WcaError(f"{name} must live on a CUDA device (no CPU fallback exists)")
    if t.dtype != torch.float32 or t.dim() < 2 or t.stride(-1) != 1:
        raise WcaError(f"{name} must be fp32 with unit stride along the width")
    pitch = t.stride(-2)
    rows = t.shape[-2]
    for dim in range(t.dim() - 3, -1, -1):  # leading dims must continue the same row pitch
        if t.shape[dim] != 1 and t.stride(dim) != rows * pitch:
            raise WcaError(f"{name}: rows are not evenly strided")
        rows *= t.shape[dim]
    return rows, pitch


def capture_attention(q_layers: Sequence[torch.Tensor], k_layers: Sequence[torch.Tensor], n_heads: int,
                      ld_q: int | None, ld_k: int | None, d_utts: torch.Tensor, n_utts: int, max_tokens: int, max_frames: int,
                      medfilt_width: int, qk_scale: float, ws: torch.Tensor, flags: int = 0, partials: torch.Tensor | None = None):
    """q_layers / k_layers: per decoder layer, (..., rows, n_heads*64) fp32 with evenly strided rows (ld_q / ld_k are
    taken from the tensors when None)."""
    n_layers = len(q_layers)
    if n_layers != len(k_layers) or not 1 <= n_layers <= WCA_MAX_LAYERS:
        raise WcaError(f"bad layer count {n_layers}")
    head_dim = 64
    q_rows, q_pitch = _rows_and_pitch(q_layers[0], "Q")
    k_rows, k_pitch = _rows_and_pitch(k_layers[0], "K")
    ld_q = q_pitch if ld_q is None else ld_q
    ld_k = k_pitch if ld_k is None else ld_k
    for q, k in zip(q_layers, k_layers):
        if _rows_and_pitch(q, "Q") != (q_rows, q_pitch) or _rows_and_pitch(k, "K") != (k_rows, k_pitch):
            raise WcaError("every layer's Q (and K) must have the same shape and row pitch")
    if q_pitch != ld_q or k_pitch != ld_k:
        raise WcaError("ld_q / ld_k disagree with the tensors' row pitch")
    qp = (ctypes.c_void_p * n_layers)(*[t.data_ptr() for t in q_layers])
    kp = (ctypes.c_void_p * n_layers)(*[t.data_ptr() for t in k_layers])
    with _timed("wca_capture_attention"):
        _check(
            load().wca_capture_attention(qp, kp, n_layers, n_heads, head_dim, ld_q, ld_k, q_rows, k_rows,
                                         _dev_ptr(d_utts), n_utts,
                                         max_tokens, max_frames, medfilt_width, float(qk_scale),
                                         _dev_ptr(ws, torch.float32, "ws"), _dev_ptr(partials, torch.float32, "partials"),
                                         flags, _stream()),
            "wca_capture_attention",
        )


def capture_writes_partials(max_frames: int, medfilt_width: int, flags: int = 0) -> bool:
    return bool(load().wca_capture_writes_partials(int(max_frames), int(medfilt_width), int(flags)))


def capture_partials_floats(n_heads: int, n_tokens: int, n_frames: int) -> int:
    return int(load().wca_capture_partials_floats(int(n_heads), int(n_tokens), int(n_frames)))


def head_scores_from_partials(partials: torch.Tensor, d_utts, n_utts, n_heads, w_col, w_row, scores):
    with _timed("wca_head_scores_from_partials"):
        _check(
            load().wca_head_scores_from_partials(_dev_ptr(partials, torch.float32, "partials"), _dev_ptr(d_utts), n_utts,
                                                 n_heads, float(w_col), float(w_row),
                                                 _dev_ptr(scores, torch.float32, "scores"), _stream()),
            "wca_head_scores_from_partials",
        )


def full_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, n_heads: int, out: torch.Tensor | None = None,
                   causal: bool = False):
    """q: (batch, n_q, n_heads*64), k, v: (batch, n_kv, n_heads*64), fp32, last dim contiguous, rows evenly
    strided.  Returns softmax(q k^T / 8) v as (batch, n_q, n_heads*64) (wca_full_attention); causal=True masks the
    keys j > i of query i (wca_causal_attention: the decoder's self-attention)."""
    batch, n_q, width = q.shape
    n_kv = k.shape[1]
    for t, name, rows in ((q, "q", n_q), (k, "k", n_kv), (v, "v", n_kv)):
        if not t.is_cuda or t.dtype != torch.float32:
            raise WcaError(f"full_attention: {name} must be an fp32 CUDA tensor (no CPU fallback exists)")
        if tuple(t.shape) != (batch, rows, width) or t.stride(2) != 1 or t.stride(0) != rows * t.stride(1):
            raise WcaError(f"full_attention: {name} must be (batch, rows, width) with contiguous rows")
    if out is None:
        out = torch.empty(batch, n_q, width, dtype=torch.float32, device=q.device)
    name = "wca_causal_attention" if causal else "wca_full_attention"
    with _timed(name):
        _check(
            getattr(load(), name)(q.data_ptr(), k.data_ptr(), v.data_ptr(), _dev_ptr(out, torch.float32, "out"), batch, n_q,
                                  n_kv, n_heads, width // n_heads, q.stride(1), k.stride(1), v.stride(1), out.stride(1),
                                  _stream()),
            name,
        )
    return out


def decode_attention_workspace_bytes(n_batch: int, n_heads: int, n_kv: int) -> int:
    return int(load().wca_decode_attention_workspace_bytes(int(n_batch), int(n_heads), int(n_kv)))


def decode_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, n_heads: int, out: torch.Tensor | None = None,
                     workspace: torch.Tensor | None = None):
    """q: (batch, n_heads*64), k, v: (batch, n_kv, n_heads*64), fp32 CUDA, last dim contiguous; any row and batch
    strides (a column slice of a wider projection, the live rows of a preallocated cache).  Returns
    softmax(q k^T / 8) v per (batch item, head) as (batch, n_heads*64) (wca_decode_attention: one query row per item,
    every key visible).  workspace: a uint8 CUDA tensor of at least decode_attention_workspace_bytes, allocated when
    None."""
    batch, width = q.shape
    n_kv = k.shape[1]
    if n_heads < 1 or width % n_heads:
        raise WcaError(f"decode_attention: width {width} is not a multiple of n_heads={n_heads}")
    for t, name in ((q, "q"), (k, "k"), (v, "v")):
        if not t.is_cuda or t.dtype != torch.float32:
            raise WcaError(f"decode_attention: {name} must be an fp32 CUDA tensor (no CPU fallback exists)")
        if t.stride(-1) != 1:
            raise WcaError(f"decode_attention: {name} must have unit stride along the width")
    for t, name in ((k, "k"), (v, "v")):
        if tuple(t.shape) != (batch, n_kv, width):
            raise WcaError(f"decode_attention: {name} must be (batch, n_kv, width) = {(batch, n_kv, width)}, got {tuple(t.shape)}")
    if out is None:
        out = torch.empty(batch, width, dtype=torch.float32, device=q.device)
    if tuple(out.shape) != (batch, width) or out.dtype != torch.float32 or not out.is_cuda or out.stride(-1) != 1:
        raise WcaError("decode_attention: out must be an fp32 CUDA (batch, width) tensor with unit stride along the width")
    need = decode_attention_workspace_bytes(batch, n_heads, n_kv)
    if workspace is None:
        workspace = torch.empty(need, dtype=torch.uint8, device=q.device)
    if not workspace.is_cuda or not workspace.is_contiguous():
        raise WcaError("decode_attention: workspace must be a contiguous CUDA tensor")
    with _timed("wca_decode_attention"):
        _check(
            load().wca_decode_attention(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), batch, n_kv, n_heads,
                                        width // n_heads, q.stride(0), k.stride(1), v.stride(1), out.stride(0), k.stride(0),
                                        v.stride(0), workspace.data_ptr(), workspace.numel() * workspace.element_size(),
                                        _stream()),
            "wca_decode_attention",
        )
    return out


def add_layernorm(x: torch.Tensor, h: torch.Tensor | None, gamma: torch.Tensor, beta: torch.Tensor, eps: float):
    """(x + h, LayerNorm(x + h) * gamma + beta) over the last dimension in one pass (wca_add_layernorm);
    h may be None (plain LayerNorm, returns (x, n))."""
    width = x.shape[-1]
    for t, name in ((x, "x"), (h, "h"), (gamma, "gamma"), (beta, "beta")):
        if t is None:
            continue
        if not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            raise WcaError(f"add_layernorm: {name} must be a contiguous fp32 CUDA tensor (no CPU fallback exists)")
    if h is not None and h.shape != x.shape:
        raise WcaError("add_layernorm: x and h must have the same shape")
    y = torch.empty_like(x) if h is not None else x
    n = torch.empty_like(x)
    with _timed("wca_add_layernorm"):
        _check(
            load().wca_add_layernorm(x.data_ptr(), None if h is None else h.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                     None if h is None else y.data_ptr(), n.data_ptr(), x.numel() // width, width,
                                     float(eps), _stream()),
            "wca_add_layernorm",
        )
    return y, n


def encoder_attention(q, k, v, n_heads, out=None):
    """Self-attention special case (n_q == n_kv) of full_attention."""
    return full_attention(q, k, v, n_heads, out)


def medfilt_softmax(x: torch.Tensor, n_rows: int, ld_in: int, n_frames: int, medfilt_width: int, qk_scale: float,
                    out: torch.Tensor):
    with _timed("wca_medfilt_softmax"):
        _check(
            load().wca_medfilt_softmax(_dev_ptr(x, torch.float32, "logits"), n_rows, ld_in, n_frames, medfilt_width,
                                       float(qk_scale), _dev_ptr(out, torch.float32, "out"), _stream()),
            "wca_medfilt_softmax",
        )


def head_scores(ws_base: int, d_utts, n_utts, n_heads, max_tokens, max_frames, w_col, w_row, w_cov, scores):
    with _timed("wca_head_scores"):
        _check(
            load().wca_head_scores(ws_base, _dev_ptr(d_utts), n_utts, n_heads, max_tokens, max_frames, float(w_col),
                                   float(w_row), float(w_cov), _dev_ptr(scores, torch.float32, "scores"), _stream()),
            "wca_head_scores",
        )


def topk_heads(scores, d_utts, n_utts, n_heads, sel, sel_scores):
    with _timed("wca_topk_heads"):
        _check(
            load().wca_topk_heads(_dev_ptr(scores, torch.float32, "scores"), _dev_ptr(d_utts), n_utts, n_heads,
                                  _dev_ptr(sel, torch.int32, "sel"), _dev_ptr(sel_scores, torch.float32, "sel_scores"),
                                  _stream()),
            "wca_topk_heads",
        )


def aggregate_heads(ws_base: int, sel, d_utts, n_utts, max_tokens, max_frames, matrix, max_sel: int = 2):
    """max_sel: an upper bound of the descriptors' n_sel (1 selects the single-head kernel of the probe sweep)."""
    with _timed("wca_aggregate_heads"):
        _check(
            load().wca_aggregate_heads(ws_base, _dev_ptr(sel, torch.int32, "sel"), _dev_ptr(d_utts), n_utts, max_tokens,
                                       max_frames, max(int(max_sel), 1), _dev_ptr(matrix, torch.float32, "matrix"), _stream()),
            "wca_aggregate_heads",
        )


def normalize_heads(ws_base: int, sel, d_utts, n_utts, max_tokens, max_frames, matrix, weights=None, weights_off=None):
    """Std-normalised head maps (`weights` + `weights_off`, both or neither) and their mean (`matrix`)."""
    if (weights is None) != (weights_off is None):
        raise WcaError("normalize_heads: give weights and weights_off together or neither")
    with _timed("wca_normalize_heads"):
        _check(
            load().wca_normalize_heads(ws_base, _dev_ptr(sel, torch.int32, "sel"), _dev_ptr(d_utts), n_utts, max_tokens,
                                       max_frames, _dev_ptr(weights, torch.float32, "weights"),
                                       _dev_ptr(weights_off, torch.int64, "weights_off"),
                                       _dev_ptr(matrix, torch.float32, "matrix"), _stream()),
            "wca_normalize_heads",
        )


def token_probs(row_addrs: np.ndarray, targets: np.ndarray, n_cols: int, probs: torch.Tensor):
    """probs[r] = softmax(logits at row_addrs[r], columns [0, n_cols))[targets[r]] (wca_token_probs).  row_addrs: host
    int64 device addresses of fp32 rows (any 4-byte alignment, any pitch); targets: host ints.  The targets are checked
    here, on the host, before anything is launched (the library cannot read them without synchronising); both arrays go
    to the device in one copy."""
    row_addrs = np.ascontiguousarray(row_addrs, dtype=np.int64).reshape(-1)
    targets = np.asarray(targets).reshape(-1)
    n = len(row_addrs)
    if len(targets) != n:
        raise WcaError(f"wca_token_probs: {n} rows but {len(targets)} targets")
    if n and (targets.min() < 0 or targets.max() >= n_cols):
        bad = int(targets[(targets < 0) | (targets >= n_cols)][0])
        raise WcaError(f"wca_token_probs: target {bad} outside [0, {n_cols})")
    if n and (row_addrs % 4).any():
        raise WcaError("wca_token_probs: row addresses must be 4-byte aligned")
    if not probs.is_cuda or probs.dtype != torch.float32 or not probs.is_contiguous() or probs.numel() < n:
        raise WcaError(f"wca_token_probs: probs must be a contiguous fp32 CUDA tensor of at least {n} elements")
    if n == 0:
        return
    packed = np.empty(12 * n, dtype=np.uint8)  # n int64 addresses, then n int32 targets
    packed[: 8 * n] = row_addrs.view(np.uint8)
    packed[8 * n:] = targets.astype(np.int32).view(np.uint8)
    host = torch.from_numpy(packed)
    dev = host.pin_memory().to(probs.device, non_blocking=True)
    with _timed("wca_token_probs"):
        _check(load().wca_token_probs(dev.data_ptr(), dev.data_ptr() + 8 * n, n, int(n_cols), probs.data_ptr(), _stream()),
               "wca_token_probs")


def dtw_workspace_bytes(n_utts, max_rows, max_frames) -> int:
    return int(load().wca_dtw_workspace_bytes(n_utts, max_rows, max_frames))


def dtw_align(matrix_base: int, d_utts, n_utts, max_rows, max_frames, negate, path_text=None, path_time=None,
              path_len=None, jump_frames=None, word_bounds=None, start_times=None, end_times=None, trace_ws=None):
    ws_bytes = 0 if trace_ws is None else trace_ws.numel() * trace_ws.element_size()
    with _timed("wca_dtw_align"):
        _check(
            load().wca_dtw_align(matrix_base, _dev_ptr(d_utts), n_utts, max_rows, max_frames, int(bool(negate)),
                                 _dev_ptr(path_text, torch.int32, "path_text"),
                                 _dev_ptr(path_time, torch.int32, "path_time"),
                                 _dev_ptr(path_len, torch.int32, "path_len"),
                                 _dev_ptr(jump_frames, torch.int32, "jump_frames"),
                                 _dev_ptr(word_bounds, torch.int32, "word_bounds"),
                                 _dev_ptr(start_times, torch.float64, "start_times"),
                                 _dev_ptr(end_times, torch.float64, "end_times"),
                                 _dev_ptr(trace_ws), ws_bytes, _stream()),
            "wca_dtw_align",
        )
