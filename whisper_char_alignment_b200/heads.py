"""Alignment-head masks: ranking heads by their measured word-boundary accuracy, and upstream Whisper's text format
for a mask (the `bytes` that whisper.model.Whisper.set_alignment_heads takes, the `_ALIGNMENT_HEADS` values of
whisper/__init__.py): base85 of the gzip-compressed (n_text_layer, n_text_head) bool array."""
from __future__ import annotations

import base64
import gzip

import numpy as np

from .metrics import get_seg_metrics


def head_f1(counts_LH3) -> np.ndarray:
    """(L, H) float64 dataset F1 of every head: get_seg_metrics(hits, hits, n_pred, n_ref) on the summed counts."""
    c = np.asarray(counts_LH3, dtype=np.int64)
    return np.asarray(get_seg_metrics(c[..., 0], c[..., 0], c[..., 1], c[..., 2])[2], dtype=np.float64)


def rank_heads(counts_LH3, n_heads: int) -> np.ndarray:
    """(L, H) bool mask of the n_heads heads of best dataset F1 (head_f1); ties go to the lower flat index l*H + h.
    counts_LH3: int (L, H, 3) of (hits, n_pred, n_ref), as timing.head_boundary_counts_batch returns them summed over
    utterances.  n_heads is clipped to L*H."""
    f1 = head_f1(counts_LH3)
    if int(n_heads) < 1:
        raise ValueError(f"n_heads={n_heads}: at least one alignment head is needed")
    flat = f1.reshape(-1)
    order = np.lexsort((np.arange(flat.size), -flat))  # F1 descending, then flat index ascending
    mask = np.zeros(flat.size, dtype=bool)
    mask[order[: int(n_heads)]] = True
    return mask.reshape(f1.shape)


def encode_alignment_heads(mask) -> bytes:
    """base64.b85encode(gzip.compress(mask.tobytes())) of an (L, H) bool mask, upstream's format.  The gzip header's
    time stamp is zeroed so that a mask always encodes to the same bytes."""
    return base64.b85encode(gzip.compress(np.ascontiguousarray(mask, dtype=bool).tobytes(), mtime=0))


def decode_alignment_heads(dump, n_layers: int, n_heads: int) -> np.ndarray:
    """(n_layers, n_heads) bool mask of an upstream dump (bytes or str), as Whisper.set_alignment_heads reads it."""
    if isinstance(dump, str):
        dump = dump.encode("ascii")
    array = np.frombuffer(gzip.decompress(base64.b85decode(dump)), dtype=bool)
    if array.size != n_layers * n_heads:
        raise ValueError(f"alignment-head mask of {array.size} entries for a model of {n_layers} x {n_heads} heads")
    return array.reshape(n_layers, n_heads).copy()
