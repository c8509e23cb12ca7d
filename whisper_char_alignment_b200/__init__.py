"""whisper_char_alignment_b200 -- B200-native (sm_100a) implementation of the alignment hot
path of 30stomercury/whisper-char-alignment: `timing.get_attentions` + `timing.force_align`.

Layout
    csrc/            hand-written CUDA kernels + the extern "C" ABI (include/wca_b200.h)
    _cabi.py         ctypes binding (raises if the library is missing: no CPU fallback)
    timing.py        get_attentions / filter_attention / force_align (+ batched variants)
    retokenize.py    encode / split_tokens_on_spaces / remove_punctuation
    metrics.py       eval_n1 / eval_n1_strict / get_seg_metrics / coverage_penalty
    whisper_model.py the Whisper module whose linears stay on cuBLAS
    tokenizer.py     offline stand-in tokenizer
"""
from .timing import (  # noqa: F401
    default_find_alignment, default_find_alignment_batch, dtw, dtw_batch, filter_attention, force_align, force_align_batch, get_attentions, get_attentions_batch,
    median_filter_softmax,
)

__version__ = "0.1.0"
