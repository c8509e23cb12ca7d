"""Host-side checks of the KV-cached greedy decoder (whisper_model.greedy_decode_cached): no device needed."""
import pytest
import torch


def test_greedy_decode_cached_rejects_cpu_features(tokenizer):
    """The cached decoder runs on wca_decode_attention only: CPU features raise WcaError instead of falling back."""
    from whisper_char_alignment_b200 import _cabi
    from whisper_char_alignment_b200.whisper_model import greedy_decode_cached, load_model

    model = load_model("random:micro")
    with pytest.raises(_cabi.WcaError):
        greedy_decode_cached(model, torch.zeros(1, model.dims.n_audio_ctx, model.dims.n_audio_state), tokenizer, 4)
