"""CPU suite: the float64 reference of tests/test_gpu_default_timing.py (std-normalisation over tokens + mean over the
alignment heads) against the fp32 CPU restatement of the reference's default_find_alignment (oracle/ref_path.py,
timing.py:156-163) on the reference fixtures, so that the GPU tests rest on a reference that is itself checked."""
import numpy as np
import pytest
import torch

from conftest import default_timing_names, load_golden
from test_gpu_default_timing import EPS, ref_normalize

# torch's fp32 std_mean against float64, in units of eps * (max_t |a| / sd + |w|): what the fp32 port can be held to
PORT_K = 64


@pytest.mark.parametrize("name", default_timing_names())
def test_fp64_normalisation_matches_the_cpu_port(name, oracle_models, tokenizer):
    from oracle import ref_path

    g = load_golden(name)
    c = g["case"]
    model = oracle_models(c["model"])
    text = g["text_tokens"].tolist()
    mel = torch.from_numpy(g["mel"])
    _, _, _, weights, _ = ref_path.default_find_alignment(model, tokenizer, text, mel, c["frames"],
                                                          medfilt_width=c["width"], qk_scale=c["qk_scale"])
    tokens = torch.tensor([*tokenizer.sot_sequence, tokenizer.no_timestamps, *text, tokenizer.eot])
    qk, _ = ref_path.capture_logits(model, mel, tokens)
    maps = ref_path.filtered_softmax(qk, c["frames"], c["width"], c["qk_scale"])  # (L, H, T, F), timing.py:157-159
    heads = model.alignment_heads.indices().T
    sel = (heads[:, 0] * model.dims.n_text_head + heads[:, 1]).numpy()
    sot, T = len(tokenizer.sot_sequence), len(tokens)
    w64, m64, scale = ref_normalize(maps.flatten(0, 1), sel, sot, T - 1)
    w64, m64, scale = w64.numpy(), m64.numpy(), np.broadcast_to(scale.numpy(), w64.shape)
    port = weights.double().numpy()
    assert port.shape == w64.shape
    np.testing.assert_array_equal(np.isnan(port), np.isnan(w64))
    ok = ~np.isnan(w64)
    assert (np.abs(port - w64)[ok] <= PORT_K * EPS * (scale + np.abs(w64))[ok]).all()
    np.testing.assert_allclose(w64, g["weights"], rtol=2e-4, atol=2e-5)  # the fixture the reference's own code wrote
    # the matrix the reference aligns (timing.py:163-165): mean over heads, rows sot_len .. T-2
    np.testing.assert_allclose(m64, weights.mean(0)[sot:-1].double().numpy(), rtol=0, atol=PORT_K * EPS * float(scale[ok].max()))
