"""CPU suite: the float64 references of tests/test_gpu_scoring.py and tests/test_gpu_capture.py against the fp32 CPU
restatement of the reference (oracle/ref_path.py), so that the GPU tests rest on references that are themselves checked."""
import numpy as np
import pytest
import torch

from test_gpu_capture import ref_capture, ref_logits
from test_gpu_scoring import NAN, ref_aggregate, ref_head_terms, ref_scores, ref_topk

RTOL = 1e-5


def _maps(seed, L, H, T, F):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(L, H, T, F, generator=g) * 3).softmax(-1)


@pytest.mark.parametrize("w", [(1.0, 1.0, 0.0), (1.0, 1.0, 0.7), (0.0, 0.0, 1.0), (1.0, 0.0, 0.0), (0.0, 1.0, 0.0),
                               (-1.0, 1.0, 0.5), (NAN, 1.0, 0.5), (2.0, NAN, 0.0), (0.5, 1.0, NAN)], ids=str)
def test_fp64_scores_match_the_cpu_port(w):
    from oracle import ref_path

    for seed, (L, H, T, F) in enumerate([(2, 3, 9, 300), (1, 4, 1, 1), (2, 2, 40, 31), (1, 2, 17, 600)]):
        maps = _maps(seed, L, H, T, F)
        maps[..., :2, :] *= 3  # column sums on both sides of the coverage threshold 0.5
        want = ref_path.head_scores(maps, *w).double().numpy()
        got, scale = (t.numpy().reshape(L, H) for t in ref_scores(ref_head_terms(maps.view(L * H, T, F)), F, *w))
        assert (np.abs(got - want) <= RTOL * scale).all(), (w, (L, H, T, F), got, want)


@pytest.mark.parametrize("aggregation", ["mean", "topk"])
def test_fp64_aggregate_matches_the_cpu_port(aggregation):
    from oracle import ref_path

    L, H, T, F = 4, 3, 12, 70
    maps = _maps(7, L, H, T, F)
    matrix, kept = ref_path.aggregate(maps, aggregation, 5)
    sel = list(range(L // 2 * H, L * H)) if aggregation == "mean" else [l * H + h for _, (l, h), _ in kept]
    got = ref_aggregate(maps.view(L * H, T, F), sel, 0, T).numpy()
    np.testing.assert_allclose(got, matrix.double().numpy(), rtol=RTOL, atol=0)
    np.testing.assert_allclose(ref_aggregate(maps.view(L * H, T, F), sel, 3, 10).numpy(), got[3:10], rtol=1e-15, atol=0)


def test_topk_reference_matches_the_cpu_port():
    """The order of filter_attention (sorted tuples, timing.py:36) with exactly tied heads, then the NaN rule of the
    kernel, which the reference leaves unspecified."""
    from oracle import ref_path

    maps = _maps(3, 2, 4, 10, 50)
    maps[1, 3] = maps[0, 1]  # two pairs of heads with identical maps: exactly tied scores
    maps[1, 0] = maps[0, 2]
    scores = ref_path.head_scores(maps).view(-1).numpy()
    for k in (1, 2, 5, 8):
        _, kept = ref_path.filter_attention(maps, k)
        np.testing.assert_array_equal(ref_topk(scores, k), [l * 4 + h for _, (l, h), _ in kept])
    rng = np.random.default_rng(0)
    for values in ([0.0, -0.0, 1.0, -1.0], [1e-45, -1e-45, 1e-40, 0.0, -0.0, np.inf, -np.inf], [0.5, 1.5]):
        s = rng.choice(np.array(values, np.float32), 300)
        for k in (1, 7, 300):
            want = [i for _, i in sorted((float(v), i) for i, v in enumerate(s))[-k:]]
            np.testing.assert_array_equal(ref_topk(s, k), want)
    s = np.array([NAN, -np.inf, 2.0, NAN, -np.inf, -0.0, 0.0], np.float32)
    np.testing.assert_array_equal(ref_topk(s, 7), [0, 3, 1, 4, 5, 6, 2])
    np.testing.assert_array_equal(ref_topk(s, 3), [5, 6, 2])
    assert len(ref_topk(s, 0)) == 0 and len(ref_topk(s, 9)) == 7


@pytest.mark.parametrize("width,qk_scale", [(1, 1.0), (3, 1.0), (5, 0.0), (7, 0.5), (7, -1.0), (9, 3.0), (31, -0.0)],
                         ids=str)
def test_fp64_capture_matches_the_cpu_port(width, qk_scale):
    """The capture reference: logits against the hooked cross-attention of the restated model (capture_logits,
    timing.py:48-63, SDPA off), maps against filtered_softmax (trim, median with reflect padding inside the row, identity
    for rows of at most width // 2 frames, scale, softmax) -- on the fp32 logits within fp32 rounding, on the float64
    logits to float64 rounding."""
    from oracle import ref_path
    from whisper.model import MultiHeadAttention, disable_sdpa

    n_heads = 2
    attn = MultiHeadAttention(64 * n_heads, n_heads)
    g = torch.Generator().manual_seed(width)
    for T, F in [(1, 1), (3, width // 2), (5, width // 2 + 1), (9, 40), (4, 300)]:
        if F < 1:
            continue
        q = torch.randn(1, T, 64 * n_heads, generator=g) * 2
        k = torch.randn(1, F + 5, 64 * n_heads, generator=g)
        with disable_sdpa():
            _, qk = attn.qkv_attention(q, k, torch.zeros_like(k))
        np.testing.assert_allclose(ref_logits(q[0], k[0]).numpy(), qk[0].double().numpy(), rtol=1e-5, atol=1e-5)
        want = ref_capture(q[0], k[0, :F], width, qk_scale)
        np.testing.assert_allclose(want.numpy(), ref_path.filtered_softmax(qk[0], F, width, qk_scale).double().numpy(),
                                   rtol=1e-4, atol=1e-7)
        port64 = ref_path.filtered_softmax(ref_logits(q[0], k[0]), F, width, qk_scale)
        np.testing.assert_allclose(want.numpy(), port64.numpy(), rtol=1e-12, atol=0)
