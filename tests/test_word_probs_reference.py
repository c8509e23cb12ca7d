"""CPU suite: the float64 restatement of upstream find_alignment's word probabilities (ref_word_probabilities below),
which tests/test_gpu_word_probs.py compares the wca_token_probs path against -- checked on a hand-computed case and on
the logits of the reference fixtures' own forward -- and the host side of the product's entry points."""
import math

import numpy as np
import pytest
import torch

from conftest import default_timing_names, golden_names, load_golden
from oracle import ref_path


def ref_word_probabilities(logits, text_tokens, tokenizer, aligned_unit_type="subword"):
    """Upstream whisper.timing.find_alignment's word confidence, in float64 on the CPU:
        sampled_logits = logits[len(tokenizer.sot_sequence):, : tokenizer.eot]
        token_probs = sampled_logits.softmax(dim=-1)
        text_token_probs = token_probs[np.arange(len(text_tokens)), text_tokens].tolist()
        word_probabilities = [np.mean(text_token_probs[i:j]) for i, j in zip(word_boundaries[:-1], word_boundaries[1:])]
    logits: (T, V) of the teacher-forced tokens [*sot_sequence, no_timestamps, *text_tokens, eot].  Words are grouped
    as force_align groups them (the oracle's restatement of retokenize.py:19-39, for either unit; upstream uses the
    "subword" grouping).  Returns (text_token_probs float64 (n_text,), word_probabilities float64 (W,))."""
    sampled_logits = logits.detach().cpu().double()[len(tokenizer.sot_sequence):, : tokenizer.eot]
    token_probs = sampled_logits.softmax(dim=-1)
    text_tokens = list(text_tokens)
    text_token_probs = token_probs[np.arange(len(text_tokens)), np.asarray(text_tokens, dtype=np.int64)].tolist()
    _, word_tokens = ref_path.split_tokens_on_spaces(text_tokens + [tokenizer.eot], tokenizer, aligned_unit_type)
    word_boundaries = np.pad(np.cumsum([len(t) for t in word_tokens[:-1]]), (1, 0))
    word_probs = [np.mean(text_token_probs[i:j]) for i, j in zip(word_boundaries[:-1], word_boundaries[1:])]
    return np.array(text_token_probs, dtype=np.float64), np.array(word_probs, dtype=np.float64)


@pytest.mark.parametrize("unit", ["char", "subword"])
def test_hand_computed_case(unit, tokenizer):
    """Row sot + i holds 0 everywhere but log(k_i) at its text token: p_i = k_i / (k_i + eot - 1) exactly.  The columns
    at and past eot (timestamps, specials) hold huge values and +inf: they are not part of the text vocabulary."""
    from whisper_char_alignment_b200.retokenize import encode, split_tokens_on_spaces

    text = encode("ab cde f", tokenizer, unit)
    sot, eot = len(tokenizer.sot_sequence), tokenizer.eot
    V = eot + 7
    logits = torch.zeros(sot + 1 + len(text) + 1, V)
    logits[:, eot:] = 1e4
    logits[:, -1] = float("inf")
    ks = [1.0 + 3 * i for i in range(len(text))]
    for i, (t, k) in enumerate(zip(text, ks)):
        logits[sot + i, t] = math.log(k)
    tp, wp = ref_word_probabilities(logits, text, tokenizer, unit)
    want_tp = [k / (k + eot - 1) for k in ks]
    np.testing.assert_allclose(tp, want_tp, rtol=1e-6)  # log(k) was rounded to fp32
    _, word_tokens = split_tokens_on_spaces(text + [eot], tokenizer, unit)
    want_wp, i = [], 0
    for toks in word_tokens[:-1]:
        want_wp.append(sum(want_tp[i:i + len(toks)]) / len(toks))
        i += len(toks)
    assert len(wp) == len(word_tokens) - 1 == 3  # "ab", " cde", " f" in either unit
    np.testing.assert_allclose(wp, want_wp, rtol=1e-6)
    # an EOT-only utterance has no word
    tp0, wp0 = ref_word_probabilities(logits[: sot + 2], [], tokenizer, unit)
    assert tp0.shape == (0,) and wp0.shape == (0,)


@pytest.mark.parametrize("name", golden_names() + default_timing_names())
def test_restatement_on_the_fixtures_logits(name, oracle_models, tokenizer):
    """The oracle's CPU forward reproduces the fixture's logits (its stored digest where it has one, as test_oracle_golden
    checks); on
    those logits the float64 restatement agrees with upstream's own fp32 lines (softmax over [:eot], gather, np.mean)
    within fp32 rounding, and yields one probability per word force_align returns, EOT aside."""
    g = load_golden(name)
    c = g["case"]
    model = oracle_models(c["model"], c.get("seed", 0), c.get("gain", 4.0))
    text = g["text_tokens"].tolist()
    tokens = torch.tensor([*tokenizer.sot_sequence, tokenizer.no_timestamps, *text, tokenizer.eot])
    _, logits = ref_path.capture_logits(model, torch.from_numpy(g["mel"]), tokens)
    if "logits_digest" in g:  # the default_find_alignment fixtures store none
        np.testing.assert_allclose(logits.double().sum().item(), g["logits_digest"][0], rtol=1e-5)
    unit = c.get("unit", "subword")
    tp, wp = ref_word_probabilities(logits, text, tokenizer, unit)

    # upstream, verbatim, in fp32
    sampled_logits = logits[len(tokenizer.sot_sequence):, : tokenizer.eot]
    token_probs = sampled_logits.softmax(dim=-1)
    text_token_probs = token_probs[np.arange(len(text)), text].tolist() if text else []
    assert len(tp) == len(text)
    np.testing.assert_allclose(tp, text_token_probs, rtol=1e-4, atol=1e-30)
    if g["sentinel"]:
        assert len(wp) == 0
        return
    assert len(wp) == len(g["words"]) - 1
    _, word_tokens = ref_path.split_tokens_on_spaces(text + [tokenizer.eot], tokenizer, unit)
    wb = np.pad(np.cumsum([len(t) for t in word_tokens[:-1]]), (1, 0))
    upstream = [np.mean(text_token_probs[i:j]) for i, j in zip(wb[:-1], wb[1:])]
    np.testing.assert_allclose(wp, upstream, rtol=1e-4, atol=1e-30)
    assert ((wp > 0) & (wp < 1)).all()


def test_word_probabilities_refuses_cpu_logits(tokenizer):
    """The product computes the probabilities on wca_token_probs only: CPU logits raise WcaError."""
    from whisper_char_alignment_b200 import _cabi, timing

    sot = len(tokenizer.sot_sequence)
    with pytest.raises(_cabi.WcaError):
        timing.word_probabilities_batch([torch.zeros(sot + 3, tokenizer.eot + 1)], [[11, 12]], tokenizer)


def test_word_probabilities_flag_is_off_by_default():
    """Without --word_probabilities the parsed flags, and so the results JSON that records them, are unchanged."""
    from whisper_char_alignment_b200.cli import infer_ali

    assert "word_probabilities" not in vars(infer_ali.parse_args(["--output_dir", "x"]))
    assert infer_ali.parse_args(["--output_dir", "x", "--word_probabilities"]).word_probabilities is True
