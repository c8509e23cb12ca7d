"""GPU suite: tuning the alignment settings -- timing.get_attentions_widths_batch against get_attentions_batch width by
width, timing.alignment_config_counts_batch against force_align_batch + metrics.py config by config, and the
tune_alignment CLI against infer_ali run with each config's flags.  Maps and end times are compared bit for bit, counts
and metrics exactly."""
import glob
import json
import os

import numpy as np
import pytest
import torch

from whisper_char_alignment_b200.metrics import eval_n1, eval_n1_strict
from whisper_char_alignment_b200.tuning import Config

pytestmark = pytest.mark.gpu

WIDTHS = (1, 3, 7, 9)  # 1-7 on the tensor-core capture (with head-score partials), 9 on the SIMT capture


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _medium_batch(tokenizer, dev, n=8, seed=8):
    """Whisper-medium dims (random init, qk_gain 4), a TIMIT-shaped batch."""
    from test_gpu_word_probs import _tokens
    from whisper_char_alignment_b200.retokenize import encode
    from whisper_char_alignment_b200.synthetic import timit_shaped
    from whisper_char_alignment_b200.whisper_model import load_model

    model = load_model("random:medium", dev, qk_gain=4.0)
    utts = timit_shaped(n, tokenizer, n_mels=model.dims.n_mels, seed=seed)
    texts = [encode(u.text, tokenizer, "subword") for u in utts]
    return model, texts, torch.stack([u.mel for u in utts]).to(dev), [u.max_frames for u in utts], _tokens(tokenizer, texts, dev)


def _small_batch(size, unit, tokenizer, oracle_models, dev, n=6, seed=13):
    """Ragged text and frame counts on a fixture model, the third utterance EOT-only."""
    from test_gpu_parity import product_model
    from test_gpu_word_probs import _synthetic_batch, _tokens

    model = product_model(oracle_models(size), dev)
    texts, mels, frames = _synthetic_batch(model, tokenizer, unit, n, seed=seed, dev=dev)
    return model, texts, mels, frames, _tokens(tokenizer, texts, dev)


# ------------------------------------------------------------------ several widths from one forward
def _check_widths(model, tokens, mels, frames, tokenizer, dev, label):
    from whisper_char_alignment_b200 import timing
    from whisper_char_alignment_b200.timing import _ScorePartials

    with torch.no_grad():
        features = model.embed_audio(mels)
    for kind, kw in (("mels", dict(mels=mels)), ("features", dict(mels=None, audio_features=features))):
        audio = kw.pop("mels")
        got = timing.get_attentions_widths_batch(audio, tokens, model, tokenizer, frames, list(WIDTHS) + [3], **kw)
        assert list(got) == list(WIDTHS)
        partial_widths = set()
        for w in WIDTHS:
            want_maps, want_logits = timing.get_attentions_batch(audio, tokens, model, tokenizer, frames, w, **kw)
            maps, logits = got[w]
            for b in range(len(tokens)):
                tag = f"{label}/{kind} width {w} utterance {b}"
                assert torch.equal(maps[b], want_maps[b]), tag
                assert torch.equal(logits[b], want_logits[b]), tag
                p, q = _ScorePartials.of(maps[b]), _ScorePartials.of(want_maps[b])
                assert (p is None) == (q is None), tag
                if p is not None:
                    partial_widths.add(w)
                    assert p.offset == q.offset and p.buffer.shape == q.buffer.shape, tag
                # head scores as force_align reads them (from the partials where the capture left them; the partials
                # buffer also holds slots the capture never writes, so it is compared through what is read of it)
                _, t1 = timing.filter_attention(maps[b], topk=0)
                _, t2 = timing.filter_attention(want_maps[b], topk=0)
                assert t1 == t2, tag
        if timing.SCORE_PARTIALS == "1":
            assert partial_widths == {1, 3, 7}, label  # both capture paths were taken


@pytest.mark.parametrize("size", ["micro", "mini"])
def test_widths_from_one_forward_small_models(size, tokenizer, oracle_models, dev):
    model, _, mels, frames, tokens = _small_batch(size, "subword", tokenizer, oracle_models, dev)
    _check_widths(model, tokens, mels, frames, tokenizer, dev, size)


def test_widths_from_one_forward_medium(tokenizer, dev):
    model, _, mels, frames, tokens = _medium_batch(tokenizer, dev)
    _check_widths(model, tokens, mels, frames, tokenizer, dev, "medium")


# ------------------------------------------------------------------ every config against force_align + metrics.py
def _grid(L, H):
    from whisper_char_alignment_b200 import tuning

    return tuning.expand_grid(WIDTHS, ["mean", "topk"], [1, 10, L * H, L * H + 5],
                              [(1.0, 1.0, 0.0), (0.0, 1.0, 0.0), (1.0, 1.0, 0.5)])


def _host_counts(maps_by_width, texts, tokenizer, unit, configs, refs, ref_words, tol):
    """What infer_ali._align_batch counts, config by config: force_align_batch, then eval_n1 / eval_n1_strict."""
    from whisper_char_alignment_b200 import timing

    out = np.zeros((len(texts), len(configs), 3), dtype=np.int64)
    ends = {}
    for i, c in enumerate(configs):
        outs = timing.force_align_batch(maps_by_width[c.medfilt_width], texts, tokenizer, aligned_unit_type=unit,
                                        aggregation=c.aggr, topk=c.topk, w_colnorm=c.w_colnorm, w_rownorm=c.w_rownorm,
                                        w_coverage=c.w_coverage)
        for b, o in enumerate(outs):
            words, _, end_times, _, _ = o
            ends[i, b] = np.asarray(end_times, dtype=np.float64)
            if ref_words is None:
                out[b, i] = (eval_n1(refs[b], end_times, tol)[0], len(end_times), len(refs[b]))
            else:
                tp, fp, fn = eval_n1_strict(refs[b], end_times, ref_words[b], " ".join(words[:-1]).split(), tol)
                out[b, i] = (tp, tp + fp, tp + fn)
    return out, ends


def _references(rng, maps, texts, tokenizer, unit, frames):
    """Reference boundaries and words near one config's alignment (so that the tolerance matters), as in
    test_gpu_boundary_hits."""
    from test_gpu_boundary_hits import _references as jitter
    from whisper_char_alignment_b200 import timing

    refs, ref_words = [], []
    for o, f in zip(timing.force_align_batch(maps, texts, tokenizer, unit, "topk", 3), frames):
        words = ["a", "b"] if isinstance(o, list) else " ".join(o[0][:-1]).split()
        ends = np.array([0.1, 0.3]) if isinstance(o, list) else o[2]
        y, rw = jitter(rng, ends[: len(words)], words, f)
        refs.append(y)
        ref_words.append(rw)
    return refs, ref_words


def _check_counts(model, texts, mels, frames, tokens, tokenizer, unit, label, seed):
    from whisper_char_alignment_b200 import _cabi, timing

    L, H = model.dims.n_text_layer, model.dims.n_text_head
    configs = _grid(L, H)
    by_width = timing.get_attentions_widths_batch(mels, tokens, model, tokenizer, frames, WIDTHS)
    maps_by_width = {w: m for w, (m, _) in by_width.items()}
    refs, ref_words = _references(np.random.default_rng(seed), maps_by_width[7], texts, tokenizer, unit, frames)
    for strict in (False, True):
        rw = ref_words if strict else None
        before = _cabi.launch_count()
        got = timing.alignment_config_counts_batch(maps_by_width, texts, tokenizer, refs, configs,
                                                   aligned_unit_type=unit, tolerance=0.02, ref_words_list=rw)
        # per width: 3 scorings + 3 top-k rankings + 1 aggregation; then DTW and scoring
        assert _cabi.launch_count() - before == len(WIDTHS) * (2 * 3 + 1) + 2, label
        want, _ = _host_counts(maps_by_width, texts, tokenizer, unit, configs, refs, rw, 0.02)
        for b in range(len(texts)):
            assert got[b].dtype == np.int64 and got[b].shape == (len(configs), 3)
            np.testing.assert_array_equal(got[b], want[b], err_msg=f"{label} strict={strict} utterance {b}")
        assert want[..., 0].sum() > 0, label
        if any(len(t) == 0 for t in texts):
            eot = [b for b, t in enumerate(texts) if len(t) == 0]
            for b in eot:
                assert (got[b][:, :2] == 0).all() and (got[b][:, 2] == len(refs[b])).all()

    # bit-identical end times: a config scored against its own end times at tolerance 0 hits every word
    _, ends = _host_counts(maps_by_width, texts, tokenizer, unit, configs, refs, None, 0.0)
    for i in range(0, len(configs), 5):
        own = [ends[i, b] for b in range(len(texts))]
        got = timing.alignment_config_counts_batch(maps_by_width, texts, tokenizer, own, configs,
                                                   aligned_unit_type=unit, tolerance=0.0)
        for b in range(len(texts)):
            n = len(own[b])
            assert tuple(got[b][i]) == (n, n, n), f"{label} config {configs[i]} utterance {b}"

    # an utterance alone gives the counts it gets inside the batch
    got = timing.alignment_config_counts_batch(maps_by_width, texts, tokenizer, refs, configs, aligned_unit_type=unit,
                                               tolerance=0.02)
    for b in range(len(texts)):
        alone = timing.alignment_config_counts_batch({w: [m[b]] for w, m in maps_by_width.items()}, [texts[b]],
                                                     tokenizer, [refs[b]], configs, aligned_unit_type=unit,
                                                     tolerance=0.02)
        np.testing.assert_array_equal(alone[0], got[b], err_msg=f"{label} utterance {b} alone")
    # a sub-grid in another order picks the same rows
    sub = configs[::-3]
    part = timing.alignment_config_counts_batch(maps_by_width, texts, tokenizer, refs, sub, aligned_unit_type=unit,
                                                tolerance=0.02)
    for b in range(len(texts)):
        np.testing.assert_array_equal(part[b], got[b][::-3])


@pytest.mark.parametrize("unit", ["char", "subword"])
@pytest.mark.parametrize("size", ["micro", "mini"])
def test_counts_equal_force_align_small_models(size, unit, tokenizer, oracle_models, dev):
    model, texts, mels, frames, tokens = _small_batch(size, unit, tokenizer, oracle_models, dev)
    assert len(texts[2]) == 0
    _check_counts(model, texts, mels, frames, tokens, tokenizer, unit, f"{size}/{unit}", seed=1)


def test_counts_equal_force_align_medium(tokenizer, dev):
    model, texts, mels, frames, tokens = _medium_batch(tokenizer, dev, n=4)
    _check_counts(model, texts, mels, frames, tokens, tokenizer, "subword", "medium", seed=2)


def test_strict_raises_like_the_reference(tokenizer, oracle_models, dev):
    """Fewer hypothesis words than end times: the IndexError of head_boundary_counts_batch; CPU maps: WcaError."""
    from whisper_char_alignment_b200 import _cabi, timing

    from test_gpu_word_probs import _tokens

    model, texts, mels, frames, _ = _small_batch("micro", "char", tokenizer, oracle_models, dev, n=2, seed=3)
    texts_ws = [texts[0] + tokenizer.encode(" ") * 3, texts[1]]  # char words of only spaces vanish from the hypothesis
    maps = timing.get_attentions_widths_batch(mels, _tokens(tokenizer, texts_ws, dev), model, tokenizer, frames, [7])
    configs = [Config(7, "mean", 15, 1.0, 1.0, 0.0)]
    with pytest.raises(IndexError):
        timing.alignment_config_counts_batch({7: maps[7][0]}, texts_ws, tokenizer, [np.array([0.5])] * 2, configs,
                                             aligned_unit_type="char", ref_words_list=[["qqqqqqq"], ["qqqqqqq"]])
    with pytest.raises(_cabi.WcaError):
        timing.alignment_config_counts_batch({7: [m.cpu() for m in maps[7][0]]}, texts_ws, tokenizer,
                                             [np.array([0.5])] * 2, configs)


# ------------------------------------------------------------------ CLI against infer_ali
@pytest.mark.parametrize("strict", [False, True], ids=["plain", "strict"])
def test_tune_alignment_cli_equals_infer_ali(strict, tmp_path, dev):
    """tune_alignment on the synthetic dataset with a random:micro model: every config's precision, recall and F1 are
    exactly what infer_ali reports with that config's flags, and the best flags are those of the top-ranked config."""
    from whisper_char_alignment_b200 import tuning
    from whisper_char_alignment_b200.cli import infer_ali, tune_alignment

    data = ["--model", "random:micro", "--dataset", "synthetic", "--scp", "timit:6", "--batch_size", "4",
            "--tolerance", "0.5"] + (["--strict"] if strict else [])
    grid = ["--medfilt_widths", "3", "9", "--aggrs", "mean", "topk", "--topks", "1", "3", "--weights", "1,1,0",
            "0,1,0.5"]
    tune_alignment.main(data + grid + ["--output_dir", str(tmp_path / "tune")])
    [path] = glob.glob(os.path.join(str(tmp_path / "tune"), "*-tune.json"))
    res = json.load(open(path))
    configs = tuning.expand_grid([3, 9], ["mean", "topk"], [1, 3], [(1, 1, 0), (0, 1, 0.5)])
    assert [Config(**{k: r[k] for k in Config._fields}) for r in res["configs"]] == configs
    counts = np.array([[r["hits"], r["n_pred"], r["n_ref"]] for r in res["configs"]], dtype=np.int64)
    assert res["ranking"] == tuning.rank_configs(counts)
    assert res["best_flags"] == tuning.infer_ali_flags(configs[res["ranking"][0]])
    assert res["strict"] == strict and counts[:, 0].sum() > 0
    for i, c in enumerate(configs):
        out = tmp_path / f"infer{i}"
        infer_ali.main(data + tuning.infer_ali_flags(c) + ["--output_dir", str(out)])
        [p] = glob.glob(os.path.join(str(out), "*.json"))
        want = json.load(open(p))
        for k in ("precision", "recall", "f1", "r_value"):
            assert res["configs"][i][k] == want[k], (c, k)
