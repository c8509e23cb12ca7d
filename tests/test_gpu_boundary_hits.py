"""GPU suite: every head's word-boundary accuracy on the device -- the wca_boundary_hits kernel
(csrc/boundary_hits.cu) against the reference's metrics.eval_n1 / eval_n1_strict, timing.head_boundary_counts_batch
against the per-head host loop it replaces, and the find_alignment_heads / infer_ali --alignment_heads workflow.
Counts are integers: every comparison is exact."""
import glob
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GEMM_MODE, ROOT
from test_gpu_scoring import Guarded
from whisper_char_alignment_b200.metrics import eval_n1, eval_n1_strict

pytestmark = pytest.mark.gpu

MAX_WORDS = 448  # Whisper's text context bounds the words of one utterance


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


# ------------------------------------------------------------------ kernel against metrics.py
def _times(rng, n, kind):
    """n float64 boundary times: kind 0 sorted on the 20 ms frame grid (what the DTW writes), 1 sorted continuous,
    2 unsorted, 3 sorted with duplicates, 4 sorted with NaNs."""
    if kind == 0:
        t = np.sort(rng.integers(0, 1500, n)) / 50.0
    elif kind == 1:
        t = np.sort(rng.random(n) * 30)
    elif kind == 2:
        t = rng.integers(0, 300, n) / 50.0
    elif kind == 3:
        t = np.sort(np.repeat(rng.integers(0, 300, n) / 50.0, 2)[:n])
    else:
        t = np.sort(rng.integers(0, 1500, n) / 50.0)
        t[rng.random(n) < 0.1] = np.nan
    return t.astype(np.float64)


def _problems(seed, n_lists, heads_per_list, long_every=97):
    """Reference lists and, per list, heads_per_list predictions; lengths 0..448 (mostly short, every long_every-th list
    long), W_ref != W_hyp in general; predictions partly derived from the reference (so that hits, exact-tolerance
    distances and duplicates occur), partly independent; word ids from a vocabulary of 1, 3 or 50 words."""
    rng = np.random.default_rng(seed)
    refs, ref_ids, preds, hyp_ids, utt_of = [], [], [], [], []
    for u in range(n_lists):
        long = u % long_every == 0
        n_ref = int(rng.integers(0, MAX_WORDS + 1)) if long else int(rng.geometric(0.08)) - 1
        vocab = (1, 3, 50)[u % 3]
        y = _times(rng, n_ref, int(rng.integers(0, 5)))
        refs.append(y)
        ref_ids.append(rng.integers(0, vocab, n_ref).astype(np.int32))
        n_hyp = int(rng.integers(0, MAX_WORDS + 1)) if long else max(int(n_ref + rng.integers(-3, 4)), 0)
        if u % 11 == 5:
            n_hyp = 0
        hyp_ids.append(rng.integers(0, vocab, n_hyp).astype(np.int32))
        for _ in range(heads_per_list):
            mode = int(rng.integers(0, 3))
            if mode == 0 and n_ref:  # the reference shifted by multiples of 10 ms: distances at the tolerances exactly
                src = y[np.minimum(np.arange(n_hyp), n_ref - 1)] if n_hyp else y[:0]
                yh = src + rng.integers(-3, 4, n_hyp) * 0.01
            else:
                yh = _times(rng, n_hyp, int(rng.integers(0, 5)))
            preds.append(yh.astype(np.float64))
            utt_of.append(u)
    return refs, ref_ids, preds, hyp_ids, np.array(utt_of, dtype=np.int64)


def _launch(preds, utt_of, refs, tol, dev, ref_ids=None, hyp_ids=None):
    """Predictions laid out as wca_dtw_align lays them out (W + 1 slots at word_off; the spare slot holds a value that
    would count as a hit if it were read), one launch; returns the hits after checking the guard zones."""
    from whisper_char_alignment_b200 import _cabi

    P = len(preds)
    n = np.array([len(p) for p in preds], dtype=np.int64)
    off = np.concatenate([[0], np.cumsum(n + 1)[:-1]]) if P else np.zeros(0, np.int64)
    flat = np.zeros(int((n + 1).sum()) + 1, dtype=np.float64)
    for p, (o, yh) in enumerate(zip(off, preds)):
        flat[o: o + len(yh)] = yh
        r = refs[utt_of[p]]
        flat[o + len(yh)] = r[0] if len(r) else 0.0
    recs = np.zeros(P, dtype=_cabi.UTT_DTYPE)
    recs["word_off"], recs["n_words"] = off, n
    d_utts = _cabi.upload_utts(recs, dev) if P else torch.zeros(8, dtype=torch.uint8, device=dev)
    end_times = torch.from_numpy(flat).to(dev)
    out = Guarded(P, torch.int32, dev)
    _cabi.boundary_hits(end_times, d_utts, utt_of, refs, tol, out.out, ref_ids=ref_ids, hyp_ids=hyp_ids,
                        n_pred=None if ref_ids is None else n)
    return out.check(np.ones(P, dtype=bool)).astype(np.int64)


def _host(preds, utt_of, refs, tol, ref_ids=None, hyp_ids=None):
    if ref_ids is None:
        return np.array([eval_n1(refs[u], yh, tol)[0] for yh, u in zip(preds, utt_of)], dtype=np.int64)
    words = lambda ids: [str(int(i)) for i in ids]  # noqa: E731
    return np.array([eval_n1_strict(refs[u], yh, words(ref_ids[u]), words(hyp_ids[u][: len(yh)]), tol)[0]
                     for yh, u in zip(preds, utt_of)], dtype=np.int64)


@pytest.mark.parametrize("strict", [False, True], ids=["plain", "strict"])
@pytest.mark.parametrize("tol", [0.0, 0.01, 0.02, 0.05, 1e300])
def test_kernel_equals_metrics(tol, strict, dev):
    """Lists of 0..448 words, sorted and unsorted, on the frame grid and off it, with duplicates and NaNs, predictions
    at exact multiples of 10 ms from the reference (distances equal to the tolerance), tolerance 0 and huge, word ids
    from vocabularies of 1, 3 and 50 words: equal to metrics.py problem by problem."""
    refs, ref_ids, preds, hyp_ids, utt_of = _problems(int(tol * 1000) % 97 + 3 * strict, 300, 4)
    ids = dict(ref_ids=ref_ids, hyp_ids=hyp_ids) if strict else {}
    got = _launch(preds, utt_of, refs, tol, dev, **ids)
    want = _host(preds, utt_of, refs, tol, **ids)
    bad = np.nonzero(got != want)[0]
    assert not len(bad), [(int(p), int(got[p]), int(want[p]), len(preds[p]), len(refs[utt_of[p]])) for p in bad[:5]]
    assert want.sum() > 0


@pytest.mark.parametrize("strict", [False, True], ids=["plain", "strict"])
def test_kernel_twenty_thousand_problems_in_one_launch(strict, dev):
    refs, ref_ids, preds, hyp_ids, utt_of = _problems(99 + strict, 5000, 4, long_every=250)
    assert len(preds) == 20000
    ids = dict(ref_ids=ref_ids, hyp_ids=hyp_ids) if strict else {}
    got = _launch(preds, utt_of, refs, 0.02, dev, **ids)
    np.testing.assert_array_equal(got, _host(preds, utt_of, refs, 0.02, **ids))


def test_kernel_problem_alone_and_in_any_batch(dev):
    """A problem's count does not depend on the batch: the same problems alone, in batches of 3 and 50, and in reverse
    order."""
    refs, ref_ids, preds, hyp_ids, utt_of = _problems(5, 60, 3)
    for ids in ({}, dict(ref_ids=ref_ids, hyp_ids=hyp_ids)):
        full = _launch(preds, utt_of, refs, 0.02, dev, **ids)
        rev = _launch(preds[::-1], utt_of[::-1], refs, 0.02, dev, **ids)
        np.testing.assert_array_equal(rev[::-1], full)
        for size in (3, 50):
            parts = np.concatenate([_launch(preds[s: s + size], utt_of[s: s + size], refs, 0.02, dev, **ids)
                                    for s in range(0, len(preds), size)])
            np.testing.assert_array_equal(parts, full)
        for p in range(0, len(preds), 17):
            np.testing.assert_array_equal(_launch(preds[p: p + 1], utt_of[p: p + 1], refs, 0.02, dev, **ids), full[p: p + 1])


def test_kernel_rejects_bad_arguments(dev):
    """Null pointers, n_problems < 0, a negative or NaN tolerance and an unknown mode return WCA_ERR_INVALID with a
    message and write nothing; the binding raises for them and for over-long strict references; n_problems == 0 is a
    valid launch that writes nothing."""
    from whisper_char_alignment_b200 import _cabi

    lib = _cabi.load()
    t = torch.zeros(16, dtype=torch.float64, device=dev)
    recs = np.zeros(4, dtype=_cabi.UTT_DTYPE)
    recs["n_words"] = 2
    d_utts = _cabi.upload_utts(recs, dev)
    utt_of = torch.zeros(4, dtype=torch.int32, device=dev)
    off = torch.tensor([0, 3], dtype=torch.int64, device=dev)
    ids = torch.zeros(4, dtype=torch.int32, device=dev)
    out = Guarded(4, torch.int32, dev)
    s = torch.cuda.current_stream().cuda_stream
    p = lambda x: x.data_ptr()  # noqa: E731
    good = [p(t), p(d_utts), p(utt_of), 4, p(t), p(off), p(ids), p(ids), p(off), 0.02, 1, p(out.out), s]
    bad = []
    for i in (0, 1, 2, 4, 5, 6, 7, 8, 11):
        a = list(good)
        a[i] = None
        bad.append(a)
    for i, v in ((3, -1), (9, -0.5), (9, float("nan")), (9, float("-inf")), (10, 2), (10, -1)):
        a = list(good)
        a[i] = v
        bad.append(a)
    for a in bad:
        assert lib.wca_boundary_hits(*a) == -1, a
        assert lib.wca_last_error().decode().startswith("wca_boundary_hits:")
    plain = list(good)
    plain[6] = plain[7] = plain[8] = None
    plain[10] = 0
    zero = list(good)
    zero[3] = 0
    assert lib.wca_boundary_hits(*zero) == 0
    torch.cuda.synchronize()
    out.check(np.zeros(4, dtype=bool))
    assert lib.wca_boundary_hits(*plain) == 0  # the plain mode needs no ids
    torch.cuda.synchronize()
    out.check(np.ones(4, dtype=bool))

    out = Guarded(2, torch.int32, dev)
    refs = [np.zeros(3), np.zeros(1)]
    for kw in (dict(tolerance=-1.0), dict(tolerance=float("nan")), dict(utt_of=np.array([0, 2])),
               dict(ref_ids=[np.zeros(3, np.int32), np.zeros(1, np.int32)]),
               dict(ref_ids=[np.zeros(2, np.int32), np.zeros(1, np.int32)], hyp_ids=[np.zeros(2, np.int32)] * 2),
               dict(refs=[np.zeros(1025), np.zeros(1)], ref_ids=[np.zeros(1025, np.int32), np.zeros(1, np.int32)],
                    hyp_ids=[np.zeros(2, np.int32)] * 2, n_pred=np.array([2, 2])),
               dict(ref_ids=[np.zeros(3, np.int32), np.zeros(1, np.int32)], hyp_ids=[np.zeros(2, np.int32)] * 2),
               dict(ref_ids=[np.zeros(3, np.int32), np.zeros(1, np.int32)], hyp_ids=[np.zeros(2, np.int32)] * 2,
                    n_pred=np.array([2, 3])),
               dict(hits=torch.zeros(2, dtype=torch.int64, device=dev)),
               dict(end_times=t.float())):
        args = dict(end_times=t, d_utts=d_utts, utt_of=np.array([0, 1]), refs=refs, tolerance=0.02, hits=out.out)
        args.update(kw)
        with pytest.raises(_cabi.WcaError):
            _cabi.boundary_hits(args["end_times"], args["d_utts"], args["utt_of"], args["refs"], args["tolerance"],
                                args["hits"], ref_ids=args.get("ref_ids"), hyp_ids=args.get("hyp_ids"),
                                n_pred=args.get("n_pred"))
    torch.cuda.synchronize()
    out.check(np.zeros(2, dtype=bool))


# ------------------------------------------------------------------ the API against the per-head host loop
def _references(rng, ends_hat, words_hat, frames):
    """Reference boundaries and words near a prediction (so that the tolerance matters): jittered on the 10 ms grid,
    a few dropped or added, words with case and punctuation changed, a few replaced."""
    n = len(ends_hat)
    keep = rng.random(n) > 0.15
    y = np.asarray(ends_hat, dtype=np.float64)[keep] + rng.integers(-4, 5, int(keep.sum())) * 0.01
    words = [w for w, k in zip(words_hat, keep) if k]
    extra = int(rng.integers(0, 3))
    y = np.concatenate([y, rng.integers(0, frames, extra) / 50.0])
    words = words + ["extra"] * extra
    order = np.argsort(y, kind="stable")
    y = y[order]
    words = [words[i] for i in order]
    style = lambda w: rng.choice([w, w.upper(), w.capitalize(), w + ",", '"' + w + '."', "zz" + w])  # noqa: E731
    return y, [str(style(w)) for w in words]


def _host_counts(w, text_tokens, tokenizer, unit, ref_ends, ref_words, tol):
    """The loop head_boundary_counts_batch replaces: force_align per head, metrics.py per head."""
    from whisper_char_alignment_b200 import timing

    L, H = w.shape[:2]
    c = np.zeros((L, H, 3), dtype=np.int64)
    for l in range(L):
        for h in range(H):
            words, _, ends_hat, _, _ = timing.force_align(w[l, h][None, None], text_tokens, tokenizer, unit,
                                                          aggregation="mean")
            if ref_words is None:
                c[l, h] = (eval_n1(ref_ends, ends_hat, tol)[0], len(ends_hat), len(ref_ends))
            else:
                tp, fp, fn = eval_n1_strict(ref_ends, ends_hat, ref_words, " ".join(words[:-1]).split(), tol)
                c[l, h] = (tp, tp + fp, tp + fn)
    return c


def _check_api(maps, texts, tokenizer, unit, frames, seed, label):
    from whisper_char_alignment_b200 import _cabi, timing

    rng = np.random.default_rng(seed)
    refs, ref_words = [], []
    for w, t, f in zip(maps, texts, frames):  # references built around one head's alignment of each utterance
        out = timing.force_align(w[-1, 0][None, None], t, tokenizer, unit, aggregation="mean")
        words = " ".join(out[0][:-1]).split() if not isinstance(out, list) else ["a", "b"]
        ends = out[2] if not isinstance(out, list) else np.array([0.1, 0.3])
        y, rw = _references(rng, ends[: len(words)], words, f)
        refs.append(y)
        ref_words.append(rw)
    for strict in (False, True):
        rw = ref_words if strict else None
        before = _cabi.launch_count()
        got = timing.head_boundary_counts_batch(maps, texts, tokenizer, refs, aligned_unit_type=unit, tolerance=0.02,
                                                ref_words_list=rw)
        assert _cabi.launch_count() - before == 3  # aggregation, DTW, scoring
        total = 0
        for b, w in enumerate(maps):
            want = _host_counts(w, texts[b], tokenizer, unit, refs[b], None if rw is None else rw[b], 0.02)
            assert got[b].dtype == np.int64 and got[b].shape == want.shape
            np.testing.assert_array_equal(got[b], want, err_msg=f"{label} strict={strict} utterance {b}")
            total += int(want[..., 0].sum())
        assert total > 0, label


@pytest.mark.parametrize("unit", ["char", "subword"])
@pytest.mark.parametrize("size", ["micro", "mini"])
def test_api_equals_host_loop_small_models(size, unit, tokenizer, oracle_models, dev):
    """A ragged batch with an EOT-only utterance on the micro and mini fixture models, plain and strict."""
    from test_gpu_parity import product_model
    from test_gpu_word_probs import _synthetic_batch, _tokens
    from whisper_char_alignment_b200 import timing

    model = product_model(oracle_models(size), dev)
    texts, mels, frames = _synthetic_batch(model, tokenizer, unit, 6, seed=13, dev=dev)
    maps, _ = timing.get_attentions_batch(mels, _tokens(tokenizer, texts, dev), model, tokenizer, frames)
    got = timing.head_boundary_counts_batch(maps, texts, tokenizer, [np.array([0.5, 1.0])] * 6, aligned_unit_type=unit)
    assert (got[2][..., 0] == 0).all() and (got[2][..., 1] == 0).all() and (got[2][..., 2] == 2).all()  # EOT-only
    _check_api(maps, texts, tokenizer, unit, frames, seed=1, label=f"{size}/{unit}")


def test_api_equals_host_loop_medium_batch(tokenizer, dev):
    """Whisper-medium dims (random init, qk_gain 4), 24 layers x 16 heads, a TIMIT-shaped batch of 4."""
    from test_gpu_word_probs import _tokens
    from whisper_char_alignment_b200 import timing
    from whisper_char_alignment_b200.retokenize import encode
    from whisper_char_alignment_b200.synthetic import timit_shaped
    from whisper_char_alignment_b200.whisper_model import load_model

    model = load_model("random:medium", dev, qk_gain=4.0)
    utts = timit_shaped(4, tokenizer, n_mels=model.dims.n_mels, seed=8)
    texts = [encode(u.text, tokenizer, "subword") for u in utts]
    frames = [u.max_frames for u in utts]
    mels = torch.stack([u.mel for u in utts]).to(dev)
    maps, _ = timing.get_attentions_batch(mels, _tokens(tokenizer, texts, dev), model, tokenizer, frames)
    _check_api(maps, texts, tokenizer, "subword", frames, seed=2, label="medium")


def test_api_strict_raises_like_the_reference(tokenizer, oracle_models, dev):
    """Fewer hypothesis words than end times: eval_n1_strict's IndexError; CPU maps: WcaError."""
    from test_gpu_parity import product_model
    from test_gpu_word_probs import _synthetic_batch, _tokens
    from whisper_char_alignment_b200 import _cabi, timing

    from whisper_char_alignment_b200.retokenize import split_tokens_on_spaces

    model = product_model(oracle_models("micro"), dev)
    texts, mels, frames = _synthetic_batch(model, tokenizer, "char", 2, seed=3, dev=dev)
    maps, _ = timing.get_attentions_batch(mels, _tokens(tokenizer, texts, dev), model, tokenizer, frames)
    # in char units every space piece opens a word: words of only spaces vanish from " ".join(words[:-1]).split()
    texts_ws = [texts[0] + tokenizer.encode(" ") * 3, texts[1]]
    words, _ = split_tokens_on_spaces(texts_ws[0] + [tokenizer.eot], tokenizer, "char")
    assert len(" ".join(words[:-1]).split()) == len(words) - 4
    maps_ws, _ = timing.get_attentions_batch(mels, _tokens(tokenizer, texts_ws, dev), model, tokenizer, frames)
    with pytest.raises(IndexError):
        _host_counts(maps_ws[0], texts_ws[0], tokenizer, "char", np.array([0.5]), ["qqqqqqq"], 0.02)
    with pytest.raises(IndexError):
        timing.head_boundary_counts_batch(maps_ws, texts_ws, tokenizer, [np.array([0.5])] * 2, aligned_unit_type="char",
                                          ref_words_list=[["qqqqqqq"], ["qqqqqqq"]])
    with pytest.raises(_cabi.WcaError):
        timing.head_boundary_counts_batch([m.cpu() for m in maps], texts, tokenizer, [np.array([0.5])] * 2)


@pytest.mark.skipif(GEMM_MODE == "bf16x9", reason="already inside the bf16x9 run")
def test_api_in_the_bf16x9_gemm_mode():
    """The API tests of this file again with the forward's linears on cuBLAS 12.9's BF16x9-emulated fp32 GEMMs (the
    libraries must be mapped before torch is imported, hence a subprocess)."""
    env = dict(os.environ, WCA_FP32_GEMM="bf16x9")
    cmd = [sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider", os.path.abspath(__file__),
           "-k", "api_equals"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=3000)
    tail = (r.stdout or "")[-6000:]
    assert r.returncode == 0, f"bf16x9 run failed (rc {r.returncode}):\n{tail}\n{(r.stderr or '')[-3000:]}"
    m = re.search(r"(\d+) passed", r.stdout)
    assert m and int(m.group(1)) >= 5, tail


# ------------------------------------------------------------------ CLI
@pytest.mark.parametrize("strict", [False, True], ids=["plain", "strict"])
def test_find_alignment_heads_cli_equals_host_loop(strict, tmp_path, dev):
    """find_alignment_heads on the synthetic dataset with a random:micro model: the table equals the per-head host loop
    over the same prepared utterances, and the mask decodes to the top --n_heads of that table."""
    from whisper_char_alignment_b200 import heads, timing
    from whisper_char_alignment_b200.cli import common, find_alignment_heads
    from whisper_char_alignment_b200.dataset import DATASET

    flags = ["--model", "random:micro", "--dataset", "synthetic", "--scp", "timit:6", "--output_dir", str(tmp_path),
             "--batch_size", "4", "--tolerance", "0.5", "--n_heads", "2"] + (["--strict"] if strict else [])
    find_alignment_heads.main(flags)
    [path] = glob.glob(os.path.join(str(tmp_path), "*-heads.json"))
    res = json.load(open(path))
    model, tk, whisper_pkg, source = common.load_model_and_tokenizer("random:micro", dev)
    dataset = DATASET["synthetic"]("timit:6", n_mels=80, device=dev)
    L, H = model.dims.n_text_layer, model.dims.n_text_head
    want = np.zeros((L, H, 3), dtype=np.int64)
    for n in range(len(dataset)):
        it = common.prepare(dataset[n], tk, "subword", dev, whisper_pkg, model)
        if it is None:
            continue
        w, _ = timing.get_attentions(it["mel"], it["tokens"], model, tk, it["max_frames"])
        want += _host_counts(w, it["text_tokens"], tk, "subword", it["ends"], it["text"].split() if strict else None, 0.5)
    table = np.array([[r["hits"], r["n_pred"], r["n_ref"]] for r in res["heads"]], dtype=np.int64).reshape(L, H, 3)
    np.testing.assert_array_equal(table, want)
    assert [(r["layer"], r["head"]) for r in res["heads"]] == [(l, h) for l in range(L) for h in range(H)]
    assert want[..., 0].sum() > 0
    mask = heads.decode_alignment_heads(res["mask"], L, H)
    np.testing.assert_array_equal(mask, heads.rank_heads(want, 2))
    assert res["alignment_heads"] == np.argwhere(mask).tolist()
    assert res["model_source"] == source and res["transcript_source"] == common.transcript_source(whisper_pkg)
    assert res["n_heads"] == 2 and res["strict"] == strict
    for r in res["heads"]:
        assert 0.0 <= r["f1"] <= 1.0 and 0.0 <= r["precision"] <= 1.0 and 0.0 <= r["recall"] <= 1.0


INFER_JSON_KEYS = {  # what infer_ali writes without the new flag, as before it existed
    "model", "dataset", "scp", "output_dir", "n_mels", "medfilt_width", "aggr", "topk", "aligned_unit_type", "tolerance",
    "w_colnorm", "w_rownorm", "w_coverage", "plot", "strict", "save_prediction", "default_whisper_timing", "batch_size",
    "precision", "recall", "f1", "r_value", "model_source", "transcript_source"}


def test_infer_ali_with_found_heads(tmp_path, dev):
    """infer_ali --default_whisper_timing --alignment_heads (a mask string or a -heads.json file) gives the end times
    default_find_alignment_batch gives on a model whose heads were set by hand; without the flag the results JSON has
    the same keys as before the flag existed."""
    import joblib

    from whisper_char_alignment_b200 import heads, timing
    from whisper_char_alignment_b200.cli import common, infer_ali
    from whisper_char_alignment_b200.dataset import DATASET

    mask = np.zeros((2, 2), dtype=bool)
    mask[0, 1] = mask[1, 0] = True  # not the default (upper half) heads
    dump = heads.encode_alignment_heads(mask).decode("ascii")
    heads_file = tmp_path / "found-heads.json"
    heads_file.write_text(json.dumps({"mask": dump}))
    base = ["--model", "random:micro", "--dataset", "synthetic", "--scp", "timit:6", "--save_prediction",
            "--batch_size", "4", "--default_whisper_timing"]
    runs = {}
    for name, extra in (("string", ["--alignment_heads", dump]), ("file", ["--alignment_heads", str(heads_file)]),
                        ("none", [])):
        out = tmp_path / name
        infer_ali.main(base + ["--output_dir", str(out)] + extra)
        runs[name] = joblib.load(glob.glob(os.path.join(str(out), "*-predictions.pkl"))[0])
        [res] = [p for p in glob.glob(os.path.join(str(out), "*.json"))]
        keys = set(json.load(open(res)))
        assert keys == (INFER_JSON_KEYS | {"alignment_heads"} if extra else INFER_JSON_KEYS), name

    model, tk, whisper_pkg, _ = common.load_model_and_tokenizer("random:micro", dev)
    default = model.alignment_heads.to_dense().cpu().numpy().copy()
    model.set_alignment_heads(heads.encode_alignment_heads(mask))
    assert torch.equal(model.alignment_heads.to_dense().cpu(), torch.from_numpy(mask))
    dataset = DATASET["synthetic"]("timit:6", n_mels=80, device=dev)
    items = [common.prepare(dataset[n], tk, "subword", dev, whisper_pkg, model) for n in range(len(dataset))]
    outs = timing.default_find_alignment_batch(model, tk, [it["text_tokens"] for it in items],
                                               [it["mel"] for it in items], [it["max_frames"] for it in items])
    differs = False
    for n, out in enumerate(outs):
        want = np.zeros(0) if isinstance(out, list) else out[2]
        for name in ("string", "file"):
            np.testing.assert_array_equal(runs[name][n]["ends_hat"], want, err_msg=f"{name} utterance {n}")
        differs |= not np.array_equal(runs["none"][n]["ends_hat"], want)
    assert differs and not np.array_equal(default, mask)  # the flag changed which heads were used
