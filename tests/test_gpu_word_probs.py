"""GPU suite: per-word probabilities (timing.word_probabilities_batch, the word confidence of upstream
whisper.timing.find_alignment) and their kernel (wca_token_probs, csrc/token_probs.cu) through the C ABI.

Bar of the kernel: |p - p64| <= TP_K * eps * (1 + log2 n_cols) * p64 + FLT_MIN against the float64 softmax of the same
fp32 logits (eps = 2^-23): a few fp32 roundings per exp and per rescale, and a sum over n_cols terms in blocks; FLT_MIN
covers results below the normal range, where fp32 has no relative precision left.  The word probabilities, means of
token probabilities, are held to the same bar.  NaN exactly where torch's float64 softmax has it, exact 0 for a -inf
target.  Every output sits between guard zones and must come back fully written."""
import glob
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GEMM_MODE, ROOT, golden_names, load_golden, record_measure
from test_gpu_scoring import Guarded
from test_word_probs_reference import ref_word_probabilities

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -23
FLT_MIN = 2.0 ** -126
TP_K = 8
# End-to-end bar of the forward against the oracle's CPU forward: the logits within E2E_LOGIT_RTOL of their largest
# magnitude (the north-star end-to-end bar; the maps measure <= 5e-5).  A logit error of at most d moves log p by at
# most 2 d (the target's own logit and the log-sum-exp), so the probabilities are held to exp(2 d) - 1 relative.
E2E_LOGIT_RTOL = 1e-4

NCOLS = [1, 2, 3, 4, 5, 255, 256, 257, 1023, 50256, 50257, 51865, 51866]
N_KINDS = 12


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def bar(n_cols):
    return TP_K * EPS * (1.0 + math.log2(n_cols))


# ------------------------------------------------------------------ hand-built rows in a poisoned buffer
def _rows_of_kind(gen, n_rows, n, dev, row0):
    """(n_rows, n) fp32 logits and int64 targets; row r is of kind (row0 + r) % N_KINDS:
    0 normal, 1-4 the maximum at column 0 / n-1 / 2 (scalar head of a misaligned row) / n-2 (scalar tail),
    5 large equal values, 6 magnitude ~100, 7 a NaN, 8 a +inf, 9 all -inf, 10 a -inf target, 11 half the row -inf."""
    x = torch.randn(n_rows, n, generator=gen, device=dev) * 3
    idx = torch.arange(n_rows, device=dev)
    kind = (idx + row0) % N_KINDS
    tgt = torch.stack([torch.zeros_like(idx), torch.full_like(idx, n - 1), torch.full_like(idx, n // 2)])[idx % 3, idx]
    rnd = torch.randint(0, n, (n_rows,), generator=gen, device=dev)
    tgt = torch.where(idx % 7 == 6, rnd, tgt)
    peak = x.amax(-1) + 5
    for k, col in ((1, 0), (2, n - 1), (3, min(2, n - 1)), (4, max(n - 2, 0))):
        rows = idx[kind == k]
        x[rows, col] = peak[rows]
        tgt[rows[::2]] = col  # the maximum is the target every other time
    x[kind == 5] = 88.0
    big = idx[kind == 6]
    x[big] = (torch.rand(len(big), n, generator=gen, device=dev) * 200 - 100)
    nan_rows, inf_rows = idx[kind == 7], idx[kind == 8]
    x[nan_rows, rnd[nan_rows]] = float("nan")
    x[inf_rows, rnd[inf_rows]] = float("inf")
    x[kind == 9] = float("-inf")
    ninf = idx[kind == 10]
    x[ninf, tgt[ninf]] = float("-inf")
    half = idx[kind == 11]
    mask = torch.rand(len(half), n, generator=gen, device=dev) < 0.5
    sub = x[half]
    sub[mask] = float("-inf")
    sub[torch.arange(len(half), device=dev), tgt[half]] = 1.0
    x[half] = sub
    return x, tgt


def _n_rows(n):
    return 3000 if n <= 1023 else (2500 if n == 51866 else 200)


def _poisoned_cases(dev):
    """Every NCOLS case's rows in one buffer at an odd pitch (row addresses cycle through every 4-byte alignment modulo
    16), plus the product's own pitch 51 872 for n_cols = 51 865; everything outside [0, n_cols) of a row is NaN or
    +-inf.  Returns (buf, [(n_cols, first float offset, pitch, logits, targets)])."""
    gen = torch.Generator(device=dev).manual_seed(7)
    layout, off = [], 3
    specs = [(n, n + (1 if n % 2 == 0 else 2)) for n in NCOLS] + [(51865, 51872)]
    for n, pitch in specs:
        layout.append((n, off, pitch))
        off += _n_rows(n) * pitch + 5
    poison = torch.tensor([float("nan"), float("inf"), float("-inf")], device=dev)
    buf = poison.repeat(off // 3 + 1)[:off].contiguous()
    cases = []
    for i, (n, o, pitch) in enumerate(layout):
        x, tgt = _rows_of_kind(gen, _n_rows(n), n, dev, row0=i)
        buf[o: o + x.shape[0] * pitch].view(x.shape[0], pitch)[:, :n] = x
        cases.append((n, o, pitch, x, tgt))
    return buf, cases


def _addrs(buf, o, pitch, n_rows):
    return buf.data_ptr() + 4 * (o + pitch * np.arange(n_rows, dtype=np.int64))


def _launch(addrs, targets, n_cols, dev):
    from whisper_char_alignment_b200 import _cabi

    out = Guarded(len(addrs), torch.float32, dev)
    _cabi.token_probs(addrs, np.asarray(targets), n_cols, out.out)
    return out.check(np.ones(len(addrs), dtype=bool))


def _fp64(x, tgt):
    """torch's float64 softmax over the row, at the target: the semantics (NaN, +-inf) the kernel follows."""
    out = []
    for a in range(0, x.shape[0], 256):
        p = torch.softmax(x[a: a + 256].double(), dim=-1)
        out.append(p.gather(1, tgt[a: a + 256, None]).squeeze(1))
    return torch.cat(out).cpu().numpy()


def _check(got, want, n_cols, what):
    np.testing.assert_array_equal(np.isnan(got), np.isnan(want), err_msg=f"{what}: NaN pattern")
    zero = want == 0
    ok = ~np.isnan(want)
    err = np.abs(got[ok].astype(np.float64) - want[ok])
    assert (err <= bar(n_cols) * want[ok] + FLT_MIN).all(), (what, float((err / (want[ok] + FLT_MIN)).max()))
    normal = ok & (want >= 2.0 ** -100)
    units = float((np.abs(got[normal] - want[normal]) / (EPS * (1 + math.log2(n_cols)) * want[normal])).max()) if normal.any() else 0.0
    return units, zero


def test_token_probs_vs_fp64(dev):
    """Every n_cols of NCOLS, rows at every 4-byte alignment modulo 16 in a NaN / +-inf poisoned buffer, all value kinds
    of _rows_of_kind, targets at 0, n_cols - 1, the middle, random and on the maximum: against float64, NaN where torch
    has it, exactly 0 for a -inf target."""
    buf, cases = _poisoned_cases(dev)
    worst = 0.0
    for i, (n, o, pitch, x, tgt) in enumerate(cases):
        got = _launch(_addrs(buf, o, pitch, x.shape[0]), tgt.cpu().numpy(), n, dev)
        want = _fp64(x, tgt)
        kind = (np.arange(x.shape[0]) + i) % N_KINDS
        assert np.isnan(got[np.isin(kind, [7, 8, 9])]).all(), n
        if n > 1:  # with one column the -inf target is an all -inf row
            assert (got[kind == 10] == 0).all() and not np.signbit(got[kind == 10]).any(), n
        units, zero = _check(got, want, n, f"n_cols={n} pitch={pitch}")
        assert (got[zero] == 0).all()
        if n > 1:
            np.testing.assert_allclose(got[kind == 5], 1.0 / n, rtol=bar(n))  # large equal values
        worst = max(worst, units)
    print(f"token_probs vs float64: max |p - p64| = {worst:.2f} x eps x (1 + log2 n_cols) x p64 (bar {TP_K})")
    record_measure("token_probs_vs_fp64_err_in_eps_log2n", worst)


def test_a_row_gives_the_same_bits_alone_in_any_batch_and_again(dev):
    """The rows of several cases launched together, again, in batches of 7 and of 300, and a sample of them alone."""
    buf, cases = _poisoned_cases(dev)
    # one launch covers one n_cols: a batch is (up to 400) rows of one case
    for n, o, pitch, x, tgt in (c for c in cases if c[0] in (5, 257, 51865, 51866)):
        k = min(400, x.shape[0])
        a, t = _addrs(buf, o, pitch, k), tgt[:k].cpu().numpy()
        full = _launch(a, t, n, dev).view(np.int32)
        np.testing.assert_array_equal(_launch(a, t, n, dev).view(np.int32), full)
        for size in (7, 300):
            parts = np.concatenate([_launch(a[s: s + size], t[s: s + size], n, dev) for s in range(0, len(a), size)])
            np.testing.assert_array_equal(parts.view(np.int32), full, err_msg=f"n_cols={n}, batches of {size}")
        for r in range(0, k, 23):
            np.testing.assert_array_equal(_launch(a[r: r + 1], t[r: r + 1], n, dev).view(np.int32), full[r: r + 1])


def test_token_probs_rejects_bad_arguments(dev):
    """Null pointers, n_rows < 0 and n_cols < 1 return WCA_ERR_INVALID with a message; a target outside [0, n_cols) is
    refused on the host before the launch.  Nothing is written; n_rows == 0 is a valid launch."""
    from whisper_char_alignment_b200 import _cabi

    lib = _cabi.load()
    x = torch.zeros(64, device=dev)
    rows = torch.tensor([x.data_ptr()] * 4, dtype=torch.int64, device=dev)
    tg = torch.zeros(4, dtype=torch.int32, device=dev)
    out = Guarded(4, torch.float32, dev)
    s = torch.cuda.current_stream().cuda_stream
    p = lambda t: t.data_ptr()  # noqa: E731
    for args in ((None, p(tg), 4, 8, p(out.out), s), (p(rows), None, 4, 8, p(out.out), s),
                 (p(rows), p(tg), 4, 8, None, s), (p(rows), p(tg), -1, 8, p(out.out), s),
                 (p(rows), p(tg), 4, 0, p(out.out), s)):
        assert lib.wca_token_probs(*args) == -1, args
        assert lib.wca_last_error().decode().startswith("wca_token_probs:")
    assert lib.wca_token_probs(p(rows), p(tg), 0, 8, p(out.out), s) == 0
    addrs = np.full(4, x.data_ptr(), dtype=np.int64)
    for bad in ([0, 1, 8, 2], [0, -1, 3, 2]):
        with pytest.raises(_cabi.WcaError, match="outside"):
            _cabi.token_probs(addrs, np.array(bad), 8, out.out)
    with pytest.raises(_cabi.WcaError):
        _cabi.token_probs(addrs + 2, np.zeros(4), 8, out.out)  # not 4-byte aligned
    torch.cuda.synchronize()
    out.check(np.zeros(4, dtype=bool))


# ------------------------------------------------------------------ end to end on the forward's logits
def _synthetic_batch(model, tokenizer, unit, n, seed, dev):
    """n utterances of ragged text and frame counts, the third one EOT-only."""
    from oracle.synth import make_mel
    from whisper_char_alignment_b200.retokenize import encode
    from whisper_char_alignment_b200.synthetic import _sentence

    rng = np.random.default_rng(seed)
    n_ctx, texts, mels, frames = model.dims.n_audio_ctx, [], [], []
    for i in range(n):
        f = int(rng.integers(20, n_ctx + 1))
        texts.append([] if i == 2 else encode(_sentence(rng, int(rng.integers(3, 60))), tokenizer, unit))
        mels.append(make_mel(model.dims.n_mels, 2 * n_ctx, 2 * f, seed + i))
        frames.append(f)
    return texts, torch.stack(mels).to(dev), frames


def _tokens(tokenizer, texts, dev):
    return [torch.tensor([*tokenizer.sot_sequence, tokenizer.no_timestamps, *t, tokenizer.eot], device=dev) for t in texts]


def _check_against_restatement(logits, texts, got, tokenizer, unit, label):
    sot, V = len(tokenizer.sot_sequence), tokenizer.eot
    worst = 0.0
    for b, (lg, t) in enumerate(zip(logits, texts)):
        tp64, wp64 = ref_word_probabilities(lg[: sot + len(t)], t, tokenizer, unit)
        tp, wp = got[b]
        assert tp.dtype == np.float32 and wp.dtype == np.float64 and tp.shape == tp64.shape and wp.shape == wp64.shape
        if not len(t):
            continue
        for g, w in ((tp, tp64), (wp, wp64)):
            assert np.isfinite(g).all()
            assert (np.abs(g - w) <= bar(V) * w + FLT_MIN).all(), (label, b, float((np.abs(g - w) / w).max()))
            normal = w >= 2.0 ** -100  # below fp32's normal range a result has no relative precision left
            if normal.any():
                worst = max(worst, float((np.abs(g - w)[normal] / (EPS * (1 + math.log2(V)) * w[normal])).max()))
    return worst


@pytest.mark.parametrize("unit", ["char", "subword"])
@pytest.mark.parametrize("size", ["micro", "mini"])
def test_end_to_end_word_probs_small_models(size, unit, tokenizer, oracle_models, dev):
    """word_probabilities_batch on the logits get_attentions_batch returns (row views of one padded tensor, read in
    place) against the float64 restatement on those same logits: a ragged batch with an EOT-only utterance; one launch."""
    from test_gpu_parity import product_model
    from whisper_char_alignment_b200 import _cabi, timing

    model = product_model(oracle_models(size), dev)
    texts, mels, frames = _synthetic_batch(model, tokenizer, unit, 7, seed=11, dev=dev)
    _, logits = timing.get_attentions_batch(mels, _tokens(tokenizer, texts, dev), model, tokenizer, frames)
    before = _cabi.launch_count()
    got = timing.word_probabilities_batch(logits, texts, tokenizer, unit)
    assert _cabi.launch_count() - before == 1
    assert got[2][0].shape == (0,) and got[2][1].shape == (0,)
    worst = _check_against_restatement(logits, texts, got, tokenizer, unit, f"{size}/{unit}")
    record_measure(f"word_probs_e2e_{size}_vs_fp64_err_in_eps_log2n", worst)


@pytest.mark.parametrize("unit", ["char", "subword"])
def test_end_to_end_word_probs_medium_timit_batch(unit, tokenizer, dev):
    """Whisper-medium dims (random init, qk_gain 4), TIMIT-shaped batch of 32 plus an EOT-only utterance."""
    from whisper_char_alignment_b200 import timing
    from whisper_char_alignment_b200.retokenize import encode
    from whisper_char_alignment_b200.synthetic import timit_shaped
    from whisper_char_alignment_b200.whisper_model import load_model

    model = load_model("random:medium", dev, qk_gain=4.0)
    utts = timit_shaped(32, tokenizer, n_mels=model.dims.n_mels, seed=4)
    texts = [encode(u.text, tokenizer, unit) for u in utts] + [[]]
    mels = torch.stack([u.mel for u in utts] + [utts[0].mel]).to(dev)
    frames = [u.max_frames for u in utts] + [utts[0].max_frames]
    _, logits = timing.get_attentions_batch(mels, _tokens(tokenizer, texts, dev), model, tokenizer, frames)
    got = timing.word_probabilities_batch(logits, texts, tokenizer, unit)
    worst = _check_against_restatement(logits, texts, got, tokenizer, unit, f"medium/{unit}")
    record_measure("word_probs_e2e_medium_timit_vs_fp64_err_in_eps_log2n", worst)


@pytest.mark.parametrize("name", [n for n in golden_names() if "eot_only" not in n])
def test_end_to_end_word_probs_against_the_cpu_forward(name, tokenizer, oracle_models, dev):
    """Against the oracle's CPU forward of a reference fixture: the logits within d <= E2E_LOGIT_RTOL of their largest
    magnitude, so the word probabilities within exp(2 d) - 1 relative (plus the kernel's bar, plus FLT_MIN for
    probabilities below fp32's normal range)."""
    from oracle import ref_path
    from test_gpu_parity import product_model
    from whisper_char_alignment_b200 import timing

    g = load_golden(name)
    c = g["case"]
    om = oracle_models(c["model"], c.get("seed", 0), c.get("gain", 4.0))
    model = product_model(om, dev)
    text = g["text_tokens"].tolist()
    tokens = torch.from_numpy(g["tokens"])
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        _, logits = timing.get_attentions(torch.from_numpy(g["mel"]).to(dev), tokens.to(dev), model, tokenizer,
                                          c["frames"], c["width"], c["qk_scale"])
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    _, cpu_logits = ref_path.capture_logits(om, torch.from_numpy(g["mel"]), tokens)
    sot, V = len(tokenizer.sot_sequence), tokenizer.eot
    rows = slice(sot, sot + len(text))
    d = float((logits[rows, :V].cpu().double() - cpu_logits[rows, :V].double()).abs().max())
    scale = float(cpu_logits[rows, :V].abs().max())
    record_measure("word_probs_fixture_logits_vs_cpu_err_rel_to_max", d / scale)
    assert d <= E2E_LOGIT_RTOL * scale, (d, scale)
    _, wp = timing.word_probabilities_batch([logits], [text], tokenizer, c["unit"])[0]
    _, wp_cpu = ref_word_probabilities(cpu_logits, text, tokenizer, c["unit"])
    assert len(wp) == len(g["words"]) - 1
    # random weights put most of the vocabulary's mass away from the text: many words' probabilities lie far below
    # fp32's range (1e-150 in float64), where the fp32 result is 0 as upstream's fp32 softmax gives it -- hence FLT_MIN
    allowed = math.expm1(2 * d) + bar(V)
    diff = np.abs(wp - wp_cpu)
    assert (diff <= allowed * wp_cpu + FLT_MIN).all(), (wp, wp_cpu, allowed)
    normal = wp_cpu >= 2.0 ** -100
    if normal.any():
        record_measure("word_probs_fixture_vs_cpu_forward_rel_err", float((diff[normal] / wp_cpu[normal]).max()))


@pytest.mark.skipif(GEMM_MODE == "bf16x9", reason="already inside the bf16x9 run")
def test_end_to_end_word_probs_in_the_bf16x9_gemm_mode():
    """The end-to-end tests of this file again with the forward's linears on cuBLAS 12.9's BF16x9-emulated fp32 GEMMs
    (the libraries must be mapped before torch is imported, hence a subprocess)."""
    env = dict(os.environ, WCA_FP32_GEMM="bf16x9")
    cmd = [sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider", os.path.abspath(__file__),
           "-k", "end_to_end and not bf16x9"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=3000)
    tail = (r.stdout or "")[-6000:]
    assert r.returncode == 0, f"bf16x9 run failed (rc {r.returncode}):\n{tail}\n{(r.stderr or '')[-3000:]}"
    m = re.search(r"(\d+) passed", r.stdout)
    assert m and int(m.group(1)) >= 8, tail
    for name, val in re.findall(r"MEASURE\[bf16x9\] (\S+) = (\S+)", r.stdout):
        record_measure("bf16x9:" + name, float(val))


# ------------------------------------------------------------------ default_find_alignment with word probabilities
def test_default_find_alignment_word_probabilities(tokenizer, oracle_models, dev):
    """With word_probabilities=True: the same words, times and weights bit for bit as without, exactly one launch more,
    and the fifth slot equal to word_probabilities_batch on the capture's logits; the single-utterance form agrees."""
    from test_gpu_parity import product_model
    from whisper_char_alignment_b200 import _cabi, timing

    model = product_model(oracle_models("micro"), dev)
    texts, mels, frames = _synthetic_batch(model, tokenizer, "subword", 6, seed=21, dev=dev)
    before = _cabi.launch_count()
    plain = timing.default_find_alignment_batch(model, tokenizer, texts, mels, frames)
    n_plain = _cabi.launch_count() - before
    before = _cabi.launch_count()
    withp = timing.default_find_alignment_batch(model, tokenizer, texts, mels, frames, word_probabilities=True)
    assert _cabi.launch_count() - before == n_plain + 1
    _, logits = timing.get_attentions_batch(mels, _tokens(tokenizer, texts, dev), model, tokenizer, frames)
    api = timing.word_probabilities_batch(logits, texts, tokenizer, "subword")
    for b, (a, w) in enumerate(zip(plain, withp)):
        if isinstance(a, list):
            assert w == a == [[], [], [], [], None]
            continue
        assert a[4] is None and w[0] == a[0]
        np.testing.assert_array_equal(w[1], a[1])
        np.testing.assert_array_equal(w[2], a[2])
        assert torch.equal(w[3], a[3])
        assert w[4].dtype == np.float64 and len(w[4]) == len(w[0]) - 1
        np.testing.assert_array_equal(w[4], api[b][1])
        one = timing.default_find_alignment(model, tokenizer, texts[b], mels[b], frames[b], word_probabilities=True)
        np.testing.assert_allclose(one[4], w[4], rtol=1e-4)


# ------------------------------------------------------------------ CLI
def _run_cli(out, extra):
    import joblib

    from whisper_char_alignment_b200.cli import infer_ali

    infer_ali.main(["--model", "random:micro", "--dataset", "synthetic", "--scp", "timit:6", "--output_dir", str(out),
                    "--save_prediction", "--batch_size", "4", "--tolerance", "0.5", *extra])
    return joblib.load(glob.glob(os.path.join(str(out), "*-predictions.pkl"))[0])


@pytest.mark.parametrize("mode", ["mean", "topk", "default"])
def test_cli_word_probabilities_equal_per_utterance_calls(mode, tmp_path, tokenizer, dev):
    """infer_ali --word_probabilities --save_prediction writes probs_hat, aligned with predwords[:-1], equal to the API
    called on each utterance alone; without the flag the predictions carry no probs_hat and the same times."""
    from whisper_char_alignment_b200 import timing
    from whisper_char_alignment_b200.cli import common
    from whisper_char_alignment_b200.dataset import DATASET

    extra = {"mean": [], "topk": ["--aggr", "topk", "--topk", "3"], "default": ["--default_whisper_timing"]}[mode]
    preds = _run_cli(tmp_path / "with", extra + ["--word_probabilities"])
    plain = _run_cli(tmp_path / "without", extra)
    model, tk, whisper_pkg, _ = common.load_model_and_tokenizer("random:micro", dev)
    dataset = DATASET["synthetic"]("timit:6", n_mels=80, device=dev)
    assert len(preds) == len(plain) == len(dataset)
    for n in range(len(dataset)):
        assert "probs_hat" not in plain[n]
        np.testing.assert_array_equal(plain[n]["ends_hat"], preds[n]["ends_hat"])
        it = common.prepare(dataset[n], tk, "subword", dev, whisper_pkg, model)
        if mode == "default":
            one = timing.default_find_alignment(model, tk, it["text_tokens"], it["mel"], it["max_frames"],
                                                word_probabilities=True)
            want = np.zeros(0) if isinstance(one, list) else one[4]
        else:
            _, logits = timing.get_attentions(it["mel"], it["tokens"], model, tk, it["max_frames"])
            want = timing.word_probabilities_batch([logits], [it["text_tokens"]], tk, "subword")[0][1]
        got = preds[n]["probs_hat"]
        assert len(got) == max(len(preds[n]["predwords"]) - 1, 0)
        np.testing.assert_allclose(got, want, rtol=1e-4, err_msg=f"utterance {n}")
