"""GPU suite: the batched stock-Whisper baseline (timing.default_find_alignment_batch, reference timing.py:116-186) and
its std-normalisation kernel (wca_normalize_heads, csrc/scores.cu) through the C ABI.

Bars: the normalised maps against float64 `std_mean(unbiased=False)` on the same fp32 maps within
NORM_K * eps * (max_t |a[t,f]| / sd[f] + |w|) per element (eps = 2^-23): the error of an fp32 mean carried through the
division by sd, plus the rounding of the quotient.  The matrix adds the fp32 sum of n_sel heads
(n_sel * eps * mean_i |w_i|).  NaN (sd = 0: a column constant over the tokens) exactly where float64 has it.  DTW bit-exact
against the C oracle on the kernel's own matrix.  Every output sits between guard zones and must come back fully written."""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import default_timing_names, load_golden, record_measure
from test_gpu_scoring import Guarded, pack_maps, planted_softmax, spans

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -23
NORM_K = 16


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


# ------------------------------------------------------------------ float64 reference (checked on the CPU against oracle/ref_path)
def ref_normalize(maps, sel, row_begin, row_end):
    """maps (H, T, F) -> float64 (weights (k, T, F), matrix (row_end - row_begin, F), scale (k, 1, F)): the heads `sel`
    std-normalised over tokens (timing.py:160-161), their mean (:163), and max_t |a[t,f]| / sd[f] for the tolerance."""
    a = maps[torch.as_tensor(np.asarray(sel, dtype=np.int64), device=maps.device)].double()
    std, mean = torch.std_mean(a, dim=-2, keepdim=True, unbiased=False)
    w = (a - mean) / std
    return w, w.mean(0)[row_begin:row_end], a.abs().amax(-2, keepdim=True) / std


def _err_units(got, want, scale):
    """|got - want| / (eps * (scale + |want|)) where both are numbers; NaN positions are compared separately."""
    ok = ~np.isnan(want)
    return float((np.abs(got[ok] - want[ok]) / (EPS * (scale[ok] + np.abs(want[ok])))).max()) if ok.any() else 0.0


# ------------------------------------------------------------------ kernel against float64
#        T    F    H    k    row_begin row_end   (k heads in random order out of H)
CASES = [(1, 1, 3, 1, 0, 1), (2, 33, 4, 2, 0, 2), (5, 32, 6, 5, 1, 4), (31, 257, 8, 5, 4, 30), (32, 255, 200, 192, 3, 31),
         (33, 31, 5, 2, 0, 33), (127, 256, 9, 7, 4, 126), (128, 1, 2, 2, 5, 120), (129, 1500, 7, 5, 4, 128),
         (448, 1500, 330, 320, 4, 447), (60, 1500, 200, 192, 2, 59)]
SHARED = [(17, 130, 8), (64, 999, 8), (3, 2, 8)]  # (T, F, H): all use the list of the first of them, 5 heads, one repeated
SHARED_SEL = np.array([6, 1, 6, 0, 3], np.int32)


def _adversarial(m, gen):
    """Columns 0-2 of every head: constant over the tokens (sd = 0), one spike, a large mean over a small spread."""
    H, T, F = m.shape
    if F > 0:
        m[:, :, 0] = 0.37
    if F > 1 and T > 1:
        m[:, :, 1] = 1e-3
        m[:, T // 2, 1] = 0.9
    if F > 2 and T > 1:
        m[:, :, 2] = 0.5 + 1e-4 * torch.rand(H, T, generator=gen, device=m.device)
    return m


def _batch(dev):
    from whisper_char_alignment_b200 import _cabi

    gen = torch.Generator(device=dev).manual_seed(41)
    rng = np.random.default_rng(41)
    shapes = [c[:3] for c in CASES] + SHARED
    B = len(shapes)
    recs = np.zeros(B, dtype=_cabi.UTT_DTYPE)
    sels, sel_flat, soff, moff, woff = [], [], 0, 0, 0
    w_off = np.zeros(B, np.int64)
    for b, (T, F, H) in enumerate(shapes):
        if b < len(CASES):
            k, rb, re = CASES[b][3:]
            sel = rng.permutation(H)[:k].astype(np.int32)
            if k >= 5:
                sel[k // 2] = sel[0]  # a repeated head
            recs[b]["sel_off"] = soff + 1
            sel_flat += [np.full(1, -1, np.int32), sel]
            soff += 1 + k
        else:
            sel, rb, re = SHARED_SEL, 4 if T > 8 else 0, T - 1
            recs[b]["sel_off"] = soff + 1  # set below: one list for all of SHARED
        recs[b]["n_tokens"], recs[b]["n_frames"], recs[b]["n_sel"] = T, F, len(sel)
        recs[b]["row_begin"], recs[b]["row_end"] = rb, re
        recs[b]["matrix_off"] = moff + 5  # five untouched elements in front of every output
        moff += 5 + (re - rb) * F
        w_off[b] = woff + 3
        woff += 3 + len(sel) * T * F
        sels.append(sel)
    recs[len(CASES):]["sel_off"] = soff + 1
    sel_flat += [np.full(1, -1, np.int32), SHARED_SEL]
    maps = [_adversarial(planted_softmax(gen, H, T, F, dev), gen) for T, F, H in shapes]
    ws = pack_maps(maps, recs, dev)
    return recs, maps, sels, ws, torch.from_numpy(np.concatenate(sel_flat)).to(dev), moff, w_off, woff


def _run(recs, ws, d_sel, n_mx, w_off, n_w, dev, with_weights=True):
    from whisper_char_alignment_b200 import _cabi

    mx = Guarded(n_mx, torch.float32, dev)
    w = Guarded(n_w, torch.float32, dev) if with_weights else None
    d_off = torch.from_numpy(w_off).to(dev) if with_weights else None
    _cabi.normalize_heads(ws.data_ptr(), d_sel, _cabi.upload_utts(recs, dev), len(recs), int(recs["n_tokens"].max()),
                          int(recs["n_frames"].max()), mx.out, None if w is None else w.out, d_off)
    n_rows = recs["row_end"] - recs["row_begin"]
    got_m = mx.check(spans(n_mx, recs["matrix_off"], n_rows * recs["n_frames"]))
    got_w = None
    if with_weights:
        got_w = w.check(spans(n_w, w_off, recs["n_sel"] * recs["n_tokens"] * recs["n_frames"]))
    return got_m, got_w


def test_normalize_heads_vs_fp64(dev):
    """Weights and matrices of one ragged launch (T 1-448, F 1-1500, lists of 1-320 heads in random order with a repeated
    head, a list shared by several utterances, kept-row ranges cut at both ends, adversarial columns) against float64;
    NaN exactly where float64 has it; then with d_weights = NULL the matrix is the same bit for bit."""
    recs, maps, sels, ws, d_sel, n_mx, w_off, n_w = _batch(dev)
    got_m, got_w = _run(recs, ws, d_sel, n_mx, w_off, n_w, dev)
    worst_w = worst_m = 0.0
    for b, r in enumerate(recs):
        T, F, k = int(r["n_tokens"]), int(r["n_frames"]), int(r["n_sel"])
        rb, re = int(r["row_begin"]), int(r["row_end"])
        w64, m64, scale = (x.cpu().numpy() for x in ref_normalize(maps[b], sels[b], rb, re))
        gw = got_w[w_off[b]: w_off[b] + k * T * F].reshape(k, T, F)
        gm = got_m[int(r["matrix_off"]): int(r["matrix_off"]) + (re - rb) * F].reshape(re - rb, F)
        np.testing.assert_array_equal(np.isnan(gw), np.isnan(w64), err_msg=f"weights NaN pattern, utterance {b}")
        np.testing.assert_array_equal(np.isnan(gm), np.isnan(m64), err_msg=f"matrix NaN pattern, utterance {b}")
        assert np.isnan(w64[:, :, 0]).all()  # the constant column
        sc = np.broadcast_to(scale, w64.shape)
        err_w = _err_units(gw, w64, sc)
        assert err_w <= NORM_K, (b, err_w)
        # matrix: the mean of the heads' bounds plus the fp32 sum of k terms
        m_scale = (sc + np.abs(w64)).mean(0)[rb:re] + k / NORM_K * np.abs(w64).mean(0)[rb:re]
        err_m = _err_units(gm, m64, m_scale - np.abs(m64))
        assert err_m <= NORM_K, (b, err_m)
        worst_w, worst_m = max(worst_w, err_w), max(worst_m, err_m)
    print(f"normalize_heads vs float64: weights {worst_w:.2f}, matrix {worst_m:.2f} x eps x (max|a|/sd + |w|)")
    record_measure("normalize_heads_weights_vs_fp64_err_in_eps_cond", worst_w)
    record_measure("normalize_heads_matrix_vs_fp64_err_in_eps_cond", worst_m)
    alone_m, _ = _run(recs, ws, d_sel, n_mx, w_off, n_w, dev, with_weights=False)
    np.testing.assert_array_equal(alone_m.view(np.int32), got_m.view(np.int32))


def test_normalize_heads_rejects_bad_arguments(dev):
    from whisper_char_alignment_b200 import _cabi

    lib = _cabi.load()
    x = torch.zeros(64, device=dev)
    sel = torch.zeros(1, dtype=torch.int32, device=dev)
    recs = np.zeros(1, dtype=_cabi.UTT_DTYPE)
    recs["n_tokens"], recs["n_frames"], recs["n_sel"], recs["row_end"] = 4, 4, 1, 3
    d = _cabi.upload_utts(recs, dev)
    off = torch.zeros(1, dtype=torch.int64, device=dev)
    s = torch.cuda.current_stream().cuda_stream
    p = lambda t: t.data_ptr()  # noqa: E731
    assert lib.wca_normalize_heads(None, p(sel), p(d), 1, 4, 4, p(x), p(off), p(x), s) == -1
    assert lib.wca_normalize_heads(p(x), p(sel), p(d), 1, 4, 4, p(x), None, p(x), s) == -1  # weights without offsets
    assert lib.wca_normalize_heads(p(x), p(sel), p(d), 1, 0, 4, None, None, p(x), s) == -1
    assert lib.wca_normalize_heads(p(x), p(sel), p(d), -1, 4, 4, None, None, p(x), s) == -1
    assert lib.wca_normalize_heads(p(x), p(sel), p(d), 1, 449, 4, None, None, p(x), s) == -2  # beyond Whisper's context
    assert lib.wca_normalize_heads(p(x), p(sel), p(d), 0, 4, 4, None, None, p(x), s) == 0
    with pytest.raises(_cabi.WcaError):
        _cabi.normalize_heads(p(x), sel, d, 1, 4, 4, x, weights=x)


# ------------------------------------------------------------------ batch invariance
def _dtw_times(matrix, recs, wb_flat, dev):
    from whisper_char_alignment_b200 import _cabi

    times = torch.full((2, int((recs["n_words"] + 1).sum()) + 8), -1.0, dtype=torch.float64, device=dev)
    max_rows, max_f = int((recs["row_end"] - recs["row_begin"]).max()), int(recs["n_frames"].max())
    nbytes = _cabi.dtw_workspace_bytes(len(recs), max_rows, max_f)
    _cabi.dtw_align(matrix.data_ptr(), _cabi.upload_utts(recs, dev), len(recs), max_rows, max_f, True,
                    word_bounds=torch.from_numpy(wb_flat).to(dev), start_times=times[0], end_times=times[1],
                    trace_ws=torch.empty(nbytes, dtype=torch.uint8, device=dev) if nbytes else None)
    return times.cpu().numpy()


def test_an_utterance_alone_equals_the_same_utterance_in_a_batch(dev):
    """Weights, matrix and DTW times of every utterance are bit-identical whether it is launched alone or inside the
    ragged batch of the fp64 test (larger max_tokens / max_frames, other lists)."""
    recs, maps, sels, ws, d_sel, n_mx, w_off, n_w = _batch(dev)
    rng = np.random.default_rng(5)
    n_rows = recs["row_end"] - recs["row_begin"]
    recs["n_words"] = np.minimum(n_rows, 3)
    recs["word_off"] = np.concatenate([[0], np.cumsum(recs["n_words"] + 1)[:-1]])
    wb = [np.sort(rng.choice(n, size=w + 1, replace=n < w + 1)).astype(np.int32) for n, w in zip(n_rows, recs["n_words"])]
    wb_flat = np.concatenate(wb)
    # finite matrices (but for T = 1) for the DTW: column 0 is no longer constant over the tokens
    for m in maps:
        if m.shape[1] > 1:
            m[:, 0, 0] += 0.25
    ws = pack_maps(maps, recs, dev)
    got_m, got_w = _run(recs, ws, d_sel, n_mx, w_off, n_w, dev)
    mx = Guarded(n_mx, torch.float32, dev)
    mx.out.copy_(torch.from_numpy(got_m))
    times = _dtw_times(mx.out, recs, wb_flat, dev)
    for b, r in enumerate(recs):
        one = recs[b:b + 1].copy()
        one["word_off"] = 0
        alone_m, alone_w = _run(one, ws, d_sel, n_mx, w_off[b:b + 1], n_w, dev)  # offsets by position in the launch
        k, T, F = int(r["n_sel"]), int(r["n_tokens"]), int(r["n_frames"])
        sw = slice(int(w_off[b]), int(w_off[b]) + k * T * F)
        sm = slice(int(r["matrix_off"]), int(r["matrix_off"]) + int(n_rows[b]) * F)
        np.testing.assert_array_equal(alone_w[sw].view(np.int32), got_w[sw].view(np.int32), err_msg=f"weights {b}")
        np.testing.assert_array_equal(alone_m[sm].view(np.int32), got_m[sm].view(np.int32), err_msg=f"matrix {b}")
        mx.out.copy_(torch.from_numpy(alone_m))
        t1 = _dtw_times(mx.out, one, wb[b], dev)
        wo, W = int(r["word_off"]), int(r["n_words"])
        np.testing.assert_array_equal(t1[:, :W], times[:, wo:wo + W], err_msg=f"times {b}")


# ------------------------------------------------------------------ through default_find_alignment_batch
def _spy_maps(monkeypatch, timing):
    """Keeps the maps default_find_alignment_batch captures (to check its normaliser against fp64 on them)."""
    seen = {}
    orig = timing.get_attentions_batch

    def spy(*a, **k):
        out = orig(*a, **k)
        seen["maps"] = out[0]
        return out

    monkeypatch.setattr(timing, "get_attentions_batch", spy)
    return seen


def _synthetic_inputs(tokenizer, n, n_mels, mel_len, n_ctx, seed):
    from oracle.synth import make_mel
    from whisper_char_alignment_b200.retokenize import encode
    from whisper_char_alignment_b200.synthetic import _sentence

    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        frames = int(rng.integers(20, n_ctx + 1))
        text = _sentence(rng, int(rng.integers(5, 40)))
        out.append((encode(text, tokenizer, "subword"), make_mel(n_mels, mel_len, 2 * frames, seed + i), frames))
    return out


@pytest.mark.parametrize("name", default_timing_names())
def test_reference_fixture_inside_a_batch(name, tokenizer, oracle_models, dev, monkeypatch):
    """The reference's own default_find_alignment output (fixture) for one utterance batched with seeded synthetic ones
    of the same model: words equal, times equal to the frame, weights within the fixture test's bounds; the weights
    against float64 std_mean of the product's own captured maps (the normaliser's error apart from the capture's).
    The batch costs the capture's launches plus exactly one normalisation and one DTW launch."""
    from test_gpu_parity import product_model
    from whisper_char_alignment_b200 import _cabi, timing

    g = load_golden(name)
    c = g["case"]
    model = product_model(oracle_models(c["model"]), dev)
    n_ctx = model.dims.n_audio_ctx
    extra = _synthetic_inputs(tokenizer, 5, g["mel"].shape[0], g["mel"].shape[1], n_ctx, seed=len(name))
    texts = [t for t, _, _ in extra[:2]] + [g["text_tokens"].tolist()] + [t for t, _, _ in extra[2:]]
    mels = [m for _, m, _ in extra[:2]] + [torch.from_numpy(g["mel"])] + [m for _, m, _ in extra[2:]]
    frames = [f for _, _, f in extra[:2]] + [c["frames"]] + [f for _, _, f in extra[2:]]
    mels = torch.stack(mels).to(dev)
    seen = _spy_maps(monkeypatch, timing)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        before = _cabi.launch_count()
        outs = timing.default_find_alignment_batch(model, tokenizer, texts, mels, frames, medfilt_width=c["width"],
                                                   qk_scale=c["qk_scale"])
        launched = _cabi.launch_count() - before
        tokens = [torch.tensor([*tokenizer.sot_sequence, tokenizer.no_timestamps, *t, tokenizer.eot], device=dev)
                  for t in texts]
        before = _cabi.launch_count()
        timing.get_attentions_batch(mels, tokens, model, tokenizer, frames, c["width"], c["qk_scale"])
        capture_only = _cabi.launch_count() - before
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert launched == capture_only + 2, (launched, capture_only)
    words, st, en, weights, none = outs[2]
    assert none is None and words == g["words"]
    np.testing.assert_array_equal(np.round(st * 50).astype(int), np.round(g["start_times"] * 50).astype(int))
    np.testing.assert_array_equal(np.round(en * 50).astype(int), np.round(g["end_times"] * 50).astype(int))
    gold = torch.from_numpy(g["weights"])
    torch.testing.assert_close(weights.cpu(), gold, rtol=2e-3, atol=2e-4)
    vs_ref = float(((weights.cpu().double() - gold.double()).abs() / (gold.double().abs() + 0.1)).max())
    print(f"{name}: weights vs the reference's fp32 weights: max |diff| / (|w| + 0.1) = {vs_ref:.3e}")
    record_measure(f"default_timing_{name}_weights_vs_reference_err", vs_ref)

    picked = model.alignment_heads.indices().T.cpu()
    sel = (picked[:, 0] * model.dims.n_text_head + picked[:, 1]).numpy()
    worst = 0.0
    for b, (maps, out) in enumerate(zip(seen["maps"], outs)):
        if isinstance(out, list):
            continue
        w64, _, scale = ref_normalize(maps.flatten(0, 1), sel, 0, 1)
        got = out[3].cpu().numpy()
        w64, scale = w64.cpu().numpy(), np.broadcast_to(scale.cpu().numpy(), w64.shape)
        np.testing.assert_array_equal(np.isnan(got), np.isnan(w64))
        worst = max(worst, _err_units(got, w64, scale))
    assert worst <= NORM_K, worst
    record_measure("default_timing_fixture_batch_weights_vs_fp64_err_in_eps_cond", worst)


def test_medium_timit_batch_dtw_bit_exact(tokenizer, dev, monkeypatch):
    """Whisper-medium dims (random init, qk_gain 4), TIMIT-shaped batch of 32: the times are those of the C oracle's DTW
    on the kernel's own matrix, bit for bit.  Reported, not asserted: the share of word boundaries that agree with
    those of a float64-normalised matrix."""
    from oracle import dtw as odtw
    from whisper_char_alignment_b200 import _cabi, timing
    from whisper_char_alignment_b200.retokenize import split_tokens_on_spaces
    from whisper_char_alignment_b200.synthetic import timit_shaped
    from whisper_char_alignment_b200.whisper_model import load_model

    model = load_model("random:medium", dev, qk_gain=4.0)
    utts = timit_shaped(32, tokenizer, n_mels=model.dims.n_mels, seed=3)
    seen = _spy_maps(monkeypatch, timing)
    outs = timing.default_find_alignment_batch(model, tokenizer, [u.text_tokens for u in utts],
                                               torch.stack([u.mel for u in utts]).to(dev), [u.max_frames for u in utts])
    maps = seen["maps"]
    picked = model.alignment_heads.indices().T
    sel = (picked[:, 0] * model.dims.n_text_head + picked[:, 1]).to(torch.int32)
    sot = len(tokenizer.sot_sequence)
    plan = timing._Plan(maps, sot, [len(sel)] * len(maps), shared_sel=True)
    matrix = torch.empty(plan.totals["matrix"], dtype=torch.float32, device=dev)
    _cabi.normalize_heads(plan.base_ptr, sel, plan.d_utts, plan.B, plan.max_tokens, plan.max_frames, matrix)
    matrix = matrix.cpu().numpy()
    agree = total = 0
    for b, (u, out) in enumerate(zip(utts, outs)):
        r = plan.recs[b]
        n, F = int(r["row_end"] - r["row_begin"]), int(r["n_frames"])
        m = matrix[int(r["matrix_off"]): int(r["matrix_off"]) + n * F].reshape(n, F)
        _, word_tokens = split_tokens_on_spaces(list(u.text_tokens) + [tokenizer.eot], tokenizer, "subword")
        wb = np.pad(np.cumsum([len(t) for t in word_tokens[:-1]]), (1, 0))
        jumps = odtw.jump_frames(*odtw.dtw_path(-m))
        np.testing.assert_array_equal(out[2], jumps[wb[1:]] / 50.0, err_msg=f"end times, utterance {b}")
        np.testing.assert_array_equal(out[1], jumps[wb[:-1]] / 50.0, err_msg=f"start times, utterance {b}")
        _, m64, _ = ref_normalize(maps[b].flatten(0, 1), sel.cpu().numpy(), sot, int(r["row_end"]))
        j64 = odtw.jump_frames(*odtw.dtw_path(-m64.float().cpu().numpy()))
        agree += int((j64[wb[1:]] == jumps[wb[1:]]).sum())
        total += len(wb) - 1
    print(f"medium TIMIT batch of 32: {agree}/{total} end boundaries agree with the float64-normalised matrix's")
    record_measure("default_timing_medium_timit_boundary_agreement_with_fp64", agree / total)


def test_cli_default_timing_equals_per_utterance_calls(tmp_path, tokenizer, dev):
    """infer_ali --default_whisper_timing (one default_find_alignment_batch call per planned batch) predicts, per
    utterance, the end times of default_find_alignment called on that utterance alone."""
    import joblib

    from whisper_char_alignment_b200 import timing
    from whisper_char_alignment_b200.cli import common, infer_ali
    from whisper_char_alignment_b200.dataset import DATASET

    out = tmp_path / "run"
    infer_ali.main(["--model", "random:micro", "--dataset", "synthetic", "--scp", "timit:6", "--output_dir", str(out),
                    "--default_whisper_timing", "--save_prediction", "--batch_size", "4", "--tolerance", "0.5"])
    preds = joblib.load(glob.glob(os.path.join(str(out), "*-predictions.pkl"))[0])
    model, tk, whisper_pkg, _ = common.load_model_and_tokenizer("random:micro", dev)
    dataset = DATASET["synthetic"]("timit:6", n_mels=80, device=dev)
    assert len(preds) == len(dataset)
    for n in range(len(dataset)):
        it = common.prepare(dataset[n], tk, "subword", dev, whisper_pkg, model)
        one = timing.default_find_alignment(model, tk, it["text_tokens"], it["mel"], it["max_frames"])
        np.testing.assert_array_equal(preds[n]["ends_hat"], one[2], err_msg=f"utterance {n}")
        np.testing.assert_array_equal(preds[n]["starts_hat"], one[1], err_msg=f"utterance {n}")
