"""GPU suite: the KV-cached greedy decoder -- wca_decode_attention (csrc/decode_attn.cu) through the C ABI, the cached
decode step of whisper_model against the full decoder, greedy_decode_cached against greedy_decode and the HF greedy loop,
the reuse of the encoder output by timing.get_attentions_batch, and the greedy CLI path.

Bars: the kernel against float64 softmax(q k^T / 8) v on the same fp32 inputs within DECODE_BAR * max_j |v_j| per
(row, head); a cached step's logits within STEP_BAR * max |logit| of the last row of the full decoder on the same
prefix.  A transcript may leave the reference's only at a step whose top-2 margin there is below that logit bar."""
import ctypes
import glob
import os

import numpy as np
import pytest
import torch

from conftest import record_measure
from test_gpu_scoring import Guarded, spans

pytestmark = pytest.mark.gpu

DECODE_BAR = 3e-6
STEP_BAR = 1e-4
POISON = (float("nan"), float("inf"), float("-inf"), 1e30, -1e30)


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


# ------------------------------------------------------------------ kernel against float64
def _poisoned(n, dev):
    return torch.tensor(POISON, dtype=torch.float32, device=dev).repeat(n // len(POISON) + 1)[:n].contiguous()


def _inputs(kind, B, H, n_kv, gen, dev):
    """(q (B, H, 64), k, v (B, n_kv, H, 64)) fp32 of one value regime:
    normal    logits ~ N(0, 4);
    large     integer logits of magnitude ~100 (q integers, k multiples of 8: every dot product is exact in fp32);
    dominant  normal, plus one key per (row, head) 60 above the rest;
    constant  normal logits over a V that is the same for every key."""
    def randn(*shape):
        return torch.randn(*shape, generator=gen, device=dev)

    if kind == "large":
        q = torch.randint(-6, 7, (B, H, 64), generator=gen, device=dev).float()
        k = 8 * torch.randint(-6, 7, (B, n_kv, H, 64), generator=gen, device=dev).float()
    else:
        q, k = 2 * randn(B, H, 64), randn(B, n_kv, H, 64)
    v = randn(B, n_kv, H, 64)
    if kind == "dominant":
        j = torch.randint(0, n_kv, (B, H), generator=gen, device=dev)
        boost = q * (8 * 60.0 / (q * q).sum(-1, keepdim=True))
        idx = j[:, None, :, None].expand(B, 1, H, 64)
        k.scatter_(1, idx, k.gather(1, idx) + boost[:, None])
    if kind == "constant":
        v = v[:, :1].expand(B, n_kv, H, 64).contiguous()
    return q, k, v


def _reference(q, k, v):
    s = torch.einsum("bhd,bjhd->bhj", q.double(), k.double()) / 8
    ref = torch.einsum("bhj,bjhd->bhd", s.softmax(-1), v.double())
    return ref, v.double().abs().amax(dim=(1, 3))


class _Layout:
    """q, k, v placed as column slices of wider buffers with batch strides that are not a multiple of the rows, every
    element around them (and every row at or past n_kv) poisoned.  shared=True: K and V side by side in one
    (B, rows, ld) buffer, as in the decoder's self-attention cache; False: two buffers of different pitches."""

    def __init__(self, q, k, v, shared, dev):
        B, n_kv, H, _ = k.shape
        W = 64 * H
        rows = n_kv + 3
        self.ld_q, q_off = W + 12, 8
        self.qbuf = _poisoned(B * self.ld_q + 16, dev)
        self.q = self.qbuf[q_off:q_off + B * self.ld_q].view(B, self.ld_q)[:, :W]
        self.q.copy_(q.reshape(B, W))
        if shared:
            ld = 2 * W + 8
            bs = rows * ld + 4
            self.kvbuf = [_poisoned(B * bs + 16, dev)]
            base = self.kvbuf[0][4:4 + B * bs].view(B, bs)[:, :rows * ld].view(B, rows, ld)
            self.k, self.v = base[:, :n_kv, :W], base[:, :n_kv, W + 4:2 * W + 4]
        else:
            ld_k, ld_v = W + 4, 3 * W
            bs_k, bs_v = rows * ld_k + 8, rows * ld_v + 20
            self.kvbuf = [_poisoned(B * bs_k + 16, dev), _poisoned(B * bs_v + 16, dev)]
            self.k = self.kvbuf[0][8:8 + B * bs_k].view(B, bs_k)[:, :rows * ld_k].view(B, rows, ld_k)[:, :n_kv, :W]
            self.v = self.kvbuf[1][12:12 + B * bs_v].view(B, bs_v)[:, :rows * ld_v].view(B, rows, ld_v)[:, :n_kv, W:2 * W]
        self.k.copy_(k.reshape(B, n_kv, W))
        self.v.copy_(v.reshape(B, n_kv, W))


def _launch(lay, H, dev, ld_out=None):
    """wca_decode_attention on a layout; the output rows between guard zones (checked fully written), the workspace
    exactly as large as the query returns, inside its own guards.  Returns (B, H*64) on the host."""
    from test_gpu_scoring import G, SENTINEL

    from whisper_char_alignment_b200 import _cabi

    B, n_kv, W = lay.k.shape
    ld_out = W + 8 if ld_out is None else ld_out
    out = Guarded(B * ld_out, torch.float32, dev)
    need = _cabi.decode_attention_workspace_bytes(B, H, n_kv)
    assert need > 0 and need % 16 == 0
    ws = torch.full((need // 4 + 2 * G,), 0, dtype=torch.int32, device=dev)
    ws.fill_(SENTINEL)
    _cabi.decode_attention(lay.q, lay.k, lay.v, H, out=out.out.view(B, ld_out)[:, :W],
                           workspace=ws[G:G + need // 4].view(torch.uint8))
    guards = torch.cat([ws[:G], ws[G + need // 4:]]).cpu().numpy()
    assert (guards == SENTINEL).all(), "the kernel wrote outside its workspace"
    got = out.check(spans(B * ld_out, np.arange(B) * ld_out, [W] * B))
    return got.reshape(B, ld_out)[:, :W]


N_KV = [1, 2, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 447, 448, 1499, 1500]
KINDS = ["normal", "large", "dominant", "constant"]
BATCHES = [1, 33, 7, 16, 2, 5]


@pytest.mark.parametrize("n_kv", N_KV)
def test_decode_attention_vs_fp64(n_kv, dev):
    gen = torch.Generator(device=dev).manual_seed(1000 + n_kv)
    worst = 0.0
    for i, H in enumerate((1, 6, 16, 20)):
        for j, kind in enumerate(KINDS):
            B = BATCHES[(i + j + N_KV.index(n_kv)) % len(BATCHES)]
            q, k, v = _inputs(kind, B, H, n_kv, gen, dev)
            got = _launch(_Layout(q, k, v, shared=(i + j) % 2 == 0, dev=dev), H, dev)
            ref, vmax = _reference(q, k, v)
            got = torch.from_numpy(np.ascontiguousarray(got)).to(dev).double().view(B, H, 64)
            assert torch.isfinite(got).all(), (kind, B, H)
            err = float(((got - ref).abs().amax(-1) / vmax).max())
            assert err <= DECODE_BAR, (kind, B, H, err)
            worst = max(worst, err)
    print(f"n_kv={n_kv}: max |out - ref| / max_j |v_j| = {worst:.3e}")
    record_measure("decode_attention_vs_fp64_err_over_vmax", worst)


def test_decode_attention_batch_invariant_and_repeatable(dev):
    """A row alone and the same row at several places of batches of several sizes: the same bits; two launches of
    the same batch: the same bits."""
    gen = torch.Generator(device=dev).manual_seed(7)
    H = 16
    for n_kv in (65, 448, 1500):
        q, k, v = _inputs("normal", 33, H, n_kv, gen, dev)
        full = _launch(_Layout(q, k, v, True, dev), H, dev)
        assert np.array_equal(full.view(np.int32), _launch(_Layout(q, k, v, True, dev), H, dev).view(np.int32))
        for row in (0, 5, 32):
            alone = _launch(_Layout(q[row:row + 1], k[row:row + 1], v[row:row + 1], False, dev), H, dev)
            assert np.array_equal(alone[0].view(np.int32), full[row].view(np.int32)), (n_kv, row)
            for B in (2, 9):
                lo = max(0, row - B + 1)
                part = _launch(_Layout(q[lo:lo + B], k[lo:lo + B], v[lo:lo + B], False, dev), H, dev)
                assert np.array_equal(part[row - lo].view(np.int32), full[row].view(np.int32)), (n_kv, row, B)


def test_decode_attention_rejects_bad_arguments(dev):
    """Host-side checks: each returns its status with a message naming the entry point, and launches nothing."""
    from whisper_char_alignment_b200 import _cabi

    lib = _cabi.load()
    B, H, n_kv = 2, 4, 10
    W = 64 * H
    buf = torch.zeros(1 << 20, dtype=torch.float32, device=dev)  # q, k, v, out 64 KB apart
    p = buf.data_ptr()
    need = _cabi.decode_attention_workspace_bytes(B, H, n_kv)
    ws_buf = torch.zeros(need, dtype=torch.uint8, device=dev)
    ws = ws_buf.data_ptr()
    good = dict(q=p, k=p + (1 << 16), v=p + (2 << 16), out=p + (3 << 16), n_batch=B, n_kv=n_kv, n_heads=H, head_dim=64, ld_q=W, ld_k=W,
                ld_v=W, ld_out=W, bs_k=n_kv * W, bs_v=n_kv * W, ws=ws, ws_bytes=need)

    def call(**over):
        a = {**good, **over}
        return lib.wca_decode_attention(a["q"], a["k"], a["v"], a["out"], a["n_batch"], a["n_kv"], a["n_heads"],
                                        a["head_dim"], a["ld_q"], a["ld_k"], a["ld_v"], a["ld_out"], a["bs_k"], a["bs_v"],
                                        a["ws"], a["ws_bytes"], ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))

    cases = [
        (dict(head_dim=32), -2), (dict(head_dim=128), -2),
        (dict(q=None), -1), (dict(k=None), -1), (dict(v=None), -1), (dict(out=None), -1), (dict(ws=None), -1),
        (dict(n_batch=0), -1), (dict(n_kv=0), -1), (dict(n_batch=-3), -1), (dict(n_kv=-1), -1),
        (dict(q=p + 4), -1), (dict(k=p + (1 << 16) + 4), -1), (dict(v=p + (2 << 16) + 8), -1),
        (dict(out=p + (3 << 16) + 12), -1), (dict(ws=ws + 4), -1),
        (dict(ld_q=W + 2), -1), (dict(ld_k=W + 1), -1), (dict(ld_v=W + 6), -1), (dict(ld_out=W + 3), -1),
        (dict(bs_k=n_kv * W + 2), -1), (dict(bs_v=n_kv * W + 1), -1), (dict(bs_k=-4), -1),
        (dict(ws_bytes=need - 1), -1), (dict(ws_bytes=0), -1),
    ]
    torch.cuda.synchronize()
    before = _cabi.launch_count()
    for over, status in cases:
        assert call(**over) == status, over
        assert b"wca_decode_attention" in lib.wca_last_error(), over
    assert _cabi.launch_count() == before
    assert call() == 0
    torch.cuda.synchronize()
    assert _cabi.decode_attention_workspace_bytes(0, H, n_kv) == 0 and _cabi.decode_attention_workspace_bytes(B, H, 0) == 0
    with pytest.raises(_cabi.WcaError):
        _cabi.decode_attention(torch.zeros(B, W), torch.zeros(B, n_kv, W), torch.zeros(B, n_kv, W), H)


# ------------------------------------------------------------------ cached decode step and greedy_decode_cached
def _features(model, n, seed, dev):
    from whisper_char_alignment_b200.synthetic import timit_shaped
    from whisper_char_alignment_b200.tokenizer import get_tokenizer

    utts = timit_shaped(n, get_tokenizer(True, language="English"), n_mels=model.dims.n_mels, seed=seed)
    mels = torch.stack([u.mel for u in utts]).to(dev)
    with torch.no_grad():
        return mels, model.embed_audio(mels)


_MODELS = {}


def _model(size, dev):
    from whisper_char_alignment_b200.whisper_model import load_model

    if size not in _MODELS:
        _MODELS.clear()  # one model at a time on the device
        _MODELS[size] = load_model(f"random:{size}", dev, qk_gain=4.0)
    return _MODELS[size]


@pytest.mark.parametrize("size,n_steps", [("micro", 60), ("mini", 60), ("medium", 24)])
def test_cached_step_logits_match_the_full_decoder(size, n_steps, tokenizer, dev):
    """Teacher-forced along a seeded token sequence (prefix, then text tokens), every cached step's logits against the
    last row of model.decoder over the whole prefix, on the same audio features."""
    from whisper_char_alignment_b200.whisper_model import DecodeCache

    model = _model(size, dev)
    _, xa = _features(model, 3, seed=11, dev=dev)
    rng = np.random.default_rng(5)
    prefix = [*tokenizer.sot_sequence, tokenizer.no_timestamps]
    text = rng.integers(0, tokenizer.eot, size=(3, n_steps - len(prefix)))
    tokens = torch.tensor(np.concatenate([np.tile(prefix, (3, 1)), text], axis=1), device=dev)
    cache = DecodeCache(model.decoder, xa)
    worst = 0.0
    with torch.no_grad():
        for p in range(tokens.shape[1]):
            step = model.decoder(tokens[:, p:p + 1], xa, cache=cache)[:, -1].double()
            full = model.decoder(tokens[:, :p + 1], xa)[:, -1].double()
            err = float(((step - full).abs().amax(-1) / full.abs().amax(-1)).max())
            assert err <= STEP_BAR, (p, err)
            worst = max(worst, err)
    assert cache.pos == tokens.shape[1]
    print(f"{size}: cached step logits vs full decoder, max |diff| / max |logit| = {worst:.3e}")
    record_measure(f"decode_step_vs_full_decoder_{size}_err_over_max_logit", worst)


def _margin(logits, eot):
    top = logits[: eot + 1].double().topk(2).values
    return float(top[0] - top[1]), float(logits[: eot + 1].abs().max())


def _check_transcripts(got, want, margin_at, label):
    """got == want row by row, except from a first divergence at which the reference's top-2 margin is below the
    logit bar.  margin_at(row, context tokens) -> (margin, max |logit|).  Returns the number of such divergences."""
    accepted = 0
    for row, (g, w) in enumerate(zip(got, want)):
        if g == w:
            continue
        i = next((i for i, (a, b) in enumerate(zip(g, w)) if a != b), min(len(g), len(w)))
        margin, scale = margin_at(row, w[:i])
        assert margin < STEP_BAR * scale, f"{label} row {row}: diverges at token {i} where the reference's margin is {margin}"
        accepted += 1
    return accepted


@pytest.mark.parametrize("size,max_tokens,batch", [("micro", 224, 32), ("mini", 224, 32), ("medium", 48, 16)])
def test_greedy_decode_cached_equals_greedy_decode(size, max_tokens, batch, tokenizer, dev):
    from whisper_char_alignment_b200.whisper_model import greedy_decode, greedy_decode_cached

    model = _model(size, dev)
    mels, xa = _features(model, batch, seed=21, dev=dev)
    want = greedy_decode(model, mels, tokenizer, max_tokens)
    got = greedy_decode_cached(model, xa, tokenizer, max_tokens)
    prefix = [*tokenizer.sot_sequence, tokenizer.no_timestamps]

    def margin_at(row, ctx):
        with torch.no_grad():
            logits = model.decoder(torch.tensor([prefix + ctx], device=dev), xa[row:row + 1])[0, -1]
        return _margin(logits, tokenizer.eot)

    accepted = _check_transcripts(got, want, margin_at, size)
    print(f"{size}: {batch - accepted}/{batch} transcripts identical to greedy_decode, {accepted} near-tie divergences; "
          f"lengths {sorted(len(t) for t in want)[::max(1, batch // 8)]}")
    record_measure(f"greedy_cached_{size}_near_tie_divergences", accepted)


def test_greedy_decode_cached_equals_hf_greedy(oracle_models, tokenizer, dev):
    """micro: the cached decoder on the GPU against the plain greedy loop over the HF model (CPU) with the same weights."""
    pytest.importorskip("transformers")
    from oracle import hf_crosscheck
    from test_gpu_parity import product_model
    from whisper_char_alignment_b200.whisper_model import greedy_decode_cached

    from oracle.synth import make_mel

    om = oracle_models("micro")
    hf = hf_crosscheck.hf_model_from(om)
    model = product_model(om, dev)
    n_in = 2 * om.dims.n_audio_ctx  # the oracle's micro has its own (shorter) audio context
    mels = torch.stack([make_mel(om.dims.n_mels, n_in, n_in * (i + 1) // 4, seed=31 + i) for i in range(3)]).to(dev)
    with torch.no_grad():
        xa = model.embed_audio(mels)
    prefix = [*tokenizer.sot_sequence, tokenizer.no_timestamps]
    n = 40
    got = greedy_decode_cached(model, xa, tokenizer, n)
    want = [hf_crosscheck.hf_greedy(hf, m.cpu(), prefix, tokenizer.eot, n) for m in mels]

    def margin_at(row, ctx):
        with torch.no_grad():
            enc = hf.model.encoder(input_features=mels[row:row + 1].cpu()).last_hidden_state
            dec = hf.model.decoder(input_ids=torch.tensor([prefix + ctx]), encoder_hidden_states=enc, use_cache=False)
            return _margin(hf.proj_out(dec.last_hidden_state[0, -1]), tokenizer.eot)

    accepted = _check_transcripts(got, want, margin_at, "micro vs HF")
    print(f"micro vs HF greedy: {3 - accepted}/3 identical, {accepted} near-tie divergences")
    record_measure("greedy_cached_vs_hf_near_tie_divergences", accepted)


# ------------------------------------------------------------------ encoder output reuse
@pytest.mark.parametrize("tapped", [False, True])
def test_get_attentions_with_audio_features_is_bit_identical(tapped, tokenizer, dev, monkeypatch):
    """get_attentions_batch(..., audio_features=model.embed_audio(mels)) with mels=None: the maps, the head-score
    partials the capture leaves, the scores force_align derives from them and the logits equal the mel path's bit for
    bit -- for the product model and for a module tree reached only through the forward hooks."""
    from whisper_char_alignment_b200 import timing, whisper_model
    from whisper_char_alignment_b200.synthetic import timit_shaped

    model = _model("mini", dev)
    if tapped:
        monkeypatch.setattr(whisper_model, "FUSED_PROJECTIONS", False)  # the hooks see every cross_attn.key call

        class StockLike(torch.nn.Module):  # no forward_with_cross_qk: timing taps cross_attn.query / .key
            def __init__(self, inner):
                super().__init__()
                self.dims, self.encoder, self.decoder = inner.dims, inner.encoder, inner.decoder

            def forward(self, mel, tokens):
                return self.decoder(tokens, self.encoder(mel))

        model = StockLike(model)
    utts = timit_shaped(6, tokenizer, n_mels=model.dims.n_mels, seed=41)
    mels = torch.stack([u.mel for u in utts]).to(dev)
    tokens = [u.tokens.to(dev) for u in utts]
    frames = [u.max_frames for u in utts]
    with torch.no_grad():
        xa = model.encoder(mels)
    w_mel, l_mel = timing.get_attentions_batch(mels, tokens, model, tokenizer, frames)
    w_xa, l_xa = timing.get_attentions_batch(None, tokens, model, tokenizer, frames, audio_features=xa)
    for a, b in zip(w_mel + l_mel, w_xa + l_xa):
        assert torch.equal(a, b)
    assert (timing._ScorePartials.of(w_mel[0]) is None) == (timing._ScorePartials.of(w_xa[0]) is None)
    texts = [u.text_tokens for u in utts]
    sa = timing.force_align_batch(w_mel, texts, tokenizer, "char", "topk", 10)
    sb = timing.force_align_batch(w_xa, texts, tokenizer, "char", "topk", 10)
    for a, b in zip(sa, sb):
        assert a[0] == b[0] and a[4] == b[4]
        assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]) and torch.equal(a[3], b[3])
    if not tapped:
        da = timing.default_find_alignment_batch(model, tokenizer, texts, mels, frames)
        db = timing.default_find_alignment_batch(model, tokenizer, texts, None, frames, audio_features=xa)
        for a, b in zip(da, db):
            assert np.array_equal(a[2], b[2]) and torch.equal(a[3], b[3])


# ------------------------------------------------------------------ CLI
def test_cli_greedy_equals_per_utterance_loop(tmp_path, tokenizer, dev, monkeypatch):
    """infer_ali with WCA_TRANSCRIBE=greedy (batched encoder + greedy_decode_cached per chunk, the encoder output reused
    for the alignment) predicts what a per-utterance loop predicts: greedy_decode -> remove_punctuation -> encode ->
    get_attentions -> force_align.  Words equal, times equal to the frame."""
    import joblib

    from whisper_char_alignment_b200 import timing, whisper_model
    from whisper_char_alignment_b200.cli import common, infer_ali
    from whisper_char_alignment_b200.dataset import DATASET
    from whisper_char_alignment_b200.retokenize import encode, remove_punctuation

    monkeypatch.setattr(common, "TRANSCRIBE", "greedy")
    monkeypatch.setattr(common, "DECODE_TOKENS", 12)
    out = tmp_path / "run"
    infer_ali.main(["--model", "random:micro", "--dataset", "synthetic", "--scp", "timit:6", "--output_dir", str(out),
                    "--save_prediction", "--batch_size", "4", "--tolerance", "0.5"])
    preds = joblib.load(glob.glob(os.path.join(str(out), "*-predictions.pkl"))[0])
    model, tk, _, _ = common.load_model_and_tokenizer("random:micro", dev)
    dataset = DATASET["synthetic"]("timit:6", n_mels=80, device=dev)
    assert len(preds) == len(dataset)
    for n in range(len(dataset)):
        _, mel, duration, *_ = dataset[n]
        mel = mel.to(dev)
        text = remove_punctuation(tk.decode(whisper_model.greedy_decode(model, mel, tk, 12)))
        text_tokens = encode(text, tk, "subword")
        tokens = torch.tensor([*tk.sot_sequence, tk.no_timestamps, *text_tokens, tk.eot], device=dev)
        w, _ = timing.get_attentions(mel, tokens, model, tk, int(duration) // common.AUDIO_SAMPLES_PER_TOKEN)
        words, starts, ends, _, _ = timing.force_align(w, text_tokens, tk, "subword", "mean", 15)
        assert preds[n]["predwords"] == words, n
        np.testing.assert_array_equal(np.round(preds[n]["ends_hat"] * 50), np.round(ends * 50), err_msg=f"utterance {n}")
        np.testing.assert_array_equal(np.round(preds[n]["starts_hat"] * 50), np.round(starts * 50), err_msg=f"utterance {n}")
