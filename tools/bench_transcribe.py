"""Throughput of transcribe-then-align (`WCA_TRANSCRIBE=greedy`): two arms in the same process, alternating, after
warm-up, median of the repetitions.

  (a) what the CLI did before the cached decoder: greedy_decode one utterance at a time (the whole prefix re-run, and
      every layer's cross-attention K/V re-projected, at every step), then the batched alignment
      (get_attentions_batch + force_align_batch) with its own encoder pass;
  (b) one embed_audio per batch, greedy_decode_cached on it, then the same alignment on that encoder output
      (audio_features=...).

Plus wca_decode_attention alone from CUDA events over many launches at the cross-attention shape (n_kv = 1500) and the
self-attention shape (n_kv = 448) of Whisper-medium, on the bytes the algorithm reads (K and V once, 4 B H n_kv 128,
plus q and out), against the 6548.5 GB/s HBM copy bandwidth of BASELINE.md.  The launches cycle over several layers'
K/V whose sum exceeds the 126 MB L2, so the figures are HBM reads, not L2 hits.

    python tools/bench_transcribe.py [--reps 3] [--timit 32 --timit_tokens 32] [--librispeech 16 --librispeech_tokens 128]

Whisper-medium dimensions, seeded random weights (qk_gain 4), synthetic TIMIT- and LibriSpeech-shaped utterances.
Random weights rarely emit EOT, so every transcript runs to the fixed token budget; the arms align the decoded token ids
directly.  Needs a CUDA device; prints the card's name and power limit with the figures."""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tools.bench_default_timing import COPY_PEAK_GBS, card, timed  # noqa: E402


def align(model, tk, texts, mels, frames, features=None):
    from whisper_char_alignment_b200 import timing

    dev = mels.device if features is None else features.device
    tokens = [torch.tensor([*tk.sot_sequence, tk.no_timestamps, *t, tk.eot], device=dev) for t in texts]
    maps, _ = timing.get_attentions_batch(None if features is not None else mels, tokens, model, tk, frames,
                                          audio_features=features)
    return timing.force_align_batch(maps, texts, tk, "subword", return_matrix=False)


def arm_loop(model, tk, mels, frames, max_tokens):
    from whisper_char_alignment_b200.whisper_model import greedy_decode

    texts = [greedy_decode(model, m, tk, max_tokens) for m in mels]
    return texts, align(model, tk, texts, mels, frames)


def arm_cached(model, tk, mels, frames, max_tokens):
    from whisper_char_alignment_b200.whisper_model import greedy_decode_cached

    with torch.no_grad():
        xa = model.embed_audio(mels)
    texts = greedy_decode_cached(model, xa, tk, max_tokens)
    return texts, align(model, tk, texts, mels, frames, xa)


def kernel_rate(B, H, n_kv, n_layers, ld, iters, dev):
    """wca_decode_attention over n_layers distinct (B, n_kv, ld) K/V buffers read as column slices (K at column 0, V
    at column H*64), one layer per launch in turn: mean time per launch and GB/s on the algorithmic bytes."""
    from whisper_char_alignment_b200 import _cabi

    W = 64 * H
    kv = [torch.randn(B, n_kv, ld, device=dev) for _ in range(n_layers)]
    q = torch.randn(B, W, device=dev)
    out = torch.empty(B, W, device=dev)
    ws = torch.empty(_cabi.decode_attention_workspace_bytes(B, H, n_kv), dtype=torch.uint8, device=dev)

    def launch(i):
        t = kv[i % n_layers]
        _cabi.decode_attention(q, t[..., :W], t[..., W:2 * W], H, out=out, workspace=ws)

    for i in range(2 * n_layers):
        launch(i)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        launch(i)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / iters
    nbytes = 4 * B * H * n_kv * 128 + 4 * 2 * B * W
    kv_mb = sum(t.numel() for t in kv) * 4 / 1e6
    return dict(B=B, H=H, n_kv=n_kv, kernel_ms=ms, algorithmic_bytes=nbytes, gbs=nbytes / ms / 1e6,
                share_of_copy_peak=nbytes / ms / 1e6 / COPY_PEAK_GBS,
                l2_note=f"cycles over {n_layers} layers' K/V buffers, {kv_mb:.0f} MB in all (> 126 MB L2)")


def main(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--timit", type=int, default=32, help="TIMIT-shaped batch size")
    p.add_argument("--timit_tokens", type=int, default=32, help="max_tokens of the TIMIT-shaped batch")
    p.add_argument("--librispeech", type=int, default=16, help="LibriSpeech-shaped batch size")
    p.add_argument("--librispeech_tokens", type=int, default=128, help="max_tokens of the LibriSpeech-shaped batch")
    p.add_argument("--kernel_iters", type=int, default=200)
    p.add_argument("--out", default=None)
    args = p.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_transcribe: needs a CUDA device (no figure is measured without one)")

    from whisper_char_alignment_b200.synthetic import librispeech_shaped, timit_shaped
    from whisper_char_alignment_b200.tokenizer import get_tokenizer
    from whisper_char_alignment_b200.whisper_model import load_model

    dev = torch.device("cuda:0")
    torch.backends.cudnn.allow_tf32 = False
    model = load_model("random:medium", dev, qk_gain=4.0)
    tk = get_tokenizer(True, language="English")
    name, limit = card()
    report = dict(card=name, power_limit=limit, model="random:medium (qk_gain 4)", workloads={}, kernel={})
    d, H = model.dims.n_text_state, model.dims.n_text_head
    # cross: one layer's K/V slice of the 4-layer cross_kv GEMM output (row pitch 2 * 4 * d); self: the step cache
    # (row pitch 2d), 8 layers
    for label, n_kv, layers, ld in (("cross", model.dims.n_audio_ctx, 4, 8 * d), ("self", model.dims.n_text_ctx, 8, 2 * d)):
        k = kernel_rate(args.timit, H, n_kv, layers, ld, args.kernel_iters, dev)
        report["kernel"][label] = k
        print(f"wca_decode_attention {label} (B {k['B']}, H {H}, n_kv {n_kv}): {k['kernel_ms'] * 1e3:.1f} us, "
              f"{k['gbs']:.0f} GB/s = {100 * k['share_of_copy_peak']:.1f} % of {COPY_PEAK_GBS} GB/s; {k['l2_note']}",
              flush=True)
        torch.cuda.empty_cache()
    for label, make, n, max_tokens in (("timit", timit_shaped, args.timit, args.timit_tokens),
                                       ("librispeech", librispeech_shaped, args.librispeech, args.librispeech_tokens)):
        utts = make(n, tk, n_mels=model.dims.n_mels, seed=1)
        mels = torch.stack([u.mel for u in utts]).to(dev)
        frames = [u.max_frames for u in utts]
        timed(lambda: arm_cached(model, tk, mels, frames, max_tokens))
        timed(lambda: arm_loop(model, tk, mels, frames, max_tokens))  # warm-up of every shape
        ta, tb = [], []
        for _ in range(args.reps):
            s, (texts_a, outs_a) = timed(lambda: arm_loop(model, tk, mels, frames, max_tokens))
            ta.append(s)
            s, (texts_b, outs_b) = timed(lambda: arm_cached(model, tk, mels, frames, max_tokens))
            tb.append(s)
        same_text = sum(int(a == b) for a, b in zip(texts_a, texts_b))
        same_ends = sum(int(a == b and np.array_equal(oa[2], ob[2]))
                        for a, b, oa, ob in zip(texts_a, texts_b, outs_a, outs_b))
        w = dict(utterances=n, max_tokens=max_tokens, loop_utt_per_s=n / float(np.median(ta)),
                 cached_utt_per_s=n / float(np.median(tb)), loop_s=sorted(ta), cached_s=sorted(tb),
                 speedup=float(np.median(ta) / np.median(tb)), same_transcripts=f"{same_text}/{n}",
                 same_transcripts_and_end_times=f"{same_ends}/{n}",
                 mean_tokens=float(np.mean([len(t) for t in texts_b])))
        report["workloads"][label] = w
        print(f"{label} (batch {n}, max_tokens {max_tokens}): per-utterance greedy_decode + alignment "
              f"{w['loop_utt_per_s']:.2f} utt/s, cached batch {w['cached_utt_per_s']:.2f} utt/s (x{w['speedup']:.1f}); "
              f"transcripts equal on {w['same_transcripts']}, transcripts and end times on "
              f"{w['same_transcripts_and_end_times']}", flush=True)
    print(f"card: {name}, power limit {limit}")
    print(json.dumps(report))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
