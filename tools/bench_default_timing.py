"""Throughput of the stock-Whisper baseline (`infer_ali.py --default_whisper_timing`): the batched
timing.default_find_alignment_batch against the per-utterance loop it replaced (one batch-1 forward + capture, torch-op
std-normalisation of the alignment heads, force_align(..., "grad_norm") per utterance), both in the same process,
alternating, after warm-up; plus the time of wca_normalize_heads alone from CUDA events and its rate on the bytes the
algorithm needs (one read of the k selected maps, one write of the k normalised maps and of the (N, F) matrix) against
the 6548.5 GB/s HBM copy bandwidth of BASELINE.md.

    python tools/bench_default_timing.py [--reps 5] [--timit 32] [--librispeech 16] [--out bench_default_timing.json]

Whisper-medium dimensions, seeded random weights (qk_gain 4), synthetic TIMIT- and LibriSpeech-shaped utterances.
Needs a CUDA device; prints the card's name and power limit with the figures."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

COPY_PEAK_GBS = 6548.5  # HBM copy bandwidth (read + write) measured on a B200, BASELINE.md section 2


def per_utterance_loop(model, tokenizer, items):
    """The baseline as it ran before the batched path: one utterance at a time, normalisation in torch ops."""
    from whisper_char_alignment_b200 import timing

    outs = []
    for text_tokens, mel, max_frames in items:
        device = mel.device
        tokens = torch.tensor([*tokenizer.sot_sequence, tokenizer.no_timestamps, *text_tokens, tokenizer.eot], device=device)
        maps, _ = timing.get_attentions(mel, tokens, model, tokenizer, max_frames)
        n_heads = maps.shape[1]
        picked = model.alignment_heads.indices().T.to(device)
        weights = maps.flatten(0, 1).index_select(0, picked[:, 0] * n_heads + picked[:, 1])
        std, mean = torch.std_mean(weights, dim=-2, keepdim=True, unbiased=False)
        weights = (weights - mean) / std
        outs.append(timing.force_align(weights.mean(dim=0), list(text_tokens), tokenizer, "subword", "grad_norm"))
    return outs


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def kernel_rate(model, tokenizer, items, iters):
    """wca_normalize_heads on the batch's captured maps: mean time over `iters` launches (CUDA events) and GB/s."""
    from whisper_char_alignment_b200 import _cabi, timing

    dev = items[0][1].device
    tokens = [torch.tensor([*tokenizer.sot_sequence, tokenizer.no_timestamps, *t, tokenizer.eot], device=dev)
              for t, _, _ in items]
    maps, _ = timing.get_attentions_batch(torch.stack([m for _, m, _ in items]), tokens, model, tokenizer,
                                          [f for _, _, f in items])
    picked = model.alignment_heads.indices().T
    sel = (picked[:, 0] * model.dims.n_text_head + picked[:, 1]).to(device=dev, dtype=torch.int32)
    k = len(sel)
    plan = timing._Plan(maps, len(tokenizer.sot_sequence), [k] * len(maps), shared_sel=True)
    T, F = plan.recs["n_tokens"].astype(np.int64), plan.recs["n_frames"].astype(np.int64)
    sizes = k * T * F
    w_off = torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)).to(dev)
    weights = torch.empty(int(sizes.sum()), dtype=torch.float32, device=dev)
    matrix = torch.empty(plan.totals["matrix"], dtype=torch.float32, device=dev)

    def launch():
        _cabi.normalize_heads(plan.base_ptr, sel, plan.d_utts, plan.B, plan.max_tokens, plan.max_frames, matrix, weights,
                              w_off)

    for _ in range(3):
        launch()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        launch()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / iters
    nbytes = 4 * (2 * int(sizes.sum()) + plan.totals["matrix"])
    return dict(kernel_ms=ms, algorithmic_bytes=nbytes, gbs=nbytes / ms / 1e6, share_of_copy_peak=nbytes / ms / 1e6 / COPY_PEAK_GBS,
                heads=k, utterances=len(items), max_tokens=plan.max_tokens, max_frames=plan.max_frames,
                l2_note="the maps of the batch (read by the capture just before) may partly sit in the 126 MB L2")


def main(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--reps", type=int, default=5)
    p.add_argument("--timit", type=int, default=32, help="TIMIT-shaped batch size")
    p.add_argument("--librispeech", type=int, default=16, help="LibriSpeech-shaped batch size")
    p.add_argument("--kernel_iters", type=int, default=50)
    p.add_argument("--out", default=None)
    args = p.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_default_timing: needs a CUDA device (no figure is measured without one)")

    from whisper_char_alignment_b200 import timing
    from whisper_char_alignment_b200.synthetic import librispeech_shaped, timit_shaped
    from whisper_char_alignment_b200.tokenizer import get_tokenizer
    from whisper_char_alignment_b200.whisper_model import load_model

    dev = torch.device("cuda:0")
    torch.backends.cudnn.allow_tf32 = False
    model = load_model("random:medium", dev, qk_gain=4.0)
    tk = get_tokenizer(True, language="English")
    name, limit = card()
    report = dict(card=name, power_limit=limit, model="random:medium (qk_gain 4)", workloads={})
    for label, make, n in (("timit", timit_shaped, args.timit), ("librispeech", librispeech_shaped, args.librispeech)):
        utts = make(n, tk, n_mels=model.dims.n_mels, seed=1)
        items = [(u.text_tokens, u.mel.to(dev), u.max_frames) for u in utts]
        mels = torch.stack([m for _, m, _ in items])

        def batched():
            return timing.default_find_alignment_batch(model, tk, [t for t, _, _ in items], mels, [f for _, _, f in items])

        def loop():
            return per_utterance_loop(model, tk, items)

        timed(batched)
        timed(loop)  # warm-up of every shape
        tb, tl = [], []
        for _ in range(args.reps):
            s, ob = timed(batched)
            tb.append(s)
            s, ol = timed(loop)
            tl.append(s)
        same = sum(int(np.array_equal(a[2], b[2])) for a, b in zip(ob, ol) if not isinstance(a, list))
        w = dict(utterances=n, batched_utt_per_s=n / float(np.median(tb)), loop_utt_per_s=n / float(np.median(tl)),
                 batched_s=sorted(tb), loop_s=sorted(tl), speedup=float(np.median(tl) / np.median(tb)),
                 same_end_times=f"{same}/{sum(not isinstance(a, list) for a in ob)}",
                 normalize_heads=kernel_rate(model, tk, items, args.kernel_iters))
        report["workloads"][label] = w
        print(f"{label}: batched {w['batched_utt_per_s']:.1f} utt/s, per-utterance loop {w['loop_utt_per_s']:.1f} utt/s "
              f"(x{w['speedup']:.1f}); wca_normalize_heads {w['normalize_heads']['kernel_ms']:.4f} ms, "
              f"{w['normalize_heads']['gbs']:.0f} GB/s = {100 * w['normalize_heads']['share_of_copy_peak']:.1f} % of "
              f"{COPY_PEAK_GBS} GB/s; end times equal to the loop's on {w['same_end_times']} utterances", flush=True)
    print(f"card: {name}, power limit {limit}")
    print(json.dumps(report))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
