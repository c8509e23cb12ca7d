"""Cost of scoring a grid of alignment configurations (the measurement behind tune_alignment), one pass against one
infer_ali-style pass per configuration:

  (a) sweep: ONE forward (timing.get_attentions_widths_batch, one capture per width) and
      timing.alignment_config_counts_batch for every configuration;
  (b) per config: timing.get_attentions_batch + timing.force_align_batch with the config's settings, then
      metrics.eval_n1 (or eval_n1_strict) per utterance on the host -- what one infer_ali run per config does per batch.

Host clock around each synchronised arm.  Arms alternate after a warm-up of both, the median of --reps is reported, and
the script fails unless both arms give equal counts on every repetition.

    python tools/bench_tune.py [--reps 3] [--timit 32] [--librispeech 16] [--strict] [--out bench_tune.json]

Whisper-medium dimensions (24 x 16 heads), seeded random weights (qk_gain 4), synthetic utterances whose reference words
are their own words with boundaries spread evenly over the utterance, tune_alignment's default grid of 48 configs
(widths 3 5 7; mean, and top-k 1 5 10 15 20 under weights 1,1,0 1,0,0 0,1,0).  Needs a CUDA device; prints the card's
name and power limit with the figures."""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_default_timing import card, timed  # noqa: E402

UNIT = "char"  # the synthetic TIMIT / LibriSpeech utterances are char-encoded


def sweep(batch, configs, tk, model, refs, ref_words, tol):
    """Arm (a)."""
    from whisper_char_alignment_b200 import timing

    mels, tokens, texts, frames = batch
    widths = list(dict.fromkeys(c.medfilt_width for c in configs))
    by_width = timing.get_attentions_widths_batch(mels, tokens, model, tk, frames, widths)
    return timing.alignment_config_counts_batch({w: m for w, (m, _) in by_width.items()}, texts, tk, refs, configs,
                                                aligned_unit_type=UNIT, tolerance=tol, ref_words_list=ref_words)


def per_config(batch, configs, tk, model, refs, ref_words, tol):
    """Arm (b)."""
    from whisper_char_alignment_b200 import timing
    from whisper_char_alignment_b200.metrics import eval_n1, eval_n1_strict

    mels, tokens, texts, frames = batch
    out = [np.zeros((len(configs), 3), dtype=np.int64) for _ in texts]
    for i, c in enumerate(configs):
        maps, _ = timing.get_attentions_batch(mels, tokens, model, tk, frames, c.medfilt_width, 1.0)
        outs = timing.force_align_batch(maps, texts, tk, aligned_unit_type=UNIT, aggregation=c.aggr, topk=c.topk,
                                        w_colnorm=c.w_colnorm, w_rownorm=c.w_rownorm, w_coverage=c.w_coverage)
        for b, (words, _, ends, _, _) in enumerate(outs):
            if ref_words is None:
                out[b][i] = (eval_n1(refs[b], ends, tol)[0], len(ends), len(refs[b]))
            else:
                tp, fp, fn = eval_n1_strict(refs[b], ends, ref_words[b], " ".join(words[:-1]).split(), tol)
                out[b][i] = (tp, tp + fp, tp + fn)
    return out


def main(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--timit", type=int, default=32, help="TIMIT-shaped batch size")
    p.add_argument("--librispeech", type=int, default=16, help="LibriSpeech-shaped batch size")
    p.add_argument("--tolerance", type=float, default=0.02)
    p.add_argument("--strict", action="store_true", help="score with eval_n1_strict instead of eval_n1")
    p.add_argument("--out", default=None)
    args = p.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_tune: needs a CUDA device (no figure is measured without one)")

    from whisper_char_alignment_b200.cli import tune_alignment
    from whisper_char_alignment_b200.synthetic import librispeech_shaped, timit_shaped
    from whisper_char_alignment_b200.tokenizer import get_tokenizer
    from whisper_char_alignment_b200.whisper_model import load_model

    dev = torch.device("cuda:0")
    model = load_model("random:medium", dev, qk_gain=4.0)
    tk = get_tokenizer(True, language="English")
    configs = tune_alignment.grid(tune_alignment.parse_args(["--output_dir", "unused"]))
    name, limit = card()
    report = dict(card=name, power_limit=limit, model="random:medium (qk_gain 4)", configs=len(configs),
                  tolerance=args.tolerance, strict=args.strict, workloads={})
    for label, make, n in (("timit", timit_shaped, args.timit), ("librispeech", librispeech_shaped, args.librispeech)):
        utts = make(n, tk, n_mels=model.dims.n_mels, seed=1)
        batch = (torch.stack([u.mel for u in utts]).to(dev), [u.tokens.to(dev) for u in utts],
                 [u.text_tokens for u in utts], [u.max_frames for u in utts])
        ref_words = [u.text.split() for u in utts]
        refs = [np.arange(1, len(w) + 1, dtype=np.float64) * (u.max_frames / 50.0) / len(w)
                for w, u in zip(ref_words, utts)]
        rw = ref_words if args.strict else None
        run = lambda fn: timed(lambda: fn(batch, configs, tk, model, refs, rw, args.tolerance))  # noqa: E731
        run(sweep)  # warm-up of every shape of both arms
        run(per_config)
        sweep_s, per_config_s, equal = [], [], True
        for _ in range(args.reps):
            s, a = run(sweep)
            sweep_s.append(s)
            s, b = run(per_config)
            per_config_s.append(s)
            equal &= all(np.array_equal(x, y) for x, y in zip(a, b))
        med = lambda x: float(np.median(x))  # noqa: E731
        total = sum(a)
        f1 = [float(2 * h / (p_ + r)) if p_ + r else 0.0 for h, p_, r in total.tolist()]
        w = dict(utterances=n, tokens=int(sum(len(t) for t in batch[2])), frames=int(sum(batch[3])),
                 sweep_s=sorted(sweep_s), per_config_s=sorted(per_config_s), speedup=med(per_config_s) / med(sweep_s),
                 best_config=int(np.argmax(f1)), equal_counts=bool(equal))
        report["workloads"][label] = w
        print(f"{label} batch of {n}: {len(configs)} configs in one pass {1e3 * med(sweep_s):.1f} ms, one pass per "
              f"config {1e3 * med(per_config_s):.1f} ms (x{w['speedup']:.1f}); equal counts: {equal}", flush=True)
        assert equal, f"{label}: the sweep and the per-config passes give different counts"
        del batch
    print(f"card: {name}, power limit {limit}")
    print(json.dumps(report))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
