"""Cost of scoring every head's single-head alignment against the reference boundaries (the measurement behind
find_alignment_heads), device against host:

  (a) device: wca_boundary_hits on the end times the DTW left on the device, as timing.head_boundary_counts_batch runs
      it (upload of the references, one launch, one copy of the hits), host clock around a synchronised call; and, with
      --profile in a run of its own, the kernel alone, its device time from torch.profiler over many calls;
  (b) host: the device->host copy of every head's start / end times plus metrics.eval_n1 (or eval_n1_strict) per head
      and per utterance, as the per-head loop of infer_ali / probe_oracle scores;
  whole step: capture (get_attentions_batch) + the L*H single-head alignments + scoring, with (a) (through
      timing.head_boundary_counts_batch) and with (b).

Arms alternate after a warm-up of every shape, and both give equal counts (checked on every repetition).

    python tools/bench_head_probe.py [--reps 3] [--timit 32] [--librispeech 16] [--profile] [--out bench_head_probe.json]

Whisper-medium dimensions (24 x 16 heads), seeded random weights (qk_gain 4), synthetic utterances whose reference
words are their own words with boundaries spread evenly over the utterance.  Needs a CUDA device; prints the card's
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


def host_counts(sh, refs, ref_words, tol):
    """Arm (b): copy every head's times to the host and score each head with metrics.py."""
    from whisper_char_alignment_b200.metrics import eval_n1, eval_n1_strict

    times_h = sh.times.cpu().numpy()
    out, p = [], 0
    for b, (words, _) in enumerate(sh.words_all):
        W, H = int(sh.n_words[b]), int((sh.utt_of == b).sum())
        hyp = " ".join(words[:-1]).split()
        c = np.empty((H, 3), dtype=np.int64)
        for k in range(H):
            ends = times_h[1, int(sh.recs["word_off"][p]): int(sh.recs["word_off"][p]) + W]
            if ref_words is None:
                c[k] = (eval_n1(refs[b], ends, tol)[0], len(ends), len(refs[b]))
            else:
                tp, fp, fn = eval_n1_strict(refs[b], ends, ref_words[b], hyp, tol)
                c[k] = (tp, tp + fp, tp + fn)
            p += 1
        out.append(c)
    return out


def device_counts(sh, refs, ref_words, tol):
    """Arm (a): the scoring half of timing.head_boundary_counts_batch."""
    from whisper_char_alignment_b200 import timing

    return timing._boundary_counts(sh, refs, tol, ref_words)


def kernel_ms(sh, refs, ref_words, tol, iters):
    """wca_boundary_hits alone: mean device time of boundary_hits_kernel over `iters` calls, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            device_counts(sh, refs, ref_words, tol)
        torch.cuda.synchronize()
    for k in prof.key_averages():
        if "boundary_hits_kernel" in k.key:
            us = getattr(k, "device_time_total", None)
            return (k.cuda_time_total if us is None else us) / k.count / 1e3
    raise RuntimeError("boundary_hits_kernel not found in the profile")


def main(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--timit", type=int, default=32, help="TIMIT-shaped batch size")
    p.add_argument("--librispeech", type=int, default=16, help="LibriSpeech-shaped batch size")
    p.add_argument("--tolerance", type=float, default=0.02)
    p.add_argument("--kernel_iters", type=int, default=200)
    p.add_argument("--profile", action="store_true",
                   help="only the kernel's device time, from torch.profiler (run it apart from the timed arms)")
    p.add_argument("--out", default=None)
    args = p.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_head_probe: needs a CUDA device (no figure is measured without one)")

    from whisper_char_alignment_b200 import timing
    from whisper_char_alignment_b200.synthetic import librispeech_shaped, timit_shaped
    from whisper_char_alignment_b200.tokenizer import get_tokenizer
    from whisper_char_alignment_b200.whisper_model import load_model

    dev = torch.device("cuda:0")
    model = load_model("random:medium", dev, qk_gain=4.0)
    tk = get_tokenizer(True, language="English")
    L, H = model.dims.n_text_layer, model.dims.n_text_head
    name, limit = card()
    report = dict(card=name, power_limit=limit, model="random:medium (qk_gain 4)", tolerance=args.tolerance,
                  workloads={})
    for label, make, n in (("timit", timit_shaped, args.timit), ("librispeech", librispeech_shaped, args.librispeech)):
        utts = make(n, tk, n_mels=model.dims.n_mels, seed=1)
        mels = torch.stack([u.mel for u in utts]).to(dev)
        tokens = [u.tokens.to(dev) for u in utts]
        texts = [u.text_tokens for u in utts]
        frames = [u.max_frames for u in utts]
        ref_words = [u.text.split() for u in utts]
        refs = [np.arange(1, len(w) + 1, dtype=np.float64) * (f / 50.0) / len(w) for w, f in zip(ref_words, frames)]
        heads = [np.arange(L * H)] * n

        for mode in ("plain", "strict"):
            rw = ref_words if mode == "strict" else None

            def step(device_arm):
                maps, _ = timing.get_attentions_batch(mels, tokens, model, tk, frames)
                if device_arm:  # the public entry point
                    return [c.reshape(-1, 3) for c in timing.head_boundary_counts_batch(
                        maps, texts, tk, refs, aligned_unit_type=UNIT, tolerance=args.tolerance, ref_words_list=rw)]
                sh = timing._launch_single_heads(maps, heads, texts, tk, UNIT)
                return host_counts(sh, refs, rw, args.tolerance)

            maps, _ = timing.get_attentions_batch(mels, tokens, model, tk, frames)
            sh = timing._launch_single_heads(maps, heads, texts, tk, UNIT)
            if args.profile:  # the kernel alone, in a run of its own (the profiler slows the host)
                device_counts(sh, refs, rw, args.tolerance)
                k_ms = kernel_ms(sh, refs, rw, args.tolerance, args.kernel_iters)
                report["workloads"][f"{label}/{mode}"] = dict(utterances=n, problems=len(sh.utt_of),
                                                              words=int(sh.n_words.sum()), kernel_ms=k_ms)
                print(f"{label}/{mode}: {len(sh.utt_of)} problems: boundary_hits_kernel {k_ms:.4f} ms", flush=True)
                del maps, sh
                continue
            for _ in range(2):  # warm-up of every shape and arm
                timed(lambda: device_counts(sh, refs, rw, args.tolerance))
                timed(lambda: host_counts(sh, refs, rw, args.tolerance))
            timed(lambda: step(True))
            timed(lambda: step(False))
            dev_s, host_s, step_dev_s, step_host_s = [], [], [], []
            equal = True
            for _ in range(args.reps):
                s, a = timed(lambda: device_counts(sh, refs, rw, args.tolerance))
                dev_s.append(s)
                s, b = timed(lambda: host_counts(sh, refs, rw, args.tolerance))
                host_s.append(s)
                equal &= all(np.array_equal(x, y) for x, y in zip(a, b))
                s, a = timed(lambda: step(True))
                step_dev_s.append(s)
                s, b = timed(lambda: step(False))
                step_host_s.append(s)
                equal &= all(np.array_equal(x, y) for x, y in zip(a, b))
            med = lambda x: float(np.median(x))  # noqa: E731
            w = dict(utterances=n, problems=len(sh.utt_of), words=int(sh.n_words.sum()),
                     ref_words=int(sum(len(r) for r in refs)), hits=int(sum(int(c[:, 0].sum()) for c in a)),
                     device_scoring_s=sorted(dev_s), host_scoring_s=sorted(host_s),
                     host_over_device=med(host_s) / med(dev_s), step_with_device_scoring_s=sorted(step_dev_s),
                     step_with_host_scoring_s=sorted(step_host_s), step_speedup=med(step_host_s) / med(step_dev_s),
                     equal_counts=bool(equal))
            report["workloads"][f"{label}/{mode}"] = w
            print(f"{label}/{mode}: {w['problems']} single-head alignments, {w['words']} words: "
                  f"scoring on the device {1e3 * med(dev_s):.2f} ms, copy + metrics.py on the host "
                  f"{1e3 * med(host_s):.1f} ms (x{w['host_over_device']:.0f}); whole step {1e3 * med(step_dev_s):.1f} "
                  f"against {1e3 * med(step_host_s):.1f} ms (x{w['step_speedup']:.2f}); equal counts: {equal}",
                  flush=True)
            assert equal, f"{label}/{mode}: device and host counts differ"
            del maps, sh
    print(f"card: {name}, power limit {limit}")
    print(json.dumps(report))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
