"""Cost of the per-word probabilities (timing.word_probabilities_batch, kernel wca_token_probs):

  * the kernel alone, from CUDA events over many launches, at the rows of a TIMIT-shaped (32 x ~40 text rows) and a
    LibriSpeech-shaped (16 x ~400 text rows) batch of Whisper-medium (n_cols = eot = 50 257 text-vocabulary columns
    read at the product's pitch of 51 872 floats), cycling over enough copies of the logits to exceed the 126 MB L2;
    its rate on the algorithmic bytes (4 n_cols read per row, plus 8 for the target and the output) against the
    6548.5 GB/s HBM copy bandwidth of BASELINE.md;
  * eager torch on the same rows: the rows gathered into one tensor, [:, :eot].softmax(-1), then a gather of the
    targets;
  * the cost added to one alignment batch: get_attentions_batch + force_align_batch with and without
    word_probabilities_batch, alternating.

    python tools/bench_word_probs.py [--reps 5] [--timit 32] [--librispeech 16] [--out bench_word_probs.json]

Whisper-medium dimensions, seeded random weights (qk_gain 4), synthetic utterances.  Needs a CUDA device; prints the
card's name and power limit with the figures."""
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
from bench_default_timing import COPY_PEAK_GBS, card, timed  # noqa: E402

L2_BYTES = 126 * 2 ** 20


def kernel_vs_torch(logits_list, texts, tokenizer, iters):
    """wca_token_probs and the eager torch arm on the text rows of the batch, each timed over `iters` launches that
    cycle over copies of the batch's padded logits (more bytes than the L2 holds)."""
    from whisper_char_alignment_b200 import _cabi

    sot, n_cols = len(tokenizer.sot_sequence), tokenizer.eot
    base = logits_list[0]
    # every utterance's (T_b, V) logits are row views of one (B, T_max, V_pad) tensor: copy that tensor
    owner_rows = max((lg.data_ptr() - base.data_ptr()) // 4 // base.stride(0) + lg.shape[0] for lg in logits_list)
    block = torch.as_strided(base, (owner_rows, base.stride(0)), (base.stride(0), 1))
    n_rows = sum(len(t) for t in texts)
    copies = max(2, int(np.ceil(2 * L2_BYTES / (4 * n_rows * n_cols))))
    blocks = [block.clone() for _ in range(copies)]
    rel = np.concatenate([(lg.data_ptr() - base.data_ptr()) // 4 + base.stride(0) * (sot + np.arange(len(t)))
                          for lg, t in zip(logits_list, texts)]).astype(np.int64)
    targets = np.concatenate([np.asarray(t, dtype=np.int64) for t in texts])
    d_tg = torch.from_numpy(targets).to(base.device)
    probs = torch.empty(n_rows, dtype=torch.float32, device=base.device)
    lib = _cabi.load()
    d_rows = [torch.from_numpy(b.data_ptr() + 4 * rel).to(base.device) for b in blocks]
    d_tg32 = d_tg.to(torch.int32)
    stream = torch.cuda.current_stream().cuda_stream

    def kernel(i):
        rc = lib.wca_token_probs(d_rows[i % copies].data_ptr(), d_tg32.data_ptr(), n_rows, n_cols, probs.data_ptr(), stream)
        assert rc == 0, lib.wca_last_error()

    row_idx = torch.from_numpy(rel // base.stride(0)).to(base.device)

    def eager(i):
        rows = blocks[i % copies].index_select(0, row_idx)  # the same rows, gathered as the eager path would
        return rows[:, :n_cols].softmax(-1).gather(1, d_tg[:, None])

    def events(fn):
        for i in range(copies):
            fn(i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(iters):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    ms_k = events(kernel)
    ms_t = events(eager)
    got = probs.clone()
    want = eager(0).squeeze(1)
    nbytes = n_rows * (4 * n_cols + 8)
    return dict(rows=n_rows, n_cols=n_cols, copies_cycled=copies, kernel_ms=ms_k, algorithmic_bytes=nbytes,
                gbs=nbytes / ms_k / 1e6, share_of_copy_peak=nbytes / ms_k / 1e6 / COPY_PEAK_GBS, torch_ms=ms_t,
                torch_over_kernel=ms_t / ms_k,
                max_rel_diff_vs_torch=float(((got - want).abs() / want.abs().clamp_min(1e-30)).max()))


def main(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--reps", type=int, default=5)
    p.add_argument("--timit", type=int, default=32, help="TIMIT-shaped batch size")
    p.add_argument("--librispeech", type=int, default=16, help="LibriSpeech-shaped batch size")
    p.add_argument("--kernel_iters", type=int, default=200)
    p.add_argument("--out", default=None)
    args = p.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_word_probs: needs a CUDA device (no figure is measured without one)")

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
        mels = torch.stack([u.mel for u in utts]).to(dev)
        tokens = [u.tokens.to(dev) for u in utts]
        texts = [u.text_tokens for u in utts]
        frames = [u.max_frames for u in utts]

        def align(with_probs):
            maps, logits = timing.get_attentions_batch(mels, tokens, model, tk, frames)
            outs = timing.force_align_batch(maps, texts, tk, aligned_unit_type="char")
            if with_probs:
                return outs, timing.word_probabilities_batch(logits, texts, tk, "char")
            return outs, None

        timed(lambda: align(False))
        timed(lambda: align(True))  # warm-up of every shape
        t0, t1 = [], []
        for _ in range(args.reps):
            s, o0 = timed(lambda: align(False))
            t0.append(s)
            s, o1 = timed(lambda: align(True))
            t1.append(s)
        same = all(np.array_equal(a[2], b[2]) for a, b in zip(o0[0], o1[0]) if not isinstance(a, list))
        _, logits = timing.get_attentions_batch(mels, tokens, model, tk, frames)
        k = kernel_vs_torch(logits, texts, tk, args.kernel_iters)
        w = dict(utterances=n, text_rows=k["rows"], align_s=sorted(t0), align_with_probs_s=sorted(t1),
                 added_ms=1e3 * (float(np.median(t1)) - float(np.median(t0))),
                 added_share=float(np.median(t1)) / float(np.median(t0)) - 1.0, same_end_times=same, token_probs=k)
        report["workloads"][label] = w
        print(f"{label}: {k['rows']} rows x {k['n_cols']} columns: wca_token_probs {k['kernel_ms']:.4f} ms, "
              f"{k['gbs']:.0f} GB/s = {100 * k['share_of_copy_peak']:.1f} % of {COPY_PEAK_GBS} GB/s; eager torch "
              f"{k['torch_ms']:.4f} ms (x{k['torch_over_kernel']:.1f}); alignment batch {1e3 * np.median(t0):.2f} ms, "
              f"+{w['added_ms']:.3f} ms ({100 * w['added_share']:.2f} %) with word probabilities; "
              f"max rel diff vs torch {k['max_rel_diff_vs_torch']:.2e}", flush=True)
    print(f"card: {name}, power limit {limit}")
    print(json.dumps(report))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
