"""`probe_oracle.py` shell: align every head on its own, pick the best-F1 ("oracle") head per utterance
and count how often the scoring would have kept it (reference probe_oracle.py:28-138).

The reference file does not run as committed; this implements its evident intent (SURVEY.md 3.4):
`plot_attns` does not exist, `best_ends_hat` is used before assignment where `ends_hat` is meant, and
`correct_pred` is undefined where the strict counts `tp, tp+fp, tp+fn` are meant.  All heads of an
utterance go through ONE batched force_align launch instead of L*H sequential calls."""
from __future__ import annotations

import argparse
import os

import torch

from .. import timing
from ..dataset import DATASET
from ..metrics import eval_n1, eval_n1_strict, get_seg_metrics
from . import common

N_PROBED_HEADS = 360  # probe_oracle.py:83 `filter_attention(w, topk=360)`
TRANSCRIBE_BATCH = 16  # utterances per greedy transcription batch (common.prepare_window)


def parse_args(argv=None):
    p = argparse.ArgumentParser(description="Arguments for whisper-based forced alignments")
    p.add_argument("--model", type=str, default="medium")
    p.add_argument("--dataset", type=str, default="TIMIT", choices=sorted(DATASET))
    p.add_argument("--scp", type=str, default="scp/test.wav.scp")
    p.add_argument("--output_dir", type=str, default="results", required=True, help="Path to the output directory")
    p.add_argument("--n_mels", type=int, default=80)
    p.add_argument("--medfilt_width", type=int, default=7)
    p.add_argument("--hit_within", type=int, default=10,
                   help="compute how often the oracle head is included in the selected heads using the proposed approach.")
    p.add_argument("--aggr", type=str, default="mean", choices=["mean", "topk"])
    p.add_argument("--topk", type=int, default=15)
    p.add_argument("--aligned_unit_type", type=str, default="subword", choices=["subword", "char"])
    p.add_argument("--tolerance", type=float, default=0.02)
    p.add_argument("--plot", action="store_true")
    p.add_argument("--strict", action="store_true")
    p.add_argument("--min_words", type=int, default=18, help="probe_oracle.py:55 skips shorter utterances")
    return p.parse_args(argv)


def infer_dataset(args):
    print(args)
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(device)
    model, tokenizer, whisper_pkg, model_source = common.load_model_and_tokenizer(args.model, device)
    dataset = DATASET[args.dataset](args.scp, n_mels=args.n_mels, device=device)
    corrects = total_preds = total_gts = includes_best = n_probed = 0
    for it in _prepared(dataset, args, tokenizer, device, whisper_pkg, model):
        if it is None:
            continue
        w, _ = timing.get_attentions(it["mel"], it["tokens"], model, tokenizer, it["max_frames"], args.medfilt_width, 1.0)
        outs, scores = timing.probe_heads_batch([w], [it["text_tokens"]], tokenizer, args.aligned_unit_type,
                                                N_PROBED_HEADS)[0]
        ref_words = it["text"].split()
        best_f1, best_ends, best_words, best_score = -1.0, None, None, None
        for out, score in zip(outs, scores):
            if isinstance(out, list):
                continue
            words, _, ends_hat, _, _ = out
            hyp_words = " ".join(words[:-1]).split()
            tp, fp, fn = eval_n1_strict(it["ends"], ends_hat, ref_words, hyp_words, args.tolerance)
            _, _, f1, _, _ = get_seg_metrics(tp, tp, tp + fp, tp + fn)
            if f1 >= best_f1:
                best_f1, best_ends, best_words, best_score = f1, ends_hat, hyp_words, score[0]
        if best_ends is None:
            continue
        n_probed += 1
        if len(scores) >= args.hit_within and best_score > scores[-args.hit_within][0]:
            includes_best += 1
        if not args.strict:
            hit, _ = eval_n1(it["ends"], best_ends, args.tolerance)
            total_gts += len(it["ends"])
            total_preds += len(best_ends)
            corrects += hit
        else:
            tp, fp, fn = eval_n1_strict(it["ends"], best_ends, ref_words, best_words, args.tolerance)
            corrects += tp
            total_gts += tp + fn
            total_preds += tp + fp
    precision, recall, f1, r_value, _ = get_seg_metrics(corrects, corrects, total_preds, total_gts)
    results = dict(precision=precision, recall=recall, f1=f1, r_value=r_value,
                   hit_rate=includes_best / max(len(dataset), 1), utterances_probed=n_probed)
    print(results)
    common.dump_results(args, {**results, "model_source": model_source,
                               "transcript_source": common.transcript_source(whisper_pkg)})
    return results


def _prepared(dataset, args, tokenizer, device, whisper_pkg, model):
    """The prepared records with at least --min_words reference words, in dataset order (None where skipped)."""
    for window in common.batches(range(len(dataset)), TRANSCRIBE_BATCH):
        records = [r for r in (dataset[n] for n in window) if len(r[3].split()) >= args.min_words]
        yield from common.prepare_window(records, tokenizer, args.aligned_unit_type, device, whisper_pkg, model,
                                         TRANSCRIBE_BATCH)


def main(argv=None):
    return infer_dataset(parse_args(argv))


if __name__ == "__main__":
    main()
