"""`infer_ali.py` shell: align a dataset and score the word boundaries.

Flags are the reference's (infer_ali.py:151-173) plus `--dataset synthetic`, `--batch_size` and
multi-GPU sharding under torchrun.  Per batch the hot path is two calls
(get_attentions_batch + force_align_batch), or one (default_find_alignment_batch) with --default_whisper_timing.  Ranks own cost-balanced shards (sharding.shard_by_cost over the
datasets' size hints), align them in length-bucketed batches (batching.plan_batches, with the reference's skip
rule for over-long inputs) and meet once, at the end."""
from __future__ import annotations

import argparse
import os
from collections import defaultdict

import numpy as np
import torch
import torch.distributed as dist

from .. import batching, sharding, timing
from ..dataset import DATASET
from ..metrics import eval_n1, eval_n1_strict, get_seg_metrics
from . import common


def parse_args(argv=None):
    p = argparse.ArgumentParser(description="Arguments for whisper-based forced alignments")
    p.add_argument("--model", type=str, default="medium")
    p.add_argument("--dataset", type=str, default="TIMIT", choices=sorted(DATASET))
    p.add_argument("--scp", type=str, default="scp/test.wav.scp")
    p.add_argument("--output_dir", type=str, default="results", required=True, help="Path to the output directory")
    p.add_argument("--n_mels", type=int, default=80)
    p.add_argument("--medfilt_width", type=int, default=7)
    p.add_argument("--aggr", type=str, default="mean", choices=["mean", "topk"])
    p.add_argument("--topk", type=int, default=15)
    p.add_argument("--aligned_unit_type", type=str, default="subword", choices=["subword", "char"])
    p.add_argument("--tolerance", type=float, default=0.02)
    p.add_argument("--w_colnorm", type=float, default=1.0)
    p.add_argument("--w_rownorm", type=float, default=1.0)
    p.add_argument("--w_coverage", type=float, default=0.0)
    p.add_argument("--plot", action="store_true")
    p.add_argument("--strict", action="store_true")
    p.add_argument("--save_prediction", action="store_true")
    p.add_argument("--default_whisper_timing", action="store_true")
    p.add_argument("--batch_size", type=int, default=16, help="utterances per launch (the reference uses 1)")
    # absent from the namespace unless given, so that the results JSON (every flag) of a run without it is unchanged
    p.add_argument("--word_probabilities", action="store_true", default=argparse.SUPPRESS,
                   help="with --save_prediction, save each predicted word's probability (whisper's word confidence) "
                        "as probs_hat")
    return p.parse_args(argv)


def infer_dataset(args):
    print(args)
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(device)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=device)
    model, tokenizer, whisper_pkg, model_source = common.load_model_and_tokenizer(args.model, device)
    dataset = DATASET[args.dataset](args.scp, n_mels=args.n_mels, device=device)
    qk_scale = 1.0
    n_maps = model.dims.n_text_layer * model.dims.n_text_head

    corrects = total_preds = total_gts = 0
    predictions = defaultdict(int)
    local_alignments = {}
    if hasattr(dataset, "size_hint"):
        hints = [dataset.size_hint(n) for n in range(len(dataset))]
        costs = [batching.utterance_cost(t, f, model.dims.n_text_layer, model.dims.n_text_state,
                                         model.dims.n_audio_layer) for t, f in hints]
        mine = sharding.shard_by_cost(costs, rank, world)
        mine.sort(key=lambda n: hints[n])  # similar lengths meet in the same window
    else:
        mine = sharding.shard_indices(len(dataset), rank, world)
    # windows of a few batches: every utterance of a window is prepared (transcribed, tokenised), then the window is
    # cut into length-bucketed batches
    for window in common.batches(mine, args.batch_size * 8):
        items = common.prepare_window([dataset[n] for n in window], tokenizer, args.aligned_unit_type, device, whisper_pkg,
                                      model, args.batch_size)
        prepared = [(n, item) for n, item in zip(window, items) if item is not None]
        plan, _ = batching.plan_batches([len(it["tokens"]) for _, it in prepared], [it["max_frames"] for _, it in prepared],
                                        args.batch_size, n_maps=n_maps)
        for chunk in plan:
            items = [prepared[j] for j in chunk]
            hit, n_pred, n_gt = _align_batch(args, items, model, tokenizer, qk_scale, local_alignments, predictions)
            corrects, total_preds, total_gts = corrects + hit, total_preds + n_pred, total_gts + n_gt
    return _finish(args, rank, world, corrects, total_preds, total_gts, local_alignments, predictions, model_source,
                   common.transcript_source(whisper_pkg))


def _align_batch(args, items, model, tokenizer, qk_scale, local_alignments, predictions):
    """One length-bucketed batch through the hot path; returns (corrects, predicted, reference) boundary counts."""
    corrects = total_preds = total_gts = 0
    # the encoder output the transcription step already computed (greedy mode), else the mels
    features = None
    if items[0][1]["audio_features"] is not None:
        features = torch.stack([it["audio_features"] for _, it in items])
    mels = None if features is not None else [it["mel"] for _, it in items]
    with_probs = getattr(args, "word_probabilities", False)
    word_probs = None  # per utterance, the probabilities of words[:-1] (--word_probabilities)
    if args.default_whisper_timing:
        outs = timing.default_find_alignment_batch(model, tokenizer, [it["text_tokens"] for _, it in items], mels,
                                                   [it["max_frames"] for _, it in items], audio_features=features,
                                                   word_probabilities=with_probs)
        if with_probs:
            word_probs = [np.zeros(0) if isinstance(out, list) else out[4] for out in outs]
    else:
        maps, logits = timing.get_attentions_batch(mels, [it["tokens"] for _, it in items], model, tokenizer,
                                                   [it["max_frames"] for _, it in items], args.medfilt_width, qk_scale,
                                                   audio_features=features)
        outs = timing.force_align_batch(maps, [it["text_tokens"] for _, it in items], tokenizer,
                                        aligned_unit_type=args.aligned_unit_type, aggregation=args.aggr,
                                        topk=args.topk, w_colnorm=args.w_colnorm, w_rownorm=args.w_rownorm,
                                        w_coverage=args.w_coverage)
        if with_probs:
            word_probs = [wp for _, wp in timing.word_probabilities_batch(
                logits, [it["text_tokens"] for _, it in items], tokenizer, args.aligned_unit_type)]
    for b, ((n, it), out) in enumerate(zip(items, outs)):
        words, start_times, end_times, ws, _scores = out
        if args.plot:
            from ..plot import plot_attn  # matplotlib is optional

            plot_attn(ws, it["text_tokens"], tokenizer, gt_alignment=it["ends"], pred_alignment=end_times,
                      fid=it["fid"], aligned_unit_type=args.aligned_unit_type,
                      path=f"{args.output_dir}/imgs/{args.dataset}")
        local_alignments[n] = (start_times, end_times)
        if args.save_prediction:
            predictions[n] = dict(starts=it["starts"], ends=it["ends"], texts=it["text"].split(),
                                  starts_hat=start_times, ends_hat=end_times, predwords=words, fids=it["fid"])
            if word_probs is not None:
                predictions[n]["probs_hat"] = word_probs[b]
        if not args.strict:
            hit, _ = eval_n1(it["ends"], end_times, args.tolerance)
            total_gts += len(it["ends"])
            total_preds += len(end_times)
            corrects += hit
        else:
            hyp_words = " ".join(words[:-1]).split()
            tp, fp, fn = eval_n1_strict(it["ends"], end_times, it["text"].split(), hyp_words, args.tolerance)
            corrects += tp
            total_gts += tp + fn
            total_preds += tp + fp

    return corrects, total_preds, total_gts


def _finish(args, rank, world, corrects, total_preds, total_gts, local_alignments, predictions, model_source,
            transcript_source):
    # the job's single collective: metric counters and the padded boundary arrays
    corrects, total_preds, total_gts = sharding.gather_counters(corrects, total_preds, total_gts)
    alignments = sharding.gather_alignments(local_alignments)
    precision, recall, f1, r_value, _ = get_seg_metrics(corrects, corrects, total_preds, total_gts)
    results = dict(precision=precision, recall=recall, f1=f1, r_value=r_value)
    provenance = dict(model_source=model_source, transcript_source=transcript_source)
    if rank == 0:
        print(results)
        if model_source.startswith("random-init"):
            print(f"NOTE: {model_source}: these figures come from RANDOM weights (synthetic / smoke run), not from a checkpoint")
        path, stamp = common.dump_results(args, {**results, **provenance})
        if args.save_prediction:
            import joblib

            if world > 1:  # other ranks' predictions travel as objects (host-side, once)
                gathered = [None] * world
                dist.gather_object(dict(predictions), gathered, dst=0)
                for part in gathered:
                    predictions.update(part)
            joblib.dump(predictions, os.path.join(args.output_dir, stamp + "-predictions.pkl"))
        print(f"{len(alignments)} utterances aligned; results in {path}")
    elif args.save_prediction and world > 1:
        dist.gather_object(dict(predictions), None, dst=0)
    if world > 1:
        dist.barrier()
    return results


def main(argv=None):
    return infer_dataset(parse_args(argv))


if __name__ == "__main__":
    main()
