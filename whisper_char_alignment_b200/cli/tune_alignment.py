"""`tune_alignment.py` shell: score a grid of alignment settings over a labelled dataset and report which one aligns
best.

The settings the method leaves free (--medfilt_width, --aggr, --topk and the head-score weights) were chosen for OpenAI's
checkpoints on TIMIT; a fine-tuned or locally trained checkpoint may want others.  Every configuration of the grid
(tuning.expand_grid) is scored with infer_ali's metric (eval_n1, or eval_n1_strict with --strict) from ONE forward per
batch: get_attentions_widths_batch captures the maps of every width, alignment_config_counts_batch aligns and scores
every configuration on the device.  The (config, (hits, predicted, reference)) table is summed over the dataset and
over ranks (one collective), and rank 0 writes <output_dir>/<stamp>-tune.json: the flags, every config with its counts,
precision, recall, F1 and R-value, the ranking by F1 and the infer_ali flags of the best config."""
from __future__ import annotations

import argparse
import os

import numpy as np
import torch
import torch.distributed as dist

from .. import batching, sharding, timing, tuning
from ..dataset import DATASET
from ..metrics import get_seg_metrics
from . import common


def _weighting(text: str):
    parts = text.split(",")
    if len(parts) != 3:
        raise argparse.ArgumentTypeError(f"{text!r}: expected colnorm,rownorm,coverage")
    try:
        return tuple(float(x) for x in parts)
    except ValueError as e:
        raise argparse.ArgumentTypeError(f"{text!r}: {e}") from None


def parse_args(argv=None):
    p = argparse.ArgumentParser(description="Tune a checkpoint's alignment settings from labelled data")
    p.add_argument("--model", type=str, default="medium")
    p.add_argument("--dataset", type=str, default="TIMIT", choices=sorted(DATASET))
    p.add_argument("--scp", type=str, default="scp/test.wav.scp")
    p.add_argument("--output_dir", type=str, default="results", required=True, help="Path to the output directory")
    p.add_argument("--n_mels", type=int, default=80)
    p.add_argument("--aligned_unit_type", type=str, default="subword", choices=["subword", "char"])
    p.add_argument("--tolerance", type=float, default=0.02)
    p.add_argument("--strict", action="store_true")
    p.add_argument("--batch_size", type=int, default=16, help="utterances per launch")
    p.add_argument("--medfilt_widths", type=int, nargs="+", default=[3, 5, 7])
    p.add_argument("--aggrs", type=str, nargs="+", default=["mean", "topk"], choices=list(tuning.AGGREGATIONS))
    p.add_argument("--topks", type=int, nargs="+", default=[1, 5, 10, 15, 20])
    p.add_argument("--weights", type=_weighting, nargs="+", default=[(1.0, 1.0, 0.0), (1.0, 0.0, 0.0), (0.0, 1.0, 0.0)],
                   metavar="COLNORM,ROWNORM,COVERAGE", help="head-score weightings of the top-k configs")
    args = p.parse_args(argv)
    try:
        grid(args)
    except ValueError as e:
        p.error(str(e))
    return args


def grid(args):
    return tuning.expand_grid(args.medfilt_widths, args.aggrs, args.topks, args.weights)


def count_dataset(args, configs):
    """(model, tokenizer, whisper_pkg, model_source, (n_configs, 3) int64 counts summed over this rank's utterances)."""
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(device)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=device)
    model, tokenizer, whisper_pkg, model_source = common.load_model_and_tokenizer(args.model, device)
    dataset = DATASET[args.dataset](args.scp, n_mels=args.n_mels, device=device)
    L, H = model.dims.n_text_layer, model.dims.n_text_head
    counts = np.zeros((len(configs), 3), dtype=np.int64)
    if hasattr(dataset, "size_hint"):
        hints = [dataset.size_hint(n) for n in range(len(dataset))]
        costs = [batching.utterance_cost(t, f, L, model.dims.n_text_state, model.dims.n_audio_layer) for t, f in hints]
        mine = sharding.shard_by_cost(costs, rank, world)
        mine.sort(key=lambda n: hints[n])
    else:
        mine = sharding.shard_indices(len(dataset), rank, world)
    widths = list(dict.fromkeys(c.medfilt_width for c in configs))
    for window in common.batches(mine, args.batch_size * 8):
        items = common.prepare_window([dataset[n] for n in window], tokenizer, args.aligned_unit_type, device, whisper_pkg,
                                      model, args.batch_size)
        items = [it for it in items if it is not None]
        # every width's maps are captured from the one forward and live together, beside one matrix per config
        plan, _ = batching.plan_batches([len(it["tokens"]) for it in items], [it["max_frames"] for it in items],
                                        args.batch_size, n_maps=len(widths) * L * H + len(configs))
        for chunk in plan:
            counts += sum(count_batch(args, configs, widths, [items[j] for j in chunk], model, tokenizer))
    return model, tokenizer, whisper_pkg, model_source, counts


def count_batch(args, configs, widths, items, model, tokenizer):
    """Per utterance of one batch, its (n_configs, 3) counts."""
    features = None
    if items[0]["audio_features"] is not None:
        features = torch.stack([it["audio_features"] for it in items])
    mels = None if features is not None else [it["mel"] for it in items]
    by_width = timing.get_attentions_widths_batch(mels, [it["tokens"] for it in items], model, tokenizer,
                                                  [it["max_frames"] for it in items], widths, 1.0,
                                                  audio_features=features)
    return timing.alignment_config_counts_batch(
        {w: maps for w, (maps, _) in by_width.items()}, [it["text_tokens"] for it in items], tokenizer,
        [it["ends"] for it in items], configs, aligned_unit_type=args.aligned_unit_type, tolerance=args.tolerance,
        ref_words_list=[it["text"].split() for it in items] if args.strict else None)


def config_table(configs, counts):
    """Per config, its settings, counts and get_seg_metrics' precision, recall, F1 and R-value, in grid order."""
    rows = []
    for c, (hit, n_pred, n_ref) in zip(configs, counts.tolist()):
        precision, recall, f1, r_value, _ = get_seg_metrics(hit, hit, n_pred, n_ref)
        rows.append(dict(c._asdict(), hits=hit, n_pred=n_pred, n_ref=n_ref, precision=float(precision),
                         recall=float(recall), f1=float(f1), r_value=float(r_value)))
    return rows


def main(argv=None):
    args = parse_args(argv)
    print(args)
    configs = grid(args)
    model, _, whisper_pkg, model_source, counts = count_dataset(args, configs)
    counts = sharding.sum_over_ranks(counts)  # the job's single collective
    ranking = tuning.rank_configs(counts)
    best = configs[ranking[0]]
    result = dict(model_source=model_source, transcript_source=common.transcript_source(whisper_pkg),
                  configs=config_table(configs, counts), ranking=ranking, best=best._asdict(),
                  best_flags=tuning.infer_ali_flags(best))
    if int(os.environ.get("RANK", 0)) == 0:
        path, _ = common.dump_results(args, result, suffix="-tune")
        row = result["configs"][ranking[0]]
        print(f"best of {len(configs)} configs: F1 {row['f1']:.4f} with {' '.join(result['best_flags'])}; table in {path}")
        if model_source.startswith("random-init"):
            print(f"NOTE: {model_source}: these settings come from RANDOM weights (synthetic / smoke run), not from a checkpoint")
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.barrier()
    return result


if __name__ == "__main__":
    main()
