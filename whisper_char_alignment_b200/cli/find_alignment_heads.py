"""`find_alignment_heads.py` shell: measure how well every cross-attention head aligns words on its own over a labelled
dataset, and pick the best heads as the checkpoint's alignment heads.

This is how upstream Whisper found the head masks it ships for its own checkpoints; a fine-tuned or locally trained
checkpoint has none.  Each head (l, h) of each utterance is aligned on its own (force_align of that one map,
aggregation "mean") and its predicted word ends are scored against the reference ends with infer_ali's metric
(eval_n1, or eval_n1_strict with --strict), on the device.  The (layer, head) table of (hits, predicted, reference)
counts is summed over the dataset and over ranks (one collective), and rank 0 writes
<output_dir>/<stamp>-heads.json: the flags, every head's counts, precision, recall and F1, the --n_heads heads of
best F1 and their mask in upstream's format, which `infer_ali --default_whisper_timing --alignment_heads` takes (as the
mask string or as this file)."""
from __future__ import annotations

import argparse
import os

import numpy as np
import torch
import torch.distributed as dist

from .. import batching, heads, sharding, timing
from ..dataset import DATASET
from ..metrics import get_seg_metrics
from . import common


def parse_args(argv=None):
    p = argparse.ArgumentParser(description="Find a checkpoint's alignment heads from labelled data")
    p.add_argument("--model", type=str, default="medium")
    p.add_argument("--dataset", type=str, default="TIMIT", choices=sorted(DATASET))
    p.add_argument("--scp", type=str, default="scp/test.wav.scp")
    p.add_argument("--output_dir", type=str, default="results", required=True, help="Path to the output directory")
    p.add_argument("--n_mels", type=int, default=80)
    p.add_argument("--medfilt_width", type=int, default=7)
    p.add_argument("--aligned_unit_type", type=str, default="subword", choices=["subword", "char"])
    p.add_argument("--tolerance", type=float, default=0.02)
    p.add_argument("--strict", action="store_true")
    p.add_argument("--batch_size", type=int, default=16, help="utterances per launch")
    p.add_argument("--n_heads", type=int, default=10, help="how many heads of best F1 become the alignment heads")
    args = p.parse_args(argv)
    if args.n_heads < 1:
        p.error("--n_heads must be at least 1")
    return args


def count_dataset(args):
    """(model, tokenizer, whisper_pkg, model_source, (L, H, 3) int64 counts summed over this rank's utterances)."""
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(device)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=device)
    model, tokenizer, whisper_pkg, model_source = common.load_model_and_tokenizer(args.model, device)
    dataset = DATASET[args.dataset](args.scp, n_mels=args.n_mels, device=device)
    L, H = model.dims.n_text_layer, model.dims.n_text_head
    counts = np.zeros((L, H, 3), dtype=np.int64)
    if hasattr(dataset, "size_hint"):
        hints = [dataset.size_hint(n) for n in range(len(dataset))]
        costs = [batching.utterance_cost(t, f, L, model.dims.n_text_state, model.dims.n_audio_layer) for t, f in hints]
        mine = sharding.shard_by_cost(costs, rank, world)
        mine.sort(key=lambda n: hints[n])
    else:
        mine = sharding.shard_indices(len(dataset), rank, world)
    for window in common.batches(mine, args.batch_size * 8):
        items = common.prepare_window([dataset[n] for n in window], tokenizer, args.aligned_unit_type, device, whisper_pkg,
                                      model, args.batch_size)
        items = [it for it in items if it is not None]
        # the single-head matrices of all L*H heads are about as large as the maps themselves
        plan, _ = batching.plan_batches([len(it["tokens"]) for it in items], [it["max_frames"] for it in items],
                                        args.batch_size, n_maps=2 * L * H)
        for chunk in plan:
            counts += sum(count_batch(args, [items[j] for j in chunk], model, tokenizer))
    return model, tokenizer, whisper_pkg, model_source, counts


def count_batch(args, items, model, tokenizer):
    """Per utterance of one batch, its (L, H, 3) counts."""
    features = None
    if items[0]["audio_features"] is not None:
        features = torch.stack([it["audio_features"] for it in items])
    mels = None if features is not None else [it["mel"] for it in items]
    maps, _ = timing.get_attentions_batch(mels, [it["tokens"] for it in items], model, tokenizer,
                                          [it["max_frames"] for it in items], args.medfilt_width, 1.0,
                                          audio_features=features)
    return timing.head_boundary_counts_batch(
        maps, [it["text_tokens"] for it in items], tokenizer, [it["ends"] for it in items],
        aligned_unit_type=args.aligned_unit_type, tolerance=args.tolerance,
        ref_words_list=[it["text"].split() for it in items] if args.strict else None)


def head_table(counts):
    """Per (layer, head), its counts and get_seg_metrics' precision, recall and F1, in flat-index order."""
    rows = []
    for l in range(counts.shape[0]):
        for h in range(counts.shape[1]):
            hit, n_pred, n_ref = (int(x) for x in counts[l, h])
            precision, recall, f1, _, _ = get_seg_metrics(hit, hit, n_pred, n_ref)
            rows.append(dict(layer=l, head=h, hits=hit, n_pred=n_pred, n_ref=n_ref, precision=float(precision),
                             recall=float(recall), f1=float(f1)))
    return rows


def main(argv=None):
    args = parse_args(argv)
    print(args)
    model, _, whisper_pkg, model_source, counts = count_dataset(args)
    counts = sharding.sum_over_ranks(counts)  # the job's single collective
    mask = heads.rank_heads(counts, args.n_heads)
    result = dict(model_source=model_source, transcript_source=common.transcript_source(whisper_pkg),
                  heads=head_table(counts), alignment_heads=np.argwhere(mask).tolist(),
                  mask=heads.encode_alignment_heads(mask).decode("ascii"))
    if int(os.environ.get("RANK", 0)) == 0:
        path, _ = common.dump_results(args, result, suffix="-heads")
        print(f"alignment heads {result['alignment_heads']}; mask {result['mask']}; table in {path}")
        if model_source.startswith("random-init"):
            print(f"NOTE: {model_source}: these heads come from RANDOM weights (synthetic / smoke run), not from a checkpoint")
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.barrier()
    return result


if __name__ == "__main__":
    main()
