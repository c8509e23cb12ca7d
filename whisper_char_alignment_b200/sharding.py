"""Multi-GPU plumbing: utterances are independent, so rank r of W owns utterances r::W and
nothing is exchanged while aligning (SURVEY.md section 8e).  The ONE collective of a job is
the final all_gather of the metric counters (infer_ali.py:53-55,122-132) and of the padded
per-utterance boundary arrays; NCCL over NVLink on GPUs, gloo in the CPU tests."""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist


def shard_indices(n_items: int, rank: int, world_size: int):
    """Round-robin ownership: the fixed 30 s encoder dominates per-utterance cost, so
    interleaving balances the shards without sorting."""
    return list(range(rank, n_items, world_size))


def shard_by_cost(costs, rank: int, world_size: int):
    """Longest-processing-time-first assignment of items with very unequal cost (LibriSpeech: 2-30 s utterances,
    BASELINE.json configs[2]): items in decreasing cost, each to the currently lightest rank.  Deterministic and
    identical on every rank (ties by index); every item belongs to exactly one rank.  Returns this rank's indices in
    increasing order.  The greedy bound is 4/3 - 1/(3W) of the optimum; with hundreds of items per rank the measured
    imbalance is well under 1 %."""
    order = sorted(range(len(costs)), key=lambda i: (-float(costs[i]), i))
    loads = [0.0] * world_size
    mine = []
    for i in order:
        r = min(range(world_size), key=lambda k: (loads[k], k))
        loads[r] += float(costs[i])
        if r == rank:
            mine.append(i)
    return sorted(mine)


def shard_imbalance(costs, world_size: int, how: str = "lpt") -> float:
    """max over ranks of the assigned cost / mean, for `how` in {"lpt", "round_robin"}."""
    loads = []
    for r in range(world_size):
        idx = shard_by_cost(costs, r, world_size) if how == "lpt" else shard_indices(len(costs), r, world_size)
        loads.append(sum(float(costs[i]) for i in idx))
    mean = sum(loads) / world_size
    return max(loads) / mean if mean > 0 else 1.0


def _comm_device():
    if dist.is_initialized() and dist.get_backend() == "nccl":
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def sum_over_ranks(counts) -> np.ndarray:
    """Element-wise sum of an integer array of the same shape on every rank, in ONE collective (every rank gets the
    totals, as int64)."""
    local = np.asarray(counts, dtype=np.int64)
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return local.copy()
    t = torch.from_numpy(np.ascontiguousarray(local).reshape(-1)).to(_comm_device())
    parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, t)
    return torch.stack(parts).sum(0).cpu().numpy().reshape(local.shape)


def gather_counters(corrects: int, total_preds: int, total_gts: int):
    """Sum of the three metric counters over all ranks (every rank gets the totals)."""
    tot = sum_over_ranks([corrects, total_preds, total_gts]).tolist()
    return int(tot[0]), int(tot[1]), int(tot[2])


def gather_alignments(local: dict):
    """local: {utterance index: (start_times, end_times)} for the utterances this rank owns.
    Returns the merged dict on every rank.  Wire format: one float64 tensor per rank,
    rows [index, n_words, starts..., ends...] padded to the global maximum word count."""
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return {int(k): (np.asarray(s, np.float64), np.asarray(e, np.float64)) for k, (s, e) in local.items()}
    dev = _comm_device()
    world = dist.get_world_size()
    n_local = len(local)
    w_local = max([len(s) for s, _ in local.values()], default=0)
    shape = torch.tensor([n_local, w_local], dtype=torch.int64, device=dev)
    shapes = [torch.empty_like(shape) for _ in range(world)]
    dist.all_gather(shapes, shape)
    shapes = torch.stack(shapes).cpu()
    n_max, w_max = int(shapes[:, 0].max()), int(shapes[:, 1].max())
    buf = np.full((n_max, 2 + 2 * w_max), np.nan)
    for row, (idx, (s, e)) in enumerate(sorted(local.items())):
        buf[row, 0], buf[row, 1] = idx, len(s)
        buf[row, 2: 2 + len(s)] = s
        buf[row, 2 + w_max: 2 + w_max + len(e)] = e
    mine = torch.from_numpy(buf).to(dev)
    parts = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine)
    merged = {}
    for r, part in enumerate(parts):
        arr = part.cpu().numpy()
        for row in range(int(shapes[r, 0])):
            idx, n = int(arr[row, 0]), int(arr[row, 1])
            merged[idx] = (arr[row, 2: 2 + n].copy(), arr[row, 2 + w_max: 2 + w_max + n].copy())
    return merged
