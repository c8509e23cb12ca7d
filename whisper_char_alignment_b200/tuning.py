"""Alignment settings tuned on labelled data: the grid of configurations `tune_alignment` sweeps, their ranking by
dataset F1, and the `infer_ali` flags of a configuration.

A configuration is (medfilt_width, aggr, topk, w_colnorm, w_rownorm, w_coverage): every `infer_ali` flag that changes
the alignment of a given transcript except the unit type (which changes the tokens, hence the forward) and qk_scale
(1.0 in infer_ali).  timing.alignment_config_counts_batch counts the word boundaries of every configuration of a grid
in one pass."""
from __future__ import annotations

import math
from typing import NamedTuple

import numpy as np

from .heads import head_f1

AGGREGATIONS = ("mean", "topk")
#: What a mean configuration carries for the flags mean aggregation ignores: infer_ali's defaults.
MEAN_TOPK = 15
MEAN_WEIGHTS = (1.0, 1.0, 0.0)


class Config(NamedTuple):
    medfilt_width: int
    aggr: str
    topk: int
    w_colnorm: float
    w_rownorm: float
    w_coverage: float


def expand_grid(widths, aggrs, topks, weightings) -> list[Config]:
    """Every configuration of a grid, in this order: for each width (as given), for each aggregation (as given),
    "mean" gives ONE config (its weights and top-k do not change the alignment: it carries MEAN_TOPK and MEAN_WEIGHTS),
    "topk" gives one config per weighting (as given) and, within a weighting, per topk (as given).  weightings:
    (w_colnorm, w_rownorm, w_coverage) triples.  A repeated config keeps its first place only.
    Raises ValueError for an empty list, a width that is not an odd positive int, an unknown aggregation, topk <= 0
    with "topk", or a negative or NaN weight."""
    widths, aggrs, topks, weightings = list(widths), list(aggrs), list(topks), [tuple(w) for w in weightings]
    for name, values in (("widths", widths), ("aggrs", aggrs), ("topks", topks), ("weightings", weightings)):
        if not values:
            raise ValueError(f"expand_grid: empty list of {name}")
    for w in widths:
        if int(w) != w or w < 1 or w % 2 != 1:
            raise ValueError(f"expand_grid: median-filter width {w} is not an odd positive int")
    for a in aggrs:
        if a not in AGGREGATIONS:
            raise ValueError(f"expand_grid: unknown aggregation {a!r} (expected one of {AGGREGATIONS})")
    if "topk" in aggrs:
        for k in topks:
            if int(k) != k or k <= 0:
                raise ValueError(f"expand_grid: topk={k} with aggregation 'topk' must be a positive int")
    for wt in weightings:
        if len(wt) != 3:
            raise ValueError(f"expand_grid: weighting {wt} is not a (colnorm, rownorm, coverage) triple")
        for x in wt:
            if math.isnan(float(x)) or float(x) < 0:
                raise ValueError(f"expand_grid: weighting {wt} has a negative or NaN weight")
    grid = []
    for w in widths:
        for a in aggrs:
            if a == "mean":
                grid.append(Config(int(w), "mean", MEAN_TOPK, *MEAN_WEIGHTS))
                continue
            for wc, wr, wv in weightings:
                for k in topks:
                    grid.append(Config(int(w), "topk", int(k), float(wc), float(wr), float(wv)))
    return list(dict.fromkeys(grid))


def config_f1(counts) -> np.ndarray:
    """(n_configs,) dataset F1 of every config: get_seg_metrics(hits, hits, n_pred, n_ref) on its summed counts."""
    return head_f1(np.asarray(counts, dtype=np.int64).reshape(-1, 3))


def rank_configs(counts) -> list[int]:
    """Config indices by dataset F1 (config_f1), best first; ties go to the config earlier in grid order.
    counts: int (n_configs, 3) of (hits, n_pred, n_ref) summed over the dataset."""
    f1 = config_f1(counts)
    return [int(i) for i in np.lexsort((np.arange(f1.size), -f1))]


def infer_ali_flags(config) -> list[str]:
    """The infer_ali arguments that align with `config` (to add to its data flags)."""
    c = Config(*config)
    return ["--medfilt_width", str(int(c.medfilt_width)), "--aggr", c.aggr, "--topk", str(int(c.topk)),
            "--w_colnorm", repr(float(c.w_colnorm)), "--w_rownorm", repr(float(c.w_rownorm)),
            "--w_coverage", repr(float(c.w_coverage))]
