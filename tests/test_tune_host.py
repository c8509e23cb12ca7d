"""CPU suite: the grid of alignment settings tune_alignment sweeps (order, deduplication, validation), the ranking of
configs by dataset F1, the infer_ali flags of a config, and the refusal of CPU maps."""
import math

import numpy as np
import pytest
import torch

from whisper_char_alignment_b200 import tuning
from whisper_char_alignment_b200.metrics import get_seg_metrics
from whisper_char_alignment_b200.tuning import Config


def test_grid_order_and_mean_deduplication():
    g = tuning.expand_grid([3, 7], ["mean", "topk"], [1, 5], [(1, 1, 0), (0, 1, 0)])
    mean = lambda w: Config(w, "mean", tuning.MEAN_TOPK, *tuning.MEAN_WEIGHTS)  # noqa: E731
    want = []
    for w in (3, 7):
        want.append(mean(w))
        for wt in ((1.0, 1.0, 0.0), (0.0, 1.0, 0.0)):
            for k in (1, 5):
                want.append(Config(w, "topk", k, *wt))
    assert g == want
    assert all(type(c.w_colnorm) is float and type(c.topk) is int for c in g)
    # the default grid: 3 widths x (mean + 5 top-k values x 3 weightings)
    assert len(tuning.expand_grid([3, 5, 7], ["mean", "topk"], [1, 5, 10, 15, 20],
                                  [(1, 1, 0), (1, 0, 0), (0, 1, 0)])) == 48
    # topk before mean, repeats dropped in place, mean needs no top-k or weighting to differ
    g = tuning.expand_grid([5, 5], ["topk", "mean", "mean"], [2, 2, 1], [(1, 1, 0), (1, 1, 0)])
    assert g == [Config(5, "topk", 2, 1.0, 1.0, 0.0), Config(5, "topk", 1, 1.0, 1.0, 0.0), mean(5)]
    assert tuning.expand_grid([1], ["mean"], [0], [(0, 0, 0)]) == [mean(1)]  # topk is not read without "topk"


@pytest.mark.parametrize("bad", [
    dict(widths=[]), dict(aggrs=[]), dict(topks=[]), dict(weightings=[]),
    dict(widths=[4]), dict(widths=[0]), dict(widths=[-1]), dict(widths=[3.5]),
    dict(aggrs=["grad_norm"]), dict(aggrs=["mean", "max"]),
    dict(topks=[0]), dict(topks=[5, -1]),
    dict(weightings=[(1, -1, 0)]), dict(weightings=[(1, 1, float("nan"))]), dict(weightings=[(1, 1)]),
])
def test_grid_validation(bad):
    args = dict(widths=[3], aggrs=["mean", "topk"], topks=[1], weightings=[(1, 1, 0)])
    args.update(bad)
    with pytest.raises(ValueError):
        tuning.expand_grid(**args)


def test_rank_configs_ties_and_zero_counts():
    counts = np.array([
        (5, 10, 10),   # F1 0.5
        (8, 10, 10),   # F1 0.8
        (0, 0, 10),    # no predictions: F1 0
        (5, 10, 10),   # ties with config 0, which comes first
        (0, 0, 0),     # no counts at all: F1 0, never NaN; ties with config 2
        (7, 10, 10),   # F1 0.7
    ], dtype=np.int64)
    f1 = tuning.config_f1(counts)
    assert np.isfinite(f1).all()
    for i, (hit, n_pred, n_ref) in enumerate(counts):
        assert f1[i] == get_seg_metrics(hit, hit, n_pred, n_ref)[2]
    assert tuning.rank_configs(counts) == [1, 5, 0, 3, 2, 4]
    assert tuning.rank_configs(np.zeros((3, 3), dtype=np.int64)) == [0, 1, 2]


def test_infer_ali_flags_round_trip():
    from whisper_char_alignment_b200.cli import infer_ali

    defaults = infer_ali.parse_args(["--output_dir", "x"])
    assert (tuning.MEAN_TOPK, *tuning.MEAN_WEIGHTS) == (defaults.topk, defaults.w_colnorm, defaults.w_rownorm,
                                                        defaults.w_coverage)
    grid = tuning.expand_grid([1, 3, 9], ["mean", "topk"], [1, 10, 500],
                              [(1, 1, 0), (0.1, 1 / 3, 2.5e-7), (0, 0, 1e300)])
    for c in grid:
        a = infer_ali.parse_args(["--output_dir", "x"] + tuning.infer_ali_flags(c))
        got = Config(a.medfilt_width, a.aggr, a.topk, a.w_colnorm, a.w_rownorm, a.w_coverage)
        assert got == c and all(type(x) is type(y) for x, y in zip(got, c)), c
        assert not a.default_whisper_timing and not a.strict


def test_tune_alignment_flags():
    from whisper_char_alignment_b200.cli import infer_ali, tune_alignment

    a = vars(tune_alignment.parse_args(["--output_dir", "x"]))
    i = vars(infer_ali.parse_args(["--output_dir", "x"]))
    for k in ("model", "dataset", "scp", "output_dir", "n_mels", "aligned_unit_type", "tolerance", "strict",
              "batch_size"):
        assert a[k] == i[k], k
    assert len(tune_alignment.grid(tune_alignment.parse_args(["--output_dir", "x"]))) == 48
    a = tune_alignment.parse_args(["--output_dir", "x", "--medfilt_widths", "1", "9", "--aggrs", "topk", "--topks", "3",
                                   "--weights", "1,0.5,0", "0,0,2"])
    assert tune_alignment.grid(a) == [Config(w, "topk", 3, *wt) for w in (1, 9) for wt in ((1.0, 0.5, 0.0), (0.0, 0.0, 2.0))]
    for bad in (["--weights", "1,1"], ["--weights", "a,b,c"], ["--weights", "1,-1,0"], ["--topks", "0"],
                ["--medfilt_widths", "4"], ["--aggrs", "max"]):
        with pytest.raises(SystemExit):
            tune_alignment.parse_args(["--output_dir", "x"] + bad)


def test_cpu_maps_are_refused():
    from whisper_char_alignment_b200 import _cabi, timing
    from whisper_char_alignment_b200.tokenizer import get_tokenizer

    tk = get_tokenizer(True, language="English")
    maps = [torch.rand(2, 2, 8, 20), torch.rand(2, 2, 9, 30)]
    texts = [[tk.encode(" a")[0]], [tk.encode(" b")[0]] * 2]
    configs = [Config(7, "mean", 15, 1.0, 1.0, 0.0), Config(7, "topk", 2, 1.0, 1.0, 0.0)]
    with pytest.raises(_cabi.WcaError):
        timing.alignment_config_counts_batch({7: maps}, texts, tk, [np.array([0.1])] * 2, configs)
    with pytest.raises(AssertionError):  # as force_align_batch
        timing.alignment_config_counts_batch({7: maps}, texts, tk, [np.array([0.1])] * 2, [Config(7, "topk", 0, 1, 1, 0)])
    with pytest.raises(ValueError):
        timing.alignment_config_counts_batch({7: maps}, texts, tk, [np.array([0.1])] * 2, [Config(5, "mean", 1, 1, 1, 0)])
    with pytest.raises(ValueError):
        timing.alignment_config_counts_batch({7: maps}, texts, tk, [np.array([0.1])] * 2, [])
    assert timing.alignment_config_counts_batch({7: []}, [], tk, [], configs) == []
    assert math.isfinite(tuning.config_f1([[0, 0, 0]])[0])
