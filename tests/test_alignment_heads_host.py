"""CPU suite: alignment-head masks (upstream's dump format, ranking by dataset F1, Whisper.set_alignment_heads), the
host word ids of the strict scoring, the array sum over ranks, and the flags of find_alignment_heads and
infer_ali --alignment_heads."""
import base64
import gzip
import json
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from whisper_char_alignment_b200 import heads, sharding
from whisper_char_alignment_b200.metrics import eval_n1_strict, get_seg_metrics


# ------------------------------------------------------------------ dump format
@pytest.mark.parametrize("shape", [(1, 1), (2, 2), (24, 16), (32, 20)])
def test_mask_round_trips_and_reads_upstream_dumps(shape):
    rng = np.random.default_rng(shape[0] * 100 + shape[1])
    for _ in range(5):
        mask = rng.random(shape) < 0.3
        dump = heads.encode_alignment_heads(mask)
        assert isinstance(dump, bytes) and dump == heads.encode_alignment_heads(mask)  # no time stamp in the bytes
        np.testing.assert_array_equal(heads.decode_alignment_heads(dump, *shape), mask)
        np.testing.assert_array_equal(heads.decode_alignment_heads(dump.decode("ascii"), *shape), mask)
        # upstream's recipe, gzip header time stamp included
        upstream = base64.b85encode(gzip.compress(mask.tobytes()))
        np.testing.assert_array_equal(heads.decode_alignment_heads(upstream, *shape), mask)
    with pytest.raises(ValueError):
        heads.decode_alignment_heads(heads.encode_alignment_heads(np.zeros(shape, bool)), shape[0] + 1, shape[1])


def test_set_alignment_heads_on_a_cpu_product_model():
    from whisper_char_alignment_b200.whisper_model import ModelDimensions, TEST_SIZES, Whisper

    model = Whisper(ModelDimensions(*TEST_SIZES["mini"]))
    L, H = model.dims.n_text_layer, model.dims.n_text_head
    mask = np.zeros((L, H), dtype=bool)
    mask[0, 1] = mask[2, 3] = mask[1, 0] = True
    model.set_alignment_heads(base64.b85encode(gzip.compress(mask.tobytes())))
    got = model.alignment_heads
    assert got.is_sparse and got.device.type == "cpu"
    assert torch.equal(got.to_dense(), torch.from_numpy(mask))
    assert got.indices().T.tolist() == [[0, 1], [1, 0], [2, 3]]  # the (layer, head) order default_find_alignment stacks
    assert "alignment_heads" not in model.state_dict()  # still a non-persistent buffer
    with pytest.raises(ValueError):
        model.set_alignment_heads(heads.encode_alignment_heads(np.ones((L + 1, H), bool)))


# ------------------------------------------------------------------ ranking
def test_rank_heads_on_a_hand_made_table():
    counts = np.zeros((3, 2, 3), dtype=np.int64)
    counts[..., 2] = 10  # 10 reference boundaries everywhere
    counts[0, 0] = (5, 10, 10)  # F1 0.5
    counts[0, 1] = (8, 10, 10)  # F1 0.8
    counts[1, 0] = (5, 10, 10)  # ties with (0, 0): the lower flat index wins
    counts[1, 1] = (0, 0, 10)   # no predictions: F1 0
    counts[2, 0] = (7, 10, 10)  # F1 0.7
    counts[2, 1] = (0, 0, 0)    # no counts at all: F1 0, never NaN; ties with (1, 1), which comes first
    f1 = heads.head_f1(counts)
    assert np.isfinite(f1).all()
    for l in range(3):
        for h in range(2):
            hit, n_pred, n_ref = counts[l, h]
            assert f1[l, h] == get_seg_metrics(hit, hit, n_pred, n_ref)[2]
    expect = [[(0, 1)], [(0, 1), (2, 0)], [(0, 0), (0, 1), (2, 0)], [(0, 0), (0, 1), (1, 0), (2, 0)],
              [(0, 0), (0, 1), (1, 0), (1, 1), (2, 0)]]
    for k, want in enumerate(expect, start=1):
        assert [tuple(x) for x in np.argwhere(heads.rank_heads(counts, k))] == want, k
    assert heads.rank_heads(counts, 100).all()
    with pytest.raises(ValueError):
        heads.rank_heads(counts, 0)


# ------------------------------------------------------------------ strict word ids
def test_word_ids_follow_eval_n1_strict_normalisation():
    from whisper_char_alignment_b200.timing import strict_word_ids

    words = ["Hello", "hello,", "'hello'", "HELLO!!", "hel-lo", "world", "World.", "", "...", "-", "don't", "Don't",
             "dont", "naïve", "NAÏVE", "a.b", "A.B.", " x", "x "]
    rng = np.random.default_rng(3)
    extra = ["".join(rng.choice(list("aAbB.,!'- "), size=int(rng.integers(0, 5)))) for _ in range(60)]
    words = words + extra
    a, b = strict_word_ids([words[:40], words[40:]])
    ids = np.concatenate([a, b])
    assert a.dtype == np.int32
    for i, wi in enumerate(words):
        for j, wj in enumerate(words):
            tp, _, _ = eval_n1_strict([0.0], [0.0], [wi], [wj], 0.0)
            assert (ids[i] == ids[j]) == (tp == 1), (wi, wj)


# ------------------------------------------------------------------ array sum over ranks
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sum_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        local = np.arange(24 * 16 * 3, dtype=np.int64).reshape(24, 16, 3) * (rank + 1) + (1 << 40) * rank
        tot = sharding.sum_over_ranks(local)
        want = sum(np.arange(24 * 16 * 3, dtype=np.int64).reshape(24, 16, 3) * (r + 1) + (1 << 40) * r for r in range(world))
        assert tot.dtype == np.int64 and tot.shape == (24, 16, 3)
        np.testing.assert_array_equal(tot, want)
        assert sharding.gather_counters(rank + 1, 10 * rank, 7) == (3, 10, 14)
        assert type(sharding.gather_counters(1, 2, 3)[0]) is int
        open(os.path.join(out_dir, f"sum{rank}"), "w").close()
    finally:
        dist.destroy_process_group()


def test_two_rank_array_sum(tmp_path):
    mp.spawn(_sum_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert all((tmp_path / f"sum{r}").exists() for r in range(2))


def test_single_process_array_sum_is_a_copy():
    a = np.array([[1, 2, 3]], dtype=np.int64)
    got = sharding.sum_over_ranks(a)
    np.testing.assert_array_equal(got, a)
    got[0, 0] = 9
    assert a[0, 0] == 1
    assert sharding.gather_counters(1, 2, 3) == (1, 2, 3)


# ------------------------------------------------------------------ flags
def test_find_alignment_heads_flags():
    from whisper_char_alignment_b200.cli import find_alignment_heads, infer_ali

    a = vars(find_alignment_heads.parse_args(["--output_dir", "x"]))
    i = vars(infer_ali.parse_args(["--output_dir", "x"]))
    for k in ("model", "dataset", "scp", "output_dir", "n_mels", "medfilt_width", "aligned_unit_type", "tolerance",
              "strict", "batch_size"):
        assert a[k] == i[k], k
    assert a["n_heads"] == 10
    with pytest.raises(SystemExit):
        find_alignment_heads.parse_args(["--output_dir", "x", "--n_heads", "0"])


def test_infer_ali_alignment_heads_flag(tmp_path):
    from whisper_char_alignment_b200.cli import infer_ali

    assert "alignment_heads" not in vars(infer_ali.parse_args(["--output_dir", "x", "--default_whisper_timing"]))
    with pytest.raises(SystemExit):  # only the stock-Whisper path aligns on the model's heads
        infer_ali.parse_args(["--output_dir", "x", "--alignment_heads", "abc"])
    a = infer_ali.parse_args(["--output_dir", "x", "--default_whisper_timing", "--alignment_heads", "abc"])
    assert a.alignment_heads == "abc"
    mask = np.zeros((2, 2), dtype=bool)
    mask[1, 0] = True
    dump = heads.encode_alignment_heads(mask)
    f = tmp_path / "x-heads.json"
    f.write_text(json.dumps({"mask": dump.decode("ascii"), "alignment_heads": [[1, 0]]}))
    assert infer_ali.alignment_heads_dump(str(f)) == dump
    assert infer_ali.alignment_heads_dump(dump.decode("ascii")) == dump
