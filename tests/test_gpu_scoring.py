"""GPU suite: head scoring, top-k selection and aggregation (csrc/scores.cu) through the C ABI, against float64
references of the same operations at the shapes and values where such kernels go wrong: one and several 256-column
chunks, 32-row groups and 128-row blocks, ties, signed zeros, subnormals, NaN and infinities, kept-row ranges, selection
lists in any order.  Every output buffer sits between guard zones and must come back fully written.

Bars: scores and matrices within 1e-5 relative (north_star); with the coverage term, whose `sum max(., .5) - .5 F`
cancels, within 1e-5 of the scale before the subtraction.  Top-k is exact."""
import numpy as np
import pytest
import torch

from conftest import max_rel_err, record_measure

pytestmark = pytest.mark.gpu

RTOL = 1e-5
G = 4096               # guard elements on either side of every output
SENTINEL = 0x7FBADBAD  # bits of a NaN payload no kernel produces; as int32, not a head index
NAN, INF = float("nan"), float("inf")


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


# ------------------------------------------------------------------ float64 references (checked on the CPU against oracle/ref_path)
def ref_head_terms(a):
    """a: (..., T, F) maps -> float64 (col, row, cov) per head: sum_f ||a[:,f]||, sum_t ||a[t,:]||, sum_f max(sum_t a[t,f], .5)."""
    a = a.double()
    col = a.square().sum(-2).sqrt().sum(-1)
    row = a.square().sum(-1).sqrt().sum(-1)
    cov = a.sum(-2).clamp_min(0.5).sum(-1)  # clamp keeps NaN, like torch.maximum in metrics.py:109
    return col, row, cov


def ref_scores(terms, n_frames, w_col, w_row, w_cov):
    """Scores from ref_head_terms and, for the tolerance, the scale before the coverage subtraction.  A term is skipped
    when its weight is <= 0 or NaN (`if w > 0`, timing.py:20-32)."""
    col, row, cov = terms
    score, scale = col * 0, col * 0
    if w_col > 0:
        score, scale = score + w_col * col, scale + w_col * col
    if w_row > 0:
        score, scale = score + w_row * row, scale + w_row * row
    if w_cov > 0:
        score, scale = score - w_cov * (cov - 0.5 * n_frames), scale + w_cov * cov
    return score, scale


def ref_aggregate(maps, sel, row_begin, row_end):
    """(1/k) sum_i a_i / ||a_i[:, f]|| in float64 over the heads `sel` of maps (H, T, F), the norm over ALL T rows; rows
    [row_begin, row_end) kept (timing.py:95-102)."""
    a = maps[torch.as_tensor(np.asarray(sel, dtype=np.int64), device=maps.device)].double()
    return (a / a.square().sum(-2, keepdim=True).sqrt()).mean(0)[row_begin:row_end]


def ref_topk(scores, k):
    """Indices of the last min(k, n) of the ascending order by (score, index), NaN below every number and NaNs by index."""
    s = np.asarray(scores, dtype=np.float32)
    n, nan = len(s), np.isnan(s)
    order = np.lexsort((np.arange(n), np.where(nan, np.float32(0), s), ~nan))  # the last key is the primary one
    return order[n - min(k, n):]


# ------------------------------------------------------------------ inputs and guarded outputs
class Guarded:
    """An fp32 / int32 output of n elements between two guard zones of G elements; all of it starts as SENTINEL bits."""

    def __init__(self, n, dtype, dev):
        self.n = int(n)
        self.buf = torch.empty(self.n + 2 * G, dtype=dtype, device=dev)
        self.buf.view(torch.int32).fill_(SENTINEL)
        self.out = self.buf[G:G + self.n]

    def check(self, written):
        """written: bool (n,), the elements the call must have written; every other element must hold the sentinel.
        Returns the output on the host."""
        bits = self.buf.view(torch.int32).cpu().numpy()
        kept = bits == SENTINEL
        assert kept[:G].all() and kept[G + self.n:].all(), "a guard zone was overwritten"
        kept = kept[G:G + self.n]
        assert not kept[written].any(), f"{int(kept[written].sum())} of {int(written.sum())} output elements not written"
        assert kept[~written].all(), f"{int((~kept[~written]).sum())} elements between the outputs were written"
        return self.out.cpu().numpy()


def spans(n, offsets, lengths):
    m = np.zeros(int(n), dtype=bool)
    for o, k in zip(offsets, lengths):
        m[int(o):int(o) + int(k)] = True
    return m


def planted_softmax(gen, H, T, F, dev):
    """Softmax over frames of logits with a planted monotone peak (token t around frame (t + .5) F / T) plus noise:
    peaky like real cross-attention, with logits in [-6, 14] so that every value stays above ~1e-12, far from where fp32
    squares turn subnormal (below ~1e-19 the kernels and the fp32 reference alike lose precision)."""
    t = (torch.arange(T, device=dev, dtype=torch.float64)[:, None] + 0.5) * (F / T)
    f = torch.arange(F, device=dev, dtype=torch.float64)[None, :]
    peak = 8.0 * torch.exp(-(((f - t) / max(1.0, F / T)) ** 2))
    noise = torch.randn(H, T, F, generator=gen, device=dev, dtype=torch.float64).clamp(-4, 4)
    return (peak + 1.5 * noise).softmax(-1).float()


def nonneg_maps(gen, H, T, F, dev):
    """Non-negative maps that are not softmax rows: column sums spread over ~(0.02, 1.2), across the coverage
    threshold 0.5."""
    u = torch.rand(H, T, F, generator=gen, device=dev) * 2 + 0.01
    s = torch.rand(H, 1, F, generator=gen, device=dev) * 1.2 + 0.02
    return u * s / T


def pack_maps(maps, recs, dev):
    """Lay the (H, T, F) blocks out back to back, each starting at an odd float (rows not 16-byte aligned), with NaN in
    the gaps so that a read outside a block poisons its result.  Sets recs["ws_off"]."""
    off = 1
    for b, m in enumerate(maps):
        recs[b]["ws_off"] = off
        off += m.numel()
        off += (1 - off) % 4 if b % 2 else (3 - off) % 4
    ws = torch.full((off + 1,), NAN, device=dev)
    for b, m in enumerate(maps):
        ws[int(recs[b]["ws_off"]): int(recs[b]["ws_off"]) + m.numel()] = m.reshape(-1)
    return ws


def col_max_floor(maps):
    """The smallest column maximum of the maps, all-zero columns aside."""
    return min(float(c[c > 0].min()) for c in (m.amax(-2) for m in maps))


# ------------------------------------------------------------------ wca_head_scores
SCORE_F = [1, 31, 255, 256, 257, 511, 512, 513, 1500]
SCORE_T = [1, 2, 7, 8, 9, 15, 16, 17, 448]
SCORE_WEIGHTS = [
    (1.0, 1.0, 0.0),
    (1.0, 1.0, 0.7), (0.3, 2.0, 1.5),                       # coverage on
    (1.0, 0.0, 0.0), (0.0, 1.0, 0.0), (0.0, 0.0, 1.0),      # each term alone
    (-1.0, 1.0, 0.5), (1.0, -2.0, 0.0), (0.5, 1.0, -1.0),   # a negative weight skips its term
    (NAN, 1.0, 0.5), (1.0, NAN, 0.0), (2.0, 0.5, NAN),      # so does a NaN weight
]


def _scores_vs_fp64(shapes, kind, H, seed, dev):
    from whisper_char_alignment_b200 import _cabi

    gen = torch.Generator(device=dev).manual_seed(seed)
    make = planted_softmax if kind == "softmax" else nonneg_maps
    maps = [make(gen, H, T, F, dev) for T, F in shapes]
    assert col_max_floor(maps) >= 1e-15
    if kind == "nonneg":
        sums = torch.cat([m.sum(-2).reshape(-1) for m in maps])
        assert bool((sums < 0.5).any()) and bool((sums > 0.5).any())
    B = len(shapes)
    recs = np.zeros(B, dtype=_cabi.UTT_DTYPE)
    recs["n_tokens"], recs["n_frames"] = [t for t, _ in shapes], [f for _, f in shapes]
    recs["score_off"] = 3 + np.arange(B) * (H + 2)  # two untouched slots between utterances
    ws = pack_maps(maps, recs, dev)
    d_utts = _cabi.upload_utts(recs, dev)
    n_out = 3 + B * (H + 2)
    written = spans(n_out, recs["score_off"], [H] * B)
    terms = [torch.stack(t).cpu().numpy() for t in zip(*(ref_head_terms(m) for m in maps))]  # 3 x (B, H)
    n_frames = recs["n_frames"][:, None].astype(np.float64)
    idx = recs["score_off"][:, None] + np.arange(H)[None, :]
    for w in SCORE_WEIGHTS:
        out = Guarded(n_out, torch.float32, dev)
        _cabi.head_scores(ws.data_ptr(), d_utts, B, H, int(recs["n_tokens"].max()), int(recs["n_frames"].max()), *w, out.out)
        got = out.check(written)[idx].astype(np.float64)
        want, scale = ref_scores(terms, n_frames, *w)
        err = np.abs(got - want) / scale
        b, h = np.unravel_index(np.argmax(err), err.shape)
        assert err.max() <= RTOL, (w, shapes[b], h, got[b, h], want[b, h], err.max())
        cov = w[2] > 0
        record_measure("head_scores_coverage_vs_fp64_max_err_over_scale" if cov else "head_scores_vs_fp64_max_rel_err",
                       err.max())


@pytest.mark.parametrize("kind", ["softmax", "nonneg"])
def test_head_scores_vs_fp64(kind, dev):
    """Every (T, F) of the grids in one ragged launch: one and several 256-column chunks (per-row sums of squares in
    shared memory), the coverage term at every F, each term alone, skipped terms; then the ABI's long case, more than
    1024 token rows with rows of at most one chunk."""
    _scores_vs_fp64([(T, F) for T in SCORE_T for F in SCORE_F], kind, 3, 1, dev)
    _scores_vs_fp64([(1100, 256), (1031, 31), (2, 255), (1025, 1)], kind, 2, 2, dev)


def test_head_scores_rejects_long_rows_with_many_tokens(dev):
    """More than 1024 token rows are only accepted with rows of at most 256 frames (the per-row partial norms of longer
    rows live in a 1024-entry shared buffer).  The descriptors are small, so the launch would be harmless anyway."""
    from whisper_char_alignment_b200 import _cabi

    recs = np.zeros(2, dtype=_cabi.UTT_DTYPE)
    recs["n_tokens"], recs["n_frames"], recs["score_off"] = 10, 10, [0, 4]
    ws = torch.rand(2 * 4 * 100, device=dev)
    recs["ws_off"] = [0, 400]
    out = Guarded(8, torch.float32, dev)
    with pytest.raises(_cabi.WcaError, match="1024 token rows"):
        _cabi.head_scores(ws.data_ptr(), _cabi.upload_utts(recs, dev), 2, 4, 1025, 257, 1.0, 1.0, 0.0, out.out)
    out.check(np.zeros(8, dtype=bool))


# ------------------------------------------------------------------ wca_head_scores_from_partials
def test_scores_from_partials_vs_fp64_of_the_captured_maps(dev):
    """The scores finished from the capture kernel's partials against float64 sums of the maps that very launch wrote:
    token counts across the 32-row groups and 128-row blocks, frame counts in clusters of 1 to 8 CTAs."""
    from test_gpu_parity import _planted_qk
    from whisper_char_alignment_b200 import _cabi
    from whisper_char_alignment_b200.timing import _cluster_bucket

    L, H, W = 2, 4, 3
    n_heads, width = L * H, H * 64
    f_cycle = [40, 224, 300, 449, 700, 1111, 1500]
    t_list = [1, 31, 32, 33, 127, 128, 129, 255, 256, 257, 448]
    tf = [(T, f_cycle[(2 * i + j) % len(f_cycle)]) for i, T in enumerate(t_list) for j in range(2)]
    B = len(tf)
    q, k = _planted_qk(5, L, width, [t for t, _ in tf], 1500, dev)
    t_max = max(t for t, _ in tf)
    recs = np.zeros(B, dtype=_cabi.UTT_DTYPE)
    off = poff = 0
    for b, (T, F) in enumerate(tf):
        recs[b]["n_tokens"], recs[b]["n_frames"] = T, F
        recs[b]["q_row0"], recs[b]["k_row0"], recs[b]["ws_off"], recs[b]["part_off"] = b * t_max, b * 1500, off, poff
        recs[b]["score_off"] = 5 + b * (n_heads + 3)
        off += n_heads * T * F
        poff += _cabi.capture_partials_floats(n_heads, T, F)
    ws = torch.full((off,), NAN, device=dev)
    partials = torch.full((poff,), NAN, device=dev)
    buckets = {}
    for b, (_, F) in enumerate(tf):
        buckets.setdefault(_cluster_bucket(F), []).append(b)
    assert len(buckets) >= 5
    for _, members in sorted(buckets.items()):
        sub = recs[members]
        assert _cabi.capture_writes_partials(int(sub["n_frames"].max()), W, 0)  # the tcgen05 kernel, which writes partials
        _cabi.capture_attention(q, k, H, width, width, _cabi.upload_utts(sub, dev), len(members), int(sub["n_tokens"].max()),
                                int(sub["n_frames"].max()), W, 1.0, ws, 0, partials)
    maps = [ws[int(r["ws_off"]): int(r["ws_off"]) + n_heads * T * F].view(n_heads, T, F) for r, (T, F) in zip(recs, tf)]
    assert col_max_floor(maps) >= 1e-15
    terms = [torch.stack(t).cpu().numpy() for t in zip(*(ref_head_terms(m) for m in maps))]
    d_utts = _cabi.upload_utts(recs, dev)
    n_out = 5 + B * (n_heads + 3)
    written = spans(n_out, recs["score_off"], [n_heads] * B)
    idx = recs["score_off"][:, None] + np.arange(n_heads)[None, :]
    for w_col, w_row in ((1.0, 1.0), (0.5, 2.0), (0.0, 1.0), (1.0, 0.0)):
        out = Guarded(n_out, torch.float32, dev)
        _cabi.head_scores_from_partials(partials, d_utts, B, n_heads, w_col, w_row, out.out)
        got = out.check(written)[idx]
        want, _ = ref_scores(terms, None, w_col, w_row, 0.0)
        err = max_rel_err(got, want, atol=0, rtol=1)
        record_measure("scores_from_partials_vs_fp64_max_rel_err", err)
        b, h = np.unravel_index(np.argmax(np.abs(got - want) / want), want.shape)
        assert err <= RTOL, ((w_col, w_row), tf[b], h, got[b, h], want[b, h])


# ------------------------------------------------------------------ wca_topk_heads
def _payload_nans(n):
    return np.resize(np.array([0x7FC0BEEF, 0xFFC00001, 0x7FC00000, 0xFFC00000], dtype=np.uint32), n).view(np.float32)


def score_sets(n, rng):
    from test_gpu_parity import rand_cost

    f32 = np.float32
    nan = rng.standard_normal(n).astype(f32)
    hit = rng.random(n) < 0.3
    nan[hit] = _payload_nans(int(hit.sum()))
    return {
        "equal": rand_cost(rng, 1, n, "const")[0],
        "tie_groups": rand_cost(rng, 1, n, "ties")[0],  # normals rounded to halves
        "signed_zeros": rng.choice(np.array([0.0, -0.0, 1.0, -1.0], f32), n),
        "nan": nan,
        # NaN after and before a -inf, next to +inf and finite scores
        "inf_nan": np.resize(np.array([-INF, NAN, INF, 1.5, NAN, -INF, -0.0, -2.0, INF, NAN], f32), n),
        "subnormal": rng.choice(np.array([1e-45, -1e-45, 3e-45, 1e-40, -1e-40, 1.1754942e-38, 1.1754944e-38, 0.0, -0.0], f32), n),
        "distinct": rng.permutation(n).astype(f32) - f32(n // 2),
    }


@pytest.mark.parametrize("n_heads", [1, 6, 255, 256, 257, 384, 640, 8192])
def test_topk_heads_exact(n_heads, dev):
    """Selection and reported scores are exact: the order (NaN first, score, head index) of a stable sort, the last
    min(n_sel, n_heads) kept, the scores' bits passed through.  n_sel from 0 to n_heads + 5 in one launch; slots past
    min(n_sel, n_heads) stay untouched; sel_scores may be NULL."""
    from whisper_char_alignment_b200 import _cabi

    rng = np.random.default_rng(n_heads)
    sets = score_sets(n_heads, rng)
    n_sels = sorted({0, 1, 2, n_heads - 1, n_heads, n_heads + 5})
    cases = [(name, k) for name in sets for k in n_sels]
    B = len(cases)
    recs = np.zeros(B, dtype=_cabi.UTT_DTYPE)
    flat, soff, seloff = [], 0, 0
    for b, (name, k) in enumerate(cases):
        flat += [np.full(3, 7.0, np.float32), sets[name]]
        recs[b]["score_off"], recs[b]["sel_off"], recs[b]["n_sel"] = soff + 3, seloff + 2, k
        soff, seloff = soff + 3 + n_heads, seloff + 2 + k
    d_scores = torch.from_numpy(np.concatenate(flat)).to(dev)
    d_utts = _cabi.upload_utts(recs, dev)
    written = spans(seloff, recs["sel_off"], np.minimum(recs["n_sel"], n_heads))
    sel, sel_scores = Guarded(seloff, torch.int32, dev), Guarded(seloff, torch.float32, dev)
    _cabi.topk_heads(d_scores, d_utts, B, n_heads, sel.out, sel_scores.out)
    got, got_sc = sel.check(written), sel_scores.check(written)
    sel_only = Guarded(seloff, torch.int32, dev)
    _cabi.topk_heads(d_scores, d_utts, B, n_heads, sel_only.out, None)
    np.testing.assert_array_equal(sel_only.check(written), got)
    for b, (name, k) in enumerate(cases):
        s, o, kk = sets[name], int(recs[b]["sel_off"]), min(k, n_heads)
        want = ref_topk(s, k)
        np.testing.assert_array_equal(got[o:o + kk], want, err_msg=f"{name}, n_sel {k}")
        np.testing.assert_array_equal(got_sc[o:o + kk].view(np.int32), s[want].view(np.int32), err_msg=f"{name}, n_sel {k}")
        if kk and not np.isnan(s).any():  # the reference's own expression, timing.py:36
            kept = sorted((float(v), i) for i, v in enumerate(s))[-kk:]
            np.testing.assert_array_equal(got[o:o + kk], [i for _, i in kept], err_msg=f"{name}, n_sel {k}")


def test_topk_nan_ranks_below_minus_inf(dev):
    """The scores of heads whose maps hold +inf or NaN, coverage term only: -inf and NaN, as oracle/ref_path computes them.
    A NaN score ranks below -inf whichever of the two heads has the smaller index, and NaNs rank among themselves by
    index."""
    from oracle import ref_path
    from whisper_char_alignment_b200 import _cabi

    gen = torch.Generator().manual_seed(3)
    H, T, F = 6, 9, 300  # two 256-column chunks
    maps = (torch.randn(H, T, F, generator=gen) * 2).softmax(-1)
    maps[1, 4, 280] = INF  # head 1: -inf;  head 2: NaN (a larger index than the -inf head)
    maps[2, 0, 10] = NAN
    maps[4, 8, 0] = NAN    # head 4: NaN;   head 5: -inf (a larger index than the NaN head)
    maps[5, 2, 100] = INF
    want_scores = ref_path.head_scores(maps.view(1, H, T, F), 0.0, 0.0, 1.0).view(-1).numpy()
    assert np.isneginf(want_scores[[1, 5]]).all() and np.isnan(want_scores[[2, 4]]).all()
    recs = np.zeros(1, dtype=_cabi.UTT_DTYPE)
    recs["n_tokens"], recs["n_frames"], recs["n_sel"] = T, F, H
    d_utts = _cabi.upload_utts(recs, dev)
    scores = Guarded(H, torch.float32, dev)
    d_maps = maps.to(dev)
    _cabi.head_scores(d_maps.data_ptr(), d_utts, 1, H, T, F, 0.0, 0.0, 1.0, scores.out)
    got_scores = scores.check(np.ones(H, dtype=bool))
    np.testing.assert_array_equal(np.isnan(got_scores), np.isnan(want_scores))
    np.testing.assert_allclose(got_scores, want_scores, rtol=RTOL)
    sel = Guarded(H, torch.int32, dev)
    _cabi.topk_heads(scores.out, d_utts, 1, H, sel.out, None)
    order = sel.check(np.ones(H, dtype=bool))
    assert list(order[:4]) == [2, 4, 1, 5], order
    np.testing.assert_array_equal(order, ref_topk(got_scores, H))


# ------------------------------------------------------------------ wca_aggregate_heads
# (T, F, heads in the maps, n_sel, row_begin, row_end)
AGG_CASES = [
    (1, 1, 4, 1, 0, 1), (1, 31, 5, 2, 0, 1), (1, 32, 6, 3, 0, 1), (1, 33, 7, 4, 0, 1), (1, 1500, 9, 5, 0, 1),
    (8, 1, 9, 6, 3, 7), (8, 31, 10, 7, 1, 8), (8, 32, 12, 8, 3, 7), (8, 33, 12, 9, 0, 8), (8, 1500, 8, 1, 3, 7),
    (9, 1, 4, 2, 4, 9), (9, 31, 200, 192, 3, 7), (9, 32, 5, 3, 0, 9), (9, 33, 330, 320, 4, 8), (9, 1500, 12, 4, 3, 7),
    (448, 1, 12, 5, 3, 447), (448, 31, 7, 6, 4, 447), (448, 32, 200, 192, 4, 447), (448, 33, 9, 7, 0, 448),
    (448, 1500, 10, 9, 4, 447),
    (9, 33, 12, 4, 5, 5),  # nothing kept: nothing written
]
SHARED = [(17, 40, 12, 4, 3, 16), (448, 300, 12, 4, 3, 447)]  # these reuse the selection list of AGG_CASES[-1]
ZERO_COLUMN = {2: "every head", 13: "one selected head"}     # column 3 of these cases is all zero: 0 / 0


def _aggregate_batch(dev):
    """The AGG_CASES + SHARED utterances: maps, selection lists in random order, descriptors."""
    from whisper_char_alignment_b200 import _cabi

    gen = torch.Generator(device=dev).manual_seed(17)
    rng = np.random.default_rng(17)
    cases = AGG_CASES + SHARED
    B = len(cases)
    recs = np.zeros(B, dtype=_cabi.UTT_DTYPE)
    maps, sels, sel_flat = [], [], []
    moff, soff = 0, 0
    for b, (T, F, H, k, rb, re) in enumerate(cases):
        recs[b]["n_tokens"], recs[b]["n_frames"], recs[b]["n_sel"] = T, F, k
        recs[b]["row_begin"], recs[b]["row_end"] = rb, re
        recs[b]["matrix_off"] = moff + 7  # seven untouched elements in front of every matrix
        moff += 7 + (re - rb) * F
        if b < len(AGG_CASES):
            sel = rng.permutation(H)[:k].astype(np.int32)
            if k > 1 and (np.diff(sel) > 0).all():
                sel = sel[::-1].copy()
            recs[b]["sel_off"] = soff + 1
            sel_flat += [np.full(1, -1, np.int32), sel]
            soff += 1 + k
        else:
            src = len(AGG_CASES) - 1
            assert cases[src][2] <= H and cases[src][3] == k
            sel, recs[b]["sel_off"] = sels[src], recs[src]["sel_off"]
        sels.append(sel)
        m = planted_softmax(gen, H, T, F, dev)
        m[:, :rb] *= 50  # the rows that are not kept carry most of each column's norm
        m[:, re:] *= 50
        if ZERO_COLUMN.get(b) == "every head":
            m[:, :, 3] = 0
        elif b in ZERO_COLUMN:
            m[int(sel[0]), :, 3] = 0
        maps.append(m)
    ws = pack_maps(maps, recs, dev)
    return cases, recs, maps, sels, ws, torch.from_numpy(np.concatenate(sel_flat)).to(dev), moff


def test_aggregate_heads_vs_fp64_and_single_heads(dev):
    """The (N, F) matrices of one ragged launch against float64, per element within 1e-5 relative, NaN exactly where torch
    fp32 `a / a.norm(dim=-2)` has it; then bit for bit: (a) the grouped kernel equals the fp32 sum, in list order, of the
    same heads aggregated one at a time, over n_sel; (b) single-head descriptors give the same bits under max_sel 1 and 4;
    (c) every utterance launched alone gives the bits it gets inside the batch."""
    from whisper_char_alignment_b200 import _cabi

    cases, recs, maps, sels, ws, d_sel, n_out = _aggregate_batch(dev)
    assert col_max_floor(maps) >= 1e-15
    B = len(cases)
    max_t, max_f = int(recs["n_tokens"].max()), int(recs["n_frames"].max())
    n_rows = recs["row_end"] - recs["row_begin"]
    written = spans(n_out, recs["matrix_off"], n_rows * recs["n_frames"])
    out = Guarded(n_out, torch.float32, dev)
    _cabi.aggregate_heads(ws.data_ptr(), d_sel, _cabi.upload_utts(recs, dev), B, max_t, max_f, out.out,
                          max_sel=int(recs["n_sel"].max()))
    got = out.check(written)

    def block(flat, r):
        o, n = int(r["matrix_off"]), int(r["row_end"] - r["row_begin"])
        return flat[o:o + n * int(r["n_frames"])].reshape(n, int(r["n_frames"]))

    worst = 0.0
    for b, (T, F, H, k, rb, re) in enumerate(cases):
        g = block(got, recs[b])
        want = ref_aggregate(maps[b], sels[b], rb, re).cpu().numpy()
        st = maps[b][torch.as_tensor(sels[b].astype(np.int64), device=dev)]
        nan_fp32 = torch.isnan((st / st.norm(dim=-2, keepdim=True)).mean(0)[rb:re]).cpu().numpy()
        np.testing.assert_array_equal(np.isnan(g), nan_fp32, err_msg=f"NaN pattern, case {cases[b]}")
        assert nan_fp32.any() == (b in ZERO_COLUMN)
        err = max_rel_err(g[~nan_fp32], want[~nan_fp32], atol=1e-30, rtol=1)
        assert err <= RTOL, (cases[b], err)
        worst = max(worst, err)
    record_measure("aggregate_heads_vs_fp64_max_rel_err", worst)

    # (a) + (b): every selected head alone, n_sel = 1, its sel_off pointing into the utterance's list
    singles = np.repeat(recs, recs["n_sel"])
    singles["n_sel"] = 1
    singles["sel_off"] = np.concatenate([np.arange(k) + r["sel_off"] for r in recs for k in [int(r["n_sel"])]])
    one_rows = singles["row_end"] - singles["row_begin"]
    singles["matrix_off"] = np.concatenate([[0], np.cumsum(one_rows * singles["n_frames"])[:-1]])
    n_one = int((one_rows * singles["n_frames"]).sum())
    d_singles = _cabi.upload_utts(singles, dev)
    one = {}
    for max_sel in (1, 4):
        o = Guarded(n_one, torch.float32, dev)
        _cabi.aggregate_heads(ws.data_ptr(), d_sel, d_singles, len(singles), max_t, max_f, o.out, max_sel=max_sel)
        one[max_sel] = o.check(spans(n_one, singles["matrix_off"], one_rows * singles["n_frames"]))
    np.testing.assert_array_equal(one[1].view(np.int32), one[4].view(np.int32))
    i = 0
    for b, r in enumerate(recs):
        acc = None
        for _ in range(int(r["n_sel"])):
            m = block(one[1], singles[i])
            acc = m.copy() if acc is None else acc + m  # float32 adds, in list order
            i += 1
        np.testing.assert_array_equal(block(got, r), acc / np.float32(r["n_sel"]), err_msg=f"case {cases[b]}")

    # (c) alone, with its own maxima (and the single-head kernel where n_sel = 1)
    for b, r in enumerate(recs):
        o = Guarded(n_out, torch.float32, dev)
        _cabi.aggregate_heads(ws.data_ptr(), d_sel, _cabi.upload_utts(recs[b:b + 1], dev), 1, int(r["n_tokens"]),
                              int(r["n_frames"]), o.out, max_sel=int(r["n_sel"]))
        alone = o.check(spans(n_out, [r["matrix_off"]], [int(r["row_end"] - r["row_begin"]) * int(r["n_frames"])]))
        np.testing.assert_array_equal(block(alone, r).view(np.int32), block(got, r).view(np.int32), err_msg=f"case {cases[b]}")


# ------------------------------------------------------------------ the three stages, alone and in a batch
def test_an_utterance_alone_equals_the_same_utterance_in_a_batch(dev):
    """Scores (coverage on), selection and matrix of every utterance are bit-identical whether it is launched alone or
    inside a ragged batch whose max_tokens / max_frames are larger."""
    from whisper_char_alignment_b200 import _cabi

    H = 16
    shapes = [(448, 1500), (9, 31), (130, 257), (300, 1111), (1, 1), (17, 513)]
    n_sel = [5, 1, 16, 9, 3, 13]  # at most H: the aggregation reads exactly the entries the selection wrote
    gen = torch.Generator(device=dev).manual_seed(29)
    maps = [planted_softmax(gen, H, T, F, dev) for T, F in shapes]
    B = len(shapes)
    recs = np.zeros(B, dtype=_cabi.UTT_DTYPE)
    recs["n_tokens"], recs["n_frames"], recs["n_sel"] = [t for t, _ in shapes], [f for _, f in shapes], n_sel
    recs["row_begin"] = [4, 0, 4, 4, 0, 4]
    recs["row_end"] = [447, 9, 129, 299, 1, 16]
    recs["score_off"] = 1 + np.arange(B) * (H + 1)
    recs["sel_off"] = np.concatenate([[1], 1 + np.cumsum(np.asarray(n_sel) + 1)[:-1]])
    n_rows = recs["row_end"] - recs["row_begin"]
    recs["matrix_off"] = np.concatenate([[1], 1 + np.cumsum(n_rows * recs["n_frames"] + 1)[:-1]])
    ws = pack_maps(maps, recs, dev)
    n_sc, n_sl = 1 + B * (H + 1), int(recs["sel_off"][-1] + n_sel[-1])
    n_mx = int(recs["matrix_off"][-1] + n_rows[-1] * recs["n_frames"][-1])

    def run(sub):
        sc, sl, ss, mx = (Guarded(n_sc, torch.float32, dev), Guarded(n_sl, torch.int32, dev),
                          Guarded(n_sl, torch.float32, dev), Guarded(n_mx, torch.float32, dev))
        d = _cabi.upload_utts(sub, dev)
        mt, mf = int(sub["n_tokens"].max()), int(sub["n_frames"].max())
        _cabi.head_scores(ws.data_ptr(), d, len(sub), H, mt, mf, 1.0, 0.5, 0.8, sc.out)
        _cabi.topk_heads(sc.out, d, len(sub), H, sl.out, ss.out)
        _cabi.aggregate_heads(ws.data_ptr(), sl.out, d, len(sub), mt, mf, mx.out, max_sel=int(sub["n_sel"].max()))
        sub_n = sub["row_end"] - sub["row_begin"]
        return (sc.check(spans(n_sc, sub["score_off"], [H] * len(sub))).view(np.int32),
                sl.check(spans(n_sl, sub["sel_off"], sub["n_sel"])),
                ss.check(spans(n_sl, sub["sel_off"], sub["n_sel"])).view(np.int32),
                mx.check(spans(n_mx, sub["matrix_off"], sub_n * sub["n_frames"])).view(np.int32))

    batch = run(recs)
    for b, r in enumerate(recs):
        alone = run(recs[b:b + 1])
        for name, o, n, a, w in zip(("scores", "sel", "sel_scores", "matrix"),
                                    (r["score_off"], r["sel_off"], r["sel_off"], r["matrix_off"]),
                                    (H, r["n_sel"], r["n_sel"], n_rows[b] * r["n_frames"]), alone, batch):
            np.testing.assert_array_equal(a[int(o):int(o) + int(n)], w[int(o):int(o) + int(n)], err_msg=f"{name}, utterance {b}")

