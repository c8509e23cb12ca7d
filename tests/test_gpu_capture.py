"""GPU suite: the capture kernel (wca_capture_attention: csrc/capture_tc.cu, and for the other widths or on request the
CUDA-core logits of capture_simt.cu + the filter of medfilt_softmax.cu) against a float64 reference of the same
operation, on inputs built to reach its rare paths: rows whose maximum climbs past the lazy softmax reference of the
tcgen05 epilogue (2^32: the blocks already in tensor memory are rescaled in place), a step of exactly 32 log2 units and
one ulp either side of it, maxima in the last partial block, at the first and last frame and inside a mirrored copy or
cluster rank other than the first, falling rows that underflow, negative and zero qk_scale, the CUDA-core widths 9-31,
NaN / inf / 1e30 in every Q and K row around the utterances.  Every output starts as NaN and must come back written.

Q / K are constructed so that the logits are known: per head, three directions on disjoint groups of 8 dimensions
(entries +-x, exact tf32 values, so the tensor core multiplies them exactly) and a little noise on the other 32.
A row's logits are then sum_j a[t, j] b_j(f) + noise with b_0(f) = f - F // 2 (a ramp), b_1 = a plateau of 4 frames
whose place depends on the head, b_2(f) = [f >= 16] (a step at the second 16-frame block).

Bars: maps within 1e-4 relative of float64 where the reference is >= 1e-30 (north_star), rows summing to 1 within 1e-5;
below 1e-30 (ex2.approx.ftz flushes under 2^-126) an element must lie in [0, ref + 1e-30].  Scores finished from the
partials within 1e-5 relative of float64 scores of the float64 maps."""
import numpy as np
import pytest
import torch
import torch.nn.functional as tnf

from conftest import record_measure
from test_gpu_scoring import Guarded, ref_head_terms, ref_scores, spans

pytestmark = pytest.mark.gpu

MAP_RTOL = 1e-4
SUM_TOL = 1e-5
SCORE_RTOL = 1e-5
TINY = 1e-30
NAN, INF = float("nan"), float("inf")

L, H = 2, 2                     # two decoder layers of two heads: four (layer, head) maps per utterance
G = L * H
WIDTH = H * 64
LD_Q, Q_COL = 2 * WIDTH + 4, WIDTH       # Q: a column slice of a wider, oddly pitched buffer
LD_K, K_COL = 4 * WIDTH, 2 * WIDTH       # K: the K half of a fused [K|V] projection of two layers
Q_GAP, K_GAP = 7, 300                    # rows between utterances (after Q's last 128-row tile / after K's last frame)

GRID_T = [1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 448]
GRID_F = [1, 3, 16, 17, 223, 224, 225, 448, 449, 1344, 1345, 1500]
KINDS = ("ramp_up", "ramp_down", "plateau", "step_32", "step_32_up", "step_32_down", "noise", "ramp_plateau")


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


# ------------------------------------------------------------------ float64 reference (checked on the CPU against oracle/ref_path)
def median_reflect(x, width):
    """Median over windows of `width` frames, reflect padding inside the row; identity when F <= width // 2."""
    half = width // 2
    F = x.shape[-1]
    if width == 1 or F <= half:
        return x
    padded = tnf.pad(x.reshape(1, -1, F), (half, half), mode="reflect")[0]
    return padded.unfold(-1, width, 1).sort(dim=-1)[0][..., half].reshape(x.shape)


def ref_logits(q, k):
    """q: (T, n_heads * 64), k: (F, n_heads * 64) fp32 rows -> (n_heads, T, F) float64 logits q.k / 8."""
    T, F = q.shape[0], k.shape[0]
    qh = q.double().reshape(T, -1, 64).transpose(0, 1)
    kh = k.double().reshape(F, -1, 64).transpose(0, 1)
    return qh @ kh.transpose(-1, -2) / 8


def ref_capture(q, k, width, qk_scale):
    """softmax_f(median_width(q.k / 8) * qk_scale) in float64: (n_heads, T, F)."""
    return (median_reflect(ref_logits(q, k), width) * qk_scale).softmax(-1)


# ------------------------------------------------------------------ constructed Q / K
def tf32(x):
    """x truncated to a tf32 value (10 mantissa bits), which the tensor core reads without loss."""
    return (np.asarray(x, np.float32).view(np.int32) & np.int32(~0x1FFF)).view(np.float32)


def scale2_f32(qk_scale):
    """The kernel's factor from raw q.k to log2 units: (qk_scale * 2^-3) * log2(e), in fp32."""
    return np.float32(np.float32(qk_scale) * np.float32(0.125)) * np.float32(1.4426950408889634)


def threshold_steps(qk_scale):
    """Raw q.k values X whose block maximum y = fl(X * scale2) lands at / just above / just below 32 (the reference of
    the first block is 0): (X with y <= 32 and next(X) above, that next X, the X below the first)."""
    s2 = scale2_f32(qk_scale)
    sign = np.float32(1.0 if s2 > 0 else -1.0)
    x = np.float32(32.0 / abs(float(s2)))
    prod = lambda v: np.float32(sign * v) * s2  # noqa: E731
    while prod(x) > np.float32(32):
        x = np.nextafter(x, np.float32(0))
    while prod(np.nextafter(x, np.float32(INF))) <= np.float32(32):
        x = np.nextafter(x, np.float32(INF))
    up, down = np.nextafter(x, np.float32(INF)), np.nextafter(x, np.float32(0))
    assert prod(up) > 32 and prod(x) <= 32 and prod(down) < 32
    return sign * x, sign * up, sign * down


def exact_pieces(x):
    """Three tf32 values whose sum is the fp32 x exactly (every partial sum too)."""
    x = np.float32(x)
    a = tf32(x)
    r = np.float32(x - a)
    b = tf32(r)
    c = np.float32(r - b)
    assert tf32(c) == c and np.float32(np.float32(a + b) + c) == x
    return [a, b, c]


def row_kinds(T):
    """(T, G) index into KINDS: every warp of token rows holds every kind, so some lanes rescale and others do not."""
    return (np.arange(T)[:, None] + np.arange(G)[None, :]) % len(KINDS)


def plateau_start(F, g):
    """The plateau of (layer, head) g: at the last frames (the last, partial block), the first frames, 5/8 and 3/8 of the
    row (a mirrored copy or cluster rank other than the first)."""
    p = [F - 4, 0, 5 * F // 8, 3 * F // 8][g]
    return min(max(p, 0), max(F - 4, 0))


def make_qk_rows(T, F, qk_scale, gen, signs):
    """Q (T, G, 64) and K (F, G, 64) float32 of one utterance, on the CPU.  The profiles are set in nats of the scaled
    logits y = qk_scale * logit (for qk_scale 0 as for 1): they do not depend on the scale."""
    S = abs(qk_scale) if qk_scale != 0 else 1.0
    kinds = row_kinds(T)
    # nats per frame: a rise of <= 100 nats along the row keeps |y| <= 50 (the tensor core's fp32 accumulation loses
    # bits in proportion to the logit's size: at |y| ~ 125 the maps were ~1e-4 off float64 already)
    slope = min(1.5, 100.0 / F)
    a = np.zeros((T, G, 3, 8), np.float32)  # per direction and dimension
    a[:, :, 0, :] = tf32(np.select([kinds == 0, kinds == 1, kinds == 2, kinds == 7],
                                   [slope, -slope, 0.02, slope / 2], 0.0) / S)[..., None]
    a[:, :, 1, :] = tf32(np.select([kinds == 2, kinds == 7], [30.0, 15.0], 0.0) / S)[..., None]
    if qk_scale != 0:
        for kind, x in zip((3, 4, 5), threshold_steps(qk_scale)):
            a[:, :, 2, :3][kinds == kind] = exact_pieces(x)
    q_noise = np.where((kinds >= 3) & (kinds <= 5), 0.0, 0.28 / S).astype(np.float32)
    f = np.arange(F)
    b = np.zeros((F, G, 3), np.float32)
    b[:, :, 0] = (f - F // 2)[:, None]
    for g in range(G):
        p = plateau_start(F, g)
        b[p:p + 4, g, 1] = 1.0
    b[:, :, 2] = (f >= 16)[:, None]
    q = np.zeros((T, G, 64), np.float32)
    k = np.zeros((F, G, 64), np.float32)
    q[:, :, :24] = (a * signs[None, :, :, :]).reshape(T, G, 24)
    k[:, :, :24] = (b[..., None] * signs[None, :, :, :]).reshape(F, G, 24)
    q[:, :, 32:] = torch.randn(T, G, 32, generator=gen).numpy() * q_noise[..., None]
    k[:, :, 32:] = torch.randn(F, G, 32, generator=gen).numpy()
    return q, k


def poison_values(kind, shape, gen):
    if kind == "finite":
        return torch.randn(shape, generator=gen) * 3
    if kind == "nan":
        return torch.full(shape, NAN)
    assert kind == "inf_big"
    cycle = torch.tensor([INF, -INF, 1e30, -1e30])
    return cycle[torch.arange(int(np.prod(shape))) % 4].reshape(shape)


class Batch:
    """Q / K of the utterances `shapes`, packed into strided per-layer buffers whose every other element (other columns,
    rows between and after the utterances, rows past the last token of a 128-row tile) holds `poison`; descriptors with
    odd q_row0 / k_row0 and ws_off, partial offsets."""

    def __init__(self, shapes, qk_scale, dev, seed=0, poison="finite"):
        from whisper_char_alignment_b200 import _cabi

        self.shapes, self.qk_scale = list(shapes), qk_scale
        gen = torch.Generator().manual_seed(seed)
        signs = np.where(torch.rand(G, 3, 8, generator=gen).numpy() < 0.5, -1.0, 1.0).astype(np.float32)
        B = len(self.shapes)
        recs = np.zeros(B, dtype=_cabi.UTT_DTYPE)
        qr, kr, off, poff = 3, 5, 1, 2
        for b, (T, F) in enumerate(self.shapes):
            r = recs[b]
            r["n_tokens"], r["n_frames"], r["q_row0"], r["k_row0"], r["ws_off"], r["part_off"] = T, F, qr, kr, off, poff
            r["score_off"] = 1 + b * (G + 1)
            qr += -(-T // 128) * 128 + Q_GAP
            kr += F + K_GAP
            off += G * T * F + (b % 3)
            poff += _cabi.capture_partials_floats(G, T, F) + 1
        self.recs, self.n_ws, self.n_part, self.n_scores = recs, off + 1, poff, 1 + B * (G + 1)
        self.rows = []  # (q (T, G, 64), k (F, G, 64)) per utterance
        qbuf = [poison_values(poison, (qr + 64, LD_Q), gen) for _ in range(L)]
        kbuf = [poison_values(poison, (kr, LD_K), gen) for _ in range(L)]
        data_gen = torch.Generator().manual_seed(seed + 1)  # the same utterances whatever the poison
        for b, (T, F) in enumerate(self.shapes):
            q, k = make_qk_rows(T, F, qk_scale, data_gen, signs)
            self.rows.append((q, k))
            q0, k0 = int(recs[b]["q_row0"]), int(recs[b]["k_row0"])
            for l in range(L):
                qbuf[l][q0:q0 + T, Q_COL:Q_COL + WIDTH] = torch.from_numpy(q[:, l * H:(l + 1) * H].reshape(T, WIDTH))
                kbuf[l][k0:k0 + F, K_COL:K_COL + WIDTH] = torch.from_numpy(k[:, l * H:(l + 1) * H].reshape(F, WIDTH))
        self.qbuf = [t.to(dev) for t in qbuf]
        self.kbuf = [t.to(dev) for t in kbuf]
        self.q = [t[:, Q_COL:Q_COL + WIDTH] for t in self.qbuf]
        self.k = [t[:, K_COL:K_COL + WIDTH] for t in self.kbuf]
        self.dev = dev

    def map_of(self, flat, b):
        T, F = self.shapes[b]
        o = int(self.recs[b]["ws_off"])
        return flat[o:o + G * T * F].reshape(G, T, F)

    def ws_written(self):
        return spans(self.n_ws, self.recs["ws_off"], [G * T * F for T, F in self.shapes])

    def partials_written(self, members=None):
        """The partial slots the tcgen05 epilogue writes: per (layer, head), token block and 32-row group holding tokens, the
        row term and the F column sums of squares."""
        m = np.zeros(self.n_part, dtype=bool)
        for b in (range(len(self.shapes)) if members is None else members):
            T, F = self.shapes[b]
            base, tbu = int(self.recs[b]["part_off"]), -(-T // 128)
            for lh in range(G):
                for tb in range(tbu):
                    for grp in range(-(-min(128, T - 128 * tb) // 32)):
                        m[base + (lh * tbu + tb) * 4 + grp] = True
                        c = base + G * tbu * 4 + ((lh * tbu + tb) * 4 + grp) * F
                        m[c:c + F] = True
        return m

    def reference(self, b, width):
        """float64 (G, T, F) maps of utterance b and its median-filtered logits."""
        q, k = (torch.from_numpy(x).to(self.dev) for x in self.rows[b])
        T, F = self.shapes[b]
        med = torch.cat([median_reflect(ref_logits(q[:, l * H:(l + 1) * H].reshape(T, WIDTH),
                                                   k[:, l * H:(l + 1) * H].reshape(F, WIDTH)), width) for l in range(L)])
        return (med * self.qk_scale).softmax(-1), med


def capture(batch, width, flags=0, partials=True, members=None, max_tokens=None, max_frames=None, by_bucket=True):
    """wca_capture_attention over the utterances `members` (all by default), one launch per cluster bucket (or one in
    all), into fresh guarded outputs.  Returns (ws, partials) on the host (partials None when not written)."""
    from whisper_char_alignment_b200 import _cabi
    from whisper_char_alignment_b200.timing import _cluster_bucket

    members = list(range(len(batch.shapes))) if members is None else list(members)
    ws = Guarded(batch.n_ws, torch.float32, batch.dev)
    part = Guarded(batch.n_part, torch.float32, batch.dev) if partials else None
    groups = {}
    for b in members:
        groups.setdefault(_cluster_bucket(batch.shapes[b][1]) if by_bucket else 0, []).append(b)
    for _, grp in sorted(groups.items()):
        sub = batch.recs[grp]
        mt = int(sub["n_tokens"].max()) if max_tokens is None else max_tokens
        mf = int(sub["n_frames"].max()) if max_frames is None else max_frames
        assert _cabi.capture_writes_partials(mf, width, flags) == (partials and True)
        _cabi.capture_attention(batch.q, batch.k, H, LD_Q, LD_K, _cabi.upload_utts(sub, batch.dev), len(grp), mt, mf, width,
                                batch.qk_scale, ws.out, flags, part.out if partials else None)
    written = spans(batch.n_ws, batch.recs["ws_off"][members], [G * T * F for T, F in (batch.shapes[b] for b in members)])
    got_ws = ws.check(written)
    got_part = part.check(batch.partials_written(members)) if partials else None
    return got_ws, got_part


# ------------------------------------------------------------------ the lazy reference, emulated
def part_ranges(T, F, csize):
    """[(token rows, (f_lo, f_hi))]: the frame range each epilogue thread of the tcgen05 kernel sweeps with its own
    reference, per 128-row token block, cluster rank and mirrored copy (decode_tile / epilogue_tile)."""
    slab = (-(-F // csize) + 15) // 16 * 16
    out = []
    for t0 in range(0, T, 128):
        rv = min(128, T - t0)
        copies = 4 if rv <= 32 else (2 if rv <= 64 else 1)
        for rank in range(csize):
            f0, f1 = rank * slab, min(F, rank * slab + slab)
            nb = -(-(f1 - f0) // 16) if f1 > f0 else 0
            for p in range(copies):
                lo, hi = -(-nb * p // copies), -(-nb * (p + 1) // copies)
                if lo < hi:
                    out.append(((t0, t0 + rv), (f0 + 16 * lo, min(f1, f0 + 16 * hi))))
    return out


def count_reference_moves(med, qk_scale, csize):
    """Per row of med (G, T, F float64 filtered logits), how often the kernel's lazy reference moves: its block maxima of
    y = fl(fl(8 med) * scale2) over each thread's blocks, a move when one exceeds the reference by more than 32."""
    s2 = float(scale2_f32(qk_scale))
    y = (med * 8).float() * s2
    _, T, F = y.shape
    moves = torch.zeros(G, T, dtype=torch.int32, device=y.device)
    for (t0, t1), (f0, f1) in part_ranges(T, F, csize):
        seg = y[:, t0:t1, f0:f1]
        nb = -(-(f1 - f0) // 16)
        seg = tnf.pad(seg, (0, nb * 16 - (f1 - f0)), value=-INF).reshape(G, t1 - t0, nb, 16).amax(-1)
        m = seg[..., 0]
        for i in range(1, nb):
            need = seg[..., i] > m + 32
            m = torch.where(need, seg[..., i], m)
            moves[:, t0:t1] += need.int()
    return moves


# ------------------------------------------------------------------ comparison
def compare_maps(got, ref):
    """got (float32) against ref (float64) maps, same shape, on the device: (max relative error where ref >= 1e-30,
    max |row sum - 1|); asserts the bound below 1e-30."""
    got = got.double()
    big = ref >= TINY
    rel = ((got - ref).abs() / ref.clamp_min(TINY))[big]
    small_got, small_ref = got[~big], ref[~big]
    assert bool(torch.isfinite(got).all()), "non-finite map element"
    assert bool((small_got >= 0).all()) and bool((small_got <= small_ref + TINY).all()), \
        f"below 1e-30: max excess {float((small_got - small_ref).max()):.3e}"
    return (float(rel.max()) if rel.numel() else 0.0), float((got.sum(-1) - 1).abs().max())


def check_batch(batch, ws, width, label, measure):
    """Every utterance's maps of ws (host, flat) against float64; returns {b: (G, T, F) float64 reference}."""
    worst = (0.0, 0.0)
    refs = {}
    for b, (T, F) in enumerate(batch.shapes):
        ref, _ = batch.reference(b, width)
        got = torch.from_numpy(batch.map_of(ws, b)).to(batch.dev)
        rel, dsum = compare_maps(got, ref)
        assert rel <= MAP_RTOL, (label, (T, F), rel)
        assert dsum <= SUM_TOL, (label, (T, F), dsum)
        worst = (max(worst[0], rel), max(worst[1], dsum))
        refs[b] = ref
    record_measure(f"{measure}_max_rel_err", worst[0])
    record_measure(f"{measure}_row_sum_max_err", worst[1])
    return refs, worst


def check_scores(batch, part, refs, members, label):
    """wca_head_scores_from_partials of the kernel's partials against float64 scores of the float64 maps."""
    from whisper_char_alignment_b200 import _cabi

    sub = batch.recs[members]
    part_d = torch.from_numpy(part).to(batch.dev)
    terms = [torch.stack(t).cpu().numpy() for t in zip(*(ref_head_terms(refs[b]) for b in members))]
    idx = sub["score_off"][:, None] + np.arange(G)[None, :]
    worst = 0.0
    for w_col, w_row in ((1.0, 1.0), (0.5, 2.0), (0.0, 1.0), (1.0, 0.0)):
        out = Guarded(batch.n_scores, torch.float32, batch.dev)
        _cabi.head_scores_from_partials(part_d, _cabi.upload_utts(sub, batch.dev), len(members), G, w_col, w_row, out.out)
        got = out.check(spans(batch.n_scores, sub["score_off"], [G] * len(members)))[idx].astype(np.float64)
        want, _ = ref_scores(terms, None, w_col, w_row, 0.0)
        err = np.abs(got - want) / want
        b, h = np.unravel_index(np.argmax(err), err.shape)
        assert err.max() <= SCORE_RTOL, (label, (w_col, w_row), batch.shapes[members[b]], h, got[b, h], want[b, h])
        worst = max(worst, float(err.max()))
    record_measure("capture_peaky_scores_from_partials_vs_fp64_max_rel_err", worst)


def report_moves(batch, width, label):
    """Print, per utterance shape class, how often the kernel's reference moved (emulated from the float64 logits) and
    return the totals (rows that moved at least once, most moves of one row, step rows that crossed)."""
    from whisper_char_alignment_b200.timing import _cluster_bucket

    moved = most = 0
    steps = {k: [0, 0] for k in (3, 4, 5)}  # kind -> [rows whose reference moved, rows whose step lies inside a sweep]
    for b, (T, F) in enumerate(batch.shapes):
        _, med = batch.reference(b, width)
        mv = count_reference_moves(med, batch.qk_scale, _cluster_bucket(F)).cpu().numpy()
        moved += int((mv > 0).sum())
        most = max(most, int(mv.max()))
        kinds = row_kinds(T).T  # (G, T)
        for (t0, t1), (f0, f1) in part_ranges(T, F, _cluster_bucket(F)):
            # this sweep holds block 0 and frames of block 1 the median leaves at the step's height
            if f0 == 0 and f1 > 16 + width // 2 and batch.qk_scale != 0:
                for kind in steps:
                    rows = kinds[:, t0:t1] == kind
                    steps[kind][0] += int((mv[:, t0:t1][rows] > 0).sum())
                    steps[kind][1] += int(rows.sum())
    print(f"{label}: rows whose lazy reference moved {moved}, at most {most} moves in one row; step rows moved / swept: "
          f"exactly 32 {steps[3]}, +1 ulp {steps[4]}, -1 ulp {steps[5]}")
    return moved, most, steps


# ------------------------------------------------------------------ 2 + 7: constructed profiles, every width of the tcgen05 kernel
GRID = [(T, F) for T in GRID_T for F in GRID_F]


@pytest.mark.parametrize("width", [1, 3, 5, 7])
def test_capture_tc_on_peaky_rows_vs_fp64(width, dev):
    """Every (T, F) of the grid in one ragged batch (one launch per cluster size 1-6, 8): ramps whose maximum climbs past
    the lazy reference once or many times, the exact threshold and one ulp either side, plateaus at the first / last
    frame, in the last partial block, in another copy or rank; maps against float64, then the head scores finished from
    the partials of the same launches."""
    batch = Batch(GRID, 1.0, dev, seed=width)
    ws, part = capture(batch, width)
    refs, worst = check_batch(batch, ws, width, f"W={width}", "capture_tc_peaky_vs_fp64")
    moved, most, steps = report_moves(batch, width, f"tcgen05 W={width} qk_scale=1")
    assert moved > 0 and most >= 3
    assert steps[4][0] == steps[4][1] > 0 and steps[3][0] == 0 and steps[5][0] == 0
    check_scores(batch, part, refs, list(range(len(GRID))), f"W={width}")


# ------------------------------------------------------------------ 3: qk_scale, both paths
SCALE_T = [1, 31, 33, 64, 65, 129, 448]
SCALE_F = [1, 3, 17, 224, 225, 449, 1345, 1500]


@pytest.mark.parametrize("qk_scale,width", [(1.0, 3), (0.5, 7), (3.0, 5), (20.0, 3), (0.0, 7), (-1.0, 3), (-0.0, 5),
                                            (-1.0, 7)], ids=str)
def test_capture_qk_scale_both_paths_vs_fp64(qk_scale, width, dev):
    """The tcgen05 kernel (the fminf branch for a negative scale, uniform rows for 0 and -0) and the CUDA-core path with
    the same inputs: each against float64, and the two against each other; scores from the partials as well."""
    from whisper_char_alignment_b200 import _cabi

    shapes = [(T, F) for T in SCALE_T for F in SCALE_F]
    batch = Batch(shapes, qk_scale, dev, seed=11)
    ws_tc, part = capture(batch, width)
    ws_simt, _ = capture(batch, width, flags=_cabi.WCA_CAPTURE_FORCE_SIMT, partials=False, by_bucket=False)
    refs, _ = check_batch(batch, ws_tc, width, f"tc qk_scale={qk_scale}", "capture_tc_qk_scale_vs_fp64")
    check_batch(batch, ws_simt, width, f"simt qk_scale={qk_scale}", "capture_simt_qk_scale_vs_fp64")
    a, s = torch.from_numpy(ws_tc).double(), torch.from_numpy(ws_simt).double()
    big = torch.from_numpy(batch.ws_written()) & (s >= TINY)
    between = float(((a - s).abs() / s.clamp_min(TINY))[big].max())
    record_measure("capture_tc_vs_simt_qk_scale_max_rel_diff", between)
    assert between <= 2 * MAP_RTOL
    if qk_scale == 0:  # every row uniform, whatever the logits
        for b, (T, F) in enumerate(shapes):
            np.testing.assert_allclose(batch.map_of(ws_tc, b), 1.0 / F, rtol=1e-6)
    else:
        moved, _, steps = report_moves(batch, width, f"tcgen05 W={width} qk_scale={qk_scale}")
        assert moved > 0 and steps[4][0] == steps[4][1] > 0 and steps[3][0] == 0 and steps[5][0] == 0
    check_scores(batch, part, refs, list(range(len(shapes))), f"qk_scale={qk_scale}")


# ------------------------------------------------------------------ 4: widths of the CUDA-core path
@pytest.mark.parametrize("width", [9, 11, 15, 31])
def test_capture_wide_median_vs_fp64(width, dev):
    """Widths 9-31 go through the CUDA-core logits and the in-place batched filter (median_window): rows of at most
    width // 2 frames (identity), of width // 2 + 1, short and 1500-frame rows in one ragged launch; no partials."""
    from whisper_char_alignment_b200 import _cabi

    half = width // 2
    shapes = [(1, 1), (33, half), (7, half + 1), (65, half + 2), (31, 17), (129, 224), (448, 1500), (3, 1500), (64, 449)]
    batch = Batch(shapes, 1.0, dev, seed=width)
    assert not _cabi.capture_writes_partials(1500, width) and not _cabi.capture_writes_partials(1, width)
    ws, _ = capture(batch, width, partials=False, by_bucket=False)
    check_batch(batch, ws, width, f"W={width}", "capture_wide_median_vs_fp64")
    part = Guarded(batch.n_part, torch.float32, dev)
    with pytest.raises(_cabi.WcaError, match="partials"):
        _cabi.capture_attention(batch.q, batch.k, H, LD_Q, LD_K, _cabi.upload_utts(batch.recs, dev), len(shapes), 448, 1500,
                                width, 1.0, Guarded(batch.n_ws, torch.float32, dev).out, 0, part.out)
    part.check(np.zeros(batch.n_part, dtype=bool))


# ------------------------------------------------------------------ 5: poisoned surroundings
POISON_T = [1, 31, 33, 65, 127, 129, 448]
POISON_F = [1, 3, 17, 224, 225, 449, 1500]


@pytest.mark.parametrize("width", [1, 7])
def test_capture_ignores_rows_outside_the_utterance(width, dev):
    """The maps and partials of an utterance depend on its Q rows q_row0 .. q_row0+T-1 and K rows k_row0 .. k_row0+F-1
    only: with every other element of the operand buffers NaN, or +-inf and +-1e30, they are bit-identical to a run where
    those are finite numbers (tcgen05 kernel; the tile reads Q rows up to its 32/64/128-row boundary, K rows into the
    right halo), and the CUDA-core path likewise."""
    from whisper_char_alignment_b200 import _cabi

    shapes = [(T, F) for T in POISON_T for F in POISON_F]
    runs = {}
    for poison in ("finite", "nan", "inf_big"):
        batch = Batch(shapes, 1.0, dev, seed=5, poison=poison)
        runs[poison] = capture(batch, width) + (capture(batch, width, flags=_cabi.WCA_CAPTURE_FORCE_SIMT, partials=False,
                                                        by_bucket=False)[0],)
    check_batch(batch, runs["finite"][0], width, f"poison W={width}", "capture_tc_poisoned_vs_fp64")
    for poison in ("nan", "inf_big"):
        for i, what in enumerate(("tcgen05 maps", "partials", "CUDA-core maps")):
            np.testing.assert_array_equal(runs[poison][i].view(np.int32), runs["finite"][i].view(np.int32),
                                          err_msg=f"{what} with {poison} around the utterances, W={width}")


# ------------------------------------------------------------------ 6: batch independence
def test_capture_utterance_alone_equals_in_a_batch(dev):
    """An utterance's maps and partials are bit-identical launched alone, inside its mixed cluster bucket (the order
    reversed: other tile-list positions), and in a launch whose max_tokens / max_frames exceed its own without changing
    the cluster size.  A max_frames that changes the cluster size splits the frames differently: compared with float64
    only."""
    shapes = [(448, 1500), (1, 1345), (33, 1400), (129, 225), (65, 300), (31, 448), (1, 1), (64, 17), (127, 224), (3, 16)]
    batch = Batch(shapes, 1.0, dev, seed=3)
    width = 5
    ws_all, part_all = capture(batch, width, members=list(reversed(range(len(shapes)))))
    refs, _ = check_batch(batch, ws_all, width, "batch", "capture_tc_batch_vs_fp64")
    from whisper_char_alignment_b200.timing import _cluster_bucket

    def same(b, got, label):
        T, F = shapes[b]
        o, n = int(batch.recs[b]["ws_off"]), G * T * F
        np.testing.assert_array_equal(got[0][o:o + n].view(np.int32), ws_all[o:o + n].view(np.int32), err_msg=label)
        m = batch.partials_written([b])
        np.testing.assert_array_equal(got[1][m].view(np.int32), part_all[m].view(np.int32), err_msg=label)

    for b, (T, F) in enumerate(shapes):
        same(b, capture(batch, width, members=[b]), f"alone, {shapes[b]}")
        big_f = min(1500, _cluster_bucket(F) * 224) if _cluster_bucket(F) < 8 else 1500
        assert _cluster_bucket(big_f) == _cluster_bucket(F)
        same(b, capture(batch, width, members=[b], max_tokens=448, max_frames=big_f), f"max 448 x {big_f}, {shapes[b]}")
        if _cluster_bucket(F) < 8:  # one more CTA per cluster: other frame ranges per rank
            ws, part = capture(batch, width, members=[b], max_frames=_cluster_bucket(F) * 224 + 1)
            rel, dsum = compare_maps(torch.from_numpy(batch.map_of(ws, b)).to(dev), refs[b])
            assert rel <= MAP_RTOL and dsum <= SUM_TOL, (shapes[b], rel, dsum)
            check_scores(batch, part, refs, [b], f"larger cluster, {shapes[b]}")
