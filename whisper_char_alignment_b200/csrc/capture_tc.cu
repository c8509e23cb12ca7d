// tcgen05 / TMEM / TMA cross-attention capture (north-star kernel 1), v2: persistent,
// warp-specialised, double-buffered in tensor memory.
//
// Replaces reference timing.py:50-66 + upstream qkv_attention (SDPA off): for every
// (utterance, layer, head, block of 128 tokens) it computes
//     P[t, f] = softmax_f( median_w( (q_t * s) . (k_f * s) )[:F] * qk_scale ),  s = 64^-1/4
// and writes it ONCE, already trimmed to F, in the (L, H, T, F) layout get_attentions
// returns.  The 1500-frame logits, the torch.cat copy, the reflect-padded copy and the two
// softmax passes of the reference never touch HBM.
//
// Mapping
//   tokens  <-> TMEM lanes (UMMA M = 128): thread r of an epilogue warpgroup owns token row
//               r, so the median window and both softmax reductions are private to a thread;
//   frames  <-> TMEM columns: the fp32 accumulator IS the row buffer (filter and exp results
//               are written back in place with tcgen05.st).  512 columns = two accumulators
//               of 256 (16 halo + 224 own + 16 halo), so the tensor pipe fills one while an
//               epilogue warpgroup drains the other;
//   F > 224 : thread-block cluster of 2/4/8 CTAs along frames; per-row max and sum travel
//               through distributed shared memory, signalled with remote mbarrier arrives;
//   fp32 in, fp32-grade out on the tensor pipe: operands are split v = hi + lo (hi = v as the
//               tensor core chops it to tf32, lo = v - hi exact) and lo*hi + hi*lo + hi*hi is
//               accumulated: 3 x 8 tcgen05.mma kind::tf32 of N = all frames of the CTA per head,
//               error ~1e-6 relative;
//   TMA     : Q / K tiles arrive as 2-D tensor-map boxes (cp.async.bulk.tensor.2d, 64 rows x
//               32 floats, 128-byte swizzle) on one mbarrier per tile, directly where the MMA
//               reads them: the swizzled boxes ARE the UMMA K-major SWIZZLE_128B layout.
//
// Roles of the 16 warps of a CTA (one persistent CTA per SM, static tile schedule):
//   warp 0      TMA producer            warp 1      MMA issuer (one thread)
//   warps 4-7   operand splitters       warps 8-11 / 12-15   epilogue warpgroups A / B,
//                                       alternating tiles (accumulator i & 1)
#include <cuda.h>  // CUtensorMap and its enums only; the encoder is fetched from the driver at run time

#include <atomic>
#include <cstring>
#include <mutex>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace wca {
namespace tc {

constexpr int kThreads = 512;
constexpr int kRows = 128;           // UMMA M: tokens per tile
constexpr int kChunk = 64;           // frames per MMA group (UMMA N of a full chunk)
constexpr int kHalo = 16;            // halo columns either side (>= largest half-width, 15)
constexpr int kOwnCol0 = 16;         // accumulator column of a CTA's first own frame
constexpr int kAccCols = 256;        // columns per accumulator
constexpr int kMaxOwn = kAccCols - 2 * kHalo;   // 224 own frames per CTA and tile
constexpr int kTmemCols = 512;
constexpr int kStageRows = 64;                     // rows per TMA box
constexpr int kBoxCols = 32;                       // floats per TMA box row: 128 B, the swizzle span
constexpr int kBoxBytes = kStageRows * kBoxCols * 4;     // 8192: one 64-row x 128-byte box
constexpr int kQHalfBytes = 2 * kBoxBytes;               // Q tile, one column half: 128 rows x 128 B
constexpr int kQBytes = 2 * kQHalfBytes;                 // 32768
constexpr int kMaxChunks = kAccCols / kChunk;            // 4 boxes of 64 frames cover an accumulator
constexpr int kKHalfBytes = kMaxChunks * kBoxBytes;      // K slab, one column half: 256 frames x 128 B
constexpr int kKBytes = 2 * kKHalfBytes;                 // 65536
constexpr int kTilePitch = 16;           // transpose tile pitch: no padding, 16-byte chunks XOR-swizzled by (row / 2) & 3
constexpr int kSplitThreads = 128;
constexpr int kEpiThreads = 128;

// Operands live in shared memory exactly as TMA lands them (128-byte swizzle = the UMMA canonical
// K-major SWIZZLE_128B layout); the `hi` part of the 3 x tf32 split is the tile itself (the tensor
// core ignores the 13 low mantissa bits), the `lo` part is a twin tile the splitter warps write.
// One tile = the Q tile (128 token rows) + the whole K slab of the CTA (up to 256 frames), so that a
// head is 24 MMAs of N = up to 256 instead of 72 of N = 64: with both operands in shared memory an
// MMA re-reads its 4 KB of A every time, and at N = 64 that made the tensor pipe wait on shared memory.
constexpr int kOffQHi = 0;
constexpr int kOffQLo = kOffQHi + kQBytes;
constexpr int kOffKHi = kOffQLo + kQBytes;
constexpr int kOffKLo = kOffKHi + kKBytes;
constexpr int kOffTile = kOffKLo + kKBytes;                     // 8 epilogue warps x 32 x 17 floats
constexpr int kStatSlots = 2 * kRows;  // per group and tile parity: [128] published rows + [128] triples of the mirrored copies
constexpr int kOffStat = kOffTile + 8 * 32 * kTilePitch * 4;    // [group][tile parity][256] x {m, sum, sum of squares, -}
constexpr int kOffBar = kOffStat + 2 * 2 * kStatSlots * 16;
enum Bar {
    kKFull = 0,                  // TMA -> splitters (transaction bytes): K slab landed
    kQFull = kKFull + 1,         // ... Q tile landed
    kKLoReady = kQFull + 1,      // splitters -> MMA issuer: K lo twin written
    kQLoReady = kKLoReady + 1,   // splitters -> MMA issuer: Q lo twin written
    kKFree = kQLoReady + 1,      // MMA (tcgen05.commit after the two passes that read K_hi, once the K twin is written) -> TMA producer: K_hi may be refilled
    kOpFree = kKFree + 1,        // MMA (tcgen05.commit after the last pass) -> producer (Q_hi) and splitters (lo twins)
    kAccFull = kOpFree + 1,
    kAccEmpty = kAccFull + 2,
    kXMax = kAccEmpty + 2,
    kXSum = kXMax + 2,
    kNumBars = kXSum + 2
};
constexpr int kOffTmem = kOffBar + kNumBars * 8;
constexpr int kOffSink = kOffTmem + 16;  // 16 floats the transposition-tile writes of lanes past the last token row go to
constexpr int kSmemBytes = kOffSink + 64;
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");

// ------------------------------------------------------------------ debug trace (WCA_CAPTURE_TRACE)
// CTA 0 stamps clock64() at the hand-over points of every role for its first kTraceTiles
// tiles; tools/trace_capture.py turns the table into a per-role timeline.
constexpr int kTraceTiles = 40;
enum Ev { kEvProdQ = 0, kEvProdK0, kEvProdKLast, kEvSplAFree, kEvSplQDone, kEvSplK0Done, kEvSplKLast, kEvMmaAccEmpty,
          kEvMmaAReady, kEvMmaB0, kEvMmaIssued, kEvEpiAccFull, kEvEpiA, kEvEpiXMax, kEvEpiB, kEvEpiXSum, kEvEpiC,
          kEvSplFull, kEvSplLoaded, kEvSplStored, kEvSplFenced, kNumEv };
__device__ long long g_trace[kTraceTiles][kNumEv];
__device__ __forceinline__ void stamp(bool on, uint32_t tile_seq, int ev) {
    if (on && tile_seq < (uint32_t)kTraceTiles) g_trace[tile_seq][ev] = clock64();
}

// ------------------------------------------------------------------ tile geometry
// (rows, H*64) fp32 matrices, boxes of 32 floats (128 B, the swizzle span) x 64 / 128 / 192 / 256 rows:
// one TMA instruction costs ~150 cycles of the producer lane whatever it moves, so a tile is fetched
// with the tallest box that fits (K slab: one box per column half).
struct TensorMaps {
    CUtensorMap q[3][WCA_MAX_LAYERS];  // boxes of 64, 128 and 32 token rows
    CUtensorMap k[4][WCA_MAX_LAYERS];
};

struct KernelArgs {
    const wca_utt_t *utts;
    float *ws;
    float *partials;  // head-score partials (see wca_capture_attention), or nullptr
    int n_heads, lh_count, tok_blocks, n_tiles;
    float s, qk_scale;
    int raw_logits;
    int trace;
    unsigned dbg;  // experiment switches (bits 8..): never set by the product path
};

struct Geo {
    bool live;       // the tile has token rows (same answer in every CTA of the cluster)
    int T, F, rows_valid;
    int f0, f1, n_own;       // frames this CTA owns
    int half;                // filter half-width actually applied (0: identity)
    int m0, mcol0, n_mma;    // first frame / accumulator column / frame count the MMA computes
    int n_chunks;
    int copies;              // <= 64 token rows are mirrored into A rows 64..127 (2), <= 32 rows into all four
                             // lane quarters (4): the epilogue warps that hold the same rows split the frames
    bool dup;                // copies > 1
    int layer, col0;         // decoder layer and first float column of the head
    int qrow0, krow0;        // first Q row of the tile / first K row of the utterance
    float *out;              // row 0 of this tile, frame 0
    float *row_part;         // head-score partials of this tile, per group of 32 token rows: sum_t ||p[t,:]||_2 (4 floats) ...
    float *col_ss;           // ... and sum_t p[t,f]^2, frame 0 ([4][F] floats); nullptr: not wanted
};

// Position of a role in the static tile schedule (tile = (utterance, layer * head, token block), tiles cid, cid + n_clusters,
// ...): the three indices advance by carries instead of being divided out of the tile number for every tile -- all 16 warps of
// a CTA walk the whole list, and the four divisions by run-time divisors were most of the ~120 instructions a tile cost each.
struct TileCursor {
    int tile, ub, lh, tb;
    int d_ub, d_lh, d_tb;  // the stride, decomposed the same way
    float rcp_heads, rcp_csize;
    __device__ __forceinline__ void init(const KernelArgs &a, int first, int stride, uint32_t csize) {
        tile = first;
        tb = first % a.tok_blocks;
        int r = first / a.tok_blocks;
        lh = r % a.lh_count;
        ub = r / a.lh_count;
        d_tb = stride % a.tok_blocks;
        r = stride / a.tok_blocks;
        d_lh = r % a.lh_count;
        d_ub = r / a.lh_count;
        rcp_heads = 1.0f / (float)a.n_heads;
        rcp_csize = 1.0f / (float)csize;
    }
    __device__ __forceinline__ void next(const KernelArgs &a, int stride) {
        tile += stride;
        tb += d_tb;
        if (tb >= a.tok_blocks) { tb -= a.tok_blocks; ++lh; }
        lh += d_lh;  // < 2 * lh_count: one correction is enough
        if (lh >= a.lh_count) { lh -= a.lh_count; ++ub; }
        ub += d_ub;
    }
};
// x / d for 0 <= x < 2^15 and d <= 32 through the reciprocal: (x + 0.5) / d is at least 1 / 64 away from an integer and
// the two roundings move it by less than x / d * 2^-22, so the floor is exact
__device__ __forceinline__ int div_small(int x, float rcp) { return __float2int_rd(((float)x + 0.5f) * rcp); }

template <int W>
__device__ __forceinline__ Geo decode_tile(const KernelArgs &a, const TileCursor &tc, uint32_t crank, uint32_t csize) {
    Geo g;
    const int tb = tc.tb, lh = tc.lh;
    const wca_utt_t u = a.utts[tc.ub];
    g.T = u.n_tokens;
    g.F = u.n_frames;
    const int t0 = tb * kRows;
    g.live = t0 < g.T;
    g.rows_valid = min(kRows, g.T - t0);
    g.layer = div_small(lh, tc.rcp_heads);
    g.col0 = (lh - g.layer * a.n_heads) * kHeadDim;
    g.qrow0 = (int)u.q_row0 + t0;
    g.krow0 = (int)u.k_row0;
    g.out = a.ws + u.ws_off + ((int64_t)lh * g.T + t0) * g.F;
    g.row_part = g.col_ss = nullptr;
    if (a.partials != nullptr && !a.raw_logits) {
        // per utterance: [lh][token block][4 row groups] row terms, then [lh][token block][4 row groups][F] column sums
        // of squares: every epilogue warp writes the partials of its own 32 token rows, nothing is combined in the kernel
        const int tbu = (g.T + kRows - 1) / kRows;
        float *base = a.partials + u.part_off;
        g.row_part = base + ((int64_t)lh * tbu + tb) * 4;
        g.col_ss = base + (int64_t)a.lh_count * tbu * 4 + ((int64_t)lh * tbu + tb) * 4 * g.F;
    }
    const int slab = (div_small(g.F + (int)csize - 1, tc.rcp_csize) + 15) & ~15;
    g.f0 = (int)crank * slab;
    g.f1 = min(g.F, g.f0 + slab);
    g.n_own = max(0, g.f1 - g.f0);
    const bool filter = !a.raw_logits && W > 1 && g.F > W / 2;  // identity for very short rows, like upstream
    g.half = filter ? W / 2 : 0;
    g.m0 = g.f0 > 0 ? g.f0 - kHalo : 0;
    g.mcol0 = g.f0 > 0 ? 0 : kOwnCol0;  // frame f always sits at accumulator column f - f0 + 16
    g.n_mma = g.n_own > 0 ? min(g.f1 + kHalo, g.F) - g.m0 : 0;
    g.n_chunks = (g.n_mma + kChunk - 1) / kChunk;
    g.copies = g.rows_valid <= 32 ? 4 : (g.rows_valid <= kStageRows ? 2 : 1);
    g.dup = g.copies > 1;
    return g;
}

// 128 splitter threads: lo twin of kBytes of a tile, linear sweep (same swizzled position, conflict-free).
template <int kBytes>
__device__ __forceinline__ void split_lo(const unsigned char *hi, unsigned char *lo, int t) {
    constexpr int kIters = kBytes / 16 / kSplitThreads;
    const float4 *src = reinterpret_cast<const float4 *>(hi);
    float4 *dst = reinterpret_cast<float4 *>(lo);
    float4 v[kIters];
#pragma unroll
    for (int it = 0; it < kIters; ++it) v[it] = src[it * kSplitThreads + t];  // all loads in flight first
#pragma unroll
    for (int it = 0; it < kIters; ++it)
        dst[it * kSplitThreads + t] = make_float4(tf32_lo(v[it].x), tf32_lo(v[it].y), tf32_lo(v[it].z), tf32_lo(v[it].w));
}

// Mirrored Q tile (Geo::dup): rows 64..127 of each column half are a second copy of rows 0..63, so one box is read
// and its lo twin is written to both (half the shared-memory reads of a plain split).
__device__ __forceinline__ void split_lo_dup(const unsigned char *hi, unsigned char *lo, int t) {
    constexpr int kIters = kBoxBytes / 16 / kSplitThreads;
    const float4 *src = reinterpret_cast<const float4 *>(hi);
    float4 *dst = reinterpret_cast<float4 *>(lo);
    float4 v[kIters];
#pragma unroll
    for (int it = 0; it < kIters; ++it) v[it] = src[it * kSplitThreads + t];
#pragma unroll
    for (int it = 0; it < kIters; ++it) {
        const float4 l = make_float4(tf32_lo(v[it].x), tf32_lo(v[it].y), tf32_lo(v[it].z), tf32_lo(v[it].w));
        dst[it * kSplitThreads + t] = l;
        dst[kBoxBytes / 16 + it * kSplitThreads + t] = l;
    }
}

// Four copies of a 32-row box (Geo::copies == 4): 4 KB read, its lo twin written four times.
__device__ __forceinline__ void split_lo_quad(const unsigned char *hi, unsigned char *lo, int t) {
    constexpr int kIters = kBoxBytes / 2 / 16 / kSplitThreads;  // 2
    const float4 *src = reinterpret_cast<const float4 *>(hi);
    float4 *dst = reinterpret_cast<float4 *>(lo);
#pragma unroll
    for (int it = 0; it < kIters; ++it) {
        const float4 v = src[it * kSplitThreads + t];
        const float4 l = make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w));
#pragma unroll
        for (int c = 0; c < 4; ++c) dst[c * (kBoxBytes / 2 / 16) + it * kSplitThreads + t] = l;
    }
}

// Sliding median over a 16-column block; every index is a compile time constant after unrolling, so the
// window lives in registers.  `ptail` = the last W/2 columns of the previous block, `next` = the next block.
template <int W>
struct Tail {
    static constexpr int kLen = W / 2 > 0 ? W / 2 : 1;
};
template <int W>
__device__ __forceinline__ void median_block(const float (&ptail)[Tail<W>::kLen], const float (&cur)[16],
                                             const float (&head)[4], float (&out)[16]) {
    constexpr int half = W / 2;
    if constexpr (W == 1) {
#pragma unroll
        for (int pos = 0; pos < 16; ++pos) out[pos] = cur[pos];
    } else if constexpr (W == 3) {
        // med(a, b, c) = max(min(a, b), min(max(a, b), c)): the (min, max) of the pair (2k, 2k+1) serves both of
        // its positions (with the left / the right neighbour): 3 instead of 5 min/max per column, still exact
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float lo = fminf(cur[2 * k], cur[2 * k + 1]);
            const float hi = fmaxf(cur[2 * k], cur[2 * k + 1]);
            const float left = k == 0 ? ptail[0] : cur[2 * k - 1];
            const float right = k == 7 ? head[0] : cur[2 * k + 2];
            out[2 * k] = fmaxf(lo, fminf(hi, left));
            out[2 * k + 1] = fmaxf(lo, fminf(hi, right));
        }
    } else {
#pragma unroll
        for (int pos = 0; pos < 16; ++pos) {
            float win[W];
#pragma unroll
            for (int j = 0; j < W; ++j) {
                const int idx = pos - half + j;  // relative to cur[0]
                win[j] = idx < 0 ? ptail[half + idx] : (idx < 16 ? cur[idx] : head[idx - 16]);
            }
            out[pos] = median_regs<W>(win);
        }
    }
}

// One 16-column block of the fused filter / exponential sweep (epilogue_tile, sweep A+B).  `cur` and `head` (the first
// columns of the next block: all the window needs of it) are dead once the filter has run, so the next block and the
// head of the one after it are loaded straight into their registers and land behind the exponentials.
struct RowStats {
    float m2, row_sum, row_ss;  // lazy reference (log2 domain), sum of e = 2^(y - m2), sum of e^2
};
template <int W>
__device__ __forceinline__ void filter_exp_block(uint32_t trow, int b, int b_lo, int b_hi, int n_blocks, int tail, bool filter,
                                                 float scale2, float (&ptail)[Tail<W>::kLen], float (&cur)[16],
                                                 float (&head)[4], RowStats &st, bool want_ss) {
    float med[16];
    median_block<W>(ptail, cur, head, med);
    if (W > 1 && !filter) {  // rows of at most W/2 frames are not filtered (as upstream): rare, kept off the hot path
#pragma unroll
        for (int i = 0; i < 16; ++i) med[i] = cur[i];
    }
    if constexpr (W > 1) {
#pragma unroll
        for (int j = 0; j < W / 2; ++j) ptail[j] = cur[16 - W / 2 + j];
    }
    if (b + 1 < b_hi) {
        tmem_ld16_issue(trow + (uint32_t)(16 * (b + 1)), cur);
        if (W > 1) tmem_ld4_issue(trow + (uint32_t)(16 * (b + 2)), head);  // b + 2 <= n_blocks: stays inside the accumulator
    }
    const int n_ok = b + 1 < n_blocks ? 16 : tail;
    if (n_ok < 16) {  // last block: columns past the row end must not win the maximum
#pragma unroll
        for (int i = 1; i < 16; ++i)
            if (i >= n_ok) med[i] = med[0];
    }
    // extreme of the block in the direction of the scale, then ONE multiply: y = med * scale2 is monotone
    float ext;
    if (scale2 >= 0.f) {
        ext = fmaxf(fmaxf(med[0], med[1]), med[2]);
#pragma unroll
        for (int i = 3; i < 15; i += 2) ext = fmaxf(fmaxf(ext, med[i]), med[i + 1]);
        ext = fmaxf(ext, med[15]);
    } else {
        ext = fminf(fminf(med[0], med[1]), med[2]);
#pragma unroll
        for (int i = 3; i < 15; i += 2) ext = fminf(fminf(ext, med[i]), med[i + 1]);
        ext = fminf(ext, med[15]);
    }
    const float bmax = ext * scale2;
    if (b == b_lo) st.m2 = bmax;
    const bool need = bmax > st.m2 + 32.f;
    if (__any_sync(0xffffffffu, need)) {  // rare: move the reference, rescale what is already stored
        const float f = need ? ex2_approx(st.m2 - bmax) : 1.f;
        if (need) st.m2 = bmax;
        st.row_sum *= f;
        st.row_ss *= f * f;
        tmem_wait_st();  // the blocks stored so far are read back
#pragma unroll 1
        for (int cc = 16 * b_lo; cc < 16 * b; cc += 4) {
            float t[4];
            tmem_ld4_issue(trow + (uint32_t)cc, t);
            tmem_ld_wait4(t);
#pragma unroll
            for (int i = 0; i < 4; ++i) t[i] *= f;
            tmem_st4(trow + (uint32_t)cc, t);
        }
    }
    const float neg_m2 = -st.m2;
#pragma unroll
    for (int i = 0; i < 16; ++i) med[i] = ex2_approx(__fmaf_rn(med[i], scale2, neg_m2));
    if (n_ok < 16) {
#pragma unroll
        for (int i = 1; i < 16; ++i)
            if (i >= n_ok) med[i] = 0.f;
    }
    st.row_sum += ((med[0] + med[1]) + (med[2] + med[3])) + ((med[4] + med[5]) + (med[6] + med[7])) +
                  (((med[8] + med[9]) + (med[10] + med[11])) + ((med[12] + med[13]) + (med[14] + med[15])));
    if (want_ss) {
        // sum of squares of the row (head scores, timing.py:24: ||a[t,:]||_2 = sqrt(sum e^2) / sum e); two chains
        float q0 = med[0] * med[0], q1 = med[1] * med[1];
#pragma unroll
        for (int i = 2; i < 16; i += 2) {
            q0 = __fmaf_rn(med[i], med[i], q0);
            q1 = __fmaf_rn(med[i + 1], med[i + 1], q1);
        }
        st.row_ss += q0 + q1;
    }
    tmem_st16(trow + (uint32_t)(16 * b), med);
    tmem_ld_wait(cur);  // the next block (and the head of the one after it) has landed; also orders the loads of the rescale path
    tmem_ld_wait4(head);
}

// The three sweeps of one tile by one epilogue warpgroup (thread <-> token row).
// Returns true when the accumulator has already been handed back (mbarrier `acc_empty`): that happens as soon as the
// last block of the store sweep is in registers, one block of stores before the tile is finished.
template <int W>
__device__ __forceinline__ bool epilogue_tile(const Geo &g, const KernelArgs &a, unsigned char *smem, uint32_t acc,
                                              int grp, int ewarp, int lane, uint32_t csize, uint32_t x_parity,
                                              bool tr, uint32_t seq, uint32_t acc_empty) {
    bool released = false;
    // Mirrored tiles (Geo::dup): lane quarters 2 and 3 hold a copy of token rows 0..63, so warps
    // 2/3 (other two schedulers) take the second half of the columns of the rows of warps 0/1.
    const int copy = g.copies == 4 ? ewarp : (g.copies == 2 ? ewarp >> 1 : 0);     // which copy of the rows this warp holds
    const int lw = g.copies == 4 ? 0 : (g.copies == 2 ? (ewarp & 1) : ewarp);      // logical 32-row group
    const int row = lw * 32 + lane;
    const bool row_ok = row < g.rows_valid;
    const int n_blocks = (g.n_own + 15) >> 4;
    // the copies split the blocks: copy p takes [ceil(n p / copies), ceil(n (p + 1) / copies))
    const int cshift = g.copies >> 1;  // log2(copies) for 1, 2, 4
    const int b_lo = (n_blocks * copy + g.copies - 1) >> cshift;
    const int b_hi = (n_blocks * (copy + 1) + g.copies - 1) >> cshift;
    const bool rows_live = (lw * 32 < g.rows_valid) && g.n_own > 0;  // warp-uniform
    const bool sweep = rows_live && b_lo < b_hi;
    const uint32_t trow = acc + ((uint32_t)(ewarp * 32) << 16) + kOwnCol0;  // own frame 0 of this lane quarter
    const int tail = g.n_own - 16 * (n_blocks - 1);  // valid columns of the last block (1..16)
    float4 *sstat = reinterpret_cast<float4 *>(smem + kOffStat) + grp * 2 * kStatSlots;  // [tile parity][256] x {m, sum, ss, -}
    const uint32_t bar_xmax = smem_u32(smem + kOffBar) + 8u * (kXMax + grp);

    float inv_sum = a.s;  // raw-logit mode: only the 2^-3 of the operand scaling is applied
    bool report_rows = false;
    float row_term = 0.f;
    if (!a.raw_logits) {
        if (sweep && g.half > 0 && min(g.f1, g.f0 + 16 * b_hi) + g.half > g.F) {  // the windows of this part reach past the last frame
            // materialise the right reflect padding in TMEM, frame F-1+i <- frame F-1-i (i = 1..3 whatever the width: what a
            // narrower window does not read is never used): one 4-column load and one 4-column store instead of a round
            // trip per frame.  (The left padding never reaches tensor memory: see ptail below.)
            float t[4];
            const uint32_t c_end = trow + (uint32_t)(g.F - g.f0);
            tmem_ld4_issue(c_end - 4u, t);
            tmem_ld_wait4(t);
            const float r[4] = {t[2], t[1], t[0], t[0]};
            tmem_st4(c_end, r);
            tmem_wait_st();
        }
        // Sweep A+B fused: median filter, * qk_scale, and e = 2^(y - m) against a LAZY per-thread reference m
        // (the maximum of the thread's first block; it only moves when a later block exceeds it by 2^32, and the
        // few blocks already written are then rescaled in place), with the running sum.  One pass over tensor
        // memory instead of two and a single exchange of (m, sum) pairs between column halves / cluster ranks.
        const float kLog2e = 1.4426950408889634f;
        const float scale2 = a.qk_scale * kLog2e;
        const bool want_ss = g.row_part != nullptr && !(a.dbg & 0x400u);  // (0x400: experiment switch)
        RowStats st{-INFINITY, 0.f, 0.f};
        if (sweep) {
            float ptail[Tail<W>::kLen], cur[16], head[4];
            {
                float prev[4];
                tmem_ld4_issue(trow + (uint32_t)(16 * b_lo) - 4u, prev);
                tmem_ld16_issue(trow + (uint32_t)(16 * b_lo), cur);
                tmem_ld4_issue(trow + (uint32_t)(16 * (b_lo + 1)), head);
                tmem_ld_wait4(prev);
                tmem_ld_wait(cur);
                tmem_ld_wait4(head);
#pragma unroll
                for (int j = 0; j < Tail<W>::kLen; ++j) ptail[j] = prev[4 - Tail<W>::kLen + j];
                if (W > 1 && g.f0 == 0 && b_lo == 0) {  // left reflect padding: frame -i <- frame i, straight from the first block
#pragma unroll
                    for (int j = 0; j < Tail<W>::kLen; ++j) ptail[j] = cur[Tail<W>::kLen - j];
                }
            }
#pragma unroll 1
            for (int b = b_lo; b < b_hi; ++b)
                filter_exp_block<W>(trow, b, b_lo, b_hi, n_blocks, tail, g.half > 0, scale2, ptail, cur, head, st, want_ss);
        }
        const float m2 = st.m2, row_sum = st.row_sum, row_ss = st.row_ss;
        stamp(tr, seq, kEvEpiA);
        stamp(tr, seq, kEvEpiXMax);
        stamp(tr, seq, kEvEpiB);
        // (m, sum, sum of squares) of the other column half (mirrored tiles) and of the other cluster ranks; the
        // statistics buffers alternate with the tile parity so that nobody overwrites a triple a slower peer still reads
        float4 *strip = sstat + x_parity * kStatSlots;
        float gmax = m2, gsum = row_sum, gss = row_ss;
        if (csize == 1 && g.copies == 2) {
            strip[ewarp * 32 + lane] = make_float4(m2, row_sum, row_ss, 0.f);
            named_bar_sync(3 + grp * 2 + (ewarp & 1), 64);  // only the two warps that hold the same rows meet
            const float4 o = strip[(ewarp ^ 2) * 32 + lane];
            gmax = fmaxf(m2, o.x);
            const float fa = m2 > -INFINITY ? ex2_approx(m2 - gmax) : 0.f, fb = o.x > -INFINITY ? ex2_approx(o.x - gmax) : 0.f;
            gsum = row_sum * fa + o.y * fb;
            gss = row_ss * (fa * fa) + o.z * (fb * fb);
        } else if (csize == 1 && g.copies == 4) {
            strip[ewarp * 32 + lane] = make_float4(m2, row_sum, row_ss, 0.f);
            named_bar_sync(1 + grp, kEpiThreads);  // all four warps hold the same 32 rows
            float4 pr[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) pr[j] = strip[j * 32 + lane];
            gmax = fmaxf(fmaxf(pr[0].x, pr[1].x), fmaxf(pr[2].x, pr[3].x));
            gsum = gss = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j)  // fixed order: every copy computes the same sums
                if (pr[j].x > -INFINITY) {
                    const float f = ex2_approx(pr[j].x - gmax);
                    gsum += pr[j].y * f;
                    gss += pr[j].z * (f * f);
                }
        }
        if (csize > 1) {
            // every CTA of the cluster takes part, even with no own frames
            const float4 mine = row_ok ? make_float4(m2, row_sum, row_ss, 0.f) : make_float4(-INFINITY, 0.f, 0.f, 0.f);
            if (g.copies == 1) {
                strip[row] = mine;
            } else {
                // mirrored rows: the copies' triples meet in the second half of the strip, the first copy adds them up
                // (fixed order) and publishes the CTA's triple of the row for the other ranks
                float4 *loc = strip + kRows;
                loc[ewarp * 32 + lane] = mine;
                named_bar_sync(7 + grp, kEpiThreads);
                if (copy == 0) {
                    const int stride = g.copies == 4 ? 32 : 64;  // warp of copy c with the same rows: ewarp + c * (4 / copies)
                    float cm = -INFINITY;
                    for (int c = 0; c < g.copies; ++c) cm = fmaxf(cm, loc[ewarp * 32 + c * stride + lane].x);
                    float cs = 0.f, cq = 0.f;
                    for (int c = 0; c < g.copies; ++c) {
                        const float4 o = loc[ewarp * 32 + c * stride + lane];
                        if (o.x > -INFINITY) {
                            const float f = ex2_approx(o.x - cm);
                            cs += o.y * f;
                            cq += o.z * (f * f);
                        }
                    }
                    strip[row] = make_float4(cm, cs, cq, 0.f);
                }
            }
            named_bar_sync(1 + grp, kEpiThreads);
            // lane r of the first warp signals rank r: ONE instruction with csize active lanes.  A loop of release-arrives
            // in one thread paid the cluster-scope release (~1.2 k cycles) once per rank, 9-10 k cycles per head.
            if (ewarp == 0 && (uint32_t)lane < csize) mbar_arrive_remote(bar_xmax, (uint32_t)lane);
            mbar_wait_cluster(bar_xmax, x_parity);
            // all ranks' triples in flight at once: a dependent chain of remote loads (maximum first, then a conditional
            // load of each sum) cost ~16 distributed-shared-memory round trips per head, 10.8 k of a 22.7 k-cycle epilogue
            float4 pr[8];
#pragma unroll
            for (uint32_t r = 0; r < 8; ++r)
                if (r < csize) pr[r] = ld_dsmem_f32x4(&strip[row], r);
            gmax = -INFINITY;
#pragma unroll
            for (uint32_t r = 0; r < 8; ++r)
                if (r < csize) gmax = fmaxf(gmax, pr[r].x);
            gsum = gss = 0.f;
#pragma unroll
            for (uint32_t r = 0; r < 8; ++r)
                if (r < csize && pr[r].x > -INFINITY) {
                    const float f = ex2_approx(pr[r].x - gmax);
                    gsum += pr[r].y * f;
                    gss += pr[r].z * (f * f);
                }
        }
        // head scores, row term of this warp's 32 token rows (timing.py:24): one thread per row reports -- rank 0 of a
        // cluster, the first copy of a mirrored row -- and a fixed shuffle tree adds them (deterministic)
        // (the shuffle tree and the store wait until the store sweep is through: they are not on the way to the accumulator's release)
        report_rows = g.row_part != nullptr && rows_live && (csize == 1 || cluster_ctarank() == 0) && copy == 0;
        if (report_rows) row_term = row_ok ? sqrtf(gss) / gsum : 0.f;
        inv_sum = __fdividef(m2 > -INFINITY ? ex2_approx(m2 - gmax) : 0.f, gsum);  // this thread's e values are relative to its own m
        stamp(tr, seq, kEvEpiXSum);
    }

    // column partials of this warp's 32 token rows for the head scores, written straight to the partial buffer
    float *colss = (g.col_ss != nullptr && !(a.dbg & 0x200u)) ? g.col_ss + (int64_t)lw * g.F + g.f0 : nullptr;  // (0x200: experiment switch)
    // sweep C: normalise, transpose 32x16 blocks through shared memory, coalesced row stores.
    // Lane (c, rsel) stores column c of rows rsel, rsel+2, ...: two 64-byte row segments per
    // instruction, the address advancing by two rows per step.
    if (sweep) {
        float *tile = reinterpret_cast<float *>(smem + kOffTile) + (grp * 4 + ewarp) * (32 * kTilePitch);
        const int rows_here = min(32, g.rows_valid - lw * 32);
        const int c = lane & 15, rsel = lane >> 4;
        const int n_steps = (rows_here - rsel + 1) >> 1;  // rows rsel + 2k < rows_here
        // 32-bit element offsets from the lane's first row (at most 128 rows of 1500 frames): one multiply-add and
        // one widening add per store instead of a 64-bit running pointer
        const int step = 2 * g.F;
        float *obase = g.out + ((lw * 32 + rsel) * g.F + g.f0 + c);
        asm volatile("" : "+l"(obase));  // keep the lane's base pointer in a register pair instead of re-deriving it per store
        // 32 x 16 tile without padding; the 16-byte chunk j of row r sits in slot j ^ ((r >> 1) & 3).  Row writes
        // (128-bit, 8 lanes per wavefront: rows r, r+2, r+4, r+6 share 16 banks) and column reads (lanes = 16 columns
        // x 2 rows; both rows of an instruction have the same (r >> 1) & 3 = k & 3) are then both conflict-free.
        const int sw = (lane >> 1) & 3;
        float4 *tdst = reinterpret_cast<float4 *>(tile + lane * kTilePitch);
        // Lanes past the last token row computed their values from the Q rows behind the utterance's last token, which a
        // caller may leave as NaN or inf (and 0 * NaN is NaN): they zero their row of the transposition tile once and send
        // their block writes to a sink, so that the column sums of the head scores only see token rows (a per-block
        // predicate or select on those writes cost 2-6 % of the kernel)
        if (!row_ok) {
#pragma unroll
            for (int i = 0; i < 4; ++i) tdst[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            tdst = reinterpret_cast<float4 *>(smem + kOffSink);
        }
        const float *tsrc[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) tsrc[j] = tile + rsel * kTilePitch + 4 * ((c >> 2) ^ j) + (c & 3);
        float v[16];
        tmem_wait_st();  // the filter sweep's stores (they drained behind the statistics exchange)
        tmem_ld16_issue(trow + (uint32_t)(16 * b_lo), v);
        tmem_ld_wait(v);
        for (int b = b_lo; b < b_hi; ++b) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                tdst[i ^ sw] = make_float4(v[4 * i] * inv_sum, v[4 * i + 1] * inv_sum, v[4 * i + 2] * inv_sum, v[4 * i + 3] * inv_sum);
            if (b + 1 < b_hi) {
                tmem_ld16_issue(trow + (uint32_t)(16 * (b + 1)), v);  // v is free again: the next block lands behind the stores
            } else {
                // nothing of this tile is left in tensor memory: the MMA issuer may refill the accumulator now
                tc_fence_before();
                mbar_arrive(acc_empty);
                released = true;
            }
            __syncwarp();
            float o[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) o[k] = tsrc[k & 3][k * 2 * kTilePitch];  // all reads in flight before the stores
            if (g.f0 + 16 * b + c < g.f1) {
                const int o0 = 16 * b;
                // one predicated path: a second, unpredicated copy for full warps saved 16 ISETP per block and cost more in
                // instruction fetch (the hot loops of the five roles together exceed the SM's 32 KB instruction cache)
#pragma unroll
                for (int k = 0; k < 16; ++k)
                    if (k < n_steps) st_stream(obase + (o0 + k * step), o[k]);
            }
            if (colss != nullptr) {
                // head scores (timing.py:21): sum over this warp's token rows of p[t,f]^2 for the 16 frames of the block;
                // lane (c, rsel) holds rows rsel, rsel + 2, ...: rows past the last token row are exact zeros in the tile
                float q0 = o[0] * o[0], q1 = o[1] * o[1];
#pragma unroll
                for (int k = 2; k < 16; k += 2) {
                    q0 = __fmaf_rn(o[k], o[k], q0);
                    q1 = __fmaf_rn(o[k + 1], o[k + 1], q1);
                }
                float q = q0 + q1;
                q += __shfl_xor_sync(0xffffffffu, q, 16);
                if (lane < 16 && g.f0 + 16 * b + lane < g.f1) colss[16 * b + lane] = q;  // 64 contiguous bytes per block
            }
            __syncwarp();
            tmem_ld_wait(v);
        }
    }
    if (report_rows) {  // warp-uniform
        const float term = warp_sum(row_term);
        if (lane == 0) g.row_part[lw] = term;
    }
    stamp(tr, seq, kEvEpiC);
    return released;
}

// ------------------------------------------------------------------ the kernel
template <int W>
__global__ void __launch_bounds__(kThreads, 1)
capture_tc_kernel(const __grid_constant__ TensorMaps maps, const __grid_constant__ KernelArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t crank = cluster_ctarank(), csize = cluster_nctarank();
    const int cid = blockIdx.x / csize, n_clusters = gridDim.x / csize;
    const uint32_t bars = smem_u32(smem + kOffBar);
    auto bar = [&](int which) { return bars + 8u * (uint32_t)which; };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + kOffTmem);

    // ---- setup ------------------------------------------------------------------------
    if (tid == 0) {
        mbar_init(bar(kKFull), 1);
        mbar_init(bar(kQFull), 1);
        mbar_init(bar(kKLoReady), kSplitThreads);
        mbar_init(bar(kQLoReady), kSplitThreads);
        mbar_init(bar(kKFree), 1);
        mbar_init(bar(kOpFree), 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar(kAccFull + i), 1);
            mbar_init(bar(kAccEmpty + i), kEpiThreads);
            mbar_init(bar(kXMax + i), csize);
            mbar_init(bar(kXSum + i), csize);
        }
        fence_mbar_init();
    }
    if (warp == 0) {
        tmem_alloc(smem_u32(tmem_slot), kTmemCols);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    cluster_sync_all();  // peers' barriers are initialised before anyone arrives remotely

    if (warp == 0) {
        // ================= TMA producer: boxes land directly in the operand buffers =================
        uint32_t n_tile = 0;
        const bool tr = a.trace && blockIdx.x == (a.dbg >> 8) && lane == 0;
        const uint32_t q_hi = smem_u32(smem + kOffQHi), k_hi = smem_u32(smem + kOffKHi);
        TileCursor cur;
        for (cur.init(a, cid, n_clusters, csize); cur.tile < a.n_tiles; cur.next(a, n_clusters)) {
            const Geo g = decode_tile<W>(a, cur, crank, csize);
            if (!g.live || g.n_own == 0) continue;
            // K_hi is refilled as soon as the two MMA passes that read it have run (a third of the MMA time and the whole
            // drain earlier than the last pass), Q_hi once all of them have: the K load -- 60 % of the bytes -- is then
            // already in shared memory when the splitters are allowed to touch the lo twins.
            const bool upper = g.dup || g.rows_valid > kStageRows;
            mbar_wait(bar(kKFree), (n_tile & 1u) ^ 1u);  // first lap passes
            if (lane == 0) {
                mbar_expect_tx(bar(kKFull), g.n_chunks * 2 * kBoxBytes);  // boxes are always full: rows past the matrix end read as zero
                const CUtensorMap *kmap = &maps.k[g.n_chunks - 1][g.layer];   // box = n_chunks * 64 frames
                for (int half = 0; half < 2; ++half)
                    tma_load_box(k_hi + half * kKHalfBytes, kmap, g.col0 + half * kBoxCols, g.krow0 + g.m0, bar(kKFull));
            }
            __syncwarp();
            mbar_wait(bar(kOpFree), (n_tile & 1u) ^ 1u);  // MMAs of the previous tile no longer read Q
            if (lane == 0) {
                // Q rows 64..127: the next 64 token rows, or (Geo::dup) a second copy of rows 0..63; with <= 64
                // rows and no mirroring the upper half is left as it is (nobody reads those lanes)
                mbar_expect_tx(bar(kQFull), upper ? kQBytes : kQBytes / 2);
                const CUtensorMap *qmap = &maps.q[g.copies == 4 ? 2 : ((upper && !g.dup) ? 1 : 0)][g.layer];
                const int copy_bytes = kQHalfBytes >> (g.copies >> 1);  // one box per copy and column half
                for (int half = 0; half < 2; ++half)
                    for (int c = 0; c < g.copies; ++c)
                        tma_load_box(q_hi + half * kQHalfBytes + c * copy_bytes, qmap, g.col0 + half * kBoxCols, g.qrow0,
                                     bar(kQFull));
            }
            __syncwarp();
            stamp(tr, n_tile, kEvProdQ);
            ++n_tile;
            // While this tile is split, multiplied and filtered, pull the next tile's boxes into L2: the
            // operand buffers are single (shared memory is full), so the next load can only be issued once
            // this tile's MMAs are done, and its latency is then an L2 hit instead of an HBM round trip.
            TileCursor ahead = cur;
            for (ahead.next(a, n_clusters); ahead.tile < a.n_tiles; ahead.next(a, n_clusters)) {
                const Geo h = decode_tile<W>(a, ahead, crank, csize);
                if (!h.live || h.n_own == 0) continue;
                if (lane == 0) {
                    const CUtensorMap *kmap = &maps.k[h.n_chunks - 1][h.layer];
                    const CUtensorMap *qmap = &maps.q[h.copies == 4 ? 2 : ((!h.dup && h.rows_valid > kStageRows) ? 1 : 0)][h.layer];
                    for (int half = 0; half < 2; ++half) {
                        tma_prefetch_box(kmap, h.col0 + half * kBoxCols, h.krow0 + h.m0);
                        tma_prefetch_box(qmap, h.col0 + half * kBoxCols, h.qrow0);
                    }
                }
                __syncwarp();
                break;
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer: the whole warp runs the loop, one elected lane issues =================
        // (only the tcgen05.mma itself is predicated: descriptor arithmetic stays on the uniform datapath)
        uint32_t n_tile = 0, acc_use0 = 0, acc_use1 = 0, it = 0;
        const bool tr = a.trace && blockIdx.x == (a.dbg >> 8) && lane == 0;
        const uint32_t elected = elect_one() ? 1u : 0u;
        const uint32_t tm = __shfl_sync(0xffffffffu, tmem_base, 0);
        // K-major, 128-byte swizzle: 8-row groups are 1024 B apart; 8 tf32 = 32 B along the row, the second
        // column half is the next half-tile (A: +16 KB, B: +32 KB)
        const uint64_t da_hi = smem_desc_sw128(smem_u32(smem + kOffQHi), 16, 1024);
        const uint64_t da_lo = smem_desc_sw128(smem_u32(smem + kOffQLo), 16, 1024);
        const uint64_t db_hi = smem_desc_sw128(smem_u32(smem + kOffKHi), 16, 1024);
        const uint64_t db_lo = smem_desc_sw128(smem_u32(smem + kOffKLo), 16, 1024);
        TileCursor cur;
        for (cur.init(a, cid, n_clusters, csize); cur.tile < a.n_tiles; cur.next(a, n_clusters)) {
            const Geo g = decode_tile<W>(a, cur, crank, csize);
            if (!g.live) continue;
            const uint32_t buf = it & 1u;
            ++it;
            if (g.n_own == 0) continue;
            const uint32_t use = buf ? acc_use1 : acc_use0;
            mbar_wait(bar(kAccEmpty + buf), (use & 1u) ^ 1u);  // epilogue drained this accumulator
            if (buf) ++acc_use1; else ++acc_use0;
            stamp(tr, n_tile, kEvMmaAccEmpty);
            const int n_cols = min(kAccCols, (g.n_mma + 15) & ~15);  // UMMA N: multiple of 16
            const uint32_t idesc = instr_desc_tf32(kRows, n_cols);
            const uint32_t d = tm + buf * kAccCols + (uint32_t)g.mcol0;
            // Pass order hi*hi, lo*hi, hi*lo.  hi*hi reads the tiles exactly as TMA landed them, so it is issued
            // as soon as the boxes are there and runs while the splitters still write the lo twins; lo*hi follows
            // the Q twin, and K_hi -- read by the first two passes only -- is released for the next head's
            // load before hi*lo (which waits for the K twin) is issued.
            mbar_wait(bar(kKFull), n_tile & 1u);
            mbar_wait(bar(kQFull), n_tile & 1u);
            tc_fence_after();
            stamp(tr, n_tile, kEvMmaAReady);
#pragma unroll
            for (int pass = 0; pass < 3; ++pass) {
                const uint64_t da = pass == 1 ? da_lo : da_hi;
                const uint64_t db = pass == 2 ? db_lo : db_hi;
                if (pass == 1) {
                    mbar_wait(bar(kQLoReady), n_tile & 1u);
                    tc_fence_after();
                }
                if (pass == 2) {
                    // the K twin is complete: the splitters no longer read K_hi either, so the commit below (it
                    // covers the two passes issued so far) hands K_hi back to the TMA producer
                    mbar_wait(bar(kKLoReady), n_tile & 1u);
                    tc_fence_after();
                    umma_commit_if(bar(kKFree), elected);
                    stamp(tr, n_tile, kEvMmaB0);
                }
#pragma unroll  // (a rolled loop saves 80 instructions of code and costs 4 % of the kernel: the issue rate of the MMAs matters)
                for (int ks = 0; ks < kHeadDim / 8; ++ks)
                    umma_tf32_ss_if(d, da + (uint64_t)(((ks >> 2) * kQHalfBytes + (ks & 3) * 32) >> 4),
                                    db + (uint64_t)(((ks >> 2) * kKHalfBytes + (ks & 3) * 32) >> 4), idesc, (pass | ks) != 0,
                                    elected);
            }
            umma_commit_if(bar(kOpFree), elected);
            umma_commit_if(bar(kAccFull + buf), elected);
            stamp(tr, n_tile, kEvMmaIssued);
            ++n_tile;
        }
    } else if (warp >= 4 && warp < 8) {
        // ================= operand splitters: write the lo twins =================
        const int t = tid - 4 * 32;
        uint32_t n_tile = 0;
        const bool tr = a.trace && blockIdx.x == (a.dbg >> 8) && t == 0;
        TileCursor cur;
        for (cur.init(a, cid, n_clusters, csize); cur.tile < a.n_tiles; cur.next(a, n_clusters)) {
            const Geo g = decode_tile<W>(a, cur, crank, csize);
            if (!g.live || g.n_own == 0) continue;
            mbar_wait(bar(kOpFree), (n_tile & 1u) ^ 1u);  // the previous tile's MMAs no longer read the lo twins (first lap passes)
            mbar_wait(bar(kKFull), n_tile & 1u);
            stamp(tr, n_tile, kEvSplFull);
            for (int half = 0; half < 2; ++half)
                for (int c = 0; c < g.n_chunks; ++c)
                    split_lo<kBoxBytes>(smem + kOffKHi + half * kKHalfBytes + c * kBoxBytes,
                                        smem + kOffKLo + half * kKHalfBytes + c * kBoxBytes, t);
            fence_proxy_async_smem();  // generic-proxy stores must be visible to the tensor core's async proxy
            mbar_arrive(bar(kKLoReady));
            stamp(tr, n_tile, kEvSplK0Done);
            mbar_wait(bar(kQFull), n_tile & 1u);
            if (g.copies == 4) {
                for (int half = 0; half < 2; ++half)
                    split_lo_quad(smem + kOffQHi + half * kQHalfBytes, smem + kOffQLo + half * kQHalfBytes, t);
            } else if (g.copies == 2) {
                for (int half = 0; half < 2; ++half)
                    split_lo_dup(smem + kOffQHi + half * kQHalfBytes, smem + kOffQLo + half * kQHalfBytes, t);
            } else {
                split_lo<kQBytes>(smem + kOffQHi, smem + kOffQLo, t);
            }
            fence_proxy_async_smem();
            mbar_arrive(bar(kQLoReady));
            stamp(tr, n_tile, kEvSplQDone);
            ++n_tile;
        }
    } else if (warp >= 8) {
        // ================= epilogue warpgroups (A: even tiles, B: odd tiles) =================
        const int grp = (warp - 8) >> 2, ewarp = warp & 3;
        uint32_t it = 0, acc_use = 0, n_x = 0;
        const bool tr = a.trace && blockIdx.x == (a.dbg >> 8) && ewarp == 0 && lane == 0;
        // the other warpgroup's tiles only have to be counted: a tile is live when its first token row exists
        TileCursor cur;
        for (cur.init(a, cid, n_clusters, csize); cur.tile < a.n_tiles; cur.next(a, n_clusters)) {
            const bool mine = (it & 1u) == (uint32_t)grp;
            if (!mine) {
                if (cur.tb * kRows < a.utts[cur.ub].n_tokens) ++it;
                continue;
            }
            const Geo g = decode_tile<W>(a, cur, crank, csize);
            if (!g.live) continue;
            const uint32_t seq = it;
            ++it;
            if (g.n_own > 0) {
                mbar_wait(bar(kAccFull + grp), acc_use & 1u);
                tc_fence_after();
            }
            stamp(tr, seq, kEvEpiAccFull);
            const bool released = epilogue_tile<W>(g, a, smem, tmem_base + (uint32_t)grp * kAccCols, grp, ewarp, lane, csize,
                                                   n_x & 1u, tr, seq, bar(kAccEmpty + grp));
            ++n_x;
            if (g.n_own > 0) {
                if (!released) {
                    tc_fence_before();
                    mbar_arrive(bar(kAccEmpty + grp));
                }
                ++acc_use;
            }
        }
    }

    // ---- teardown: nobody leaves while a peer may still read our statistics ----------------
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

}  // namespace tc

int read_capture_trace(long long *h_out, int capacity) {
    const int n = tc::kTraceTiles * tc::kNumEv;
    if (capacity < n) {
        set_error("wca_debug_capture_trace: capacity %d < %d", capacity, n);
        return WCA_ERR_INVALID;
    }
    WCA_CUDA(cudaMemcpyFromSymbol(h_out, tc::g_trace, sizeof(long long) * n));
    return n;
}

bool capture_tc_supported(int max_tokens, int max_frames, int medfilt_width) {
    (void)max_tokens;
    const bool width_ok = medfilt_width == 1 || medfilt_width == 3 || medfilt_width == 5 || medfilt_width == 7;
    return width_ok && max_frames <= 8 * tc::kMaxOwn;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int encode_map(EncodeTiledFn encode, CUtensorMap *map, const float *base, int64_t rows, int64_t cols, int64_t ld,
                      int box_rows) {
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)tc::kBoxCols, (cuuint32_t)box_rows};
    const cuuint32_t elem[2] = {1, 1};
    const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims, strides, box, elem,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows %lld, cols %lld, ld %lld)", (int)r, (long long)rows,
                  (long long)cols, (long long)ld);
        return WCA_ERR_CUDA;
    }
    return WCA_OK;
}

int launch_capture_tc(const float *const *h_q_layers, const float *const *h_k_layers, int n_layers, int n_heads,
                      int64_t ld_q, int64_t ld_k, int64_t q_rows, int64_t k_rows, const wca_utt_t *d_utts, int n_utts,
                      int max_tokens, int max_frames, int medfilt_width, float qk_scale, float *d_ws, float *d_partials,
                      unsigned flags, int sm_count, cudaStream_t stream) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        WCA_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !fn) {
            set_error("capture_tc: the driver does not export cuTensorMapEncodeTiled");
            return WCA_ERR_CUDA;
        }
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    // The descriptors only depend on the operand buffers (base pointers, rows, pitch), not on the utterances of the launch:
    // the launches of one batch (one per cluster-size bucket) and, with a caching allocator, of consecutive batches reuse
    // them.  144 cuTensorMapEncodeTiled calls cost 0.15-0.3 ms of host time per launch, which the GPU spent idle between
    // the bucket launches of a LibriSpeech-shaped step.  One entry, keyed by the device and the operand buffers, guarded by a
    // mutex (the entry points stay thread-safe; threads driving different devices only evict each other's entry).
    struct MapKey {
        const float *q[WCA_MAX_LAYERS], *k[WCA_MAX_LAYERS];
        int64_t ld_q, ld_k, q_rows, k_rows;
        int n_layers, n_heads, device;
    };
    int device = 0;
    WCA_CUDA(cudaGetDevice(&device));
    static std::mutex cache_mutex;
    static MapKey cache_key;
    static tc::TensorMaps cache_maps;
    static bool cache_valid = false;
    MapKey key;
    memset(&key, 0, sizeof(key));
    for (int l = 0; l < n_layers; ++l) {
        key.q[l] = h_q_layers[l];
        key.k[l] = h_k_layers[l];
    }
    key.ld_q = ld_q; key.ld_k = ld_k; key.q_rows = q_rows; key.k_rows = k_rows;
    key.n_layers = n_layers; key.n_heads = n_heads; key.device = device;
    tc::TensorMaps maps;
    bool hit = false;
    {
        std::lock_guard<std::mutex> lock(cache_mutex);
        if (cache_valid && memcmp(&key, &cache_key, sizeof(key)) == 0) {
            memcpy(&maps, &cache_maps, sizeof(maps));
            hit = true;
        }
    }
    if (!hit) {
        memset(&maps, 0, sizeof(maps));
        for (int l = 0; l < n_layers; ++l) {
            for (int v = 0; v < 3; ++v) {
                const int rc = encode_map(encode, &maps.q[v][l], h_q_layers[l], q_rows, (int64_t)n_heads * kHeadDim, ld_q,
                                          v == 2 ? tc::kStageRows / 2 : (v + 1) * tc::kStageRows);
                if (rc) return rc;
            }
            for (int v = 0; v < 4; ++v) {
                const int rc = encode_map(encode, &maps.k[v][l], h_k_layers[l], k_rows, (int64_t)n_heads * kHeadDim, ld_k,
                                          (v + 1) * tc::kStageRows);
                if (rc) return rc;
            }
        }
        std::lock_guard<std::mutex> lock(cache_mutex);
        memcpy(&cache_key, &key, sizeof(key));
        memcpy(&cache_maps, &maps, sizeof(maps));
        cache_valid = true;
    }
    // CTAs per cluster = 224-frame slabs the longest utterance of the launch needs: 1-6 or 8.  (7 would leave more SMs idle
    // than 8: clusters do not straddle GPCs, and a GPC of 18 SMs holds two clusters of 7 or of 8, three of 5 or 6, six of 3.)
    int csize = (max_frames + tc::kMaxOwn - 1) / tc::kMaxOwn;
    if (csize == 7) csize = 8;
    const int tok_blocks = (max_tokens + tc::kRows - 1) / tc::kRows;
    const int lh_count = n_layers * n_heads;
    const long long tiles = (long long)n_utts * lh_count * tok_blocks;
    if (tiles > 0x7fffffffLL) {
        set_error("capture_tc: %lld tiles exceed the tile index range", tiles);
        return WCA_ERR_UNSUPPORTED;
    }
    tc::KernelArgs a;
    a.utts = d_utts;
    a.ws = d_ws;
    a.partials = d_partials;
    a.n_heads = n_heads;
    a.lh_count = lh_count;
    a.tok_blocks = tok_blocks;
    a.n_tiles = (int)tiles;
    // (q s).(k s) with s = 64^-1/4 is q.k / 8: the operands go to the tensor core unscaled and the exact
    // power of two is applied after the median filter (scaling by 2^-3 commutes with it bit for bit)
    a.s = 0.125f;
    a.qk_scale = qk_scale * 0.125f;
    a.raw_logits = (flags & WCA_CAPTURE_RAW_LOGITS) ? 1 : 0;
    a.trace = (flags & WCA_CAPTURE_TRACE) ? 1 : 0;
    a.dbg = flags & 0xff00u;
    const int width = a.raw_logits ? 1 : medfilt_width;

    long long clusters = sm_count / csize;  // one persistent CTA per SM
    if (clusters > tiles) clusters = tiles;
    if (clusters < 1) clusters = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(clusters * csize));
    cfg.blockDim = dim3(tc::kThreads);
    cfg.dynamicSmemBytes = tc::kSmemBytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)csize;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;

    // A persistent grid must be co-resident: clusters cannot straddle GPCs, so fewer clusters of 4 / 8 CTAs fit than
    // sm_count / csize (16 of 8 on a B200, not 18) and the surplus ones would run as a second wave after the first has
    // walked its whole tile list - twice the time.  Ask the runtime how many fit and size the grid to that.
#define WCA_GO(Wv)                                                                                              \
    do {                                                                                                        \
        WCA_CUDA(cudaFuncSetAttribute(tc::capture_tc_kernel<Wv>, cudaFuncAttributeMaxDynamicSharedMemorySize,    \
                                      tc::kSmemBytes));                                                         \
        if (csize > 1) {                                                                                        \
            static std::atomic<int> fit_tab[64][9]; /* [device][cluster size], zero-initialised */             \
            std::atomic<int> *fit = fit_tab[device & 63];                                                       \
            const int slot = csize;                                                                             \
            if (fit[slot] == 0) {                                                                               \
                int n = 0;                                                                                      \
                if (cudaOccupancyMaxActiveClusters(&n, tc::capture_tc_kernel<Wv>, &cfg) != cudaSuccess || n < 1) { \
                    (void)cudaGetLastError();                                                                   \
                    n = sm_count / csize;                                                                       \
                }                                                                                               \
                fit[slot] = n;                                                                                  \
            }                                                                                                   \
            if (clusters > fit[slot]) {                                                                         \
                clusters = fit[slot];                                                                           \
                cfg.gridDim = dim3((unsigned)(clusters * csize));                                               \
            }                                                                                                   \
        }                                                                                                       \
        WCA_CUDA(cudaLaunchKernelEx(&cfg, tc::capture_tc_kernel<Wv>, maps, a));                                 \
    } while (0)
    switch (width) {
        case 1: WCA_GO(1); break;
        case 3: WCA_GO(3); break;
        case 5: WCA_GO(5); break;
        case 7: WCA_GO(7); break;
        default:
            set_error("capture_tc: medfilt_width=%d has no tensor-core instantiation", width);
            return WCA_ERR_UNSUPPORTED;
    }
#undef WCA_GO
    WCA_LAUNCH_CHECK("capture_tc_kernel");
    return WCA_OK;
}

}  // namespace wca
