// swb_trace_tile.cu -- traceback of the short-read path, one THREAD per maximum cell.
//
// GetAlignment.call (reference SmithWaterman.java:354-436): from a maximum cell walk while the
// score is positive; the type of a positive cell is the first of alignment / insertion /
// deletion whose candidate equals H, i.e. the ">=" cascade of GetCellScore.call (:228,:236,:245)
// (SWB_F_TIE_GT: deletion / insertion / alignment, DistributedSW.java:310-326).
//
// The fill leaves, per (read pair, reference, block of CB steps):
//   * the CHECKPOINT: every lane's K cells + diagonal boundary at the block start,
//   * the SEAMS: per lane and step the boundary row the lane received from the lane above
//     (matrix row t*K of the step's column).
// A TILE = (lane t, block b) = K rows x CB skewed columns is therefore recomputable on its own:
// left column from the checkpoint, top row from the seam, corner = the checkpointed diagonal.
// A path of ~170 columns crosses ~19 tiles of 304 cells (5.8k cells) instead of the ~12 full
// 8-lane blocks (29k cells) the group-based kernel (swb_trace.cu) recomputes.
//
// One thread owns one maximum cell at a time: it recomputes the tile that holds the current
// cell (unpacked int32, column-biased like the fill: one IMAD + two DPX ops per cell) into its private column-major
// byte tile in shared memory, walks until the path leaves the tile, and repeats.  No lane
// ever talks to another lane, so there are no shuffles and no barriers inside a traceback.
//
// Bytes are enough: the walker knows the exact score of its current cell (it starts from the
// pair's maximum and subtracts the score of every move), and a candidate (NW+s, N+gap, W+gap)
// never lies more than 2*(smax+|gap|)+max|s| below H, so equality of the low 8 bits IS equality
// (tile8_ok() checks that bound; other score sets use swb_trace.cu).
#include "swb_internal.h"
#include "swb_device.cuh"

#include <algorithm>
#include <cstdlib>

namespace swb {

namespace {

constexpr int NT = 128;                      // threads per CTA
constexpr int TRACE_ROLL_K = 25;              // from this K on the tile's column loop is rolled in quads (code size)

template <int K> struct TileGeo {
    static constexpr int ROWW = Geo<K>::KW / 4;          // words per tile column: boundary row + K rows, one byte each
    static constexpr int COLS = CB + 1;                   // column 0 = the checkpointed column
    static constexpr int TILE_WORDS = ROWW * COLS;        // per thread
    static constexpr int PROF_WORDS = 5 * GL * Geo<K>::KS;   // int32 scores: [lane*4 + code] + [32 + lane] for "no column"
};

// byte (row rr, column cc) of this thread's tile; words are interleaved over the CTA's threads
// (word index * NT + tid), so every access of a warp is conflict-free whatever (rr, cc) each lane reads
template <int K>
__device__ __forceinline__ int tile_byte(const uint8_t *tile8, int rr, int cc)
{
    return tile8[(size_t)((cc * TileGeo<K>::ROWW + (rr >> 2)) * NT) * 4 + (rr & 3)];
}

// one tile column: byte 0 = boundary row, bytes 1..K = the lane's rows (low 8 bits of each score).
// Two scores per IMAD (FMA pipe: v1 * 65536 + v0, scores are in [0, 32767]), one PRMT per word.
template <int K>
__device__ __forceinline__ void store_col8(uint32_t *col, int top, const int (&H)[K], uint32_t k64k)
{
    constexpr int ROWW = TileGeo<K>::ROWW;
#pragma unroll
    for (int w = 0; w < ROWW; ++w) {
        const uint32_t v0 = (w == 0) ? (uint32_t)top : (uint32_t)H[4 * w - 1 < K ? 4 * w - 1 : 0];
        const uint32_t v1 = (4 * w + 0 < K) ? (uint32_t)H[4 * w + 0 < K ? 4 * w + 0 : 0] : 0u;
        const uint32_t v2 = (4 * w + 1 < K) ? (uint32_t)H[4 * w + 1 < K ? 4 * w + 1 : 0] : 0u;
        const uint32_t v3 = (4 * w + 2 < K) ? (uint32_t)H[4 * w + 2 < K ? 4 * w + 2 : 0] : 0u;
        const uint32_t p01 = v1 * k64k + ((w == 0 || 4 * w - 1 < K) ? v0 : 0u);
        const uint32_t p23 = v3 * k64k + v2;
        col[w * NT] = __byte_perm(p01, p23, 0x6420);
    }
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

template <int K, bool TIE_GT>
__global__ void __launch_bounds__(NT) tile_trace_kernel(const BatchParams P, const uint64_t *keys, uint32_t n_cells,
                                                        int chunk, int32_t *beginnings, int32_t *op_lens, uint32_t *ops,
                                                        int ops_stride, uint32_t k64k)
{
    using G = Geo<K>;
    using TG = TileGeo<K>;
    constexpr int KS = G::KS, ROWW = TG::ROWW;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ uint32_t seg_next;
    int *prof = reinterpret_cast<int *>(smem);                                   // [5*GL][KS]
    uint32_t *tile = smem + TG::PROF_WORDS + threadIdx.x;                         // + word * NT
    const uint8_t *tile8 = reinterpret_cast<const uint8_t *>(tile);
    uint8_t *rcodes_s = reinterpret_cast<uint8_t *>(smem + TG::PROF_WORDS + (size_t)TG::TILE_WORDS * NT);   // [GL*K]
    const int gap = P.gap, match = P.match, mismatch = P.mismatch, sbias = P.seam_bias;
    const int ag = -gap;                                                          // > 0 (tile_trace_ok)
    const uint32_t kone = k64k >> 16;                                             // 1, opaque to ptxas: keeps NW + s an IMAD

    const uint32_t c_lo = blockIdx.x * (uint32_t)chunk;
    const uint32_t c_hi = min(n_cells, c_lo + (uint32_t)chunk);
    uint32_t seg_lo = c_lo;
    while (seg_lo < c_hi) {
        // ---- segment = run of cells of one read (slot): one score profile for the whole CTA ----------
        const uint32_t slot = (uint32_t)(key_pair(keys[seg_lo]) / (uint64_t)P.n_refs);
        uint32_t seg_hi;
        {
            const uint64_t target = make_key((uint64_t)(slot + 1) * (uint64_t)P.n_refs, 0, 0);
            uint32_t lo = seg_lo, hi = c_hi;
            while (lo < hi) { const uint32_t mid = lo + ((hi - lo) >> 1); if (keys[mid] < target) lo = mid + 1; else hi = mid; }
            seg_hi = lo;
        }
        const int read_idx = P.rp_reads[slot];
        const int rh = (int)(slot & 1u);                             // the read's half in the fill's checkpoints
        const int64_t roff = P.read_off[read_idx];
        const int m = (int)(P.read_off[read_idx + 1] - roff);
        __syncthreads();
        for (int idx = threadIdx.x; idx < 5 * GL * K; idx += NT) {
            const int cc = idx / (GL * K), rem = idx - cc * GL * K;
            const int tt = rem / K, r = rem - tt * K;
            const int row = tt * K + r;
            int s = S_PAD;
            if (row < m && cc < 4) s = ((int)P.read_codes[roff + row] == cc) ? match : mismatch;
            prof[(cc < 4 ? tt * 4 + cc : 4 * GL + tt) * KS + r] = s + ag;      // the recompute is column-biased (below)
        }
        for (int idx = threadIdx.x; idx < GL * K; idx += NT)
            rcodes_s[idx] = idx < m ? P.read_codes[roff + idx] : (uint8_t)0xFE;
        if (threadIdx.x == 0) seg_next = seg_lo;
        __syncthreads();

        bool busy = false;
        int ci = 0, cj = 0, n = 0;
        const uint32_t *rw = P.ref_words;
        int64_t bk = 0;
        uint32_t w_cell = 0, w_opword = 0;
        int w_h = 0, w_beg = 0, w_len = 0;

        for (;;) {
            if (!busy) {
                const uint32_t e = atomicAdd(&seg_next, 1u);
                if (e < seg_hi) {
                    const uint64_t key = keys[e];
                    const int ro = (int)(key_pair(key) - (uint64_t)slot * (uint64_t)P.n_refs);
                    const int ref = P.ref_sorted_of[ro];
                    ci = (int)key_i(key); cj = (int)key_j(key);
                    n = P.ref_len[ref];
                    rw = P.ref_words + P.ref_word_off[ref];
                    bk = (int64_t)(slot >> 1) * P.blocks_per_rp + P.ref_blk_off[ref];
                    w_cell = e; w_opword = 0; w_beg = 0; w_len = 0;
                    w_h = P.scores[(int64_t)ro * P.n_reads + read_idx];
                    busy = w_h > 0;
                    if (!busy) { beginnings[e] = 0; op_lens[e] = 0; }       // cannot happen: keys exist for positive scores only
                }
            }
            if (!__any_sync(FULL, busy)) break;

            // ---- the tile that holds the current cell: lane t, block b -------------------------------
            const int t = busy ? (ci - 1) / K : 0;
            const int step = cj - 1 + t;
            const int b = busy ? step / CB : 0;
            int H[K], diag = 0;
            {
                load_checkpoint<K>(rec_lane<K>(P.rec, bk + b, t), busy && b > 0, [&](int w, uint32_t v) {
                    if (w < K) H[w < K ? w : 0] = half_of(v, rh); else diag = half_of(v, rh);
                });
            }
            int top[CB];
            {
                const uint32_t *sq = rec_lane<K>(P.rec, bk + b, t) + G::CKP * REC_P;
                const bool ld = busy && t > 0;                      // lane 0's boundary row is matrix row 0
                const int bias0 = sbias * (9 - t);
#pragma unroll
                for (int p = 0; p < CB / 8; ++p) {
                    uint32_t v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                    if (ld) ldg256(sq + p * REC_P, v);
#pragma unroll
                    for (int e = 0; e < 8; ++e)
                        top[8 * p + e] = ld ? half_of(v[e], rh) - (bias0 + sbias * (8 * p + e)) : 0;
                }
            }
            // reference codes of the block's 16 steps for this lane: 0-based columns j0 .. j0 + 15
            uint32_t win; int ulo, uhi;
            {
                const int j0 = b * CB - t;
                const int wi = j0 >> 4;                                  // floor (j0 may be negative in block 0)
                const uint32_t a0 = (busy && wi >= 0 && wi * 16 < n) ? __ldg(rw + wi) : 0u;
                const uint32_t a1 = (busy && wi + 1 >= 0 && (wi + 1) * 16 < n) ? __ldg(rw + wi + 1) : 0u;
                win = __funnelshift_r(a0, a1, 2 * (j0 & 15));
                ulo = -j0; uhi = busy ? n - j0 - 1 : -1;                  // step u is a real column iff ulo <= u <= uhi
            }
            store_col8<K>(tile, diag, H, k64k);

            // The tile is recomputed COLUMN-BIASED like the fill (swb_fill_bias.cu): column c = u + 1 of the tile holds
            // H'' = H + |gap| * c (column 0, the checkpoint, is unbiased), so that W + gap is the register itself and the
            // cell costs an IMAD (NW'' + s + |gap|, FMA pipe) and two DPX ops instead of three DPX ops:
            //     pre = max3(NW'' + s'', W'', |gap| * c)      the third operand is the biased zero
            //     H'' = max(N'' + gap, pre)
            // The bytes the walker reads are biased the same way (see the walk below).
            const int *pbase = prof + t * 4 * KS, *ppad = prof + (4 * GL + t) * KS;
            // one column of the tile: u = step inside the block, tv = the (unbiased) boundary value of that step
            auto column = [&](int u, int tv, uint32_t code) {
                const bool real = (u >= ulo) && (u <= uhi);
                const int *pv = real ? pbase + code * KS : ppad;
                int sv[G::KP];
                {
                    const int4 *p4 = reinterpret_cast<const int4 *>(pv);
#pragma unroll
                    for (int q = 0; q < G::KP / 4; ++q) {
                        const int4 v = p4[q];
                        sv[4 * q] = v.x; sv[4 * q + 1] = v.y; sv[4 * q + 2] = v.z; sv[4 * q + 3] = v.w;
                    }
                }
                const int floorc = ag * (u + 1);
                const int topb = tv + floorc;
                int nw = diag, nn = topb;
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    const int tt = nw * (int)kone + sv[r];               // NW'' + s''           (IMAD, FMA pipe)
                    const int pre = __vimax3_s32(tt, H[r], floorc);      // max(., W'', 0'')
                    nw = H[r];
                    H[r] = __viaddmax_s32(nn, gap, pre);                 // max(N'' + gap, .)
                    nn = H[r];
                }
                diag = topb;
                store_col8<K>(tile + (u + 1) * ROWW * NT, topb, H, k64k);
            };
            if constexpr (K < TRACE_ROLL_K) {
#pragma unroll
                for (int u = 0; u < CB; ++u) column(u, top[u], (win >> (2 * u)) & 3u);
            } else {
                // K >= 25: 16 unrolled columns of 32 .. 64 rows are 34 .. 60 KB of code (ncu, K = 64: no_instruction stalls;
                // K = 32: 250 bp batches 10.3 -> 8.9 ms); rolled in quads, the quad's four boundary values picked without
                // dynamic register indexing.  K = 19 is faster unrolled (4.0 vs 4.1 ms per step).
#pragma unroll 1
                for (int q = 0; q < CB / 4; ++q) {
                    int tv[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        int x = top[e];
#pragma unroll
                        for (int qq = 1; qq < CB / 4; ++qq) x = (q == qq) ? top[4 * qq + e] : x;
                        tv[e] = x;
                    }
                    const uint32_t wq = win >> (8 * q);
#pragma unroll
                    for (int e = 0; e < 4; ++e) column(4 * q + e, tv[e], (wq >> (2 * e)) & 3u);
                }
            }

            // ---- walk inside the tile (SmithWaterman.java:380-409) ------------------------------------
            // pw = shared-memory address of the tile word that holds the current cell (row r = 4*w + rb, column c);
            // the word above (rows 4w-4..4w-1) and the two words of column c-1 sit at constant offsets, and one
            // PRMT over (word above : word) picks byte rb+3 = row r-1 or rb+4 = row r, whatever rb is.
            if (busy) {
                constexpr int UPB = NT * 4, COLB = ROWW * NT * 4;       // byte offsets: one word up, one column left
                int r = ci - t * K;                                     // 1..K
                int c = step - b * CB + 1;                              // 1..CB
                const int cbase = cj - c;                               // global column = cbase + c
                const uint8_t *pw = tile8 + (size_t)((c * ROWW + (r >> 2)) * NT) * 4;
                uint32_t sel3 = (uint32_t)(r & 3) + 3u;                 // PRMT selector of row r-1; +1: row r
                // codes of the block's columns in reverse order: column c at bits 2*(CB - c), so a step left is >> 2
                uint32_t wsh = __brev(win);
                wsh = ((wsh & 0x55555555u) << 1) | ((wsh >> 1) & 0x55555555u);
                wsh >>= 2 * (CB - c);                                   // reference code of column c in bits 0..1
                const uint8_t *qp = rcodes_s + (ci - 1);
                uint32_t *op_ptr = ops + (size_t)w_cell * ops_stride + (w_len >> 4);
                uint32_t sh = 2u * ((uint32_t)w_len & 15u);
                int lastc = c;
                for (;;) {
                    const uint32_t w_c = *reinterpret_cast<const uint32_t *>(pw), u_c = *reinterpret_cast<const uint32_t *>(pw - UPB);
                    const uint32_t w_l = *reinterpret_cast<const uint32_t *>(pw - COLB), u_l = *reinterpret_cast<const uint32_t *>(pw - COLB - UPB);
                    // low byte = the score's low 8 bits; the other bytes are masked after the add
                    const int hn = (int)prmt(u_c, w_c, sel3), hw = (int)prmt(u_l, w_l, sel3 + 1u), hnw = (int)prmt(u_l, w_l, sel3);
                    const int sc = ((uint32_t)*qp == (wsh & 3u)) ? match : mismatch;
                    // biased bytes: column c holds H + |gap| * c, so with whb = H(r, c) + |gap| * c
                    //   alignment  H = NW + s    <=>  NW'' + s + |gap| == whb      (NW'' carries |gap| * (c - 1))
                    //   insertion  H = N + gap   <=>  N'' + gap == whb            (same column)
                    //   deletion   H = W + gap   <=>  W'' == whb
                    const int whb = w_h + ag * c;
                    const bool eq_a = ((hnw + sc + ag - whb) & 0xff) == 0, eq_i = ((hn + gap - whb) & 0xff) == 0,
                               eq_d = ((hw - whb) & 0xff) == 0;
                    const uint32_t op = TIE_GT ? (eq_d ? 3u : (eq_i ? 2u : 1u)) : (eq_a ? 1u : (eq_i ? 2u : 3u));
                    lastc = c;
                    w_opword |= op << sh;
                    sh = (sh + 2u) & 31u;
                    if (sh == 0u) { *op_ptr = w_opword; w_opword = 0; }
                    op_ptr += (sh == 0u);
                    ++w_len;
                    w_h -= (op == 1u) ? sc : gap;
                    const int up = op != 3u, left = op != 2u;           // alignment: both
                    r -= up; qp -= up; sel3 -= up;
                    if (sel3 < 3u) { sel3 = 6u; pw -= UPB; }
                    c -= left; pw -= left ? COLB : 0; wsh >>= 2 * left;
                    if (w_h <= 0 || r == 0 || c == 0) break;            // done, or the path left this tile
                }
                ci = t * K + r; cj = cbase + c;
                w_beg = cbase + lastc;
                if (w_h <= 0) {
                    if (sh) *op_ptr = w_opword;
                    beginnings[w_cell] = w_beg;
                    op_lens[w_cell] = w_len;
                    busy = false;
                }
            }
        }
        seg_lo = seg_hi;
    }
}

// ---------------------------------------------------------------------------------------
// Max-cell enumeration (ScoreMatrix.call, SmithWaterman.java:176-185), one thread per candidate tile.
//
// The fill's tile maxima may be SUBSAMPLED (BatchParams::tmx_slack > 0): flag_tiles then hands over every tile
// whose tracked maximum is within the slack of the pair's tracked maximum, and the pair score in P.scores is a
// lower bound (score - slack <= tracked <= score).  Two passes make everything exact:
//   scan : recompute the tile from its record (unpacked int32 DPX, 3 ops/cell + compare/select score), find its
//          exact maximum E over the real rows (only values >= the tracked pair score matter) and the cells == E
//          (<= 4 buffered per tile); atomicMax of E into the pair score  ->  P.scores is exact after the pass
//   emit : tiles with E == the (now exact) pair score write their cells as keys (pair, i, j) -- one
//          warp-aggregated reservation; tiles with more than 4 such cells (tie-heavy) recompute and emit directly.
// The radix sort of the keys is the reference's row-major list order.  With exact tile maxima (slack 0) every
// candidate is a real one and the scan finds E == score at once.
// The step loop is rolled in quads (fully unrolled it thrashed the instruction cache: 68 warps stalled on
// no_instruction per issue, 1.86 ms instead of 0.19).
// bit mask over a lane's K rows: 32 bits, 64 for the LONG classes (K = 40 .. 64)
template <int K> struct RowMask { using type = uint32_t; };
template <> struct RowMask<40> { using type = uint64_t; };
template <> struct RowMask<48> { using type = uint64_t; };
template <> struct RowMask<56> { using type = uint64_t; };
template <> struct RowMask<64> { using type = uint64_t; };
__device__ __forceinline__ int mask_ffs(uint32_t m) { return __ffs((int)m); }
__device__ __forceinline__ int mask_ffs(uint64_t m) { return __ffsll((long long)m); }

template <int K>
struct TileSweep {
    using mask_t = typename RowMask<K>::type;
    static_assert(K <= 8 * (int)sizeof(mask_t), "row mask too narrow for K");
    int rc[K], H[K];
    int diag, S, t, b;
    uint32_t win;
    mask_t rowok;
    int ulo, uhi;
    const uint32_t *sq;
    bool has_top;
    uint64_t pkey;
    int64_t pair;

    __device__ __forceinline__ void setup(const BatchParams &P, const TileTask &T, bool live)
    {
        using G = Geo<K>;
        const int rp = (int)(T.rp_half >> 1), rh = (int)(T.rp_half & 1u), ref = (int)T.ref_sorted;
        t = (int)T.lane; b = (int)T.block;
        S = 0x7fffffff; pkey = 0; pair = 0; diag = 0; win = 0; rowok = 0; ulo = 0; uhi = -1;
        sq = P.rec; has_top = false;
#pragma unroll
        for (int r = 0; r < K; ++r) { rc[r] = 0xFE; H[r] = 0; }
        if (!live) return;
        const int read_idx = P.rp_reads[2 * rp + rh];
        const int64_t off = P.read_off[read_idx];
        const int m = (int)(P.read_off[read_idx + 1] - off);
        const int n = P.ref_len[ref];
        const int64_t ro = P.ref_orig[ref];
        pair = ro * P.n_reads + read_idx;
        S = P.scores[pair];
        pkey = (uint64_t)T.rp_half * (uint64_t)P.n_refs + (uint64_t)ro;
#pragma unroll
        for (int r = 0; r < K; ++r) {
            const int row = t * K + r;
            rc[r] = (row < m) ? (int)P.read_codes[off + row] : 0xFE;
            if (row < m) rowok |= (mask_t)1 << r;
        }
        const int64_t blk = (int64_t)rp * P.blocks_per_rp + P.ref_blk_off[ref] + b;
        if (b > 0) {
            load_checkpoint<K>(rec_lane<K>(P.rec, blk, t), true, [&](int w, uint32_t v) {
                if (w < K) H[w < K ? w : 0] = half_of(v, rh); else diag = half_of(v, rh);
            });
        }
        sq = rec_lane<K>(P.rec, blk, t) + G::CKP * REC_P;
        has_top = t > 0;                                         // lane 0's boundary row is matrix row 0
        const uint32_t *rw = P.ref_words + P.ref_word_off[ref];
        const int j0 = b * CB - t;
        const int wi = j0 >> 4;
        const uint32_t a0 = (wi >= 0 && wi * 16 < n) ? __ldg(rw + wi) : 0u;
        const uint32_t a1 = (wi + 1 >= 0 && (wi + 1) * 16 < n) ? __ldg(rw + wi + 1) : 0u;
        win = __funnelshift_r(a0, a1, 2 * (j0 & 15));
        ulo = -j0; uhi = n - j0 - 1;
        (void)rh;
    }

    // fn(j, cmax, H) after every real column; cmax = maximum over ALL K rows of the column
    template <class Fn>
    __device__ __forceinline__ void run(const BatchParams &P, int rh, Fn &&fn)
    {
        const int gap = P.gap, match = P.match, mismatch = P.mismatch;
        const int bias0 = P.seam_bias * (9 - t);
        uint32_t sv[CB];                                        // the seam: two 32-byte pieces
#pragma unroll
        for (int p = 0; p < CB / 8; ++p) {
            uint32_t v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            if (has_top) ldg256(sq + p * REC_P, v);
#pragma unroll
            for (int e = 0; e < 8; ++e) sv[8 * p + e] = v[e];
        }
#pragma unroll 1
        for (int q = 0; q < CB / 4; ++q) {
            // the quad's four seam words without dynamic register indexing
            uint32_t av[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                uint32_t x = sv[e];
#pragma unroll
                for (int qq = 1; qq < CB / 4; ++qq) x = (q == qq) ? sv[4 * qq + e] : x;
                av[e] = x;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int u = 4 * q + e;
                const int top = has_top ? half_of(av[e], rh) - (bias0 + P.seam_bias * u) : 0;
                const bool real = (u >= ulo) && (u <= uhi);
                const int c = real ? (int)((win >> (2 * u)) & 3u) : 0xFD;       // 0xFD: matches no row
                int nw = diag, nn = top, cmax = 0;
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    const int sc = (rc[r] == c) ? match : mismatch;
                    const int x = __viaddmax_s32_relu(nw, sc, 0);
                    const int pre = __viaddmax_s32(H[r], gap, x);
                    nw = H[r];
                    H[r] = real ? __viaddmax_s32(nn, gap, pre) : 0;       // left of the matrix: zeros; right of it: never used
                    nn = H[r];
                    cmax = max(cmax, H[r]);
                }
                diag = top;
                if (real) fn(b * CB - t + u + 1, cmax, H);
            }
        }
    }
};

struct TileHit { int32_t emax; uint32_t n; uint32_t code[4]; };

template <int K>
__global__ void __launch_bounds__(NT) tile_scan_kernel(const BatchParams P, const TileTask *tasks,
                                                       const uint32_t *n_tasks_ptr, uint32_t cap_tasks, TileHit *hits)
{
    __shared__ uint32_t hitbuf[4 * NT];
    const uint32_t n_tasks = min(*n_tasks_ptr, cap_tasks);        // written by flag_tiles on the same stream
    const uint32_t n_threads = gridDim.x * blockDim.x;
    for (uint32_t task = blockIdx.x * blockDim.x + threadIdx.x; task < n_tasks; task += n_threads) {
        const TileTask T = tasks[task];
        TileSweep<K> W;
        W.setup(P, T, true);
        // rows beyond the read's end sit below every real row, never feed one, and may exceed the real maximum
        // when mismatch > 0: the exact maximum is taken over the real rows only (rowok)
        int E = max(W.S, 1);                                     // cells below the tracked pair score cannot be maximal
        uint32_t n_hit = 0;
        const int t = W.t;
        using mask_t = typename TileSweep<K>::mask_t;
        const mask_t rowok = W.rowok;
        W.run(P, (int)(T.rp_half & 1u), [&](int j, int cmax, const int (&H)[K]) {
            if (cmax < E) return;
            int vm = 0;
#pragma unroll
            for (int r = 0; r < K; ++r) vm = max(vm, ((rowok >> r) & 1u) ? H[r] : 0);
            if (vm < E) return;
            if (vm > E) { E = vm; n_hit = 0; }
            mask_t rm = 0;
#pragma unroll
            for (int r = 0; r < K; ++r) rm |= (H[r] == E) ? ((mask_t)1 << r) : (mask_t)0;
            rm &= rowok;
            while (rm) {
                const int r = mask_ffs(rm) - 1;
                rm &= rm - 1;
                if (n_hit < 4) hitbuf[n_hit * NT + threadIdx.x] = ((uint32_t)(t * K + r + 1) << KEY_J_BITS) | (uint32_t)j;
                ++n_hit;
            }
        });
        if (n_hit && E > W.S) atomicMax(P.scores + W.pair, E);
        TileHit o;
        o.emax = n_hit ? E : 0; o.n = n_hit;
#pragma unroll
        for (int h = 0; h < 4; ++h) o.code[h] = (uint32_t)h < n_hit ? hitbuf[h * NT + threadIdx.x] : 0u;
        hits[task] = o;
    }
}

// SEL (hits mode): a pair emits only if its bit in P.sel is set; a separate instantiation keeps the plain emit as it was
template <int K, bool SEL>
__global__ void __launch_bounds__(NT) tile_emit_kernel(const BatchParams P, const TileTask *tasks,
                                                       const uint32_t *n_tasks_ptr, uint32_t cap_tasks, const TileHit *hits,
                                                       uint64_t *keys, uint32_t cap, uint32_t *count)
{
    const uint32_t n_tasks = min(*n_tasks_ptr, cap_tasks);
    const int lane = threadIdx.x & 31;
    const uint32_t n_threads = gridDim.x * blockDim.x;
    const uint32_t iters = (n_tasks + n_threads - 1) / n_threads; // whole warps iterate together
    for (uint32_t it = 0; it < iters; ++it) {
        const uint32_t task = it * n_threads + blockIdx.x * blockDim.x + threadIdx.x;
        const bool live = task < n_tasks;
        TileTask T = TileTask{0, 0, 0, 0};
        TileHit h; h.emax = 0; h.n = 0;
        uint64_t pkey = 0;
        bool hot = false;
        if (live) {
            T = tasks[task];
            h = hits[task];
            const int read_idx = P.rp_reads[T.rp_half];
            const int64_t ro = P.ref_orig[T.ref_sorted];
            pkey = ((uint64_t)T.rp_half * (uint64_t)P.n_refs + (uint64_t)ro) << (KEY_J_BITS + KEY_I_BITS);
            hot = h.n > 0 && h.emax == P.scores[ro * P.n_reads + read_idx];   // exact since the scan pass
            if (SEL) {
                const uint64_t b = (uint64_t)T.rp_half * (uint64_t)P.n_refs + (uint64_t)ro;
                hot = hot && ((P.sel[b >> 5] >> (b & 31)) & 1u);
            }
        }
        const uint32_t mine = hot ? min(h.n, 4u) : 0u;
        uint32_t inc = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
        const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
        uint32_t base = 0;
        if (lane == 31 && total) base = atomicAdd(count, total);
        base = __shfl_sync(0xffffffffu, base, 31) + inc - mine;
        if (hot && h.n <= 4) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if ((uint32_t)k < mine && base + k < cap) keys[base + k] = pkey | h.code[k];
        } else if (hot) {
            // tie-heavy tile: more cells than the scan could buffer -- recompute, one atomic per cell beyond the first four
            TileSweep<K> W;
            W.setup(P, T, true);
            const int S = h.emax;
            const int t = W.t;
            using mask_t = typename TileSweep<K>::mask_t;
            const mask_t rowok = W.rowok;
            uint32_t seen = 0;
            W.run(P, (int)(T.rp_half & 1u), [&](int j, int cmax, const int (&H)[K]) {
                if (cmax < S) return;
                mask_t rm = 0;
#pragma unroll
                for (int r = 0; r < K; ++r) rm |= (H[r] == S) ? ((mask_t)1 << r) : (mask_t)0;
                rm &= rowok;
                while (rm) {
                    const int r = mask_ffs(rm) - 1;
                    rm &= rm - 1;
                    const uint32_t k = seen < 4 ? base + seen : atomicAdd(count, 1u);
                    ++seen;
                    if (k < cap) keys[k] = pkey | ((uint32_t)(t * K + r + 1) << KEY_J_BITS) | (uint32_t)j;
                }
            });
        }
    }
}

template <int K>
cudaError_t launch_tile_locate_k(const BatchParams &P, const TileTask *tasks, const uint32_t *n_tasks, uint32_t cap_tasks,
                                 void *hits, uint64_t *keys, uint32_t cap, uint32_t *count, int sm_count, int phase, cudaStream_t st)
{
    // the task count is read on the device; size the grid for the capacity, capped at a few waves
    const int64_t ctas = std::max<int64_t>(1, std::min<int64_t>(((int64_t)cap_tasks + NT - 1) / NT, (int64_t)sm_count * 32));
    if (phase == 0) tile_scan_kernel<K><<<(unsigned)ctas, NT, 0, st>>>(P, tasks, n_tasks, cap_tasks, static_cast<TileHit *>(hits));
    else if (P.sel) tile_emit_kernel<K, true><<<(unsigned)ctas, NT, 0, st>>>(P, tasks, n_tasks, cap_tasks, static_cast<const TileHit *>(hits), keys, cap, count);
    else tile_emit_kernel<K, false><<<(unsigned)ctas, NT, 0, st>>>(P, tasks, n_tasks, cap_tasks, static_cast<const TileHit *>(hits), keys, cap, count);
    return cudaGetLastError();
}

template <int K>
cudaError_t launch_tile_trace_k(const BatchParams &P, const uint64_t *keys, uint32_t n_cells, int32_t *beginnings,
                                int32_t *op_lens, uint32_t *ops, int ops_stride, int sm_count, cudaStream_t st)
{
    using TG = TileGeo<K>;
    if (n_cells == 0) return cudaSuccess;
    const size_t smem = ((size_t)TG::PROF_WORDS + (size_t)TG::TILE_WORDS * NT) * sizeof(uint32_t) + (((size_t)GL * K + 15) / 16) * 16;
    static PerDeviceOnce attr;
    {
        const cudaError_t e = attr.run([&] {
            cudaError_t e1 = cudaFuncSetAttribute(tile_trace_kernel<K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(tile_trace_kernel<K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            return e1;
        });
        if (e != cudaSuccess) return e;
    }
    // chunks of the sorted cell list: many per SM for balance, each long enough to amortise its profile.  In hits mode
    // (P.sel) a read has a handful of cells: a CTA walks its chunk's reads one after another, so a chunk of 2 * NT
    // cells would serialise up to 2 * NT walks in one CTA; every cell may start a chunk of its own there.
    const int per_sm = 16;
    const int chunk = (int)std::max<int64_t>(P.sel ? 1 : 2 * NT, ((int64_t)n_cells + (int64_t)sm_count * per_sm - 1) / ((int64_t)sm_count * per_sm));
    const int64_t ctas = ((int64_t)n_cells + chunk - 1) / chunk;
    if (P.tie_gt) tile_trace_kernel<K, true><<<(unsigned)ctas, NT, smem, st>>>(P, keys, n_cells, chunk, beginnings, op_lens, ops, ops_stride, 65536u);
    else          tile_trace_kernel<K, false><<<(unsigned)ctas, NT, smem, st>>>(P, keys, n_cells, chunk, beginnings, op_lens, ops, ops_stride, 65536u);
    return cudaGetLastError();
}

}  // namespace

// Equality of the low 8 bits must be equality: a candidate lies at most 2*(smax+|gap|) + max|s| below H.
bool tile_trace_ok(int match, int mismatch, int gap)
{
    if (gap >= 0) return false;
    const int64_t smax = std::max<int64_t>({match, mismatch, 0});
    const int64_t sabs = std::max<int64_t>(std::llabs((long long)match), std::llabs((long long)mismatch));
    return 2 * (smax - (int64_t)gap) + sabs < 250;
}

size_t locate_hit_bytes() { return sizeof(TileHit); }

// phase 0: scan (exact tile maxima -> exact pair scores, buffered cells); phase 1: emit keys
cudaError_t launch_locate(int K, const BatchParams &P, const TileTask *tasks, const uint32_t *n_tasks,
                          uint32_t cap_tasks, void *hits, uint64_t *keys, uint32_t cap, uint32_t *count, int sm_count,
                          int phase, cudaStream_t st)
{
    switch (K) {
        case 4:  return launch_tile_locate_k<4>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 5:  return launch_tile_locate_k<5>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 7:  return launch_tile_locate_k<7>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 10: return launch_tile_locate_k<10>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 8:  return launch_tile_locate_k<8>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 13: return launch_tile_locate_k<13>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 16: return launch_tile_locate_k<16>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 19: return launch_tile_locate_k<19>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 25: return launch_tile_locate_k<25>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 32: return launch_tile_locate_k<32>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 40: return launch_tile_locate_k<40>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 48: return launch_tile_locate_k<48>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 56: return launch_tile_locate_k<56>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
        case 64: return launch_tile_locate_k<64>(P, tasks, n_tasks, cap_tasks, hits, keys, cap, count, sm_count, phase, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_tile_trace(int K, const BatchParams &P, const uint64_t *keys, uint32_t n_cells, int32_t *beginnings,
                              int32_t *op_lens, uint32_t *ops, int ops_stride_words, int sm_count, cudaStream_t st)
{
    switch (K) {
        case 4:  return launch_tile_trace_k<4>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 5:  return launch_tile_trace_k<5>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 7:  return launch_tile_trace_k<7>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 10: return launch_tile_trace_k<10>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 8:  return launch_tile_trace_k<8>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 13: return launch_tile_trace_k<13>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 16: return launch_tile_trace_k<16>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 19: return launch_tile_trace_k<19>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 25: return launch_tile_trace_k<25>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 32: return launch_tile_trace_k<32>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 40: return launch_tile_trace_k<40>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 48: return launch_tile_trace_k<48>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 56: return launch_tile_trace_k<56>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 64: return launch_tile_trace_k<64>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
    }
    return cudaErrorInvalidValue;
}

}  // namespace swb
