// swb_wide.cu -- the general ("wide") path: int32 scores, any read length, any scores that do
// not overflow int32, 8-bit symbol codes (any alphabet).  Used for long pairs (BASELINE config 3:
// 100 kbp x 100 kbp), for reads longer than the s16x2 short path's 256 rows (the reference's own
// read-length sweep goes to 500 bp, EngineerData.java:87-104) and for every score set outside
// the s16x2 domain.
//
// Same design as the short path, in int32:
//   * the matrix is cut in BANDS of 32 lanes x KL rows (KL = 8, 16 or 32, chosen per read); one
//     warp sweeps a band along the reference as a 32-lane skewed wavefront (lane t computes column
//     s - t + 1 at step s; the boundary row moves down the lanes with one __shfl_up_sync per step);
//   * the cell costs one IMAD (NW + s, FMA pipe; s from a per-warp shared-memory profile) and two
//     DPX ops (VIADDMNMX.RELU, VIADDMNMX) on the integer pipe -- SmithWaterman.java:217-252, :277-280,
//     :309-318;
//   * consecutive bands of a pair run concurrently on different warps, coupled through the band's
//     bottom row in HBM (brow), whose words validate themselves (no counter, no fence; see ld_relaxed).
//     Work is handed out by a global ticket in (band, pair) order, so a warp only ever waits for a
//     lower ticket, which is held by a running warp: no deadlock, no cooperative launch;
//   * the fill is score-only and leaves, per (band, block of 32 steps, lane), one contiguous RECORD:
//     the lane's CHECKPOINT (KL cells + the diagonal boundary at the block start) and its SEAM (the
//     boundary row it receives at each of the 32 steps), plus the lane's tile maximum.  A record is
//     all one THREAD needs to recompute the TILE (band, block, lane) = KL rows x 32 skewed columns;
//   * locate: one thread per tile whose maximum equals the pair's score (ScoreMatrix.call's max-cell
//     list, SmithWaterman.java:176-185; the radix sort of the keys gives its row-major order);
//   * traceback (GetAlignment.call, SmithWaterman.java:354-436): tiles are recomputed into byte tiles
//     in shared memory, one per thread.  G = 1: one thread per max cell (many cells, short walks).
//     G = 32: one warp per max cell (fewer cells than threads): the lanes recompute a CORRIDOR of 32 tiles
//     along the predicted diagonal ahead of the walker, the warp walks through them in lock step (one
//     ballot per diagonal run) until the path leaves the corridor; wrong predictions only cost another
//     round.  CTA-wide (no more cells than SMs, long walks -- cfg3's 100k-column paths): a cluster of CTAs
//     per cell; corridors of 128 tiles are recomputed rounds ahead together with per-tile EXIT TABLES (where
//     does a path that enters the tile here leave it, in how many moves, at what score), so the serial part
//     of a walk is one table look-up per tile; the moves themselves are re-walked in parallel, 32 tile
//     visits at a time.
#include "swb_internal.h"

#include <algorithm>
#include <cstdlib>

namespace swb {

using namespace wide;

namespace {

constexpr int PAD_NEG = -(1 << 29);          // profile score of a row beyond the read's end (gap < 0: stays below every real cell)

// Band-to-band hand-off without fences: every word of a band's bottom row (brow) validates itself.  The host
// fills brow with -1, scores are never negative, so a consumer that reads a value >= 0 has the producer's value
// (relaxed, GPU-scope accesses of single 32-bit words: no ordering between different words is needed).
__device__ __forceinline__ int ld_relaxed(const int32_t *p)
{
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed(int32_t *p, int v) { asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ void st_relaxed4(int32_t *p, int a, int b, int c, int d)
{
    asm volatile("st.relaxed.gpu.global.v4.s32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

__device__ __forceinline__ int ld_acquire(const int32_t *p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int32_t *p, int v) { asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }

struct WCtx {
    const uint8_t *ref;     // codes of this pair's reference (n bytes)
    const uint8_t *read;    // codes of this pair's read in the padded buffer (16-byte aligned, 0xFE beyond m)
    int n, m;
    int match, mismatch, gap;
    int n_blocks;           // blocks per band = ceil((n + 31) / 32)
    int32_t *brow;          // [bands][n_blocks * 32] bottom row of lane 31, indexed by STEP
    int32_t *rec;           // [bands][n_blocks][32 lanes][RW]
    int32_t *tmx;           // [bands][n_blocks][32]
};

template <int KL>
__device__ __forceinline__ WCtx make_ctx(const WideParams &P, int pair)
{
    WCtx C;
    const int ro = P.pair_ref[pair], rd = P.pair_read[pair];
    C.ref = P.ref_codes + P.ref_off[ro];
    C.n = (int)(P.ref_off[ro + 1] - P.ref_off[ro]);
    C.read = P.rpad + P.rpad_off[rd];
    C.m = (int)(P.read_off[rd + 1] - P.read_off[rd]);
    C.match = P.match; C.mismatch = P.mismatch; C.gap = P.gap;
    C.n_blocks = (C.n + WL - 1 + WCB - 1) / WCB;
    C.brow = P.brow + P.brow_off[pair];
    C.rec = P.rec + P.blk_off[pair] * (int64_t)(WL * WGeo<KL>::RW);
    C.tmx = P.tmx + P.blk_off[pair] * (int64_t)WL;
    return C;
}

// the KL read codes of lane-row T (rows T*KL .. T*KL+KL-1) from the padded read buffer
template <int KL>
__device__ __forceinline__ void load_row_codes(const uint8_t *read, int T, int (&rc)[KL])
{
    const uint2 *p = reinterpret_cast<const uint2 *>(read + (int64_t)T * KL);      // KL is a multiple of 8, the buffer 16-aligned
#pragma unroll
    for (int q = 0; q < KL / 8; ++q) {
        const uint2 v = __ldg(p + q);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            rc[8 * q + e] = (int)((v.x >> (8 * e)) & 0xffu);
            rc[8 * q + 4 + e] = (int)((v.y >> (8 * e)) & 0xffu);
        }
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------
// Fill.  NC = 4 / 8 (alphabets of up to NC symbols, gap < 0): substitution scores from a per-warp
// shared-memory profile [code][KL/4][lane][4] (conflict-free LDS.128), NW + s as an IMAD on the FMA
// pipe, two DPX ops per cell.  NC = 0: compare + select, row masks (any alphabet, any gap sign).
template <int KL, int NC>
__global__ void __launch_bounds__(128, KL >= 32 ? 2 : 4)
wide_fill_kernel(const WideParams P, const int2 *items, int n_items, uint32_t *ticket, int one)
{
    using G = WGeo<KL>;
    constexpr bool PROF = NC > 0;
    constexpr int PW = PROF ? NC * KL * WL : 0;                   // profile words per warp
    constexpr int SW = 2 * (WL + 16);                             // staging per warp: 2 x (32 top words + 64 code bytes)
    extern __shared__ __align__(16) int32_t wsm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int32_t *wprof = wsm + warp * (PW + SW);
    int32_t *stage = wprof + PW;
    const int gap = P.gap;

    for (;;) {
        uint32_t it = 0;
        if (lane == 0) it = atomicAdd(ticket, 1u);
        it = __shfl_sync(0xffffffffu, it, 0);
        if (it >= (uint32_t)n_items) break;
        const int pair = items[it].x, band = items[it].y;
        const WCtx C = make_ctx<KL>(P, pair);
        const int T = band * WL + lane;                           // this lane's lane-row
        const int nvalid = min(KL, max(0, C.m - T * KL));         // real rows of this lane
        int rc[KL];
        load_row_codes<KL>(C.read, T, rc);
        __syncwarp();
        if (PROF) {
#pragma unroll
            for (int c = 0; c < (PROF ? NC : 1); ++c)
#pragma unroll
                for (int r = 0; r < KL; ++r)
                    wprof[((c * (KL / 4) + (r >> 2)) * WL + lane) * 4 + (r & 3)] =
                        r < nvalid ? ((rc[r] == c) ? C.match : C.mismatch) : PAD_NEG;
        } else {
#pragma unroll
            for (int r = 0; r < KL; ++r) if (r >= nvalid) rc[r] = 0x100 + r;      // matches nothing
        }
        int H[KL], diag = 0;
#pragma unroll
        for (int r = 0; r < KL; ++r) H[r] = 0;
        int tmax = 0, bmax = 0;
        const int nsteps = C.n + WL - 1;
        const int nchunks = (nsteps + WCB - 1) / WCB;
        int32_t *my_brow = C.brow + (int64_t)band * (C.n_blocks * WCB);
        const int32_t *up_brow = my_brow - (int64_t)C.n_blocks * WCB;
        const bool feeds_below = (int64_t)(band + 1) * G::BH < C.m;       // another band reads this band's bottom row
        int32_t *recp = C.rec + (((int64_t)band * C.n_blocks) * WL + lane) * G::RW;     // record of block 0
        int32_t *tmxp = C.tmx + ((int64_t)band * C.n_blocks) * WL + lane;
        // bottom row of the band above for lane 0: lane L holds column s0 + 1 + L = step s0 + 31 + L up there;
        // requested one chunk ahead (the words validate themselves), re-polled while any is still -1
        auto fetch_top = [&](int s0) -> int {
            return (band > 0 && s0 + 1 + lane <= C.n) ? ld_relaxed(up_brow + s0 + WL - 1 + lane) : 0;
        };
        int tnext = fetch_top(0);

        // reference codes of a chunk: bytes s0-32 .. s0+31 (0-based columns) -> lane L fetches bytes L and L+32
        auto fetch_codes = [&](int s0, int &c_lo, int &c_hi) {
            const int j_lo = s0 - 32 + lane, j_hi = s0 + lane;
            c_lo = (j_lo >= 0 && j_lo < C.n) ? (int)__ldg(C.ref + j_lo) : 0xFF;
            c_hi = (j_hi >= 0 && j_hi < C.n) ? (int)__ldg(C.ref + j_hi) : 0xFF;
        };
        int c_lo, c_hi;
        fetch_codes(0, c_lo, c_hi);

        for (int ch = 0; ch < nchunks; ++ch) {
            const int s0 = ch * WCB;
            int32_t *stg = stage + (ch & 1) * (WL + 16);
            uint8_t *stg_codes = reinterpret_cast<uint8_t *>(stg + WL);
            // ---- top boundary of lane 0
            int tval = tnext;
            if (band > 0) {
                while (__any_sync(0xffffffffu, tval < 0)) {
                    __nanosleep(100);
                    if (tval < 0) tval = ld_relaxed(up_brow + s0 + WL - 1 + lane);
                }
                if (ch + 1 < nchunks) tnext = fetch_top(s0 + WCB);
            }
            stg[lane] = tval;
            stg_codes[lane] = (uint8_t)c_lo;
            stg_codes[lane + 32] = (uint8_t)c_hi;
            __syncwarp();
            if (ch + 1 < nchunks) fetch_codes(s0 + WCB, c_lo, c_hi);             // prefetch: lands during this chunk
            const uint8_t *cb = stg_codes + 32 - lane;            // code of step u: cb[u]  (column s0 + u - lane, 0-based)
            int32_t *seam = recp + G::KW;

            const bool interior = PROF && (s0 >= WL) && (s0 + WCB <= C.n);
            if (interior) {
                // every lane's 32 columns are inside the matrix: no per-step branch, steps overlap
#pragma unroll 2
                for (int q = 0; q < WCB / 4; ++q) {
                    const int4 t4 = *reinterpret_cast<const int4 *>(stg + 4 * q);
                    const int tq[4] = {t4.x, t4.y, t4.z, t4.w};
                    int sm[4], bw[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int u = 4 * q + e;
                        int top = __shfl_up_sync(0xffffffffu, H[KL - 1], 1);
                        if (lane == 0) top = tq[e];
                        const int c = cb[u];
                        const int4 *pp = reinterpret_cast<const int4 *>(wprof) + (c & (NC - 1)) * (KL / 4) * WL + lane;
                        int nw = diag, nn = top;
#pragma unroll
                        for (int g4 = 0; g4 < KL / 4; ++g4) {
                            const int4 v = pp[g4 * WL];
                            const int sv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                            for (int x = 0; x < 4; ++x) {
                                const int r = 4 * g4 + x;
                                const int tt = nw * one + sv[x];                       // NW + s   (IMAD, FMA pipe)
                                const int pre = __viaddmax_s32_relu(H[r], gap, tt);    // max(W + gap, NW + s, 0)
                                nw = H[r];
                                H[r] = __viaddmax_s32(nn, gap, pre);                   // max(N + gap, pre)
                                nn = H[r];
                            }
                        }
#pragma unroll
                        for (int r = 0; r < KL; r += 2) tmax = __vimax3_s32(tmax, H[r], H[r + 1]);
                        diag = top;
                        sm[e] = top; bw[e] = H[KL - 1];
                    }
                    *reinterpret_cast<int4 *>(seam + 4 * q) = make_int4(sm[0], sm[1], sm[2], sm[3]);
                    if (feeds_below && lane == WL - 1) st_relaxed4(my_brow + s0 + 4 * q, bw[0], bw[1], bw[2], bw[3]);
                    // the next chunk's top row was requested at this chunk's start; words the band above had not written
                    // yet are asked for again on the way (the load lands while the chunk computes), so that the poll at
                    // the next chunk's start rarely has to wait for a round trip
                    if ((q & 1) && tnext < 0) tnext = ld_relaxed(up_brow + s0 + WCB + WL - 1 + lane);
                }
            } else {
#pragma unroll 1
                for (int u = 0; u < WCB; ++u) {
                    int top = __shfl_up_sync(0xffffffffu, H[KL - 1], 1);
                    if (lane == 0) top = stg[u];
                    const int c = cb[u];
                    const int j = s0 + u - lane + 1;
                    if (j >= 1 && j <= C.n) {
                        int nw = diag, nn = top;
                        if (PROF) {
                            const int4 *pp = reinterpret_cast<const int4 *>(wprof) + (c & ((PROF ? NC : 1) - 1)) * (KL / 4) * WL + lane;
#pragma unroll
                            for (int g4 = 0; g4 < KL / 4; ++g4) {
                                const int4 v = pp[g4 * WL];
                                const int sv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                                for (int x = 0; x < 4; ++x) {
                                    const int r = 4 * g4 + x;
                                    const int tt = nw * one + sv[x];
                                    const int pre = __viaddmax_s32_relu(H[r], gap, tt);
                                    nw = H[r];
                                    H[r] = __viaddmax_s32(nn, gap, pre);
                                    nn = H[r];
                                }
                            }
#pragma unroll
                            for (int r = 0; r < KL; r += 2) tmax = __vimax3_s32(tmax, H[r], H[r + 1]);
                        } else {
#pragma unroll
                            for (int r = 0; r < KL; ++r) {
                                const int sc = (rc[r] == c) ? C.match : C.mismatch;
                                const int pre = __viaddmax_s32_relu(H[r], gap, nw + sc);
                                nw = H[r];
                                H[r] = __viaddmax_s32(nn, gap, pre);
                                nn = H[r];
                                if (r < nvalid) tmax = max(tmax, H[r]);          // rows beyond the read may exceed the real maximum when gap >= 0
                            }
                        }
                    }
                    diag = top;
                    seam[u] = top;
                    if (feeds_below && lane == WL - 1) st_relaxed(my_brow + s0 + u, H[KL - 1]);
                }
            }
            // ---- block boundary: tile maximum, next block's checkpoint
            tmxp[(int64_t)ch * WL] = tmax;
            bmax = max(bmax, tmax);
            tmax = 0;
            recp += WL * G::RW;
            if (ch + 1 < nchunks) {
#pragma unroll
                for (int q = 0; q < G::KW / 4; ++q) {
                    int v[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int w = 4 * q + e;
                        v[e] = w < KL ? H[w < KL ? w : 0] : (w == KL ? diag : 0);
                    }
                    *reinterpret_cast<int4 *>(recp + 4 * q) = make_int4(v[0], v[1], v[2], v[3]);
                }
            }
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) bmax = max(bmax, __shfl_xor_sync(0xffffffffu, bmax, o));
        if (lane == 0 && bmax > 0)
            atomicMax(P.scores + (int64_t)P.pair_ref[pair] * P.n_reads + P.pair_read[pair], bmax);
    }
}

// copies the wide reads into the padded, 16-byte aligned code buffer (0xFE beyond the read's end)
__global__ void wide_pad_reads_kernel(const uint8_t *codes, const int64_t *read_off, const int32_t *reads, int n_reads,
                                      const int64_t *rpad_off, const int64_t *rpad_len, uint8_t *rpad)
{
    for (int k = blockIdx.y; k < n_reads; k += gridDim.y) {
        const int rd = reads[k];
        const int64_t src = read_off[rd], m = read_off[rd + 1] - src, dst = rpad_off[rd], len = rpad_len[k];
        for (int64_t x = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; x < len; x += (int64_t)gridDim.x * blockDim.x)
            rpad[dst + x] = x < m ? codes[src + x] : (uint8_t)0xFE;
    }
}

// one warp per (pair, band, block): the lanes whose tile maximum equals the pair's score become tasks
__global__ void __launch_bounds__(256) wide_flag_kernel(const WideParams P, int64_t total_blocks, WideTask *tasks,
                                                         uint32_t cap, uint32_t *count)
{
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t idx = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; idx < total_blocks; idx += n_warps) {
        int lo = 0, hi = P.n_pairs;
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (P.blk_off[mid] <= idx) lo = mid; else hi = mid; }
        const int pair = lo;
        const int ro = P.pair_ref[pair];
        const int S = P.scores[(int64_t)ro * P.n_reads + P.pair_read[pair]];
        if (S <= 0) continue;
        const bool hit = P.tmx[idx * WL + lane] == S;
        const uint32_t mask = __ballot_sync(0xffffffffu, hit);
        if (!mask) continue;
        const int64_t rel = idx - P.blk_off[pair];
        const int n = (int)(P.ref_off[ro + 1] - P.ref_off[ro]);
        const int nb = (n + WL - 1 + WCB - 1) / WCB;
        const int band = (int)(rel / nb), blk = (int)(rel - (int64_t)band * nb);
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(count, (uint32_t)__popc(mask));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (hit) {
            const uint32_t k = base + (uint32_t)__popc(mask & ((1u << lane) - 1u));
            if (k < cap) tasks[k] = WideTask{pair, band, blk, (uint32_t)lane};
        }
    }
}

namespace {

// One tile (band, block, lane) recomputed by one thread from its record.
template <int KL>
struct WTile {
    int H[KL], rc[KL];
    int diag, j0;
    const int32_t *rec;

    __device__ __forceinline__ void load(const WCtx &C, int band, int t, int blk)
    {
        using G = WGeo<KL>;
        rec = C.rec + (((int64_t)band * C.n_blocks + blk) * WL + t) * G::RW;
        diag = 0;
#pragma unroll
        for (int r = 0; r < KL; ++r) H[r] = 0;
        if (blk > 0) {
#pragma unroll
            for (int q = 0; q < G::KW / 4; ++q) {
                const int4 a = __ldg(reinterpret_cast<const int4 *>(rec) + q);
                const int v[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int w = 4 * q + e;
                    if (w < KL) H[w < KL ? w : 0] = v[e];
                    else if (w == KL) diag = v[e];
                }
            }
        }
        load_row_codes<KL>(C.read, band * WL + t, rc);
        j0 = blk * WCB - t + 1;                                   // column of step u = j0 + u
    }

    // fn(u, top, H, code) after every step (code = 0xFD outside the matrix); the column is computed when it is
    // inside the matrix.  The seam quad and the reference codes of the next four steps are requested one quad ahead.
    template <class Fn>
    __device__ __forceinline__ void run(const WCtx &C, Fn &&fn)
    {
        const int gap = C.gap, match = C.match, mismatch = C.mismatch;
        const int4 *sq = reinterpret_cast<const int4 *>(rec + WGeo<KL>::KW);
        auto codes4 = [&](int q, int (&cc)[4]) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int j = j0 + 4 * q + e;
                cc[e] = (j >= 1 && j <= C.n) ? (int)__ldg(C.ref + j - 1) : 0xFD;
            }
        };
        int4 a_nxt = __ldg(sq);
        int c_nxt[4];
        codes4(0, c_nxt);
#pragma unroll 1
        for (int q = 0; q < WCB / 4; ++q) {
            const int tq[4] = {a_nxt.x, a_nxt.y, a_nxt.z, a_nxt.w};
            const int cq[4] = {c_nxt[0], c_nxt[1], c_nxt[2], c_nxt[3]};
            if (q + 1 < WCB / 4) { a_nxt = __ldg(sq + q + 1); codes4(q + 1, c_nxt); }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int u = 4 * q + e;
                const int top = tq[e], c = cq[e];
                if (c != 0xFD) {
                    int nw = diag, nn = top;
#pragma unroll
                    for (int r = 0; r < KL; ++r) {
                        const int sc = (rc[r] == c) ? match : mismatch;
                        const int x = __viaddmax_s32_relu(nw, sc, 0);        // max(NW + s, 0)
                        const int pre = __viaddmax_s32(H[r], gap, x);        // max(W + gap, .)
                        nw = H[r];
                        H[r] = __viaddmax_s32(nn, gap, pre);                 // max(N + gap, .)
                        nn = H[r];
                    }
                }
                fn(u, top, H, c);
                diag = top;
            }
        }
    }
};

}  // namespace

// Exit tables.  While a tile is recomputed, every cell also carries WHERE the traceback that passes through it leaves
// the tile, in how many moves, and what score it consumes on the way -- the same three-neighbour dependency as H
// itself, so it rides along in the same pass:
//     packed = exit code | moves << 8 | consumed score << 16
//     exit code: 0..32 = boundary row above the lane (row 0 of the tile) at tile column code; 33..64 = checkpointed
//     column (column 0) at tile row code - 32; 127 = the path ends inside the tile (a cell of score 0)
// The type of a positive cell is the reference's cascade (GetCellScore, SmithWaterman.java:227-249: alignment over
// insertion over deletion on ties; DistributedSW.java:310-326 the other way round).
constexpr int EXIT_END = 127;

template <int KL, class Fn>
__device__ __forceinline__ void run_with_exits(WTile<KL> &W, const WCtx &C, bool tie_gt, uint32_t *tab, Fn &&fn)
{
    static_assert(KL <= WCB, "right-column entries share the second half of the table");
    const int gap = C.gap, match = C.match, mismatch = C.mismatch;
    const int4 *sq = reinterpret_cast<const int4 *>(W.rec + WGeo<KL>::KW);
    uint32_t Pr[KL];
#pragma unroll
    for (int r = 0; r < KL; ++r) Pr[r] = (uint32_t)(WCB + 1 + r);                  // column 0: leaves through (row r + 1, column 0)
    const uint32_t inc_gap = (1u << 8) + ((uint32_t)gap << 16);
    int diag = W.diag;
#pragma unroll 1
    for (int q = 0; q < WCB / 4; ++q) {
        const int4 a = __ldg(sq + q);
        const int tq[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int u = 4 * q + e;
            const int j = W.j0 + u;
            const int c = (j >= 1 && j <= C.n) ? (int)__ldg(C.ref + j - 1) : 0xFD;
            const int top = tq[e];
            if (c != 0xFD) {
                int nw = diag, nn = top;
                uint32_t pnw = (uint32_t)u, pn = (uint32_t)(u + 1);               // boundary row: (0, c - 1) and (0, c)
#pragma unroll
                for (int r = 0; r < KL; ++r) {
                    const int sc = (W.rc[r] == c) ? match : mismatch;
                    const int dv = nw + sc, wv = W.H[r] + gap, nv = nn + gap;
                    const int hn = max(max(dv, 0), max(wv, nv));
                    const uint32_t pa = pnw + (1u << 8) + ((uint32_t)sc << 16), pi2 = pn + inc_gap, pd = Pr[r] + inc_gap;
                    uint32_t sel = tie_gt ? (wv == hn ? pd : (nv == hn ? pi2 : pa)) : (dv == hn ? pa : (nv == hn ? pi2 : pd));
                    if (hn <= 0) sel = EXIT_END;
                    pnw = Pr[r]; Pr[r] = sel; pn = sel;
                    nw = W.H[r]; W.H[r] = hn; nn = hn;
                }
            } else {
#pragma unroll
                for (int r = 0; r < KL; ++r) Pr[r] = EXIT_END;
            }
            tab[u] = Pr[KL - 1];
            fn(u, top, W.H, c);
            diag = top;
        }
    }
#pragma unroll
    for (int r = 0; r < KL; ++r) tab[WCB + r] = Pr[r];
}

// one thread per flagged tile: every cell of the tile that equals the pair's score becomes a key
template <int KL>
__global__ void __launch_bounds__(128) wide_locate_kernel(const WideParams P, const WideTask *tasks,
                                                           const uint32_t *n_tasks_ptr, uint32_t cap_tasks,
                                                           uint64_t *keys, uint32_t cap, uint32_t *count)
{
    const uint32_t n_tasks = min(*n_tasks_ptr, cap_tasks);
    const uint32_t n_threads = gridDim.x * blockDim.x;
    for (uint32_t task = blockIdx.x * blockDim.x + threadIdx.x; task < n_tasks; task += n_threads) {
        const WideTask T = tasks[task];
        const WCtx C = make_ctx<KL>(P, T.pair);
        const int t = (int)T.lane;
        const int S = P.scores[(int64_t)P.pair_ref[T.pair] * P.n_reads + P.pair_read[T.pair]];
        const int row0 = (T.band * WL + t) * KL;                  // 0-based first row of the tile
        const int nvalid = min(KL, max(0, C.m - row0));
        WTile<KL> W;
        W.load(C, T.band, t, T.block);
        W.run(C, [&](int u, int, const int (&Hc)[KL], int c) {
            if (c == 0xFD) return;
            uint32_t rm = 0;
#pragma unroll
            for (int r = 0; r < KL; ++r) rm |= (Hc[r] == S) ? (1u << r) : 0u;
            if (nvalid < 32) rm &= (1u << nvalid) - 1u;
            while (rm) {
                const int r = __ffs((int)rm) - 1;
                rm &= rm - 1;
                const uint32_t k = atomicAdd(count, 1u);
                if (k < cap) keys[k] = wide_key((uint64_t)T.pair, (uint32_t)(row0 + r + 1), (uint32_t)(W.j0 + u));
            }
        });
    }
}

// ---------------------------------------------------------------------------------------
// Traceback.  Every thread owns one tile slot in shared memory (stride TW words, odd: the lanes' slots start in
// different banks, so the lock-step column stores of a warp are conflict-free):
//   elements [cc][rr], cc = 0 .. 32 (0 = the checkpointed column), rr = 0 .. KL (0 = the boundary row above the
//   lane), then the lane-row's KL read codes and the reference codes of the tile's 32 steps.
// A step up / left / diagonal in the matrix is a constant pointer decrement inside the slot.
// BYTE: only the low 8 bits of every score are kept.  That is enough because the walker carries the exact score
// of its cell (the pair maximum minus the moves so far) and a candidate never lies 250 or more below H
// (tile_trace_ok): equality of the low bytes is equality.  Other score sets use int32 tiles.
// The walker checks up to four diagonal moves per iteration ('>=' rule: an alignment move wins whenever
// NW + s == H): all their loads are independent, so a run of matches costs one shared-memory latency per four
// columns instead of one per column.
template <int KL, bool BYTE> struct TraceGeo {
    static constexpr int ES = BYTE ? 1 : 4;                         // bytes per element
    static constexpr int ROWW = BYTE ? (KL + 1 + 3) / 4 : KL + 1;   // words per tile column
    static constexpr int COLB = ROWW * 4;                           // bytes per tile column
    static constexpr int CODE0 = ROWW * (WCB + 1);                  // first code word
    static constexpr int TW = (CODE0 + KL / 4 + WCB / 4) | 1;       // slot stride in words (odd)
    static constexpr int GUARD = 4 * (COLB + ES) / 4 + 4;           // words before slot 0: the diagonal look-ahead may reach below a slot
    static size_t smem_bytes(int nt) { return ((size_t)nt + GUARD + (size_t)nt * TW) * 4; }
};
// CTA-wide mode (few max cells, long walks): see the pipelined block in wide_trace_kernel.
constexpr int CTAW_TILES = 128, CTAW_THREADS = 256;
constexpr int SUB_STAGE = (15 + 32 * 2 * WCB) / 16 + 4;                             // staging words for one batch of chained tile visits (32 visits of <= 64 moves)
constexpr int NXT_STRIDE = 66;                                                     // next-entry table: 65 exit codes per tile (uint16), padded
constexpr int SUB_SMEM_WORDS = CTAW_TILES * 64 + CTAW_TILES * NXT_STRIDE / 2 + SUB_STAGE;   // exit tables [tile][64], next-entry tables, op staging


template <int KL, int NT, int G, bool BYTE>
__global__ void __launch_bounds__(NT) wide_trace_kernel(const WideParams P, const uint64_t *keys, uint32_t n_cells,
                                                         int32_t *beginnings, int32_t *op_lens, uint32_t *ops,
                                                         int64_t ops_stride)
{
    using TG = TraceGeo<KL, BYTE>;
    constexpr int ES = TG::ES, ROWW = TG::ROWW, COLB = TG::COLB, TW = TG::TW;
    constexpr int DG = COLB + ES;                                   // one diagonal step, in bytes
    constexpr bool CTAW = G > 32;                                  // the whole CTA works on one max cell
    constexpr int TILES = CTAW ? CTAW_TILES : G;                   // tiles of a corridor
    constexpr int DB = CTAW ? 4 : (G > 1 ? 2 : 1);                 // blocks per lane-row of the corridor
    constexpr int HS = TILES / DB;                                 // lane-rows a corridor covers
    constexpr int NSLOT = CTAW ? TILES : NT;                       // tile slots of the CTA
    constexpr int TPW = 32;                                        // tiles per warp: the recompute is issue-bound, not latency-bound
                                                                   // (8 busy lanes in each of 16 warps: 2.3x slower than 32 in 4)
    static_assert(G == 1 || G == 32 || G == NT, "a group is a thread, a warp or the whole CTA");
    static_assert(HS <= 32, "one lane of the first warp per lane-row");
    extern __shared__ uint32_t tsm[];
    __shared__ int bc_state[3];                                    // CTA-wide groups: the walker's state for the next round
    int32_t *slot_blk = reinterpret_cast<int32_t *>(tsm);           // [NSLOT] block of the tile in each slot
    uint32_t *slots = tsm + NSLOT + TG::GUARD;
    const int gl = threadIdx.x % G;                                // lane in group
    const int leader = CTAW ? 0 : threadIdx.x - gl;
    // tile of the corridor this thread recomputes (-1: none), which is also its slot
    const int tg = !CTAW ? gl : (((threadIdx.x & 31) < TPW && (int)(threadIdx.x >> 5) * TPW + (int)(threadIdx.x & 31) < TILES)
                                     ? (int)(threadIdx.x >> 5) * TPW + (int)(threadIdx.x & 31) : -1);
    const int myslot = CTAW ? max(tg, 0) : (int)threadIdx.x;
    uint32_t *mytile = slots + (size_t)myslot * TW;
    int32_t *subrec = reinterpret_cast<int32_t *>(slots + (size_t)NSLOT * TW);   // CTA-wide: exit tables [TILES][64], then stage[SUB_STAGE]
    const unsigned gmask = 0xffffffffu;
    const uint32_t n_groups = gridDim.x * (NT / G);
    const uint32_t gid = (blockIdx.x * NT + threadIdx.x) / G;
    const int gap = P.gap, match = P.match, mismatch = P.mismatch;
    const bool tie_gt = P.tie_gt != 0;
    constexpr int M = BYTE ? 0xff : -1;

    auto store_col = [&](int cc, int top, const int (&Hc)[KL]) {
        uint32_t *col = mytile + cc * ROWW;
        if (BYTE) {
#pragma unroll
            for (int w = 0; w < ROWW; ++w) {
                uint32_t v[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int k = 4 * w + e;                       // element k: 0 = boundary row, 1..KL = the lane's rows
                    v[e] = k == 0 ? (uint32_t)top : (k <= KL ? (uint32_t)Hc[(k >= 1 && k <= KL) ? k - 1 : 0] : 0u);
                }
                col[w] = __byte_perm(__byte_perm(v[0], v[1], 0x0040), __byte_perm(v[2], v[3], 0x0040), 0x5410);
            }
        } else {
            col[0] = (uint32_t)top;
#pragma unroll
            for (int r = 0; r < KL; ++r) col[r + 1] = (uint32_t)Hc[r];
        }
    };
    auto elem = [&](const uint8_t *p) -> int {
        return BYTE ? (int)*p : *reinterpret_cast<const int32_t *>(p);
    };


    if constexpr (CTAW) {
        // ================================================================================================
        // CTA-wide mode, PIPELINED over the CTAs of a cluster.  A long path is cut into ROUNDS of HS lane-rows
        // (fixed rows: round r covers lane-rows T00 - HS r .. T00 - HS r - HS + 1).  CTA q of the cell's cluster owns the
        // rounds q, q + C, q + 2C, ...  For each of them it PREPARES -- recomputes the corridor of tiles along the
        // diagonal predicted from the latest published walker state and runs the speculative sub-walks -- while the
        // walker is still rounds away, then waits for the round's TOKEN (the walker state at the round's first row,
        // in global memory, release / acquire), CONSUMES (chains the sub-walk records, exact walker for what they
        // miss, corrective corridors if the path left the predicted one) and publishes the next token.  Only the
        // chain and the exact walker are serial along a path; the expensive recompute runs C rounds ahead.
        // The CTAs of a cluster are co-scheduled, so a waiting CTA's producer is always running.
        const int Cc = P.pipe_c;
        const uint32_t cell = blockIdx.x / (uint32_t)Cc;
        const int q = (int)(blockIdx.x % (uint32_t)Cc);
        if (cell >= n_cells) return;
        const uint64_t key = keys[cell];
        const int pair = (int)wide_key_pair(key);
        const int ci0 = (int)wide_key_i(key), cj0 = (int)wide_key_j(key);
        const WCtx C = make_ctx<KL>(P, pair);
        const int h0 = P.scores[(int64_t)P.pair_ref[pair] * P.n_reads + P.pair_read[pair]];
        int32_t *tok = P.mail + (int64_t)cell * P.mail_stride * 8;      // token k = walker state at the first row of round k
        int32_t *latest = P.mail_latest + cell;                        // highest token index published so far
        uint32_t *myops = ops + (int64_t)cell * ops_stride;
        const int T00 = (ci0 - 1) / KL;
        // corridor shape: 32 lane-rows x 4 blocks along the predicted diagonal, or 16 x 8 for a path of low score density
        // (many gaps: it wanders off a diagonal -- the random pair of cfg3 left a 4-block corridor 1.4 times per round)
        const bool wide_shape = (long long)h0 * 2 < (long long)max(match, 1) * (long long)min(ci0, cj0);
        const int DBr = wide_shape ? 8 : 4, HSr = TILES / DBr;
        const int wl = (int)threadIdx.x;                                // lane of the walking warp (threads 0..31)
        const int big = max(abs(match), abs(mismatch));
        const int bigp = max(max(match, mismatch), 1);
        uint32_t *tabs = reinterpret_cast<uint32_t *>(subrec);           // [TILES][64] exit tables
        uint16_t *nxt = reinterpret_cast<uint16_t *>(tabs + TILES * 64); // [TILES][NXT_STRIDE]: exit code -> slot * 64 + entry of the next tile
        uint32_t *stage = tabs + TILES * 64 + TILES * NXT_STRIDE / 2;
        __shared__ int bc[8];
        int hcur = h0, ci = ci0, cj = cj0, beginning = 0;
        int64_t oplen = 0;
        uint32_t opword = 0;
        int T0 = 0;                                                    // the prepared corridor: lane-rows T0, T0 - 1, .., T0 - HS + 1

        // corridor of tiles along the diagonal through (qi, qj): byte tiles + exit tables
        auto prepare = [&](int qi, int qj, int Tlo) {
            T0 = (qi - 1) / KL;
            int myblk = -1;
            if (tg >= 0) {
                const int k = tg / DBr, d = tg % DBr;
                const int Tk = T0 - k;
                if (Tk >= 0) {
                    const int t = Tk % WL;
                    const int di = k == 0 ? 0 : qi - (Tk * KL + KL);   // rows the path climbs to reach lane-row Tk
                    const int step = qj - di - 1 + t;
                    const int b = (step >= 0 ? step / WCB : -1) + DBr / 2 - 1 - d;   // blocks b_k + 1 .. b_k - 2 (b_k + 3 .. b_k - 4)
                    if (b >= 0 && b < C.n_blocks) myblk = b;
                }
                if (myblk >= 0) {
                    WTile<KL> W;
                    W.load(C, Tk / WL, Tk % WL, myblk);
                    store_col(0, W.diag, W.H);
                    uint32_t *cw = mytile + TG::CODE0;
#pragma unroll
                    for (int q4 = 0; q4 < KL / 4; ++q4)
                        cw[q4] = (uint32_t)W.rc[4 * q4] | ((uint32_t)W.rc[4 * q4 + 1] << 8) | ((uint32_t)W.rc[4 * q4 + 2] << 16) | ((uint32_t)W.rc[4 * q4 + 3] << 24);
                    uint32_t cacc = 0;
                    run_with_exits<KL>(W, C, tie_gt, tabs + tg * 64, [&](int u, int top, const int (&Hc)[KL], int c) {
                        store_col(u + 1, top, Hc);
                        cacc |= (uint32_t)c << (8 * (u & 3));
                        if ((u & 3) == 3) { cw[KL / 4 + (u >> 2)] = cacc; cacc = 0; }
                    });
                }
                slot_blk[tg] = myblk;
            }
            __syncthreads();
            // next-entry table of my tile: the cell a path leaves the tile through is an entry cell (bottom row or right
            // column) of a neighbouring tile -- which slot, which entry -- or of none (outside the corridor / the round)
            if (tg >= 0 && myblk >= 0) {
                const int kk = tg / DBr, Tk = T0 - kk, t = Tk % WL;
                // the only tiles a path can step into from this one: the lane-row above (blocks b - 1, b, b + 1: its skew
                // differs by one step, or by 31 across a band boundary) and block b - 1 of this lane-row
                auto find = [&](int kk2, int b2) -> int {
                    if (kk2 < 0 || kk2 >= HSr || T0 - kk2 < Tlo || T0 - kk2 < 0 || b2 < 0) return -1;
                    int sl = -1;
                    for (int dd = 0; dd < DBr; ++dd) if (slot_blk[DBr * kk2 + dd] == b2) sl = DBr * kk2 + dd;
                    return sl;
                };
                const int sUm = find(kk + 1, myblk - 1), sU0 = find(kk + 1, myblk), sUp = find(kk + 1, myblk + 1), sL = find(kk, myblk - 1);
                const int t2 = (Tk - 1 + WL) % WL;                                   // skew of the lane-row above
                for (int code = 0; code <= 2 * WCB; ++code) {
                    int nx = 0xFFFF;
                    if (code <= WCB) {                                              // leaves through the boundary row, tile column `code`
                        const int xj = myblk * WCB + code - t;
                        if (Tk >= 1 && xj >= 1) {
                            const int step2 = xj - 1 + t2, b2 = step2 / WCB;
                            const int sl = b2 == myblk ? sU0 : (b2 == myblk - 1 ? sUm : (b2 == myblk + 1 ? sUp : -1));
                            if (sl >= 0) nx = sl * 64 + (step2 - b2 * WCB);         // bottom row of the tile above, column c2 = step2 - b2 * WCB + 1
                        }
                    } else if (sL >= 0 && myblk * WCB - t >= 1) {
                        nx = sL * 64 + WCB + (code - WCB) - 1;                      // right column of the tile to the left, row code - WCB
                    }
                    nxt[tg * NXT_STRIDE + code] = (uint16_t)nx;
                }
            }
            __syncthreads();
        };

        // the walking warp (threads 0..31, every lane keeps the whole state); never above lane-row Tlo.
        //  (a) CHAIN: while the walker stands on an entry edge of a tile (bottom row or right column), the tile's exit
        //      table says where the path leaves it, in how many moves and what score that consumes -- one look-up per
        //      tile; up to 32 tile visits per batch, then lane v re-walks visit v inside its byte tile to get the moves
        //      themselves (n is known, so no score is carried) and prefix sums place them in the op stream;
        //  (b) the exact walker for one tile visit when (a) cannot move: an interior start cell, the last tiles of a
        //      path (the exact score decides where it stops).
        auto consume = [&](int Tlo) {
            auto push = [&](uint32_t op, int n) {
                const uint32_t pattern = op * 0x55555555u;
                while (n > 0) {
                    const int used = (int)(oplen & 15);
                    const int take = min(n, 16 - used);
                    const uint32_t bits = take == 16 ? pattern : (pattern & ((1u << (2 * take)) - 1u));
                    opword |= bits << (2 * used);
                    oplen += take; n -= take;
                    if ((oplen & 15) == 0) { if (wl == 0) myops[(oplen >> 4) - 1] = opword; opword = 0; }
                }
            };
            for (;;) {
                // ---- (a) chain
                int nv = 0, hc = hcur, xi = ci, xj = cj;
                int my_slot = 0, my_r = 0, my_c = 0, my_n = 0;
                if (hc > 0 && xi >= 1 && xj >= 1) {
                    // the tile and entry the walker stands on (found the slow way once per batch) ...
                    const int T = (xi - 1) / KL;
                    const int kk = T0 - T;
                    int cur = -1;
                    if (T >= Tlo && kk >= 0 && kk < HSr) {
                        const int step = xj - 1 + T % WL;
                        const int b = step / WCB;
                        int slot = DBr * kk, dd = 0;
                        while (dd < DBr && slot_blk[slot + dd] != b) ++dd;
                        const int r = xi - T * KL, c = step - b * WCB + 1;            // 1..KL, 1..WCB
                        if (dd < DBr && (r == KL || c == WCB)) cur = (slot + dd) * 64 + (r == KL ? c - 1 : WCB + r - 1);
                    }
                    // ... then two look-ups per tile visit: the exit table of the entry, the next-entry table of the exit
                    int last_cur = -1, last_code = 0;
                    while (nv < 32 && cur >= 0) {
                        const uint32_t pk = tabs[cur];
                        const int code = (int)(pk & 127u), n = (int)((pk >> 8) & 127u), ds = (int)pk >> 16;
                        if (code == EXIT_END || n == 0 || hc <= n * bigp) break;  // the path may end inside: (b)
                        if (wl == nv) { my_slot = cur >> 6; const int e = cur & 63; my_r = e < WCB ? KL : e - WCB + 1; my_c = e < WCB ? e + 1 : WCB; my_n = n; }
                        hc -= ds;
                        last_cur = cur; last_code = code;
                        ++nv;
                        const int nx = (int)nxt[(cur >> 6) * NXT_STRIDE + code];
                        cur = nx == 0xFFFF ? -1 : nx;
                    }
                    if (nv > 0) {
                        const int slot = last_cur >> 6;
                        const int T2 = T0 - slot / DBr, t2 = T2 % WL, b2 = slot_blk[slot];
                        if (last_code <= WCB) { xi = T2 * KL; xj = b2 * WCB + last_code - t2; }
                        else { xi = T2 * KL + (last_code - WCB); xj = b2 * WCB - t2; }
                    }
                }
                if (nv > 0) {
                    // lane v: the moves of visit v (walk order), 2 bits each
                    unsigned long long lo = 0, hi = 0;
                    if (wl < nv) {
                        const uint8_t *base = reinterpret_cast<const uint8_t *>(slots + (size_t)my_slot * TW);
                        const uint8_t *p = base + my_c * COLB + my_r * ES;
                        const uint8_t *pr = base + TG::CODE0 * 4 + (my_r - 1);
                        const uint8_t *pq = base + TG::CODE0 * 4 + KL + (my_c - 1);
                        for (int k = 0; k < my_n; ++k) {
                            const int e0 = elem(p), e1 = elem(p - DG), hn = elem(p - ES), hw = elem(p - COLB);
                            const int s0 = (pr[0] == pq[0]) ? match : mismatch;
                            const bool eq_a = ((e1 + s0 - e0) & M) == 0, eq_i = ((hn + gap - e0) & M) == 0, eq_d = ((hw + gap - e0) & M) == 0;
                            const uint32_t op = tie_gt ? (eq_d ? 3u : (eq_i ? 2u : 1u)) : (eq_a ? 1u : (eq_i ? 2u : 3u));
                            const int up = op != 3u, left = op != 2u;
                            pr -= up; pq -= left;
                            p -= up * ES + left * COLB;
                            if (k < 32) lo |= (unsigned long long)op << (2 * k); else hi |= (unsigned long long)op << (2 * k - 64);
                        }
                    }
                    const int n = wl < nv ? my_n : 0;
                    int pn = n;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int a = __shfl_up_sync(0xffffffffu, pn, o);
                        if (wl >= o) pn += a;
                    }
                    const int used0 = (int)(oplen & 15);
                    const int total = __shfl_sync(0xffffffffu, pn, nv - 1);
                    const int nwords = (used0 + total + 15) >> 4;
                    for (int w = wl; w <= nwords; w += 32) stage[w] = (w == 0) ? opword : 0u;
                    __syncwarp();
                    if (wl < nv) {
                        const int pos = used0 + (pn - n);
                        const int word0 = pos >> 4, sh = 2 * (pos & 15);
                        const uint32_t w4[4] = {(uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32)};
#pragma unroll
                        for (int q4 = 0; q4 < 4; ++q4)
                            if (n > 16 * q4) {
                                const unsigned long long v = (unsigned long long)w4[q4] << sh;
                                atomicOr(&stage[word0 + q4], (uint32_t)v);
                                if ((uint32_t)(v >> 32)) atomicOr(&stage[word0 + q4 + 1], (uint32_t)(v >> 32));
                            }
                    }
                    __syncwarp();
                    const int64_t oplen_new = oplen + total;
                    const int full_words = (int)((oplen_new >> 4) - (oplen >> 4));
                    for (int w = wl; w < full_words; w += 32) myops[(oplen >> 4) + w] = stage[w];
                    opword = stage[full_words];
                    __syncwarp();
                    oplen = oplen_new;
                    hcur = hc; ci = xi; cj = xj;
                    continue;
                }
                // ---- (b) exact walker (SmithWaterman.java:380-409), one tile visit, all 32 lanes in lock step: lane k probes
                // the diagonal cell (r - k, c - k), one ballot finds a whole run of alignment moves
                if (!(hcur > 0 && ci >= 1 && cj >= 1)) return;
                const int T = (ci - 1) / KL;
                const int kk = T0 - T;
                if (T < Tlo || kk < 0 || kk >= HSr) return;
                const int t = T % WL;
                const int step = cj - 1 + t;
                const int b = step / WCB;
                int slot = DBr * kk, dd = 0;
                while (dd < DBr && slot_blk[slot + dd] != b) ++dd;
                if (dd == DBr) return;
                slot += dd;
                int r = ci - T * KL;                           // 1..KL
                int c = step - b * WCB + 1;                    // 1..WCB
                const uint8_t *base = reinterpret_cast<const uint8_t *>(slots + (size_t)slot * TW);
                const uint8_t *p = base + c * COLB + r * ES;
                const uint8_t *pr = base + TG::CODE0 * 4 + (r - 1);
                const uint8_t *pq = base + TG::CODE0 * 4 + KL + (c - 1);
                for (;;) {
                    const int lim = min(r, c);
                    const bool inside = wl < lim;
                    const uint8_t *pk = p - wl * DG;
                    const int hk = inside ? elem(pk) : 0, hnwk = inside ? elem(pk - DG) : 1;
                    const bool is_m = inside && pr[-wl] == pq[-wl];
                    const int sck = is_m ? match : mismatch;
                    const bool okk = inside && (((hnwk + sck - hk) & M) == 0);
                    const unsigned okm = __ballot_sync(0xffffffffu, okk), mm = __ballot_sync(0xffffffffu, is_m);
                    const int run = tie_gt ? 0 : (okm == 0xffffffffu ? 32 : __ffs((int)~okm) - 1);
                    const int L = (hcur > 32 * big) ? run : min(run, 1);
                    if (L > 0) {
                        const unsigned lm = L >= 32 ? 0xffffffffu : ((1u << L) - 1u);
                        const int nm = __popc(mm & lm);
                        hcur -= nm * match + (L - nm) * mismatch;
                        beginning = cj - (L - 1);
                        ci -= L; cj -= L; r -= L; c -= L;
                        p -= L * DG; pr -= L; pq -= L;
                        push(1u, L);
                    }
                    if (hcur <= 0 || r == 0 || c == 0) break;
                    if (L == run && run < lim) {
                        const int hn = elem(p - ES), hw = elem(p - COLB);
                        const bool eq_i = ((hn + gap - hcur) & M) == 0, eq_d = ((hw + gap - hcur) & M) == 0;
                        const int s0 = (pr[0] == pq[0]) ? match : mismatch;
                        const uint32_t op = tie_gt ? (eq_d ? 3u : (eq_i ? 2u : 1u)) : (eq_i ? 2u : 3u);
                        beginning = cj;
                        hcur -= (op == 1u) ? s0 : gap;
                        const int up = op != 3u, left = op != 2u;
                        r -= up; ci -= up; pr -= up;
                        c -= left; cj -= left; pq -= left;
                        p -= up * ES + left * COLB;
                        push(op, 1);
                        if (hcur <= 0 || r == 0 || c == 0) break;
                    }
                }
                if (hcur <= 0) return;
            }
        };

        for (int r = q;; r += Cc) {
            const int Tr_hi = T00 - HSr * r;
            if (Tr_hi < 0 || h0 <= 0) break;
            const int Tr_lo = max(Tr_hi - HSr + 1, 0);
            // ---- 1. where will the path enter this round?  The diagonal through the latest published state.
            if (threadIdx.x == 0) {
                int lt = r == 0 ? 0 : min(ld_acquire(latest), r);
                int tci = ci0, tcj = cj0, tdone = 0;
                if (lt >= 1) { tci = ld_relaxed(tok + lt * 8 + 2); tcj = ld_relaxed(tok + lt * 8 + 3); tdone = ld_relaxed(tok + lt * 8 + 7); }
                bc[0] = tci; bc[1] = tcj; bc[2] = tdone;
            }
            __syncthreads();
            const int tci = bc[0], tcj = bc[1];
            const bool tdone = bc[2] != 0;
            __syncthreads();
            if (tdone) break;
            const int row_r = r == 0 ? ci0 : (Tr_hi + 1) * KL;
            prepare(row_r, tcj - (tci - row_r), Tr_lo);
            // ---- 2. the round's token
            if (r > 0) {
                if (threadIdx.x == 0) {
                    int done = 0;
                    for (;;) {
                        if (ld_acquire(tok + r * 8) == r + 1) break;
                        const int lt = ld_acquire(latest);
                        if (lt >= 1 && lt < r && ld_relaxed(tok + lt * 8 + 7)) { done = 1; break; }       // the path ended in an earlier round
                        __nanosleep(200);
                    }
                    bc[7] = done;
                    if (!done) for (int k = 1; k < 7; ++k) bc[k] = ld_relaxed(tok + r * 8 + k);
                    if (!done && ld_relaxed(tok + r * 8 + 7)) bc[7] = 1;
                }
                __syncthreads();
                const bool done = bc[7] != 0;
                hcur = bc[1]; ci = bc[2]; cj = bc[3]; oplen = bc[4]; opword = (uint32_t)bc[5]; beginning = bc[6];
                __syncthreads();
                if (done) break;
            }
            // ---- 3. walk the round's lane-rows
            bool first = true;
            for (;;) {
                if (!first) prepare(ci, cj, Tr_lo);                    // the path left the prepared corridor: one around the true cell
                const int ci_before = ci, cj_before = cj;
                if (threadIdx.x < 32) {
                    consume(Tr_lo);
                    if (wl == 0) { bc[0] = hcur; bc[1] = ci; bc[2] = cj; }
                }
                __syncthreads();
                hcur = bc[0]; ci = bc[1]; cj = bc[2];
                __syncthreads();
                if (!first && ci == ci_before && cj == cj_before) hcur = 0;   // cannot happen (a corridor around the true cell holds it); never spin
                first = false;
                if (hcur <= 0 || ci < 1 || cj < 1 || (ci - 1) / KL < Tr_lo) break;
            }
            // ---- 4. publish the next token
            const bool done = hcur <= 0 || ci < 1 || cj < 1;
            if (threadIdx.x == 0) {
                int32_t *tk = tok + (r + 1) * 8;
                tk[1] = hcur; tk[2] = ci; tk[3] = cj; tk[4] = (int)oplen; tk[5] = (int)opword; tk[6] = beginning; tk[7] = done ? 1 : 0;
                __threadfence();
                st_release(tk, r + 2);
                __threadfence();
                atomicMax(latest, r + 1);
                if (done) {
                    if (oplen & 15) myops[oplen >> 4] = opword;
                    beginnings[cell] = beginning;
                    op_lens[cell] = (int32_t)oplen;
                }
            }
            if (done) break;
        }
        return;
    }

    if constexpr (!CTAW)
    for (uint32_t cell = gid; cell < n_cells; cell += n_groups) {            // group-uniform
        const uint64_t key = keys[cell];
        const int pair = (int)wide_key_pair(key);
        int ci = (int)wide_key_i(key), cj = (int)wide_key_j(key);
        const WCtx C = make_ctx<KL>(P, pair);
        int hcur = P.scores[(int64_t)P.pair_ref[pair] * P.n_reads + P.pair_read[pair]];
        int beginning = 0;
        int64_t oplen = 0;
        uint32_t opword = 0;
        uint32_t *myops = ops + (int64_t)cell * ops_stride;
        while (hcur > 0) {                                         // group-uniform: the state is broadcast below
            // ---- corridor: slot (k, d) = lane-row T0 - k, block b_k - d, b_k from the diagonal through (ci, cj)
            // (DB = 2: blocks b_k, b_k - 1; DB = 4: b_k + 1 .. b_k - 2 -- a path with many gaps drifts off the diagonal)
            const int T0 = (ci - 1) / KL;
            const int k = tg / DB, d = tg % DB;
            const int Tk = T0 - k;
            int myblk = -1;
            if (tg >= 0 && Tk >= 0) {
                const int t = Tk % WL;
                const int di = k == 0 ? 0 : ci - (Tk * KL + KL);   // rows the path climbs to reach lane-row Tk
                const int step = cj - di - 1 + t;
                const int b = (step >= 0 ? step / WCB : -1) + (DB == 4 ? 1 : 0) - d;
                if (b >= 0 && b < C.n_blocks) myblk = b;
            }
            if (myblk >= 0) {
                WTile<KL> W;
                W.load(C, Tk / WL, Tk % WL, myblk);
                store_col(0, W.diag, W.H);
                uint32_t *cw = mytile + TG::CODE0;
#pragma unroll
                for (int q = 0; q < KL / 4; ++q)
                    cw[q] = (uint32_t)W.rc[4 * q] | ((uint32_t)W.rc[4 * q + 1] << 8) | ((uint32_t)W.rc[4 * q + 2] << 16) | ((uint32_t)W.rc[4 * q + 3] << 24);
                uint32_t cacc = 0;
                W.run(C, [&](int u, int top, const int (&Hc)[KL], int c) {
                    store_col(u + 1, top, Hc);
                    cacc |= (uint32_t)c << (8 * (u & 3));
                    if ((u & 3) == 3) { cw[KL / 4 + (u >> 2)] = cacc; cacc = 0; }
                });
            }
            if (tg >= 0) slot_blk[myslot] = myblk;
            if (G == 32) __syncwarp(gmask);
            else if (G > 32) __syncthreads();
            if (G == 1) {
                // ---- walk (SmithWaterman.java:380-409): one thread per max cell
                for (;;) {
                    const int T = (ci - 1) / KL;
                    const int kk = T0 - T;
                    if (kk >= HS) break;
                    const int t = T % WL;
                    const int step = cj - 1 + t;
                    const int b = step / WCB;
                    int slot = leader + DB * kk;
                    if (slot_blk[slot] != b) {
                        int dd = 1;
                        while (dd < DB && slot_blk[slot + dd] != b) ++dd;
                        if (dd == DB) break;
                        slot += dd;
                    }
                    int r = ci - T * KL;                           // 1..KL
                    int c = step - b * WCB + 1;                    // 1..WCB
                    const uint8_t *base = reinterpret_cast<const uint8_t *>(slots + (size_t)slot * TW);
                    const uint8_t *p = base + c * COLB + r * ES;   // element (r, c)
                    const uint8_t *pr = base + TG::CODE0 * 4 + (r - 1);          // read code of row r
                    const uint8_t *pq = base + TG::CODE0 * 4 + KL + (c - 1);     // reference code of column c
                    for (;;) {
                        // everything a diagonal run of four and a single gap move can need; the loads are independent
                        const int h1 = elem(p - DG), h2 = elem(p - 2 * DG), h3 = elem(p - 3 * DG), h4 = elem(p - 4 * DG);
                        const int hn = elem(p - ES), hw = elem(p - COLB);
                        const int s0 = (pr[0] == pq[0]) ? match : mismatch, s1 = (pr[-1] == pq[-1]) ? match : mismatch;
                        const int s2 = (pr[-2] == pq[-2]) ? match : mismatch, s3 = (pr[-3] == pq[-3]) ? match : mismatch;
                        const int lim = min(r, c);                 // cells (r - k, c - k), k < lim, lie inside this tile
                        const int hc1 = hcur - s0, hc2 = hc1 - s1, hc3 = hc2 - s2, hc4 = hc3 - s3;
                        const bool eq_a = ((h1 + s0 - hcur) & M) == 0;
                        int L = 0;
                        if (!tie_gt && eq_a) {
                            const bool ok1 = lim > 1 && hc1 > 0 && ((h2 + s1 - hc1) & M) == 0;
                            const bool ok2 = ok1 && lim > 2 && hc2 > 0 && ((h3 + s2 - hc2) & M) == 0;
                            const bool ok3 = ok2 && lim > 3 && hc3 > 0 && ((h4 + s3 - hc3) & M) == 0;
                            L = 1 + (int)ok1 + (int)ok2 + (int)ok3;
                        }
                        const uint32_t sh = 2u * ((uint32_t)oplen & 15u);
                        if (L > 0) {
                            hcur = L == 1 ? hc1 : (L == 2 ? hc2 : (L == 3 ? hc3 : hc4));
                            beginning = cj - (L - 1);
                            ci -= L; cj -= L; r -= L; c -= L;
                            p -= L * DG; pr -= L; pq -= L;
                            const unsigned long long acc = (unsigned long long)opword | ((unsigned long long)(0x55u >> (8 - 2 * L)) << sh);
                            oplen += L;
                            if (sh + 2u * (uint32_t)L >= 32u) { myops[(oplen >> 4) - 1] = (uint32_t)acc; opword = (uint32_t)(acc >> 32); }
                            else opword = (uint32_t)acc;
                        } else {
                            const bool eq_i = ((hn + gap - hcur) & M) == 0, eq_d = ((hw + gap - hcur) & M) == 0;
                            const uint32_t op = tie_gt ? (eq_d ? 3u : (eq_i ? 2u : 1u)) : (eq_i ? 2u : 3u);
                            beginning = cj;
                            hcur -= (op == 1u) ? s0 : gap;         // exact score of the next cell
                            const int up = op != 3u, left = op != 2u;
                            r -= up; ci -= up; pr -= up;
                            c -= left; cj -= left; pq -= left;
                            p -= up * ES + left * COLB;
                            opword |= op << sh;
                            ++oplen;
                            if ((oplen & 15) == 0) { myops[(oplen >> 4) - 1] = opword; opword = 0; }
                        }
                        if (hcur <= 0 || r == 0 || c == 0) break;  // done, or the path left this tile
                    }
                    if (hcur <= 0) break;
                }
            }
            if (G > 1 && gl < 32) {
                // ---- walk (SmithWaterman.java:380-409), all 32 lanes of the group's first warp in lock step.  Every lane
                // keeps the whole walker state (no shuffles); lane k probes the diagonal cell (r - k, c - k): it is an
                // alignment move iff NW + s == H (the '>=' cascade's first choice), so one ballot finds a whole run of
                // alignment moves; the gap move that ends the run is decided in the same iteration.
                const int wl = gl;
                const int big = max(abs(match), abs(mismatch));
                auto push = [&](uint32_t op, int n) {               // n columns of the same op
                    const uint32_t pattern = op * 0x55555555u;
                    while (n > 0) {
                        const int used = (int)(oplen & 15);
                        const int take = min(n, 16 - used);
                        const uint32_t bits = take == 16 ? pattern : (pattern & ((1u << (2 * take)) - 1u));
                        opword |= bits << (2 * used);
                        oplen += take; n -= take;
                        if ((oplen & 15) == 0) { if (wl == 0) myops[(oplen >> 4) - 1] = opword; opword = 0; }
                    }
                };
                for (;;) {
                    const int T = (ci - 1) / KL;
                    const int kk = T0 - T;
                    if (kk >= HS) break;
                    const int t = T % WL;
                    const int step = cj - 1 + t;
                    const int b = step / WCB;
                    int slot = leader + DB * kk;
                    if (slot_blk[slot] != b) {
                        int dd = 1;
                        while (dd < DB && slot_blk[slot + dd] != b) ++dd;
                        if (dd == DB) break;
                        slot += dd;
                    }
                    int r = ci - T * KL;                           // 1..KL
                    int c = step - b * WCB + 1;                    // 1..WCB
                    const uint8_t *base = reinterpret_cast<const uint8_t *>(slots + (size_t)slot * TW);
                    const uint8_t *p = base + c * COLB + r * ES;   // element (r, c)
                    const uint8_t *pr = base + TG::CODE0 * 4 + (r - 1);          // read code of row r
                    const uint8_t *pq = base + TG::CODE0 * 4 + KL + (c - 1);     // reference code of column c
                    for (;;) {
                        const int lim = min(r, c);                 // cells (r - k, c - k), k < lim, lie inside this tile
                        const bool inside = wl < lim;
                        const uint8_t *pk = p - wl * DG;
                        const int hk = inside ? elem(pk) : 0, hnwk = inside ? elem(pk - DG) : 1;
                        const bool is_m = inside && pr[-wl] == pq[-wl];
                        const int sck = is_m ? match : mismatch;
                        const bool okk = inside && (((hnwk + sck - hk) & M) == 0);
                        const unsigned okm = __ballot_sync(0xffffffffu, okk), mm = __ballot_sync(0xffffffffu, is_m);
                        const int run = tie_gt ? 0 : (okm == 0xffffffffu ? 32 : __ffs((int)~okm) - 1);
                        // a cell is only visited while its score is positive: exact along the run unless the walk is about
                        // to end -- then advance one cell at a time
                        const int L = (hcur > 32 * big) ? run : min(run, 1);
                        if (L > 0) {
                            const unsigned lm = L >= 32 ? 0xffffffffu : ((1u << L) - 1u);
                            const int nm = __popc(mm & lm);
                            hcur -= nm * match + (L - nm) * mismatch;
                            beginning = cj - (L - 1);
                            ci -= L; cj -= L; r -= L; c -= L;
                            p -= L * DG; pr -= L; pq -= L;
                            push(1u, L);
                        }
                        if (hcur <= 0 || r == 0 || c == 0) break;  // done, or the path left this tile
                        if (L == run && run < lim) {
                            // the cell here is known not to take the alignment move ('>=' rule), or the rule is '>'
                            const int hn = elem(p - ES), hw = elem(p - COLB);
                            const bool eq_i = ((hn + gap - hcur) & M) == 0, eq_d = ((hw + gap - hcur) & M) == 0;
                            const int s0 = (pr[0] == pq[0]) ? match : mismatch;
                            const uint32_t op = tie_gt ? (eq_d ? 3u : (eq_i ? 2u : 1u)) : (eq_i ? 2u : 3u);
                            beginning = cj;
                            hcur -= (op == 1u) ? s0 : gap;
                            const int up = op != 3u, left = op != 2u;
                            r -= up; ci -= up; pr -= up;
                            c -= left; cj -= left; pq -= left;
                            p -= up * ES + left * COLB;
                            push(op, 1);
                            if (hcur <= 0 || r == 0 || c == 0) break;
                        }
                    }
                    if (hcur <= 0) break;
                }
            }
            if (G == 32) {
                __syncwarp(gmask);                                 // every lane walked: the state is already uniform
            } else if (G > 32) {
                if (gl == 0) { bc_state[0] = hcur; bc_state[1] = ci; bc_state[2] = cj; }
                __syncthreads();
                hcur = bc_state[0]; ci = bc_state[1]; cj = bc_state[2];
                __syncthreads();
            }
        }
        if (gl == 0) {
            if (oplen & 15) myops[oplen >> 4] = opword;
            beginnings[cell] = beginning;
            op_lens[cell] = (int32_t)oplen;
        }
    }
}

// ---------------------------------------------------------------------------------------
namespace {

template <int KL, int NC>
cudaError_t launch_fill_k(const WideParams &P, const int2 *items, int n_items, uint32_t *ticket, int sm_count, cudaStream_t st)
{
    constexpr int PW = NC > 0 ? NC * KL * WL : 0, SW = 2 * (WL + 16);
    const size_t smem = (size_t)4 * (PW + SW) * sizeof(int32_t);
    int per_sm = KL >= 32 ? 2 : 4;                                          // registers (__launch_bounds__)
    per_sm = std::min<int>(per_sm, (int)((220 * 1024) / (smem + 1024)));    // shared memory
    per_sm = std::max(per_sm, 1);
    const int ctas = (int)std::min<int64_t>(((int64_t)n_items + 3) / 4, (int64_t)sm_count * per_sm);
    cudaError_t e = cudaFuncSetAttribute(wide_fill_kernel<KL, NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    wide_fill_kernel<KL, NC><<<ctas, 128, smem, st>>>(P, items, n_items, ticket, 1);
    return cudaGetLastError();
}

template <int KL>
cudaError_t launch_fill_kl(const WideParams &P, const int2 *items, int n_items, uint32_t *ticket, int sm_count, cudaStream_t st)
{
    if (P.gap < 0 && P.n_symbols <= 4) return launch_fill_k<KL, 4>(P, items, n_items, ticket, sm_count, st);
    if (P.gap < 0 && P.n_symbols <= 8) return launch_fill_k<KL, 8>(P, items, n_items, ticket, sm_count, st);
    return launch_fill_k<KL, 0>(P, items, n_items, ticket, sm_count, st);
}

template <int KL, int NT, int G, bool BYTE>
cudaError_t launch_trace_k(const WideParams &P, const uint64_t *keys, uint32_t n_cells, int32_t *beginnings,
                           int32_t *op_lens, uint32_t *ops, int64_t ops_stride, int sm_count, cudaStream_t st)
{
    const size_t smem = G > 32 ? TraceGeo<KL, BYTE>::smem_bytes(CTAW_TILES) + (size_t)SUB_SMEM_WORDS * 4 : TraceGeo<KL, BYTE>::smem_bytes(NT);
    cudaError_t e = cudaFuncSetAttribute(wide_trace_kernel<KL, NT, G, BYTE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int per_sm = std::max(1, std::min(8, (int)((220 * 1024) / (smem + 1024))));
    const int64_t groups = ((int64_t)n_cells + (NT / G) - 1) / (NT / G);
    const int64_t ctas = std::max<int64_t>(1, std::min<int64_t>(groups, (int64_t)sm_count * per_sm));
    wide_trace_kernel<KL, NT, G, BYTE><<<(unsigned)ctas, NT, smem, st>>>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride);
    return cudaGetLastError();
}

// CTA-wide, pipelined mode: one cluster of C CTAs per max cell (co-scheduled: a CTA waits for tokens of its cluster mates)
template <int KL>
cudaError_t launch_trace_pipe(const WideParams &P0, const uint64_t *keys, uint32_t n_cells, int32_t *beginnings,
                              int32_t *op_lens, uint32_t *ops, int64_t ops_stride, int sm_count, cudaStream_t st)
{
    auto kern = wide_trace_kernel<KL, CTAW_THREADS, CTAW_THREADS, true>;
    const size_t smem = TraceGeo<KL, true>::smem_bytes(CTAW_TILES) + (size_t)SUB_SMEM_WORDS * 4;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    // CTAs per cell.  Measured on cfg3 (ten 100 kbp pairs): 1 / 2 / 3 / 4 / 8 CTAs -> 9.3 / 4.9 / 4.7 / 5.6 / 7.8 ms.  Three keep one
    // prepare hidden behind two walks; more only lengthen the distance over which the entry point is predicted (the
    // path drifts off the predicted diagonal and the prepared corridor has to be redone).
    int c = 3;
    while (c > 1 && (int64_t)n_cells * c > (int64_t)sm_count) --c;           // every cluster resident at once
    WideParams P = P0;
    for (;; --c) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(n_cells * (uint32_t)c));
        cfg.blockDim = dim3(CTAW_THREADS);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)c; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        int n_clusters = 0;
        e = c > 1 ? cudaOccupancyMaxActiveClusters(&n_clusters, kern, &cfg) : cudaSuccess;
        if (c > 1 && (e != cudaSuccess || n_clusters < 1)) { cudaGetLastError(); continue; }   // this cluster size does not fit: halve
        P.pipe_c = c;
        return cudaLaunchKernelEx(&cfg, kern, P, keys, n_cells, beginnings, op_lens, ops, ops_stride);
    }
}

template <int KL>
cudaError_t launch_trace_kl(const WideParams &P, const uint64_t *keys, uint32_t n_cells, int32_t *beginnings,
                            int32_t *op_lens, uint32_t *ops, int64_t ops_stride, int sm_count, cudaStream_t st)
{
    const bool bytes = tile_trace_ok(P.match, P.mismatch, P.gap);        // same bound as the short path's byte tiles
    // lanes per max cell: a whole CTA (corridor of 32 lane-rows x 4 blocks) while there are fewer cells than SMs, a warp
    // (16 x 2) while the cells cannot fill the machine with one thread each, else one thread per cell
    const int g = (int64_t)n_cells <= (int64_t)sm_count ? 128 : ((int64_t)n_cells < (int64_t)sm_count * 256 ? 32 : 1);
    constexpr int NTB = KL >= 32 ? 64 : 128;                              // byte tiles: 80 / 91 / 56 KB per CTA
    if (bytes) {
        if (g >= 128 && P.mail) return launch_trace_pipe<KL>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride, sm_count, st);
        if (g == 32) return launch_trace_k<KL, NTB, 32, true>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride, sm_count, st);
        return launch_trace_k<KL, NTB, 1, true>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride, sm_count, st);
    }
    if (g >= 32) return launch_trace_k<KL, 32, 32, false>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride, sm_count, st);
    return launch_trace_k<KL, 32, 1, false>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride, sm_count, st);
}

}  // namespace

cudaError_t launch_wide_pad_reads(const uint8_t *codes, const int64_t *read_off, const int32_t *reads, int n_reads,
                                  const int64_t *rpad_off, const int64_t *rpad_len, uint8_t *rpad, int64_t max_len,
                                  cudaStream_t st)
{
    if (n_reads == 0) return cudaSuccess;
    const dim3 grid((unsigned)std::max<int64_t>(1, std::min<int64_t>((max_len + 255) / 256, 256)), (unsigned)std::min(n_reads, 4096));
    wide_pad_reads_kernel<<<grid, 256, 0, st>>>(codes, read_off, reads, n_reads, rpad_off, rpad_len, rpad);
    return cudaGetLastError();
}

cudaError_t launch_wide_fill(int KL, const WideParams &P, const int2 *items, int n_items, uint32_t *ticket, int sm_count,
                             cudaStream_t st)
{
    if (n_items == 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    switch (KL) {
        case 8:  return launch_fill_kl<8>(P, items, n_items, ticket, sm_count, st);
        case 16: return launch_fill_kl<16>(P, items, n_items, ticket, sm_count, st);
        case 32: return launch_fill_kl<32>(P, items, n_items, ticket, sm_count, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_wide_flag(const WideParams &P, int64_t total_blocks, WideTask *tasks, uint32_t cap, uint32_t *count,
                             int sm_count, cudaStream_t st)
{
    if (total_blocks == 0) return cudaSuccess;
    const int64_t ctas = std::max<int64_t>(1, std::min<int64_t>((total_blocks + 7) / 8, (int64_t)sm_count * 16));
    wide_flag_kernel<<<(unsigned)ctas, 256, 0, st>>>(P, total_blocks, tasks, cap, count);
    return cudaGetLastError();
}

cudaError_t launch_wide_locate(int KL, const WideParams &P, const WideTask *tasks, const uint32_t *n_tasks, uint32_t cap_tasks,
                               uint64_t *keys, uint32_t cap, uint32_t *count, int sm_count, cudaStream_t st)
{
    const int64_t ctas = std::max<int64_t>(1, std::min<int64_t>(((int64_t)cap_tasks + 127) / 128, (int64_t)sm_count * 8));
    switch (KL) {
        case 8:  wide_locate_kernel<8><<<(unsigned)ctas, 128, 0, st>>>(P, tasks, n_tasks, cap_tasks, keys, cap, count); break;
        case 16: wide_locate_kernel<16><<<(unsigned)ctas, 128, 0, st>>>(P, tasks, n_tasks, cap_tasks, keys, cap, count); break;
        case 32: wide_locate_kernel<32><<<(unsigned)ctas, 128, 0, st>>>(P, tasks, n_tasks, cap_tasks, keys, cap, count); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t launch_wide_trace(int KL, const WideParams &P, const uint64_t *keys, uint32_t n_cells, int32_t *beginnings,
                              int32_t *op_lens, uint32_t *ops, int64_t ops_stride, int sm_count, cudaStream_t st)
{
    if (n_cells == 0) return cudaSuccess;
    switch (KL) {
        case 8:  return launch_trace_kl<8>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride, sm_count, st);
        case 16: return launch_trace_kl<16>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride, sm_count, st);
        case 32: return launch_trace_kl<32>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride, sm_count, st);
    }
    return cudaErrorInvalidValue;
}

}  // namespace swb
