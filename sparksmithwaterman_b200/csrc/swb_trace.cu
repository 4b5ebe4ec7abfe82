// swb_trace.cu -- short-read path: tile flagging, the group-based traceback (fallback), small reductions.
//
// The fill (swb_fill*.cu) leaves, per pair, the (tracked) maximum score, per-(block, lane) tile maxima and the
// block records.  Here:
//   flag_tiles : tiles whose maximum is within P.tmx_slack of the pair's tracked maximum (slack 0: equal to it)
//   trace      : GROUP-based traceback, used when the byte tiles of the default kernel (swb_trace_tile.cu) cannot
//                represent the score set (tile_trace_ok): per max cell, GetAlignment.call (SmithWaterman.java:
//                354-436): walk while the score is positive; the type of a positive cell is re-derived from the
//                scores with the priority of the ">=" cascade (:228,:236,:245): alignment, then insertion, then
//                deletion.  Blocks are recomputed lazily, right to left, each from its own checkpoints (all 8
//                lanes of the group), so every H the walk reads is exact.
//   ref_totals, best_hits, key sort: the per-call reductions of Distribution.MapRef (:424) and
//                the best-hit records merged across GPUs.
// Max-cell enumeration and the default traceback live in swb_trace_tile.cu.
#include "swb_internal.h"
#include "swb_device.cuh"

#include <algorithm>
#include <cub/device/device_radix_sort.cuh>

namespace swb {

// ---------------------------------------------------------------------------------------
// One thread per global checkpoint block gb (x) and slice of the read pairs (y): the owning reference is
// searched once and reused for every read pair; one task per (half, lane) whose tile maximum is within
// P.tmx_slack of the pair's (tracked) maximum -- with exact tile maxima (slack 0) that is equality.
constexpr int FLAG_WARPS = 8;
__global__ void __launch_bounds__(FLAG_WARPS * 32) flag_tiles_kernel(const BatchParams P, TileTask *tasks, uint32_t cap, uint32_t *count)
{
    __shared__ uint32_t wsum[FLAG_WARPS];
    __shared__ uint32_t bbase;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slack = P.tmx_slack;                               // 0: exact tile maxima; > 0: subsampled (swb_fill_bias.cu)
    const int64_t gb = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const bool in = gb < P.blocks_per_rp;
    int ref = 0, b = 0;
    int64_t ro = 0;
    if (in) {
        int lo = 0, hi = P.n_refs;
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (P.ref_blk_off[mid] <= gb) lo = mid; else hi = mid; }
        ref = lo;
        b = (int)(gb - P.ref_blk_off[ref]);
        ro = P.ref_orig[ref];
    }
    // four read pairs per round: all loads of a round are issued before any is used (the kernel is latency-bound)
    for (int rp0 = blockIdx.y * 4; rp0 < P.n_rp; rp0 += gridDim.y * 4) {
        uint4 v0[4], v1[4];
        int sa[4], sb[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int rp = rp0 + k;
            const bool ok = in && rp < P.n_rp;
            const int ra = ok ? P.rp_reads[2 * rp] : 0, rb = ok ? P.rp_reads[2 * rp + 1] : -1;
            sa[k] = ok ? P.scores[ro * P.n_reads + ra] : 0;
            sb[k] = rb >= 0 ? P.scores[ro * P.n_reads + rb] : 0;
            const uint4 *tm = reinterpret_cast<const uint4 *>(P.tmx + ((int64_t)rp * P.blocks_per_rp + gb) * GL);
            v0[k] = ok ? __ldcs(tm) : make_uint4(0, 0, 0, 0);
            v1[k] = ok ? __ldcs(tm + 1) : make_uint4(0, 0, 0, 0);
        }
        uint32_t ma[4], mb[4], nt = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            ma[k] = 0; mb[k] = 0;
            const uint32_t w[GL] = {v0[k].x, v0[k].y, v0[k].z, v0[k].w, v1[k].x, v1[k].y, v1[k].z, v1[k].w};
#pragma unroll
            for (int t = 0; t < GL; ++t) {
                const int wa = half_of(w[t], 0), wb = half_of(w[t], 1);
                if (sa[k] > 0 && wa > 0 && wa >= sa[k] - slack) ma[k] |= 1u << t;
                if (sb[k] > 0 && wb > 0 && wb >= sb[k] - slack) mb[k] |= 1u << t;
            }
            nt += (uint32_t)(__popc(ma[k]) + __popc(mb[k]));
        }
        // ONE atomic per CTA and round: the counter is a single address, and ~half of all warps find a tile
        // (one atomic per warp serialised in L2: 0.6 of the kernel's 0.7 ms)
        uint32_t inc = nt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            const uint32_t mine = lane < FLAG_WARPS ? wsum[lane] : 0u;
            uint32_t x = mine;
#pragma unroll
            for (int o = 1; o < FLAG_WARPS; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += v; }
            if (lane < FLAG_WARPS) wsum[lane] = x - mine;
            if (lane == FLAG_WARPS - 1) bbase = x ? atomicAdd(count, x) : 0u;
        }
        __syncthreads();
        uint32_t kk = bbase + wsum[warp] + inc - nt;
        __syncthreads();                                            // wsum / bbase are rewritten next round
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int rp = rp0 + k;
            for (uint32_t mm = ma[k]; mm; mm &= mm - 1, ++kk)
                if (kk < cap) tasks[kk] = TileTask{(uint32_t)rp * 2u, (uint32_t)ref, (uint32_t)b, (uint32_t)(__ffs((int)mm) - 1)};
            for (uint32_t mm = mb[k]; mm; mm &= mm - 1, ++kk)
                if (kk < cap) tasks[kk] = TileTask{(uint32_t)rp * 2u + 1u, (uint32_t)ref, (uint32_t)b, (uint32_t)(__ffs((int)mm) - 1)};
        }
    }
}

cudaError_t launch_flag_tiles(const BatchParams &P, TileTask *tasks, uint32_t cap, uint32_t *count, int sm_count, cudaStream_t st)
{
    if (P.blocks_per_rp == 0 || P.n_rp == 0) return cudaSuccess;
    const int threads = FLAG_WARPS * 32;
    const int64_t bx = (P.blocks_per_rp + threads - 1) / threads;
    const int64_t by = std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>((P.n_rp + 3) / 4, 65535), ((int64_t)sm_count * 16 + bx - 1) / bx));
    flag_tiles_kernel<<<dim3((unsigned)bx, (unsigned)by), threads, 0, st>>>(P, tasks, cap, count);
    return cudaGetLastError();
}

template <int K> struct TraceGeo {
    // lanes of a half's tile: a walk of CB steps climbs at most CB rows (plus rare insertion runs,
    // which simply end the block early), i.e. ceil(CB / K) lanes above the current one
    static constexpr int NLW = ((CB + K - 1) / K + 1) < GL ? ((CB + K - 1) / K + 1) : GL;
    static constexpr int KW = Geo<K>::KW;
    static constexpr int HALF_WORDS = NLW * (CB + 1) * KW;            // one half's tile: [slot][column][KW packed words]
    static constexpr int CODE_WORDS = ((2 * NLW * (CB + 1) + 1 + 15) / 16) * 4;   // [half][slot][column] bytes + 1 trash byte
    static constexpr int GROUP_WORDS = 2 * HALF_WORDS + CODE_WORDS + KW;         // + one trash column
};

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// one tile column: word 0 = boundary row received from the lane above, words 1..K = this lane's rows
template <int K>
__device__ __forceinline__ void store_col(uint32_t *dst, uint32_t top, const uint32_t (&H)[K])
{
    constexpr int KW = Geo<K>::KW;
#pragma unroll
    for (int q = 0; q < KW / 4; ++q) {
        uint4 v;
        v.x = (4 * q == 0) ? top : ((4 * q - 1 < K) ? H[(4 * q - 1 < K && 4 * q >= 1) ? 4 * q - 1 : 0] : 0u);
        v.y = (4 * q + 0 < K) ? H[(4 * q + 0 < K) ? 4 * q + 0 : 0] : 0u;
        v.z = (4 * q + 1 < K) ? H[(4 * q + 1 < K) ? 4 * q + 1 : 0] : 0u;
        v.w = (4 * q + 2 < K) ? H[(4 * q + 2 < K) ? 4 * q + 2 : 0] : 0u;
        reinterpret_cast<uint4 *>(dst)[q] = v;
    }
}

// ---------------------------------------------------------------------------------------
// Traceback, packed: one 8-lane group walks TWO max cells at once, one per s16 half.
// Keys are sorted (read slot, ref, i, j), so a run of cells shares its read: the two halves
// align the same read rows against two (usually different) references, and the score
// profile depends on the read only:
//     prof2[cA*5 + cB][lane][row] = pack(s(read[row], cA), s(read[row], cB)),  code 4 = "no column"
// (S_PAD: a column left of the matrix stays all-zero, one right of it is never read).
// Each half restarts from ITS block's checkpoint (own ref, own block index); the group then
// runs the same three-op cell as the (unbiased) fill for CB steps.  Only the lanes a walk of CB
// steps can reach are kept, [tc - NLW + 1, tc] around the current cell's lane tc, per half:
//     tile[half][slot][c][w]   c = 0..CB (c = 0: the checkpointed column), w = 0: boundary row
//                              received from lane-1 (matrix row lane*K), w = 1..K: the lane's rows
// so W, N and NW of a cell with c >= 1 lie in the same slot.  Lanes outside a window store to a
// trash column (no branches in the step loop).  Lane h of the group walks half h
// (GetAlignment.call, SmithWaterman.java:380-409) until the path leaves what the block holds, then
// the block that holds the current cell is recomputed -- exact, because every block starts
// from the fill's own registers.
template <int K>
__global__ void __launch_bounds__(128) trace_kernel(const BatchParams P, const uint64_t *keys, uint32_t n_cells,
                                                     int chunk, int32_t *beginnings, int32_t *op_lens, uint32_t *ops,
                                                     int ops_stride, uint32_t zero)
{
    using G = Geo<K>;
    using TG = TraceGeo<K>;
    constexpr int KW = G::KW;
    constexpr int NLW = TG::NLW;
    constexpr int HALF_WORDS = TG::HALF_WORDS;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ uint32_t seg_next;
    uint32_t *prof2 = smem;                                         // [25][GL][KS]
    const int lane = threadIdx.x & 31, t = lane & (GL - 1), g = lane >> 3, warp = threadIdx.x >> 5;
    uint32_t *gbase = smem + 25 * G::CSTRIDE + (size_t)(warp * 4 + g) * TG::GROUP_WORDS;
    uint32_t *tile = gbase;
    uint8_t *codes = reinterpret_cast<uint8_t *>(gbase + 2 * HALF_WORDS);   // [half][slot][CB + 1]
    uint8_t *trash_code = codes + 2 * NLW * (CB + 1);
    uint32_t *trash = gbase + 2 * HALF_WORDS + TG::CODE_WORDS;
    uint8_t *rcodes_s = reinterpret_cast<uint8_t *>(smem + 25 * G::CSTRIDE + (size_t)(blockDim.x >> 3) * TG::GROUP_WORDS);   // [GL*K]
    const uint32_t g2 = pack2(P.gap, P.gap);
    const int my_prof = t * G::KS;

    const uint32_t c_lo = blockIdx.x * (uint32_t)chunk;
    const uint32_t c_hi = min(n_cells, c_lo + (uint32_t)chunk);
    uint32_t seg_lo = c_lo;
    while (seg_lo < c_hi) {
        // ---- segment = run of cells of one read (slot) -----------------------------------
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
        for (int idx = threadIdx.x; idx < 25 * GL * K; idx += blockDim.x) {
            const int cc = idx / (GL * K), rem = idx - cc * GL * K;
            const int tt = rem / K, r = rem - tt * K;
            const int row = tt * K + r;
            const int ca = cc / 5, cb = cc - ca * 5;
            int lo = S_PAD, hi = S_PAD;
            if (row < m) {
                const int q = P.read_codes[roff + row];
                if (ca < 4) lo = (q == ca) ? P.match : P.mismatch;
                if (cb < 4) hi = (q == cb) ? P.match : P.mismatch;
            }
            prof2[cc * G::CSTRIDE + tt * G::KS + r] = pack2(lo, hi);
        }
        for (int idx = threadIdx.x; idx < GL * K; idx += blockDim.x)
            rcodes_s[idx] = idx < m ? P.read_codes[roff + idx] : (uint8_t)0xFE;
        if (threadIdx.x == 0) seg_next = seg_lo;
        __syncthreads();

        // ---- per-half state, replicated in the 8 lanes of the group ----------------------
        bool busy0 = false, busy1 = false;
        int ci0 = 0, cj0 = 0, ci1 = 0, cj1 = 0, n0 = 0, n1 = 0;
        const uint32_t *rw0 = P.ref_words, *rw1 = P.ref_words;
        int64_t bk0 = 0, bk1 = 0;
        // walker state, replicated in the 4 lanes of a half's walk team (lanes 0-3: half 0, 4-7: half 1);
        // the team leader (lane 0 / 4) writes the results
        uint32_t w_cell = 0, w_opword = 0;
        int w_h = 0, w_beg = 0, w_len = 0;

        for (;;) {
            // fetch a new cell for every idle half
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const bool idle = h ? !busy1 : !busy0;
                uint32_t e = 0xffffffffu;
                if (idle && t == 4 * h) e = atomicAdd(&seg_next, 1u);
                e = __shfl_sync(FULL, e, 4 * h, GL);
                if (idle && e < seg_hi) {
                    const uint64_t key = keys[e];
                    const int ro = (int)(key_pair(key) - (uint64_t)slot * (uint64_t)P.n_refs);
                    const int ref = P.ref_sorted_of[ro];
                    const int ii = (int)key_i(key), jj = (int)key_j(key);
                    if (h == 0) { busy0 = true; ci0 = ii; cj0 = jj; n0 = P.ref_len[ref]; rw0 = P.ref_words + P.ref_word_off[ref];
                                  bk0 = (int64_t)(slot >> 1) * P.blocks_per_rp + P.ref_blk_off[ref]; }
                    else        { busy1 = true; ci1 = ii; cj1 = jj; n1 = P.ref_len[ref]; rw1 = P.ref_words + P.ref_word_off[ref];
                                  bk1 = (int64_t)(slot >> 1) * P.blocks_per_rp + P.ref_blk_off[ref]; }
                    if ((t >> 2) == h) {                             // the 4 lanes of this half's walk team
                        w_cell = e; w_opword = 0; w_beg = 0; w_len = 0;
                        w_h = P.scores[(int64_t)ro * P.n_reads + read_idx];
                    }
                }
            }
            if (!__any_sync(FULL, busy0 || busy1)) break;

            // ---- block of each half, checkpoint -> registers ---------------------------------
            const int tca = (ci0 - 1) / K, tcb = (ci1 - 1) / K;
            const int b0 = busy0 ? (cj0 - 1 + tca) / CB : 0;
            const int b1 = busy1 ? (cj1 - 1 + tcb) / CB : 0;
            // this lane's slot in each half's window [tc - NLW + 1, tc]; outside: the trash column
            const int sa = busy0 ? t - (tca - NLW + 1) : -1;
            const int sb = busy1 ? t - (tcb - NLW + 1) : -1;
            const bool ina = sa >= 0 && sa < NLW, inb = sb >= 0 && sb < NLW;
            // ONE packed column store per lane and step (shared-memory bandwidth is this kernel's tightest
            // resource): physical slots 0..NLW-1 hold half 0's window, NLW..2NLW-1 the lanes that are only in
            // half 1's window; a lane in both windows lives in half 0's slot and half 1's walker looks it up there
            const int phys = ina ? sa : (inb ? NLW + sb : -1);
            uint32_t *pa = phys >= 0 ? tile + (size_t)phys * (CB + 1) * KW : trash;
            uint8_t *qa = ina ? codes + sa * (CB + 1) : trash_code;
            uint8_t *qb = inb ? codes + (NLW + sb) * (CB + 1) : trash_code;
            const int inca = phys >= 0 ? KW : 0, incqa = ina ? 1 : 0, incqb = inb ? 1 : 0;

            uint32_t H[K], diag = 0;
            {
                const uint32_t *ckA = rec_lane<K>(P.rec, bk0 + b0, t);
                const uint32_t *ckB = rec_lane<K>(P.rec, bk1 + b1, t);
                const bool la = busy0 && b0 > 0, lb = busy1 && b1 > 0;
                const uint32_t sel = rh ? 0x7632u : 0x5410u;        // (A.half rh) | (B.half rh) << 16
#pragma unroll
                for (int p = 0; p < G::CKP; ++p) {
                    uint32_t a[8] = {0, 0, 0, 0, 0, 0, 0, 0}, bq[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                    if (la) ldg256(ckA + p * REC_P, a);
                    if (lb) ldg256(ckB + p * REC_P, bq);
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const int w = 8 * p + e;
                        const uint32_t v = __byte_perm(a[e], bq[e], sel);
                        if (w < K) H[w < K ? w : 0] = v;
                        else if (w == K) diag = v;
                    }
                }
            }
            // the path almost always continues into the block to the left: pull its records towards L2
            if (busy0 && b0 > 1) prefetch_l2(rec_lane<K>(P.rec, bk0 + b0 - 1, t));
            if (busy1 && b1 > 1) prefetch_l2(rec_lane<K>(P.rec, bk1 + b1 - 1, t));
            // reference-code windows of this lane for the block: 0-based columns j0 .. j0+15
            uint32_t win0, win1; int ulo0, uhi0, ulo1, uhi1;
            {
                const int j0 = b0 * CB - t, j1 = b1 * CB - t;
                const int wi0 = j0 >> 4, wi1 = j1 >> 4;                   // floor (j may be negative in block 0)
                const uint32_t a0 = (busy0 && wi0 >= 0 && wi0 * 16 < n0) ? __ldg(rw0 + wi0) : 0u;
                const uint32_t a1 = (busy0 && wi0 + 1 >= 0 && (wi0 + 1) * 16 < n0) ? __ldg(rw0 + wi0 + 1) : 0u;
                const uint32_t c0 = (busy1 && wi1 >= 0 && wi1 * 16 < n1) ? __ldg(rw1 + wi1) : 0u;
                const uint32_t c1 = (busy1 && wi1 + 1 >= 0 && (wi1 + 1) * 16 < n1) ? __ldg(rw1 + wi1 + 1) : 0u;
                win0 = __funnelshift_r(a0, a1, 2 * (j0 & 15));
                win1 = __funnelshift_r(c0, c1, 2 * (j1 & 15));
                // step u computes 0-based column j0 + u: valid iff 0 <= j0 + u < n
                ulo0 = -j0; uhi0 = busy0 ? n0 - j0 - 1 : -1;
                ulo1 = -j1; uhi1 = busy1 ? n1 - j1 - 1 : -1;
            }
            // halo column c = 0
            store_col<K>(pa, diag, H);
            pa += inca; qa += incqa; qb += incqb;

            // interior block: every step of every lane / half is a real column -> no per-step validity tests
            const bool interior = ulo0 <= 0 && uhi0 >= CB - 1 && ulo1 <= 0 && uhi1 >= CB - 1;
            if (__all_sync(FULL, interior)) {
#pragma unroll 4
                for (int u = 0; u < CB; ++u) {
                    uint32_t top = __shfl_up_sync(FULL, H[K - 1], 1, GL);
                    if (t == 0) top = 0;
                    const uint32_t ca = (win0 >> (2 * u)) & 3u, cb = (win1 >> (2 * u)) & 3u;
                    uint32_t sv[G::KP];
                    load_profile<G::KP>(prof2 + (ca * 5 + cb) * G::CSTRIDE + my_prof, sv);
                    uint32_t nw = diag, nn = top;
#pragma unroll
                    for (int r = 0; r < K; ++r) {
                        const uint32_t x = viaddmax_relu(nw, sv[r], zero);
                        const uint32_t pre = viaddmax(H[r], g2, x);
                        nw = H[r];
                        H[r] = viaddmax(nn, g2, pre);
                        nn = H[r];
                    }
                    diag = top;
                    store_col<K>(pa, top, H);
                    *qa = (uint8_t)ca; *qb = (uint8_t)cb;
                    pa += inca; qa += incqa; qb += incqb;
                }
            } else {
#pragma unroll 1
                for (int u = 0; u < CB; ++u) {
                    uint32_t top = __shfl_up_sync(FULL, H[K - 1], 1, GL);
                    if (t == 0) top = 0;
                    const uint32_t ca = (u >= ulo0 && u <= uhi0) ? ((win0 >> (2 * u)) & 3u) : 4u;
                    const uint32_t cb = (u >= ulo1 && u <= uhi1) ? ((win1 >> (2 * u)) & 3u) : 4u;
                    uint32_t sv[G::KP];
                    load_profile<G::KP>(prof2 + (ca * 5 + cb) * G::CSTRIDE + my_prof, sv);
                    uint32_t nw = diag, nn = top;
#pragma unroll
                    for (int r = 0; r < K; ++r) {
                        const uint32_t x = viaddmax_relu(nw, sv[r], zero);
                        const uint32_t pre = viaddmax(H[r], g2, x);
                        nw = H[r];
                        H[r] = viaddmax(nn, g2, pre);
                        nn = H[r];
                    }
                    diag = top;
                    store_col<K>(pa, top, H);
                    *qa = (uint8_t)ca; *qb = (uint8_t)cb;
                    pa += inca; qa += incqa; qb += incqb;
                }
            }
            __syncwarp();

            // ---- walk (GetAlignment.call, SmithWaterman.java:380-409), four lanes per half ----------------
            // Lane q of a team looks at the cell q steps up the diagonal from the current one and derives ITS
            // move from the tile.  Alignment paths are mostly diagonal, so a ballot finds the run of leading
            // "alignment" moves and the whole run (plus the first gap move after it) is applied in one round:
            // ~3 path steps per round instead of one load -> compare -> select chain per step.
            const int h = t >> 2, q = t & 3;
            const bool mybusy = h ? busy1 : busy0;
            int ci = h ? ci1 : ci0, cj = h ? cj1 : cj0;
            const int b = h ? b1 : b0;
            const int lane_lo = (h ? tcb : tca) - NLW + 1;              // first lane held in this half's window
            const int a_lo = tca - NLW + 1;
            const int16_t *T16 = reinterpret_cast<const int16_t *>(tile);   // halfword 2*w + h of packed word w
            const uint8_t *tcodes = codes + h * NLW * (CB + 1);
            auto phys_of = [&](int s_) -> int {                           // physical slot of window position s_
                if (h == 0) return s_;
                const int in_a = (lane_lo + s_) - a_lo;
                return (busy0 && in_a >= 0 && in_a < NLW) ? in_a : NLW + s_;
            };
            // position of the current cell inside the tile, kept incrementally
            const int tc0 = (ci - 1) / K;
            int r = ci - tc0 * K;                                        // 1..K
            int c = cj - (b * CB - tc0);
            int sl = tc0 - lane_lo;
            bool walking = mybusy;                                        // this half still walks in this block
            int done = 0;
            const int team = lane & ~3;
            while (__any_sync(FULL, walking)) {
                // my cell: q steps up the diagonal
                int r_q = r - q, sl_q = sl, c_q = c - q;
                if (r_q <= 0) { r_q += K; --sl_q; --c_q; }
                const int ci_q = ci - q, cj_q = cj - q;
                const bool in = walking && ci_q >= 1 && cj_q >= 1 && c_q >= 1 && sl_q >= 0;
                int hc = 0, hw = 0, hn = 0, hnw = 0, rc = 0, qc = 1;
                if (in) {
                    const int idx = 2 * ((phys_of(sl_q) * (CB + 1) + c_q) * KW + r_q) + h;
                    hc = T16[idx]; hw = T16[idx - 2 * KW]; hn = T16[idx - 2]; hnw = T16[idx - 2 * KW - 2];
                    rc = tcodes[sl_q * (CB + 1) + c_q];
                    qc = rcodes_s[ci_q - 1];
                }
                const int sc = (qc == rc) ? P.match : P.mismatch;
                // type of a positive cell = first of (alignment, insertion, deletion) whose candidate equals H:
                // the ">=" cascade of GetCellScore.call; SWB_F_TIE_GT: first of (deletion, insertion, alignment)
                const bool eq_a = (hnw + sc == hc), eq_i = (hn + P.gap == hc), eq_d = (hw + P.gap == hc);
                const uint32_t op = P.tie_gt ? (eq_d ? 3u : (eq_i ? 2u : 1u)) : (eq_a ? 1u : (eq_i ? 2u : 3u));
                const bool alive = in && hc > 0;
                const int hnext = op == 1u ? hnw : (op == 2u ? hn : hw);
                const uint32_t bal = (__ballot_sync(FULL, alive && op == 1u) >> team) & 0xFu;
                const int n_a = __ffs((int)(~bal & 0x1Fu)) - 1;         // leading alignment moves: 0..4
                const int src = team + min(n_a, 3);
                const bool alive_s = __shfl_sync(FULL, (int)alive, src) != 0;
                const uint32_t op_s = __shfl_sync(FULL, op, src);
                const int hnext_s = __shfl_sync(FULL, hnext, src);
                const int hnw_prev = __shfl_sync(FULL, hnw, team + max(n_a - 1, 0));
                const bool extra = n_a < 4 && alive_s;                   // lane n_a's own (gap) move is applied too
                const int steps = n_a + (extra ? 1 : 0);
                if (walking) {
                    if (steps == 0) {
                        // the current cell is outside what this block holds (or its score is 0: cannot happen here)
                        walking = false;
                    } else {
                        const int up = extra ? (op_s != 3u) : 0, left = extra ? (op_s != 2u) : 0;
                        w_beg = extra ? cj - n_a : cj - n_a + 1;        // column of the last cell that made a move
                        const uint64_t bits = (n_a ? (0x55ull >> (8 - 2 * n_a)) : 0ull) | (extra ? (uint64_t)op_s << (2 * n_a) : 0ull);
                        const uint64_t acc = (uint64_t)w_opword | (bits << (2 * (w_len & 15)));
                        const int nl = w_len + steps;
                        if ((nl >> 4) != (w_len >> 4)) {                 // a 16-column word is complete
                            if (q == 0) ops[(size_t)w_cell * ops_stride + (w_len >> 4)] = (uint32_t)acc;
                            w_opword = (uint32_t)(acc >> 32);
                        } else {
                            w_opword = (uint32_t)acc;
                        }
                        w_len = nl;
                        w_h = extra ? hnext_s : ((n_a == 4) ? hnext_s : hnw_prev);
                        ci -= n_a + up; cj -= n_a + left;
                        r -= n_a + up; c -= n_a + left;
                        if (r <= 0) { r += K; --sl; --c; }
                        if (r <= 0) { r += K; --sl; --c; }
                        if (w_h <= 0) { walking = false; done = 1; }
                    }
                }
            }
            if (done && q == 0) {
                if (w_len & 15) ops[(size_t)w_cell * ops_stride + (w_len >> 4)] = w_opword;
                beginnings[w_cell] = w_beg;
                op_lens[w_cell] = w_len;
            }
            {
                const int d0 = __shfl_sync(FULL, done, 0, GL), d1 = __shfl_sync(FULL, done, 4, GL);
                const int i0 = __shfl_sync(FULL, ci, 0, GL), j0 = __shfl_sync(FULL, cj, 0, GL);
                const int i1 = __shfl_sync(FULL, ci, 4, GL), j1 = __shfl_sync(FULL, cj, 4, GL);
                if (busy0) { ci0 = i0; cj0 = j0; if (d0) busy0 = false; }
                if (busy1) { ci1 = i1; cj1 = j1; if (d1) busy1 = false; }
            }
            __syncwarp();
        }
        seg_lo = seg_hi;
    }
}

template <int K>
static cudaError_t launch_trace_k(const BatchParams &P, const uint64_t *keys, uint32_t n_cells, int32_t *beginnings,
                                  int32_t *op_lens, uint32_t *ops, int ops_stride, int sm_count, cudaStream_t st)
{
    using G = Geo<K>;
    if (n_cells == 0) return cudaSuccess;
    const size_t per_group = (size_t)TraceGeo<K>::GROUP_WORDS * sizeof(uint32_t);
    const size_t prof_bytes = (size_t)25 * G::CSTRIDE * sizeof(uint32_t);
    const size_t tail_bytes = (((size_t)GL * K + 15) / 16) * 16;
    int warps = 4;
    while (warps > 1 && prof_bytes + per_group * 4 * warps + tail_bytes > 112 * 1024) --warps;   // two CTAs per SM
    const size_t smem = prof_bytes + per_group * 4 * warps + tail_bytes;
    static PerDeviceOnce attr;                    // one per template instantiation (K)
    {
        const cudaError_t e = attr.run([&] { return cudaFuncSetAttribute(trace_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
        if (e != cudaSuccess) return e;
    }
    // chunks of the sorted cell list: several per SM for balance, each long enough to amortise its profile (hits mode,
    // P.sel: a few cells per read, one chunk may be a single cell -- see launch_tile_trace_k)
    int chunk = (int)std::max<int64_t>(P.sel ? 1 : 256, ((int64_t)n_cells + sm_count * 4 - 1) / (sm_count * 4));
    const int64_t ctas = ((int64_t)n_cells + chunk - 1) / chunk;
    trace_kernel<K><<<(unsigned)ctas, warps * 32, smem, st>>>(P, keys, n_cells, chunk, beginnings, op_lens, ops, ops_stride, 0u);
    return cudaGetLastError();
}

cudaError_t launch_trace(int K, const BatchParams &P, const uint64_t *keys, uint32_t n_cells, int32_t *beginnings,
                         int32_t *op_lens, uint32_t *ops, int ops_stride_words, int sm_count, cudaStream_t st)
{
    switch (K) {
        case 4:  return launch_trace_k<4>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 5:  return launch_trace_k<5>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 7:  return launch_trace_k<7>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 10: return launch_trace_k<10>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 8:  return launch_trace_k<8>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 13: return launch_trace_k<13>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 16: return launch_trace_k<16>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 19: return launch_trace_k<19>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 25: return launch_trace_k<25>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
        case 32: return launch_trace_k<32>(P, keys, n_cells, beginnings, op_lens, ops, ops_stride_words, sm_count, st);
    }
    return cudaErrorInvalidValue;
}

// ---------------------------------------------------------------------------------------
// per-reference wrapping int32 total over reads (Distribution.java:424): one warp per ref
__global__ void ref_totals_kernel(const int32_t *scores, int64_t n_refs, int64_t n_reads, int32_t *totals)
{
    const int64_t ref = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (ref >= n_refs) return;
    uint32_t acc = 0;
    for (int64_t q = lane; q < n_reads; q += 32) acc += (uint32_t)scores[ref * n_reads + q];
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) totals[ref] = (int32_t)acc;
}

cudaError_t launch_ref_totals(const int32_t *scores, int64_t n_refs, int64_t n_reads, int32_t *totals, cudaStream_t st)
{
    if (n_refs == 0) return cudaSuccess;
    const int threads = 256;
    const int64_t blocks = (n_refs * 32 + threads - 1) / threads;
    ref_totals_kernel<<<(unsigned)blocks, threads, 0, st>>>(scores, n_refs, n_reads, totals);
    return cudaGetLastError();
}

// per-read best reference: highest score, lowest ref index on ties.  best[4q] = score, [4q+1] = ref.
// Phase 1: thread = (read q, slice of the references), coalesced over q; 64-bit atomicMax of
// (score << 32 | ~ref) into the first two words of the read's record.  Phase 2 decodes.
__global__ void best_hits_scan_kernel(const int32_t *scores, int64_t n_refs, int64_t n_reads, unsigned long long *best64)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_reads) return;
    int bs = -1; int64_t br = -1;
    for (int64_t r = blockIdx.y; r < n_refs; r += gridDim.y) {
        const int s = scores[r * n_reads + q];
        if (s > bs) { bs = s; br = r; }
    }
    if (br >= 0)
        atomicMax(best64 + 2 * q, ((unsigned long long)(uint32_t)max(bs, 0) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)br));
}

__global__ void best_hits_finish_kernel(int32_t *best, int64_t n_reads)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_reads) return;
    const unsigned long long k = reinterpret_cast<const unsigned long long *>(best)[2 * q];
    int4 o;
    o.x = (int)(uint32_t)(k >> 32);
    o.y = k ? (int)(0xffffffffu - (uint32_t)k) : -1;          // no reference at all: (0, -1)
    o.z = 0; o.w = 0;
    reinterpret_cast<int4 *>(best)[q] = o;
}

cudaError_t launch_best_hits(const int32_t *scores, int64_t n_refs, int64_t n_reads, int32_t *best, int sm_count, cudaStream_t st)
{
    if (n_reads == 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(best, 0, (size_t)n_reads * 16, st);
    if (e != cudaSuccess) return e;
    const int threads = 128;
    const int64_t bx = (n_reads + threads - 1) / threads;
    if (n_refs > 0) {
        const int64_t by = std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(n_refs, 65535), ((int64_t)sm_count * 16 + bx - 1) / bx));
        best_hits_scan_kernel<<<dim3((unsigned)bx, (unsigned)by), threads, 0, st>>>(scores, n_refs, n_reads,
                                                                                    reinterpret_cast<unsigned long long *>(best));
    }
    best_hits_finish_kernel<<<(unsigned)bx, threads, 0, st>>>(best, n_reads);
    return cudaGetLastError();
}

size_t sort_keys_tmp_bytes(uint32_t n)
{
    size_t bytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, bytes, (const uint64_t *)nullptr, (uint64_t *)nullptr, (int)n);
    return bytes;
}

cudaError_t sort_keys(uint64_t *keys_in, uint64_t *keys_out, uint32_t n, void *tmp, size_t tmp_bytes, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    return cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, keys_in, keys_out, (int)n, 0, 64, st);
}

}  // namespace swb
