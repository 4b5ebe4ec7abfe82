// swb_fill.cu -- score-matrix fill of the short-read path (sm_100a, DPX s16x2).
//
// Computes, for every (read, reference) pair of a batch, the maximum of
//   H(i,j) = max(0, H(i,j-1)+gap, H(i-1,j)+gap, H(i-1,j-1)+match|mismatch)
// which is the score recurrence of GetCellScore.call / InsDelScore.call /
// AlignmentScore.call (reference SmithWaterman.java:217-252, :277-280, :309-318) as
// iterated by ScoreMatrix.call (:157-187).  Scores only: the tie rule of the ">="
// cascade affects alignment types, never H, so the fill needs no direction state.
// The locate / traceback kernels (swb_trace_tile.cu, swb_trace.cu) restart from the block records written here.
//
// Per cell pair (two reads packed in s16x2):  VIADDMNMX.RELU  x   = max(NW + s, 0)
//                                             VIADDMNMX       pre = max(W + gap, x)
//                                             VIADDMNMX       H   = max(N + gap, pre)
// plus half a VIMNMX3 for the running tile maximum.  The dependent chain down a lane's
// K rows is one VIADDMNMX per row; x and pre of all rows are independent.
#include "swb_internal.h"
#include "swb_device.cuh"

#include <algorithm>
#include <cstdlib>

namespace swb {

template <int K>
__global__ void __launch_bounds__(512) fill_kernel(const BatchParams P, uint32_t *work_counter, uint32_t zero)
{
    using G = Geo<K>;
    extern __shared__ __align__(16) uint32_t prof_all[];        // per warp: [4 codes][GL lanes][KS]

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t = lane & (GL - 1), g = lane >> 3;
    uint32_t *prof = prof_all + warp * G::PROF_WORDS;
    const int n_quads = (P.n_vrefs + 3) >> 2;
    const uint32_t n_items = (uint32_t)n_quads * (uint32_t)P.n_rp;

    const uint32_t g2 = pack2(P.gap, P.gap);
    // `zero` is a kernel argument (always 0): ptxas cannot fold it, so the RELU ops take it from a
    // register instead of re-materialising a packed zero with one PRMT per cell
    const uint32_t lmask = t ? 0xffffffffu : 0u;
    const int my_prof = t * G::KS;
    int cur_rp = -1, ra = 0, rb = -1;

    // persistent warps: items (quad, read pair) are handed out quad-major, i.e. longest
    // references first, through one global counter -> no tail, no per-CTA imbalance
    for (;;) {
        uint32_t item = 0;
        if (lane == 0) item = atomicAdd(work_counter, 1u);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const int q = (int)(item / (uint32_t)P.n_rp);
        const int rp = (int)(item - (uint32_t)q * (uint32_t)P.n_rp);
        if (rp != cur_rp) {
            // ---- query profile of this warp's read pair ------------------------------------
            cur_rp = rp;
            ra = P.rp_reads[2 * rp]; rb = P.rp_reads[2 * rp + 1];
            const int64_t offa = P.read_off[ra];
            const int ma = (int)(P.read_off[ra + 1] - offa);
            const int64_t offb = rb >= 0 ? P.read_off[rb] : 0;
            const int mb = rb >= 0 ? (int)(P.read_off[rb + 1] - offb) : 0;
            __syncwarp();
            for (int idx = lane; idx < GL * K; idx += 32) {
                const int tt = idx / K, r = idx - tt * K;
                const int row = tt * K + r;
                const int qa = row < ma ? (int)P.read_codes[offa + row] : -1;
                const int qb = row < mb ? (int)P.read_codes[offb + row] : -1;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int lo = qa < 0 ? (int)S_PAD : (qa == c ? P.match : P.mismatch);
                    const int hi = qb < 0 ? (int)S_PAD : (qb == c ? P.match : P.mismatch);
                    prof[c * G::CSTRIDE + tt * G::KS + r] = pack2(lo, hi);
                }
            }
            __syncwarp();
        }
        // this group's SEGMENT: a window [c0, c0 + n_g) of a reference (the whole reference unless it is
        // very long).  A segment owns the checkpoint blocks [skip, own_end) of its local step space; the
        // blocks before `skip` only warm up the window (every owned cell is further than the longest
        // possible alignment from the window's left edge, so it is exact), see make_segments().
        const int v = 4 * q + g;
        const bool has_ref = v < P.n_vrefs;
        const int ref = has_ref ? P.v_ref[v] : 0;
        const int c0 = has_ref ? P.v_c0[v] : 0;
        const int n_g = has_ref ? P.v_len[v] : 0;
        const int skip = has_ref ? P.v_skip[v] : 0;
        const int own_end = has_ref ? P.v_end[v] : 0;
        const int nmax = P.v_len[4 * q];                          // sorted descending
        const int nmin = (4 * q + 3 < P.n_vrefs) ? P.v_len[4 * q + 3] : 0;
        const uint32_t *wp = P.ref_words + (has_ref ? P.ref_word_off[ref] + (uint32_t)(c0 >> 4) : 0u);
        const int64_t blk0 = (int64_t)rp * P.blocks_per_rp + (has_ref ? P.ref_blk_off[ref] + c0 / CB : 0);
        const int my_steps = has_ref ? min(n_g + GL - 1, own_end * CB) : 0;   // steps whose blocks this group owns

        uint32_t H[K];
#pragma unroll
        for (int r = 0; r < K; ++r) H[r] = 0;
        uint32_t diag = 0, tmax = 0, gmax = 0, wprev = 0;

        const int nsteps = nmax + GL - 1;
        for (int s0 = 0; s0 < nsteps; s0 += 16) {
            const uint32_t wnew = (s0 < n_g) ? __ldg(wp + (s0 >> 4)) : 0u;
            // window of this lane's 16 codes for steps s0..s0+15: columns (0-based) s0-t ..
            const uint32_t win = __funnelshift_rc(wprev, wnew, 32 - 2 * t);
            wprev = wnew;
            const bool fast = (s0 >= GL - 1) && (s0 + 16 <= nmin);

            // SEAMS: the boundary row this lane receives at every step (matrix row t*K) is kept next to the block
            // checkpoint, so that the traceback can recompute ONE lane's tile (K rows x CB steps) without the lanes
            // above it.  Record of (block, lane) = checkpoint + seam in 32-byte pieces (swb_device.cuh): every piece is
            // written straight from registers, one 256-bit store per 8 steps, 256 contiguous bytes per group store.
            const bool own_chunk = (s0 < my_steps) && ((s0 >> 4) >= skip);
            uint32_t *seam = rec_lane<K>(P.rec, blk0 + (s0 >> 4), t) + G::CKP * REC_P;       // this block's seam pieces
            uint32_t tq[8] = {0, 0, 0, 0, 0, 0, 0, 0};

            if (fast) {
                // K >= 25: two rounds of 8 steps instead of 16 unrolled ones (49-62 KB of code stall on instruction fetch,
                // see swb_fill_bias.cu)
                constexpr int UNR = K < 25 ? 16 : 8;
#pragma unroll 1
                for (int uq = 0; uq < 16; uq += UNR) {
                    const uint32_t winq = win >> (2 * uq);
#pragma unroll
                    for (int uu = 0; uu < UNR; ++uu) {
                        const uint32_t top = __shfl_up_sync(0xffffffffu, H[K - 1], 1) & lmask;
                        const uint32_t c = (winq >> (2 * uu)) & 3u;
                        uint32_t sv[G::KP];
                        load_profile<G::KP>(prof + c * G::CSTRIDE + my_prof, sv);
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
                        tmax = colmax<K>(tmax, H);
                        tq[uu & 7] = top;
                        if ((uu & 7) == 7 && own_chunk)
                            stg256(seam + ((uq + uu) >> 3) * REC_P, tq[0], tq[1], tq[2], tq[3], tq[4], tq[5], tq[6], tq[7]);
                    }
                }
            } else {
#pragma unroll 1
                for (int uq = 0; uq < 16; uq += 8) {
#pragma unroll
                    for (int uu = 0; uu < 8; ++uu) {
                        const int u = uq + uu;
                        const int s = s0 + u;
                        const uint32_t top = __shfl_up_sync(0xffffffffu, H[K - 1], 1) & lmask;
                        const uint32_t c = (win >> (2 * u)) & 3u;
                        const bool valid = (s >= t) && (s < n_g + t);        // column j = s-t+1 in [1, n_g]
                        if (valid) {
                            uint32_t sv[G::KP];
                            load_profile<G::KP>(prof + c * G::CSTRIDE + my_prof, sv);
                            uint32_t nw = diag, nn = top;
#pragma unroll
                            for (int r = 0; r < K; ++r) {
                                const uint32_t x = viaddmax_relu(nw, sv[r], zero);
                                const uint32_t pre = viaddmax(H[r], g2, x);
                                nw = H[r];
                                H[r] = viaddmax(nn, g2, pre);
                                nn = H[r];
                            }
                            tmax = colmax<K>(tmax, H);
                        }
                        diag = top;
                        tq[uu] = top;
                        if (uu == 7 && own_chunk) stg256(seam + (uq >> 3) * REC_P, tq[0], tq[1], tq[2], tq[3], tq[4], tq[5], tq[6], tq[7]);
                    }
                }
            }

            // ---- end of a checkpoint block: tile max, the next block's checkpoint
            const int s_next = s0 + 16;
            {
                const int b = s_next / CB;                       // block that starts at s_next
                if (s_next - CB < my_steps && b - 1 >= skip) {    // block b-1 is owned by this group
                    P.tmx[(blk0 + b - 1) * GL + t] = tmax;
                    gmax = vmax2(gmax, tmax);
                }
                tmax = 0;
                if (s_next < my_steps && b >= skip)               // block b is owned by this group
                    store_checkpoint<K>(rec_lane<K>(P.rec, blk0 + b, t), H, diag);       // state before step s_next
            }
        }
        // last (partial) block
        {
            const int s_end = ((nsteps + 15) >> 4) << 4;          // first step not executed
            if ((s_end % CB) != 0) {
                const int b_last = s_end / CB;
                if (b_last * CB < my_steps && b_last >= skip) {
                    P.tmx[(blk0 + b_last) * GL + t] = tmax;
                    gmax = vmax2(gmax, tmax);
                }
            }
        }
        // ---- pair scores: maximum over the group's 8 lanes, both halves ---------------
        gmax = vmax2(gmax, __shfl_xor_sync(0xffffffffu, gmax, 1));
        gmax = vmax2(gmax, __shfl_xor_sync(0xffffffffu, gmax, 2));
        gmax = vmax2(gmax, __shfl_xor_sync(0xffffffffu, gmax, 4));
        if (t == 0 && has_ref) {
            const int64_t ro = P.ref_orig[ref];
            // several segments of one reference may contribute: scores are zero-initialised
            atomicMax(P.scores + ro * P.n_reads + ra, (int)(int16_t)(gmax & 0xffffu));
            if (rb >= 0) atomicMax(P.scores + ro * P.n_reads + rb, (int)(int16_t)(gmax >> 16));
        }
    }
}

template <int K>
static cudaError_t launch_fill_k(const BatchParams &P, uint32_t *work_counter, int sm_count, cudaStream_t st)
{
    using G = Geo<K>;
    const int n_quads = (P.n_vrefs + 3) / 4;
    const int warps = 12;
    const int64_t items = (int64_t)n_quads * P.n_rp;
    // persistent CTAs, never more than there is work; one CTA per SM: measured 54 ms vs 69 ms for two (warp starvation)
    const int64_t ctas = std::min<int64_t>((items + warps - 1) / warps, (int64_t)sm_count);
    const size_t smem = (size_t)warps * G::PROF_WORDS * sizeof(uint32_t);
    cudaError_t e = cudaSuccess;
    {
        // ask for the largest shared-memory carve-out: the traceback CTAs of the previous batch (68 KB of
        // shared memory each) must be able to co-reside with this kernel's CTA on the same SM
        static PerDeviceOnce carve;
        e = carve.run([] { return cudaFuncSetAttribute(fill_kernel<K>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); });
        if (e != cudaSuccess) return e;
    }
    if (smem > 48 * 1024) {
        e = cudaFuncSetAttribute(fill_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    e = cudaMemsetAsync(work_counter, 0, sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    fill_kernel<K><<<dim3((unsigned)ctas), dim3(warps * 32), smem, st>>>(P, work_counter, 0u);
    return cudaGetLastError();
}

cudaError_t launch_fill(int K, const BatchParams &P, uint32_t *work_counter, int sm_count, cudaStream_t st)
{
    switch (K) {
        case 4:  return launch_fill_k<4>(P, work_counter, sm_count, st);
        case 5:  return launch_fill_k<5>(P, work_counter, sm_count, st);
        case 7:  return launch_fill_k<7>(P, work_counter, sm_count, st);
        case 10: return launch_fill_k<10>(P, work_counter, sm_count, st);
        case 8:  return launch_fill_k<8>(P, work_counter, sm_count, st);
        case 13: return launch_fill_k<13>(P, work_counter, sm_count, st);
        case 16: return launch_fill_k<16>(P, work_counter, sm_count, st);
        case 19: return launch_fill_k<19>(P, work_counter, sm_count, st);
        case 25: return launch_fill_k<25>(P, work_counter, sm_count, st);
        case 32: return launch_fill_k<32>(P, work_counter, sm_count, st);
    }
    return cudaErrorInvalidValue;
}

}  // namespace swb
