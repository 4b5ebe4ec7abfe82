// swb_fill_bias.cu -- the fill kernel with the horizontal gap folded into a column bias.
//
// Same job, geometry, scheduling, outputs and checkpoint format as swb_fill.cu, but every register
// holds  H''(i,j) = H(i,j) + |gap| * (j - jref)  instead of H.  With that bias
//     W + gap      ->  W''                       (the bias of column j-1 plus |gap| IS the bias of column j)
//     N + gap      ->  N'' + gap                 (same column)
//     NW + s       ->  NW'' + (s + |gap|)        (non-negative addend)
//     0            ->  floor_j = |gap| * (j - jref)
// so the cell costs ONE packed add with a non-negative addend -- done as IMAD on the FMA pipe, which
// runs beside the ALU/DPX pipe (profiles/dpx_microbench_r01.json: VIADDMNMX + IMAD = 3.4 warp-instr/
// clk/SM vs 2.0 for the ALU pipe alone) -- plus two ALU ops:
//     t   = IMAD(NW'', 1, s'')              FMA pipe; carry-free: both halves are non-negative and small
//     pre = VIMNMX3(t, W'', floor_j)        ALU
//     H'' = VIADDMNMX(N'', gap, pre)        ALU, the only op on the row-to-row dependency chain
// i.e. 2.5 ALU ops per cell pair (with the half VIMNMX3 of the tile maximum) instead of 3.5.
// jref advances by CB at every checkpoint block (all registers -= CB*|gap|), so the bias stays in
// [|gap|, 24*|gap|]; tile maxima and checkpoints are stored UNBIASED, the traceback kernels are unchanged.
// Domain (checked by the host, else swb_fill.cu runs): gap < 0, match + |gap| >= 0, mismatch + |gap| >= 0,
// max score + 32*|gap| within s16.  Padding rows score s = gap on the diagonal (s'' = 0): every padded
// cell is then an earlier cell minus |gap|, i.e. strictly below the true maximum, as before.
// Recurrence: reference SmithWaterman.java:217-252 (GetCellScore.call), :277-280, :309-318.
#include "swb_internal.h"
#include "swb_device.cuh"

#include <algorithm>
#include <cstdlib>

namespace swb {

__device__ __forceinline__ uint32_t imad_add(uint32_t a, uint32_t one, uint32_t b)
{
    // a * 1 + b with `one` opaque to ptxas: stays an IMAD (FMA pipe) instead of becoming IADD3 (ALU pipe)
    return a * one + b;
}

// one column of a lane: K cells.  K <= 32: the lane's KP profile words are loaded up front (5 LDS.128 for K = 19);
// the LONG classes (K = 40 .. 64) load them a quad at a time inside the row loop -- K score registers plus K profile
// registers would not fit the 128-register budget of a 16-warp CTA.
template <int K>
__device__ __forceinline__ void fill_column(uint32_t (&H)[K], const uint32_t *pcol, uint32_t diag, uint32_t top,
                                            uint32_t floorv, uint32_t g2, uint32_t one)
{
    using G = Geo<K>;
    uint32_t nw = diag, nn = top;
    if constexpr (K <= MAX_K_BASE) {
        uint32_t sv[G::KP];
        load_profile<G::KP>(pcol, sv);
#pragma unroll
        for (int r = 0; r < K; ++r) {
            const uint32_t tt = imad_add(nw, one, sv[r]);       // NW'' + s''          (FMA pipe)
            const uint32_t pre = vmax3(tt, H[r], floorv);       // max(t, W'', floor)  (ALU)
            nw = H[r];
            H[r] = viaddmax(nn, g2, pre);                       // max(N'' + gap, pre) (ALU)
            nn = H[r];
        }
    } else {
        const uint4 *p4 = reinterpret_cast<const uint4 *>(pcol);
#pragma unroll
        for (int q = 0; q < G::KP / 4; ++q) {
            const uint4 v = p4[q];
            const uint32_t sv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int x = 0; x < 4; ++x) {
                const int r = 4 * q + x;
                if (r < K) {
                    const uint32_t tt = imad_add(nw, one, sv[x]);
                    const uint32_t pre = vmax3(tt, H[r < K ? r : 0], floorv);
                    nw = H[r < K ? r : 0];
                    H[r < K ? r : 0] = viaddmax(nn, g2, pre);
                    nn = H[r < K ? r : 0];
                }
            }
        }
    }
}

// from this K on the 16 steps of a block run as two rounds of 8 (code size, see the fast path)
constexpr int FILL_ROLL_K = 25;
constexpr int fill_bias_threads(int K) { return K <= MAX_K_BASE ? 512 : (K <= 48 ? 384 : 256); }

// SUB: the tile maximum (and with it the pair score the fill leaves) is taken over a SUBSAMPLE of the cells --
// even rows + the lane's last row, on the odd steps of a block (CB is even: the last step is odd) -- which costs
// 3.0 instead of 10.5 DPX ops per step.  Every cell (r, u) of a tile has a tracked cell of the SAME tile among (r, u), (r+1, u),
// (r, u+1), (r+1, u+1), so the tracked maximum M of a tile satisfies  true max - slack <= M <= true max  with
// slack = max(|gap|, min(|mismatch|, 2|gap|)) (fill_sub_slack).  The locate stage recomputes every tile within
// slack of the pair's tracked maximum, makes the pair score exact and enumerates the exact maximum cells.
template <int K, bool SUB>
__global__ void __launch_bounds__(fill_bias_threads(K)) fill_bias_kernel(const BatchParams P, uint32_t *work_counter, uint32_t one)
{
    using G = Geo<K>;
    extern __shared__ __align__(16) uint32_t prof_all[];        // per warp: [4 codes][GL lanes][KS], entries s + |gap|

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t = lane & (GL - 1), g = lane >> 3;
    uint32_t *prof = prof_all + warp * G::PROF_WORDS;
    const int n_quads = (P.n_vrefs + 3) >> 2;
    const uint32_t n_items = (uint32_t)n_quads * (uint32_t)P.n_rp;

    const int ag = -P.gap;                                        // |gap| > 0
    const uint32_t g2 = pack2(P.gap, P.gap);
    const uint32_t gpos = pack2(ag, ag);
    const uint32_t base_bias = pack2(ag * (8 - t), ag * (8 - t)); // bias of this lane's stored column at a block start
    const uint32_t renorm = (uint32_t)(-(int32_t)(pack2(ag * CB, ag * CB)));   // 32-bit add of -(CB*|gap|) in both halves (no borrow: bias >= CB*|gap| there)
    const uint32_t unbias = (uint32_t)(-(int32_t)base_bias);      // for 32-bit IMAD subtraction (no borrow across halves)
    const uint32_t negbase = pack2(-ag * (8 - t), -ag * (8 - t)); // per-half negation, for the packed s16x2 ops
    // negfloor += gap in both halves as ONE 32-bit IMAD (FMA pipe) instead of a VIADD.16x2 (ALU pipe, DPX rate): both
    // halves stay negative, so the low half's add always carries into the high half -- take that carry out of the addend
    const uint32_t g2c = g2 - 0x10000u, g2c2 = 2u * g2c;
    static_assert((CB & 1) == 0, "the subsampled tile maximum tracks the odd steps of a block");
    const int my_prof = t * G::KS;
    int cur_rp = -1, ra = 0, rb = -1;

    for (;;) {
        uint32_t item = 0;
        if (lane == 0) item = atomicAdd(work_counter, 1u);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const int q = (int)(item / (uint32_t)P.n_rp);
        const int rp = (int)(item - (uint32_t)q * (uint32_t)P.n_rp);
        if (rp != cur_rp) {
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
                    const int lo = qa < 0 ? 0 : (qa == c ? P.match : P.mismatch) + ag;
                    const int hi = qb < 0 ? 0 : (qb == c ? P.match : P.mismatch) + ag;
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

        // all-zero matrix left of column 1, biased: every register = the floor of its column
        uint32_t H[K];
#pragma unroll
        for (int r = 0; r < K; ++r) H[r] = base_bias;
        uint32_t diag = base_bias, floorv = base_bias, negfloor = negbase;
        uint32_t tmax = 0, gmax = 0, wprev = 0;

        const int nsteps = nmax + GL - 1;
        for (int s0 = 0; s0 < nsteps; s0 += 16) {
            const uint32_t wnew = (s0 < n_g) ? __ldg(wp + (s0 >> 4)) : 0u;
            const uint32_t win = __funnelshift_rc(wprev, wnew, 32 - 2 * t);
            wprev = wnew;
            const bool fast = (s0 >= GL - 1) && (s0 + 16 <= nmin);

            // SEAMS (see swb_fill.cu): the boundary row this lane receives at every step, written straight to the
            // block's record (one 256-bit store per 8 steps), BIASED -- the
            // bias of step u of a block is |gap| * (9 - t + u) in both halves (P.seam_bias tells the traceback).
            const bool own_chunk = (s0 < my_steps) && ((s0 >> 4) >= skip);
            uint32_t *seam = rec_lane<K>(P.rec, blk0 + (s0 >> 4), t) + G::CKP * REC_P;       // this block's seam pieces
            uint32_t tq[8] = {0, 0, 0, 0, 0, 0, 0, 0};

            if (fast) {
                // K <= 19: all 16 steps unrolled (<= 20 KB of code).  Larger classes stall on instruction fetch when fully
                // unrolled (ncu, K = 64, 56 KB: no_instruction 1.1 warps per issue; K = 32, 31 KB: 250 bp batches 5 % slower):
                // two rounds of 8 steps there.  Rolling K = 19 as well costs 2 % (35.3 -> 35.9 ms; with the 90 registers
                // it then needs, 20 warps per CTA: 36.1 ms).
                constexpr int UNR = K < FILL_ROLL_K ? 16 : 8;
#pragma unroll 1
                for (int uq = 0; uq < 16; uq += UNR) {
                    const uint32_t winq = win >> (2 * uq);
#pragma unroll
                    for (int uu = 0; uu < UNR; ++uu) {
                        floorv = imad_add(floorv, one, gpos);                  // floor of the new column
                        if (!SUB) negfloor = imad_add(negfloor, one, g2c);      // its negative (packed; see g2c)
                        uint32_t top = __shfl_up_sync(0xffffffffu, H[K - 1], 1);
                        if (t == 0) top = floorv;                               // row 0 is all zero
                        const uint32_t c = (winq >> (2 * uu)) & 3u;
                        fill_column<K>(H, prof + c * G::CSTRIDE + my_prof, diag, top, floorv, g2, one);
                        diag = top;
                        if (!SUB) tmax = viaddmax(colmax<K>(floorv, H), negfloor, tmax);  // unbiased running maximum
                        else if (uu & 1) {                                      // odd steps: CB and UNR are even, the last step is one
                            negfloor = imad_add(negfloor, one, g2c2);           // two columns on
                            tmax = viaddmax(colmax_even<K>(floorv, H), negfloor, tmax);
                        }
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
                        floorv = imad_add(floorv, one, gpos);
                        negfloor = imad_add(negfloor, one, g2c);
                        uint32_t top = __shfl_up_sync(0xffffffffu, H[K - 1], 1);
                        if (t == 0) top = floorv;
                        const uint32_t c = (win >> (2 * u)) & 3u;
                        const bool valid = (s >= t) && (s < n_g + t);
                        if (valid) {
                            fill_column<K>(H, prof + c * G::CSTRIDE + my_prof, diag, top, floorv, g2, one);
                            tmax = viaddmax(colmax<K>(floorv, H), negfloor, tmax);
                        } else {
                            // outside the matrix: the column is all zero (left of it) or never read (right of it)
#pragma unroll
                            for (int r = 0; r < K; ++r) H[r] = floorv;
                        }
                        diag = top;
                        tq[uu] = top;
                        if (uu == 7 && own_chunk) stg256(seam + (uq >> 3) * REC_P, tq[0], tq[1], tq[2], tq[3], tq[4], tq[5], tq[6], tq[7]);
                    }
                }
            }

            // ---- block boundary: move jref by CB columns, then (un-biased) tile max + the next block's checkpoint
            const int s_next = s0 + 16;
            {
#pragma unroll
                for (int r = 0; r < K; ++r) H[r] = imad_add(H[r], one, renorm);
                diag = imad_add(diag, one, renorm);
                floorv = base_bias;
                negfloor = negbase;
                const int b = s_next / CB;
                if (s_next - CB < my_steps && b - 1 >= skip) {
                    P.tmx[(blk0 + b - 1) * GL + t] = tmax;
                    gmax = vmax2(gmax, tmax);
                }
                tmax = 0;
                if constexpr (K <= MAX_K_BASE) {
                    uint32_t U[K];
#pragma unroll
                    for (int r = 0; r < K; ++r) U[r] = imad_add(H[r], one, unbias);     // H'' - bias >= 0: no borrow
                    if (s_next < my_steps && b >= skip)                                 // block b is owned by this group
                        store_checkpoint<K>(rec_lane<K>(P.rec, blk0 + b, t), U, imad_add(diag, one, unbias));
                } else if (s_next < my_steps && b >= skip) {
                    // LONG classes: un-bias piece by piece (no second copy of the K score registers)
                    uint32_t *lane_rec = rec_lane<K>(P.rec, blk0 + b, t);
#pragma unroll
                    for (int p = 0; p < G::CKP; ++p) {
                        uint32_t v[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const int w = 8 * p + e;
                            v[e] = (w < K) ? imad_add(H[w < K ? w : 0], one, unbias) : (w == K ? imad_add(diag, one, unbias) : 0u);
                        }
                        stg256(lane_rec + p * REC_P, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]);
                    }
                }
            }
        }
        {
            const int s_end = ((nsteps + 15) >> 4) << 4;
            if ((s_end % CB) != 0) {
                const int b_last = s_end / CB;
                if (b_last * CB < my_steps && b_last >= skip) {
                    P.tmx[(blk0 + b_last) * GL + t] = tmax;
                    gmax = vmax2(gmax, tmax);
                }
            }
        }
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

template <int K, bool SUB>
static cudaError_t launch_fill_bias_k2(const BatchParams &P, uint32_t *work_counter, int sm_count, cudaStream_t st)
{
    using G = Geo<K>;
    const int n_quads = (P.n_vrefs + 3) / 4;
    const int max_warps = fill_bias_threads(K) / 32;
    const int warps = std::min(16, max_warps);   // measured (K = 19): 10/12/14/16 warps -> 42.0/39.8/39.4/39.2 ms
    const int64_t items = (int64_t)n_quads * P.n_rp;
    const int64_t ctas = std::min<int64_t>((items + warps - 1) / warps, (int64_t)sm_count);   // one CTA per SM
    const size_t smem = (size_t)warps * G::PROF_WORDS * sizeof(uint32_t);
    cudaError_t e = cudaSuccess;
    {
        // ask for the largest shared-memory carve-out: the traceback CTAs of the previous batch (68 KB of
        // shared memory each) must be able to co-reside with this kernel's CTA on the same SM
        static PerDeviceOnce carve;
        e = carve.run([] { return cudaFuncSetAttribute(fill_bias_kernel<K, SUB>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); });
        if (e != cudaSuccess) return e;
    }
    if (smem > 48 * 1024) {
        e = cudaFuncSetAttribute(fill_bias_kernel<K, SUB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    e = cudaMemsetAsync(work_counter, 0, sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    fill_bias_kernel<K, SUB><<<dim3((unsigned)ctas), dim3(warps * 32), smem, st>>>(P, work_counter, 1u);
    return cudaGetLastError();
}

template <int K>
static cudaError_t launch_fill_bias_k(const BatchParams &P, uint32_t *work_counter, int sm_count, cudaStream_t st)
{
    return P.tmx_slack > 0 ? launch_fill_bias_k2<K, true>(P, work_counter, sm_count, st)
                           : launch_fill_bias_k2<K, false>(P, work_counter, sm_count, st);
}

cudaError_t launch_fill_bias(int K, const BatchParams &P, uint32_t *work_counter, int sm_count, cudaStream_t st)
{
    switch (K) {
        case 4:  return launch_fill_bias_k<4>(P, work_counter, sm_count, st);
        case 5:  return launch_fill_bias_k<5>(P, work_counter, sm_count, st);
        case 7:  return launch_fill_bias_k<7>(P, work_counter, sm_count, st);
        case 10: return launch_fill_bias_k<10>(P, work_counter, sm_count, st);
        case 8:  return launch_fill_bias_k<8>(P, work_counter, sm_count, st);
        case 13: return launch_fill_bias_k<13>(P, work_counter, sm_count, st);
        case 16: return launch_fill_bias_k<16>(P, work_counter, sm_count, st);
        case 19: return launch_fill_bias_k<19>(P, work_counter, sm_count, st);
        case 25: return launch_fill_bias_k<25>(P, work_counter, sm_count, st);
        case 32: return launch_fill_bias_k<32>(P, work_counter, sm_count, st);
        case 40: return launch_fill_bias_k<40>(P, work_counter, sm_count, st);
        case 48: return launch_fill_bias_k<48>(P, work_counter, sm_count, st);
        case 56: return launch_fill_bias_k<56>(P, work_counter, sm_count, st);
        case 64: return launch_fill_bias_k<64>(P, work_counter, sm_count, st);
    }
    return cudaErrorInvalidValue;
}

// host-side domain check of the biased kernel
// Slack of the subsampled tile maximum, or 0 when the subsample may not be used: a positive cell must not hide
// behind a tracked maximum of 0, i.e. one match has to exceed the slack (then score_lo == 0 implies score == 0).
int fill_sub_slack(int match, int mismatch, int gap)
{
    if (gap >= 0) return 0;
    const int ag = -gap;
    const int diag = mismatch >= 0 ? 0 : std::min(-mismatch, 2 * ag);   // (r+1, u+1) >= H + max(mismatch, 2 gap)
    const int slack = std::max(ag, diag);
    return (match > slack && slack < 4096) ? slack : 0;
}

bool fill_bias_ok(int match, int mismatch, int gap, int64_t max_score)
{
    if (gap >= 0) return false;
    const int ag = -gap;
    return match + ag >= 0 && mismatch + ag >= 0 && match + ag <= 4000 && mismatch + ag <= 4000 &&
           max_score + 32LL * ag <= 30000;
}

}  // namespace swb
