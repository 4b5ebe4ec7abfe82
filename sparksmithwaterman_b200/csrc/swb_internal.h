// swb_internal.h -- shared declarations of libswb200 (host structs, kernel launch API).
//
// Geometry of the short-read path (reads up to 8*32 = 256 rows; up to 511 rows with the LONG classes K = 40 .. 64)
//   * a GROUP of GL = 8 lanes owns one (read pair, reference) task; lane t owns the K
//     consecutive read rows t*K+1 .. t*K+K and marches along the reference columns,
//   * the 8 lanes form a skewed wavefront: at STEP s lane t computes column j = s - t + 1,
//     the boundary row travels to lane t+1 with one __shfl_up_sync per step,
//   * two reads are packed in the two s16 halves of every register (DPX s16x2 ops),
//   * per block of CB steps and lane the fill writes one RECORD to HBM: the CHECKPOINT (the lane's
//     K cells + the diagonal boundary at the block start) and the SEAM (the boundary row the
//     lane receives at each of the CB steps), plus the lane's tile maximum.  A record is all a
//     TILE (block, lane) = K rows x CB skewed columns needs to be recomputed on its own; the
//     locate / traceback kernels recompute only the tiles that hold maximum cells or that a
//     path crosses, so no direction plane is ever written.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/swb200.h"

namespace swb {

constexpr int GL = 8;        // lanes per group
constexpr int CB = 16;       // steps per checkpoint block (multiple of 16; the trace kernel's code window needs 16)
constexpr int MAX_SHORT_ROWS = GL * 32;       // every short-path kernel (incl. the fallbacks swb_fill.cu / swb_trace.cu)
static_assert(CB == 16, "the fill kernels store one seam quad per 4 steps of a 16-step chunk");

// rows-per-lane variants compiled for the short path
constexpr int kNumK = 14;
constexpr int kKList[kNumK] = {4, 5, 7, 8, 10, 13, 16, 19, 25, 32,    // 8 K >= m: 36/50/75-80/100/125/150/200/250 bp reads fit with <= 7 % padding
                               40, 48, 56, 64};                        // LONG classes: 257 .. 511 rows (the reference's read-length sweep
                                                                       // goes to 500 bp, EngineerData.java:87-104); biased fill + tile kernels only
constexpr int MAX_K_BASE = 32;                // largest K of the fallback kernels
constexpr int MAX_LONG_ROWS = 511;            // row index i has KEY_I_BITS = 9 bits in a max-cell key

template <int K> struct Geo {
    static constexpr int KW = ((K + 1 + 3) / 4) * 4;            // checkpoint words per lane (K cells + diag), padded to 16 bytes
    static constexpr int CKP = (K + 1 + 7) / 8;                 // checkpoint PIECES (32 bytes each) of a record
    static constexpr int RP = CKP + CB / 8;                     // pieces per (block, lane) record: checkpoint + seam
    static constexpr int RW = RP * 8;                           // record words
    static constexpr int KP = ((K + 3) / 4) * 4;                // profile words per lane per code
    static constexpr int KS = ((KP / 4) % 2 == 1) ? KP : KP + 4; // padded: odd number of 16B units -> conflict-free LDS.128
    static constexpr int CSTRIDE = GL * KS;                     // words per reference code
    static constexpr int PROF_WORDS = 4 * CSTRIDE;
    static constexpr int RS = ((K + 1 + 1) / 2) * 2;            // traceback tile row stride (halfwords)
    static constexpr int TILE_HALFWORDS = GL * (CB + 1) * RS;   // per group
};

constexpr int16_t S_PAD = -16384;   // profile score of a padding row (beyond the read's end)

// key of one maximum cell: pair key = read slot * n_refs + ref (33 bits) | i (9 bits) | j (22 bits);
// sorting the keys gives, per (read, ref) pair, the reference's row-major max-cell order
constexpr int KEY_J_BITS = 22, KEY_I_BITS = 9;
__host__ __device__ inline uint64_t make_key(uint64_t p, uint32_t i, uint32_t j)
{ return (p << (KEY_J_BITS + KEY_I_BITS)) | ((uint64_t)i << KEY_J_BITS) | j; }
__host__ __device__ inline uint64_t key_pair(uint64_t k) { return k >> (KEY_J_BITS + KEY_I_BITS); }
__host__ __device__ inline uint32_t key_i(uint64_t k) { return (uint32_t)(k >> KEY_J_BITS) & ((1u << KEY_I_BITS) - 1); }
__host__ __device__ inline uint32_t key_j(uint64_t k) { return (uint32_t)k & ((1u << KEY_J_BITS) - 1); }

// cudaFuncSetAttribute is per device (context): a process may hold one swb_ctx per GPU (Spark local[N] over 8 GPUs
// in one JVM), so "already set" is tracked per device.  need() is true the first time it is called on the current device.
struct PerDeviceOnce {
    std::mutex mu;
    bool done[64] = {};
    // runs f() once per device, under a lock, and only records success: two contexts on one device (Spark local[N]
    // threads of one JVM) can no longer skip an attribute that has not been set yet
    template <class F> cudaError_t run(F &&f)
    {
        int d = 0;
        if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return f();
        std::lock_guard<std::mutex> lk(mu);
        if (done[d]) return cudaSuccess;
        const cudaError_t e = f();
        if (e == cudaSuccess) done[d] = true;
        return e;
    }
};

struct TileTask { uint32_t rp_half; uint32_t ref_sorted; uint32_t block; uint32_t lane; };   // one flagged tile

// Everything the short-path kernels need for one batch of read pairs of one K class.
struct BatchParams {
    // reference set (sorted by descending length)
    const uint32_t *ref_words;      // 2-bit codes, 16 per word
    const uint32_t *ref_word_off;   // [n_refs] first word of sorted ref
    const int32_t  *ref_len;        // [n_refs]
    const int32_t  *ref_orig;       // [n_refs] sorted -> original index
    const int32_t  *ref_sorted_of;  // [n_refs] original -> sorted index
    const int64_t  *ref_blk_off;    // [n_refs+1] prefix of checkpoint blocks per sorted ref
    int32_t n_refs;
    int64_t blocks_per_rp;          // ref_blk_off[n_refs]
    // fill work units: segments of references, sorted by descending length (see make_segments)
    const int32_t *v_ref, *v_c0, *v_len, *v_skip, *v_end;
    int32_t n_vrefs;
    // reads
    const uint8_t *read_codes;      // 1 byte per base: 0..3, 0xFF = matches nothing
    const int64_t *read_off;        // [n_reads+1]
    const int32_t *rp_reads;        // [n_rp][2] read indices of the batch's pairs (-1 = none)
    const int32_t *read_slot;       // [n_reads] rp_local*2+half for reads of this batch, else -1
    int32_t n_rp;
    int64_t n_reads;                // reads in the whole call (pair index stride)
    // scores
    int32_t match, mismatch, gap;
    int32_t tie_gt;                 // traceback tie rule: 0 = '>=' cascade (a > i > d), 1 = strict '>' (d > i > a)
    // outputs / workspace
    int32_t  *scores;               // [n_refs_orig * n_reads]
    // block records [n_rp][blocks_per_rp][RP pieces][GL lanes][8 words]: per lane the CHECKPOINT at the block start
    // (K cells + diagonal boundary, unbiased) and the SEAM of the block (the boundary row the lane receives at each
    // of its CB steps) -- everything a traceback needs to recompute the tile (block, lane) -- in 32-byte pieces;
    // piece p of a block's eight lanes is contiguous (swb_device.cuh).
    uint32_t *rec;
    uint32_t *tmx;                  // tile maxima  [n_rp][blocks_per_rp][GL]
    int32_t tmx_slack;              // 0: tile maxima / pair scores of the fill are exact; > 0: subsampled, true max - slack <= tmx <= true max
    int32_t seam_bias;              // seam word of step u, lane t = H + seam_bias * (9 - t + u) (biased fill), 0 = plain
    const uint32_t *sel;            // hits mode: bit rp_half * n_refs + ref_orig = the pair is selected, only those emit
                                    // max cells; nullptr = every pair emits
};

// ---- general ("wide") int32 path: bands of 32 lanes x KL rows, see swb_wide.cu ------------------
namespace wide {
constexpr int WL = 32;       // lanes per band (one warp)
constexpr int WCB = 32;      // steps per checkpoint block
constexpr int kNumKL = 3;
constexpr int kKLList[kNumKL] = {8, 16, 32};                  // rows per lane (band height 256 / 512 / 1024)
template <int KL> struct WGeo {
    static constexpr int BH = WL * KL;                        // rows per band
    static constexpr int KW = ((KL + 1 + 3) / 4) * 4;         // checkpoint words per lane (KL cells + diag)
    static constexpr int RW = KW + WCB;                       // record words per (band, block, lane): checkpoint + seam
};
constexpr int wide_rw(int kl) { return ((kl + 1 + 3) / 4) * 4 + WCB; }
// key: local pair (21 bits) | i (21 bits) | j (22 bits)
__host__ __device__ inline uint64_t wide_key(uint64_t pair, uint32_t i, uint32_t j) { return (pair << 43) | ((uint64_t)i << 22) | j; }
__host__ __device__ inline uint64_t wide_key_pair(uint64_t k) { return k >> 43; }
__host__ __device__ inline uint32_t wide_key_i(uint64_t k) { return (uint32_t)(k >> 22) & ((1u << 21) - 1); }
__host__ __device__ inline uint32_t wide_key_j(uint64_t k) { return (uint32_t)k & ((1u << 22) - 1); }
}  // namespace wide

struct WideTask { int32_t pair, band, block; uint32_t lane; };   // one flagged tile

struct WideParams {
    int32_t n_pairs;
    const int32_t *pair_ref;     // [n_pairs] reference index (original order)
    const int32_t *pair_read;    // [n_pairs] read index
    const uint8_t *ref_codes;    // 1 byte per base, original reference order
    const int64_t *ref_off;      // [n_refs + 1]
    const uint8_t *rpad;         // read codes, each wide read 16-byte aligned and padded with 0xFE to a multiple of 1024 rows
    const int64_t *rpad_off;     // [n_reads] offset of the read in rpad (reads of this call that take the wide path)
    const int64_t *read_off;     // [n_reads + 1] offsets in the unpadded read codes (lengths)
    int32_t match, mismatch, gap;
    int32_t tie_gt;
    int32_t n_symbols;           // alphabet size of the reference set (codes 0 .. n_symbols-1)
    int64_t n_reads;
    const int64_t *band_off;     // [n_pairs + 1] prefix of bands
    const int64_t *blk_off;      // [n_pairs + 1] prefix of bands * blocks
    const int64_t *brow_off;     // [n_pairs + 1] prefix of bands * blocks * 32 (steps)
    int32_t *brow;               // per band: lane 31's bottom row, indexed by step; -1 = not written yet (host memset)
    int32_t *rec;                // block records [bands * blocks][32 lanes][RW]
    int32_t *tmx;                // tile maxima   [bands * blocks][32 lanes]
    int32_t *scores;
    int32_t *mail;               // pipelined CTA-wide traceback: tokens [cells][mail_stride][8] (zeroed by the host), nullptr = mode off
    int32_t *mail_latest;        // [cells] highest token index published
    int32_t mail_stride;         // tokens per cell = rounds + 2
    int32_t pipe_c;              // CTAs per cell (cluster size), set by the launcher
};

// one batch of max cells as the assembly kernels see it (swb_assemble.cu)
struct BatchDesc {
    const uint64_t *keys; const int32_t *beg; const int32_t *oplen; const uint32_t *ops;
    const int32_t *slot_read;   // short path: read slot -> read index
    const int64_t *pair_map;    // wide path: local pair -> ABI pair index
    int64_t ops_stride;
    uint32_t base;              // index of the batch's first cell in the concatenation
    uint32_t n_cells;
    int32_t wide;
};
size_t      assemble_tmp_bytes(uint32_t n_cells);
// keep (nullable): hits mode, bit p of the ABI pairs whose cells stay; the others sort after them as p + n_pairs
cudaError_t assemble_sort(const BatchDesc *batches, int nb, uint32_t n_cells, int64_t n_refs, int64_t n_reads,
                          const uint32_t *keep, uint64_t *pair_tmp, uint32_t *src_tmp, uint64_t *pair_sorted, uint32_t *order, void *tmp,
                          size_t tmp_bytes, int pair_bits, cudaStream_t st);
cudaError_t assemble_gather_cells(const BatchDesc *batches, int nb, uint32_t n_cells, const uint32_t *order, int32_t *cells,
                                  int32_t *beginnings, int32_t *op_lens, int64_t *words, int64_t *ops_off, void *tmp,
                                  size_t tmp_bytes, cudaStream_t st);
cudaError_t assemble_gather_ops(const BatchDesc *batches, int nb, uint32_t n_cells, const uint32_t *order,
                                const int64_t *ops_off, uint32_t *ops_out, cudaStream_t st);
cudaError_t assemble_offsets(const uint64_t *pair_sorted, uint32_t n_cells, int64_t n_pairs, int64_t *cell_off,
                             int32_t *best, int64_t n_reads, const int32_t *cells, cudaStream_t st);

// hits mode: *n_kept = cells of kept pairs (a device word); hits[q][h] (i, j) and the (i, j) of best hits below min_score
cudaError_t assemble_kept_count(const uint64_t *pair_sorted, uint32_t n_cells, int64_t n_pairs, uint32_t *n_kept, cudaStream_t st);
cudaError_t assemble_hit_cells(const BatchDesc *batches, int nb, const uint64_t *pair_sorted, const uint32_t *order, uint32_t n_all,
                               int64_t n_pairs, int64_t n_reads, const int64_t *cell_off, const int32_t *cells, int32_t *best,
                               int32_t *hits, int k, cudaStream_t st);
// all-hits mode: (i, j) of every list entry = its pair's first kept cell
cudaError_t assemble_list_cells(const int64_t *hit_off, int64_t n_reads, int32_t *list, int64_t n_hits, const int64_t *cell_off,
                                const int32_t *cells, cudaStream_t st);

// swb_hits.cu: per-read top k (score desc, ref asc) of scores[ref * n_reads + q] over q = slots[s] (slots null: q = s,
// slot -1: skipped), written to hits[s * k ..] / bits as hits_merge_kernel describes.
size_t      select_hits_tmp_elems(int64_t n_refs, int64_t n_slots, int k);
cudaError_t launch_select_hits(const int32_t *scores, int64_t n_refs, int64_t n_reads, const int32_t *slots, int64_t n_slots,
                               int k, int32_t min_score, int with_best, int4 *hits, uint32_t *bits, int64_t bit_slot,
                               int64_t bit_ref, bool oriented_bits, uint64_t *tmp, size_t tmp_elems, cudaStream_t st);
// all-hits mode: best[s] = key of read slots[s]'s best pair ((score << 32) | ~ref, 0 = none); bits (nullable) as
// hits_merge_kernel for every pair with score >= max(min_score, best - margin), plus the best pair if with_best
cudaError_t launch_select_margin(const int32_t *scores, int64_t n_refs, int64_t n_reads, const int32_t *slots, int64_t n_slots,
                                 int32_t min_score, int32_t margin, int with_best, uint32_t *bits, int64_t bit_slot, int64_t bit_ref,
                                 bool oriented_bits, uint64_t *best, cudaStream_t st);
// the final lists over all reads (best from launch_select_margin with slots null): count[n_reads * chunks + 1] -> off
// (exclusive scan; off[last] = n_hits), then list[n_hits] (score, ref, 0, 0) by read, score descending, reference
// ascending, and hit_off[n_reads + 1]
size_t      margin_list_tmp_bytes(int64_t n_refs, int64_t n_reads, int64_t n_hits);
size_t      margin_count_elems(int64_t n_refs, int64_t n_reads);
cudaError_t launch_margin_count(const int32_t *scores, int64_t n_refs, int64_t n_reads, int32_t min_score, int32_t margin,
                                const uint64_t *best, int64_t *count, int64_t *off, void *tmp, size_t tmp_bytes, cudaStream_t st);
cudaError_t launch_margin_write(const int32_t *scores, int64_t n_refs, int64_t n_reads, int32_t min_score, int32_t margin,
                                const uint64_t *best, const int64_t *off, int64_t n_hits, int4 *list_tmp, uint64_t *keys_tmp,
                                uint64_t *keys_sorted, uint32_t *idx_tmp, uint32_t *order, int4 *list, int64_t *hit_off, void *tmp,
                                size_t tmp_bytes, cudaStream_t st);

cudaError_t launch_wide_pad_reads(const uint8_t *codes, const int64_t *read_off, const int32_t *reads, int n_reads,
                                  const int64_t *rpad_off, const int64_t *rpad_len, uint8_t *rpad, int64_t max_len,
                                  cudaStream_t st);
cudaError_t launch_wide_fill(int KL, const WideParams &P, const int2 *items, int n_items, uint32_t *ticket, int sm_count,
                             cudaStream_t st);
cudaError_t launch_wide_flag(const WideParams &P, int64_t total_blocks, WideTask *tasks, uint32_t cap, uint32_t *count,
                             int sm_count, cudaStream_t st);
cudaError_t launch_wide_locate(int KL, const WideParams &P, const WideTask *tasks, const uint32_t *n_tasks, uint32_t cap_tasks,
                               uint64_t *keys, uint32_t cap, uint32_t *count, int sm_count, cudaStream_t st);
cudaError_t launch_wide_trace(int KL, const WideParams &P, const uint64_t *keys, uint32_t n_cells, int32_t *beginnings,
                              int32_t *op_lens, uint32_t *ops, int64_t ops_stride, int sm_count, cudaStream_t st);

// swb_fill.cu
cudaError_t launch_fill(int K, const BatchParams &P, uint32_t *work_counter, int sm_count, cudaStream_t st);
// swb_fill_bias.cu: same contract, horizontal gap folded into a column bias (2.5 instead of 3.5 ALU ops / cell pair)
cudaError_t launch_fill_bias(int K, const BatchParams &P, uint32_t *work_counter, int sm_count, cudaStream_t st);
bool fill_bias_ok(int match, int mismatch, int gap, int64_t max_score);
int fill_sub_slack(int match, int mismatch, int gap);
// swb_trace.cu
cudaError_t launch_flag_tiles(const BatchParams &P, TileTask *tasks, uint32_t cap, uint32_t *count, int sm_count, cudaStream_t st);
cudaError_t launch_locate(int K, const BatchParams &P, const TileTask *tasks, const uint32_t *n_tasks,
                          uint32_t cap_tasks, void *hits, uint64_t *keys, uint32_t cap, uint32_t *count, int sm_count,
                          int phase, cudaStream_t st);
size_t      locate_hit_bytes();
cudaError_t launch_trace(int K, const BatchParams &P, const uint64_t *keys, uint32_t n_cells,
                         int32_t *beginnings, int32_t *op_lens, uint32_t *ops, int ops_stride_words,
                         int sm_count, cudaStream_t st);
// swb_trace_tile.cu: one thread per max cell, single-lane tiles from checkpoint + seam (default when the scores allow)
cudaError_t launch_tile_trace(int K, const BatchParams &P, const uint64_t *keys, uint32_t n_cells,
                              int32_t *beginnings, int32_t *op_lens, uint32_t *ops, int ops_stride_words,
                              int sm_count, cudaStream_t st);
bool tile_trace_ok(int match, int mismatch, int gap);
cudaError_t launch_ref_totals(const int32_t *scores, int64_t n_refs, int64_t n_reads, int32_t *totals, cudaStream_t st);
cudaError_t launch_best_hits(const int32_t *scores, int64_t n_refs, int64_t n_reads, int32_t *best, int sm_count, cudaStream_t st);
cudaError_t sort_keys(uint64_t *keys_in, uint64_t *keys_out, uint32_t n, void *tmp, size_t tmp_bytes, cudaStream_t st);
size_t      sort_keys_tmp_bytes(uint32_t n);

}  // namespace swb
