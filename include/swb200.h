/*
 * swb200.h -- C ABI of the B200-native Smith-Waterman engine (libswb200.so).
 *
 * This is the drop-in boundary for the reference's `sw` hot path.  Every entry
 * point is plain C (extern "C", pointers + fixed-width integers, no structs by
 * value) so it binds from Java (Panama FFM or a JNI shim), ctypes, or C++.
 * "Replaces" cites the reference interface (files under /root/reference/src) the
 * entry point stands in for; INTEGRATION.md shows the Java-side binding.
 *
 * Conventions
 *   - all functions return 0 on success or a negative SWB_E_* code; the message is
 *     available from swb_last_error() (per calling thread).  Nothing aborts/exits.
 *   - sequences are ASCII bytes (0x00-0x7F); equality is case-insensitive as in
 *     AlignmentScore.call (SmithWaterman.java:309-318); output keeps the original case.
 *   - "pair" p = ref_index * n_reads + read_index: the order in which MapRef.call
 *     (Distribution.java:419-426) visits pairs for one reference, references outermost.
 *   - cells are (i, j), 1-based, i = read row, j = reference column, listed in the
 *     reference's row-major order (SmithWaterman.java:157-185).
 *   - there is no CPU fallback: without a CUDA device every compute entry fails.
 */
#ifndef SWB200_H
#define SWB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SWB_ABI_VERSION 2

/* status codes */
#define SWB_OK              0
#define SWB_E_INVALID      -1   /* bad argument (null pointer, negative size, bad offsets)      */
#define SWB_E_CUDA         -2   /* CUDA runtime error / no device                                 */
#define SWB_E_UNSUPPORTED  -3   /* input outside the supported domain (non-ASCII byte, score
                                   range, alphabet) -- never silently computed elsewhere          */
#define SWB_E_NOMEM        -4
#define SWB_E_RANGE        -5   /* index out of range in an accessor                              */

/* swb_align flags */
#define SWB_F_SCORES_ONLY   1u  /* fill only: scores + ref totals + best hits, no cell lists     */
#define SWB_F_NO_FETCH      2u  /* leave results in HBM; call swb_result_fetch() later           */
#define SWB_F_TIE_GT        4u  /* DistributedSW.GetCellScore's strict '>' cascade (DistributedSW.java:300-330):
                                   on equal candidates deletion wins over insertion over alignment.  Scores and
                                   the max-cell SET are unchanged; cells are still listed row-major (the host
                                   layer re-orders them diagonal-major + stable by beginning, :209, :480)   */
#define SWB_F_BOTH_STRANDS  8u  /* align every read as given AND its reverse complement (see BOTH STRANDS below) */

/* BOTH STRANDS (SWB_F_BOTH_STRANDS; accepted by swb_align, swb_align_resident, swb_align_hits,
 * swb_align_resident_hits, the all-hits entries, swb_multi_align and swb_multi_align_hits, combinable with every other flag;
 * swb_align_pair refuses it with SWB_E_INVALID).  Sequencing reads come from either strand; this mode aligns
 * each read q and its reverse complement rc(q) against every reference in the same call.
 *   - the result has swb_result_n_refs == 2 * R ORIENTED references over the set's R references:
 *     o = 2r is reference r with the read as given, o = 2r + 1 is reference r with rc(read).  Pair
 *     p = o * n_reads + q; every accessor applies unchanged (scores, cell offsets, cells, beginnings,
 *     op lengths, ops, pair_cell_count, pair_cell, hits).
 *   - for an odd o, cell (i, j) has i = row of rc(read) (1-based) and j = column of reference r: positions are
 *     forward-reference coordinates.  Beginnings, op lengths and ops are those of that alignment.
 *   - ref_totals[o] sums over reads per oriented reference; best_hits[q] and the hit lists are taken over all 2R
 *     oriented references with the usual rule (score descending, then lowest index): on a tie the lower reference
 *     wins, and on the same reference the forward strand wins (a palindromic read reports o = 2r).
 *   - swb_result_materialize takes the caller's ORIGINAL read; for a cell of an odd o it builds the read string
 *     from rc(read), keeping case (a -> t).
 *   - complement: the IUPAC DNA involution A<->T, C<->G, R<->Y, K<->M, B<->V, D<->H; S, W, N map to themselves
 *     (case-insensitive).  A set with any other symbol is SWB_E_UNSUPPORTED for this mode.  Position i of rc(read)
 *     matches nothing when read[m-1-i], or its complement, is absent from the set.
 *   - stats out[6] / out[7] (cells, pairs) count both strands.
 *   - multi-GPU: shard results are oriented over the shard's references; the merge works on oriented global ids
 *     2 * global_ref + s, so the merged records equal one context's.  swb_comm_allgather_best / _hits take oriented
 *     ids for a both-strands result: n_local_refs = 2 * shard refs, global_ids[2r + s] = 2 * gid(r) + s. */

typedef struct swb_ctx    swb_ctx;     /* one CUDA device + streams + workspace                */
typedef struct swb_refset swb_refset;  /* packed reference set resident in HBM                  */
typedef struct swb_reads  swb_reads;   /* encoded read batch resident in HBM                    */
typedef struct swb_result swb_result;  /* results of one swb_align call                         */

int         swb_abi_version(void);
const char *swb_last_error(void);

/* Number of visible CUDA devices (0 if none); never fails. */
int swb_device_count(void);

/* Context for CUDA device `device`.  workspace_bytes bounds the HBM scratch used for
 * fill's block records (0 = default: 45 % of the free HBM, at most 64 GiB; always clamped to half the free memory). */
int  swb_create(int device, int64_t workspace_bytes, swb_ctx **out);
void swb_destroy(swb_ctx *ctx);

/* Load a reference set: n_refs sequences, ref k = bytes[offsets[k] .. offsets[k+1]).
 * Case-folds, validates, packs 2 bits/base, sorts into length buckets and uploads.
 * Replaces: the ref[1] strings of InOutOps.GetRefSeqs (InOutOps.java:100-169) as
 * carried into CombineReadsToRef.call (Distribution.java:714-724).
 * The set stays resident in HBM until swb_refset_free. */
int     swb_refset_load(swb_ctx *ctx, int64_t n_refs, const char *bytes, const int64_t *offsets,
                        swb_refset **out);
void    swb_refset_free(swb_refset *rs);
int64_t swb_refset_count(const swb_refset *rs);
int64_t swb_refset_total_bases(const swb_refset *rs);

/* Upload + encode a read batch against a reference set's alphabet (HBM-resident). */
int     swb_reads_upload(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *bytes,
                         const int64_t *offsets, swb_reads **out);
void    swb_reads_free(swb_reads *rd);
int64_t swb_reads_count(const swb_reads *rd);

/* Align every read against every reference of the set: score-matrix fill, all
 * maximum-score cells, traceback of each.
 * Replaces: the loop body of Distribution.MapRef.call (Distribution.java:419-426),
 * i.e. `new SmithWaterman.OptAlignments().call({ref, read}, {match, mismatch, gap}, types)`
 * (SmithWaterman.java:62-92) for all refs x reads, plus the per-ref totalScore (:424).
 * Host-buffer form: copies the reads in, runs, copies the results out. */
int swb_align(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes,
              const int64_t *read_offsets, int32_t match, int32_t mismatch, int32_t gap,
              uint32_t flags, swb_result **out);

/* Same, reads already resident (swb_reads_upload).  With SWB_F_NO_FETCH the results
 * stay in HBM until swb_result_fetch. */
int swb_align_resident(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd,
                       int32_t match, int32_t mismatch, int32_t gap, uint32_t flags,
                       swb_result **out);
int swb_result_fetch(swb_result *res);
void swb_result_free(swb_result *res);

/* HITS MODE: the same call, but alignments only where a read aligns best.  Every pair is still scored; each read's
 * top_k best pairs are traced, and nothing else.  Arguments as swb_align / swb_align_resident plus
 *   top_k      1 .. 32
 *   min_score  >= 1: a hit has score >= min_score (a score-0 pair is never a hit)
 * anything else is SWB_E_INVALID.
 *   - scores, ref_totals and best_hits are those of the plain call, bit for bit; SWB_F_SCORES_ONLY, SWB_F_TIE_GT,
 *     SWB_F_NO_FETCH + swb_result_fetch apply as there.
 *   - hits (swb_result_hits): hits[(q * k + h) * 4 ..] = (score, ref, i, j), h = 0 .. k-1, read q's k best pairs
 *     with score >= min_score, score descending, then reference index ascending (the best-hit rule: hits[q][0] ==
 *     best_hits[q] whenever best_hits[q].score >= min_score).  (i, j) = the pair's first max cell in row-major
 *     order, (0, 0) under SWB_F_SCORES_ONLY.  A read with fewer than k hits is padded with (0, -1, 0, 0).
 *   - cells: only hit pairs have max cells, beginnings, op lengths and ops, each equal to what the plain call
 *     returns for that pair (swb_result_materialize too).  cell_offsets still spans all pairs, so every accessor
 *     applies; every other pair has an empty range and swb_result_pair_cell_count 0 (no implicit m*n cells).
 *     A reference set that is cut into parts is aligned as one set here.
 * Prefer it to SWB_F_SCORES_ONLY when the alignments of a read's best references are wanted, and to the plain call
 * when the cells of all other pairs are not: the traceback, the assembly and the device->host copy shrink to k
 * pairs per read. */
int swb_align_hits(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                   int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score,
                   swb_result **out);
int swb_align_resident_hits(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                            int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score, swb_result **out);
/* [n_reads * k * 4] of a fetched hits-mode result (NULL before the fetch), *top_k = k; NULL and *top_k = 0 for a plain result */
const int32_t *swb_result_hits(const swb_result *res, int32_t *top_k);

/* ALL-HITS MODE: the same call, but every good hit of a read, with no cap on the count.  Every pair is still scored;
 * with best_q = read q's best score in the call, pair (ref, q) is LISTED iff score >= min_score and
 * score >= best_q - margin (computed in 64 bits: a large margin cannot wrap).  Arguments as swb_align /
 * swb_align_resident plus
 *   min_score  >= 1 (a score-0 pair is never listed)
 *   margin     >= 0: 0 gives the co-optimal set (the multi-mapping set), INT32_MAX the plain threshold score >= min_score
 * anything else is SWB_E_INVALID.
 *   - lists (swb_result_hit_offsets / swb_result_hit_list): read q's entries are hit_list[4 * k ..], k = hit_offsets[q] ..
 *     hit_offsets[q + 1] - 1, each (score, ref, i, j), score descending, then reference index ascending.  (i, j) is the
 *     pair's first max cell in row-major order, (0, 0) under SWB_F_SCORES_ONLY.  Whenever hits mode lists k entries for
 *     a read, its list is the first k entries of this one (same min_score, a large margin).
 *   - scores, ref_totals and best_hits are those of the plain call, bit for bit.  Only listed pairs have max cells,
 *     beginnings, op lengths and ops, each equal to what the plain call returns (swb_result_materialize too); every
 *     other pair has an empty range and swb_result_pair_cell_count 0.  A read's best pair below min_score is traced
 *     too, so best_hits keeps its (i, j).
 *   - SWB_F_SCORES_ONLY, SWB_F_TIE_GT, SWB_F_NO_FETCH + swb_result_fetch and SWB_F_BOTH_STRANDS apply; under both
 *     strands `ref` is the oriented index o = 2r + s and best_q is taken over both strands.  A reference set that is cut
 *     into parts is aligned as one set here.
 * Prefer it to hits mode when a read may have more than 32 good references (a repeat family) or when the question is
 * a threshold, and to the plain call + a host filter when only good hits need alignments: the traceback, the assembly
 * and the device->host copy shrink to the listed pairs.  The margin is the caller's cost knob: with a very large
 * margin and a low min_score almost every pair is listed, and the call costs about what the plain call costs. */
int swb_align_all_hits(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                       int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, int32_t min_score, int32_t margin,
                       swb_result **out);
int swb_align_resident_all_hits(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                                int32_t gap, uint32_t flags, int32_t min_score, int32_t margin, swb_result **out);
/* fetched all-hits result: [n_reads + 1] offsets into the list, *n_hits = total; NULL / 0 for any other result */
const int64_t *swb_result_hit_offsets(const swb_result *res, int64_t *n_hits);
/* [n_hits * 4] (score, ref, i, j) */
const int32_t *swb_result_hit_list(const swb_result *res);

/* ONE pair through the context's submission queue.
 * Replaces: `new SmithWaterman.OptAlignments().call({ref, read}, {match, mismatch, gap}, types)` exactly as the
 * UNCHANGED driver issues it -- once per pair, from N Spark task threads (Distribution.java:419-426, :593;
 * operator SmithWaterman.java:62-92).  Thread-safe and meant to be called concurrently: calls that arrive while
 * the device is busy are coalesced -- one of the waiting threads loads the distinct references of all queued
 * requests (same scores and flags) as one set, their distinct reads as one batch, runs one align sequence and
 * hands every caller its own 1 x 1 result (pair index 0; every swb_result_* accessor applies; free it with
 * swb_result_free).  SWB_F_NO_FETCH is ignored: the result is always on the host. */
int swb_align_pair(swb_ctx *ctx, const char *ref, int64_t ref_len, const char *read, int64_t read_len,
                   int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, swb_result **out);
/* out[0] = swb_align_pair calls so far, out[1] = batches they were served in, out[2] = largest batch */
int swb_queue_stats(swb_ctx *ctx, int64_t *out, int n);

/* ---- result accessors (valid after fetch; pointers live until swb_result_free) ---- */
int64_t swb_result_n_refs(const swb_result *res);
int64_t swb_result_n_reads(const swb_result *res);
/* scores[p]: maximum cell score of pair p (ScoreMatrix.call result _1, SmithWaterman.java:189) */
const int32_t *swb_result_scores(const swb_result *res);
/* ref_totals[r]: wrapping int32 sum over reads (Distribution.java:424) */
const int32_t *swb_result_ref_totals(const swb_result *res);
/* best_hits[4*q .. 4*q+3] = (score, ref index, i, j) of read q's best reference: highest
 * score, lowest ref index on ties, first max cell in row-major order ((0,0) if score 0).
 * The reference has no per-read best hit (it reduces per REFERENCE, Distribution.java:424); this
 * record and its tie rule are this engine's definition (BASELINE north_star: "per-read (score,
 * ref id, cell) best-hit records"). */
const int32_t *swb_result_best_hits(const swb_result *res);

/* cell_offsets[p] .. cell_offsets[p+1] index the materialised max cells of pair p.
 * A pair whose score is 0 has, per the reference, EVERY cell as a max cell with an empty
 * alignment (SmithWaterman.java:180-185, :380): those m*n cells are not materialised;
 * swb_result_pair_cell_count reports them and swb_result_pair_cell enumerates them. */
const int64_t *swb_result_cell_offsets(const swb_result *res);
int64_t        swb_result_total_cells(const swb_result *res);
const int32_t *swb_result_cells(const swb_result *res);       /* 2 per cell: i, j       */
const int32_t *swb_result_beginnings(const swb_result *res);  /* per cell               */
const int32_t *swb_result_op_lens(const swb_result *res);     /* per cell: #columns     */

/* number of max cells of pair p including the implicit score-0 case (none in hits mode) */
int64_t swb_result_pair_cell_count(const swb_result *res, int64_t pair);
/* k-th max cell of pair p (reference list order): i, j, beginning, op_len */
int swb_result_pair_cell(const swb_result *res, int64_t pair, int64_t k,
                         int32_t *i, int32_t *j, int32_t *beginning, int32_t *op_len);
/* alignment columns of materialised cell c (global cell index), start-to-end,
 * one byte per column: 1 = aligned pair, 2 = insertion (gap in ref), 3 = deletion
 * (gap in read).  Writes op_len bytes; cap must be >= op_len. */
int swb_result_ops(const swb_result *res, int64_t cell, uint8_t *out, int64_t cap);
/* Builds the two strings GetAlignment.call returns (SmithWaterman.java:418-435):
 * aligned reference and aligned read with '_' gaps, original case.  ref/read are the
 * caller's original sequences of that pair.  Writes op_len bytes + NUL to each. */
int swb_result_materialize(const swb_result *res, int64_t cell,
                           const char *ref, int64_t ref_len, const char *read, int64_t read_len,
                           char *ref_aln, char *read_aln, int64_t cap);

/* timings of the call in milliseconds (CUDA events on the engine's stream) and counters:
 * out[0]=h2d  out[1]=fill  out[2]=locate+sort  out[3]=traceback  out[4]=d2h  out[5]=total device
 * out[6]=cells (sum m*n)  out[7]=pairs  out[8]=materialised max cells  out[9]=kernel launches
 * out[10]=checkpoint bytes written  out[11]=read batches (swb_align_pair: requests served by the pair's batch)
 * out[12]=hits mode: top-k selection ms (the selections of the short path run inside out[2]'s span) */
int swb_result_stats(const swb_result *res, double *out, int n);

/* Device pointers of the HBM-resident outputs (for collectives over NVLink without a
 * host round trip): which = 0 scores, 1 ref_totals, 2 best_hits. */
int swb_result_device_ptr(const swb_result *res, int which, void **ptr, int64_t *n_elems);

/* The CUDA stream (cudaStream_t) every kernel and copy of this context is issued on, so a
 * host can bracket calls with its own events on that stream. */
int swb_get_stream(swb_ctx *ctx, void **stream);

/* ---- multi-GPU: the reference set sharded over devices, best hits merged over NVLink ----------------
 * Replaces: the partition point of the reference's driver, `sc.parallelize(refs)` + map(MapRef)
 * (Distribution.java:337-338): the pair set refs x reads is cut by REFERENCE, every device aligns
 * all reads against its own shard (scores, max-cell lists, alignments and per-reference totals stay
 * with the owning device), and only the per-read best-hit records (score, GLOBAL ref index, i, j)
 * cross NVLink -- one ncclAllGather issued on each device's engine stream right after the best-hit
 * kernel, followed by a merge kernel on the device.  The reference has no per-read best hit; the
 * merge rule is this engine's own: highest score, then lowest global reference index (the running
 * maximum with first-wins order of a single device scanning the references in index order).
 * NCCL is loaded at run time (dlopen of libnccl.so.2, or $SWB_NCCL_LIB); a single device needs none.
 *
 * Two forms.  swb_multi_*: ONE process drives all devices (a JVM / Spark local[N] host) -- one host
 * thread per device inside the call.  swb_comm_*: one process per device (torchrun, MPI); the host
 * only carries the 128-byte NCCL id from rank 0 to the other ranks. */
typedef struct swb_multi        swb_multi;         /* n devices: contexts, sharded reference set, NCCL communicators */
typedef struct swb_multi_result swb_multi_result;
typedef struct swb_comm         swb_comm;          /* one rank of a multi-process job */

/* devices[n_devices] = CUDA device indices (n_devices >= 1); workspace as in swb_create, per device. */
int  swb_multi_create(const int32_t *devices, int32_t n_devices, int64_t workspace_bytes, swb_multi **out);
void swb_multi_destroy(swb_multi *m);
int32_t swb_multi_device_count(const swb_multi *m);
/* Context of shard d (borrowed; e.g. for swb_get_stream). */
swb_ctx *swb_multi_ctx(swb_multi *m, int32_t d);

/* Shard + load: references sorted by descending length (stable) and dealt in snake order
 * (0..n-1, n-1..0, ...) so that every device holds the same number of bases to within one reference;
 * shard d keeps its references in ascending global index.  Replaces an earlier set of this handle. */
int  swb_multi_refset_load(swb_multi *m, int64_t n_refs, const char *bytes, const int64_t *offsets);
int64_t swb_multi_ref_count(const swb_multi *m);
/* global reference index -> (shard, index inside the shard) */
int  swb_multi_ref_location(const swb_multi *m, int64_t global_ref, int32_t *shard, int64_t *local_ref);
/* global indices of shard d's references, ascending; *n = their number */
const int64_t *swb_multi_shard_refs(const swb_multi *m, int32_t d, int64_t *n);

/* All reads against all shards (swb_align on every device, concurrently) + the best-hit merge. */
int  swb_multi_align(swb_multi *m, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                     int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, swb_multi_result **out);
void swb_multi_result_free(swb_multi_result *res);
/* shard d's own result (borrowed; pair p = local_ref * n_reads + read): every swb_result_* accessor applies */
swb_result *swb_multi_result_shard(swb_multi_result *res, int32_t d);
/* merged[4*q .. 4*q+3] = (score, GLOBAL ref index, i, j) of read q over all shards */
const int32_t *swb_multi_result_best_hits(const swb_multi_result *res);
/* Hits mode: swb_align_hits on every shard (local reference indices, all cells with their shard), then each shard's
 * hit lists -> global ids -> one more ncclAllGather (n_reads * k * 16 bytes) -> a k-way merge kernel.  The merged
 * list is the top k over the union of the shards' lists in the same order -- exact, since the global top k lies in
 * that union -- so it is the same for any device count and equal to one context's hits over the whole set.
 * Entries without a reference never win.  (Up to 64 devices.) */
int  swb_multi_align_hits(swb_multi *m, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                          int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score,
                          swb_multi_result **out);
/* merged[(q * k + h) * 4 ..] = (score, GLOBAL ref index, i, j), *top_k = k; NULL and 0 for a plain result */
const int32_t *swb_multi_result_hits(const swb_multi_result *res, int32_t *top_k);
/* All-hits mode: swb_align_all_hits on every shard.  Each shard selects against its LOCAL best score, which is never
 * above the global one, so a shard's list holds every pair of it that survives.  Merge: the lists -> global ids, one
 * ncclAllGather of the per-read offsets, one host sync for the largest per-shard total, one ncclAllGather of the
 * lists padded to that total, then a merge kernel per read: the global best from the lists' heads, the entries
 * filtered to score >= max(min_score, global best - margin), a k-way merge in list order.  The merged lists are the
 * same for any device count and equal to one context's lists over the whole set.  A shard result keeps the cells of
 * its LOCAL selection, a superset of the merged one's pairs on that shard.  (Up to 64 devices.) */
int  swb_multi_align_all_hits(swb_multi *m, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                              int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, int32_t min_score, int32_t margin,
                              swb_multi_result **out);
/* merged lists of an all-hits result: [n_reads + 1] offsets, *n_hits = total, and [n_hits * 4] (score, GLOBAL ref
 * index, i, j); NULL / 0 for any other result */
const int64_t *swb_multi_result_hit_offsets(const swb_multi_result *res, int64_t *n_hits);
const int32_t *swb_multi_result_hit_list(const swb_multi_result *res);
/* out[0] = wall ms of the call, out[1] = max over devices of the align's device ms, out[2] = allgather + merge ms */
int  swb_multi_result_stats(const swb_multi_result *res, double *out, int n);

/* multi-process form: rank 0 calls swb_comm_unique_id and ships the 128 bytes to every rank. */
int  swb_comm_unique_id(char *id128);
int  swb_comm_create(swb_ctx *ctx, const char *id128, int32_t rank, int32_t world, swb_comm **out);
void swb_comm_destroy(swb_comm *c);
/* Best hits of `res` (a result of this rank's shard, fetched or not) -> global ids through
 * global_ids[n_local_refs] (host array) -> ncclAllGather on the context's stream -> merge kernel.
 * merged_host (nullable) receives [n_reads * 4]; the merged records also stay on the device
 * (swb_comm_merged_device_ptr) until the next call. */
int  swb_comm_allgather_best(swb_comm *c, const swb_result *res, const int64_t *global_ids, int64_t n_local_refs,
                             int32_t *merged_host);
int  swb_comm_merged_device_ptr(swb_comm *c, void **ptr, int64_t *n_elems);
/* The same for the hit lists of a hits-mode result (every rank passes the same top_k): merged_host (nullable)
 * receives [n_reads * k * 4], (score, GLOBAL ref index, i, j), merged as in swb_multi_align_hits. */
int  swb_comm_allgather_hits(swb_comm *c, const swb_result *res, const int64_t *global_ids, int64_t n_local_refs,
                             int32_t *merged_host);
/* The same for the lists of an all-hits result (every rank passes the same min_score and margin), merged as in
 * swb_multi_align_all_hits: *offsets = [n_reads + 1], *list = [*n_hits * 4] (score, GLOBAL ref index, i, j), host
 * arrays owned by the communicator, valid until its next call or swb_comm_destroy.  Both strands: oriented ids as for
 * swb_comm_allgather_hits. */
int  swb_comm_allgather_all_hits(swb_comm *c, const swb_result *res, const int64_t *global_ids, int64_t n_local_refs,
                                 const int64_t **offsets, const int32_t **list, int64_t *n_hits);

/* Integer / DPX issue-rate microbenchmark (roofline denominator, SURVEY.md 8d). */
int swb_microbench_json(int device, int iters, char *buf, int buflen);

#ifdef __cplusplus
}
#endif
#endif /* SWB200_H */
