// swb_align.cu -- the align driver: the steps of one call over a packed set (K classes of short reads in batches of
// read pairs, the wide reads, the selections of hits and all-hits mode, the device-side assembly), a set cut into parts
// aligned part by part with each part's results crossing PCIe while the next one computes, and the fetch of a result to
// the host.
#include "swb_host.h"

using namespace swbh;

// Work units of the fill: every reference is one segment unless it is very long.  A long reference
// is cut into windows of SEG columns, each started W_al columns early from an all-zero boundary.
// H(i,j) only depends on the columns (j - W, j], W = m + floor(max(match,mismatch,0)*m/|gap|) + 1 (a
// positive-score path over i <= m rows can pay for at most that many deletions), so every cell
// further than W from the window's left edge is exact; the segment OWNS (writes tile maxima and
// checkpoints for) exactly the blocks of its own SEG columns.  This bounds the longest item (tail of
// the persistent fill) and gives a single long reference enough items to fill the machine.
namespace {
struct Segments { std::vector<int32_t> ref, c0, len, skip, end; };
void make_segments(const swb_refset *rs, int K, int match, int mismatch, int gap, bool few_items, Segments &S)
{
    const int64_t m = (int64_t)GL * K;
    const int64_t big = std::max({match, mismatch, 0});
    const int64_t W = m + (big * m) / (-(int64_t)gap) + 1;
    const int64_t W_al = ((W + 8 + 15) / 16) * 16;
    int64_t SEG = few_items ? 1024 : 8192;                                        // few items: favour parallelism
    SEG = std::max<int64_t>(SEG, ((2 * W_al + 15) / 16) * 16);
    const int32_t BIG = 1 << 26;
    struct One { int32_t ref, c0, len, skip, end; };
    std::vector<One> v;
    v.reserve((size_t)rs->n_refs + 64);
    for (int64_t s = 0; s < rs->n_refs; ++s) {
        const int64_t n = rs->len_sorted[(size_t)s];
        if (n <= 2 * SEG) { v.push_back(One{(int32_t)s, 0, (int32_t)n, 0, BIG}); continue; }
        const int64_t nseg = (n + SEG - 1) / SEG;
        for (int64_t k = 0; k < nseg; ++k) {
            const int64_t lo = k * SEG, hi = std::min<int64_t>(n, (k + 1) * SEG);
            const int64_t c0 = std::max<int64_t>(0, lo - W_al);
            v.push_back(One{(int32_t)s, (int32_t)c0, (int32_t)(hi - c0), (int32_t)((lo - c0) / CB),
                            k == nseg - 1 ? BIG : (int32_t)((hi - c0) / CB)});
        }
    }
    std::stable_sort(v.begin(), v.end(), [](const One &a, const One &b) { return a.len > b.len; });
    S.ref.clear(); S.c0.clear(); S.len.clear(); S.skip.clear(); S.end.clear();
    for (const One &o : v) { S.ref.push_back(o.ref); S.c0.push_back(o.c0); S.len.push_back(o.len); S.skip.push_back(o.skip); S.end.push_back(o.end); }
}

int pick_k(int m)
{
    for (int k = 0; k < kNumK; ++k)
        if (GL * kKList[k] >= m) return kKList[k];
    return 0;
}

int record_words(int K) { return ((K + 1 + 7) / 8 + CB / 8) * 8; }         // per (block, lane): Geo<K>::RW

// a result of rs x rd; it counts as a live handle of its context from here on (swb_result_free releases it, also on the
// error paths).  SWB_F_BOTH_STRANDS: rd holds the 2n internal reads and the result is oriented, 2R references x n reads;
// its cells and pairs count both strands.
using ResultPtr = std::unique_ptr<swb_result, void (*)(swb_result *)>;
ResultPtr new_result(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, uint32_t flags, const Selection &sel)
{
    ResultPtr res(new swb_result(), swb_result_free);
    ctx->live.fetch_add(1);
    res->ctx = ctx; res->n_refs = rs->n_refs; res->n_reads = rd->n_reads; res->flags = flags; res->sel = sel;
    res->ref_len = rs->len_orig; res->read_len = rd->len;
    if (flags & SWB_F_BOTH_STRANDS) {
        res->n_refs = 2 * rs->n_refs; res->n_reads = rd->n_reads / 2;
        res->ref_len.resize((size_t)res->n_refs);
        for (int64_t o = 0; o < res->n_refs; ++o) res->ref_len[(size_t)o] = rs->len_orig[(size_t)(o >> 1)];
        res->read_len.resize((size_t)res->n_reads);
    }
    int64_t read_bases = 0;
    for (int32_t m : rd->len) read_bases += m;
    res->stats[STAT_CELLS] = (double)rs->total_bases * (double)read_bases;
    res->stats[STAT_PAIRS] = (double)rs->n_refs * (double)rd->n_reads;
    return res;
}
}  // namespace

// one batch of read pairs of a K class; its host table stays alive until the class's sync (async copies read it)
struct AlignCall::Batch {
    int n_rp = 0, m_max = 0;
    std::vector<int32_t> h_rp;                   // read pair slot -> read, -1 = empty half
    BatchParams P;
};

// ext_scores / ext_totals: rows of the parent's score matrix / totals a part writes into (nullptr: own arrays)
int AlignCall::run(int32_t *ext_scores, int32_t *ext_totals)
{
    const int64_t n_refs = rs->n_refs, n_reads = rd->n_reads;
    const size_t n_pairs = (size_t)(n_refs * n_reads);
    if (ext_scores) res->d_scores.view(ext_scores, n_pairs); else CU(res->d_scores.alloc(n_pairs, st));
    if (ext_totals) res->d_totals.view(ext_totals, (size_t)o_refs); else CU(res->d_totals.alloc((size_t)o_refs, st));
    CU(res->d_best.alloc((size_t)o_reads * 4, st));
    CU(cudaMemsetAsync(res->d_scores.p, 0, std::max<size_t>(n_pairs, 1) * 4, st));
    if (sel.mode == Selection::TOP_K) CU(res->d_hits.alloc((size_t)o_reads * sel.top_k * 4, st));

    const auto t_wall0 = std::chrono::steady_clock::now();
    ctx->ev_used = 0;                                    // the timer's spans reuse the context's events
    CU(ctx->counters.reserve(16, st));
    int rc;
    if (n_refs > 0 && n_reads > 0) {
        std::vector<std::vector<int32_t>> classes(kNumK);
        std::vector<int32_t> wide;
        classify_reads(classes, wide);
        for (int kc = 0; kc < kNumK; ++kc)
            if (!classes[(size_t)kc].empty() && (rc = run_class(kKList[kc], classes[(size_t)kc]))) return rc;
        if (!wide.empty() && (rc = run_wide_reads(wide))) return rc;
    }
    DevBuf<uint32_t> keep;
    if (sel.mode != Selection::NONE && (rc = select_final(keep))) return rc;
    if ((rc = assemble(keep))) return rc;
    return finish_stats(t_wall0);
}

// reads by rows-per-lane class of the short path, longest first inside a class after run_class; the rest take the wide path.
// Both strands: read q and its reverse complement n + q go in next to each other.  They have the same length, so the
// stable length sort keeps them next to each other, and every class holds whole (q, n + q) read pairs.
void AlignCall::classify_reads(std::vector<std::vector<int32_t>> &classes, std::vector<int32_t> &wide) const
{
    // s16x2 short-read kernels: gap < 0 (padding stays below the maximum), small scores, 2-bit alphabet;
    // everything else goes through the int32 wide path (swb_wide.cu)
    const bool short_scores_ok = rs->two_bit_ok && gap < 0 && std::abs((int64_t)match) <= 8000 &&
                                 std::abs((int64_t)mismatch) <= 8000 && std::abs((int64_t)gap) <= 8000;
    // reads of 257 .. 511 rows: the LONG classes (K = 40 .. 64) exist for the biased fill and the tile kernels only;
    // other score sets send such reads through the wide path
    const bool long_kernels_ok = tile_trace_ok(match, mismatch, gap);
    for (int64_t x = 0; x < rd->n_reads; ++x) {
        const int64_t q = both ? (x >> 1) + (x & 1) * o_reads : x;
        const int m = rd->len[(size_t)q];
        if (m == 0) continue;                                  // score 0, no cells
        const int64_t smax = (int64_t)std::max({match, mismatch, 0}) * std::min<int64_t>(m, rs->max_len);   // a positive mismatch scores too
        const bool is_short = short_scores_ok && smax <= 16000 &&
                              (m <= MAX_SHORT_ROWS || (m <= MAX_LONG_ROWS && long_kernels_ok && fill_bias_ok(match, mismatch, gap, smax)));
        if (!is_short) { wide.push_back((int32_t)q); continue; }
        const int K = pick_k(m);
        for (int k = 0; k < kNumK; ++k) if (kKList[k] == K) classes[(size_t)k].push_back((int32_t)q);
    }
}

// the reads of one K class, two per read pair, in equal batches of read pairs: fill batch k, then trace batch k
int AlignCall::run_class(int K, std::vector<int32_t> &reads)
{
    std::stable_sort(reads.begin(), reads.end(), [&](int32_t a, int32_t b) { return rd->len[(size_t)a] > rd->len[(size_t)b]; });
    const int64_t n_rp_total = ((int64_t)reads.size() + 1) / 2;
    std::shared_ptr<swb_refset::SegTables> segt;
    int rc = seg_tables(K, n_rp_total * ((rs->n_refs + 3) / 4) < (int64_t)ctx->sm_count * 24, segt);
    if (rc) return rc;
    // as many read pairs per batch as the workspace holds block records (checkpoint + seam) and tile maxima for
    const int64_t bytes_per_rp = rs->blocks_per_rp * ((int64_t)record_words(K) * GL * 4 + GL * 4);
    int64_t rp_per_batch = std::max<int64_t>(1, ctx->ws_bytes / std::max<int64_t>(bytes_per_rp, 1));
    rp_per_batch = std::min<int64_t>(rp_per_batch, 1 << 16);
    if (rp_per_batch * rs->n_refs * 2 >= ((int64_t)1 << 30)) rp_per_batch = std::max<int64_t>(1, (((int64_t)1 << 30) - 1) / (rs->n_refs * 2));
    // equal-sized batches (no small straggler batch at the end)
    const int64_t nb = (n_rp_total + rp_per_batch - 1) / rp_per_batch;
    rp_per_batch = (n_rp_total + nb - 1) / nb;
    std::vector<Batch> batches((size_t)nb);
    for (int64_t k = 0; k < nb; ++k) {
        const int64_t rp0 = k * rp_per_batch;
        Batch &b = batches[(size_t)k];
        if ((rc = fill_batch(K, reads, rp0, (int)std::min<int64_t>(rp_per_batch, n_rp_total - rp0), *segt, b))) return rc;
        if ((rc = trace_batch(K, b))) return rc;
    }
    CU(cudaStreamSynchronize(st));
    return SWB_OK;
}

// the segment tables of class K (make_segments) only depend on (K, scores, few-items flag): built once per reference
// set and kept on the device
int AlignCall::seg_tables(int K, bool few_items, std::shared_ptr<swb_refset::SegTables> &out)
{
    const swb_refset::SegKey skey{K, match, mismatch, gap, few_items ? 1 : 0};
    auto sit = rs->seg_cache.find(skey);
    if (sit == rs->seg_cache.end()) {
        Segments segs;
        make_segments(rs, K, match, mismatch, gap, few_items, segs);
        auto sc = std::make_shared<swb_refset::SegTables>();
        sc->nv = segs.ref.size();
        CU(sc->ref.alloc(sc->nv, st)); CU(sc->c0.alloc(sc->nv, st)); CU(sc->len.alloc(sc->nv, st));
        CU(sc->skip.alloc(sc->nv, st)); CU(sc->end.alloc(sc->nv, st));
        CU(cudaMemcpyAsync(sc->ref.p, segs.ref.data(), sc->nv * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(sc->c0.p, segs.c0.data(), sc->nv * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(sc->len.p, segs.len.data(), sc->nv * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(sc->skip.p, segs.skip.data(), sc->nv * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(sc->end.p, segs.end.data(), sc->nv * 4, cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));         // segs is a local
        if (rs->seg_cache.size() >= 16) rs->seg_cache.clear();
        sit = rs->seg_cache.emplace(skey, sc).first;
    }
    out = sit->second;
    return SWB_OK;
}

// read pairs [rp0, rp0 + n_rp) of the class: the fill writes their pair scores, block records and tile maxima
int AlignCall::fill_batch(int K, const std::vector<int32_t> &reads, int64_t rp0, int n_rp, const swb_refset::SegTables &segt, Batch &b)
{
    b.n_rp = n_rp;
    b.h_rp.assign((size_t)n_rp * 2, -1);
    for (int r = 0; r < n_rp; ++r)
        for (int h = 0; h < 2; ++h) {
            const int64_t x = (rp0 + r) * 2 + h;
            if (x < (int64_t)reads.size()) {
                b.h_rp[(size_t)r * 2 + h] = reads[(size_t)x];
                b.m_max = std::max(b.m_max, rd->len[(size_t)reads[(size_t)x]]);
            }
        }
    ++n_batches;
    // both strands in hits / all-hits mode: the selection's slots, the forward read of each read pair, follow the read pairs
    const bool fwd_slots = both && sel.mode != Selection::NONE && !(flags & SWB_F_SCORES_ONLY);
    if (fwd_slots)
        for (int r = 0; r < n_rp; ++r) b.h_rp.push_back(b.h_rp[(size_t)r * 2]);
    CU(ctx->rp.reserve(b.h_rp.size(), st));
    CU(cudaMemcpyAsync(ctx->rp.p, b.h_rp.data(), b.h_rp.size() * 4, cudaMemcpyHostToDevice, st));
    if (fwd_slots) b.h_rp.resize((size_t)n_rp * 2);
    const size_t ck_words = (size_t)n_rp * rs->blocks_per_rp * record_words(K) * GL;
    const size_t tmx_words = (size_t)n_rp * rs->blocks_per_rp * GL;
    CU(ctx->ck.reserve(ck_words, st));
    CU(ctx->tmx.reserve(tmx_words, st));
    ck_bytes += (double)(ck_words + tmx_words) * 4;
    BatchParams &P = b.P;
    P.ref_words = rs->words.p; P.ref_word_off = rs->word_off.p; P.ref_len = rs->len.p;
    P.ref_orig = rs->orig.p; P.ref_sorted_of = rs->sorted_of.p; P.ref_blk_off = rs->blk_off.p;
    P.n_refs = (int32_t)rs->n_refs; P.blocks_per_rp = rs->blocks_per_rp;
    P.v_ref = segt.ref.p; P.v_c0 = segt.c0.p; P.v_len = segt.len.p; P.v_skip = segt.skip.p;
    P.v_end = segt.end.p; P.n_vrefs = (int32_t)segt.nv;
    P.read_codes = rd->codes.p; P.read_off = rd->off.p; P.rp_reads = ctx->rp.p; P.read_slot = nullptr;
    P.n_rp = n_rp; P.n_reads = rd->n_reads;
    P.match = match; P.mismatch = mismatch; P.gap = gap; P.tie_gt = (flags & SWB_F_TIE_GT) ? 1 : 0;
    P.scores = res->d_scores.p; P.rec = ctx->ck.p; P.tmx = ctx->tmx.p; P.sel = nullptr;
    uint32_t *d_work = ctx->counters.p + 4;
    const bool biased = fill_bias_ok(match, mismatch, gap, (int64_t)std::max({match, mismatch, 0}) * std::min<int64_t>(b.m_max, rs->max_len));
    P.seam_bias = biased ? -gap : 0;               // the biased fill stores its seams biased
    P.tmx_slack = biased ? fill_sub_slack(match, mismatch, gap) : 0;
    CU(timer.begin(STAT_FILL_MS));
    if (biased)
        CU(launch_fill_bias(K, P, d_work, ctx->sm_count, st));
    else
        CU(launch_fill(K, P, d_work, ctx->sm_count, st));
    ++launches;
    CU(timer.end());
    return SWB_OK;
}

// exact scores of a filled batch and, with cells, its sorted max-cell keys and their tracebacks (one BatchOut)
int AlignCall::trace_batch(int K, Batch &b)
{
    const bool scores_only = (flags & SWB_F_SCORES_ONLY) != 0;
    // hits / all-hits mode: the scan makes the batch's score rows exact, the selection marks the pairs the emit keeps
    size_t sel_words = 0;
    if (sel.mode != Selection::NONE && !scores_only) {
        sel_words = ((size_t)b.n_rp * 2 * (size_t)rs->n_refs + 31) / 32;
        CU(ctx->hit_sel.reserve(sel_words, st));
        b.P.sel = ctx->hit_sel.p;
    }
    const BatchParams &P = b.P;
    if (scores_only && P.tmx_slack == 0) return SWB_OK;      // the fill's pair scores are exact
    CU(timer.begin(STAT_LOCATE_MS));
    uint32_t n_cells = 0;
    const int rc = locate_cells(K, b, sel_words, n_cells);
    if (rc) return rc;
    if (scores_only) { CU(timer.end()); return SWB_OK; }
    BatchOut bo;
    bo.n_cells = n_cells;
    CU(bo.keys.alloc(n_cells, st));
    const size_t tmp_bytes = sort_keys_tmp_bytes(n_cells);
    CU(ctx->sort_tmp.reserve(tmp_bytes, st));
    CU(sort_keys(ctx->keys_tmp.p, bo.keys.p, n_cells, ctx->sort_tmp.p, tmp_bytes, st));
    launches += 4;
    CU(timer.end());

    CU(timer.begin(STAT_TRACE_MS));
    const int64_t big = std::max({match, mismatch, 0});
    int64_t lmax = (int64_t)b.m_max + (big * b.m_max - 1) / (-(int64_t)gap) + 1;
    lmax = std::min<int64_t>(lmax, (int64_t)b.m_max + rs->max_len);
    bo.ops_stride = (int)((lmax + 15) / 16);
    CU(bo.beg.alloc(n_cells, st));
    CU(bo.oplen.alloc(n_cells, st));
    CU(bo.ops.alloc((size_t)n_cells * bo.ops_stride, st));
    if (tile_trace_ok(match, mismatch, gap))
        CU(launch_tile_trace(K, P, bo.keys.p, n_cells, bo.beg.p, bo.oplen.p, bo.ops.p, (int)bo.ops_stride, ctx->sm_count, st));
    else
        CU(launch_trace(K, P, bo.keys.p, n_cells, bo.beg.p, bo.oplen.p, bo.ops.p, (int)bo.ops_stride, ctx->sm_count, st));
    ++launches;
    CU(timer.end());
    res->stats[STAT_MAX_CELLS] += n_cells;
    CU(bo.d_slot_read.alloc(b.h_rp.size(), st));
    CU(cudaMemcpyAsync(bo.d_slot_read.p, b.h_rp.data(), b.h_rp.size() * 4, cudaMemcpyHostToDevice, st));
    res->batches.push_back(std::move(bo));
    return SWB_OK;
}

// candidate tiles -> exact pair scores and, unless scores only, the batch's max-cell keys (unsorted, ctx->keys_tmp).
// sel_words > 0 (a selection): marked between the scan and the emit, the pairs whose cells the emit keeps.
// One host sync for the two counts; lists that did not fit are made again with the counted sizes.
int AlignCall::locate_cells(int K, const Batch &b, size_t sel_words, uint32_t &n_cells)
{
    const BatchParams &P = b.P;
    const bool scores_only = (flags & SWB_F_SCORES_ONLY) != 0;
    uint32_t *d_ntasks = ctx->counters.p, *d_ncells = ctx->counters.p + 1;
    const int64_t pairs_b = (int64_t)b.n_rp * 2 * rs->n_refs;
    uint32_t cap_tasks = (uint32_t)std::min<int64_t>(pairs_b * (P.tmx_slack > 0 ? 4 : 2) + 1024, (int64_t)1 << 31);
    uint32_t cap_cells = (uint32_t)std::min<int64_t>(pairs_b * 2 + 4096, (int64_t)1 << 31);
    uint32_t h_counts[2] = {0, 0};
    for (int attempt = 0; attempt < 3; ++attempt) {
        CU(ctx->tasks.reserve(cap_tasks, st));
        CU(ctx->task_hits.reserve((size_t)cap_tasks * locate_hit_bytes(), st));
        CU(ctx->keys_tmp.reserve(cap_cells, st));
        CU(cudaMemsetAsync(ctx->counters.p, 0, 8, st));
        CU(launch_flag_tiles(P, ctx->tasks.p, cap_tasks, d_ntasks, ctx->sm_count, st));
        CU(launch_locate(K, P, ctx->tasks.p, d_ntasks, cap_tasks, ctx->task_hits.p, ctx->keys_tmp.p, cap_cells, d_ncells,
                         ctx->sm_count, 0, st));
        launches += 2;
        if (sel_words) {
            CU(cudaMemsetAsync(ctx->hit_sel.p, 0, sel_words * 4, st));
            // both strands: one slot per read pair over the 2R oriented references; oriented o = 2r + s marks bit
            // (2 * rp + s) * R + r, the emit's bit of pair (r, strand s of read pair rp).  A batch covers all references
            // of its reads, so each read's best score (the margin's bar) is exact here
            const int rc = both ? mark_selection(P.rp_reads + (size_t)b.n_rp * 2, b.n_rp, 1, ctx->hit_sel.p, 2 * rs->n_refs, rs->n_refs, true)
                                : mark_selection(P.rp_reads, (int64_t)b.n_rp * 2, 1, ctx->hit_sel.p, rs->n_refs, 1);
            if (rc) return rc;
        }
        if (!scores_only) {
            CU(launch_locate(K, P, ctx->tasks.p, d_ntasks, cap_tasks, ctx->task_hits.p, ctx->keys_tmp.p, cap_cells, d_ncells,
                             ctx->sm_count, 1, st));
            ++launches;
        }
        CU(cudaMemcpyAsync(h_counts, ctx->counters.p, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (h_counts[0] <= cap_tasks && h_counts[1] <= cap_cells) break;
        if (attempt == 2) return fail(SWB_E_NOMEM, "swb_align: max-cell list did not fit after two retries");
        // a partial scan only raised pair scores towards their exact value: the retry stays correct
        cap_tasks = std::max(cap_tasks, h_counts[0]);
        cap_cells = std::max<uint32_t>(cap_cells, (uint32_t)std::min<uint64_t>((uint64_t)h_counts[1] * 2, 1ull << 31));
    }
    n_cells = h_counts[1];
    return SWB_OK;
}

// marks the pairs the selection keeps among the reads `slots` (nullptr: every read; their score rows are exact by now)
// in `bits`, and each read's best pair with `with_best`; hits mode also writes the reads' top k lists to `hits` when
// it is not null (swb_hits.cu).  Over the oriented view: slots are oriented reads, the references oriented references;
// pair (slot, o) is bit slot * bit_slot + o * bit_ref, or with `oriented_bits` slot * bit_slot + (o & 1) * bit_ref + (o >> 1)
int AlignCall::mark_selection(const int32_t *slots, int64_t n_slots, int with_best, uint32_t *bits, int64_t bit_slot,
                              int64_t bit_ref, bool oriented_bits, int4 *hits)
{
    CU(timer.begin(STAT_SELECT_MS));
    if (sel.mode == Selection::TOP_K) {
        const size_t te = select_hits_tmp_elems(o_refs, n_slots, sel.top_k);
        CU(ctx->hit_tmp.reserve(te, st));
        CU(launch_select_hits(res->d_scores.p, o_refs, o_reads, slots, n_slots, sel.top_k, sel.min_score, with_best, hits, bits,
                              bit_slot, bit_ref, oriented_bits, ctx->hit_tmp.p, te, st));
    } else {
        CU(ctx->margin_best.reserve((size_t)std::max<int64_t>(n_slots, 1), st));
        CU(launch_select_margin(res->d_scores.p, o_refs, o_reads, slots, n_slots, sel.min_score, sel.margin, with_best, bits, bit_slot,
                                bit_ref, oriented_bits, ctx->margin_best.p, st));
    }
    CU(timer.end());
    launches += 2;
    return SWB_OK;
}

// the reads of the int32 wide path.  With a selection: exact scores of every wide pair first, then the whole wide path
// over each read's selected pairs and its best pair.  Slot x's selected references are row x of a bit matrix
// [slots x o_refs], which the host reads once.  Both strands: `wide` holds (q, n + q) next to each other
// (classify_reads); the selection runs once per read q over the oriented references, and each strand takes the
// references of its own orientation.
int AlignCall::run_wide_reads(const std::vector<int32_t> &wide)
{
    const bool scores_only = (flags & SWB_F_SCORES_ONLY) != 0;
    if (sel.mode == Selection::NONE || scores_only) return run_wide_path(wide, scores_only);
    int rc = run_wide_path(wide, true);
    if (rc) return rc;
    std::vector<int32_t> slots;
    for (size_t x = 0; x < wide.size(); x += both ? 2 : 1) slots.push_back(wide[x]);
    const int64_t nw = (int64_t)slots.size();
    const size_t words = ((size_t)nw * (size_t)o_refs + 31) / 32;
    DevBuf<int32_t> d_wr;
    DevBuf<uint32_t> d_bits;
    CU(d_wr.alloc((size_t)nw, st));
    CU(d_bits.alloc(words, st));
    CU(cudaMemcpyAsync(d_wr.p, slots.data(), (size_t)nw * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(d_bits.p, 0, words * 4, st));
    if ((rc = mark_selection(d_wr.p, nw, 1, d_bits.p, o_refs, 1))) return rc;
    std::vector<uint32_t> h_bits(words);
    CU(cudaMemcpyAsync(h_bits.data(), d_bits.p, words * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    std::vector<std::vector<int32_t>> refs_of(wide.size());
    for (size_t w = 0; w < words; ++w)
        for (uint32_t m = h_bits[w]; m; m &= m - 1) {                   // ascending bits: each row's references ascending
            const int64_t bit = (int64_t)w * 32 + __builtin_ctz(m), x = bit / o_refs, o = bit % o_refs;
            if (both) refs_of[(size_t)(2 * x + (o & 1))].push_back((int32_t)(o >> 1));
            else refs_of[(size_t)x].push_back((int32_t)o);
        }
    return run_wide_path(wide, false, &refs_of);
}

// the final selection over all reads (every score is exact now): the result's lists and, with cells, the selected
// pairs as the pairs whose cells the assembly keeps.  Hits mode: the top k lists.  All-hits mode: the lists built from
// the marking pass's per-read best, with one host sync for their length.
int AlignCall::select_final(DevBuf<uint32_t> &keep)
{
    const size_t n_pairs = (size_t)(rs->n_refs * rd->n_reads);
    if (!(flags & SWB_F_SCORES_ONLY)) {
        CU(keep.alloc((n_pairs + 31) / 32, st));
        CU(cudaMemsetAsync(keep.p, 0, ((n_pairs + 31) / 32) * 4, st));
    }
    int rc = mark_selection(nullptr, o_reads, 0, keep.p, 1, o_reads, false, reinterpret_cast<int4 *>(res->d_hits.p));
    if (rc || sel.mode == Selection::TOP_K) return rc;
    CU(timer.begin(STAT_SELECT_MS));
    const size_t n_count = margin_count_elems(o_refs, o_reads);
    DevBuf<int64_t> count, off;
    DevBuf<uint8_t> tmp;
    CU(count.alloc(n_count, st));
    CU(off.alloc(n_count, st));
    size_t tmp_bytes = margin_list_tmp_bytes(o_refs, o_reads, 0);
    CU(tmp.alloc(tmp_bytes, st));
    CU(launch_margin_count(res->d_scores.p, o_refs, o_reads, sel.min_score, sel.margin, ctx->margin_best.p, count.p, off.p, tmp.p,
                           tmp_bytes, st));
    int64_t n_hits = 0;
    CU(cudaMemcpyAsync(&n_hits, off.p + n_count - 1, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (n_hits >= ((int64_t)1 << 31)) return fail(SWB_E_UNSUPPORTED, "swb_align_all_hits: more than 2^31 listed pairs in one call");
    res->n_hits = n_hits;
    CU(res->d_hit_off.alloc((size_t)o_reads + 1, st));
    CU(res->d_hit_list.alloc((size_t)n_hits * 4, st));
    DevBuf<int4> list_tmp;
    DevBuf<uint64_t> keys_tmp, keys_sorted;
    DevBuf<uint32_t> idx_tmp, order;
    CU(list_tmp.alloc((size_t)n_hits, st));
    CU(keys_tmp.alloc((size_t)n_hits, st)); CU(keys_sorted.alloc((size_t)n_hits, st));
    CU(idx_tmp.alloc((size_t)n_hits, st)); CU(order.alloc((size_t)n_hits, st));
    tmp_bytes = margin_list_tmp_bytes(o_refs, o_reads, n_hits);
    CU(tmp.alloc(tmp_bytes, st));
    CU(launch_margin_write(res->d_scores.p, o_refs, o_reads, sel.min_score, sel.margin, ctx->margin_best.p, off.p, n_hits, list_tmp.p,
                           keys_tmp.p, keys_sorted.p, idx_tmp.p, order.p, reinterpret_cast<int4 *>(res->d_hit_list.p),
                           res->d_hit_off.p, tmp.p, tmp_bytes, st));
    CU(timer.end());
    launches += 6;
    return SWB_OK;
}

// per-reference totals, best hits and, with cells, the final ABI-ordered cell arrays on the device (swb_assemble.cu)
int AlignCall::assemble(const DevBuf<uint32_t> &keep)
{
    const int64_t n_refs = rs->n_refs, n_reads = rd->n_reads;
    const size_t n_pairs = (size_t)(n_refs * n_reads);
    CU(launch_ref_totals(res->d_scores.p, o_refs, o_reads, res->d_totals.p, st));
    CU(launch_best_hits(res->d_scores.p, o_refs, o_reads, res->d_best.p, ctx->sm_count, st));
    launches += 3;
    if (flags & SWB_F_SCORES_ONLY) {
        CU(cudaStreamSynchronize(st));
        return SWB_OK;
    }
    std::vector<BatchDesc> descs;
    uint64_t n_total = 0;
    for (auto &bo : res->batches) {
        BatchDesc d;
        d.keys = bo.keys.p; d.beg = bo.beg.p; d.oplen = bo.oplen.p; d.ops = bo.ops.p;
        d.slot_read = bo.d_slot_read.p; d.pair_map = bo.d_pair_map.p;
        d.ops_stride = bo.ops_stride; d.base = (uint32_t)n_total; d.n_cells = bo.n_cells; d.wide = bo.wide ? 1 : 0;
        if (bo.n_cells) descs.push_back(d);
        n_total += bo.n_cells;
    }
    if (n_total >= ((uint64_t)1 << 31)) return fail(SWB_E_UNSUPPORTED, "swb_align: more than 2^31 max cells in one call");
    const uint32_t N = (uint32_t)n_total;
    res->total_cells = N;
    CU(res->f_cell_off.alloc(n_pairs + 1, st));
    CU(res->f_cells.alloc((size_t)N * 2, st));
    CU(res->f_beg.alloc(N, st));
    CU(res->f_len.alloc(N, st));
    CU(res->f_ops_off.alloc((size_t)N + 1, st));
    DevBuf<BatchDesc> d_desc;
    DevBuf<uint64_t> d_pair_tmp, d_pair_sorted;
    DevBuf<uint32_t> d_src_tmp, d_order;
    DevBuf<int64_t> d_words;
    DevBuf<uint8_t> d_tmp;
    CU(d_desc.alloc(descs.size(), st));
    CU(d_pair_tmp.alloc(N, st)); CU(d_pair_sorted.alloc(N, st));
    CU(d_src_tmp.alloc(N, st)); CU(d_order.alloc(N, st));
    CU(d_words.alloc((size_t)N + 1, st));
    const size_t tmp_bytes = assemble_tmp_bytes(N);
    CU(d_tmp.alloc(tmp_bytes, st));
    if (!descs.empty()) CU(cudaMemcpyAsync(d_desc.p, descs.data(), descs.size() * sizeof(BatchDesc), cudaMemcpyHostToDevice, st));
    int pair_bits = 1;
    const uint64_t key_end = keep.p ? 2 * (uint64_t)n_pairs : (uint64_t)n_pairs;    // hits mode: dropped cells sort as p + n_pairs
    while (pair_bits < 64 && ((uint64_t)1 << pair_bits) < std::max<uint64_t>(key_end, 1)) ++pair_bits;
    CU(assemble_sort(d_desc.p, (int)descs.size(), N, n_refs, n_reads, keep.p, d_pair_tmp.p, d_src_tmp.p, d_pair_sorted.p, d_order.p,
                     d_tmp.p, tmp_bytes, pair_bits, st));
    uint32_t NK = N;                          // cells that stay: all of them, or in hits mode those of the hits
    if (keep.p) {
        CU(assemble_kept_count(d_pair_sorted.p, N, (int64_t)n_pairs, ctx->counters.p + 2, st));
        CU(cudaMemcpyAsync(&NK, ctx->counters.p + 2, 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        res->total_cells = NK;
        res->stats[STAT_MAX_CELLS] = NK;
    }
    CU(cudaMemsetAsync(d_words.p + NK, 0, 8, st));
    CU(assemble_gather_cells(d_desc.p, (int)descs.size(), NK, d_order.p, res->f_cells.p, res->f_beg.p, res->f_len.p,
                             d_words.p, res->f_ops_off.p, d_tmp.p, tmp_bytes, st));
    int64_t total_words = 0;
    CU(cudaMemcpyAsync(&total_words, res->f_ops_off.p + NK, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    res->total_words = total_words;
    CU(res->f_ops.alloc((size_t)total_words, st));
    CU(assemble_gather_ops(d_desc.p, (int)descs.size(), NK, d_order.p, res->f_ops_off.p, res->f_ops.p, st));
    CU(assemble_offsets(d_pair_sorted.p, NK, (int64_t)n_pairs, res->f_cell_off.p, res->d_best.p, o_reads, res->f_cells.p, st));
    launches += 8;
    if (keep.p) {
        CU(assemble_hit_cells(d_desc.p, (int)descs.size(), d_pair_sorted.p, d_order.p, N, (int64_t)n_pairs, o_reads, res->f_cell_off.p,
                              res->f_cells.p, res->d_best.p, res->d_hits.p, sel.top_k, st));
        launches += 2;
    }
    if (sel.mode == Selection::MARGIN) {
        CU(assemble_list_cells(res->d_hit_off.p, o_reads, res->d_hit_list.p, res->n_hits, res->f_cell_off.p, res->f_cells.p, st));
        ++launches;
    }
    CU(cudaStreamSynchronize(st));
    res->batches.clear();                     // per-batch buffers go back to the pool
    return SWB_OK;
}

int AlignCall::finish_stats(std::chrono::steady_clock::time_point t_wall0)
{
    CU(timer.add_to(res->stats));
    res->stats[STAT_DEVICE_MS] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_wall0).count();
    res->stats[STAT_LAUNCHES] = launches; res->stats[STAT_CK_BYTES] = ck_bytes; res->stats[STAT_BATCHES] = n_batches;
    return SWB_OK;
}

// the checks of an align call on a reference set handle, before it takes the context
static int check_call(const swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch, int32_t gap,
                      uint32_t flags)
{
    if (rd->rs != rs) return fail(SWB_E_INVALID, "swb_align: reads were encoded against a different reference set");
    if (rs->ctx != ctx || rd->ctx != ctx) return fail(SWB_E_INVALID, "swb_align: handles belong to another context");
    const int64_t strands = (flags & SWB_F_BOTH_STRANDS) ? 2 : 1;
    if (strands * rs->n_refs * rd->n_reads >= ((int64_t)1 << 33)) return fail(SWB_E_UNSUPPORTED, "swb_align: more than 2^33 pairs per call");
    int32_t max_m = 0;
    for (int32_t m : rd->len) max_m = std::max(max_m, m);
    // Java int arithmetic wraps; this engine refuses inputs whose scores could leave int32 instead
    const int64_t big = std::max({std::abs((int64_t)match), std::abs((int64_t)mismatch), std::abs((int64_t)gap)});
    if (big * ((int64_t)max_m + rs->max_len + 2) >= ((int64_t)1 << 30))
        return fail(SWB_E_UNSUPPORTED, "swb_align: |score| * (m + n) could overflow int32");
    return SWB_OK;
}

// One packed set (a whole small set, or one part of a large one): AlignCall::run, then the fetch unless SWB_F_NO_FETCH
static int align_leaf(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                      int32_t gap, uint32_t flags, const Selection &sel, int32_t *ext_scores, int32_t *ext_totals, swb_result **out)
{
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    ResultPtr res = new_result(ctx, rs, rd, flags, sel);
    AlignCall call{ctx, rs, rd, match, mismatch, gap, flags, sel, res.get(), ctx->stream, {ctx, ctx->stream}};
    call.both = (flags & SWB_F_BOTH_STRANDS) != 0;
    call.o_refs = res->n_refs; call.o_reads = res->n_reads;
    int rc = call.run(ext_scores, ext_totals);
    if (rc) return rc;
    swb_result *r = res.release();
    if (!(flags & SWB_F_NO_FETCH) && (rc = swb_result_fetch(r))) { swb_result_free(r); return rc; }
    *out = r;
    return SWB_OK;
}

extern "C" {

namespace {

__global__ void add_base_kernel(int64_t *a, int64_t n, int64_t base)
{
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) a[k] += base;
}

// best = better(best, part's best with its reference index moved to the global numbering): highest score, lowest reference
__global__ void fold_best_kernel(int32_t *best, const int32_t *part, int64_t n_reads, int32_t first, int is_first)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_reads) return;
    int4 b = reinterpret_cast<const int4 *>(part)[q];
    if (b.y >= 0) b.y += first;
    if (!is_first) {
        const int4 a = reinterpret_cast<const int4 *>(best)[q];
        if (a.y >= 0 && (b.y < 0 || a.x >= b.x)) b = a;            // parts come in ascending reference order: ties keep the earlier
    }
    reinterpret_cast<int4 *>(best)[q] = b;
}

// grows a pinned host array, keeping its first `used` bytes (the parts copied so far)
int pin_ensure(swb_ctx *ctx, swb_ctx::PinBuf &b, size_t need, size_t used, size_t want)
{
    if (b.p && b.bytes >= need) return SWB_OK;
    if (used) CU(cudaStreamSynchronize(ctx->stream_copy));
    swb_ctx::PinBuf nb = ctx->pin_get(std::max<size_t>(std::max(need, want), 16));
    if (!nb.p) return fail(SWB_E_NOMEM, "swb_align: pinned host allocation failed");
    if (used && b.p) memcpy(nb.p, b.p, used);
    ctx->pin_put(b);
    b = nb;
    return SWB_OK;
}

// part k of a multi-part result -> its segment of the host arrays, on the copy stream (the compute stream goes on)
int copy_part(swb_result *res, size_t k)
{
    swb_ctx *ctx = res->ctx;
    swb_result *sub = res->subs[k];
    cudaStream_t sc = ctx->stream_copy;
    const size_t S = std::max(res->parts_total, res->subs.size());
    const int64_t first = res->sub_first[k];
    const size_t np_k = (size_t)(sub->n_refs * sub->n_reads), N_k = sub->total_cells;
    const size_t n_pairs = (size_t)(res->n_refs * res->n_reads);
    const size_t cb = (size_t)res->cells_done, wb = (size_t)res->words_done;
    // capacity guess after the first part: the parts hold equal base counts
    const size_t wantN = (size_t)((double)(cb + N_k) * (double)S / (double)(k + 1) * 1.15) + 1024;
    const size_t wantW = (size_t)((double)(wb + (size_t)sub->total_words) * (double)S / (double)(k + 1) * 1.15) + 1024;
    int rc;
    if ((rc = pin_ensure(ctx, res->h_cell_off, (n_pairs + 1) * 8, 0, 0))) return rc;
    if ((rc = pin_ensure(ctx, res->h_cells, (cb + N_k) * 8, cb * 8, wantN * 8))) return rc;
    if ((rc = pin_ensure(ctx, res->h_beg, (cb + N_k) * 4, cb * 4, wantN * 4))) return rc;
    if ((rc = pin_ensure(ctx, res->h_len, (cb + N_k) * 4, cb * 4, wantN * 4))) return rc;
    if ((rc = pin_ensure(ctx, res->h_ops_off, (cb + N_k + 1) * 8, cb * 8, (wantN + 1) * 8))) return rc;
    if ((rc = pin_ensure(ctx, res->h_ops, (wb + (size_t)sub->total_words) * 4, wb * 4, wantW * 4))) return rc;
    cudaEvent_t ev;
    CU(ctx->next_event(&ev));
    CU(cudaEventRecord(ev, ctx->stream));
    CU(cudaStreamWaitEvent(sc, ev, 0));
    if (np_k) {
        if (cb) add_base_kernel<<<grid_for((int64_t)np_k, 256, ctx->sm_count), 256, 0, sc>>>(sub->f_cell_off.p, (int64_t)np_k, (int64_t)cb);
        CU(cudaMemcpyAsync((int64_t *)res->h_cell_off.p + (size_t)first * (size_t)res->n_reads, sub->f_cell_off.p, np_k * 8, cudaMemcpyDeviceToHost, sc));
    }
    if (N_k) {
        if (wb) add_base_kernel<<<grid_for((int64_t)N_k, 256, ctx->sm_count), 256, 0, sc>>>(sub->f_ops_off.p, (int64_t)N_k, (int64_t)wb);
        CU(cudaMemcpyAsync((int32_t *)res->h_cells.p + cb * 2, sub->f_cells.p, N_k * 8, cudaMemcpyDeviceToHost, sc));
        CU(cudaMemcpyAsync((int32_t *)res->h_beg.p + cb, sub->f_beg.p, N_k * 4, cudaMemcpyDeviceToHost, sc));
        CU(cudaMemcpyAsync((int32_t *)res->h_len.p + cb, sub->f_len.p, N_k * 4, cudaMemcpyDeviceToHost, sc));
        CU(cudaMemcpyAsync((int64_t *)res->h_ops_off.p + cb, sub->f_ops_off.p, N_k * 8, cudaMemcpyDeviceToHost, sc));
        if (sub->total_words)
            CU(cudaMemcpyAsync((uint32_t *)res->h_ops.p + wb, sub->f_ops.p, (size_t)sub->total_words * 4, cudaMemcpyDeviceToHost, sc));
    }
    CU(cudaGetLastError());
    res->cells_done += N_k;
    res->words_done += sub->total_words;
    res->sub_copied[k] = 1;
    return SWB_OK;
}

// the arrays that are only complete after the last part, the closing entries, and the host views
int finish_parts_fetch(swb_result *res)
{
    swb_ctx *ctx = res->ctx;
    cudaStream_t sc = ctx->stream_copy;
    const bool full = !(res->flags & SWB_F_SCORES_ONLY);
    const size_t n_pairs = (size_t)(res->n_refs * res->n_reads);
    int rc;
    if (full)
        for (size_t k = 0; k < res->subs.size(); ++k)
            if (!res->sub_copied[k] && (rc = copy_part(res, k))) return rc;
    if ((rc = pin_ensure(ctx, res->h_scores, std::max<size_t>(n_pairs, 1) * 4, 0, 0))) return rc;
    if ((rc = pin_ensure(ctx, res->h_totals, std::max<size_t>((size_t)res->n_refs, 1) * 4, 0, 0))) return rc;
    if ((rc = pin_ensure(ctx, res->h_best, std::max<size_t>((size_t)res->n_reads, 1) * 16, 0, 0))) return rc;
    cudaEvent_t ev;
    CU(ctx->next_event(&ev));
    CU(cudaEventRecord(ev, ctx->stream));
    CU(cudaStreamWaitEvent(sc, ev, 0));
    CU(cudaEventRecord(ctx->ev[0], sc));
    if (n_pairs) CU(cudaMemcpyAsync(res->h_scores.p, res->d_scores.p, n_pairs * 4, cudaMemcpyDeviceToHost, sc));
    if (res->n_refs) CU(cudaMemcpyAsync(res->h_totals.p, res->d_totals.p, (size_t)res->n_refs * 4, cudaMemcpyDeviceToHost, sc));
    if (res->n_reads) CU(cudaMemcpyAsync(res->h_best.p, res->d_best.p, (size_t)res->n_reads * 16, cudaMemcpyDeviceToHost, sc));
    CU(cudaEventRecord(ctx->ev[1], sc));
    CU(cudaStreamSynchronize(sc));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    res->stats[STAT_D2H_MS] = ms;                                 // what was left to copy after the last part's compute
    res->scores = (const int32_t *)res->h_scores.p; res->totals = (const int32_t *)res->h_totals.p;
    res->best = (const int32_t *)res->h_best.p;
    if (full) {
        if ((rc = pin_ensure(ctx, res->h_cell_off, (n_pairs + 1) * 8, 0, 0))) return rc;
        if ((rc = pin_ensure(ctx, res->h_ops_off, ((size_t)res->cells_done + 1) * 8, (size_t)res->cells_done * 8, 0))) return rc;
        ((int64_t *)res->h_cell_off.p)[n_pairs] = (int64_t)res->cells_done;
        ((int64_t *)res->h_ops_off.p)[res->cells_done] = res->words_done;
        res->cell_off = (const int64_t *)res->h_cell_off.p; res->cells = (const int32_t *)res->h_cells.p;
        res->beginnings = (const int32_t *)res->h_beg.p; res->op_lens = (const int32_t *)res->h_len.p;
        res->ops_off = (const int64_t *)res->h_ops_off.p; res->ops = (const uint32_t *)res->h_ops.p;
        res->total_cells = (uint32_t)res->cells_done; res->total_words = res->words_done;
    }
    res->fetched = true;
    return SWB_OK;
}

}  // namespace

}  // extern "C"

static int align_resident(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                          int32_t gap, uint32_t flags, const Selection &sel, swb_result **out)
{
    if (!ctx || !rs || !rd || !out) return fail(SWB_E_INVALID, "swb_align: null argument");
    *out = nullptr;
    if (rs->parent) return fail(SWB_E_INVALID, "swb_align: a part of a reference set is not a handle");
    int rc = check_call(ctx, rs, rd, match, mismatch, gap, flags);
    if (rc) return rc;
    // both strands: the 2n internal reads [reads; rc(reads)] of this call, on the set as one (whole, when it has parts)
    if (flags & SWB_F_BOTH_STRANDS) {
        std::unique_ptr<swb_reads> rd2;
        if ((rc = both_strands_reads(ctx, rs, rd, rd2))) return rc;
        return align_leaf(ctx, rs->parts.empty() ? rs : rs->whole, rd2.get(), match, mismatch, gap, flags, sel, nullptr, nullptr, out);
    }
    if (rs->parts.empty()) return align_leaf(ctx, rs, rd, match, mismatch, gap, flags, sel, nullptr, nullptr, out);
    // a selection also runs on the set as one: its cell arrays are small (nothing to overlap), and the selection is then
    // over all references at once, so no part keeps cells of a pair that a later part displaces from the top k, and a
    // read's best score, and with it the margin's bar, is known over the whole set
    if (rs->whole && ((flags & (SWB_F_NO_FETCH | SWB_F_SCORES_ONLY)) || sel.mode != Selection::NONE))
        return align_leaf(ctx, rs->whole, rd, match, mismatch, gap, flags, sel, nullptr, nullptr, out);
    // ---- a set of several parts: part by part; part k's results cross PCIe while part k + 1 computes -------------
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const auto t_wall0 = std::chrono::steady_clock::now();
    ResultPtr res = new_result(ctx, rs, rd, flags, sel);
    const int64_t n_refs = rs->n_refs, n_reads = rd->n_reads;
    const size_t n_pairs = (size_t)(n_refs * n_reads);
    CU(res->d_scores.alloc(n_pairs, st));
    CU(res->d_totals.alloc((size_t)n_refs, st));
    CU(res->d_best.alloc((size_t)n_reads * 4, st));
    const bool full = !(flags & SWB_F_SCORES_ONLY), fetch_now = !(flags & SWB_F_NO_FETCH);
    const int threads = 256;
    res->parts_total = rs->parts.size();
    for (size_t k = 0; k < rs->parts.size(); ++k) {
        const swb_refset *part = rs->parts[k];
        const int64_t first = rs->part_first[k];
        swb_result *sub = nullptr;
        rc = align_leaf(ctx, part, rd, match, mismatch, gap, flags | SWB_F_NO_FETCH, sel, res->d_scores.p + (size_t)first * (size_t)n_reads,
                        res->d_totals.p + first, &sub);
        if (rc) return rc;
        res->subs.push_back(sub); res->sub_first.push_back(first); res->sub_copied.push_back(0);
        for (Stat x : {STAT_FILL_MS, STAT_LOCATE_MS, STAT_TRACE_MS, STAT_MAX_CELLS, STAT_LAUNCHES, STAT_CK_BYTES, STAT_BATCHES})
            res->stats[x] += sub->stats[x];
        if ((uint64_t)res->cells_done + sub->total_cells >= ((uint64_t)1 << 31) || res->total_cells + (uint64_t)sub->total_cells >= ((uint64_t)1 << 31))
            return fail(SWB_E_UNSUPPORTED, "swb_align: more than 2^31 max cells in one call");
        res->total_cells += sub->total_cells; res->total_words += sub->total_words;
        if (n_reads)
            fold_best_kernel<<<(unsigned)((n_reads + threads - 1) / threads), threads, 0, st>>>(res->d_best.p, sub->d_best.p, n_reads, (int32_t)first, k == 0);
        CU(cudaGetLastError());
        if (fetch_now && full && (rc = copy_part(res.get(), k))) return rc;
    }
    CU(cudaStreamSynchronize(st));
    if (fetch_now && (rc = finish_parts_fetch(res.get()))) return rc;
    res->stats[STAT_DEVICE_MS] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_wall0).count();
    *out = res.release();
    return SWB_OK;
}

int swbh::align_host(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                     int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, const Selection &sel, swb_result **out)
{
    if (!out) return fail(SWB_E_INVALID, "swb_align: out is null");
    *out = nullptr;
    if (!ctx) return fail(SWB_E_INVALID, "swb_align: ctx is null");
    swb_reads *rd = nullptr;
    cudaEvent_t e0, e1;
    CU(cudaSetDevice(ctx->device));
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0, ctx->stream));
    int rc = swb_reads_upload(ctx, rs, n_reads, read_bytes, read_offsets, &rd);
    if (rc) { cudaEventDestroy(e0); cudaEventDestroy(e1); return rc; }
    cudaEventRecord(e1, ctx->stream);
    cudaEventSynchronize(e1);
    float h2d = 0;
    cudaEventElapsedTime(&h2d, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    rc = align_resident(ctx, rs, rd, match, mismatch, gap, flags, sel, out);
    swb_reads_free(rd);
    if (rc == SWB_OK) (*out)->stats[STAT_H2D_MS] = h2d;
    return rc;
}

extern "C" {

int swb_align_resident(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                       int32_t gap, uint32_t flags, swb_result **out)
{
    return align_resident(ctx, rs, rd, match, mismatch, gap, flags, Selection{}, out);
}

int swb_align_resident_hits(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                            int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score, swb_result **out)
{
    const Selection sel{Selection::TOP_K, top_k, min_score};
    if (out) *out = nullptr;
    const int rc = check_selection("swb_align_resident_hits", sel);
    return rc ? rc : align_resident(ctx, rs, rd, match, mismatch, gap, flags, sel, out);
}

int swb_align_resident_all_hits(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                                int32_t gap, uint32_t flags, int32_t min_score, int32_t margin, swb_result **out)
{
    const Selection sel{Selection::MARGIN, 0, min_score, margin};
    if (out) *out = nullptr;
    const int rc = check_selection("swb_align_resident_all_hits", sel);
    return rc ? rc : align_resident(ctx, rs, rd, match, mismatch, gap, flags, sel, out);
}

int swb_align(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
              int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, swb_result **out)
{
    return align_host(ctx, rs, n_reads, read_bytes, read_offsets, match, mismatch, gap, flags, Selection{}, out);
}

int swb_align_hits(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                   int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score, swb_result **out)
{
    const Selection sel{Selection::TOP_K, top_k, min_score};
    if (out) *out = nullptr;
    const int rc = check_selection("swb_align_hits", sel);
    return rc ? rc : align_host(ctx, rs, n_reads, read_bytes, read_offsets, match, mismatch, gap, flags, sel, out);
}

int swb_align_all_hits(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                       int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, int32_t min_score, int32_t margin, swb_result **out)
{
    const Selection sel{Selection::MARGIN, 0, min_score, margin};
    if (out) *out = nullptr;
    const int rc = check_selection("swb_align_all_hits", sel);
    return rc ? rc : align_host(ctx, rs, n_reads, read_bytes, read_offsets, match, mismatch, gap, flags, sel, out);
}

int swb_result_fetch(swb_result *res)
{
    if (!res) return fail(SWB_E_INVALID, "swb_result_fetch: null");
    if (res->fetched) return SWB_OK;
    swb_ctx *ctx = res->ctx;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    if (!res->subs.empty()) return finish_parts_fetch(res);
    cudaStream_t st = ctx->stream;
    CU(cudaEventRecord(ctx->ev[0], st));
    const size_t n_pairs = (size_t)(res->n_refs * res->n_reads);
    const size_t N = res->total_cells;
    const bool full = !(res->flags & SWB_F_SCORES_ONLY);
    // one pinned buffer per array, recycled through the context
    auto pull = [&](const void *dev, size_t bytes, const void **host) -> int {
        swb_ctx::PinBuf b = ctx->pin_get(std::max<size_t>(bytes, 16));
        if (!b.p) return fail(SWB_E_NOMEM, "swb_result_fetch: pinned host allocation failed");
        res->pins.push_back(b);
        *host = b.p;
        if (bytes) CU(cudaMemcpyAsync(b.p, dev, bytes, cudaMemcpyDeviceToHost, st));
        return SWB_OK;
    };
    int rc;
    if ((rc = pull(res->d_scores.p, n_pairs * 4, (const void **)&res->scores))) return rc;
    if ((rc = pull(res->d_totals.p, (size_t)res->n_refs * 4, (const void **)&res->totals))) return rc;
    if ((rc = pull(res->d_best.p, (size_t)res->n_reads * 16, (const void **)&res->best))) return rc;
    if (res->sel.mode == Selection::TOP_K && (rc = pull(res->d_hits.p, (size_t)res->n_reads * res->sel.top_k * 16, (const void **)&res->hits)))
        return rc;
    if (res->sel.mode == Selection::MARGIN) {
        if ((rc = pull(res->d_hit_off.p, ((size_t)res->n_reads + 1) * 8, (const void **)&res->hit_off))) return rc;
        if ((rc = pull(res->d_hit_list.p, (size_t)res->n_hits * 16, (const void **)&res->hit_list))) return rc;
    }
    if (full) {
        if ((rc = pull(res->f_cell_off.p, (n_pairs + 1) * 8, (const void **)&res->cell_off))) return rc;
        if ((rc = pull(res->f_cells.p, N * 8, (const void **)&res->cells))) return rc;
        if ((rc = pull(res->f_beg.p, N * 4, (const void **)&res->beginnings))) return rc;
        if ((rc = pull(res->f_len.p, N * 4, (const void **)&res->op_lens))) return rc;
        if ((rc = pull(res->f_ops_off.p, (N + 1) * 8, (const void **)&res->ops_off))) return rc;
        if ((rc = pull(res->f_ops.p, (size_t)res->total_words * 4, (const void **)&res->ops))) return rc;
    }
    CU(cudaEventRecord(ctx->ev[1], st));
    CU(cudaStreamSynchronize(st));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    res->stats[STAT_D2H_MS] = ms;
    res->fetched = true;
    return SWB_OK;
}

}  // extern "C"
