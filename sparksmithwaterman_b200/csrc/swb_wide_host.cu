// swb_wide_host.cu -- host driver of the int32 wide path (swb_wide.cu): pair batching by
// workspace, band tickets, flag -> locate -> sort -> trace, results appended as BatchOut.
#include "swb_host.h"

namespace swbh {

using namespace swb::wide;

// rows per lane for a read of m rows: the band count times the per-step cost of a band (3 ops per row + ~25 per step)
static int pick_kl(int64_t m)
{
    int best = 0;
    int64_t best_cost = 0;
    for (int k = 0; k < kNumKL; ++k) {
        const int kl = kKLList[k];
        const int64_t bands = (m + (int64_t)WL * kl - 1) / ((int64_t)WL * kl);
        const int64_t cost = bands * (3 * kl + 25);
        if (!best || cost <= best_cost) { best = kl; best_cost = cost; }
    }
    return best;
}

int AlignCall::run_wide_path(const std::vector<int32_t> &reads, bool scores_only, const std::vector<std::vector<int32_t>> *refs_of)
{
    const int64_t n_refs = rs->n_refs, n_reads = rd->n_reads;

    // ---- the wide reads, 16-byte aligned and padded to whole bands (0xFE: matches nothing) ----------------
    {
        std::vector<int64_t> rpad_off((size_t)n_reads, 0), rpad_len(reads.size());
        int64_t total = 0, max_len = 0;
        for (size_t k = 0; k < reads.size(); ++k) {
            const int64_t m = rd->len[(size_t)reads[k]];
            const int64_t len = ((m + 1023) / 1024) * 1024;
            rpad_off[(size_t)reads[k]] = total; rpad_len[k] = len;
            total += len; max_len = std::max(max_len, len);
        }
        CU(ctx->w_rpad.reserve((size_t)total + 16, st));
        CU(ctx->w_rpad_off.reserve((size_t)n_reads, st));
        CU(ctx->w_rpad_len.reserve(reads.size(), st));
        CU(ctx->w_wreads.reserve(reads.size(), st));
        CU(cudaMemcpyAsync(ctx->w_rpad_off.p, rpad_off.data(), (size_t)n_reads * 8, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(ctx->w_rpad_len.p, rpad_len.data(), reads.size() * 8, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(ctx->w_wreads.p, reads.data(), reads.size() * 4, cudaMemcpyHostToDevice, st));
        CU(launch_wide_pad_reads(rd->codes.p, rd->off.p, ctx->w_wreads.p, (int)reads.size(), ctx->w_rpad_off.p,
                                 ctx->w_rpad_len.p, ctx->w_rpad.p, max_len, st));
        ++launches;
        CU(cudaStreamSynchronize(st));      // the host tables above are locals
    }

    for (int kc = 0; kc < kNumKL; ++kc) {
    const int KL = kKLList[kc];
    const int64_t BH = (int64_t)WL * KL, RW = wide_rw(KL);
    // all (read, ref) pairs of this rows-per-lane class with a non-empty matrix, read-major
    std::vector<int32_t> pr, pq;
    for (size_t x = 0; x < reads.size(); ++x) {
        const int32_t q = reads[x];
        if (pick_kl(rd->len[(size_t)q]) != KL) continue;
        if (refs_of) {
            for (int32_t r : (*refs_of)[x])
                if (rs->len_orig[(size_t)r] > 0) { pr.push_back(r); pq.push_back(q); }
            continue;
        }
        for (int64_t r = 0; r < n_refs; ++r)
            if (rs->len_orig[(size_t)r] > 0) { pr.push_back((int32_t)r); pq.push_back(q); }
    }
    const size_t total_pairs = pr.size();
    auto pair_bytes = [&](size_t k) -> int64_t {
        const int64_t n = rs->len_orig[(size_t)pr[k]], m = rd->len[(size_t)pq[k]];
        const int64_t bands = (m + BH - 1) / BH, nb = (n + WL - 1 + WCB - 1) / WCB;
        return bands * nb * (WL * (RW + 1) * 4 + WCB * 4) + bands * 4;
    };
    size_t k0 = 0;
    while (k0 < total_pairs) {
        // ---- next batch: as many pairs as the workspace holds ---------------------------------
        size_t k1 = k0;
        int64_t bytes = 0;
        while (k1 < total_pairs && k1 - k0 < (size_t)((1 << 21) - 1)) {
            const int64_t b = pair_bytes(k1);
            if (k1 > k0 && bytes + b > ctx->ws_bytes) break;
            bytes += b; ++k1;
        }
        const int np = (int)(k1 - k0);
        ++n_batches;
        ck_bytes += (double)bytes;
        std::vector<int64_t> band_off((size_t)np + 1), blk_off((size_t)np + 1), brow_off((size_t)np + 1);
        std::vector<int2> items;
        int64_t nbands = 0, nblk = 0;
        int max_bands = 0, m_max = 0, n_max = 0;
        for (int k = 0; k < np; ++k) {
            const int64_t n = rs->len_orig[(size_t)pr[k0 + k]], m = rd->len[(size_t)pq[k0 + k]];
            const int64_t bands = (m + BH - 1) / BH, nb = (n + WL - 1 + WCB - 1) / WCB;
            band_off[(size_t)k] = nbands; blk_off[(size_t)k] = nblk; brow_off[(size_t)k] = nblk * WCB;
            nbands += bands; nblk += bands * nb;
            max_bands = std::max<int>(max_bands, (int)bands);
            m_max = std::max<int>(m_max, (int)m); n_max = std::max<int>(n_max, (int)n);
        }
        band_off[(size_t)np] = nbands; blk_off[(size_t)np] = nblk; brow_off[(size_t)np] = nblk * WCB;
        // tickets in (band, pair) order: a warp only ever waits for a lower ticket
        items.reserve((size_t)nbands);
        for (int b = 0; b < max_bands; ++b)
            for (int k = 0; k < np; ++k)
                if (b < band_off[(size_t)k + 1] - band_off[(size_t)k]) items.push_back(make_int2(k, b));

        CU(ctx->w_pair_ref.reserve((size_t)np, st));
        CU(ctx->w_pair_read.reserve((size_t)np, st));
        CU(ctx->w_band_off.reserve((size_t)np + 1, st));
        CU(ctx->w_blk_off.reserve((size_t)np + 1, st));
        CU(ctx->w_brow_off.reserve((size_t)np + 1, st));
        CU(ctx->w_items.reserve(items.size(), st));
        CU(ctx->w_brow.reserve((size_t)nblk * WCB, st));
        CU(ctx->w_rec.reserve((size_t)nblk * WL * RW, st));
        CU(ctx->w_tmx.reserve((size_t)nblk * WL, st));
        CU(ctx->counters.reserve(16, st));
        CU(cudaMemcpyAsync(ctx->w_pair_ref.p, pr.data() + k0, (size_t)np * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(ctx->w_pair_read.p, pq.data() + k0, (size_t)np * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(ctx->w_band_off.p, band_off.data(), band_off.size() * 8, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(ctx->w_blk_off.p, blk_off.data(), blk_off.size() * 8, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(ctx->w_brow_off.p, brow_off.data(), brow_off.size() * 8, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(ctx->w_items.p, items.data(), items.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
        if (max_bands > 1) CU(cudaMemsetAsync(ctx->w_brow.p, 0xFF, (size_t)nblk * WCB * 4, st));   // -1: not written yet

        WideParams P;
        P.n_pairs = np; P.pair_ref = ctx->w_pair_ref.p; P.pair_read = ctx->w_pair_read.p;
        P.ref_codes = rs->codes8.p; P.ref_off = rs->off8.p;
        P.rpad = ctx->w_rpad.p; P.rpad_off = ctx->w_rpad_off.p; P.read_off = rd->off.p;
        P.match = match; P.mismatch = mismatch; P.gap = gap; P.n_reads = n_reads; P.n_symbols = rs->n_symbols; P.tie_gt = (flags & SWB_F_TIE_GT) ? 1 : 0;
        P.band_off = ctx->w_band_off.p; P.blk_off = ctx->w_blk_off.p; P.brow_off = ctx->w_brow_off.p;
        P.brow = ctx->w_brow.p; P.rec = ctx->w_rec.p; P.tmx = ctx->w_tmx.p;
        P.scores = res->d_scores.p;
        uint32_t *d_ntasks = ctx->counters.p, *d_ncells = ctx->counters.p + 1, *d_ticket = ctx->counters.p + 2;

        CU(timer.begin(STAT_FILL_MS));
        CU(launch_wide_fill(KL, P, ctx->w_items.p, (int)items.size(), d_ticket, ctx->sm_count, st));
        ++launches;
        CU(timer.end());
        if (scores_only) { CU(cudaStreamSynchronize(st)); k0 = k1; continue; }

        CU(timer.begin(STAT_LOCATE_MS));
        uint32_t cap_tasks = (uint32_t)std::min<int64_t>((int64_t)np * 4 + 4096, (int64_t)1 << 30);
        uint32_t cap_cells = cap_tasks;
        uint32_t h_counts[2] = {0, 0};
        for (int attempt = 0; attempt < 3; ++attempt) {
            CU(ctx->w_tasks.reserve(cap_tasks, st));
            CU(ctx->keys_tmp.reserve(cap_cells, st));
            CU(cudaMemsetAsync(ctx->counters.p, 0, 8, st));
            CU(launch_wide_flag(P, nblk, ctx->w_tasks.p, cap_tasks, d_ntasks, ctx->sm_count, st));
            CU(launch_wide_locate(KL, P, ctx->w_tasks.p, d_ntasks, cap_tasks, ctx->keys_tmp.p, cap_cells, d_ncells,
                                  ctx->sm_count, st));
            launches += 2;
            CU(cudaMemcpyAsync(h_counts, ctx->counters.p, 8, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            if (h_counts[0] <= cap_tasks && h_counts[1] <= cap_cells) break;
            if (attempt == 2) return fail(SWB_E_NOMEM, "swb_align: max-cell list did not fit after two retries");
            cap_tasks = std::max(cap_tasks, h_counts[0]);
            cap_cells = std::max(cap_cells, h_counts[1]);
        }
        const uint32_t n_cells = h_counts[1];
        BatchOut bo;
        bo.wide = true; bo.n_cells = n_cells;
        bo.wide_pair_p.resize((size_t)np);
        for (int k = 0; k < np; ++k) bo.wide_pair_p[(size_t)k] = (int64_t)pr[k0 + k] * n_reads + pq[k0 + k];
        CU(bo.d_pair_map.alloc((size_t)np, st));
        CU(cudaMemcpyAsync(bo.d_pair_map.p, bo.wide_pair_p.data(), (size_t)np * 8, cudaMemcpyHostToDevice, st));
        CU(bo.keys.alloc(n_cells, st));
        const size_t tmp_bytes = sort_keys_tmp_bytes(n_cells);
        CU(ctx->sort_tmp.reserve(tmp_bytes, st));
        CU(sort_keys(ctx->keys_tmp.p, bo.keys.p, n_cells, ctx->sort_tmp.p, tmp_bytes, st));
        launches += 4;
        CU(timer.end());

        CU(timer.begin(STAT_TRACE_MS));
        // longest alignment of a positive-score path: m rows + the deletions its score can pay for
        const int64_t big = std::max({match, mismatch, 0});
        int64_t lmax = (int64_t)m_max + n_max;
        if (gap < 0) lmax = std::min<int64_t>(lmax, (int64_t)m_max + (big * m_max) / (-(int64_t)gap) + 1);
        bo.ops_stride = (lmax + 15) / 16 + 1;
        CU(bo.beg.alloc(n_cells, st));
        CU(bo.oplen.alloc(n_cells, st));
        CU(bo.ops.alloc((size_t)n_cells * (size_t)bo.ops_stride, st));
        P.mail = nullptr; P.mail_latest = nullptr; P.mail_stride = 0; P.pipe_c = 1;
        if (n_cells > 0 && n_cells <= 65536u) {
            // few, long walks: the pipelined CTA-wide traceback (swb_wide.cu) passes the walker's state from round to round
            // through tokens in global memory; one round = 32 lane-rows of KL rows
            const int64_t stride = (int64_t)m_max / ((int64_t)KL * 16) + 4;      // a round is 32 or 16 lane-rows
            const size_t words = (size_t)n_cells * (size_t)stride * 8 + n_cells;
            CU(ctx->w_mail.reserve(words, st));
            CU(cudaMemsetAsync(ctx->w_mail.p, 0, words * 4, st));
            P.mail = ctx->w_mail.p; P.mail_latest = ctx->w_mail.p + (size_t)n_cells * (size_t)stride * 8; P.mail_stride = (int32_t)stride;
        }
        CU(launch_wide_trace(KL, P, bo.keys.p, n_cells, bo.beg.p, bo.oplen.p, bo.ops.p, bo.ops_stride, ctx->sm_count, st));
        ++launches;
        CU(timer.end());
        CU(cudaStreamSynchronize(st));      // the host tables of this batch are reused by the next one
        res->stats[STAT_MAX_CELLS] += n_cells;
        res->batches.push_back(std::move(bo));
        k0 = k1;
    }
    }
    return SWB_OK;
}

}  // namespace swbh
