// swb_queue.cu -- the context's SUBMISSION QUEUE: single-pair calls from many host threads, coalesced.
//
// The reference's unchanged driver issues `new SmithWaterman.OptAlignments().call({ref, read}, scores, types)` once per
// pair from N Spark task threads (Distribution.java:419-426, one MapRef.call per reference, references spread over the
// threads).  Served one by one through swb_refset_load(1) + swb_align(1) every such call is a full launch sequence
// (measured: 660 us per pair, no gain from more threads: the context is one device).  swb_align_pair instead parks
// the request in a queue; ONE of the waiting threads (the leader) takes every queued request with the same scores and
// flags, loads their distinct references as one set and their distinct reads as one batch, runs ONE align sequence
// (references x reads; the requested pairs are a subset of that cross product) and hands every waiter a 1 x 1 result
// cut out of the batch result.  The first caller of an idle context runs alone, whatever arrives while the device is
// busy forms the next batch, and a short bounded linger (below) lets N threads settle into batches of N pairs.
#include "swb_host.h"

#include <chrono>
#include <condition_variable>
#include <deque>
#include <string_view>
#include <unordered_map>

using namespace swbh;

namespace {

struct PairReq {
    const char *ref = nullptr, *read = nullptr;
    int64_t ref_len = 0, read_len = 0;
    int32_t match = 0, mismatch = 0, gap = 0;
    uint32_t flags = 0;
    swb_result *res = nullptr;
    int rc = SWB_OK;
    std::string err;
    bool done = false;
    bool same_job(const PairReq &o) const { return match == o.match && mismatch == o.mismatch && gap == o.gap && flags == o.flags; }
};

constexpr size_t MAX_COALESCED = 256;        // requests per batch; the cross product stays <= 65,536 pairs

struct SubmitQueue {
    std::mutex mu;
    std::condition_variable cv;                 // a batch finished
    std::condition_variable cv_arrive;          // a request was queued (the lingering leader listens)
    std::deque<PairReq *> pending;
    bool leader_active = false;
    size_t callers_hint = 1;                    // how many threads were inside swb_align_pair when the last batch ended
    int64_t calls = 0, batches = 0, largest = 0;
};

// A leader that finds fewer requests than there were concurrent callers a moment ago LINGERS for the rest: the callers
// of the batch that just finished are on their way back (they only unmarshal), and one launch sequence for all of them
// beats two for a half each (the sequence is latency-bound: ~1 ms whether it carries 1 pair or 100).  Bounded by
// SWB_QUEUE_LINGER_US (default 200); the hint decays by a quarter per batch when callers go away.
int linger_us()
{
    static const int v = getenv("SWB_QUEUE_LINGER_US") ? atoi(getenv("SWB_QUEUE_LINGER_US")) : 200;
    return v;
}

// one queue per context, created on first use and kept until the process ends (a context's address may be reused
// after swb_destroy: the queue is empty by then, which is all a new context needs)
SubmitQueue &queue_of(swb_ctx *ctx)
{
    static std::mutex mu;
    static std::unordered_map<swb_ctx *, std::unique_ptr<SubmitQueue>> all;
    std::lock_guard<std::mutex> lk(mu);
    auto &q = all[ctx];
    if (!q) q.reset(new SubmitQueue());
    return *q;
}

// the 1 x 1 result of pair (r, q) of `big` (fetched, host arrays): own storage, every accessor of swb200.h applies
swb_result *cut_pair(swb_ctx *ctx, const swb_result *big, int64_t r, int64_t q, int64_t ref_len, int64_t read_len, size_t coalesced)
{
    const bool full = !(big->flags & SWB_F_SCORES_ONLY);
    const int64_t p = r * big->n_reads + q;
    const int32_t score = big->scores[(size_t)p];
    const int64_t c0 = full ? big->cell_off[(size_t)p] : 0, c1 = full ? big->cell_off[(size_t)p + 1] : 0;
    const int64_t n = c1 - c0;
    const int64_t w0 = (full && n) ? big->ops_off[(size_t)c0] : 0, w1 = (full && n) ? big->ops_off[(size_t)c1] : 0;
    std::unique_ptr<swb_result> res(new swb_result());
    res->ctx = ctx; res->n_refs = 1; res->n_reads = 1; res->flags = big->flags & ~SWB_F_NO_FETCH;
    res->ref_len.assign(1, (int32_t)ref_len); res->read_len.assign(1, (int32_t)read_len);
    // layout of the arena (8-byte aligned pieces first)
    const size_t n_i64 = 2 + (size_t)n + 1, n_i32 = 1 + 1 + 4 + (size_t)n * 4, n_u32 = (size_t)(w1 - w0);
    res->own.assign(n_i64 * 8 + n_i32 * 4 + n_u32 * 4 + 8, 0);
    int64_t *i64 = reinterpret_cast<int64_t *>(res->own.data());
    int32_t *i32 = reinterpret_cast<int32_t *>(i64 + n_i64);
    uint32_t *u32 = reinterpret_cast<uint32_t *>(i32 + n_i32);
    int64_t *cell_off = i64, *ops_off = i64 + 2;
    int32_t *scores = i32, *totals = i32 + 1, *best = i32 + 2, *cells = i32 + 6, *beg = cells + 2 * n, *len = beg + n;
    scores[0] = score; totals[0] = score;
    cell_off[0] = 0; cell_off[1] = n;
    for (int64_t k = 0; k < n; ++k) {
        cells[2 * k] = big->cells[2 * (size_t)(c0 + k)]; cells[2 * k + 1] = big->cells[2 * (size_t)(c0 + k) + 1];
        beg[k] = big->beginnings[(size_t)(c0 + k)]; len[k] = big->op_lens[(size_t)(c0 + k)];
        ops_off[k] = big->ops_off[(size_t)(c0 + k)] - w0;
    }
    ops_off[n] = w1 - w0;
    if (n_u32) memcpy(u32, big->ops + w0, n_u32 * 4);
    best[0] = score; best[1] = 0; best[2] = n ? cells[0] : 0; best[3] = n ? cells[1] : 0;
    res->scores = scores; res->totals = totals; res->best = best;
    if (full) {
        res->cell_off = cell_off; res->cells = cells; res->beginnings = beg; res->op_lens = len; res->ops_off = ops_off; res->ops = u32;
        res->total_cells = (uint32_t)n; res->total_words = w1 - w0;
    }
    for (int k = 0; k < STAT_COUNT; ++k) res->stats[k] = big->stats[k];  // timings of the batch the pair rode in
    res->stats[STAT_CELLS] = (double)ref_len * (double)read_len; res->stats[STAT_PAIRS] = 1; res->stats[STAT_MAX_CELLS] = (double)n;
    res->stats[STAT_BATCHES] = (double)coalesced;                         // requests served by that batch
    res->fetched = true;
    ctx->live.fetch_add(1);
    return res.release();
}

// one batch: distinct references x distinct reads through the ordinary entry points
void run_batch(swb_ctx *ctx, const std::vector<PairReq *> &batch)
{
    std::unordered_map<std::string_view, int64_t> ref_ix, read_ix;
    std::vector<std::string_view> refs, reads;
    std::vector<int64_t> rq_ref(batch.size()), rq_read(batch.size());
    for (size_t k = 0; k < batch.size(); ++k) {
        const PairReq &rq = *batch[k];
        const std::string_view rv(rq.ref ? rq.ref : "", (size_t)rq.ref_len), qv(rq.read ? rq.read : "", (size_t)rq.read_len);
        auto a = ref_ix.emplace(rv, (int64_t)refs.size());
        if (a.second) refs.push_back(rv);
        rq_ref[k] = a.first->second;
        auto b = read_ix.emplace(qv, (int64_t)reads.size());
        if (b.second) reads.push_back(qv);
        rq_read[k] = b.first->second;
    }
    auto pack = [](const std::vector<std::string_view> &v, std::string &bytes, std::vector<int64_t> &off) {
        off.assign(1, 0);
        for (const auto &s : v) { bytes.append(s); off.push_back((int64_t)bytes.size()); }
        if (bytes.empty()) bytes.push_back('\0');                          // a non-null pointer for an all-empty batch
    };
    std::string ref_bytes, read_bytes;
    std::vector<int64_t> ref_off, read_off;
    pack(refs, ref_bytes, ref_off);
    pack(reads, read_bytes, read_off);
    const PairReq &head = *batch[0];
    swb_refset *rs = nullptr;
    swb_result *big = nullptr;
    int rc = swb_refset_load(ctx, (int64_t)refs.size(), ref_bytes.data(), ref_off.data(), &rs);
    if (rc == SWB_OK)
        rc = swb_align(ctx, rs, (int64_t)reads.size(), read_bytes.data(), read_off.data(), head.match, head.mismatch, head.gap,
                       head.flags & ~SWB_F_NO_FETCH, &big);
    if (rc != SWB_OK) {
        const std::string err = last_error();
        if (rs) swb_refset_free(rs);
        if (batch.size() > 1) {
            // one request's input may be what the engine refused (a non-ASCII byte, an unsupported score range): the
            // others must not fail with it -> every request on its own
            for (PairReq *rq : batch) run_batch(ctx, std::vector<PairReq *>{rq});
            return;
        }
        batch[0]->rc = rc; batch[0]->err = err;
        return;
    }
    for (size_t k = 0; k < batch.size(); ++k)
        batch[k]->res = cut_pair(ctx, big, rq_ref[k], rq_read[k], batch[k]->ref_len, batch[k]->read_len, batch.size());
    swb_result_free(big);
    swb_refset_free(rs);
}

}  // namespace

extern "C" {

int swb_align_pair(swb_ctx *ctx, const char *ref, int64_t ref_len, const char *read, int64_t read_len, int32_t match,
                   int32_t mismatch, int32_t gap, uint32_t flags, swb_result **out)
{
    if (!out) return fail(SWB_E_INVALID, "swb_align_pair: out is null");
    *out = nullptr;
    if (!ctx) return fail(SWB_E_INVALID, "swb_align_pair: ctx is null");
    if (ref_len < 0 || read_len < 0 || (ref_len > 0 && !ref) || (read_len > 0 && !read))
        return fail(SWB_E_INVALID, "swb_align_pair: bad sequence argument");
    if (flags & SWB_F_BOTH_STRANDS) return fail(SWB_E_INVALID, "swb_align_pair: SWB_F_BOTH_STRANDS is not accepted here");
    PairReq rq;
    rq.ref = ref; rq.ref_len = ref_len; rq.read = read; rq.read_len = read_len;
    rq.match = match; rq.mismatch = mismatch; rq.gap = gap; rq.flags = flags & ~SWB_F_NO_FETCH;
    SubmitQueue &q = queue_of(ctx);
    std::unique_lock<std::mutex> lk(q.mu);
    q.pending.push_back(&rq);
    ++q.calls;
    q.cv_arrive.notify_one();
    while (!rq.done) {
        if (q.leader_active) { q.cv.wait(lk); continue; }
        // lead: the oldest request and everything queued that belongs to the same job
        q.leader_active = true;
        const size_t want = std::min(q.callers_hint, MAX_COALESCED);
        if (q.pending.size() < want && linger_us() > 0)
            q.cv_arrive.wait_for(lk, std::chrono::microseconds(linger_us()), [&] { return q.pending.size() >= want; });
        std::vector<PairReq *> batch;
        const PairReq &head = *q.pending.front();
        for (auto it = q.pending.begin(); it != q.pending.end() && batch.size() < MAX_COALESCED;) {
            if ((*it)->same_job(head)) { batch.push_back(*it); it = q.pending.erase(it); } else ++it;
        }
        ++q.batches;
        q.largest = std::max<int64_t>(q.largest, (int64_t)batch.size());
        lk.unlock();
        run_batch(ctx, batch);
        lk.lock();
        for (PairReq *b : batch) b->done = true;
        q.callers_hint = std::max(batch.size() + q.pending.size(), q.callers_hint - (q.callers_hint + 3) / 4);
        if (q.callers_hint < 1) q.callers_hint = 1;
        q.leader_active = false;
        q.cv.notify_all();
    }
    lk.unlock();
    if (rq.rc != SWB_OK) return fail(rq.rc, rq.err);                      // the message lands in THIS thread's last error
    *out = rq.res;
    return SWB_OK;
}

int swb_queue_stats(swb_ctx *ctx, int64_t *out, int n)
{
    if (!ctx || !out) return fail(SWB_E_INVALID, "swb_queue_stats: null");
    SubmitQueue &q = queue_of(ctx);
    std::lock_guard<std::mutex> lk(q.mu);
    const int64_t v[3] = {q.calls, q.batches, q.largest};
    for (int k = 0; k < n && k < 3; ++k) out[k] = v[k];
    return SWB_OK;
}

}  // extern "C"
