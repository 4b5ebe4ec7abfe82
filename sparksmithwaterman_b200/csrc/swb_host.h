// swb_host.h -- host-side structures of libswb200 shared by swb_api.cu, swb_align.cu and swb_wide_host.cu.
#pragma once
#include "swb_internal.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <map>
#include <tuple>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <numeric>

namespace swbh {
using namespace swb;

std::string &last_error();
inline int fail(int code, const std::string &msg) { last_error() = msg; return code; }
inline int cuda_fail(cudaError_t e, const char *what)
{
    last_error() = std::string(what) + ": " + cudaGetErrorString(e);
    return SWB_E_CUDA;
}
#define CU(x)                                                                  \
    do {                                                                       \
        cudaError_t e_ = (x);                                                  \
        if (e_ != cudaSuccess) return swbh::cuda_fail(e_, #x);                 \
    } while (0)

// Large device blocks (>= 4 MiB) are recycled by EXACT size per stream, outside the CUDA pool: the stream-ordered
// pool splits and merges its free blocks, so a 730 MB result array released by one call is carved up by the next
// call's smaller requests and the pool has to be reshaped when the 730 MB request comes back -- measured on B200 as
// single cudaMallocAsync calls of 0.2 - 1.4 s, 15 % of a 100,000-read job.  A block cached here is handed out again
// only for the same (rounded) size on the same stream, which keeps stream order: whatever still uses it was issued
// on that stream before.  The cache is bounded; overflow goes back to the pool.
struct BlockCache {
    std::mutex mu;
    std::multimap<std::pair<cudaStream_t, size_t>, void *> free_blocks;
    size_t cached = 0;
    static constexpr size_t MIN_BYTES = (size_t)4 << 20, MAX_CACHED = (size_t)24 << 30;
    static BlockCache &get() { static BlockCache c; return c; }
    void *take(cudaStream_t st, size_t bytes)
    {
        std::lock_guard<std::mutex> lk(mu);
        auto it = free_blocks.find({st, bytes});
        if (it == free_blocks.end()) return nullptr;
        void *p = it->second;
        free_blocks.erase(it);
        cached -= bytes;
        return p;
    }
    bool give(cudaStream_t st, size_t bytes, void *p)
    {
        std::lock_guard<std::mutex> lk(mu);
        if (cached + bytes > MAX_CACHED) return false;
        free_blocks.emplace(std::make_pair(st, bytes), p);
        cached += bytes;
        return true;
    }
    // the pool ran dry: hand this stream's cached blocks back (stream-ordered), the caller retries its allocation
    size_t spill(cudaStream_t st)
    {
        std::lock_guard<std::mutex> lk(mu);
        size_t freed = 0;
        for (auto it = free_blocks.begin(); it != free_blocks.end();)
            if (it->first.first == st) { cudaFreeAsync(it->second, st); freed += it->first.second; cached -= it->first.second; it = free_blocks.erase(it); } else ++it;
        return freed;
    }
    // a context goes away: its streams' blocks return to the pool (the caller has synchronised the streams)
    void purge(cudaStream_t st)
    {
        std::lock_guard<std::mutex> lk(mu);
        for (auto it = free_blocks.begin(); it != free_blocks.end();)
            if (it->first.first == st) { cudaFree(it->second); cached -= it->first.second; it = free_blocks.erase(it); } else ++it;
    }
};

// Device buffer from the stream-ordered pool (cudaMallocAsync): allocation and release are
// ordered on the engine's stream and reuse pool memory, so the align loop never hits the
// synchronising cudaMalloc/cudaFree.
template <class T> struct DevBuf {
    T *p = nullptr; size_t n = 0; cudaStream_t st = nullptr;
    bool owned = true;                          // false: a view into somebody else's allocation
    size_t cap_bytes = 0;                       // what was asked from the allocator (size class)
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(o.p), n(o.n), st(o.st), owned(o.owned), cap_bytes(o.cap_bytes) { o.p = nullptr; o.n = 0; o.owned = true; o.cap_bytes = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept
    {
        if (this != &o) { release(); p = o.p; n = o.n; st = o.st; owned = o.owned; cap_bytes = o.cap_bytes; o.p = nullptr; o.n = 0; o.owned = true; o.cap_bytes = 0; }
        return *this;
    }
    ~DevBuf() { release(); }
    void release()
    {
        if (p && owned && !(cap_bytes >= BlockCache::MIN_BYTES && BlockCache::get().give(st, cap_bytes, p))) cudaFreeAsync(p, st);
        p = nullptr; n = 0; owned = true; cap_bytes = 0;
    }
    void view(T *ptr, size_t count) { release(); p = ptr; n = count; owned = false; }
    cudaError_t alloc(size_t count, cudaStream_t stream)
    {
        release();
        if (count == 0) count = 1;
        st = stream;
        // size classes (eight per octave, <= 12.5 % over) above 1 MiB: the arrays of consecutive calls differ by a
        // percent or so (max-cell counts) and land in the same class
        size_t bytes = count * sizeof(T);
        if (bytes >= ((size_t)1 << 20)) {
            size_t step = (size_t)1 << 17;
            while ((step << 4) <= bytes) step <<= 1;               // step = 2^(floor(log2 bytes) - 3)
            bytes = (bytes + step - 1) / step * step;
        }
        cap_bytes = bytes;
        if (bytes >= BlockCache::MIN_BYTES) {
            p = static_cast<T *>(BlockCache::get().take(stream, bytes));
            if (p) { n = count; return cudaSuccess; }
        }
        cudaError_t e = cudaMallocAsync(&p, bytes, stream);
        if (e == cudaErrorMemoryAllocation && BlockCache::get().spill(stream) > 0) {
            cudaGetLastError();
            e = cudaMallocAsync(&p, bytes, stream);                // once more with the cached blocks back in the pool
        }
        if (e == cudaSuccess) n = count; else { p = nullptr; cap_bytes = 0; }
        return e;
    }
    cudaError_t reserve(size_t count, cudaStream_t stream) { return n >= count && p ? cudaSuccess : alloc(count + count / 8, stream); }
};

inline int upper(int c) { return (c >= 'a' && c <= 'z') ? c - 32 : c; }

// Which pairs of a call are traced (include/swb200.h): all of them (swb_align), each read's top_k best pairs with score
// >= min_score (hits mode, swb_align_hits), or each read's pairs with score >= max(min_score, read's best - margin)
// (all-hits mode, swb_align_all_hits).  The entry points build it and check it once (check_selection).
struct Selection {
    enum Mode { NONE, TOP_K, MARGIN } mode = NONE;
    int32_t top_k = 0, min_score = 1, margin = 0;
};

// the argument rules of the selecting entry points; `who` names the entry in the message
inline int check_selection(const char *who, const Selection &sel)
{
    if (sel.mode == Selection::TOP_K && (sel.top_k < 1 || sel.top_k > 32)) return fail(SWB_E_INVALID, std::string(who) + ": top_k must be 1 .. 32");
    if (sel.mode != Selection::NONE && sel.min_score < 1) return fail(SWB_E_INVALID, std::string(who) + ": min_score must be >= 1");
    if (sel.mode == Selection::MARGIN && sel.margin < 0) return fail(SWB_E_INVALID, std::string(who) + ": margin must be >= 0");
    return SWB_OK;
}

// grid of a grid-stride loop over n elements
inline int grid_for(int64_t n, int threads, int sm_count)
{
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + threads - 1) / threads, (int64_t)sm_count * 16));
}

// the entries of swb_result_stats (include/swb200.h, engine.STAT_NAMES)
enum Stat {
    STAT_H2D_MS, STAT_FILL_MS, STAT_LOCATE_MS, STAT_TRACE_MS, STAT_D2H_MS, STAT_DEVICE_MS, STAT_CELLS, STAT_PAIRS,
    STAT_MAX_CELLS, STAT_LAUNCHES, STAT_CK_BYTES, STAT_BATCHES, STAT_SELECT_MS, STAT_COUNT
};

}  // namespace swbh

using swbh::DevBuf;
using swb::TileTask;
using swb::WideTask;

struct swb_ctx {
    int device = 0;
    int sm_count = 0;
    int64_t ws_bytes = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream_copy = nullptr;         // results of reference part k cross PCIe while part k+1 computes
    cudaEvent_t ev[2] = {nullptr, nullptr};
    std::recursive_mutex mu;
    std::atomic<int> live{0};                   // handles (refsets, read batches, results) that still point here
    std::atomic<bool> dying{false};             // swb_destroy was called while handles were alive: the last free destroys
    // grow-only scratch reused by every align call on this context
    DevBuf<uint32_t> ck, tmx, counters;         // checkpoint workspace, tile maxima, device counters of one batch
    DevBuf<int32_t> rp;                         // read pairs of one batch
    DevBuf<TileTask> tasks;
    DevBuf<uint8_t> task_hits;                 // per candidate tile: exact maximum + buffered cells (locate scan -> emit)
    DevBuf<uint64_t> keys_tmp;
    DevBuf<uint8_t> sort_tmp;
    // wide (int32, long-pair) path scratch
    DevBuf<int32_t> w_brow, w_rec, w_tmx, w_pair_ref, w_pair_read, w_wreads;
    DevBuf<uint8_t> w_rpad;                     // wide reads, aligned + padded (0xFE) to whole bands
    DevBuf<int64_t> w_rpad_off, w_rpad_len;
    DevBuf<int32_t> w_mail;                     // tokens of the pipelined CTA-wide traceback
    DevBuf<int64_t> w_band_off, w_blk_off, w_brow_off;
    DevBuf<int2> w_items;
    DevBuf<WideTask> w_tasks;
    // hits mode (swb_hits.cu): partial top-k lists, the selection bits of one batch
    DevBuf<uint64_t> hit_tmp;
    DevBuf<uint32_t> hit_sel;
    DevBuf<uint64_t> margin_best;               // all-hits mode: best key per slot of one selection
    // pinned host buffers, recycled between results (cudaHostAlloc is slow; D2H into pageable memory too)
    struct PinBuf { void *p = nullptr; size_t bytes = 0; };
    std::vector<PinBuf> pin_free;
    // Pinned host buffers come in power-of-two size classes (>= 64 KiB): a step whose result is a few percent larger
    // than the previous one's finds its buffers in the pool instead of paying cudaHostAlloc (milliseconds per 100 MB).
    static size_t pin_class(size_t bytes)
    {
        size_t c = (size_t)64 << 10;
        while (c < bytes) c <<= 1;
        return c;
    }
    PinBuf pin_get(size_t bytes)
    {
        const size_t want = pin_class(bytes);
        size_t best = pin_free.size();
        for (size_t k = 0; k < pin_free.size(); ++k)
            if (pin_free[k].bytes >= want && (best == pin_free.size() || pin_free[k].bytes < pin_free[best].bytes)) best = k;
        if (best != pin_free.size()) { PinBuf b = pin_free[best]; pin_free.erase(pin_free.begin() + best); return b; }
        PinBuf b;
        b.bytes = want;
        if (cudaHostAlloc(&b.p, b.bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); b.p = nullptr; b.bytes = 0; }
        return b;
    }
    void pin_put(PinBuf b) { if (b.p) pin_free.push_back(b); }
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    cudaError_t next_event(cudaEvent_t *e)
    {
        if (ev_used == ev_pool.size()) {
            cudaEvent_t n;
            cudaError_t rc = cudaEventCreate(&n);
            if (rc != cudaSuccess) return rc;
            ev_pool.push_back(n);
        }
        *e = ev_pool[ev_used++];
        return cudaSuccess;
    }
};

struct swb_refset {
    swb_ctx *ctx = nullptr;
    int64_t n_refs = 0, total_bases = 0, blocks_per_rp = 0;
    int32_t max_len = 0;
    int n_symbols = 0;
    uint8_t code_of[128];                       // upper-cased ASCII byte -> code (rank among the set's symbols), 0xFF = absent
    bool two_bit_ok = false;                    // <= 4 symbols: the 2-bit packed short-read path is available
    DevBuf<uint8_t> codes8;                     // 1 byte per base, original order (wide path)
    DevBuf<int64_t> off8;                       // [n_refs + 1]
    std::vector<int32_t> len_orig;
    std::vector<int32_t> len_sorted;            // lengths in the device (descending-length) order
    DevBuf<uint32_t> words, word_off;
    DevBuf<int32_t> len, orig, sorted_of;
    DevBuf<int64_t> blk_off;
    // A large set is cut into PARTS: contiguous ranges of the caller's reference indices, each a complete packed set
    // of its own.  An align call walks the parts in order; the results of part k are a contiguous segment of every
    // ABI array (pair = ref * n_reads + read), so they cross PCIe while part k + 1 computes.  The parent keeps the
    // alphabet, the lengths and the totals; `parts` is empty for a part (and for a set small enough to be one).
    // fill work units (reference segments, make_segments) per (K, scores): device tables built on first use.  Guarded by
    // the context mutex like every align call.
    struct SegKey {
        int K, match, mismatch, gap, few;
        bool operator<(const SegKey &o) const { return std::tie(K, match, mismatch, gap, few) < std::tie(o.K, o.match, o.mismatch, o.gap, o.few); }
    };
    struct SegTables { size_t nv = 0; DevBuf<int32_t> ref, c0, len, skip, end; };
    mutable std::map<SegKey, std::shared_ptr<SegTables>> seg_cache;
    std::vector<swb_refset *> parts;
    std::vector<int64_t> part_first;            // first global reference index of each part
    swb_refset *whole = nullptr;                // a set with parts: the same references as one set (device-resident / scores-only calls)
    const swb_refset *parent = nullptr;
};

struct swb_reads {
    swb_ctx *ctx = nullptr;
    const swb_refset *rs = nullptr;
    int64_t n_reads = 0;
    std::vector<int32_t> len;
    DevBuf<uint8_t> codes;
    DevBuf<int64_t> off;
};

struct BatchOut {
    bool wide = false;                           // produced by the int32 long-pair path (different key layout)
    std::vector<int64_t> wide_pair_p;            // wide: local pair -> ABI pair index p
    uint32_t n_cells = 0;
    int64_t ops_stride = 0;
    DevBuf<uint64_t> keys;
    DevBuf<int32_t> beg, oplen;
    DevBuf<uint32_t> ops;
    DevBuf<int32_t> d_slot_read;                 // read slot of this batch -> read index of the call, for the assembly
    DevBuf<int64_t> d_pair_map;                  // wide path: local pair -> p, on the device
};

struct swb_result {
    swb_ctx *ctx = nullptr;
    int64_t n_refs = 0, n_reads = 0;
    uint32_t flags = 0;
    bool fetched = false;
    std::vector<int32_t> ref_len, read_len;
    DevBuf<int32_t> d_scores, d_totals, d_best;
    swbh::Selection sel;
    DevBuf<int32_t> d_hits;                      // hits mode: [n_reads][k][4] (score, ref, i, j)
    const int32_t *hits = nullptr;               // host view after fetch
    int64_t n_hits = 0;                          // all-hits mode: entries of d_hit_list
    DevBuf<int64_t> d_hit_off;                   // [n_reads + 1] offsets into d_hit_list
    DevBuf<int32_t> d_hit_list;                  // [n_hits][4] (score, ref, i, j)
    const int64_t *hit_off = nullptr;            // host views after fetch
    const int32_t *hit_list = nullptr;
    std::vector<BatchOut> batches;               // released once the result is assembled
    // assembled on the device (swb_assemble.cu), ABI order
    uint32_t total_cells = 0;
    int64_t total_words = 0;
    DevBuf<int32_t> f_cells, f_beg, f_len;
    DevBuf<int64_t> f_ops_off, f_cell_off;
    DevBuf<uint32_t> f_ops;
    // host views into pinned buffers (after fetch)
    std::vector<swb_ctx::PinBuf> pins;
    const int32_t *scores = nullptr, *totals = nullptr, *best = nullptr;
    const int64_t *cell_off = nullptr, *ops_off = nullptr;
    const int32_t *cells = nullptr, *beginnings = nullptr, *op_lens = nullptr;
    const uint32_t *ops = nullptr;
    double stats[swbh::STAT_COUNT] = {0};
    std::vector<char> own;                      // host arrays of a 1 x 1 result cut out of a coalesced batch (swb_queue.cu)
    // result of a multi-part reference set: one sub-result per part (device arrays), stitched into the host arrays
    std::vector<swb_result *> subs;
    std::vector<int64_t> sub_first;
    size_t parts_total = 0;                     // parts the call will produce (capacity guess of the host arrays)
    std::vector<char> sub_copied;               // part k's arrays are already on their way to the host buffers
    swb_ctx::PinBuf h_scores, h_totals, h_best, h_cell_off, h_cells, h_beg, h_len, h_ops_off, h_ops;
    uint64_t cells_done = 0;                    // cells / words of the parts copied so far
    int64_t words_done = 0;
};


namespace swbh {

// Device time per phase of one call: event pairs around the work, read once after the call's last sync.  Spans nest
// (a selection inside the locate span); end() closes the innermost open one.
struct PhaseTimer {
    struct Span { cudaEvent_t a, b; Stat stat; };
    swb_ctx *ctx;
    cudaStream_t st;
    std::vector<Span> spans;
    std::vector<size_t> open;
    cudaError_t begin(Stat stat)
    {
        Span s{nullptr, nullptr, stat};
        cudaError_t e;
        if ((e = ctx->next_event(&s.a)) || (e = ctx->next_event(&s.b)) || (e = cudaEventRecord(s.a, st))) return e;
        open.push_back(spans.size());
        spans.push_back(s);
        return cudaSuccess;
    }
    cudaError_t end()
    {
        const size_t k = open.back();
        open.pop_back();
        return cudaEventRecord(spans[k].b, st);
    }
    // adds each span's milliseconds to its entry of `stats`
    cudaError_t add_to(double *stats) const
    {
        float ms = 0;
        for (const Span &s : spans) {
            if (cudaError_t e = cudaEventElapsedTime(&ms, s.a, s.b)) return e;
            stats[s.stat] += ms;
        }
        return cudaSuccess;
    }
};

// both-strands mode (swb_strands.cu): the IUPAC DNA complement of a byte keeping case (a -> t; a byte outside the
// table stays itself), the complement codes of a set's alphabet, and the 2n internal reads [reads; rc(reads)] of a call
char complement_keep_case(char c);
int strand_complement_codes(const swb_refset *rs, uint8_t comp_code[256]);
int both_strands_reads(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, std::unique_ptr<swb_reads> &out);

// One align call over one packed set (a whole set, or one part of a large one), step by step (swb_align.cu; the wide
// path in swb_wide_host.cu).  With a selection (hits or all-hits mode) every pair is scored and only the selected ones
// are traced: a short-read batch marks its selection between the tile scan and the emit, the wide reads are scored
// first and then traced over their selected references, and a final selection over all reads makes the result's lists
// and the pairs whose cells the assembly keeps.
// Two views of the pairs: the fill, locate, traceback and assembly sort run over (rs->n_refs, rd->n_reads); the
// totals, best hits and selections over the result's oriented (o_refs, o_reads).  They are the same unless `both`
// (SWB_F_BOTH_STRANDS): rd then holds the 2n internal reads [reads; rc(reads)], and pair r * 2n + s * n + q of the
// internal view is pair (2r + s) * n + q of the oriented one -- the same index.
struct AlignCall {
    swb_ctx *ctx;
    const swb_refset *rs;
    const swb_reads *rd;
    int32_t match, mismatch, gap;
    uint32_t flags;
    Selection sel;
    swb_result *res;
    cudaStream_t st;
    PhaseTimer timer;
    int launches = 1, n_batches = 0;
    double ck_bytes = 0;
    bool both = false;
    int64_t o_refs = 0, o_reads = 0;

    struct Batch;
    int run(int32_t *ext_scores, int32_t *ext_totals);
    void classify_reads(std::vector<std::vector<int32_t>> &classes, std::vector<int32_t> &wide) const;
    int run_class(int K, std::vector<int32_t> &reads);
    int seg_tables(int K, bool few_items, std::shared_ptr<swb_refset::SegTables> &out);
    int fill_batch(int K, const std::vector<int32_t> &reads, int64_t rp0, int n_rp, const swb_refset::SegTables &segt, Batch &b);
    int trace_batch(int K, Batch &b);
    int locate_cells(int K, const Batch &b, size_t sel_words, uint32_t &n_cells);
    int mark_selection(const int32_t *slots, int64_t n_slots, int with_best, uint32_t *bits, int64_t bit_slot, int64_t bit_ref,
                       bool oriented_bits = false, int4 *hits = nullptr);
    int run_wide_reads(const std::vector<int32_t> &wide);
    // refs_of (nullable): refs_of[k] = the references (ascending) read reads[k] is aligned against; nullptr = all of them
    int run_wide_path(const std::vector<int32_t> &reads, bool scores_only, const std::vector<std::vector<int32_t>> *refs_of = nullptr);
    int select_final(DevBuf<uint32_t> &keep);
    int assemble(const DevBuf<uint32_t> &keep);
    int finish_stats(std::chrono::steady_clock::time_point t_wall0);
};

// an align call on host reads (swb_align*): upload, align, the H2D time in the result's stats
int align_host(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
               int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, const Selection &sel, swb_result **out);

}  // namespace swbh
