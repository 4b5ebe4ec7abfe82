// swb_api.cu -- the C ABI (include/swb200.h): contexts, HBM-resident reference sets and
// read batches, and result access; the align driver is swb_align.cu.
// No CPU fallback: every compute entry needs a CUDA device and fails loudly without one.
#include "swb_host.h"

using namespace swbh;

namespace swbh {
std::string &last_error()
{
    thread_local std::string e;
    return e;
}
}  // namespace swbh

// ---- device-side ingest: validate, case-fold, encode and 2-bit pack on the GPU (the reference's strings come from
// InOutOps.GetRefSeqs / GetReads, InOutOps.java:60-88, :100-169; here they arrive as raw ASCII bytes) ------------
namespace {

// which byte values occur (after upper-casing): 128-bit presence mask + a non-ASCII flag
__global__ void seq_scan_kernel(const uint8_t *raw, int64_t n, uint32_t *present, uint32_t *bad)
{
    uint32_t m[4] = {0, 0, 0, 0};
    uint32_t b = 0;
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        uint32_t c = raw[k];
        if (c >= 128) { b = 1; continue; }
        if (c >= 'a' && c <= 'z') c -= 32;
        m[c >> 5] |= 1u << (c & 31);
    }
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        uint32_t v = m[w];
        for (int o = 16; o; o >>= 1) v |= __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicOr(present + w, v);
    }
    if (b) atomicOr(bad, 1u);
}

// raw ASCII -> symbol codes (code_of[upper(byte)], 0xFF = symbol absent from the reference set)
__global__ void seq_encode_kernel(const uint8_t *raw, int64_t n, const uint8_t *code_of, uint8_t *codes, uint32_t *bad)
{
    __shared__ uint8_t tab[128];
    if (threadIdx.x < 128) tab[threadIdx.x] = code_of[threadIdx.x];
    __syncthreads();
    uint32_t b = 0;
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        uint32_t c = raw[k];
        if (c >= 128) { b = 1; c = 0; }
        if (c >= 'a' && c <= 'z') c -= 32;
        codes[k] = tab[c];
    }
    if (b && bad) atomicOr(bad, 1u);
}

// 2-bit pack, 16 codes per word, references in the device (descending-length) order: one thread per output word
__global__ void ref_pack_kernel(const uint8_t *codes8, const int64_t *src_off, const int32_t *len, const uint32_t *word_off,
                                int64_t n_refs, uint64_t n_words, uint32_t *words)
{
    for (uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; w < n_words; w += (uint64_t)gridDim.x * blockDim.x) {
        int64_t lo = 0, hi = n_refs;                              // last reference whose first word is <= w
        while (hi - lo > 1) { const int64_t mid = (lo + hi) >> 1; if ((uint64_t)word_off[mid] <= w) lo = mid; else hi = mid; }
        const int64_t c0 = (int64_t)(w - word_off[lo]) * 16;
        const int64_t n = len[lo];
        const uint8_t *src = codes8 + src_off[lo] + c0;
        uint32_t v = 0;
        for (int k = 0; k < 16 && c0 + k < n; ++k) v |= (uint32_t)(src[k] & 3u) << (2 * k);
        words[w] = v;
    }
}

}  // namespace

extern "C" {

int swb_abi_version(void) { return SWB_ABI_VERSION; }
const char *swb_last_error(void) { return last_error().c_str(); }

int swb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int swb_create(int device, int64_t workspace_bytes, swb_ctx **out)
{
    if (!out) return fail(SWB_E_INVALID, "swb_create: out is null");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(SWB_E_CUDA, "swb_create: no CUDA device available (this engine has no CPU fallback)");
    }
    if (device < 0 || device >= n) return fail(SWB_E_INVALID, "swb_create: bad device index");
    CU(cudaSetDevice(device));
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, device));
    if (p.major < 9) return fail(SWB_E_UNSUPPORTED, "swb_create: DPX kernels need sm_90+ (built for sm_100a)");
    // owned until *out is set: a failing call below releases the streams / events created so far
    std::unique_ptr<swb_ctx, void (*)(swb_ctx *)> guard(new swb_ctx(), swb_destroy);
    swb_ctx *c = guard.get();
    c->device = device;
    c->sm_count = p.multiProcessorCount;
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    // default: 45 % of the free HBM, at most 64 GiB (a B200 has 180 GB: the number every published figure uses).  The
    // block records of one batch live here; a larger workspace means fewer, larger batches (cfg3 needs 27 GB for one).
    int64_t ws = workspace_bytes > 0 ? workspace_bytes : std::min<int64_t>((int64_t)64 << 30, (int64_t)(free_b / 100 * 45));
    ws = std::min<int64_t>(ws, (int64_t)(free_b / 2));
    c->ws_bytes = ws;
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c->stream_copy, cudaStreamNonBlocking));
    CU(cudaEventCreate(&c->ev[0]));
    CU(cudaEventCreate(&c->ev[1]));
    cudaMemPool_t pool;
    CU(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t keep = UINT64_MAX;                                    // keep freed blocks in the pool
    CU(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    *out = guard.release();
    return SWB_OK;
}

// Handles (reference sets, read batches, results) point into their context and release device memory on its
// streams: a context destroyed while handles are alive (Python __del__ order at interpreter exit, a JVM's global
// arena) only marks itself; the last handle's *_free finishes the destruction.
static void ctx_handle_released(swb_ctx *c)
{
    if (c->live.fetch_sub(1) == 1 && c->dying.load()) swb_destroy(c);
}

void swb_destroy(swb_ctx *c)
{
    if (!c) return;
    if (c->live.load() > 0) { c->dying.store(true); return; }
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    c->ck.release(); c->tmx.release(); c->counters.release(); c->rp.release();
    c->tasks.release(); c->task_hits.release(); c->keys_tmp.release(); c->sort_tmp.release();
    c->w_brow.release(); c->w_rec.release(); c->w_wreads.release(); c->w_rpad.release(); c->w_rpad_off.release(); c->w_rpad_len.release(); c->w_mail.release(); c->w_tmx.release(); c->w_pair_ref.release();
    c->w_pair_read.release(); c->w_band_off.release(); c->w_blk_off.release(); c->w_brow_off.release();
    c->w_items.release(); c->w_tasks.release(); c->hit_tmp.release(); c->hit_sel.release(); c->margin_best.release();
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    for (auto &b : c->pin_free) cudaFreeHost(b.p);
    cudaStreamSynchronize(c->stream);
    if (c->ev[0]) cudaEventDestroy(c->ev[0]);
    if (c->ev[1]) cudaEventDestroy(c->ev[1]);
    for (cudaStream_t s : {c->stream, c->stream_copy}) if (s) { cudaStreamSynchronize(s); swbh::BlockCache::get().purge(s); }
    if (c->stream_copy) { cudaStreamSynchronize(c->stream_copy); cudaStreamDestroy(c->stream_copy); }
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int swb_get_stream(swb_ctx *ctx, void **stream)
{
    if (!ctx || !stream) return fail(SWB_E_INVALID, "swb_get_stream: null");
    *stream = (void *)ctx->stream;
    return SWB_OK;
}

static int check_offsets(const char *who, int64_t n, const char *bytes, const int64_t *off)
{
    if (n < 0) return fail(SWB_E_INVALID, std::string(who) + ": negative count");
    if (!off) return fail(SWB_E_INVALID, std::string(who) + ": offsets is null");
    if (off[0] < 0) return fail(SWB_E_INVALID, std::string(who) + ": negative offset");
    for (int64_t k = 0; k < n; ++k)
        if (off[k + 1] < off[k]) return fail(SWB_E_INVALID, std::string(who) + ": offsets not monotone");
    if (off[n] > off[0] && !bytes) return fail(SWB_E_INVALID, std::string(who) + ": bytes is null");
    return SWB_OK;
}

// One packed set over references [0, n_refs) of `offsets`, whose raw bytes already sit on the device at d_raw
// (d_raw[0] = byte offsets[0]); the alphabet is the caller's.  Encodes (8-bit codes, caller's order: wide path) and
// 2-bit packs (descending-length order: short path) on the device.
static int build_leaf(swb_ctx *ctx, int64_t n_refs, const int64_t *offsets, const uint8_t *d_raw, const uint8_t *code_of,
                      int n_symbols, swb_refset **out)
{
    cudaStream_t st = ctx->stream;
    std::unique_ptr<swb_refset> rs(new swb_refset());
    rs->ctx = ctx;
    rs->n_refs = n_refs;
    rs->len_orig.resize((size_t)n_refs);
    for (int64_t k = 0; k < n_refs; ++k) {
        const int64_t n = offsets[k + 1] - offsets[k];
        rs->len_orig[(size_t)k] = (int32_t)n;
        rs->total_bases += n;
        rs->max_len = std::max<int32_t>(rs->max_len, (int32_t)n);
    }
    const int64_t total = rs->total_bases;
    memcpy(rs->code_of, code_of, sizeof rs->code_of);
    rs->n_symbols = n_symbols;
    rs->two_bit_ok = n_symbols <= 4;           // otherwise only the 8-bit int32 path can hold the set

    // length buckets: descending length, stable
    std::vector<int32_t> order((size_t)n_refs);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(),
                     [&](int32_t a, int32_t b) { return rs->len_orig[(size_t)a] > rs->len_orig[(size_t)b]; });
    std::vector<int32_t> sorted_of((size_t)n_refs), len_sorted((size_t)n_refs);
    std::vector<uint32_t> word_off((size_t)n_refs);
    std::vector<int64_t> blk_off((size_t)n_refs + 1), src_off((size_t)n_refs), o8((size_t)n_refs + 1);
    uint64_t words_total = 0;
    int64_t blocks = 0;
    for (int64_t s = 0; s < n_refs; ++s) {
        const int32_t o = order[(size_t)s];
        const int32_t n = rs->len_orig[(size_t)o];
        sorted_of[(size_t)o] = (int32_t)s;
        len_sorted[(size_t)s] = n;
        word_off[(size_t)s] = (uint32_t)words_total;
        src_off[(size_t)s] = offsets[o] - offsets[0];
        words_total += (uint64_t)(n + 15) / 16;
        blk_off[(size_t)s] = blocks;
        blocks += (n + GL - 1 + CB - 1) / CB > 0 ? (n + GL - 1 + CB - 1) / CB : 1;
    }
    blk_off[(size_t)n_refs] = blocks;
    for (int64_t k = 0; k <= n_refs; ++k) o8[(size_t)k] = offsets[k] - offsets[0];
    rs->len_sorted = len_sorted;
    rs->blocks_per_rp = blocks;
    if (words_total >= ((uint64_t)1 << 32)) return fail(SWB_E_UNSUPPORTED, "swb_refset_load: reference set too large");

    DevBuf<int64_t> d_src_off;
    DevBuf<uint8_t> d_tab;
    CU(d_tab.alloc(128, st));
    CU(rs->codes8.alloc((size_t)total + 16, st));
    CU(rs->off8.alloc(o8.size(), st));
    CU(rs->words.alloc((size_t)words_total + 1, st));
    CU(rs->word_off.alloc((size_t)n_refs, st));
    CU(rs->len.alloc((size_t)n_refs, st));
    CU(rs->orig.alloc((size_t)n_refs, st));
    CU(rs->sorted_of.alloc((size_t)n_refs, st));
    CU(rs->blk_off.alloc((size_t)n_refs + 1, st));
    CU(d_src_off.alloc((size_t)n_refs, st));
    CU(cudaMemcpyAsync(d_tab.p, rs->code_of, 128, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(rs->off8.p, o8.data(), o8.size() * 8, cudaMemcpyHostToDevice, st));
    if (n_refs) {
        CU(cudaMemcpyAsync(rs->word_off.p, word_off.data(), (size_t)n_refs * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(rs->len.p, len_sorted.data(), (size_t)n_refs * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(rs->orig.p, order.data(), (size_t)n_refs * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(rs->sorted_of.p, sorted_of.data(), (size_t)n_refs * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_src_off.p, src_off.data(), (size_t)n_refs * 8, cudaMemcpyHostToDevice, st));
    }
    CU(cudaMemcpyAsync(rs->blk_off.p, blk_off.data(), ((size_t)n_refs + 1) * 8, cudaMemcpyHostToDevice, st));
    if (total) seq_encode_kernel<<<grid_for(total, 256, ctx->sm_count), 256, 0, st>>>(d_raw, total, d_tab.p, rs->codes8.p, nullptr);
    CU(cudaMemsetAsync(rs->words.p + words_total, 0, 4, st));
    if (words_total && rs->two_bit_ok)
        ref_pack_kernel<<<grid_for((int64_t)words_total, 256, ctx->sm_count), 256, 0, st>>>(rs->codes8.p, d_src_off.p, rs->len.p, rs->word_off.p,
                                                                                             n_refs, words_total, rs->words.p);
    else if (words_total) CU(cudaMemsetAsync(rs->words.p, 0, (size_t)words_total * 4, st));
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));                 // the host tables above are locals
    *out = rs.release();
    return SWB_OK;
}

// how many parts a set of `total_bases` is cut into: a part should hold about 96 read pairs' block records
// (74 bytes per base and read pair) in the workspace, so that a typical call is one batch per part
static int part_count(const swb_ctx *ctx, int64_t total_bases, int64_t n_refs)
{
    const double part_bases = (double)ctx->ws_bytes / (74.0 * 96.0);
    int s = (int)((double)total_bases / std::max(part_bases, 1.0) + 0.5);
    if (s >= 2) ++s;                  // one more, smaller, last part: 8 ranks of one box pull their results at the same moment and share the host's memory bandwidth (measured 8 x B200: 120 MB per rank in 3.7 ms exposed with 2 parts)
    return (int)std::min<int64_t>(std::max(1, std::min(s, 8)), std::max<int64_t>(n_refs, 1));
}

int swb_refset_load(swb_ctx *ctx, int64_t n_refs, const char *bytes, const int64_t *offsets, swb_refset **out)
{
    if (!ctx || !out) return fail(SWB_E_INVALID, "swb_refset_load: null argument");
    *out = nullptr;
    int rc = check_offsets("swb_refset_load", n_refs, bytes, offsets);
    if (rc) return rc;
    if (n_refs > (int64_t)1 << 30) return fail(SWB_E_UNSUPPORTED, "swb_refset_load: more than 2^30 references");
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    for (int64_t k = 0; k < n_refs; ++k)
        if (offsets[k + 1] - offsets[k] >= ((int64_t)1 << KEY_J_BITS))
            return fail(SWB_E_UNSUPPORTED, "swb_refset_load: reference longer than 4,194,303 bases");
    // ---- raw bytes to the device; symbols present and the non-ASCII check there ----------------------
    const int64_t total = offsets[n_refs] - offsets[0];
    DevBuf<uint8_t> d_raw;
    DevBuf<uint32_t> d_flags;                                      // [0..3] presence mask, [4] non-ASCII seen
    CU(d_raw.alloc((size_t)total + 16, st));
    CU(d_flags.alloc(8, st));
    CU(cudaMemsetAsync(d_flags.p, 0, 32, st));
    if (total) CU(cudaMemcpyAsync(d_raw.p, bytes + offsets[0], (size_t)total, cudaMemcpyHostToDevice, st));
    if (total) seq_scan_kernel<<<grid_for(total, 256, ctx->sm_count), 256, 0, st>>>(d_raw.p, total, d_flags.p, d_flags.p + 4);
    CU(cudaGetLastError());
    uint32_t h_flags[8] = {0};
    CU(cudaMemcpyAsync(h_flags, d_flags.p, 32, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (h_flags[4]) return fail(SWB_E_UNSUPPORTED, "swb_refset_load: non-ASCII byte in a reference");
    uint8_t code_of[128];
    int n_symbols = 0;
    memset(code_of, 0xFF, sizeof code_of);
    for (int c = 0; c < 128; ++c)
        if ((h_flags[c >> 5] >> (c & 31)) & 1u) code_of[c] = (uint8_t)n_symbols++;

    const int S = part_count(ctx, total, n_refs);
    swb_refset *rs = nullptr;
    if (S <= 1) {
        rc = build_leaf(ctx, n_refs, offsets, d_raw.p, code_of, n_symbols, &rs);
        if (rc) return rc;
    } else {
        // parts of DECREASING base counts (weights S, S-1, ..., 1), cut at reference boundaries: what stays exposed of
        // the device->host traffic is the LAST part's share (measured, cfg2 step on one B200: equal halves 44.2 ms,
        // one part 44.8 ms, device-resident 42.5 ms; every part costs ~0.5 ms of fixed work)
        std::unique_ptr<swb_refset> parent(new swb_refset());
        parent->ctx = ctx; parent->n_refs = n_refs; parent->total_bases = total;
        parent->n_symbols = n_symbols; parent->two_bit_ok = n_symbols <= 4;
        memcpy(parent->code_of, code_of, sizeof code_of);
        parent->len_orig.resize((size_t)n_refs);
        for (int64_t k = 0; k < n_refs; ++k) {
            parent->len_orig[(size_t)k] = (int32_t)(offsets[k + 1] - offsets[k]);
            parent->max_len = std::max(parent->max_len, parent->len_orig[(size_t)k]);
        }
        auto drop = [&] { for (swb_refset *q : parent->parts) delete q; parent->parts.clear(); };
        int64_t r0 = 0;
        for (int k = 0; k < S && r0 < n_refs; ++k) {
            const int64_t wsum = (int64_t)S * (S + 1) / 2, wdone = wsum - (int64_t)(S - k - 1) * (S - k) / 2;
            const int64_t goal = offsets[0] + (int64_t)((double)total * (double)wdone / (double)wsum);
            int64_t r1 = r0 + 1;
            while (r1 < n_refs && (k == S - 1 || offsets[r1] < goal)) ++r1;
            if (k == S - 1) r1 = n_refs;
            swb_refset *leaf = nullptr;
            rc = build_leaf(ctx, r1 - r0, offsets + r0, d_raw.p + (offsets[r0] - offsets[0]), code_of, n_symbols, &leaf);
            if (rc) { drop(); return rc; }
            leaf->parent = parent.get();
            parent->parts.push_back(leaf);
            parent->part_first.push_back(r0);
            r0 = r1;
        }
        // the same references once more as ONE set: calls whose results stay on the device (SWB_F_NO_FETCH) or are small
        // (SWB_F_SCORES_ONLY) have nothing to overlap and skip the parts' fixed cost (~0.4 ms each)
        rc = build_leaf(ctx, n_refs, offsets, d_raw.p, code_of, n_symbols, &parent->whole);
        if (rc) { drop(); return rc; }
        parent->whole->parent = parent.get();
        rs = parent.release();
    }
    ctx->live.fetch_add(1);
    *out = rs;
    return SWB_OK;
}

void swb_refset_free(swb_refset *rs)
{
    if (!rs) return;
    swb_ctx *c = rs->ctx;
    cudaSetDevice(c->device);
    for (swb_refset *q : rs->parts) delete q;
    delete rs->whole;
    delete rs;
    ctx_handle_released(c);
}
int64_t swb_refset_count(const swb_refset *rs) { return rs ? rs->n_refs : 0; }
int64_t swb_refset_total_bases(const swb_refset *rs) { return rs ? rs->total_bases : 0; }

int swb_reads_upload(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *bytes, const int64_t *offsets,
                     swb_reads **out)
{
    if (!ctx || !rs || !out) return fail(SWB_E_INVALID, "swb_reads_upload: null argument");
    *out = nullptr;
    int rc = check_offsets("swb_reads_upload", n_reads, bytes, offsets);
    if (rc) return rc;
    if (n_reads > (int64_t)1 << 30) return fail(SWB_E_UNSUPPORTED, "swb_reads_upload: more than 2^30 reads");
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    std::unique_ptr<swb_reads> rd(new swb_reads());
    rd->ctx = ctx; rd->rs = rs; rd->n_reads = n_reads;
    rd->len.resize((size_t)n_reads);
    std::vector<int64_t> off((size_t)n_reads + 1);
    int64_t total = 0;
    for (int64_t k = 0; k < n_reads; ++k) {
        off[(size_t)k] = total;
        const int64_t m = offsets[k + 1] - offsets[k];
        if (m >= (1 << 21))
            return fail(SWB_E_UNSUPPORTED, "swb_reads_upload: read longer than 2,097,151 bases");
        rd->len[(size_t)k] = (int32_t)m;
        total += m;
    }
    off[(size_t)n_reads] = total;
    // raw bytes up, case-fold + encode against the set's alphabet on the device
    cudaStream_t st = ctx->stream;
    DevBuf<uint8_t> d_raw, d_tab;
    DevBuf<uint32_t> d_bad;
    CU(d_raw.alloc((size_t)total + 16, st));
    CU(d_tab.alloc(128, st));
    CU(d_bad.alloc(1, st));
    CU(rd->codes.alloc((size_t)total + 16, st));
    CU(rd->off.alloc(off.size(), st));
    CU(cudaMemsetAsync(d_bad.p, 0, 4, st));
    CU(cudaMemcpyAsync(d_tab.p, rs->code_of, 128, cudaMemcpyHostToDevice, st));
    if (total) CU(cudaMemcpyAsync(d_raw.p, bytes + offsets[0], (size_t)total, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(rd->off.p, off.data(), off.size() * 8, cudaMemcpyHostToDevice, st));
    if (total) seq_encode_kernel<<<grid_for(total, 256, ctx->sm_count), 256, 0, st>>>(d_raw.p, total, d_tab.p, rd->codes.p, d_bad.p);
    CU(cudaGetLastError());
    uint32_t h_bad = 0;
    CU(cudaMemcpyAsync(&h_bad, d_bad.p, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (h_bad) return fail(SWB_E_UNSUPPORTED, "swb_reads_upload: non-ASCII byte in a read");
    ctx->live.fetch_add(1);
    *out = rd.release();
    return SWB_OK;
}

void swb_reads_free(swb_reads *rd)
{
    if (!rd) return;
    swb_ctx *c = rd->ctx;
    cudaSetDevice(c->device);
    delete rd;
    ctx_handle_released(c);
}
int64_t swb_reads_count(const swb_reads *rd) { return rd ? rd->n_reads : 0; }

void swb_result_free(swb_result *res)
{
    if (!res) return;
    swb_ctx *c = res->ctx;
    cudaSetDevice(c->device);
    if (!res->subs.empty()) cudaStreamSynchronize(c->stream_copy);       // the parts' arrays may still be on their way
    for (swb_result *sub : res->subs) swb_result_free(sub);
    {
        std::lock_guard<std::recursive_mutex> lk(c->mu);
        for (auto &b : res->pins) c->pin_put(b);
        for (swb_ctx::PinBuf *b : {&res->h_scores, &res->h_totals, &res->h_best, &res->h_cell_off, &res->h_cells, &res->h_beg,
                                   &res->h_len, &res->h_ops_off, &res->h_ops}) { c->pin_put(*b); b->p = nullptr; b->bytes = 0; }
    }
    delete res;
    ctx_handle_released(c);
}

int64_t swb_result_n_refs(const swb_result *r) { return r ? r->n_refs : 0; }
int64_t swb_result_n_reads(const swb_result *r) { return r ? r->n_reads : 0; }
const int32_t *swb_result_scores(const swb_result *r) { return (r && r->fetched) ? r->scores : nullptr; }
const int32_t *swb_result_ref_totals(const swb_result *r) { return (r && r->fetched) ? r->totals : nullptr; }
const int32_t *swb_result_best_hits(const swb_result *r) { return (r && r->fetched) ? r->best : nullptr; }
const int32_t *swb_result_hits(const swb_result *r, int32_t *top_k)
{
    if (top_k) *top_k = r ? r->sel.top_k : 0;                    // 0 outside hits mode
    return (r && r->fetched && r->sel.mode == Selection::TOP_K) ? r->hits : nullptr;
}
const int64_t *swb_result_hit_offsets(const swb_result *r, int64_t *n_hits)
{
    const bool ok = r && r->fetched && r->sel.mode == Selection::MARGIN;
    if (n_hits) *n_hits = ok ? r->n_hits : 0;
    return ok ? r->hit_off : nullptr;
}
const int32_t *swb_result_hit_list(const swb_result *r) { return (r && r->fetched && r->sel.mode == Selection::MARGIN) ? r->hit_list : nullptr; }
const int64_t *swb_result_cell_offsets(const swb_result *r) { return (r && r->fetched) ? r->cell_off : nullptr; }
int64_t swb_result_total_cells(const swb_result *r) { return r ? (int64_t)r->total_cells : 0; }
const int32_t *swb_result_cells(const swb_result *r) { return (r && r->fetched) ? r->cells : nullptr; }
const int32_t *swb_result_beginnings(const swb_result *r) { return (r && r->fetched) ? r->beginnings : nullptr; }
const int32_t *swb_result_op_lens(const swb_result *r) { return (r && r->fetched) ? r->op_lens : nullptr; }

int64_t swb_result_pair_cell_count(const swb_result *r, int64_t pair)
{
    if (!r || !r->fetched || pair < 0 || pair >= r->n_refs * r->n_reads) return -1;
    if (r->flags & SWB_F_SCORES_ONLY) return -1;
    if (r->scores[(size_t)pair] == 0 && r->sel.mode == Selection::NONE) {   // hits / all-hits mode: a score-0 pair is never listed, its range is empty
        const int64_t ref = pair / r->n_reads, rd = pair % r->n_reads;
        return (int64_t)r->ref_len[(size_t)ref] * r->read_len[(size_t)rd];     // every cell ties at 0
    }
    return r->cell_off[(size_t)pair + 1] - r->cell_off[(size_t)pair];
}

int swb_result_pair_cell(const swb_result *r, int64_t pair, int64_t k, int32_t *i, int32_t *j, int32_t *beginning,
                         int32_t *op_len)
{
    const int64_t cnt = swb_result_pair_cell_count(r, pair);
    if (cnt < 0) return fail(SWB_E_RANGE, "swb_result_pair_cell: bad pair");
    if (k < 0 || k >= cnt) return fail(SWB_E_RANGE, "swb_result_pair_cell: bad cell index");
    if (r->scores[(size_t)pair] == 0 && r->sel.mode == Selection::NONE) {
        const int64_t n = r->ref_len[(size_t)(pair / r->n_reads)];
        if (i) *i = (int32_t)(k / n + 1);
        if (j) *j = (int32_t)(k % n + 1);
        if (beginning) *beginning = 0;
        if (op_len) *op_len = 0;
        return SWB_OK;
    }
    const size_t c = (size_t)(r->cell_off[(size_t)pair] + k);
    if (i) *i = r->cells[2 * c];
    if (j) *j = r->cells[2 * c + 1];
    if (beginning) *beginning = r->beginnings[c];
    if (op_len) *op_len = r->op_lens[c];
    return SWB_OK;
}

int swb_result_ops(const swb_result *r, int64_t cell, uint8_t *outp, int64_t cap)
{
    if (!r || !r->fetched || !outp) return fail(SWB_E_INVALID, "swb_result_ops: null / not fetched");
    if (cell < 0 || cell >= (int64_t)r->total_cells || !r->ops) return fail(SWB_E_RANGE, "swb_result_ops: bad cell");
    const int32_t len = r->op_lens[(size_t)cell];
    if (cap < len) return fail(SWB_E_RANGE, "swb_result_ops: buffer too small");
    const uint32_t *w = r->ops + r->ops_off[(size_t)cell];
    // the device stores the walk order (end -> start); hand out start -> end
    for (int32_t k = 0; k < len; ++k) {
        const int32_t src = len - 1 - k;
        outp[k] = (uint8_t)((w[src >> 4] >> (2 * (src & 15))) & 3u);
    }
    return SWB_OK;
}

int swb_result_materialize(const swb_result *r, int64_t cell, const char *ref, int64_t ref_len, const char *read,
                           int64_t read_len, char *ref_aln, char *read_aln, int64_t cap)
{
    if (!r || !r->fetched || !ref_aln || !read_aln) return fail(SWB_E_INVALID, "swb_result_materialize: null / not fetched");
    if (cell < 0 || cell >= (int64_t)r->total_cells || !r->ops) return fail(SWB_E_RANGE, "swb_result_materialize: bad cell");
    const int32_t len = r->op_lens[(size_t)cell];
    if (cap < (int64_t)len + 1) return fail(SWB_E_RANGE, "swb_result_materialize: buffer too small");
    std::vector<uint8_t> ops((size_t)len + 1);
    int rc = swb_result_ops(r, cell, ops.data(), len);
    if (rc) return rc;
    // both strands: a cell of an odd oriented reference is a cell of the read's reverse complement (case kept)
    std::string rc_read;
    if ((r->flags & SWB_F_BOTH_STRANDS) && r->cell_off) {
        const int64_t n_pairs = r->n_refs * r->n_reads;
        const int64_t p = (int64_t)(std::upper_bound(r->cell_off, r->cell_off + n_pairs + 1, cell) - r->cell_off) - 1;
        if ((p / r->n_reads) & 1) {
            rc_read.resize((size_t)std::max<int64_t>(read_len, 0));
            for (int64_t k = 0; k < read_len; ++k) rc_read[(size_t)k] = complement_keep_case(read[read_len - 1 - k]);
            read = rc_read.data();
        }
    }
    // walk the columns backwards from the end cell (SmithWaterman.java:380-409), fill forwards
    int64_t i = r->cells[2 * (size_t)cell], j = r->cells[2 * (size_t)cell + 1];
    if (i > read_len || j > ref_len) return fail(SWB_E_RANGE, "swb_result_materialize: sequences shorter than the cell");
    for (int32_t k = len - 1; k >= 0; --k) {
        const uint8_t op = ops[(size_t)k];
        if (op == 1)      { if (i < 1 || j < 1) return fail(SWB_E_RANGE, "materialize: path leaves the matrix"); ref_aln[k] = ref[j - 1]; read_aln[k] = read[i - 1]; --i; --j; }
        else if (op == 2) { if (i < 1) return fail(SWB_E_RANGE, "materialize: path leaves the matrix"); ref_aln[k] = '_'; read_aln[k] = read[i - 1]; --i; }
        else              { if (j < 1) return fail(SWB_E_RANGE, "materialize: path leaves the matrix"); ref_aln[k] = ref[j - 1]; read_aln[k] = '_'; --j; }
    }
    ref_aln[len] = 0; read_aln[len] = 0;
    return SWB_OK;
}

int swb_result_stats(const swb_result *r, double *outp, int n)
{
    if (!r || !outp) return fail(SWB_E_INVALID, "swb_result_stats: null");
    for (int k = 0; k < n && k < STAT_COUNT; ++k) outp[k] = r->stats[k];
    return SWB_OK;
}

int swb_result_device_ptr(const swb_result *r, int which, void **ptr, int64_t *n_elems)
{
    if (!r || !ptr) return fail(SWB_E_INVALID, "swb_result_device_ptr: null");
    switch (which) {
        case 0: *ptr = r->d_scores.p; if (n_elems) *n_elems = r->n_refs * r->n_reads; return SWB_OK;
        case 1: *ptr = r->d_totals.p; if (n_elems) *n_elems = r->n_refs; return SWB_OK;
        case 2: *ptr = r->d_best.p; if (n_elems) *n_elems = r->n_reads * 4; return SWB_OK;
    }
    return fail(SWB_E_RANGE, "swb_result_device_ptr: bad selector");
}

}  // extern "C"
