// swb_api.cu -- the C ABI (include/swb200.h): contexts, HBM-resident reference sets and
// read batches, the align driver (batching, kernel sequencing, timing) and result access.
// No CPU fallback: every compute entry needs a CUDA device and fails loudly without one.
#include "swb_host.h"

#include <chrono>

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

int grid_for(int64_t n, int threads, int sm_count)
{
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + threads - 1) / threads, (int64_t)sm_count * 16));
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
    CU(cudaStreamCreateWithFlags(&c->stream_fill, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c->stream_copy, cudaStreamNonBlocking));
    // Two-stream pipelining (fill of batch k+1 beside the traceback of batch k) is OFF by default: measured on
    // B200 the persistent fill warps keep the integer pipe ~94 % busy and starve co-resident kernels (locate
    // 0.55 -> 5.5 ms), so the overlap buys nothing (62.0 vs 61.1 ms per step).  SWB_PIPELINE=1 enables it.
    c->pipeline = getenv("SWB_PIPELINE") != nullptr;
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
    c->ck.release(); c->tmx.release(); c->counters.release(); c->rp.release(); c->slot.release();
    c->tasks.release(); c->task_hits.release(); c->keys_tmp.release(); c->sort_tmp.release();
    for (int k = 0; k < 2; ++k) { c->ck2[k].release(); c->tmx2[k].release(); c->rp2[k].release(); }
    cudaStreamSynchronize(c->stream_fill);
    c->v_ref.release(); c->v_c0.release(); c->v_len.release(); c->v_skip.release(); c->v_end.release();
    c->w_brow.release(); c->w_rec.release(); c->w_wreads.release(); c->w_rpad.release(); c->w_rpad_off.release(); c->w_rpad_len.release(); c->w_dbg.release(); c->w_mail.release(); c->w_tmx.release(); c->w_prog.release(); c->w_pair_ref.release();
    c->w_pair_read.release(); c->w_band_off.release(); c->w_blk_off.release(); c->w_brow_off.release();
    c->w_items.release(); c->w_tasks.release(); c->hit_tmp.release(); c->hit_sel.release();
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    for (auto &b : c->pin_free) cudaFreeHost(b.p);
    cudaStreamSynchronize(c->stream);
    if (c->ev[0]) cudaEventDestroy(c->ev[0]);
    if (c->ev[1]) cudaEventDestroy(c->ev[1]);
    for (cudaStream_t s : {c->stream, c->stream_fill, c->stream_copy}) if (s) { cudaStreamSynchronize(s); swbh::BlockCache::get().purge(s); }
    if (c->stream_copy) { cudaStreamSynchronize(c->stream_copy); cudaStreamDestroy(c->stream_copy); }
    if (c->stream_fill) cudaStreamDestroy(c->stream_fill);
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
    static const int env_parts = getenv("SWB_REF_PARTS") ? atoi(getenv("SWB_REF_PARTS")) : 0;
    if (env_parts > 0) return (int)std::min<int64_t>(env_parts, std::max<int64_t>(n_refs, 1));
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

// Work units of the fill: every reference is one segment unless it is very long.  A long reference
// is cut into windows of SEG columns, each started W_al columns early from an all-zero boundary.
// H(i,j) only depends on the columns (j - W, j], W = m + floor(max(match,mismatch,0)*m/|gap|) + 1 (a
// positive-score path over i <= m rows can pay for at most that many deletions), so every cell
// further than W from the window's left edge is exact; the segment OWNS (writes tile maxima and
// checkpoints for) exactly the blocks of its own SEG columns.  This bounds the longest item (tail of
// the persistent fill) and gives a single long reference enough items to fill the machine.
namespace {
struct Segments { std::vector<int32_t> ref, c0, len, skip, end; };
void make_segments(const swb_refset *rs, int K, int match, int mismatch, int gap, int64_t n_rp, int sm_count, Segments &S)
{
    const int64_t m = (int64_t)GL * K;
    const int64_t big = std::max({match, mismatch, 0});
    const int64_t W = m + (big * m) / (-(int64_t)gap) + 1;
    const int64_t W_al = ((W + 8 + 15) / 16) * 16;
    int64_t SEG = 8192;
    if (n_rp * ((rs->n_refs + 3) / 4) < (int64_t)sm_count * 24) SEG = 1024;     // few items: favour parallelism
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
}  // namespace

static int pick_k(int m)
{
    for (int k = 0; k < kNumK; ++k)
        if (GL * kKList[k] >= m) return kKList[k];
    return 0;
}

// One packed set (a whole small set, or one part of a large one).  ext_scores / ext_totals: rows of the parent's
// score matrix / totals this part writes into (nullptr: own arrays).  top_k > 0: hits mode (swb_align_hits) -- only the
// pairs of each read's top k and its best pair are traced, and only the top k's cells are kept.
static int align_leaf(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                      int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score, int32_t *ext_scores, int32_t *ext_totals,
                      swb_result **out)
{
    if (!ctx || !rs || !rd || !out) return fail(SWB_E_INVALID, "swb_align: null argument");
    *out = nullptr;
    if (rd->rs != rs && rd->rs != rs->parent) return fail(SWB_E_INVALID, "swb_align: reads were encoded against a different reference set");
    if (rs->ctx != ctx || rd->ctx != ctx) return fail(SWB_E_INVALID, "swb_align: handles belong to another context");
    const int64_t n_refs = rs->n_refs, n_reads = rd->n_reads;
    if (n_refs * n_reads >= ((int64_t)1 << 33)) return fail(SWB_E_UNSUPPORTED, "swb_align: more than 2^33 pairs per call");
    int32_t max_m = 0;
    for (int32_t m : rd->len) max_m = std::max(max_m, m);
    // Java int arithmetic wraps; this engine refuses inputs whose scores could leave int32 instead
    {
        const int64_t big = std::max({std::abs((int64_t)match), std::abs((int64_t)mismatch), std::abs((int64_t)gap)});
        if (big * ((int64_t)max_m + rs->max_len + 2) >= ((int64_t)1 << 30))
            return fail(SWB_E_UNSUPPORTED, "swb_align: |score| * (m + n) could overflow int32");
    }
    // s16x2 short-read kernels: gap < 0 (padding stays below the maximum), small scores, 2-bit alphabet;
    // everything else goes through the int32 wide path (swb_wide.cu)
    const bool short_scores_ok = rs->two_bit_ok && gap < 0 && std::abs((int64_t)match) <= 8000 &&
                                 std::abs((int64_t)mismatch) <= 8000 && std::abs((int64_t)gap) <= 8000;
    // reads of 257 .. 511 rows: the LONG classes (K = 40 .. 64) exist for the biased fill and the tile kernels only;
    // other score sets send such reads through the wide path as before (SWB_NO_LONG_CLASSES=1: always)
    static const bool no_long = getenv("SWB_NO_LONG_CLASSES") != nullptr;
    const bool long_kernels_ok = !no_long && tile_trace_ok(match, mismatch, gap);
    auto read_is_short = [&](int32_t m) {
        if (!short_scores_ok) return false;
        const int64_t smax = (int64_t)std::max({match, mismatch, 0}) * std::min<int64_t>(m, rs->max_len);   // a positive mismatch scores too
        if (smax > 16000) return false;
        if (m <= MAX_SHORT_ROWS) return true;
        return m <= MAX_LONG_ROWS && long_kernels_ok && fill_bias_ok(match, mismatch, gap, smax);
    };

    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // a result counts as a live handle of its context from here on (released by swb_result_free, also on the error paths)
    auto res_del = [](swb_result *r) { swb_result_free(r); };
    std::unique_ptr<swb_result, decltype(res_del)> res(new swb_result(), res_del);
    ctx->live.fetch_add(1);
    res->ctx = ctx; res->n_refs = n_refs; res->n_reads = n_reads; res->flags = flags;
    res->ref_len = rs->len_orig; res->read_len = rd->len;
    const size_t n_pairs = (size_t)(n_refs * n_reads);
    if (ext_scores) res->d_scores.view(ext_scores, n_pairs); else CU(res->d_scores.alloc(n_pairs, st));
    if (ext_totals) res->d_totals.view(ext_totals, (size_t)n_refs); else CU(res->d_totals.alloc((size_t)n_refs, st));
    CU(res->d_best.alloc((size_t)n_reads * 4, st));
    CU(cudaMemsetAsync(res->d_scores.p, 0, std::max<size_t>(n_pairs, 1) * 4, st));
    res->top_k = top_k; res->min_score = min_score;
    if (top_k > 0) CU(res->d_hits.alloc((size_t)n_reads * top_k * 4, st));
    // hits mode: top k + best pair of the reads `slots` (score rows exact by now) -> `bits` / `hits` (swb_hits.cu)
    auto select_hits = [&](const int32_t *slots, int64_t n_slots, int with_best, int4 *hits, uint32_t *bits, int64_t bit_slot,
                      int64_t bit_ref) -> cudaError_t {
        const size_t te = select_hits_tmp_elems(n_refs, n_slots, top_k);
        cudaError_t e = ctx->hit_tmp.reserve(te, st);
        if (e == cudaSuccess) e = launch_select_hits(res->d_scores.p, n_refs, n_reads, slots, n_slots, top_k, min_score, with_best,
                                                     hits, bits, bit_slot, bit_ref, ctx->hit_tmp.p, te, st);
        return e;
    };

    const auto t_wall0 = std::chrono::steady_clock::now();
    const bool tlh = getenv("SWB_TIMELINE_HOST") != nullptr;
    auto mark = [&](const char *what) {
        if (tlh) fprintf(stderr, "[swb host] %8.3f ms  %s\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_wall0).count(), what);
    };
    // phase timing: event pairs are only recorded inside the loop and read after the last sync
    ctx->ev_used = 0;
    struct Span { cudaEvent_t a, b; int phase; };
    std::vector<Span> spans;
    // spans may interleave (two streams): tic returns the span's index, toc closes that index
    cudaError_t span_err = cudaSuccess;
    auto tic = [&](int phase, cudaStream_t on) -> int {
        Span sp; sp.phase = phase;
        cudaError_t e = ctx->next_event(&sp.a);
        if (e == cudaSuccess) e = ctx->next_event(&sp.b);
        if (e == cudaSuccess) e = cudaEventRecord(sp.a, on);
        if (e != cudaSuccess) { span_err = e; return -1; }
        spans.push_back(sp);
        return (int)spans.size() - 1;
    };
    auto toc = [&](int idx, cudaStream_t on) -> cudaError_t {
        if (idx < 0) return span_err;
        return cudaEventRecord(spans[(size_t)idx].b, on);
    };
    // single-stream adapters for the wide path
    int wide_span = -1;
    std::function<cudaError_t(int)> tic1 = [&](int phase) -> cudaError_t { wide_span = tic(phase, st); return wide_span < 0 ? span_err : cudaSuccess; };
    std::function<cudaError_t()> toc1 = [&]() -> cudaError_t { return toc(wide_span, st); };
    (void)max_m;

    std::vector<int32_t> h_read_batch, h_read_slot_all, wide_reads_all;
    double ck_bytes = 0;
    int launches = 1, n_batches = 0;
    CU(ctx->counters.reserve(16, st));

    if (n_refs > 0 && n_reads > 0) {
        // group reads by rows-per-lane class, longest first inside a class
        std::vector<std::vector<int32_t>> classes(kNumK);
        std::vector<int32_t> wide_reads;
        for (int64_t q = 0; q < n_reads; ++q) {
            const int m = rd->len[(size_t)q];
            if (m == 0) continue;                                  // score 0, no cells
            if (!read_is_short(m)) { wide_reads.push_back((int32_t)q); continue; }
            const int K = pick_k(m);
            for (int k = 0; k < kNumK; ++k) if (kKList[k] == K) classes[(size_t)k].push_back((int32_t)q);
        }
        wide_reads_all = wide_reads;
        CU(ctx->slot.reserve((size_t)n_reads, st));
        std::vector<int32_t> h_slot((size_t)n_reads);
        h_read_batch.assign((size_t)n_reads, -1);
        h_read_slot_all.assign((size_t)n_reads, -1);

        for (int kc = 0; kc < kNumK; ++kc) {
            auto &idx = classes[(size_t)kc];
            if (idx.empty()) continue;
            const int K = kKList[kc];
            const int RW = ((K + 1 + 7) / 8 + CB / 8) * 8;        // record words per (block, lane): Geo<K>::RW
            std::stable_sort(idx.begin(), idx.end(),
                             [&](int32_t a, int32_t b) { return rd->len[(size_t)a] > rd->len[(size_t)b]; });
            const int64_t n_rp_total = ((int64_t)idx.size() + 1) / 2;
            // the segment tables only depend on (K, scores, few-items flag): built once per reference set and kept on the device
            const bool few_items = n_rp_total * ((rs->n_refs + 3) / 4) < (int64_t)ctx->sm_count * 24;
            const swb_refset::SegKey skey{K, match, mismatch, gap, few_items ? 1 : 0};
            auto sit = rs->seg_cache.find(skey);
            if (sit == rs->seg_cache.end()) {
                Segments segs;
                make_segments(rs, K, match, mismatch, gap, n_rp_total, ctx->sm_count, segs);
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
            const std::shared_ptr<swb_refset::SegTables> segt = sit->second;
            const size_t nv = segt->nv;
            // ---- batches of read pairs, two-stage pipeline on two streams -----------------------------
            // stage F (ctx->stream_fill): fill of batch k+1;  stage T (ctx->stream): flag/locate/sort/trace of
            // batch k.  The fill saturates the integer pipe, the traceback is latency-bound: run together they
            // share the SMs.  Two checkpoint workspaces, ping-pong; events order the reuse.
            const int64_t bytes_per_rp = rs->blocks_per_rp * ((int64_t)RW * GL * 4 + GL * 4);   // block records (checkpoint + seam) + tile max
            int64_t rp_per_batch = std::max<int64_t>(1, ctx->ws_bytes / std::max<int64_t>(bytes_per_rp, 1));
            const bool pipelined = !(flags & SWB_F_SCORES_ONLY) && n_rp_total > rp_per_batch / 2 && ctx->pipeline;
            if (pipelined) rp_per_batch = std::max<int64_t>(1, rp_per_batch / 2);       // two workspaces
            rp_per_batch = std::min<int64_t>(rp_per_batch, 1 << 16);
            if (rp_per_batch * rs->n_refs * 2 >= ((int64_t)1 << 30)) rp_per_batch = std::max<int64_t>(1, (((int64_t)1 << 30) - 1) / (rs->n_refs * 2));
            // equal-sized batches (no small straggler batch at the end)
            const int64_t nb = (n_rp_total + rp_per_batch - 1) / rp_per_batch;
            rp_per_batch = (n_rp_total + nb - 1) / nb;
            cudaStream_t sF = pipelined ? ctx->stream_fill : st;

            struct Stage { int n_rp = 0, m_max = 0, buf = 0; std::vector<int32_t> h_rp; BatchParams P; cudaEvent_t ev_fill = nullptr; };
            std::vector<Stage> stages((size_t)nb);
            cudaEvent_t ev_trace_done[2] = {nullptr, nullptr};

            auto fill_stage = [&](int64_t k) -> int {
                Stage &S = stages[(size_t)k];
                const int64_t rp0 = k * rp_per_batch;
                S.n_rp = (int)std::min<int64_t>(rp_per_batch, n_rp_total - rp0);
                S.buf = pipelined ? (int)(k & 1) : 0;
                S.h_rp.assign((size_t)S.n_rp * 2, -1);
                for (int r = 0; r < S.n_rp; ++r)
                    for (int h = 0; h < 2; ++h) {
                        const int64_t x = (rp0 + r) * 2 + h;
                        if (x < (int64_t)idx.size()) {
                            S.h_rp[(size_t)r * 2 + h] = idx[(size_t)x];
                            S.m_max = std::max(S.m_max, rd->len[(size_t)idx[(size_t)x]]);
                        }
                    }
                ++n_batches;
                DevBuf<uint32_t> &ck = ctx->ck2[S.buf], &tmx = ctx->tmx2[S.buf];
                DevBuf<int32_t> &rpb = ctx->rp2[S.buf];
                // the workspace of this parity is free once the traceback that last used it has finished
                if (ev_trace_done[S.buf]) CU(cudaStreamWaitEvent(sF, ev_trace_done[S.buf], 0));
                CU(rpb.reserve(S.h_rp.size(), sF));
                CU(cudaMemcpyAsync(rpb.p, S.h_rp.data(), S.h_rp.size() * 4, cudaMemcpyHostToDevice, sF));
                const size_t ck_words = (size_t)S.n_rp * rs->blocks_per_rp * RW * GL;
                const size_t tmx_words = (size_t)S.n_rp * rs->blocks_per_rp * GL;
                CU(ck.reserve(ck_words, sF));
                CU(tmx.reserve(tmx_words, sF));
                ck_bytes += (double)(ck_words + tmx_words) * 4;
                BatchParams &P = S.P;
                P.ref_words = rs->words.p; P.ref_word_off = rs->word_off.p; P.ref_len = rs->len.p;
                P.ref_orig = rs->orig.p; P.ref_sorted_of = rs->sorted_of.p; P.ref_blk_off = rs->blk_off.p;
                P.n_refs = (int32_t)n_refs; P.blocks_per_rp = rs->blocks_per_rp;
                P.v_ref = segt->ref.p; P.v_c0 = segt->c0.p; P.v_len = segt->len.p; P.v_skip = segt->skip.p;
                P.v_end = segt->end.p; P.n_vrefs = (int32_t)nv;
                P.read_codes = rd->codes.p; P.read_off = rd->off.p; P.rp_reads = rpb.p; P.read_slot = nullptr;
                P.n_rp = S.n_rp; P.n_reads = n_reads;
                P.match = match; P.mismatch = mismatch; P.gap = gap; P.tie_gt = (flags & SWB_F_TIE_GT) ? 1 : 0;
                P.scores = res->d_scores.p; P.rec = ck.p; P.tmx = tmx.p; P.sel = nullptr;
                uint32_t *d_work = ctx->counters.p + 4 + S.buf;
                const bool biased = fill_bias_ok(match, mismatch, gap, (int64_t)std::max({match, mismatch, 0}) * std::min<int64_t>(S.m_max, rs->max_len));
                P.seam_bias = biased ? -gap : 0;               // the biased fill stores its seams biased
                P.tmx_slack = biased ? fill_sub_slack(match, mismatch, gap) : 0;
                const int sp_fill = tic(1, sF);
                if (biased)
                    CU(launch_fill_bias(K, P, d_work, ctx->sm_count, sF));
                else
                    CU(launch_fill(K, P, d_work, ctx->sm_count, sF));
                ++launches;
                mark("fill issued");
                CU(toc(sp_fill, sF));
                CU(ctx->next_event(&S.ev_fill));
                CU(cudaEventRecord(S.ev_fill, sF));
                return SWB_OK;
            };

            auto trace_stage = [&](int64_t k) -> int {
                Stage &S = stages[(size_t)k];
                const bool scores_only = (flags & SWB_F_SCORES_ONLY) != 0;
                // hits mode: the scan makes the batch's score rows exact, the selection marks the pairs the emit keeps
                const bool hits_sel = top_k > 0 && !scores_only;
                const size_t sel_words = ((size_t)S.n_rp * 2 * (size_t)n_refs + 31) / 32;
                if (hits_sel) {
                    CU(ctx->hit_sel.reserve(sel_words, st));
                    S.P.sel = ctx->hit_sel.p;
                }
                const BatchParams &P = S.P;
                const int n_rp = S.n_rp;
                if (sF != st) CU(cudaStreamWaitEvent(st, S.ev_fill, 0));
                if (scores_only && P.tmx_slack == 0) return SWB_OK;      // the fill's pair scores are exact
                uint32_t *d_ntasks = ctx->counters.p, *d_ncells = ctx->counters.p + 1;
                // ---- candidate tiles -> exact scores + max cells -> sorted keys (one host sync: the two counts) ----
                const int sp_loc = tic(2, st);
                const int64_t pairs_b = (int64_t)n_rp * 2 * n_refs;
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
                    if (hits_sel) {
                        const int sp_sel = tic(5, st);
                        CU(cudaMemsetAsync(ctx->hit_sel.p, 0, sel_words * 4, st));
                        CU(select_hits(P.rp_reads, (int64_t)n_rp * 2, 1, nullptr, ctx->hit_sel.p, n_refs, 1));
                        CU(toc(sp_sel, st));
                        launches += 2;
                    }
                    if (!scores_only) {
                        CU(launch_locate(K, P, ctx->tasks.p, d_ntasks, cap_tasks, ctx->task_hits.p, ctx->keys_tmp.p, cap_cells, d_ncells,
                                         ctx->sm_count, 1, st));
                        ++launches;
                    }
                    mark("flag + locate issued");
                    CU(cudaMemcpyAsync(h_counts, ctx->counters.p, 8, cudaMemcpyDeviceToHost, st));
                    CU(cudaStreamSynchronize(st));
                    mark("counts on the host");
                    if (h_counts[0] <= cap_tasks && h_counts[1] <= cap_cells) break;
                    if (attempt == 2) return fail(SWB_E_NOMEM, "swb_align: max-cell list did not fit after two retries");
                    // a partial scan only raised pair scores towards their exact value: the retry stays correct
                    cap_tasks = std::max(cap_tasks, h_counts[0]);
                    cap_cells = std::max<uint32_t>(cap_cells, (uint32_t)std::min<uint64_t>((uint64_t)h_counts[1] * 2, 1ull << 31));
                }
                if (scores_only) { CU(toc(sp_loc, st)); return SWB_OK; }
                const uint32_t n_cells = h_counts[1];
                BatchOut bo;
                bo.K = K;
                bo.n_cells = n_cells;
                CU(bo.keys.alloc(n_cells, st));
                const size_t tmp_bytes = sort_keys_tmp_bytes(n_cells);
                CU(ctx->sort_tmp.reserve(tmp_bytes, st));
                CU(sort_keys(ctx->keys_tmp.p, bo.keys.p, n_cells, ctx->sort_tmp.p, tmp_bytes, st));
                launches += 4;
                CU(toc(sp_loc, st));

                // ---- traceback ----------------------------------------------------------
                const int sp_tr = tic(3, st);
                const int64_t big = std::max({match, mismatch, 0});
                int64_t lmax = (int64_t)S.m_max + (big * S.m_max - 1) / (-(int64_t)gap) + 1;
                lmax = std::min<int64_t>(lmax, (int64_t)S.m_max + rs->max_len);
                bo.ops_stride = (int)((lmax + 15) / 16);
                CU(bo.beg.alloc(n_cells, st));
                CU(bo.oplen.alloc(n_cells, st));
                CU(bo.ops.alloc((size_t)n_cells * bo.ops_stride, st));
                if (tile_trace_ok(match, mismatch, gap))
                    CU(launch_tile_trace(K, P, bo.keys.p, n_cells, bo.beg.p, bo.oplen.p, bo.ops.p, (int)bo.ops_stride, ctx->sm_count, st));
                else
                    CU(launch_trace(K, P, bo.keys.p, n_cells, bo.beg.p, bo.oplen.p, bo.ops.p, (int)bo.ops_stride, ctx->sm_count, st));
                ++launches;
                CU(toc(sp_tr, st));
                CU(ctx->next_event(&ev_trace_done[S.buf]));
                CU(cudaEventRecord(ev_trace_done[S.buf], st));
                res->stats[8] += n_cells;
                bo.slot_read = S.h_rp;
                CU(bo.d_slot_read.alloc(S.h_rp.size(), st));
                CU(cudaMemcpyAsync(bo.d_slot_read.p, bo.slot_read.data(), S.h_rp.size() * 4, cudaMemcpyHostToDevice, st));
                res->batches.push_back(std::move(bo));
                mark("sort + trace issued");
                return SWB_OK;
            };

            // the fill stream must see the scores memset and the segment tables issued on `st`
            if (sF != st) {
                cudaEvent_t ev0;
                CU(ctx->next_event(&ev0));
                CU(cudaEventRecord(ev0, st));
                CU(cudaStreamWaitEvent(sF, ev0, 0));
            }
            int rc = SWB_OK;
            if (pipelined) {
                if ((rc = fill_stage(0))) return rc;
                for (int64_t k = 0; k < nb; ++k) {
                    if (k + 1 < nb && (rc = fill_stage(k + 1))) return rc;
                    if ((rc = trace_stage(k))) return rc;
                }
            } else {
                for (int64_t k = 0; k < nb; ++k) {      // one workspace: strictly fill, then trace
                    if ((rc = fill_stage(k))) return rc;
                    if ((rc = trace_stage(k))) return rc;
                }
            }
            if (sF != st) {                       // everything of this class is ordered before what follows on `st`
                cudaEvent_t evl;
                CU(ctx->next_event(&evl));
                CU(cudaEventRecord(evl, sF));
                CU(cudaStreamWaitEvent(st, evl, 0));
            }
            CU(cudaStreamSynchronize(st));        // stages hold host vectors used by async copies
            mark("class done (sync)");
        }
    }
    if (n_refs > 0 && !wide_reads_all.empty()) {
        if (top_k > 0 && !(flags & SWB_F_SCORES_ONLY)) {
            // hits mode: exact scores of every wide pair first, then the whole wide path over each read's top k + best pair
            int rc = run_wide_path(ctx, rs, rd, wide_reads_all, match, mismatch, gap, flags | SWB_F_SCORES_ONLY, res.get(), &launches,
                                   &n_batches, &ck_bytes, tic1, toc1);
            if (rc) return rc;
            const int64_t nw = (int64_t)wide_reads_all.size();
            DevBuf<int32_t> d_wr;
            CU(d_wr.alloc((size_t)nw, st));
            CU(cudaMemcpyAsync(d_wr.p, wide_reads_all.data(), (size_t)nw * 4, cudaMemcpyHostToDevice, st));
            const int sp_sel = tic(5, st);
            int4 *d_sel = reinterpret_cast<int4 *>(res->d_hits.p);              // scratch here: the final selection rewrites it
            CU(select_hits(d_wr.p, nw, 1, d_sel, nullptr, 0, 0));
            CU(toc(sp_sel, st));
            launches += 2;
            std::vector<int4> h_sel((size_t)nw * top_k);
            CU(cudaMemcpyAsync(h_sel.data(), d_sel, h_sel.size() * sizeof(int4), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            std::vector<std::vector<int32_t>> refs_of((size_t)nw);
            for (int64_t x = 0; x < nw; ++x) {
                for (int h = 0; h < top_k; ++h)
                    if (h_sel[(size_t)(x * top_k + h)].y >= 0) refs_of[(size_t)x].push_back(h_sel[(size_t)(x * top_k + h)].y);
                std::sort(refs_of[(size_t)x].begin(), refs_of[(size_t)x].end());
            }
            rc = run_wide_path(ctx, rs, rd, wide_reads_all, match, mismatch, gap, flags, res.get(), &launches, &n_batches, &ck_bytes,
                               tic1, toc1, &refs_of);
            if (rc) return rc;
        } else {
            int rc = run_wide_path(ctx, rs, rd, wide_reads_all, match, mismatch, gap, flags, res.get(), &launches, &n_batches,
                                   &ck_bytes, tic1, toc1);
            if (rc) return rc;
        }
    }
    // hits mode: the final lists (every score is exact now) and, with cells, the pairs whose cells the assembly keeps
    DevBuf<uint32_t> keep;
    if (top_k > 0) {
        const bool with_cells = !(flags & SWB_F_SCORES_ONLY);
        if (with_cells) {
            CU(keep.alloc((n_pairs + 31) / 32, st));
            CU(cudaMemsetAsync(keep.p, 0, ((n_pairs + 31) / 32) * 4, st));
        }
        const int sp_sel = tic(5, st);
        CU(select_hits(nullptr, n_reads, 0, reinterpret_cast<int4 *>(res->d_hits.p), keep.p, 1, n_reads));
        CU(toc(sp_sel, st));
        launches += 2;
    }
    const int sp_misc = tic(4, st);
    CU(launch_ref_totals(res->d_scores.p, n_refs, n_reads, res->d_totals.p, st));
    CU(launch_best_hits(res->d_scores.p, n_refs, n_reads, res->d_best.p, ctx->sm_count, st));
    launches += 3;
    // ---- assemble the final, ABI-ordered result on the device (swb_assemble.cu) ----------------
    if (!(flags & SWB_F_SCORES_ONLY)) {
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
        static const bool tl4 = getenv("SWB_TIMELINE") != nullptr;
        const auto t4 = std::chrono::steady_clock::now();
        auto ms4 = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t4).count(); };
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
        if (tl4) {
            cudaMemPool_t pool; uint64_t resv = 0, used = 0; size_t fr = 0, tot = 0;
            cudaDeviceGetDefaultMemPool(&pool, ctx->device);
            cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &resv);
            cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used);
            cudaMemGetInfo(&fr, &tot);
            fprintf(stderr, "[swb assemble] N %u: allocations issued at %.3f ms; pool reserved %.2f GB used %.2f GB, device free %.2f GB\n", N, ms4(),
                    resv / 1e9, used / 1e9, fr / 1e9);
        }
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
            res->stats[8] = NK;
        }
        CU(cudaMemsetAsync(d_words.p + NK, 0, 8, st));
        CU(assemble_gather_cells(d_desc.p, (int)descs.size(), NK, d_order.p, res->f_cells.p, res->f_beg.p, res->f_len.p,
                                 d_words.p, res->f_ops_off.p, d_tmp.p, tmp_bytes, st));
        int64_t total_words = 0;
        mark("assemble sort + cells issued");
        CU(cudaMemcpyAsync(&total_words, res->f_ops_off.p + NK, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        mark("total words on the host");
        if (tl4) fprintf(stderr, "[swb assemble] sort + cell gather done at %.3f ms\n", ms4());
        res->total_words = total_words;
        CU(res->f_ops.alloc((size_t)total_words, st));
        if (tl4) fprintf(stderr, "[swb assemble] ops array (%lld words) allocated at %.3f ms\n", (long long)total_words, ms4());
        CU(assemble_gather_ops(d_desc.p, (int)descs.size(), NK, d_order.p, res->f_ops_off.p, res->f_ops.p, st));
        CU(assemble_offsets(d_pair_sorted.p, NK, (int64_t)n_pairs, res->f_cell_off.p, res->d_best.p, n_reads, res->f_cells.p, st));
        launches += 8;
        if (keep.p) {
            CU(assemble_hit_cells(d_desc.p, (int)descs.size(), d_pair_sorted.p, d_order.p, N, (int64_t)n_pairs, n_reads, res->f_cell_off.p,
                                  res->f_cells.p, res->d_best.p, res->d_hits.p, top_k, st));
            launches += 2;
        }
        CU(toc(sp_misc, st));
        CU(cudaStreamSynchronize(st));
        mark("assembled (sync)");
        if (tl4) fprintf(stderr, "[swb assemble] ops gathered at %.3f ms\n", ms4());
        res->batches.clear();                     // per-batch buffers go back to the pool
        if (tl4) fprintf(stderr, "[swb assemble] batch buffers released at %.3f ms\n", ms4());
    } else {
        CU(toc(sp_misc, st));
        CU(cudaStreamSynchronize(st));
    }
    double t_phase[6] = {0, 0, 0, 0, 0, 0};
    if (getenv("SWB_TIMELINE") && !spans.empty())
        for (const Span &sp : spans) {
            float a = 0, b = 0;
            cudaEventElapsedTime(&a, spans[0].a, sp.a);
            cudaEventElapsedTime(&b, spans[0].a, sp.b);
            fprintf(stderr, "[swb timeline] phase %d  %8.3f .. %8.3f ms\n", sp.phase, a, b);
        }
    for (const Span &sp : spans) {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, sp.a, sp.b));
        t_phase[sp.phase] += ms;
    }

    int64_t read_bases = 0;
    for (int32_t m : rd->len) read_bases += m;
    res->stats[1] = t_phase[1]; res->stats[2] = t_phase[2]; res->stats[3] = t_phase[3];
    res->stats[5] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_wall0).count();   // wall: phases overlap
    res->stats[6] = (double)rs->total_bases * (double)read_bases;
    res->stats[7] = (double)n_refs * (double)n_reads;
    res->stats[9] = launches; res->stats[10] = ck_bytes; res->stats[11] = n_batches; res->stats[12] = t_phase[5];
    swb_result *r = res.release();
    mark("before fetch");
    if (!(flags & SWB_F_NO_FETCH)) {
        int rc = swb_result_fetch(r);
        mark("fetched");
        if (rc) { swb_result_free(r); return rc; }
    }
    *out = r;
    return SWB_OK;
}

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
    if (getenv("SWB_TIMELINE")) fprintf(stderr, "[swb parts] pinned array grows: has %zu, needs %zu, keeps %zu\n", b.bytes, need, used);
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
    const bool tl = getenv("SWB_TIMELINE") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    auto ms = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
    cudaEvent_t ev;
    CU(ctx->next_event(&ev));
    CU(cudaEventRecord(ev, ctx->stream));
    CU(cudaStreamWaitEvent(sc, ev, 0));
    if (tl) fprintf(stderr, "[swb parts]   copy_part %zu: event %.3f ms\n", k, ms());
    if (np_k) {
        if (cb) add_base_kernel<<<grid_for((int64_t)np_k, 256, ctx->sm_count), 256, 0, sc>>>(sub->f_cell_off.p, (int64_t)np_k, (int64_t)cb);
        CU(cudaMemcpyAsync((int64_t *)res->h_cell_off.p + (size_t)first * (size_t)res->n_reads, sub->f_cell_off.p, np_k * 8, cudaMemcpyDeviceToHost, sc));
    }
    if (tl) fprintf(stderr, "[swb parts]   copy_part %zu: cell_off issued %.3f ms\n", k, ms());
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
    if (tl) fprintf(stderr, "[swb parts]   copy_part %zu: all issued %.3f ms\n", k, ms());
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
    res->stats[4] = ms;                                           // what was left to copy after the last part's compute
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

static int check_hits_args(const char *who, int32_t top_k, int32_t min_score)
{
    if (top_k < 1 || top_k > 32) return fail(SWB_E_INVALID, std::string(who) + ": top_k must be 1 .. 32");
    if (min_score < 1) return fail(SWB_E_INVALID, std::string(who) + ": min_score must be >= 1");
    return SWB_OK;
}

static int align_resident(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                          int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score, swb_result **out)
{
    if (!ctx || !rs || !rd || !out) return fail(SWB_E_INVALID, "swb_align: null argument");
    *out = nullptr;
    if (rs->parent) return fail(SWB_E_INVALID, "swb_align: a part of a reference set is not a handle");
    if (rs->parts.empty()) return align_leaf(ctx, rs, rd, match, mismatch, gap, flags, top_k, min_score, nullptr, nullptr, out);
    // hits mode also runs on the set as one: its cell arrays are small (nothing to overlap), and the selection is then
    // over all references at once, so no part keeps cells of a pair that a later part displaces from the top k
    if (rs->whole && ((flags & (SWB_F_NO_FETCH | SWB_F_SCORES_ONLY)) || top_k > 0))
        return align_leaf(ctx, rs->whole, rd, match, mismatch, gap, flags, top_k, min_score, nullptr, nullptr, out);
    // ---- a set of several parts: part by part; part k's results cross PCIe while part k + 1 computes -------------
    if (rd->rs != rs) return fail(SWB_E_INVALID, "swb_align: reads were encoded against a different reference set");
    if (rs->ctx != ctx || rd->ctx != ctx) return fail(SWB_E_INVALID, "swb_align: handles belong to another context");
    const int64_t n_refs = rs->n_refs, n_reads = rd->n_reads;
    if (n_refs * n_reads >= ((int64_t)1 << 33)) return fail(SWB_E_UNSUPPORTED, "swb_align: more than 2^33 pairs per call");
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const auto t_wall0 = std::chrono::steady_clock::now();
    auto res_del = [](swb_result *r) { swb_result_free(r); };
    std::unique_ptr<swb_result, decltype(res_del)> res(new swb_result(), res_del);
    ctx->live.fetch_add(1);
    res->ctx = ctx; res->n_refs = n_refs; res->n_reads = n_reads; res->flags = flags;
    res->ref_len = rs->len_orig; res->read_len = rd->len;
    const size_t n_pairs = (size_t)(n_refs * n_reads);
    CU(res->d_scores.alloc(n_pairs, st));
    CU(res->d_totals.alloc((size_t)n_refs, st));
    CU(res->d_best.alloc((size_t)n_reads * 4, st));
    const bool full = !(flags & SWB_F_SCORES_ONLY), fetch_now = !(flags & SWB_F_NO_FETCH);
    const int threads = 256;
    res->parts_total = rs->parts.size();
    static const bool timeline = getenv("SWB_TIMELINE") != nullptr;
    auto wall_ms = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_wall0).count(); };
    for (size_t k = 0; k < rs->parts.size(); ++k) {
        const swb_refset *part = rs->parts[k];
        const int64_t first = rs->part_first[k];
        swb_result *sub = nullptr;
        if (timeline) fprintf(stderr, "[swb parts] part %zu starts at %.3f ms (pinned allocations so far %lld)\n", k, wall_ms(), (long long)ctx->pin_allocs);
        const int rc = align_leaf(ctx, part, rd, match, mismatch, gap, flags | SWB_F_NO_FETCH, 0, 1, res->d_scores.p + (size_t)first * (size_t)n_reads,
                                  res->d_totals.p + first, &sub);
        if (rc) return rc;
        res->subs.push_back(sub); res->sub_first.push_back(first); res->sub_copied.push_back(0);
        for (int x : {1, 2, 3, 8, 9, 10, 11}) res->stats[x] += sub->stats[x];
        if ((uint64_t)res->cells_done + sub->total_cells >= ((uint64_t)1 << 31) || res->total_cells + (uint64_t)sub->total_cells >= ((uint64_t)1 << 31))
            return fail(SWB_E_UNSUPPORTED, "swb_align: more than 2^31 max cells in one call");
        res->total_cells += sub->total_cells; res->total_words += sub->total_words;
        if (n_reads)
            fold_best_kernel<<<(unsigned)((n_reads + threads - 1) / threads), threads, 0, st>>>(res->d_best.p, sub->d_best.p, n_reads, (int32_t)first, k == 0);
        CU(cudaGetLastError());
        if (timeline) fprintf(stderr, "[swb parts] part %zu computed at %.3f ms\n", k, wall_ms());
        if (fetch_now && full) { const int rc2 = copy_part(res.get(), k); if (rc2) return rc2; }
        if (timeline) fprintf(stderr, "[swb parts] part %zu copy issued at %.3f ms\n", k, wall_ms());
    }
    CU(cudaStreamSynchronize(st));
    int64_t read_bases = 0;
    for (int32_t m : rd->len) read_bases += m;
    res->stats[6] = (double)rs->total_bases * (double)read_bases;
    res->stats[7] = (double)n_refs * (double)n_reads;
    if (fetch_now) { const int rc = finish_parts_fetch(res.get()); if (rc) return rc; }
    if (timeline) fprintf(stderr, "[swb parts] fetched at %.3f ms (pinned allocations %lld)\n", wall_ms(), (long long)ctx->pin_allocs);
    res->stats[5] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_wall0).count();
    *out = res.release();
    return SWB_OK;
}

int swb_align_resident(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                       int32_t gap, uint32_t flags, swb_result **out)
{
    return align_resident(ctx, rs, rd, match, mismatch, gap, flags, 0, 1, out);
}

int swb_align_resident_hits(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, int32_t match, int32_t mismatch,
                            int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score, swb_result **out)
{
    if (out) *out = nullptr;
    const int rc = check_hits_args("swb_align_resident_hits", top_k, min_score);
    if (rc) return rc;
    return align_resident(ctx, rs, rd, match, mismatch, gap, flags, top_k, min_score, out);
}

static int align_host(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                      int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score, swb_result **out)
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
    rc = align_resident(ctx, rs, rd, match, mismatch, gap, flags, top_k, min_score, out);
    swb_reads_free(rd);
    if (rc == SWB_OK) (*out)->stats[0] = h2d;
    return rc;
}

int swb_align(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
              int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, swb_result **out)
{
    return align_host(ctx, rs, n_reads, read_bytes, read_offsets, match, mismatch, gap, flags, 0, 1, out);
}

int swb_align_hits(swb_ctx *ctx, const swb_refset *rs, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                   int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score, swb_result **out)
{
    if (out) *out = nullptr;
    const int rc = check_hits_args("swb_align_hits", top_k, min_score);
    if (rc) return rc;
    return align_host(ctx, rs, n_reads, read_bytes, read_offsets, match, mismatch, gap, flags, top_k, min_score, out);
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
    if (res->top_k > 0 && (rc = pull(res->d_hits.p, (size_t)res->n_reads * res->top_k * 16, (const void **)&res->hits))) return rc;
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
    res->stats[4] = ms;
    res->fetched = true;
    return SWB_OK;
}

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
    if (top_k) *top_k = r ? r->top_k : 0;
    return (r && r->fetched && r->top_k > 0) ? r->hits : nullptr;
}
const int64_t *swb_result_cell_offsets(const swb_result *r) { return (r && r->fetched) ? r->cell_off : nullptr; }
int64_t swb_result_total_cells(const swb_result *r) { return r ? (int64_t)r->total_cells : 0; }
const int32_t *swb_result_cells(const swb_result *r) { return (r && r->fetched) ? r->cells : nullptr; }
const int32_t *swb_result_beginnings(const swb_result *r) { return (r && r->fetched) ? r->beginnings : nullptr; }
const int32_t *swb_result_op_lens(const swb_result *r) { return (r && r->fetched) ? r->op_lens : nullptr; }

int64_t swb_result_pair_cell_count(const swb_result *r, int64_t pair)
{
    if (!r || !r->fetched || pair < 0 || pair >= r->n_refs * r->n_reads) return -1;
    if (r->flags & SWB_F_SCORES_ONLY) return -1;
    if (r->scores[(size_t)pair] == 0 && r->top_k == 0) {      // hits mode: a score-0 pair is never a hit, its range is empty
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
    if (r->scores[(size_t)pair] == 0 && r->top_k == 0) {
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
    for (int k = 0; k < n && k < 13; ++k) outp[k] = r->stats[k];
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
