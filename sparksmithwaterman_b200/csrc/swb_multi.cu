// swb_multi.cu -- multi-GPU inside the C ABI (include/swb200.h, "multi-GPU" section).
//
// The reference partitions the pair set by REFERENCE (`sc.parallelize(refs)` + map(MapRef),
// Distribution.java:337-338).  Here every device keeps a length-balanced shard of the reference set
// resident in its HBM, aligns all reads against it (swb_align on its own context), and only the
// per-read best-hit records (score, global ref, i, j) cross NVLink: one ncclAllGather issued on each
// device's engine stream after the best-hit kernel, then a merge kernel on the device.
//   swb_multi_*  one process, n devices, one host thread per device inside swb_multi_align
//   swb_comm_*   one process per device (torchrun / MPI); the host ships the 128-byte NCCL id
// NCCL is resolved at run time (dlopen): the library has no link-time dependency on it and a
// single-device host never loads it.
#include "swb_host.h"

#include <dlfcn.h>
#include <nccl.h>          // types and prototypes only; the entry points are looked up with dlsym

#include <cub/device/device_scan.cuh>

#include <chrono>
#include <thread>

using namespace swbh;

namespace {

struct NcclApi {
    void *handle = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitAll) CommInitAll = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    std::string error;
};

NcclApi *nccl_api()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char *names[] = {getenv("SWB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char *n : names) {
            if (!n || !*n) continue;
            api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (!api.handle) { api.error = std::string("NCCL not found (set SWB_NCCL_LIB): ") + (dlerror() ? dlerror() : ""); return; }
#define SWB_NCCL_SYM(field, sym)                                                       \
        api.field = reinterpret_cast<decltype(api.field)>(dlsym(api.handle, sym));     \
        if (!api.field) { api.error = std::string("NCCL symbol missing: ") + sym; return; }
        SWB_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
        SWB_NCCL_SYM(CommInitAll, "ncclCommInitAll")
        SWB_NCCL_SYM(CommInitRank, "ncclCommInitRank")
        SWB_NCCL_SYM(CommDestroy, "ncclCommDestroy")
        SWB_NCCL_SYM(AllGather, "ncclAllGather")
        SWB_NCCL_SYM(GroupStart, "ncclGroupStart")
        SWB_NCCL_SYM(GroupEnd, "ncclGroupEnd")
        SWB_NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef SWB_NCCL_SYM
    });
    return &api;
}

int nccl_fail(ncclResult_t r, const char *what)
{
    NcclApi *a = nccl_api();
    return fail(SWB_E_CUDA, std::string(what) + ": " + (a->GetErrorString ? a->GetErrorString(r) : "NCCL error"));
}
#define NC(x)                                                                  \
    do {                                                                       \
        ncclResult_t r_ = (x);                                                 \
        if (r_ != ncclSuccess) return nccl_fail(r_, #x);                       \
    } while (0)

// all-gather of `count` elements per rank into recv [world][count] on `st`; a world of one copies on the device (and
// never loads NCCL)
int gather(const void *send, void *recv, size_t count, ncclDataType_t type, ncclComm_t comm, int world, cudaStream_t st)
{
    if (count == 0) return SWB_OK;
    if (world > 1) {
        const ncclResult_t r = nccl_api()->AllGather(send, recv, count, type, comm, st);
        return r == ncclSuccess ? SWB_OK : nccl_fail(r, "ncclAllGather");
    }
    CU(cudaMemcpyAsync(recv, send, count * (type == ncclInt64 ? 8 : 4), cudaMemcpyDeviceToDevice, st));
    return SWB_OK;
}

// shard-local reference index -> global index (ids), -1 stays -1 (a shard without references)
__global__ void best_to_global_kernel(const int32_t *best, const int64_t *ids, int64_t n_ids, int64_t n_reads, int32_t *out)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_reads) return;
    int4 b = reinterpret_cast<const int4 *>(best)[q];
    b.y = (b.y >= 0 && b.y < n_ids) ? (int32_t)ids[b.y] : -1;
    reinterpret_cast<int4 *>(out)[q] = b;
}

// gathered[w][q] -> merged[q]: highest score, then lowest global reference index; a record without a reference
// (ref < 0, an empty shard) loses against every real one
__global__ void merge_best_kernel(const int32_t *gathered, int world, int64_t n_reads, int32_t *merged)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_reads) return;
    int4 best = make_int4(0, -1, 0, 0);
    for (int w = 0; w < world; ++w) {
        const int4 b = reinterpret_cast<const int4 *>(gathered)[(int64_t)w * n_reads + q];
        if (b.y < 0) continue;
        if (best.y < 0 || b.x > best.x || (b.x == best.x && b.y < best.y)) best = b;
    }
    reinterpret_cast<int4 *>(merged)[q] = best;
}

// hits mode: hit lists [n_reads][k] with shard-local reference indices -> global ids; padding stays (0, -1, 0, 0)
__global__ void hits_to_global_kernel(const int32_t *hits, const int64_t *ids, int64_t n_ids, int64_t n, int32_t *out)
{
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= n) return;
    int4 h = reinterpret_cast<const int4 *>(hits)[e];
    if (h.y >= 0 && h.y < n_ids) h.y = (int32_t)ids[h.y];
    else h = make_int4(0, -1, 0, 0);
    reinterpret_cast<int4 *>(out)[e] = h;
}

constexpr int kMaxHitsWorld = 64;

// gathered[w][q][k] -> merged[q][k]: k-way merge of the world's sorted lists in the same order (score descending, then
// global reference ascending); a list ends at its first entry without a reference, so an empty shard never wins.
// Exact: the global top k is contained in the union of the shards' top k's.
__global__ void merge_hits_kernel(const int32_t *gathered, int world, int64_t n_reads, int k, int32_t *merged)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_reads) return;
    const int4 *g = reinterpret_cast<const int4 *>(gathered);
    int pos[kMaxHitsWorld];
    for (int w = 0; w < world; ++w) pos[w] = 0;
    for (int h = 0; h < k; ++h) {
        int bw = -1;
        int4 best = make_int4(0, -1, 0, 0);
        for (int w = 0; w < world; ++w) {
            if (pos[w] >= k) continue;
            const int4 e = g[((int64_t)w * n_reads + q) * k + pos[w]];
            if (e.y < 0) continue;
            if (bw < 0 || e.x > best.x || (e.x == best.x && e.y < best.y)) { best = e; bw = w; }
        }
        if (bw >= 0) ++pos[bw];
        reinterpret_cast<int4 *>(merged)[q * k + h] = best;
    }
}

// all-hits mode: the world's lists, read w's list at lists[w * T ..] with offsets offs[w * (n_reads + 1) ..] (relative
// to the list's start), each in list order.  bar = max(min_score, global best - margin), the global best being the
// largest head; count[q] = entries >= bar over all lists
__device__ __forceinline__ int64_t all_hits_bar(const int4 *lists, const int64_t *offs, int world, int64_t n_reads, int64_t T,
                                                int64_t q, int32_t min_score, int32_t margin)
{
    int64_t best = 0;
    for (int w = 0; w < world; ++w) {
        const int64_t *o = offs + (int64_t)w * (n_reads + 1);
        if (o[q + 1] > o[q]) best = max(best, (int64_t)lists[(int64_t)w * T + o[q]].x);
    }
    return max((int64_t)min_score, best - (int64_t)margin);
}

__global__ void all_hits_count_kernel(const int32_t *lists, const int64_t *offs, int world, int64_t n_reads, int64_t T,
                                      int32_t min_score, int32_t margin, int64_t *count)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_reads) return;
    const int4 *l = reinterpret_cast<const int4 *>(lists);
    const int64_t bar = all_hits_bar(l, offs, world, n_reads, T, q, min_score, margin);
    int64_t n = 0;
    for (int w = 0; w < world; ++w) {
        const int64_t *o = offs + (int64_t)w * (n_reads + 1);
        for (int64_t k = o[q]; k < o[q + 1] && l[(int64_t)w * T + k].x >= bar; ++k) ++n;
    }
    count[q] = n;
}

// k-way merge of read q's filtered lists into merged[moff[q] ..]: score descending, then global reference ascending
__global__ void all_hits_merge_kernel(const int32_t *lists, const int64_t *offs, int world, int64_t n_reads, int64_t T,
                                      int32_t min_score, int32_t margin, const int64_t *moff, int32_t *merged)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_reads) return;
    const int4 *l = reinterpret_cast<const int4 *>(lists);
    const int64_t bar = all_hits_bar(l, offs, world, n_reads, T, q, min_score, margin);
    int64_t pos[kMaxHitsWorld];
    for (int w = 0; w < world; ++w) pos[w] = offs[(int64_t)w * (n_reads + 1) + q];
    int4 *out = reinterpret_cast<int4 *>(merged);
    for (int64_t h = moff[q]; h < moff[q + 1]; ++h) {
        int bw = -1;
        int4 best = make_int4(0, -1, 0, 0);
        for (int w = 0; w < world; ++w) {
            if (pos[w] >= offs[(int64_t)w * (n_reads + 1) + q + 1]) continue;
            const int4 e = l[(int64_t)w * T + pos[w]];
            if (e.x < bar) continue;
            if (bw < 0 || e.x > best.x || (e.x == best.x && e.y < best.y)) { best = e; bw = w; }
        }
        if (bw < 0) break;
        ++pos[bw];
        out[h] = best;
    }
}

// send/gather/merge buffers of one device
struct GatherBufs {
    DevBuf<int32_t> send, gathered, merged;
    DevBuf<int32_t> hsend, hgathered, hmerged;   // hits mode: [n_reads][k][4] per shard
    DevBuf<int64_t> ids;
    int64_t n_ids = 0;
    DevBuf<int64_t> oids;                        // both strands: oriented local 2r + s -> oriented global 2 * ids[r] + s
    // all-hits mode: gathered offsets [world][n_reads + 1], lists padded to the largest total [world][T][4], the merge
    DevBuf<int64_t> aoffs, acount, amoff;
    DevBuf<int32_t> asend, alists, amerged;
    DevBuf<uint8_t> atmp;
    std::vector<int64_t> h_off;                  // merged lists on the host
    std::vector<int32_t> h_list;
    void release()
    {
        send.release(); gathered.release(); merged.release(); hsend.release(); hgathered.release(); hmerged.release(); ids.release(); oids.release();
        aoffs.release(); acount.release(); amoff.release(); asend.release(); alists.release(); amerged.release(); atmp.release();
    }
};

// The three steps of an exchange, on `st` of the current device: localize (shard-local reference ids -> global ids, into
// the send buffer), gather (into the gathered buffer), merge.
cudaError_t enqueue_localize(GatherBufs &g, const int64_t *ids, int64_t n_ids, const int32_t *d_best, int64_t n_reads, int world, cudaStream_t st)
{
    cudaError_t e = g.send.reserve((size_t)n_reads * 4, st);
    if (e == cudaSuccess) e = g.gathered.reserve((size_t)n_reads * 4 * world, st);
    if (e == cudaSuccess) e = g.merged.reserve((size_t)n_reads * 4, st);
    if (e != cudaSuccess || n_reads == 0) return e;
    const int threads = 256;
    best_to_global_kernel<<<(unsigned)((n_reads + threads - 1) / threads), threads, 0, st>>>(d_best, ids, n_ids, n_reads, g.send.p);
    return cudaGetLastError();
}
cudaError_t enqueue_merge(GatherBufs &g, int64_t n_reads, int world, cudaStream_t st)
{
    if (n_reads == 0) return cudaSuccess;
    const int threads = 256;
    merge_best_kernel<<<(unsigned)((n_reads + threads - 1) / threads), threads, 0, st>>>(g.gathered.p, world, n_reads, g.merged.p);
    return cudaGetLastError();
}

// the same two steps for the hit lists of a hits-mode result
cudaError_t enqueue_localize_hits(GatherBufs &g, const int64_t *ids, int64_t n_ids, const int32_t *d_hits, int64_t n_reads, int k, int world,
                                  cudaStream_t st)
{
    const size_t n = (size_t)n_reads * k;
    cudaError_t e = g.hsend.reserve(n * 4, st);
    if (e == cudaSuccess) e = g.hgathered.reserve(n * 4 * world, st);
    if (e == cudaSuccess) e = g.hmerged.reserve(n * 4, st);
    if (e != cudaSuccess || n == 0) return e;
    const int threads = 256;
    hits_to_global_kernel<<<(unsigned)((n + threads - 1) / threads), threads, 0, st>>>(d_hits, ids, n_ids, (int64_t)n, g.hsend.p);
    return cudaGetLastError();
}
cudaError_t enqueue_merge_hits(GatherBufs &g, int64_t n_reads, int k, int world, cudaStream_t st)
{
    if (n_reads == 0) return cudaSuccess;
    const int threads = 128;
    merge_hits_kernel<<<(unsigned)((n_reads + threads - 1) / threads), threads, 0, st>>>(g.hgathered.p, world, n_reads, k, g.hmerged.p);
    return cudaGetLastError();
}

// all-hits mode, step 1: the list of `res` -> global ids in g.asend (room for T entries)
cudaError_t enqueue_localize_all_hits(GatherBufs &g, const int64_t *ids, int64_t n_ids, const swb_result *res, int64_t T, int world,
                                      cudaStream_t st)
{
    cudaError_t e = g.asend.reserve((size_t)std::max<int64_t>(T, 1) * 4, st);
    if (e == cudaSuccess) e = g.aoffs.reserve((size_t)(res->n_reads + 1) * world, st);
    if (e == cudaSuccess) e = g.alists.reserve((size_t)std::max<int64_t>(T, 1) * 4 * world, st);
    if (e != cudaSuccess || res->n_hits == 0) return e;
    const int threads = 256;
    hits_to_global_kernel<<<(unsigned)((res->n_hits + threads - 1) / threads), threads, 0, st>>>(res->d_hit_list.p, ids, n_ids, res->n_hits,
                                                                                               g.asend.p);
    return cudaGetLastError();
}

// all-hits mode, last step (after the gathers into g.aoffs / g.alists): count, scan, one sync for the merged length,
// k-way merge, merged lists -> g.h_off / g.h_list
int merge_all_hits(GatherBufs &g, int world, int64_t n_reads, int64_t T, int32_t min_score, int32_t margin, cudaStream_t st)
{
    const int threads = 128;
    const unsigned blocks = (unsigned)((n_reads + threads - 1) / threads);
    CU(g.acount.reserve((size_t)n_reads + 1, st));
    CU(g.amoff.reserve((size_t)n_reads + 1, st));
    CU(cudaMemsetAsync(g.acount.p + n_reads, 0, 8, st));
    if (n_reads) all_hits_count_kernel<<<blocks, threads, 0, st>>>(g.alists.p, g.aoffs.p, world, n_reads, T, min_score, margin, g.acount.p);
    CU(cudaGetLastError());
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, (const int64_t *)nullptr, (int64_t *)nullptr, (int)n_reads + 1);
    CU(g.atmp.reserve(std::max<size_t>(tmp_bytes, 1), st));
    CU(cub::DeviceScan::ExclusiveSum(g.atmp.p, tmp_bytes, g.acount.p, g.amoff.p, (int)n_reads + 1, st));
    g.h_off.assign((size_t)n_reads + 1, 0);
    CU(cudaMemcpyAsync(g.h_off.data(), g.amoff.p, ((size_t)n_reads + 1) * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const int64_t n = g.h_off[(size_t)n_reads];
    g.h_list.assign((size_t)n * 4, 0);
    if (n == 0) return SWB_OK;
    CU(g.amerged.reserve((size_t)n * 4, st));
    all_hits_merge_kernel<<<blocks, threads, 0, st>>>(g.alists.p, g.aoffs.p, world, n_reads, T, min_score, margin, g.amoff.p, g.amerged.p);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(g.h_list.data(), g.amerged.p, (size_t)n * 16, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return SWB_OK;
}

}  // namespace

struct swb_comm {
    swb_ctx *ctx = nullptr;
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
    GatherBufs g;
    int64_t n_reads = 0;
};

struct swb_multi {
    std::vector<int> devices;
    std::vector<swb_ctx *> ctx;
    std::vector<swb_refset *> rs;
    std::vector<std::vector<int64_t>> ids;       // per shard: global reference indices, ascending
    std::vector<int32_t> shard_of;               // global reference -> shard
    std::vector<int64_t> local_of;               // global reference -> index in the shard
    std::vector<ncclComm_t> comms;
    std::vector<GatherBufs> g;
    int64_t n_refs = 0;
    std::mutex mu;
};

struct swb_multi_result {
    swb_multi *m = nullptr;
    std::vector<swb_result *> shard;
    std::vector<int32_t> merged;
    Selection sel;
    std::vector<int32_t> merged_hits;            // hits mode: [n_reads][k][4], global reference ids
    std::vector<int64_t> merged_off;             // all-hits mode: merged lists, global reference ids
    std::vector<int32_t> merged_list;
    int64_t n_reads = 0;
    double stats[3] = {0, 0, 0};
};

// the checks of a swb_comm_allgather_* call on a result that must be of selection `mode` (NONE: any), then the shard's
// global ids on the device (c->g.ids).  The caller holds the context's lock.
static int comm_prepare(const char *who, swb_comm *c, const swb_result *res, Selection::Mode mode, const int64_t *global_ids,
                        int64_t n_local_refs)
{
    const std::string w(who);
    if (res->ctx != c->ctx) return fail(SWB_E_INVALID, w + ": the result belongs to another context");
    if (mode == Selection::TOP_K && res->sel.mode != mode) return fail(SWB_E_INVALID, w + ": not a hits-mode result (swb_align_hits)");
    if (mode == Selection::MARGIN && res->sel.mode != mode) return fail(SWB_E_INVALID, w + ": not an all-hits result (swb_align_all_hits)");
    if (mode != Selection::NONE && c->world > kMaxHitsWorld) return fail(SWB_E_UNSUPPORTED, w + ": more than 64 ranks");
    if (n_local_refs != res->n_refs) return fail(SWB_E_INVALID, w + ": global_ids must cover the shard's references");
    if (n_local_refs > 0 && !global_ids) return fail(SWB_E_INVALID, w + ": global_ids is null");
    cudaStream_t st = c->ctx->stream;
    CU(cudaSetDevice(c->ctx->device));
    CU(c->g.ids.reserve((size_t)std::max<int64_t>(n_local_refs, 1), st));
    c->g.n_ids = n_local_refs;
    if (n_local_refs) CU(cudaMemcpyAsync(c->g.ids.p, global_ids, (size_t)n_local_refs * 8, cudaMemcpyHostToDevice, st));
    return SWB_OK;
}

extern "C" {

int swb_comm_unique_id(char *id128)
{
    if (!id128) return fail(SWB_E_INVALID, "swb_comm_unique_id: null");
    NcclApi *a = nccl_api();
    if (!a->handle || !a->GetUniqueId) return fail(SWB_E_UNSUPPORTED, "swb_comm_unique_id: " + a->error);
    static_assert(sizeof(ncclUniqueId) == 128, "the ABI ships the NCCL id as 128 bytes");
    ncclUniqueId id;
    NC(a->GetUniqueId(&id));
    memcpy(id128, &id, 128);
    return SWB_OK;
}

int swb_comm_create(swb_ctx *ctx, const char *id128, int32_t rank, int32_t world, swb_comm **out)
{
    if (!ctx || !out || (world > 1 && !id128)) return fail(SWB_E_INVALID, "swb_comm_create: null argument");
    *out = nullptr;
    if (world < 1 || rank < 0 || rank >= world) return fail(SWB_E_INVALID, "swb_comm_create: bad rank / world");
    std::unique_ptr<swb_comm> c(new swb_comm());
    c->ctx = ctx; c->rank = rank; c->world = world;
    if (world > 1) {
        NcclApi *a = nccl_api();
        if (!a->handle || !a->CommInitRank) return fail(SWB_E_UNSUPPORTED, "swb_comm_create: " + a->error);
        CU(cudaSetDevice(ctx->device));
        ncclUniqueId id;
        memcpy(&id, id128, 128);
        NC(a->CommInitRank(&c->comm, world, id, rank));
    }
    *out = c.release();
    return SWB_OK;
}

void swb_comm_destroy(swb_comm *c)
{
    if (!c) return;
    cudaSetDevice(c->ctx->device);
    cudaStreamSynchronize(c->ctx->stream);
    c->g.release();
    if (c->comm) nccl_api()->CommDestroy(c->comm);
    delete c;
}

int swb_comm_allgather_best(swb_comm *c, const swb_result *res, const int64_t *global_ids, int64_t n_local_refs,
                            int32_t *merged_host)
{
    if (!c || !res) return fail(SWB_E_INVALID, "swb_comm_allgather_best: null argument");
    std::lock_guard<std::recursive_mutex> lk(c->ctx->mu);
    int rc = comm_prepare("swb_comm_allgather_best", c, res, Selection::NONE, global_ids, n_local_refs);
    if (rc) return rc;
    cudaStream_t st = c->ctx->stream;
    const int64_t n_reads = res->n_reads;
    c->n_reads = n_reads;
    CU(enqueue_localize(c->g, c->g.ids.p, c->g.n_ids, res->d_best.p, n_reads, c->world, st));
    if ((rc = gather(c->g.send.p, c->g.gathered.p, (size_t)n_reads * 4, ncclInt32, c->comm, c->world, st))) return rc;
    CU(enqueue_merge(c->g, n_reads, c->world, st));
    if (merged_host && n_reads) CU(cudaMemcpyAsync(merged_host, c->g.merged.p, (size_t)n_reads * 16, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));        // global_ids / merged_host are the caller's
    return SWB_OK;
}

int swb_comm_allgather_hits(swb_comm *c, const swb_result *res, const int64_t *global_ids, int64_t n_local_refs,
                            int32_t *merged_host)
{
    if (!c || !res) return fail(SWB_E_INVALID, "swb_comm_allgather_hits: null argument");
    std::lock_guard<std::recursive_mutex> lk(c->ctx->mu);
    int rc = comm_prepare("swb_comm_allgather_hits", c, res, Selection::TOP_K, global_ids, n_local_refs);
    if (rc) return rc;
    cudaStream_t st = c->ctx->stream;
    const int64_t n_reads = res->n_reads;
    const int k = res->sel.top_k;
    const size_t n = (size_t)n_reads * k;
    CU(enqueue_localize_hits(c->g, c->g.ids.p, c->g.n_ids, res->d_hits.p, n_reads, k, c->world, st));
    if ((rc = gather(c->g.hsend.p, c->g.hgathered.p, n * 4, ncclInt32, c->comm, c->world, st))) return rc;
    CU(enqueue_merge_hits(c->g, n_reads, k, c->world, st));
    if (merged_host && n) CU(cudaMemcpyAsync(merged_host, c->g.hmerged.p, n * 16, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));        // global_ids / merged_host are the caller's
    return SWB_OK;
}

int swb_comm_allgather_all_hits(swb_comm *c, const swb_result *res, const int64_t *global_ids, int64_t n_local_refs,
                                const int64_t **offsets, const int32_t **list, int64_t *n_hits)
{
    if (!c || !res || !offsets || !list || !n_hits) return fail(SWB_E_INVALID, "swb_comm_allgather_all_hits: null argument");
    *offsets = nullptr; *list = nullptr; *n_hits = 0;
    std::lock_guard<std::recursive_mutex> lk(c->ctx->mu);
    int rc = comm_prepare("swb_comm_allgather_all_hits", c, res, Selection::MARGIN, global_ids, n_local_refs);
    if (rc) return rc;
    cudaStream_t st = c->ctx->stream;
    const int64_t n_reads = res->n_reads, no = n_reads + 1;
    const int world = c->world;
    CU(c->g.aoffs.reserve((size_t)no * world, st));
    // the per-read offsets, then the largest total (one host sync), then the lists padded to it
    if ((rc = gather(res->d_hit_off.p, c->g.aoffs.p, (size_t)no, ncclInt64, c->comm, world, st))) return rc;
    int64_t T = res->n_hits;
    if (world > 1) {
        std::vector<int64_t> h((size_t)no * world);
        CU(cudaMemcpyAsync(h.data(), c->g.aoffs.p, h.size() * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        for (int w = 0; w < world; ++w) T = std::max(T, h[(size_t)w * no + n_reads]);
    }
    CU(enqueue_localize_all_hits(c->g, c->g.ids.p, c->g.n_ids, res, T, world, st));
    if ((rc = gather(c->g.asend.p, c->g.alists.p, (size_t)T * 4, ncclInt32, c->comm, world, st))) return rc;
    if ((rc = merge_all_hits(c->g, world, n_reads, T, res->sel.min_score, res->sel.margin, st))) return rc;
    *offsets = c->g.h_off.data(); *list = c->g.h_list.data(); *n_hits = c->g.h_off[(size_t)n_reads];
    return SWB_OK;
}

int swb_comm_merged_device_ptr(swb_comm *c, void **ptr, int64_t *n_elems)
{
    if (!c || !ptr) return fail(SWB_E_INVALID, "swb_comm_merged_device_ptr: null");
    *ptr = c->g.merged.p;
    if (n_elems) *n_elems = c->n_reads * 4;
    return SWB_OK;
}

// ---------------------------------------------------------------------------------------------------
int swb_multi_create(const int32_t *devices, int32_t n_devices, int64_t workspace_bytes, swb_multi **out)
{
    if (!devices || !out || n_devices < 1) return fail(SWB_E_INVALID, "swb_multi_create: bad arguments");
    *out = nullptr;
    for (int a = 0; a < n_devices; ++a)
        for (int b = a + 1; b < n_devices; ++b)
            if (devices[a] == devices[b]) return fail(SWB_E_INVALID, "swb_multi_create: a device is listed twice");
    std::unique_ptr<swb_multi> m(new swb_multi());
    auto cleanup = [&] { for (swb_ctx *c : m->ctx) swb_destroy(c); m->ctx.clear(); };
    for (int d = 0; d < n_devices; ++d) {
        swb_ctx *c = nullptr;
        const int rc = swb_create(devices[d], workspace_bytes, &c);
        if (rc) { cleanup(); return rc; }
        m->ctx.push_back(c);
        m->devices.push_back(devices[d]);
    }
    m->rs.assign((size_t)n_devices, nullptr);
    m->ids.resize((size_t)n_devices);
    m->g.resize((size_t)n_devices);
    if (n_devices > 1) {
        NcclApi *a = nccl_api();
        if (!a->handle || !a->CommInitAll) { cleanup(); return fail(SWB_E_UNSUPPORTED, "swb_multi_create: " + a->error); }
        m->comms.assign((size_t)n_devices, nullptr);
        const ncclResult_t r = a->CommInitAll(m->comms.data(), n_devices, m->devices.data());
        if (r != ncclSuccess) { cleanup(); return nccl_fail(r, "ncclCommInitAll"); }
    }
    *out = m.release();
    return SWB_OK;
}

void swb_multi_destroy(swb_multi *m)
{
    if (!m) return;
    for (size_t d = 0; d < m->ctx.size(); ++d) {
        cudaSetDevice(m->devices[d]);
        cudaStreamSynchronize(m->ctx[d]->stream);
        m->g[d].release();
        if (m->rs[d]) swb_refset_free(m->rs[d]);
        if (d < m->comms.size() && m->comms[d]) nccl_api()->CommDestroy(m->comms[d]);
    }
    for (swb_ctx *c : m->ctx) swb_destroy(c);
    delete m;
}

int32_t swb_multi_device_count(const swb_multi *m) { return m ? (int32_t)m->ctx.size() : 0; }
swb_ctx *swb_multi_ctx(swb_multi *m, int32_t d) { return (m && d >= 0 && d < (int32_t)m->ctx.size()) ? m->ctx[(size_t)d] : nullptr; }
int64_t swb_multi_ref_count(const swb_multi *m) { return m ? m->n_refs : 0; }

int swb_multi_refset_load(swb_multi *m, int64_t n_refs, const char *bytes, const int64_t *offsets)
{
    if (!m) return fail(SWB_E_INVALID, "swb_multi_refset_load: null");
    if (n_refs < 0 || !offsets) return fail(SWB_E_INVALID, "swb_multi_refset_load: bad arguments");
    for (int64_t k = 0; k < n_refs; ++k)
        if (offsets[k + 1] < offsets[k]) return fail(SWB_E_INVALID, "swb_multi_refset_load: offsets not monotone");
    std::lock_guard<std::mutex> lk(m->mu);
    const int n = (int)m->ctx.size();
    // descending length (stable), dealt in snake order: 0..n-1, n-1..0, ...
    std::vector<int64_t> order((size_t)n_refs);
    std::iota(order.begin(), order.end(), (int64_t)0);
    std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
        return offsets[a + 1] - offsets[a] > offsets[b + 1] - offsets[b];
    });
    for (auto &v : m->ids) v.clear();
    m->shard_of.assign((size_t)n_refs, 0);
    m->local_of.assign((size_t)n_refs, 0);
    for (int64_t pos = 0; pos < n_refs; ++pos) {
        const int64_t round = pos / n, slot = pos % n;
        const int d = (int)((round % 2 == 0) ? slot : n - 1 - slot);
        m->ids[(size_t)d].push_back(order[(size_t)pos]);
    }
    for (int d = 0; d < n; ++d) {
        auto &v = m->ids[(size_t)d];
        std::sort(v.begin(), v.end());
        for (size_t k = 0; k < v.size(); ++k) { m->shard_of[(size_t)v[k]] = d; m->local_of[(size_t)v[k]] = (int64_t)k; }
    }
    m->n_refs = n_refs;
    // one loader thread per device: gather the shard's bytes, pack, upload
    std::vector<int> rcs((size_t)n, SWB_OK);
    std::vector<std::string> errs((size_t)n);
    std::vector<std::thread> th;
    for (int d = 0; d < n; ++d)
        th.emplace_back([&, d] {
            const auto &v = m->ids[(size_t)d];
            std::vector<int64_t> off(v.size() + 1, 0);
            for (size_t k = 0; k < v.size(); ++k) off[k + 1] = off[k] + (offsets[v[k] + 1] - offsets[v[k]]);
            std::string buf((size_t)off[v.size()], '\0');
            for (size_t k = 0; k < v.size(); ++k)
                memcpy(&buf[(size_t)off[k]], bytes + offsets[v[k]], (size_t)(off[k + 1] - off[k]));
            if (m->rs[(size_t)d]) { swb_refset_free(m->rs[(size_t)d]); m->rs[(size_t)d] = nullptr; }
            int rc = swb_refset_load(m->ctx[(size_t)d], (int64_t)v.size(), buf.data(), off.data(), &m->rs[(size_t)d]);
            if (rc == SWB_OK) {
                swb_ctx *c = m->ctx[(size_t)d];
                GatherBufs &g = m->g[(size_t)d];
                cudaError_t e = cudaSetDevice(c->device);
                if (e == cudaSuccess) e = g.ids.reserve(std::max<size_t>(v.size(), 1), c->stream);
                if (e == cudaSuccess && !v.empty()) e = cudaMemcpyAsync(g.ids.p, v.data(), v.size() * 8, cudaMemcpyHostToDevice, c->stream);
                std::vector<int64_t> ov(2 * v.size());
                for (size_t k = 0; k < ov.size(); ++k) ov[k] = 2 * v[k / 2] + (int64_t)(k & 1);
                if (e == cudaSuccess) e = g.oids.reserve(std::max<size_t>(ov.size(), 1), c->stream);
                if (e == cudaSuccess && !ov.empty()) e = cudaMemcpyAsync(g.oids.p, ov.data(), ov.size() * 8, cudaMemcpyHostToDevice, c->stream);
                if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
                g.n_ids = (int64_t)v.size();
                if (e != cudaSuccess) rc = cuda_fail(e, "swb_multi_refset_load: id table");
            }
            rcs[(size_t)d] = rc;
            if (rc) errs[(size_t)d] = swb_last_error();
        });
    for (auto &t : th) t.join();
    for (int d = 0; d < n; ++d)
        if (rcs[(size_t)d]) return fail(rcs[(size_t)d], "shard " + std::to_string(d) + ": " + errs[(size_t)d]);
    return SWB_OK;
}

int swb_multi_ref_location(const swb_multi *m, int64_t global_ref, int32_t *shard, int64_t *local_ref)
{
    if (!m) return fail(SWB_E_INVALID, "swb_multi_ref_location: null");
    if (global_ref < 0 || global_ref >= m->n_refs) return fail(SWB_E_RANGE, "swb_multi_ref_location: bad reference index");
    if (shard) *shard = m->shard_of[(size_t)global_ref];
    if (local_ref) *local_ref = m->local_of[(size_t)global_ref];
    return SWB_OK;
}

const int64_t *swb_multi_shard_refs(const swb_multi *m, int32_t d, int64_t *n)
{
    if (!m || d < 0 || d >= (int32_t)m->ids.size()) { if (n) *n = 0; return nullptr; }
    if (n) *n = (int64_t)m->ids[(size_t)d].size();
    return m->ids[(size_t)d].data();
}

}  // extern "C"

// one align call per shard (phase 1), then each mode's per-read records exchanged between the devices (phase 2) and the
// shards' results fetched (phase 3).  `who` names the entry point in the messages.
static int multi_align(const char *who, swb_multi *m, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets,
                       int32_t match, int32_t mismatch, int32_t gap, uint32_t flags, const Selection &sel, swb_multi_result **out)
{
    if (!m || !out) return fail(SWB_E_INVALID, "swb_multi_align: null argument");
    *out = nullptr;
    const int n = (int)m->ctx.size();
    if (sel.mode != Selection::NONE && n > kMaxHitsWorld) return fail(SWB_E_UNSUPPORTED, std::string(who) + ": more than 64 devices");
    for (int d = 0; d < n; ++d)
        if (!m->rs[(size_t)d]) return fail(SWB_E_INVALID, "swb_multi_align: no reference set loaded");
    std::lock_guard<std::mutex> lk(m->mu);
    const auto t0 = std::chrono::steady_clock::now();
    std::unique_ptr<swb_multi_result> res(new swb_multi_result());
    res->m = m; res->n_reads = n_reads; res->sel = sel;
    res->shard.assign((size_t)n, nullptr);
    auto drop = [&] { for (swb_result *r : res->shard) if (r) swb_result_free(r); res->shard.clear(); };

    std::vector<int> rcs((size_t)n, SWB_OK);
    std::vector<std::string> errs((size_t)n);
    // phase 1: every device aligns all reads against its shard; the results stay in HBM
    {
        std::vector<std::thread> th;
        for (int d = 0; d < n; ++d)
            th.emplace_back([&, d] {
                rcs[(size_t)d] = align_host(m->ctx[(size_t)d], m->rs[(size_t)d], n_reads, read_bytes, read_offsets, match, mismatch, gap,
                                            flags | SWB_F_NO_FETCH, sel, &res->shard[(size_t)d]);
                if (rcs[(size_t)d]) errs[(size_t)d] = swb_last_error();
            });
        for (auto &t : th) t.join();
    }
    for (int d = 0; d < n; ++d)
        if (rcs[(size_t)d]) { const int rc = rcs[(size_t)d]; const std::string e = errs[(size_t)d]; drop(); return fail(rc, "shard " + std::to_string(d) + ": " + e); }

    // phase 2: the best hits (and the mode's lists) -> global ids -> all-gathered over NVLink -> merged, on every device's
    // engine stream.  Both strands: the shards' records hold oriented local ids 2r + s, localized to oriented global ids
    // 2 * gid + s, so the merge's order is the single-context order over the oriented references
    const auto t1 = std::chrono::steady_clock::now();
    const bool both = (flags & SWB_F_BOTH_STRANDS) != 0;
    // all-hits mode: the shards' list lengths are known on the host after their calls; T = the largest
    int64_t T = 0;
    if (sel.mode == Selection::MARGIN)
        for (int d = 0; d < n; ++d) T = std::max(T, res->shard[(size_t)d]->n_hits);
    for (int d = 0; d < n; ++d) {
        swb_ctx *c = m->ctx[(size_t)d];
        GatherBufs &g = m->g[(size_t)d];
        const swb_result *sh = res->shard[(size_t)d];
        const int64_t *ids = both ? g.oids.p : g.ids.p;
        const int64_t n_ids = both ? 2 * g.n_ids : g.n_ids;
        cudaError_t e = cudaSetDevice(c->device);
        if (e == cudaSuccess) e = enqueue_localize(g, ids, n_ids, sh->d_best.p, n_reads, n, c->stream);
        if (e == cudaSuccess && sel.mode == Selection::TOP_K)
            e = enqueue_localize_hits(g, ids, n_ids, sh->d_hits.p, n_reads, sel.top_k, n, c->stream);
        if (e == cudaSuccess && sel.mode == Selection::MARGIN) e = enqueue_localize_all_hits(g, ids, n_ids, sh, T, n, c->stream);
        if (e != cudaSuccess) { drop(); return cuda_fail(e, "swb_multi_align: best hits -> global ids"); }
    }
    // the gathers of all devices, as one NCCL group
    NcclApi *a = n > 1 ? nccl_api() : nullptr;
    ncclResult_t r = a ? a->GroupStart() : ncclSuccess;
    int rc = r == ncclSuccess ? SWB_OK : nccl_fail(r, "ncclGroupStart");
    for (int d = 0; d < n && !rc; ++d) {
        GatherBufs &g = m->g[(size_t)d];
        const ncclComm_t comm = a ? m->comms[(size_t)d] : nullptr;
        cudaStream_t st = m->ctx[(size_t)d]->stream;
        rc = gather(g.send.p, g.gathered.p, (size_t)n_reads * 4, ncclInt32, comm, n, st);
        if (!rc && sel.mode == Selection::TOP_K) rc = gather(g.hsend.p, g.hgathered.p, (size_t)n_reads * sel.top_k * 4, ncclInt32, comm, n, st);
        if (!rc && sel.mode == Selection::MARGIN)
            rc = gather(res->shard[(size_t)d]->d_hit_off.p, g.aoffs.p, (size_t)n_reads + 1, ncclInt64, comm, n, st);
        if (!rc && sel.mode == Selection::MARGIN) rc = gather(g.asend.p, g.alists.p, (size_t)T * 4, ncclInt32, comm, n, st);
    }
    if (a && (r = a->GroupEnd()) != ncclSuccess && !rc) rc = nccl_fail(r, "ncclGroupEnd");
    if (rc) { const std::string err = swb_last_error(); drop(); return fail(rc, "swb_multi_align: " + err); }
    // the merges of every device; the host copies come from device 0
    res->merged.assign((size_t)n_reads * 4, 0);
    if (sel.mode == Selection::TOP_K) res->merged_hits.assign((size_t)n_reads * sel.top_k * 4, 0);
    for (int d = 0; d < n; ++d) {
        swb_ctx *c = m->ctx[(size_t)d];
        GatherBufs &g = m->g[(size_t)d];
        cudaError_t e = cudaSetDevice(c->device);
        if (e == cudaSuccess) e = enqueue_merge(g, n_reads, n, c->stream);
        if (e == cudaSuccess && d == 0 && n_reads)
            e = cudaMemcpyAsync(res->merged.data(), g.merged.p, (size_t)n_reads * 16, cudaMemcpyDeviceToHost, c->stream);
        if (sel.mode == Selection::TOP_K && n_reads) {
            if (e == cudaSuccess) e = enqueue_merge_hits(g, n_reads, sel.top_k, n, c->stream);
            if (e == cudaSuccess && d == 0)
                e = cudaMemcpyAsync(res->merged_hits.data(), g.hmerged.p, (size_t)n_reads * sel.top_k * 16, cudaMemcpyDeviceToHost, c->stream);
        }
        if (e != cudaSuccess) { drop(); return cuda_fail(e, "swb_multi_align: merge"); }
    }
    // all-hits mode: the lists are merged on device 0 (one more host sync there for the merged length)
    if (sel.mode == Selection::MARGIN) {
        const cudaError_t e = cudaSetDevice(m->ctx[0]->device);
        rc = e == cudaSuccess ? merge_all_hits(m->g[0], n, n_reads, T, sel.min_score, sel.margin, m->ctx[0]->stream)
                              : cuda_fail(e, "swb_multi_align_all_hits: merge");
        if (rc) { const std::string err = swb_last_error(); drop(); return fail(rc, err); }
        res->merged_off = m->g[0].h_off; res->merged_list = m->g[0].h_list;
    }
    for (int d = 0; d < n; ++d) {
        cudaSetDevice(m->ctx[(size_t)d]->device);
        const cudaError_t e = cudaStreamSynchronize(m->ctx[(size_t)d]->stream);
        if (e != cudaSuccess) { drop(); return cuda_fail(e, "swb_multi_align: all-gather"); }
    }
    const auto t2 = std::chrono::steady_clock::now();
    // phase 3: results to the host (unless the caller keeps them in HBM), all devices at once
    if (!(flags & SWB_F_NO_FETCH)) {
        std::vector<std::thread> th;
        for (int d = 0; d < n; ++d)
            th.emplace_back([&, d] {
                rcs[(size_t)d] = swb_result_fetch(res->shard[(size_t)d]);
                if (rcs[(size_t)d]) errs[(size_t)d] = swb_last_error();
            });
        for (auto &t : th) t.join();
        for (int d = 0; d < n; ++d)
            if (rcs[(size_t)d]) { const int rc = rcs[(size_t)d]; const std::string e = errs[(size_t)d]; drop(); return fail(rc, "shard " + std::to_string(d) + ": " + e); }
    }
    const auto t3 = std::chrono::steady_clock::now();
    res->stats[0] = std::chrono::duration<double, std::milli>(t3 - t0).count();
    for (int d = 0; d < n; ++d) res->stats[1] = std::max(res->stats[1], res->shard[(size_t)d]->stats[5]);
    res->stats[2] = std::chrono::duration<double, std::milli>(t2 - t1).count();
    *out = res.release();
    return SWB_OK;
}

extern "C" {

int swb_multi_align(swb_multi *m, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets, int32_t match,
                    int32_t mismatch, int32_t gap, uint32_t flags, swb_multi_result **out)
{
    return multi_align("swb_multi_align", m, n_reads, read_bytes, read_offsets, match, mismatch, gap, flags, Selection{}, out);
}

int swb_multi_align_hits(swb_multi *m, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets, int32_t match,
                         int32_t mismatch, int32_t gap, uint32_t flags, int32_t top_k, int32_t min_score, swb_multi_result **out)
{
    const Selection sel{Selection::TOP_K, top_k, min_score};
    if (out) *out = nullptr;
    const int rc = check_selection("swb_multi_align_hits", sel);
    return rc ? rc : multi_align("swb_multi_align_hits", m, n_reads, read_bytes, read_offsets, match, mismatch, gap, flags, sel, out);
}

int swb_multi_align_all_hits(swb_multi *m, int64_t n_reads, const char *read_bytes, const int64_t *read_offsets, int32_t match,
                             int32_t mismatch, int32_t gap, uint32_t flags, int32_t min_score, int32_t margin, swb_multi_result **out)
{
    const Selection sel{Selection::MARGIN, 0, min_score, margin};
    if (out) *out = nullptr;
    const int rc = check_selection("swb_multi_align_all_hits", sel);
    return rc ? rc : multi_align("swb_multi_align_all_hits", m, n_reads, read_bytes, read_offsets, match, mismatch, gap, flags, sel, out);
}

void swb_multi_result_free(swb_multi_result *res)
{
    if (!res) return;
    for (swb_result *r : res->shard) if (r) swb_result_free(r);
    delete res;
}

swb_result *swb_multi_result_shard(swb_multi_result *res, int32_t d)
{
    return (res && d >= 0 && d < (int32_t)res->shard.size()) ? res->shard[(size_t)d] : nullptr;
}
const int32_t *swb_multi_result_best_hits(const swb_multi_result *res) { return res ? res->merged.data() : nullptr; }
const int32_t *swb_multi_result_hits(const swb_multi_result *res, int32_t *top_k)
{
    const bool ok = res && res->sel.mode == Selection::TOP_K;
    if (top_k) *top_k = ok ? res->sel.top_k : 0;
    return ok ? res->merged_hits.data() : nullptr;
}
const int64_t *swb_multi_result_hit_offsets(const swb_multi_result *res, int64_t *n_hits)
{
    const bool ok = res && res->sel.mode == Selection::MARGIN;
    if (n_hits) *n_hits = ok ? res->merged_off[(size_t)res->n_reads] : 0;
    return ok ? res->merged_off.data() : nullptr;
}
const int32_t *swb_multi_result_hit_list(const swb_multi_result *res) { return (res && res->sel.mode == Selection::MARGIN) ? res->merged_list.data() : nullptr; }
int swb_multi_result_stats(const swb_multi_result *res, double *out, int n)
{
    if (!res || !out) return fail(SWB_E_INVALID, "swb_multi_result_stats: null");
    for (int k = 0; k < n && k < 3; ++k) out[k] = res->stats[k];
    return SWB_OK;
}

}  // extern "C"
