// swb_hits.cu -- per-read top-k selection of the hits mode (swb_align_hits, include/swb200.h).
//
// A read's k best references under the best-hit order (score descending, then reference ascending) are picked from
// the exact score rows scores[ref * n_reads + q] of one reference set.  One warp keeps a sorted list of up to 32
// keys, one per lane; a key is (score << 32) | ~ref, so "larger key" is exactly "earlier in the order".  A thread-
// per-read loop over 10^4 - 10^5 references would leave most of the GPU idle, so the references are cut into
// chunks: kernel 1 gives every (read, chunk) a warp and a partial top-k, kernel 2 merges a read's partial lists.
//
// The all-hits mode (swb_align_all_hits) lists every pair within a margin of the read's best score; its lists have no
// fixed length, so it has kernels of its own over the same (read, chunk) warps: a per-read maximum, a marking pass that
// sets the emit's selection bits, and the final list build (count, exclusive scan, write in reference order, stable
// radix sort by read and score descending).
#include "swb_internal.h"

#include <algorithm>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

namespace swb {

namespace {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ uint64_t hit_key(int32_t score, int64_t ref)
{
    return ((uint64_t)(uint32_t)score << 32) | (uint64_t)(0xffffffffu - (uint32_t)ref);
}

// the warp's list: lane h < k holds the h-th largest key seen so far (0 = empty).  Every lane offers `x` when `ok`;
// offers are inserted one at a time in lane order, the rest of the list moves down one lane.
__device__ __forceinline__ void warp_offer(uint64_t &mine, uint64_t x, bool ok, int k, int lane)
{
    const uint64_t bar = __shfl_sync(FULL, mine, k - 1);          // every lane takes part in the shuffle
    uint32_t m = __ballot_sync(FULL, ok && x > bar);
    while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const uint64_t v = __shfl_sync(FULL, x, src);
        if (v <= __shfl_sync(FULL, mine, k - 1)) continue;          // an earlier offer of this round raised the bar
        const int pos = __popc(__ballot_sync(FULL, lane < k && mine > v));
        const uint64_t up = __shfl_up_sync(FULL, mine, 1);
        if (lane > pos) mine = up;
        if (lane == pos) mine = v;
    }
}

// warp w = (slot, chunk): top k of read slots[slot]'s references [chunk * chunk_refs, +chunk_refs) with score >= 1
__global__ void __launch_bounds__(128) hits_partial_kernel(const int32_t *__restrict__ scores, int64_t n_refs, int64_t n_reads,
                                                           const int32_t *slots, int64_t slot0, int64_t n_slots,
                                                           int64_t chunk_refs, int n_chunks, int k, uint64_t *part)
{
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_slots * n_chunks) return;                          // whole warps
    const int64_t slot = slot0 + w / n_chunks;
    const int64_t c = w % n_chunks;
    const int32_t q = slots ? slots[slot] : (int32_t)slot;
    uint64_t mine = 0;
    if (q >= 0) {
        const int64_t r0 = c * chunk_refs, r1 = min(n_refs, r0 + chunk_refs);
        for (int64_t b = r0; b < r1; b += 4 * 32) {
            int32_t s[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {                          // four loads in flight before the first ballot
                const int64_t r = b + u * 32 + lane;
                s[u] = r < r1 ? __ldg(scores + r * n_reads + q) : 0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) warp_offer(mine, hit_key(s[u], b + u * 32 + lane), s[u] >= 1, k, lane);
        }
    }
    if (lane < k) part[w * k + lane] = mine;
}

// warp per slot: merge the slot's partial lists.  Entry h is TAKEN if it exists and (score >= min_score, or h = 0 and
// with_best: the read's best pair).  Taken entries go to hits[slot * k + h] = (score, ref, 0, 0), the others are
// padding (0, -1, 0, 0); a taken entry also sets bit slot * bit_slot + ref * bit_ref of `bits`.  Oriented (both strands,
// the refs are oriented o = 2r + s): bit slot * bit_slot + s * bit_ref + r, the bit of strand s's half of the read pair.
template <bool Oriented>
__global__ void __launch_bounds__(128) hits_merge_kernel(const uint64_t *part, int n_chunks, int k, const int32_t *slots,
                                                         int64_t slot0, int64_t n_slots, int32_t min_score, int with_best,
                                                         int4 *hits, uint32_t *bits, int64_t bit_slot, int64_t bit_ref)
{
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_slots) return;
    const int64_t slot = slot0 + w;
    const int32_t q = slots ? slots[slot] : (int32_t)slot;
    if (q < 0) return;
    const int64_t n = (int64_t)n_chunks * k;
    const uint64_t *in = part + w * n;
    uint64_t mine = 0;
    for (int64_t b = 0; b < n; b += 32) {
        const uint64_t x = b + lane < n ? in[b + lane] : 0;
        warp_offer(mine, x, x != 0, k, lane);
    }
    if (lane >= k) return;
    const int32_t score = (int32_t)(mine >> 32);
    const int32_t ref = (int32_t)(0xffffffffu - (uint32_t)mine);
    const bool take = mine != 0 && (score >= min_score || (lane == 0 && with_best));
    if (hits) hits[slot * k + lane] = take ? make_int4(score, ref, 0, 0) : make_int4(0, -1, 0, 0);
    if (bits && take) {
        const int64_t bit = Oriented ? slot * bit_slot + (int64_t)(ref & 1) * bit_ref + (ref >> 1) : slot * bit_slot + (int64_t)ref * bit_ref;
        atomicOr(bits + (bit >> 5), 1u << (bit & 31));
    }
}

int64_t chunk_refs_of(int64_t n_refs)
{
    // at least 1024 references per warp (32 rounds of the list), at most 256 chunks per read (bounds the partial lists)
    return std::max<int64_t>(1024, ((n_refs + 255) / 256 + 31) / 32 * 32);
}

// ---- all-hits mode (swb_align_all_hits): every pair with score >= max(min_score, best_q - margin) ------------------
// The same warp per (slot, chunk of references) as hits_partial_kernel.  A read's best key is the largest hit_key of
// its pairs with score >= 1: the best score and, on ties, the lowest reference -- the read's best pair.

// listed iff score >= this bar (>= 1); best_q - margin in 64 bits, so a large margin cannot wrap
__device__ __forceinline__ int64_t margin_bar(uint64_t best_key, int32_t min_score, int32_t margin)
{
    return max((int64_t)min_score, (int64_t)(best_key >> 32) - (int64_t)margin);
}

__device__ __forceinline__ uint64_t warp_max_u64(uint64_t v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, (uint64_t)__shfl_xor_sync(FULL, v, o));
    return v;
}

// best[slot] = max(best[slot], largest key of the chunk); best is zeroed by the caller
__global__ void __launch_bounds__(128) margin_best_kernel(const int32_t *__restrict__ scores, int64_t n_refs, int64_t n_reads,
                                                          const int32_t *slots, int64_t n_slots, int64_t chunk_refs, int n_chunks,
                                                          unsigned long long *best)
{
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_slots * n_chunks) return;                          // whole warps
    const int64_t slot = w / n_chunks, c = w % n_chunks;
    const int32_t q = slots ? slots[slot] : (int32_t)slot;
    if (q < 0) return;
    const int64_t r0 = c * chunk_refs, r1 = min(n_refs, r0 + chunk_refs);
    uint64_t mine = 0;
    for (int64_t r = r0 + lane; r < r1; r += 32) {
        const int32_t s = __ldg(scores + r * n_reads + q);
        if (s >= 1) mine = max(mine, hit_key(s, r));
    }
    mine = warp_max_u64(mine);
    if (lane == 0 && mine) atomicMax(best + slot, (unsigned long long)mine);
}

// sets the emit's selection bit of every listed pair of the chunk and, with_best, of the read's best pair.  Bit layout
// as hits_merge_kernel: slot * bit_slot + ref * bit_ref, or, oriented, slot * bit_slot + (o & 1) * bit_ref + (o >> 1)
__global__ void __launch_bounds__(128) margin_mark_kernel(const int32_t *__restrict__ scores, int64_t n_refs, int64_t n_reads,
                                                          const int32_t *slots, int64_t n_slots, int64_t chunk_refs, int n_chunks,
                                                          const unsigned long long *best, int32_t min_score, int32_t margin,
                                                          int with_best, uint32_t *bits, int64_t bit_slot, int64_t bit_ref, int oriented)
{
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_slots * n_chunks) return;
    const int64_t slot = w / n_chunks, c = w % n_chunks;
    const int32_t q = slots ? slots[slot] : (int32_t)slot;
    if (q < 0) return;
    const uint64_t key = best[slot];
    const int64_t bar = margin_bar(key, min_score, margin);
    const int64_t best_ref = (with_best && key) ? (int64_t)(0xffffffffu - (uint32_t)key) : -1;
    const int64_t r0 = c * chunk_refs, r1 = min(n_refs, r0 + chunk_refs);
    for (int64_t r = r0 + lane; r < r1; r += 32) {
        const int32_t s = __ldg(scores + r * n_reads + q);
        if (s < bar && r != best_ref) continue;
        const int64_t bit = oriented ? slot * bit_slot + (r & 1) * bit_ref + (r >> 1) : slot * bit_slot + r * bit_ref;
        atomicOr(bits + (bit >> 5), 1u << (bit & 31));
    }
}

// the final lists, over all reads (slot = read): listed pairs per (read, chunk)
__global__ void __launch_bounds__(128) margin_count_kernel(const int32_t *__restrict__ scores, int64_t n_refs, int64_t n_reads,
                                                           int64_t chunk_refs, int n_chunks, const unsigned long long *best,
                                                           int32_t min_score, int32_t margin, int64_t *count)
{
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_reads * n_chunks) return;
    const int64_t q = w / n_chunks, c = w % n_chunks;
    const int64_t bar = margin_bar(best[q], min_score, margin);
    const int64_t r0 = c * chunk_refs, r1 = min(n_refs, r0 + chunk_refs);
    int n = 0;
    for (int64_t r = r0 + lane; r < r1; r += 32) n += __ldg(scores + r * n_reads + q) >= bar;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(FULL, n, o);
    if (lane == 0) count[w] = n;
}

// (read, chunk) w writes its listed pairs from off[w] on, in reference order: (score, ref, 0, 0) and the sort key
// (read, score descending)
__global__ void __launch_bounds__(128) margin_write_kernel(const int32_t *__restrict__ scores, int64_t n_refs, int64_t n_reads,
                                                           int64_t chunk_refs, int n_chunks, const unsigned long long *best,
                                                           int32_t min_score, int32_t margin, const int64_t *off, int4 *list,
                                                           uint64_t *keys, uint32_t *idx)
{
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_reads * n_chunks) return;
    const int64_t q = w / n_chunks, c = w % n_chunks;
    const int64_t bar = margin_bar(best[q], min_score, margin);
    const int64_t r0 = c * chunk_refs, r1 = min(n_refs, r0 + chunk_refs);
    int64_t pos = off[w];
    for (int64_t b = r0; b < r1; b += 32) {
        const int64_t r = b + lane;
        const int32_t s = r < r1 ? __ldg(scores + r * n_reads + q) : 0;
        const bool take = r < r1 && s >= bar;
        const uint32_t m = __ballot_sync(FULL, take);
        if (take) {
            const int64_t k = pos + __popc(m & ((1u << lane) - 1u));
            list[k] = make_int4(s, (int32_t)r, 0, 0);
            keys[k] = ((uint64_t)q << 31) | (uint64_t)(0x7fffffff - s);
            idx[k] = (uint32_t)k;
        }
        pos += __popc(m);
    }
}

// hit_off[q] = off[q * n_chunks]
__global__ void margin_read_offsets_kernel(const int64_t *off, int64_t n_reads, int n_chunks, int64_t *hit_off)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q <= n_reads) hit_off[q] = off[q * n_chunks];
}

__global__ void gather_list_kernel(const int4 *in, const uint32_t *order, int64_t n, int4 *out)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k < n) out[k] = in[order[k]];
}

}  // namespace

size_t select_hits_tmp_elems(int64_t n_refs, int64_t n_slots, int k)
{
    const int64_t n_chunks = std::max<int64_t>(1, (n_refs + chunk_refs_of(n_refs) - 1) / chunk_refs_of(n_refs));
    const int64_t per = std::max<int64_t>(1, ((int64_t)8 << 20) / (n_chunks * k));       // <= 64 MB of partial lists
    return (size_t)(std::max<int64_t>(1, std::min(n_slots, per)) * n_chunks * k);
}

cudaError_t launch_select_hits(const int32_t *scores, int64_t n_refs, int64_t n_reads, const int32_t *slots, int64_t n_slots,
                               int k, int32_t min_score, int with_best, int4 *hits, uint32_t *bits, int64_t bit_slot,
                               int64_t bit_ref, bool oriented_bits, uint64_t *tmp, size_t tmp_elems, cudaStream_t st)
{
    if (n_slots <= 0) return cudaSuccess;
    const int64_t chunk = chunk_refs_of(n_refs);
    const int n_chunks = (int)std::max<int64_t>(1, (n_refs + chunk - 1) / chunk);
    const int64_t per = std::max<int64_t>(1, (int64_t)tmp_elems / ((int64_t)n_chunks * k));
    const int threads = 128;
    for (int64_t s0 = 0; s0 < n_slots; s0 += per) {
        const int64_t ns = std::min(per, n_slots - s0);
        const int64_t warps1 = ns * n_chunks;
        hits_partial_kernel<<<(unsigned)((warps1 * 32 + threads - 1) / threads), threads, 0, st>>>(scores, n_refs, n_reads, slots, s0, ns,
                                                                                                 chunk, n_chunks, k, tmp);
        const unsigned blocks2 = (unsigned)((ns * 32 + threads - 1) / threads);
        if (oriented_bits)
            hits_merge_kernel<true><<<blocks2, threads, 0, st>>>(tmp, n_chunks, k, slots, s0, ns, min_score, with_best, hits, bits, bit_slot, bit_ref);
        else
            hits_merge_kernel<false><<<blocks2, threads, 0, st>>>(tmp, n_chunks, k, slots, s0, ns, min_score, with_best, hits, bits, bit_slot, bit_ref);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

static unsigned warp_blocks(int64_t warps, int threads) { return (unsigned)((warps * 32 + threads - 1) / threads); }

cudaError_t launch_select_margin(const int32_t *scores, int64_t n_refs, int64_t n_reads, const int32_t *slots, int64_t n_slots,
                                 int32_t min_score, int32_t margin, int with_best, uint32_t *bits, int64_t bit_slot, int64_t bit_ref,
                                 bool oriented_bits, uint64_t *best, cudaStream_t st)
{
    if (n_slots <= 0) return cudaSuccess;
    const int64_t chunk = chunk_refs_of(n_refs);
    const int n_chunks = (int)std::max<int64_t>(1, (n_refs + chunk - 1) / chunk);
    const int threads = 128;
    cudaError_t e = cudaMemsetAsync(best, 0, (size_t)n_slots * 8, st);
    if (e != cudaSuccess) return e;
    auto *b = reinterpret_cast<unsigned long long *>(best);
    margin_best_kernel<<<warp_blocks(n_slots * n_chunks, threads), threads, 0, st>>>(scores, n_refs, n_reads, slots, n_slots, chunk, n_chunks, b);
    if (bits)
        margin_mark_kernel<<<warp_blocks(n_slots * n_chunks, threads), threads, 0, st>>>(scores, n_refs, n_reads, slots, n_slots, chunk,
                                                                                         n_chunks, b, min_score, margin, with_best, bits,
                                                                                         bit_slot, bit_ref, oriented_bits ? 1 : 0);
    return cudaGetLastError();
}

size_t margin_count_elems(int64_t n_refs, int64_t n_reads)
{
    const int64_t chunk = chunk_refs_of(n_refs);
    return (size_t)(n_reads * std::max<int64_t>(1, (n_refs + chunk - 1) / chunk) + 1);
}

size_t margin_list_tmp_bytes(int64_t n_refs, int64_t n_reads, int64_t n_hits)
{
    const int64_t chunk = chunk_refs_of(n_refs);
    const int64_t n_chunks = std::max<int64_t>(1, (n_refs + chunk - 1) / chunk);
    size_t a = 0, b = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, a, (const int64_t *)nullptr, (int64_t *)nullptr, (int)(n_reads * n_chunks + 1));
    cub::DeviceRadixSort::SortPairs(nullptr, b, (const uint64_t *)nullptr, (uint64_t *)nullptr, (const uint32_t *)nullptr,
                                    (uint32_t *)nullptr, (int)n_hits);
    return std::max(a, b);
}

cudaError_t launch_margin_count(const int32_t *scores, int64_t n_refs, int64_t n_reads, int32_t min_score, int32_t margin,
                                const uint64_t *best, int64_t *count, int64_t *off, void *tmp, size_t tmp_bytes, cudaStream_t st)
{
    const int64_t chunk = chunk_refs_of(n_refs);
    const int n_chunks = (int)std::max<int64_t>(1, (n_refs + chunk - 1) / chunk);
    const int64_t nw = n_reads * n_chunks;
    const int threads = 128;
    cudaError_t e = cudaMemsetAsync(count + nw, 0, 8, st);
    if (e != cudaSuccess) return e;
    if (nw)
        margin_count_kernel<<<warp_blocks(nw, threads), threads, 0, st>>>(scores, n_refs, n_reads, chunk, n_chunks,
                                                                          reinterpret_cast<const unsigned long long *>(best),
                                                                          min_score, margin, count);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    return cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, count, off, (int)(nw + 1), st);
}

cudaError_t launch_margin_write(const int32_t *scores, int64_t n_refs, int64_t n_reads, int32_t min_score, int32_t margin,
                                const uint64_t *best, const int64_t *off, int64_t n_hits, int4 *list_tmp, uint64_t *keys_tmp,
                                uint64_t *keys_sorted, uint32_t *idx_tmp, uint32_t *order, int4 *list, int64_t *hit_off, void *tmp,
                                size_t tmp_bytes, cudaStream_t st)
{
    const int64_t chunk = chunk_refs_of(n_refs);
    const int n_chunks = (int)std::max<int64_t>(1, (n_refs + chunk - 1) / chunk);
    const int64_t nw = n_reads * n_chunks;
    const int threads = 128;
    margin_read_offsets_kernel<<<(unsigned)((n_reads + 1 + 255) / 256), 256, 0, st>>>(off, n_reads, n_chunks, hit_off);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess || n_hits == 0) return e;
    margin_write_kernel<<<warp_blocks(nw, threads), threads, 0, st>>>(scores, n_refs, n_reads, chunk, n_chunks,
                                                                      reinterpret_cast<const unsigned long long *>(best), min_score,
                                                                      margin, off, list_tmp, keys_tmp, idx_tmp);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    // stable: equal (read, score) keep the reference order of the write
    int end_bit = 31;
    while (end_bit < 64 && (n_reads - 1) >> (end_bit - 31)) ++end_bit;
    if ((e = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys_tmp, keys_sorted, idx_tmp, order, (int)n_hits, 0, end_bit, st)))
        return e;
    gather_list_kernel<<<(unsigned)((n_hits + 255) / 256), 256, 0, st>>>(list_tmp, order, n_hits, list);
    return cudaGetLastError();
}

}  // namespace swb
