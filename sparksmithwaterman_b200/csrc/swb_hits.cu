// swb_hits.cu -- per-read top-k selection of the hits mode (swb_align_hits, include/swb200.h).
//
// A read's k best references under the best-hit order (score descending, then reference ascending) are picked from
// the exact score rows scores[ref * n_reads + q] of one reference set.  One warp keeps a sorted list of up to 32
// keys, one per lane; a key is (score << 32) | ~ref, so "larger key" is exactly "earlier in the order".  A thread-
// per-read loop over 10^4 - 10^5 references would leave most of the GPU idle, so the references are cut into
// chunks: kernel 1 gives every (read, chunk) a warp and a partial top-k, kernel 2 merges a read's partial lists.
#include "swb_internal.h"

#include <algorithm>

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

}  // namespace swb
