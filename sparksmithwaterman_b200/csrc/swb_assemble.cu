// swb_assemble.cu -- device-side assembly of the final result of one align call.
// The batches (short path: sorted by (read slot, ref, i, j); wide path: (local pair, i, j))
// hold disjoint pairs.  A stable radix sort of all cells by the ABI pair index
// p = ref * n_reads + read therefore yields the reference's order: pairs as MapRef visits them
// (Distribution.java:419-426), and inside a pair the row-major max-cell list
// (SmithWaterman.java:157-185).  Cells, beginnings, lengths and the packed alignment columns are
// then gathered into dense arrays (ops compacted to their real length), so that the host fetch is
// a handful of large device-to-pinned-host copies.
#include "swb_internal.h"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

namespace swb {

__device__ __forceinline__ int find_batch(const BatchDesc *b, int nb, uint32_t src)
{
    int lo = 0, hi = nb;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (b[mid].base <= src) lo = mid; else hi = mid; }
    return lo;
}

// keep (hits mode): cells of pairs without their bit sort after every kept cell, as pair + n_pairs
__global__ void cell_pairs_kernel(const BatchDesc *batches, int nb, uint32_t n_cells, int64_t n_refs, int64_t n_reads,
                                  const uint32_t *keep, uint64_t *pair_of, uint32_t *src)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_cells) return;
    const BatchDesc &B = batches[find_batch(batches, nb, k)];
    const uint64_t key = B.keys[k - B.base];
    uint64_t p;
    if (B.wide) p = (uint64_t)B.pair_map[wide::wide_key_pair(key)];
    else {
        const uint64_t pk = key_pair(key);
        const uint64_t slot = pk / (uint64_t)n_refs, ref = pk - slot * (uint64_t)n_refs;
        p = ref * (uint64_t)n_reads + (uint64_t)B.slot_read[slot];
    }
    if (keep && !((keep[p >> 5] >> (p & 31)) & 1u)) p += (uint64_t)n_refs * (uint64_t)n_reads;
    pair_of[k] = p;
    src[k] = k;
}

__global__ void gather_cells_kernel(const BatchDesc *batches, int nb, uint32_t n_cells, const uint32_t *order,
                                    int32_t *cells, int32_t *beginnings, int32_t *op_lens, int64_t *words)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_cells) return;
    const uint32_t s = order[k];
    const BatchDesc &B = batches[find_batch(batches, nb, s)];
    const uint32_t l = s - B.base;
    const uint64_t key = B.keys[l];
    cells[2 * k] = (int32_t)(B.wide ? wide::wide_key_i(key) : key_i(key));
    cells[2 * k + 1] = (int32_t)(B.wide ? wide::wide_key_j(key) : key_j(key));
    beginnings[k] = B.beg[l];
    const int32_t len = B.oplen[l];
    op_lens[k] = len;
    words[k] = ((int64_t)len + 15) >> 4;
}

// eight lanes per cell (an alignment of ~170 columns is 11 words): copy its packed columns into the dense buffer
__global__ void gather_ops_kernel(const BatchDesc *batches, int nb, uint32_t n_cells, const uint32_t *order,
                                  const int64_t *ops_off, uint32_t *ops_out)
{
    const uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    const int lane = threadIdx.x & 7;
    if (k >= n_cells) return;
    const uint32_t s = order[k];
    const BatchDesc &B = batches[find_batch(batches, nb, s)];
    const uint32_t *in = B.ops + (int64_t)(s - B.base) * B.ops_stride;
    uint32_t *out = ops_out + ops_off[k];
    const int64_t n = ops_off[k + 1] - ops_off[k];
    for (int64_t w = lane; w < n; w += 8) out[w] = in[w];
}

// cell_off[p] = first sorted cell whose pair index >= p  (p = 0 .. n_pairs)
__global__ void pair_offsets_kernel(const uint64_t *pair_sorted, uint32_t n_cells, int64_t n_pairs, int64_t *cell_off)
{
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p > n_pairs) return;
    uint32_t lo = 0, hi = n_cells;
    while (lo < hi) { const uint32_t mid = lo + ((hi - lo) >> 1); if (pair_sorted[mid] < (uint64_t)p) lo = mid + 1; else hi = mid; }
    cell_off[p] = lo;
}

// (i, j) of each read's best hit = first max cell of pair (best ref, read)
__global__ void best_cells_kernel2(int32_t *best, int64_t n_reads, const int64_t *cell_off, const int32_t *cells)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_reads) return;
    const int ref = best[4 * q + 1];
    if (ref < 0 || best[4 * q] <= 0) return;
    const int64_t p = (int64_t)ref * n_reads + q;
    if (cell_off[p + 1] > cell_off[p]) {
        best[4 * q + 2] = cells[2 * cell_off[p]];
        best[4 * q + 3] = cells[2 * cell_off[p] + 1];
    }
}

__device__ __forceinline__ uint32_t lower_bound_u64(const uint64_t *a, uint32_t n, uint64_t v)
{
    uint32_t lo = 0, hi = n;
    while (lo < hi) { const uint32_t mid = lo + ((hi - lo) >> 1); if (a[mid] < v) lo = mid + 1; else hi = mid; }
    return lo;
}

__global__ void kept_count_kernel(const uint64_t *pair_sorted, uint32_t n_cells, int64_t n_pairs, uint32_t *n_kept)
{
    *n_kept = lower_bound_u64(pair_sorted, n_cells, (uint64_t)n_pairs);
}

// hits mode, thread per read: (i, j) of every hit = its pair's first kept cell; a best hit that is not a hit (score below
// min_score) takes the first of its pair's dropped cells, which sort as pair + n_pairs
__global__ void hit_cells_kernel(const BatchDesc *batches, int nb, const uint64_t *pair_sorted, const uint32_t *order,
                                 uint32_t n_all, int64_t n_pairs, int64_t n_reads, const int64_t *cell_off, const int32_t *cells,
                                 int32_t *best, int32_t *hits, int k)
{
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_reads) return;
    for (int h = 0; h < k; ++h) {
        int32_t *e = hits + (q * k + h) * 4;
        if (e[1] < 0) break;
        const int64_t p = (int64_t)e[1] * n_reads + q;
        if (cell_off[p + 1] > cell_off[p]) { e[2] = cells[2 * cell_off[p]]; e[3] = cells[2 * cell_off[p] + 1]; }
    }
    const int ref = best[4 * q + 1];
    if (ref < 0 || best[4 * q] <= 0) return;
    const int64_t p = (int64_t)ref * n_reads + q;
    if (cell_off[p + 1] > cell_off[p]) return;                    // a hit: best_cells_kernel2 has its cell
    const uint32_t c = lower_bound_u64(pair_sorted, n_all, (uint64_t)(p + n_pairs));
    if (c >= n_all || pair_sorted[c] != (uint64_t)(p + n_pairs)) return;
    const uint32_t s = order[c];
    const BatchDesc &B = batches[find_batch(batches, nb, s)];
    const uint64_t key = B.keys[s - B.base];
    best[4 * q + 2] = (int32_t)(B.wide ? wide::wide_key_i(key) : key_i(key));
    best[4 * q + 3] = (int32_t)(B.wide ? wide::wide_key_j(key) : key_j(key));
}

// all-hits mode, thread per list entry: its read is found in hit_off, (i, j) = the pair's first kept cell
__global__ void list_cells_kernel(const int64_t *hit_off, int64_t n_reads, int32_t *list, int64_t n_hits, const int64_t *cell_off,
                                  const int32_t *cells)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= n_hits) return;
    int64_t lo = 0, hi = n_reads;                                  // q = last read with hit_off[q] <= k
    while (hi - lo > 1) { const int64_t mid = (lo + hi) >> 1; if (hit_off[mid] <= k) lo = mid; else hi = mid; }
    int32_t *e = list + 4 * k;
    const int64_t p = (int64_t)e[1] * n_reads + lo;
    if (cell_off[p + 1] > cell_off[p]) { e[2] = cells[2 * cell_off[p]]; e[3] = cells[2 * cell_off[p] + 1]; }
}

size_t assemble_tmp_bytes(uint32_t n_cells)
{
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (const uint64_t *)nullptr, (uint64_t *)nullptr, (const uint32_t *)nullptr,
                                    (uint32_t *)nullptr, (int)n_cells);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (const int64_t *)nullptr, (int64_t *)nullptr, (int)n_cells + 1);
    return std::max(a, b);
}

cudaError_t assemble_sort(const BatchDesc *batches, int nb, uint32_t n_cells, int64_t n_refs, int64_t n_reads,
                          const uint32_t *keep, uint64_t *pair_tmp, uint32_t *src_tmp, uint64_t *pair_sorted, uint32_t *order, void *tmp,
                          size_t tmp_bytes, int pair_bits, cudaStream_t st)
{
    if (n_cells == 0) return cudaSuccess;
    const int threads = 256;
    cell_pairs_kernel<<<(n_cells + threads - 1) / threads, threads, 0, st>>>(batches, nb, n_cells, n_refs, n_reads, keep, pair_tmp, src_tmp);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, pair_tmp, pair_sorted, src_tmp, order, (int)n_cells, 0, pair_bits, st);
}

cudaError_t assemble_gather_cells(const BatchDesc *batches, int nb, uint32_t n_cells, const uint32_t *order, int32_t *cells,
                                  int32_t *beginnings, int32_t *op_lens, int64_t *words, int64_t *ops_off, void *tmp,
                                  size_t tmp_bytes, cudaStream_t st)
{
    const int threads = 256;
    if (n_cells) {
        gather_cells_kernel<<<(n_cells + threads - 1) / threads, threads, 0, st>>>(batches, nb, n_cells, order, cells,
                                                                                  beginnings, op_lens, words);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    // words has n_cells + 1 entries (last = 0): exclusive sum gives ops_off[0 .. n_cells]
    return cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, words, ops_off, (int)n_cells + 1, st);
}

cudaError_t assemble_gather_ops(const BatchDesc *batches, int nb, uint32_t n_cells, const uint32_t *order,
                                const int64_t *ops_off, uint32_t *ops_out, cudaStream_t st)
{
    if (n_cells == 0) return cudaSuccess;
    const int threads = 256;
    const int64_t blocks = ((int64_t)n_cells * 8 + threads - 1) / threads;
    gather_ops_kernel<<<(unsigned)blocks, threads, 0, st>>>(batches, nb, n_cells, order, ops_off, ops_out);
    return cudaGetLastError();
}

cudaError_t assemble_offsets(const uint64_t *pair_sorted, uint32_t n_cells, int64_t n_pairs, int64_t *cell_off,
                             int32_t *best, int64_t n_reads, const int32_t *cells, cudaStream_t st)
{
    const int threads = 256;
    pair_offsets_kernel<<<(unsigned)((n_pairs + 1 + threads - 1) / threads), threads, 0, st>>>(pair_sorted, n_cells, n_pairs, cell_off);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess || n_reads == 0) return e;
    best_cells_kernel2<<<(unsigned)((n_reads + threads - 1) / threads), threads, 0, st>>>(best, n_reads, cell_off, cells);
    return cudaGetLastError();
}

}  // namespace swb

namespace swb {

cudaError_t assemble_kept_count(const uint64_t *pair_sorted, uint32_t n_cells, int64_t n_pairs, uint32_t *n_kept, cudaStream_t st)
{
    kept_count_kernel<<<1, 1, 0, st>>>(pair_sorted, n_cells, n_pairs, n_kept);
    return cudaGetLastError();
}

cudaError_t assemble_hit_cells(const BatchDesc *batches, int nb, const uint64_t *pair_sorted, const uint32_t *order, uint32_t n_all,
                               int64_t n_pairs, int64_t n_reads, const int64_t *cell_off, const int32_t *cells, int32_t *best,
                               int32_t *hits, int k, cudaStream_t st)
{
    if (n_reads == 0) return cudaSuccess;
    const int threads = 256;
    hit_cells_kernel<<<(unsigned)((n_reads + threads - 1) / threads), threads, 0, st>>>(batches, nb, pair_sorted, order, n_all, n_pairs,
                                                                                      n_reads, cell_off, cells, best, hits, k);
    return cudaGetLastError();
}

cudaError_t assemble_list_cells(const int64_t *hit_off, int64_t n_reads, int32_t *list, int64_t n_hits, const int64_t *cell_off,
                                const int32_t *cells, cudaStream_t st)
{
    if (n_hits == 0) return cudaSuccess;
    const int threads = 256;
    list_cells_kernel<<<(unsigned)((n_hits + threads - 1) / threads), threads, 0, st>>>(hit_off, n_reads, list, n_hits, cell_off, cells);
    return cudaGetLastError();
}

}  // namespace swb
