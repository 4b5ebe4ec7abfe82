// swb_strands.cu -- the reads of a both-strands call (SWB_F_BOTH_STRANDS, include/swb200.h).
//
// A both-strands call over n reads aligns the 2n internal reads [reads; rc(reads)]: internal read n + q is the
// reverse complement of read q.  Scores and cells of internal read v = s * n + q against reference r sit at pair
// r * 2n + v = (2r + s) * n + q, which is pair (o = 2r + s, q) of the oriented result, so the fill, locate, traceback
// and assembly run unchanged over the internal reads.  The reverse strand is built from the encoded codes, so it also
// serves resident reads, whose raw bytes are gone.
#include "swb_host.h"

namespace swbh {

namespace {

// IUPAC DNA complement of an upper-case symbol; 0 = no complement (the symbol is outside the IUPAC DNA alphabet)
char iupac_complement(int c)
{
    switch (c) {
        case 'A': return 'T'; case 'T': return 'A'; case 'C': return 'G'; case 'G': return 'C';
        case 'R': return 'Y'; case 'Y': return 'R'; case 'K': return 'M'; case 'M': return 'K';
        case 'B': return 'V'; case 'V': return 'B'; case 'D': return 'H'; case 'H': return 'D';
        case 'S': return 'S'; case 'W': return 'W'; case 'N': return 'N';
    }
    return 0;
}

// block per read: rev[off[q] + i] = comp[codes[off[q] + m - 1 - i]], the reverse strand at the forward read's offsets
__global__ void __launch_bounds__(128) rc_reads_kernel(const uint8_t *__restrict__ codes, const int64_t *__restrict__ off,
                                                       int64_t n_reads, const uint8_t *__restrict__ comp, uint8_t *__restrict__ rev)
{
    __shared__ uint8_t tab[256];
    for (int c = threadIdx.x; c < 256; c += blockDim.x) tab[c] = comp[c];
    __syncthreads();
    for (int64_t q = blockIdx.x; q < n_reads; q += gridDim.x) {
        const int64_t a = off[q], b = off[q + 1];
        for (int64_t i = a + threadIdx.x; i < b; i += blockDim.x) rev[i] = tab[codes[a + b - 1 - i]];
    }
}

}  // namespace

char complement_keep_case(char c)
{
    const bool lower = c >= 'a' && c <= 'z';
    const char k = iupac_complement(lower ? c - 32 : c);
    return !k ? c : lower ? (char)(k + 32) : k;
}

// comp_code[c] = code of the complement of the symbol with code c (0xFF: the complement is absent from the set, or
// c is 0xFF); SWB_E_UNSUPPORTED when the set holds a symbol outside the IUPAC DNA alphabet
int strand_complement_codes(const swb_refset *rs, uint8_t comp_code[256])
{
    memset(comp_code, 0xFF, 256);
    for (int c = 0; c < 128; ++c) {
        if (rs->code_of[c] == 0xFF) continue;
        const char k = iupac_complement(c);
        if (!k) {
            char msg[128];
            snprintf(msg, sizeof msg, "swb_align: SWB_F_BOTH_STRANDS needs an IUPAC DNA alphabet; the set holds byte 0x%02X", c);
            return fail(SWB_E_UNSUPPORTED, msg);
        }
        comp_code[rs->code_of[c]] = rs->code_of[(int)k];
    }
    return SWB_OK;
}

// the 2n internal reads of a both-strands call over rd: a per-call copy, rd itself is not changed
int both_strands_reads(swb_ctx *ctx, const swb_refset *rs, const swb_reads *rd, std::unique_ptr<swb_reads> &out)
{
    uint8_t comp_code[256];
    int rc = strand_complement_codes(rs, comp_code);
    if (rc) return rc;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int64_t n = rd->n_reads;
    std::unique_ptr<swb_reads> r2(new swb_reads());
    r2->ctx = ctx; r2->rs = rd->rs; r2->n_reads = 2 * n;
    r2->len.resize((size_t)(2 * n));
    std::vector<int64_t> off((size_t)(2 * n + 1));
    int64_t total = 0;
    for (int64_t v = 0; v < 2 * n; ++v) {
        const int32_t m = rd->len[(size_t)(v < n ? v : v - n)];
        r2->len[(size_t)v] = m;
        off[(size_t)v] = total;
        total += m;
    }
    off[(size_t)(2 * n)] = total;
    const int64_t half = total / 2;
    DevBuf<uint8_t> d_comp;
    CU(d_comp.alloc(256, st));
    CU(r2->codes.alloc((size_t)total + 16, st));
    CU(r2->off.alloc(off.size(), st));
    CU(cudaMemcpyAsync(d_comp.p, comp_code, 256, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(r2->off.p, off.data(), off.size() * 8, cudaMemcpyHostToDevice, st));
    if (half) {
        CU(cudaMemcpyAsync(r2->codes.p, rd->codes.p, (size_t)half, cudaMemcpyDeviceToDevice, st));
        rc_reads_kernel<<<(unsigned)std::min<int64_t>(n, (int64_t)ctx->sm_count * 16), 128, 0, st>>>(rd->codes.p, rd->off.p, n, d_comp.p,
                                                                                                    r2->codes.p + half);
        CU(cudaGetLastError());
    }
    CU(cudaStreamSynchronize(st));                 // the host tables above are locals
    out = std::move(r2);
    return SWB_OK;
}

}  // namespace swbh
