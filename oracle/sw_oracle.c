/*
 * oracle/sw_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE (see sw_oracle.h).
 *
 * Plain-C restatement of the reference's per-pair operator. Each function names
 * the reference lines it follows. All arithmetic is 32-bit signed, as Java int.
 * Parity unpinned by reference-run outputs (no JVM available); pinned by the
 * SURVEY.md section-8c known answers and the independent twin oracle/sw_twin.py.
 */
#include "sw_oracle.h"

#include <stdlib.h>
#include <string.h>

/* alignment-type codes kept in the type matrix; the reference stores the chars
 * alignTypes = {'a','i','d','-'} (Distribution.java:37) -- only identity matters */
enum { T_NONE = 0, T_ALIGN = 1, T_INS = 2, T_DEL = 3 };

/* Character.toUpperCase restricted to ASCII bytes (SmithWaterman.java:311-312) */
static inline int up(int c) { return (c >= 'a' && c <= 'z') ? c - 32 : c; }

typedef struct { int32_t score; uint8_t type; } cell_t;

/* SmithWaterman.java:217-252 -- GetCellScore.call: three ">=" tests in the order
 * deletion (west), insertion (north), alignment (north-west); the last test that
 * passes wins, so ties resolve a over i over d over none.
 * :277-280 InsDelScore = cell + gap; :309-318 AlignmentScore = nw + match|mismatch
 * on case-folded equality. Java int addition wraps; use unsigned adds to mirror. */
static inline cell_t cell_score(int32_t nw, int32_t north, int32_t west,
                                int ref_base, int read_base,
                                int32_t match, int32_t mismatch, int32_t gap)
{
    cell_t c; c.score = 0; c.type = T_NONE;
    int32_t t = (int32_t)((uint32_t)west + (uint32_t)gap);
    if (t >= c.score) { c.score = t; c.type = T_DEL; }
    t = (int32_t)((uint32_t)north + (uint32_t)gap);
    if (t >= c.score) { c.score = t; c.type = T_INS; }
    int32_t s = (up(ref_base) == up(read_base)) ? match : mismatch;
    t = (int32_t)((uint32_t)nw + (uint32_t)s);
    if (t >= c.score) { c.score = t; c.type = T_ALIGN; }
    return c;
}

typedef struct { int32_t *v; int64_t n, cap; } ivec;
static int ivec_push2(ivec *a, int32_t x, int32_t y)
{
    if (a->n + 2 > a->cap) {
        int64_t nc = a->cap ? a->cap * 2 : 64;
        int32_t *nv = (int32_t *)realloc(a->v, (size_t)nc * sizeof(int32_t));
        if (!nv) return -1;
        a->v = nv; a->cap = nc;
    }
    a->v[a->n++] = x; a->v[a->n++] = y;
    return 0;
}

typedef struct { char *v; int64_t n, cap; } cvec;
static int cvec_reserve(cvec *a, int64_t extra)
{
    if (a->n + extra > a->cap) {
        int64_t nc = a->cap ? a->cap : 256;
        while (nc < a->n + extra) nc *= 2;
        char *nv = (char *)realloc(a->v, (size_t)nc);
        if (!nv) return -1;
        a->v = nv; a->cap = nc;
    }
    return 0;
}

void sw_oracle_free(sw_oracle_result *r)
{
    if (!r) return;
    free(r->cells); free(r->beginning); free(r->aln_off); free(r->ref_aln); free(r->read_aln);
    memset(r, 0, sizeof(*r));
}

/* Append one traced alignment; `stack` holds (ref char, read char) pairs pushed
 * end-to-start, emitted start-to-end (SmithWaterman.java:418-427). */
static int emit_alignment(sw_oracle_result *out, cvec *ra, cvec *qa, int64_t k,
                          const char *stack, int64_t depth, int32_t beginning)
{
    if (cvec_reserve(ra, depth + 1) || cvec_reserve(qa, depth + 1)) return -1;
    for (int64_t p = depth - 1; p >= 0; --p) {
        ra->v[ra->n++] = stack[2 * p];
        qa->v[qa->n++] = stack[2 * p + 1];
    }
    out->beginning[k] = beginning;
    out->aln_off[k + 1] = ra->n;
    return 0;
}

/* SmithWaterman.java:62-92 with :129-190 and :354-436, literal matrices. */
int sw_oracle_align(const char *ref, int64_t n, const char *read, int64_t m,
                    int32_t match, int32_t mismatch, int32_t gap,
                    sw_oracle_result *out)
{
    memset(out, 0, sizeof(*out));
    const int64_t W = n + 1;
    /* :68-69 fresh matrices; :142-149 explicit init pass (score 0, type none) */
    int32_t *S = (int32_t *)malloc((size_t)((m + 1) * W) * sizeof(int32_t));
    uint8_t *A = (uint8_t *)malloc((size_t)((m + 1) * W));
    if (!S || !A) { free(S); free(A); return -1; }
    for (int64_t i = 0; i <= m; ++i)
        for (int64_t j = 0; j <= n; ++j) { S[i * W + j] = 0; A[i * W + j] = T_NONE; }

    /* :153-187 row-major fill with max bookkeeping: ">" restarts the list,
     * "==" appends (so a zero matrix lists every cell) */
    ivec cells = {0, 0, 0};
    int32_t max_score = 0;
    for (int64_t i = 1; i <= m; ++i) {
        for (int64_t j = 1; j <= n; ++j) {
            cell_t c = cell_score(S[(i - 1) * W + j - 1], S[(i - 1) * W + j], S[i * W + j - 1],
                                  (unsigned char)ref[j - 1], (unsigned char)read[i - 1],
                                  match, mismatch, gap);
            S[i * W + j] = c.score;
            A[i * W + j] = c.type;
            if (c.score > max_score) {
                cells.n = 0; max_score = c.score;
                if (ivec_push2(&cells, (int32_t)i, (int32_t)j)) goto oom;
            } else if (c.score == max_score) {
                if (ivec_push2(&cells, (int32_t)i, (int32_t)j)) goto oom;
            }
        }
    }

    out->score = max_score;
    out->n_cells = cells.n / 2;
    out->cells = cells.v; cells.v = NULL;
    out->beginning = (int32_t *)calloc((size_t)out->n_cells + 1, sizeof(int32_t));
    out->aln_off = (int64_t *)calloc((size_t)out->n_cells + 1, sizeof(int64_t));
    if (!out->beginning || !out->aln_off) goto oom;

    {
        /* :85-88 one traceback per max cell, in list order; :380-409 walk while the
         * SCORE of the current cell is positive, beginning = last visited column */
        cvec ra = {0, 0, 0}, qa = {0, 0, 0};
        char *stack = (char *)malloc((size_t)(2 * (m + n) + 2));
        if (!stack) goto oom;
        for (int64_t k = 0; k < out->n_cells; ++k) {
            int64_t i = out->cells[2 * k], j = out->cells[2 * k + 1];
            int32_t score = S[i * W + j];
            int32_t beginning = 0;
            int64_t depth = 0;
            while (score > 0) {
                beginning = (int32_t)j;
                uint8_t t = A[i * W + j];
                if (t == T_ALIGN) {
                    stack[2 * depth] = ref[j - 1]; stack[2 * depth + 1] = read[i - 1];
                    --i; --j;
                } else if (t == T_INS) {
                    stack[2 * depth] = '_'; stack[2 * depth + 1] = read[i - 1];
                    --i;
                } else { /* the reference's final else: deletion (also taken for none) */
                    stack[2 * depth] = ref[j - 1]; stack[2 * depth + 1] = '_';
                    --j;
                }
                ++depth;
                score = S[i * W + j];
            }
            if (emit_alignment(out, &ra, &qa, k, stack, depth, beginning)) { free(stack); goto oom; }
        }
        free(stack);
        out->ref_aln = ra.v; out->read_aln = qa.v;
        if (!out->ref_aln) out->ref_aln = (char *)calloc(1, 1);
        if (!out->read_aln) out->read_aln = (char *)calloc(1, 1);
    }
    free(S); free(A);
    return 0;
oom:
    free(S); free(A); free(cells.v);
    sw_oracle_free(out);
    return -1;
}

/* Same semantics, two score rows + a 2-bit-per-cell plane.  Plane codes:
 * 0 = score is zero (the walk stops here), 1/2/3 = a/i/d of a positive cell.
 * That is all SmithWaterman.java:380-409 ever reads: the type of a positive cell,
 * and whether the next cell's score is positive. */
int sw_oracle_align_lowmem(const char *ref, int64_t n, const char *read, int64_t m,
                           int32_t match, int32_t mismatch, int32_t gap,
                           sw_oracle_result *out)
{
    memset(out, 0, sizeof(*out));
    const int64_t W = n + 1;
    const int64_t total = (m + 1) * W;
    uint8_t *plane = (uint8_t *)calloc((size_t)(total / 4 + 1), 1);
    int32_t *prev = (int32_t *)calloc((size_t)W, sizeof(int32_t));
    int32_t *cur = (int32_t *)calloc((size_t)W, sizeof(int32_t));
    ivec cells = {0, 0, 0};
    if (!plane || !prev || !cur) goto oom;

    int32_t max_score = 0;
    for (int64_t i = 1; i <= m; ++i) {
        cur[0] = 0;
        const int rb = (unsigned char)read[i - 1];
        for (int64_t j = 1; j <= n; ++j) {
            cell_t c = cell_score(prev[j - 1], prev[j], cur[j - 1],
                                  (unsigned char)ref[j - 1], rb, match, mismatch, gap);
            cur[j] = c.score;
            if (c.score > 0) {
                int64_t idx = i * W + j;
                plane[idx >> 2] |= (uint8_t)(c.type << ((idx & 3) * 2));
            }
            if (c.score > max_score) {
                cells.n = 0; max_score = c.score;
                if (ivec_push2(&cells, (int32_t)i, (int32_t)j)) goto oom;
            } else if (c.score == max_score) {
                if (ivec_push2(&cells, (int32_t)i, (int32_t)j)) goto oom;
            }
        }
        int32_t *t = prev; prev = cur; cur = t;
    }
    free(prev); free(cur); prev = cur = NULL;

    out->score = max_score;
    out->n_cells = cells.n / 2;
    out->cells = cells.v; cells.v = NULL;
    out->beginning = (int32_t *)calloc((size_t)out->n_cells + 1, sizeof(int32_t));
    out->aln_off = (int64_t *)calloc((size_t)out->n_cells + 1, sizeof(int64_t));
    if (!out->beginning || !out->aln_off) goto oom;
    {
        cvec ra = {0, 0, 0}, qa = {0, 0, 0};
        char *stack = (char *)malloc((size_t)(2 * (m + n) + 2));
        if (!stack) goto oom;
        for (int64_t k = 0; k < out->n_cells; ++k) {
            int64_t i = out->cells[2 * k], j = out->cells[2 * k + 1];
            int32_t beginning = 0;
            int64_t depth = 0;
            for (;;) {
                int64_t idx = i * W + j;
                int code = (plane[idx >> 2] >> ((idx & 3) * 2)) & 3;
                if (code == 0) break;               /* score(i,j) == 0 */
                beginning = (int32_t)j;
                if (code == T_ALIGN) {
                    stack[2 * depth] = ref[j - 1]; stack[2 * depth + 1] = read[i - 1];
                    --i; --j;
                } else if (code == T_INS) {
                    stack[2 * depth] = '_'; stack[2 * depth + 1] = read[i - 1];
                    --i;
                } else {
                    stack[2 * depth] = ref[j - 1]; stack[2 * depth + 1] = '_';
                    --j;
                }
                ++depth;
            }
            if (emit_alignment(out, &ra, &qa, k, stack, depth, beginning)) { free(stack); goto oom; }
        }
        free(stack);
        out->ref_aln = ra.v; out->read_aln = qa.v;
        if (!out->ref_aln) out->ref_aln = (char *)calloc(1, 1);
        if (!out->read_aln) out->read_aln = (char *)calloc(1, 1);
    }
    free(plane);
    return 0;
oom:
    free(plane); free(prev); free(cur); free(cells.v);
    sw_oracle_free(out);
    return -1;
}

/* ---- DistributedSW variant (SURVEY.md 8f row N3) -------------------------------------------------
 * /root/reference/src/sw/DistributedSW.java: same recurrence, but
 *  - GetCellScore (:280-330) tests with strict ">" in the order deletion, insertion, alignment, so on
 *    equal candidates the FIRST one wins (d over i over a) and a zero cell keeps the type "none";
 *  - ScoreMatrix (:143-245) walks anti-diagonals (i + j ascending), each sorted by j (:209, CellResultComp
 *    :907-911), so the max-cell list is diagonal-major;
 *  - GetAlignments (:456-490) stably sorts the alignments by beginning (MatchSiteComp).
 * Output cells/sites are in that final (sorted) order. */
int sw_oracle_align_gt(const char *ref, int64_t n, const char *read, int64_t m,
                       int32_t match, int32_t mismatch, int32_t gap, sw_oracle_result *out)
{
    memset(out, 0, sizeof(*out));
    const int64_t W = n + 1;
    int32_t *S = (int32_t *)calloc((size_t)((m + 1) * W), sizeof(int32_t));
    uint8_t *A = (uint8_t *)calloc((size_t)((m + 1) * W), 1);
    ivec cells = {0, 0, 0};
    if (!S || !A) goto oom;
    int32_t max_score = 0;
    if (m > 0 && n > 0)
        for (int64_t d = 2; d <= m + n; ++d) {
            int64_t jlo = d - m < 1 ? 1 : d - m, jhi = d - 1 > n ? n : d - 1;
            for (int64_t j = jlo; j <= jhi; ++j) {
                const int64_t i = d - j;
                int32_t best = 0; uint8_t type = T_NONE;
                int32_t t = (int32_t)((uint32_t)S[i * W + j - 1] + (uint32_t)gap);
                if (t > best) { best = t; type = T_DEL; }
                t = (int32_t)((uint32_t)S[(i - 1) * W + j] + (uint32_t)gap);
                if (t > best) { best = t; type = T_INS; }
                int32_t sc = (up((unsigned char)ref[j - 1]) == up((unsigned char)read[i - 1])) ? match : mismatch;
                t = (int32_t)((uint32_t)S[(i - 1) * W + j - 1] + (uint32_t)sc);
                if (t > best) { best = t; type = T_ALIGN; }
                S[i * W + j] = best; A[i * W + j] = type;
                if (best > max_score) { cells.n = 0; max_score = best; if (ivec_push2(&cells, (int32_t)i, (int32_t)j)) goto oom; }
                else if (best == max_score) { if (ivec_push2(&cells, (int32_t)i, (int32_t)j)) goto oom; }
            }
        }
    {
        const int64_t nc = cells.n / 2;
        out->score = max_score; out->n_cells = nc;
        out->cells = (int32_t *)calloc((size_t)nc * 2 + 2, sizeof(int32_t));
        out->beginning = (int32_t *)calloc((size_t)nc + 1, sizeof(int32_t));
        out->aln_off = (int64_t *)calloc((size_t)nc + 1, sizeof(int64_t));
        int32_t *beg = (int32_t *)calloc((size_t)nc + 1, sizeof(int32_t));
        int64_t *len = (int64_t *)calloc((size_t)nc + 1, sizeof(int64_t));
        int64_t *order = (int64_t *)calloc((size_t)nc + 1, sizeof(int64_t));
        char **ra = (char **)calloc((size_t)nc + 1, sizeof(char *)), **qa = (char **)calloc((size_t)nc + 1, sizeof(char *));
        char *stack = (char *)malloc((size_t)(2 * (m + n) + 2));
        if (!out->cells || !out->beginning || !out->aln_off || !beg || !len || !order || !ra || !qa || !stack) goto oom;
        for (int64_t k = 0; k < nc; ++k) {
            int64_t i = cells.v[2 * k], j = cells.v[2 * k + 1];
            int32_t score = S[i * W + j]; int64_t depth = 0;
            while (score > 0) {
                beg[k] = (int32_t)j;
                const uint8_t t = A[i * W + j];
                if (t == T_ALIGN) { stack[2 * depth] = ref[j - 1]; stack[2 * depth + 1] = read[i - 1]; --i; --j; }
                else if (t == T_INS) { stack[2 * depth] = '_'; stack[2 * depth + 1] = read[i - 1]; --i; }
                else { stack[2 * depth] = ref[j - 1]; stack[2 * depth + 1] = '_'; --j; }
                ++depth; score = S[i * W + j];
            }
            len[k] = depth;
            ra[k] = (char *)malloc((size_t)depth + 1); qa[k] = (char *)malloc((size_t)depth + 1);
            for (int64_t p = 0; p < depth; ++p) { ra[k][p] = stack[2 * (depth - 1 - p)]; qa[k][p] = stack[2 * (depth - 1 - p) + 1]; }
            order[k] = k;
        }
        /* stable sort by beginning: a bottom-up merge sort, O(n log n) also when a list of ~10^5 cells arrives with
           its beginnings far from sorted (a tandem repeat lists its max cells diagonal by diagonal) */
        {
            int64_t *tmp = (int64_t *)malloc(((size_t)nc + 1) * sizeof(int64_t));
            if (!tmp) goto oom;
            int64_t *src = order, *dst = tmp;
            for (int64_t w = 1; w < nc; w *= 2) {
                for (int64_t lo = 0; lo < nc; lo += 2 * w) {
                    const int64_t mid = lo + w < nc ? lo + w : nc, hi = lo + 2 * w < nc ? lo + 2 * w : nc;
                    int64_t a = lo, b = mid, k = lo;
                    while (a < mid && b < hi) dst[k++] = beg[src[b]] < beg[src[a]] ? src[b++] : src[a++];
                    while (a < mid) dst[k++] = src[a++];
                    while (b < hi) dst[k++] = src[b++];
                }
                int64_t *t = src; src = dst; dst = t;
            }
            if (src != order) memcpy(order, src, (size_t)nc * sizeof(int64_t));
            free(tmp);
        }
        int64_t total = 0;
        for (int64_t k = 0; k < nc; ++k) total += len[k];
        out->ref_aln = (char *)calloc((size_t)total + 1, 1); out->read_aln = (char *)calloc((size_t)total + 1, 1);
        int64_t pos = 0;
        for (int64_t k = 0; k < nc; ++k) {
            const int64_t x = order[k];
            out->cells[2 * k] = cells.v[2 * x]; out->cells[2 * k + 1] = cells.v[2 * x + 1];
            out->beginning[k] = beg[x];
            memcpy(out->ref_aln + pos, ra[x], (size_t)len[x]); memcpy(out->read_aln + pos, qa[x], (size_t)len[x]);
            pos += len[x]; out->aln_off[k + 1] = pos;
        }
        for (int64_t k = 0; k < nc; ++k) { free(ra[k]); free(qa[k]); }
        free(ra); free(qa); free(stack); free(beg); free(len); free(order);
    }
    free(S); free(A); free(cells.v);
    return 0;
oom:
    free(S); free(A); free(cells.v);
    sw_oracle_free(out);
    return -1;
}

int sw_oracle_score(const char *ref, int64_t n, const char *read, int64_t m,
                    int32_t match, int32_t mismatch, int32_t gap,
                    int32_t *score, int64_t *n_cells)
{
    int32_t *prev = (int32_t *)calloc((size_t)(n + 1), sizeof(int32_t));
    int32_t *cur = (int32_t *)calloc((size_t)(n + 1), sizeof(int32_t));
    if (!prev || !cur) { free(prev); free(cur); return -1; }
    int32_t max_score = 0; int64_t cnt = 0;
    for (int64_t i = 1; i <= m; ++i) {
        cur[0] = 0;
        const int rb = (unsigned char)read[i - 1];
        for (int64_t j = 1; j <= n; ++j) {
            cell_t c = cell_score(prev[j - 1], prev[j], cur[j - 1],
                                  (unsigned char)ref[j - 1], rb, match, mismatch, gap);
            cur[j] = c.score;
            if (c.score > max_score) { max_score = c.score; cnt = 1; }
            else if (c.score == max_score) ++cnt;
        }
        int32_t *t = prev; prev = cur; cur = t;
    }
    free(prev); free(cur);
    *score = max_score; if (n_cells) *n_cells = cnt;
    return 0;
}

static inline uint64_t fnv(uint64_t h, const void *p, size_t len)
{
    const unsigned char *b = (const unsigned char *)p;
    for (size_t k = 0; k < len; ++k) { h ^= b[k]; h *= 0x100000001b3ULL; }
    return h;
}

uint64_t sw_oracle_digest(const sw_oracle_result *r)
{
    uint64_t h = 0xcbf29ce484222325ULL;
    h = fnv(h, &r->score, 4);
    h = fnv(h, &r->n_cells, 8);
    for (int64_t k = 0; k < r->n_cells; ++k) {
        h = fnv(h, &r->cells[2 * k], 8);
        h = fnv(h, &r->beginning[k], 4);
        int64_t len = r->aln_off[k + 1] - r->aln_off[k];
        h = fnv(h, &len, 8);
        h = fnv(h, r->ref_aln + r->aln_off[k], (size_t)len);
        h = fnv(h, r->read_aln + r->aln_off[k], (size_t)len);
    }
    return h;
}
