"""GPU: long references against the oracle.  The short path cuts a reference longer than 2 * SEG columns into fill
segments (make_segments, swb_align.cu): windows of SEG columns, each started W_al columns early from an all-zero
boundary, each owning only the blocks of its own columns.  SEG is 1024 when a class has few (read pair x reference
quad) items and 8192 otherwise, raised to 2 * W_al when the warm-up window is wider.  Every case mirrors that rule
(segments, few_items), asserts the regime it claims before it compares anything, and plants reads whose unique best
cell falls on each of the 16 columns around a cut, with paths that start in the previous segment.

W is a loose bound: the planted paths are much narrower than the warm-up window, so a window a few columns too short
would still give exact cells here.  What these cases pin is the cut itself: the warm-up, the blocks a segment owns,
and the lengths at which a reference is cut, and the column limit of a reference (2^22 - 1 bases, KEY_J_BITS) on
both sides."""
import ctypes as C
import random
from functools import lru_cache

import numpy as np
import pytest
import torch

import oracle
import sparksmithwaterman_b200 as swb
from tests.helpers import (assert_pair_equal, assert_ranges_equal, check_pairs, launched_kernels, launches, oracle_arrays,
                           result_arrays, result_ops, result_range)
from tests.test_gpu_all_hits import check_all_hits
from tests.test_gpu_hits import check_hits
from tests.test_gpu_strands import check_strands

pytestmark = pytest.mark.gpu

GL, CB = 8, 16                                   # lanes per group, columns per block (swb_internal.h)
K_LIST = (4, 5, 7, 8, 10, 13, 16, 19, 25, 32, 40, 48, 56, 64)
N_MAX = (1 << 22) - 1                            # KEY_J_BITS = 22: the longest reference a set takes
SWB_E_UNSUPPORTED = -3


# ---- the rule, mirrored ----------------------------------------------------------------------------------------------

def _up16(x):
    return (x + 15) // 16 * 16


def pick_k(m):
    """pick_k (swb_align.cu): the rows-per-lane class of a short read of m rows."""
    return next(k for k in K_LIST if GL * k >= m)


def segments(n, K, scores, few):
    """make_segments (swb_align.cu) for one reference of n bases and class K: (SEG, W_al, cuts), cuts the first
    columns (0-based) of every segment after the first.  W = m + max(match, mismatch, 0) * m / |gap| + 1 over the
    class's m = 8 K rows, W_al = W + 8 rounded up to 16; a reference of up to 2 * SEG bases is not cut."""
    match, mismatch, gap = scores
    m = GL * K
    W = m + max(match, mismatch, 0) * m // -gap + 1
    W_al = _up16(W + 8)
    seg = max(1024 if few else 8192, _up16(2 * W_al))
    return seg, W_al, ([] if n <= 2 * seg else list(range(seg, n, seg)))


def few_items(n_reads_in_class, n_refs, sm):
    """run_class (swb_align.cu): a class has few items below 24 per SM, an item being a read pair x a reference quad."""
    return (n_reads_in_class + 1) // 2 * ((n_refs + 3) // 4) < 24 * sm


def fill_bias_ok(match, mismatch, gap, smax):
    """fill_bias_ok (swb_fill_bias.cu): the biased fill for a batch whose best score is at most smax."""
    ag = -gap
    return gap < 0 and 0 <= match + ag <= 4000 and 0 <= mismatch + ag <= 4000 and smax + 32 * ag <= 30000


def tile_trace_ok(match, mismatch, gap):
    """tile_trace_ok (swb_trace_tile.cu): the byte-tile traceback, the only one of the long classes."""
    return gap < 0 and 2 * (max(match, mismatch, 0) - gap) + max(abs(match), abs(mismatch)) < 250


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _fillers_for_many(n_class_reads, n_refs, sm):
    """How many short filler references take a class of n_class_reads reads past 24 * sm items (one quad to spare)."""
    quads = -(-24 * sm // ((n_class_reads + 1) // 2)) + 1
    return max(0, 4 * quads - n_refs)


# ---- inputs ----------------------------------------------------------------------------------------------------------

def _rand(rnd, n):
    return "".join(rnd.choice("ACGT") for _ in range(n))


def _plant(rnd, ref, j, m):
    """Writes the source of a new read of m rows into `ref` (a list) so that it ends at 1-based column j and returns
    the read: the source less one base in its middle, with two substitutions.  Its unique best cell is (m, j) and
    its path, with one gap, starts m + 1 columns earlier."""
    src = _rand(rnd, m + 1)
    ref[j - m - 1:j] = src
    read = list(src[:m // 2] + src[m // 2 + 1:])
    for p in (m // 3, 2 * m // 3):
        read[p] = "ACGT"[("ACGT".index(read[p]) + 1) % 4]
    return "".join(read)


UNIT = "ACGTTGCAAG"                              # period 10: a read of it aligns every 10 columns along a repeat


def _repeat_across(ref, lo, m):
    """A tandem repeat over columns lo - (m + 150) .. lo + m + 150 and a read of m rows of it: the read's max cells
    sit every 10 columns on row m, on both sides of column lo."""
    hw = m + 150
    ref[lo - hw:lo + hw] = (UNIT * (2 * hw // len(UNIT) + 1))[:2 * hw]
    return (UNIT * (m // len(UNIT) + 1))[:m]


def _lengths(seg, k=17):
    """2 SEG (not cut), 2 SEG + 1 (three segments, the last owning one column), 3 SEG, and k SEG + 1 (k - 1 cuts
    of full segments, then a one-column segment)."""
    return [2 * seg, 2 * seg + 1, 3 * seg, k * seg + 1]


def _regime_set(seed, m, seg, many, sm):
    """The long references of one regime with their planted reads.  Returns refs, reads, `full` -- the (ref, read)
    pairs whose every cell is compared (each read against the reference it was planted in) -- and `plants`
    [(ref, read, j, lo)], lo the cut a plant crosses (None on the uncut reference).  Many items: the reads repeat up
    to 64, and short filler references follow the long ones."""
    rnd = random.Random(seed)
    ns = _lengths(seg)
    refs = [list(_rand(rnd, n)) for n in ns]
    reads, plants = [], []

    def plant(r, j, lo):
        plants.append((r, len(reads), j, lo))
        reads.append(_plant(rnd, refs[r], j, m))
    plant(0, seg, None)                                             # where a cut at 2 SEG would be, and the last column
    plant(0, 2 * seg, None)
    plant(1, seg + 1, seg)
    plant(1, 2 * seg + 1, 2 * seg)                                  # the one-column last segment
    plant(2, 2 * seg - 3, 2 * seg)
    plant(2, 3 * seg, 2 * seg)
    for d in range(16):                                             # lo - 7 .. lo + 8, one at each cut of the longest
        lo = (d + 1) * seg
        plant(3, lo + d - 7, lo)
    plant(3, ns[3], 17 * seg)
    q_rep = len(reads)
    reads.append(_repeat_across(refs[2], seg, m))
    reads.append(_rand(rnd, m))
    refs = ["".join(r) for r in refs]
    full = [(r, q) for r, q, _, _ in plants] + [(2, q_rep), (2, q_rep + 1)]
    if many:
        base = list(reads)
        reads = (base * (64 // len(base) + 1))[:64]
        full = [(r, q) for q in range(64) for (r, q0) in full if base[q0] == reads[q]]
        refs += [_rand(rnd, 40) for _ in range(_fillers_for_many(len(reads), len(refs), sm))]
    return refs, reads, full, plants, q_rep


def _check_call(eng, refs, reads, scores, full, tie_gt=False, memo=None):
    """One plain call against the oracle: every max cell of each pair in `full` (assert_pair_equal), the score and the
    max-cell count of every other pair (oracle.score), and the wrapping per-reference totals.  Returns the set, the
    fetched result, the kernels the call ran and the oracle's arrays of the `full` pairs by (ref, read string)."""
    rs = eng.load_refset(refs)
    res, kernels = launched_kernels(lambda: rs.align(reads, scores, tie_gt=tie_gt))
    res.cache()
    memo = {} if memo is None else memo
    for r, q in full:
        key = (r, reads[q])
        if key not in memo:
            memo[key] = oracle_arrays(refs[r], reads[q], scores, tie_gt=tie_gt)
        assert_pair_equal(result_arrays(res, r, q), memo[key], tie_gt, where=f"ref={r} read={q}")
    sc = res.scores
    cnt = np.diff(res.cell_offsets).reshape(sc.shape)
    in_full, rest = set(full), {}
    for r in range(len(refs)):
        for q in range(len(reads)):
            if (r, q) in in_full:
                continue
            key = (r, reads[q])
            if key not in rest:
                rest[key] = oracle.score(refs[r], reads[q], *scores)
            s, c = rest[key]
            assert sc[r, q] == s, f"score ref={r} read={q}: {sc[r, q]} != {s}"
            assert cnt[r, q] == (c if s > 0 else 0), f"max cells ref={r} read={q}: {cnt[r, q]} != {c}"
    tot = (sc.astype(np.int64).sum(axis=1) & 0xFFFFFFFF).astype(np.uint32).view(np.int32)
    assert (res.ref_totals == tot).all()
    return rs, res, kernels, memo


# ---- every regime of the cut -------------------------------------------------------------------------------------------

BIAS, FILL, TILE, GROUP = r"\bfill_bias_kernel<{k}, ", r"\bfill_kernel<{k}>", r"\btile_trace_kernel<{k}, {tie}>", r"\btrace_kernel<{k}>"
WIDE = r"\bwide_fill_kernel<"

# (id, read rows, scores, few items, the SEG the mirror must give, fill kernel, traceback kernel)
REGIMES = [
    ("few-1024", 150, (5, -3, -4), True, 1024, BIAS, TILE),
    ("many-8192", 150, (5, -3, -4), False, 8192, BIAS, TILE),
    ("long-class-2wal", 500, (5, -3, -4), True, 2336, BIAS, TILE),                  # K = 64: 2 W_al = 2336 > 1024
    ("wide-warmup-many", 150, (30, -1, -1), False, 9472, BIAS, TILE),               # W = 4713: 2 W_al = 9472 > 8192
    ("unbiased-fill-many", 150, (10, -9, -1), False, 8192, FILL, TILE),
    ("group-trace-few", 150, (60, -30, -40), True, 1024, BIAS, GROUP),
]


def _assert_regime(reads_in_class, n_refs, K, scores, few, seg_want, sm):
    assert few_items(reads_in_class, n_refs, sm) == few, (reads_in_class, n_refs)
    seg, W_al, _ = segments(0, K, scores, few)
    assert seg == seg_want, (seg, W_al)
    return seg, W_al


@pytest.mark.parametrize("regime", REGIMES, ids=[r[0] for r in REGIMES])
def test_cuts_of_each_regime(engine, regime):
    """Every planted cell around the cuts of 2 SEG, 2 SEG + 1, 3 SEG and 17 SEG + 1 bases against the oracle; then the
    read of a tandem repeat across a cut (max cells in two segments) under the strict '>' tie rule too."""
    name, m, scores, few, seg_want, fill, trace = regime
    K, sm = pick_k(m), _sm_count()
    refs, reads, full, plants, q_rep = _regime_set(sum(map(ord, name)), m, seg_want, not few, sm)
    seg, W_al = _assert_regime(len(reads), len(refs), K, scores, few, seg_want, sm)
    for n, n_cuts in zip(_lengths(seg), (0, 2, 2, 17)):
        cuts = segments(n, K, scores, few)[2]
        assert len(cuts) == n_cuts and (not cuts or n - cuts[-1] in (1, seg)), (n, cuts)
    if name == "wide-warmup-many":
        assert 2 * W_al > 8192
    assert fill_bias_ok(*scores, max(scores[0], scores[1], 0) * m) == (fill == BIAS)       # the kernels this set selects
    assert tile_trace_ok(*scores) == (trace == TILE)
    rs, res, kernels, memo = _check_call(engine, refs, reads, scores, full)
    assert launches(kernels, fill.format(k=K)) and launches(kernels, trace.format(k=K, tie="false")), \
        sorted({k for k, _ in kernels})
    assert not launches(kernels, WIDE)
    for r, q, j, lo in plants:                                      # each plant is what it claims to be
        exp = memo[(r, reads[q])]
        assert exp["cells"].tolist() == [[m, j]], (r, q, j, exp["cells"][:3])
        assert lo is None or (j - m - 1 < lo and lo - 7 <= j <= lo + 8) or j == len(refs[r]), (r, j, lo)
    rep = memo[(2, reads[q_rep])]["cells"][:, 1]
    assert rep.min() <= seg < rep.max() and len(rep) > 20
    res.free(); rs.free()

    gt_reads = [reads[q_rep]] * (1 if few else 64)
    _assert_regime(len(gt_reads), len(refs), K, scores, few, seg_want, sm)
    rs, res, kernels, _ = _check_call(engine, refs, gt_reads, scores, [(2, q) for q in range(len(gt_reads))], tie_gt=True)
    assert launches(kernels, trace.format(k=K, tie="true"))
    res.free(); rs.free()


# ---- one pair set in two regimes -----------------------------------------------------------------------------------

def test_same_pairs_in_both_regimes(engine):
    """One reference of 3 * 8192 + 1 bases with K = 19 and K = 64 reads planted around the cuts of every regime they
    meet: alone (both classes few items: segments of 1024 and 2336 columns), then with filler reads and references
    that take the K = 19 class to many items (8192 columns) while the K = 64 class, in the same call, stays at 2336.
    Every score, cell, beginning and op of the pair set is the same in both calls and the oracle's."""
    sm, scores = _sm_count(), (5, -3, -4)
    rnd = random.Random(8192)
    n = 3 * 8192 + 1
    ref = list(_rand(rnd, n))
    reads19 = [_plant(rnd, ref, j, 150) for j in (5 * 1024 + 2, 8192 - 3, 2 * 8192 + 5, n)]
    reads64 = [_plant(rnd, ref, j, 500) for j in (3 * 2336 + 4, 9 * 2336 + 1)]
    ref = "".join(ref)
    pair_reads = reads19 + reads64
    assert [segments(n, 19, scores, True)[0], segments(n, 64, scores, True)[0], segments(n, 19, scores, False)[0]] == \
        [1024, 2336, 8192]
    assert few_items(4, 1, sm) and few_items(2, 1, sm)
    full = [(0, q) for q in range(len(pair_reads))]
    rs_a, res_a, _, memo = _check_call(engine, [ref], pair_reads, scores, full)
    for q, j in enumerate((5 * 1024 + 2, 8192 - 3, 2 * 8192 + 5, n)):
        assert memo[(0, reads19[q])]["cells"].tolist() == [[150, j]]

    fill_reads = [_rand(rnd, 150) for _ in range(60)]
    refs = [ref] + [_rand(rnd, 40) for _ in range(_fillers_for_many(64, 1, sm))]
    reads = reads19 + fill_reads + reads64
    assert not few_items(len(reads19) + len(fill_reads), len(refs), sm) and few_items(len(reads64), len(refs), sm)
    q_of = list(range(4)) + [64, 65]                                  # the pair set's reads in the larger call
    rs_b, res_b, _, _ = _check_call(engine, refs, reads, scores, [(0, q) for q in q_of], memo=memo)
    for qa, qb in enumerate(q_of):
        assert res_a.scores[0, qa] == res_b.scores[0, qb]
        assert_ranges_equal(result_range(res_a, qa), result_range(res_b, qb), (qa, qb))
    res_a.free(); rs_a.free(); res_b.free(); rs_b.free()


# ---- the modes on segmented references ------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", ["hits", "all-hits", "both-strands"])
def test_modes_on_segmented_references(engine, mode):
    """Hits (k = 3), all-hits (margin 0) and both-strands calls on the many-items set of 8192-column segments, each
    against the plain call the way its own tests check it."""
    sm = _sm_count()
    refs, reads, _, _, _ = _regime_set(77, 150, 8192, True, sm)
    _assert_regime(len(reads) * (2 if mode == "both-strands" else 1), len(refs), 19, (5, -3, -4), False, 8192, sm)
    if mode == "hits":
        check_hits(engine, refs, reads, k=3)
    elif mode == "all-hits":
        check_all_hits(engine, refs, reads, margin=0)
    else:
        check_strands(engine, refs, reads)


# ---- the segment cache -----------------------------------------------------------------------------------------------

CACHE_SCORES = [(5, -3, -4), (1, -1, -1), (2, -1, -2), (3, -3, -1), (2, -1, -3), (7, -5, -2), (10, -2, -7), (10, -9, -1),
                (60, -30, -40)]


def test_segment_cache_past_16_entries(engine):
    """A loaded set keeps the segment tables of up to 16 (K, scores, regime) keys and clears them at the 17th
    (seg_tables, swb_align.cu).  After 17 more keys the first call gives the same arrays, equal to the oracle's."""
    sm, rnd = _sm_count(), random.Random(16)
    ref = list(_rand(rnd, 17 * 1024 + 1))
    planted = [_plant(rnd, ref, (d + 1) * 1024 + d - 7, 150) for d in range(16)]
    refs = ["".join(ref)] + [_rand(rnd, 40) for _ in range(_fillers_for_many(64, 1, sm))]
    many = (planted * 4)[:64]
    few = planted[:2]
    keys = [(s, r) for s in CACHE_SCORES for r in ("many", "few")]
    assert len({(19, s, few_items(len(many if r == "many" else few), len(refs), sm)) for s, r in keys}) == len(keys) > 16
    rs = engine.load_refset(refs)

    def arrays(res):
        res.cache()
        return [res.scores, res.cell_offsets, res.cells, res.beginnings, res.op_lens, result_ops(res, 0, res.total_cells)]
    first = rs.align(many, CACHE_SCORES[0])
    want = arrays(first)
    for q in range(16):
        exp = oracle_arrays(refs[0], planted[q])
        assert exp["cells"].tolist() == [[150, (q + 1) * 1024 + q - 7]]
        assert_pair_equal(result_arrays(first, 0, q), exp, where=f"read={q}")
    first.free()
    for s, r in keys[1:]:
        rs.align(many if r == "many" else few, s, scores_only=True).free()
    again = rs.align(many, CACHE_SCORES[0])
    for a, b in zip(arrays(again), want):
        assert a.shape == b.shape and np.array_equal(a, b)
    again.free(); rs.free()


# ---- the column limit --------------------------------------------------------------------------------------------------

@lru_cache(maxsize=1)
def _longest():
    """A random reference of 2^22 - 1 bases and two reads, K = 19 and K = 64, the first one the second one's rows
    -155 .. -6.  Copies of the K = 64 read end at 3 * 2^20 + 3 and on the last column, a copy of the K = 19 read at
    2^21 + 7: max cells at those columns (K = 64) and at 2^21 + 7, 3 * 2^20 - 2 and 5 columns before the last
    (K = 19)."""
    rnd = random.Random(22)
    ref = bytearray(np.frombuffer(b"ACGT", np.uint8)[np.random.default_rng(22).integers(0, 4, N_MAX)].tobytes())
    r64 = _rand(rnd, 449)
    r19 = r64[-155:-5]
    for j in LONGEST_ENDS[1]:
        ref[j - 449:j] = r64.encode()
    ref[LONGEST_ENDS[0][0] - 150:LONGEST_ENDS[0][0]] = r19.encode()
    return bytes(ref), [r19, r64]


LONGEST_ENDS = (((1 << 21) + 7, 3 * (1 << 20) - 2, N_MAX - 5), (3 * (1 << 20) + 3, N_MAX))


def test_reference_length_limit(engine):
    """2^22 - 1 bases load; one base more is refused with SWB_E_UNSUPPORTED and no handle."""
    ref, _ = _longest()
    rs = engine.load_refset([ref])
    assert rs.n == 1 and rs.total_bases == N_MAX
    rs.free()
    longer = ref + b"A"
    off = np.array([0, len(longer)], np.int64)
    h = C.c_void_p()
    rc = engine.lib.swb_refset_load(engine.h, 1, longer, off.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(h))
    assert rc == SWB_E_UNSUPPORTED and not h.value
    with pytest.raises(swb.SwbError) as e:
        engine.load_refset(["ACGT", longer])
    assert e.value.code == SWB_E_UNSUPPORTED


def test_cells_past_2_21_columns(engine):
    """Max cells at j >= 2^21 and in the last 16 columns of the longest reference, for K = 19 and K = 64 (segments of
    1024 and 2336 columns, few items), every cell against the oracle."""
    ref, reads = _longest()
    scores = (5, -3, -4)
    assert [pick_k(len(q)) for q in reads] == [19, 64] and few_items(1, 1, _sm_count())
    assert len(segments(N_MAX, 19, scores, True)[2]) == N_MAX // 1024
    assert segments(N_MAX, 64, scores, True)[0] == 2336
    for q, ends in zip(reads, LONGEST_ENDS):
        assert oracle.score(ref, q, *scores) == (5 * len(q), len(ends))
    assert check_pairs(engine, [ref], reads, scores, lowmem=True) == 2


def test_wide_path_past_2_21_columns(engine):
    """The same K = 19 read on the int32 wide path: a fifth symbol far from the copies takes every read there."""
    ref, reads = _longest()
    ref = b"N" + ref[1:]
    rs = engine.load_refset([ref])
    res, kernels = launched_kernels(lambda: rs.align(reads[:1]))
    assert launches(kernels, WIDE) and not launches(kernels, r"\b(fill|fill_bias)_kernel<")
    res.free(); rs.free()
    assert check_pairs(engine, [ref], reads[:1], lowmem=True) == 1


def test_class_in_several_batches(engine):
    """A workspace that holds one read pair's block records of the longest reference (1312 bytes per 16-column block
    at K = 19): four reads run in two batches and give the arrays of one read in one batch."""
    ref, reads = _longest()
    q = reads[0]
    blocks = (N_MAX + GL - 1 + CB - 1) // CB
    words = ((19 + 1 + 7) // 8 + CB // 8) * 8                      # record_words(19)
    per_rp = blocks * (words * GL * 4 + GL * 4)
    assert few_items(4, 1, _sm_count()) and segments(N_MAX, 19, (5, -3, -4), True)[0] == 1024
    rs = engine.load_refset([ref])
    one = rs.align([q]).cache()
    eng = swb.Engine(0, workspace_bytes=per_rp)
    try:
        rs2 = eng.load_refset([ref])
        res = rs2.align([q] * 4).cache()
        assert res.stats["batches"] == 2
        for k in range(4):
            assert res.scores[0, k] == one.scores[0, 0] == 5 * len(q)
            assert_ranges_equal(result_range(res, k), result_range(one, 0), k)
        res.free(); rs2.free()
    finally:
        eng.close()
    one.free(); rs.free()
