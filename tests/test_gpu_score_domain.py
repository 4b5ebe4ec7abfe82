"""GPU: every score-domain boundary of the kernel selection, on both sides.  Each align call sends a read to one of
about a dozen kernel variants, chosen from the scores, the read length and the longest reference by a handful of host
predicates, each of which protects an int16 or 8-bit representation:

  call domain        check_call (swb_align.cu)         max(|match|, |mismatch|, |gap|) * (max_m + max_len + 2) < 2^30
  s16x2 short path   classify_reads (swb_align.cu)     2-bit set, gap < 0, |score| <= 8000 each,
                                                       smax = max(match, mismatch, 0) * min(m, max_len) <= 16000
  long classes       same place                        257 .. 511 rows: also tile_trace_ok and fill_bias_ok
  biased fill        fill_bias_ok (swb_fill_bias.cu)   0 <= match + |gap|, mismatch + |gap| <= 4000, smax + 32 |gap| <= 30000
  subsampled maxima  fill_sub_slack (swb_fill_bias.cu) match > slack
  byte-tile trace    tile_trace_ok (swb_trace_tile.cu) 2 (smax_s - gap) + max |s| < 250 (short and wide traceback)

A limit that is off by one shows as wrong scores or alignments right at the limit, so each row below is one side of one
boundary: it asserts the kernels the call ran (and the ones it must not run), that the largest score of the call is
the bound max(match, mismatch, 0) * min(m, max_len), and every pair bit-exact against the C oracle."""
import random

import numpy as np
import pytest

import oracle
import sparksmithwaterman_b200 as swb
from sparksmithwaterman_b200 import sw
from sparksmithwaterman_b200._ffi import SwbError
from tests.helpers import launched_kernels, launches, parts_workspace
from tests.test_gpu_all_hits import check_all_hits
from tests.test_gpu_hits import check_hits
from tests.test_score_domain_host import BAND_EDGE_LENGTHS, BIG_IN, BIG_OUT, EDGE_M, EDGE_N, edge_score_sets, wrap32

pytestmark = pytest.mark.gpu

SWB_E_UNSUPPORTED = -3


def _rand(rnd, n, alphabet="ACGT"):
    return "".join(rnd.choice(alphabet) for _ in range(n))


def _mutate(rnd, s, sub=0.05, indel=0.02):
    out = []
    for ch in s:
        u = rnd.random()
        if u < indel / 2:
            continue
        if u < indel:
            out.append(rnd.choice("ACGT"))
        out.append(rnd.choice("ACGT") if rnd.random() < sub else ch)
    return "".join(out)


ANTI = str.maketrans("ACGT", "CGTA")            # every base to another one: a read that mismatches its source everywhere


def _workload(seed, m, ns):
    """References of lengths ns (ns[0] the longest, random; the last a tandem repeat) and reads of exactly m rows: one
    that matches refs[0] exactly over min(m, ns[0]) bases, its mismatch-everywhere twin, a tandem repeat (ties and many
    max cells against the tandem reference), a mutated and a gappy copy, and a random read."""
    assert ns[0] == max(ns)
    rnd = random.Random(seed)
    refs = [_rand(rnd, n) for n in ns[:-1]] + [("AC" * ns[-1])[:ns[-1]]]
    r0 = refs[0]
    if m <= len(r0):
        a = (len(r0) - m) // 2
        exact = r0[a:a + m]
    else:
        lead = (m - len(r0)) // 2
        exact = _rand(rnd, lead) + r0 + _rand(rnd, m - len(r0) - lead)
    anti = exact.translate(ANTI)
    fill = lambda s: (s + _rand(rnd, m))[:m]
    reads = [exact, anti, fill(("AC" * m)[:m - m // 4]), fill(_mutate(rnd, exact)), fill(_mutate(rnd, exact, 0.2, 0.25)),
             _rand(rnd, m)]
    return refs, reads


def _check(res, refs, reads, scores, tie_gt=False, max_cells=None):
    """Every pair of a fetched result against the oracle (score, cell count, cells, beginnings, both strings), the
    wrapping per-reference totals (Distribution.java:424) and the best hit of every read."""
    res.cache()
    sc = res.scores
    for r in range(len(refs)):
        for q in range(len(reads)):
            exp = oracle.align(refs[r], reads[q], *scores, max_cells=max_cells, tie_gt=tie_gt)
            score, cells, sites = res.pair(r, q, max_cells)
            if tie_gt:
                cells, sites = sw.distributed_order(cells, sites)
            assert score == exp.score, (r, q, score, exp.score)
            n_exp = len(refs[r]) * len(reads[q]) if exp.score == 0 else oracle.score(refs[r], reads[q], *scores)[1]
            assert res.pair_cell_count(r, q) == n_exp, (r, q)
            assert cells == exp.cells, (r, q, cells[:3], exp.cells[:3])
            assert sites == exp.sites, (r, q)
    tot = (sc.astype(np.int64).sum(axis=1) & 0xFFFFFFFF).astype(np.uint32).view(np.int32)
    assert (res.ref_totals == tot).all()
    best = res.best_hits
    for q in range(len(reads)):
        col = sc[:, q]
        assert best[q, 0] == col.max() and best[q, 1] == int(np.argmax(col)), q


def _run(eng, refs, reads, scores, tie_gt=False):
    rs = eng.load_refset(refs)
    res, kernels = launched_kernels(lambda: rs.align(reads, scores, tie_gt=tie_gt))
    return rs, res, kernels


WIDE = r"\bwide_fill_kernel<"
SHORT_FILL = r"\b(fill|fill_bias)_kernel<"
BIAS = r"\bfill_bias_kernel<"
TILE = r"\btile_trace_kernel<"


def _wide(kl, nc, byte_tiles):
    return [rf"\bwide_fill_kernel<{kl}, {nc}>", rf"\bwide_trace_kernel<{kl}, \d+, \d+, {'true' if byte_tiles else 'false'}>"]


# (id, scores, read rows m, reference lengths, kernels that must run, kernels that must not run, run both tie rules).
# {tie} in a pattern is the tie rule of the call: tile_trace_kernel<K, true> is the strict-'>' code.
ROWS = [
    # smax = 64 * 250 = 16000, the s16 ceiling; mismatch + |gap| < 0: the plain fill; 2 * 65 + 64 = 194: byte tiles
    ("s16-short-in", (64, -64, -1), 250, (250, 100, 250), [r"\bfill_kernel<32>", r"\btile_trace_kernel<32, {tie}>"], [WIDE], True),
    ("s16-short-out", (64, -64, -1), 251, (251, 100, 251), _wide(8, 4, True), [SHORT_FILL], False),
    # 257 .. 511 rows: smax = 32 * 500 = 16000, biased (16000 + 32 <= 30000), slack 1 < 32: subsampled maxima, K = 64
    ("s16-long-in", (32, -1, -1), 500, (500, 300, 500), [r"\bfill_bias_kernel<64, true>", r"\btile_trace_kernel<64, {tie}>"], [WIDE], False),
    ("s16-long-out", (32, -1, -1), 501, (501, 300, 501), _wide(16, 4, True), [SHORT_FILL], False),
    # smax takes min(m, max_len): a 500-row read against references of at most 250 bases scores at most 64 * 250
    ("min-len-in", (64, -1, -1), 500, (250, 120, 250), [r"\bfill_bias_kernel<64, true>", r"\btile_trace_kernel<64, {tie}>"], [WIDE], False),
    ("min-len-out", (64, -1, -1), 500, (251, 120, 250), _wide(16, 4, True), [SHORT_FILL], False),
    # |score| <= 8000 each: smax = 8000 * 2 = 16000; no biased fill, no byte tiles: the group traceback
    ("score8000-in", (8000, -8000, -8000), 2, (40, 2, 40), [r"\bfill_kernel<4>", r"\btrace_kernel<4>"], [WIDE, BIAS, TILE], False),
    ("match8001-out", (8001, -1, -1), 1, (40, 1, 40), _wide(8, 4, False), [SHORT_FILL], False),
    ("mismatch8001-out", (8000, -8001, -8000), 2, (40, 2, 40), _wide(8, 4, False), [SHORT_FILL], False),
    ("gap8001-out", (8000, -1, -8001), 2, (40, 2, 40), _wide(8, 4, False), [SHORT_FILL], False),
    # biased fill: smax + 32 |gap| = 56 * 250 + 32 * 500 = 30000; slack 500 >= match: exact tile maxima
    ("bias30000-in", (56, -56, -500), 250, (250, 90, 250), [r"\bfill_bias_kernel<32, false>", r"\btrace_kernel<32>"], [WIDE], False),
    ("bias30000-out", (57, -56, -500), 250, (250, 90, 250), [r"\bfill_kernel<32>", r"\btrace_kernel<32>"], [WIDE, BIAS], False),
    # match + |gap| <= 4000 (slack 1: subsampled maxima); the outside row still reaches smax = 16000 on the plain fill
    ("bias-match4000-in", (3999, -1, -1), 4, (50, 4, 50), [r"\bfill_bias_kernel<4, true>", r"\btrace_kernel<4>"], [WIDE], False),
    ("bias-match4000-out", (4000, -1, -1), 4, (50, 4, 50), [r"\bfill_kernel<4>", r"\btrace_kernel<4>"], [WIDE, BIAS], False),
    # mismatch + |gap| <= 4000 with a positive mismatch: the mismatch-everywhere read reaches 3999 * 4; slack 1 = match
    ("bias-mismatch4000-in", (1, 3999, -1), 4, (50, 4, 50), [r"\bfill_bias_kernel<4, false>", r"\btrace_kernel<4>"], [WIDE], False),
    ("bias-mismatch4000-out", (1, 4000, -1), 4, (50, 4, 50), [r"\bfill_kernel<4>", r"\btrace_kernel<4>"], [WIDE, BIAS], False),
    # mismatch + |gap| >= 0
    ("bias-mismatch0-in", (5, -4, -4), 150, (300, 150, 300), [r"\bfill_bias_kernel<19, true>", r"\btile_trace_kernel<19, {tie}>"], [WIDE], False),
    ("bias-mismatch0-out", (5, -5, -4), 150, (300, 150, 300), [r"\bfill_kernel<19>", r"\btile_trace_kernel<19, {tie}>"], [WIDE, BIAS], False),
    # subsampled tile maxima while match > slack = max(|gap|, min(|mismatch|, 2 |gap|)): 5 > 4, then 4 = 4 (K = 40)
    ("slack-in", (5, -4, -4), 300, (600, 300, 600), [r"\bfill_bias_kernel<40, true>", r"\btile_trace_kernel<40, {tie}>"], [WIDE], False),
    ("slack-out", (4, -3, -4), 300, (600, 300, 600), [r"\bfill_bias_kernel<40, false>", r"\btile_trace_kernel<40, {tie}>"], [WIDE], False),
    # byte tiles of the short traceback: 2 (40 + 1) + 167 = 249, then 250
    ("bytes-short-in", (40, -167, -1), 150, (300, 150, 300), [r"\bfill_kernel<19>", r"\btile_trace_kernel<19, {tie}>"], [WIDE], True),
    ("bytes-short-out", (40, -168, -1), 150, (300, 150, 300), [r"\bfill_kernel<19>", r"\btrace_kernel<19>"], [WIDE, TILE], True),
    # long classes need byte tiles: 2 (40 + 64) + 41 = 249 stays at K = 40, 250 takes the wide path
    ("bytes-long-in", (40, -41, -64), 300, (600, 300, 600), [r"\bfill_bias_kernel<40, false>", r"\btile_trace_kernel<40, {tie}>"], [WIDE], True),
    ("bytes-long-out", (40, -42, -64), 300, (600, 300, 600), _wide(16, 4, False), [SHORT_FILL], False),
    # byte tiles of the wide traceback (400 rows, mismatch + |gap| < 0: no biased fill, so no long class)
    ("bytes-wide-in", (40, -167, -1), 400, (800, 400, 800), _wide(16, 4, True), [SHORT_FILL], True),
    ("bytes-wide-out", (40, -168, -1), 400, (800, 400, 800), _wide(16, 4, False), [SHORT_FILL], False),
]

CASES = [pytest.param(row, False, id=row[0]) for row in ROWS] + \
        [pytest.param(row, True, id=row[0] + "-tie-gt") for row in ROWS if row[6]]


@pytest.mark.parametrize("row, tie_gt", CASES)
def test_selection_boundary(engine, row, tie_gt):
    name, scores, m, ns, expect, absent, _ = row
    refs, reads = _workload(sum(map(ord, name)), m, ns)
    rs, res, kernels = _run(engine, refs, reads, scores, tie_gt)
    tie = "true" if tie_gt else "false"
    for pattern in expect:
        assert launches(kernels, pattern.format(tie=tie)), (pattern, sorted({k for k, _ in kernels}))
    for pattern in absent:
        assert not launches(kernels, pattern), pattern
    bound = max(scores[0], scores[1], 0) * min(m, max(ns))
    assert int(res.scores.max()) == bound
    _check(res, refs, reads, scores, tie_gt, max_cells=None if tie_gt else 300)
    res.free(); rs.free()


# ---- the int32 edge of the call domain --------------------------------------------------------------------------

def _edge_workload():
    rnd = random.Random(2024)
    refs = [_rand(rnd, EDGE_N), ("ACG" * EDGE_N)[:700], _rand(rnd, 300)]
    src = refs[0][200:200 + EDGE_M]
    reads = [src, src.translate(ANTI), (_mutate(rnd, src) + _rand(rnd, EDGE_M))[:EDGE_M], ("ACG" * 200)[:EDGE_M - 1],
             _rand(rnd, EDGE_M), refs[2][100:250]]
    return refs, reads


@pytest.mark.parametrize("scores", edge_score_sets(BIG_IN), ids=["match", "gap", "mismatch"])
def test_largest_scores_inside_the_call_domain(engine, scores):
    """big * (600 + 1000 + 2) < 2^30 for the largest big: the int32 wide path at scores of about 4 * 10^8, and hits /
    all-hits mode on top of it (the lists the numpy rules of the plain scores)."""
    refs, reads = _edge_workload()
    rs, res, kernels = _run(engine, refs, reads, scores)
    assert launches(kernels, WIDE) and not launches(kernels, SHORT_FILL)
    assert int(res.scores.max()) == max(scores[0], scores[1], 0) * EDGE_M
    _check(res, refs, reads, scores, max_cells=100)
    res.free(); rs.free()
    check_hits(engine, refs, reads, scores, k=2)
    for margin in (0, 2**31 - 1):
        check_all_hits(engine, refs, reads, scores, margin=margin)


@pytest.mark.parametrize("scores", edge_score_sets(BIG_OUT), ids=["match", "gap", "mismatch"])
def test_smallest_scores_outside_the_call_domain(engine, scores):
    """big * (600 + 1000 + 2) >= 2^30: every entry point refuses the call with SWB_E_UNSUPPORTED; the pair queue goes
    on serving valid requests afterwards."""
    refs, reads = _edge_workload()
    rs = engine.load_refset(refs)
    up = rs.upload_reads(reads)
    calls = {"plain": lambda: rs.align(reads, scores), "resident": lambda: up.align(scores),
             "hits": lambda: rs.align(reads, scores, top_k=2), "all-hits": lambda: rs.align(reads, scores, margin=0),
             "resident-hits": lambda: up.align(scores, top_k=2), "resident-all-hits": lambda: up.align(scores, margin=0),
             "pair": lambda: engine.align_pair(refs[0], reads[0], scores)}
    for name, call in calls.items():
        with pytest.raises(SwbError) as e:
            call()
        assert e.value.code == SWB_E_UNSUPPORTED, name
    up.free(); rs.free()
    inside = tuple(max(-BIG_IN, min(BIG_IN, s)) for s in scores)
    for sc in (inside, (5, -3, -4)):
        res = engine.align_pair(refs[0], reads[0], sc).cache()
        exp = oracle.align(refs[0], reads[0], *sc)
        assert res.pair(0, 0) == (exp.score, exp.cells, exp.sites), sc
        res.free()


# ---- totals that wrap ---------------------------------------------------------------------------------------------

def test_wide_totals_wrap(engine):
    """Four reads of about 7 * 10^8 each (a positive gap: the all-gap path to (m, n)) against one reference: the
    reference's total passes 2^31 and wraps like Java's int."""
    rnd = random.Random(77)
    g = 437_500                                                      # 437,500 * 1,602 < 2^30
    scores = (1, -1, g)
    refs = [_rand(rnd, EDGE_N)]
    reads = [_rand(rnd, m) for m in (EDGE_M, EDGE_M - 1, EDGE_M - 2, EDGE_M - 3)]
    rs, res, kernels = _run(engine, refs, reads, scores)
    assert launches(kernels, r"\bwide_fill_kernel<32, 0>")
    exp = [g * (EDGE_N + m - 1) for m in map(len, reads)]
    assert res.scores[0].tolist() == exp
    assert sum(exp) > 2**31 and res.ref_totals[0] == wrap32(sum(exp))
    assert res.best_hits.tolist() == [[s, 0, len(q), EDGE_N] for s, q in zip(exp, reads)]
    _check(res, refs, reads, scores)
    res.free(); rs.free()


def test_s16_totals_wrap(engine):
    """134,218 copies of one 250-row read against itself with (64, -64, -1): 16000 each on the s16 path, a total of
    16000 * 134218 > 2^31.  One oracle call stands for every copy."""
    n = 134_218
    assert 16000 * n > 2**31
    rnd = random.Random(5)
    ref = _rand(rnd, 250)
    scores = (64, -64, -1)
    rs, res, kernels = _run(engine, [ref], [ref] * n, scores)
    assert launches(kernels, r"\bfill_kernel<32>") and launches(kernels, r"\btile_trace_kernel<32, false>")
    assert not launches(kernels, WIDE)
    exp = oracle.align(ref, ref, *scores)
    assert exp.score == 16000 and exp.cells == [(250, 250)]
    assert (res.scores == 16000).all()
    assert res.ref_totals.tolist() == [wrap32(16000 * n)]
    assert (res.best_hits == np.array([16000, 0, 250, 250], np.int32)).all()
    assert res.total_cells == n and (np.diff(res.cell_offsets) == 1).all()
    assert (res.cells == np.array(exp.cells[0], np.int32)).all()
    assert (res.beginnings == exp.sites[0][0]).all() and (res.op_lens == len(exp.sites[0][1])).all()
    res.cache()
    for q in (0, 1, n // 2, n - 1):
        assert res.pair(0, q) == (exp.score, exp.cells, exp.sites), q
    res.free(); rs.free()


# ---- the wide path with gap >= 0 or a positive mismatch, over several bands ----------------------------------------

@pytest.mark.parametrize("scores", [(5, -3, 0), (1, 0, 0), (1, -1, 1), (2, 200, -1)])
def test_wide_multi_band_non_negative_gap_and_positive_mismatch(engine, scores):
    """Rows beyond a read's end in its last band may exceed the real maximum when gap >= 0 (swb_wide.cu): reads that
    end one row into a band, one row short of a band edge and on it."""
    rnd = random.Random(sum(scores))
    base = _rand(rnd, 2600)
    refs = [base[:1200], _rand(rnd, 700), ("ACG" * 400)[:1000], base[1300:2600]]
    reads = []
    for m in BAND_EDGE_LENGTHS:
        s = rnd.randint(0, len(base) - m - 40)
        reads.append((_mutate(rnd, base[s:s + m + 40]) + _rand(rnd, m))[:m])
    reads += [_rand(rnd, 1536), ("ACG" * 700)[:2049]]
    rs, res, kernels = _run(engine, refs, reads, scores)
    nc = 4 if scores[2] < 0 else 0
    for kl in (16, 32):
        assert launches(kernels, rf"\bwide_fill_kernel<{kl}, {nc}>"), kl
    assert not launches(kernels, SHORT_FILL)
    _check(res, refs, reads, scores, max_cells=200)
    res.free(); rs.free()


# ---- a reference set in parts on both sides of a gate -------------------------------------------------------------

def test_parts_on_both_sides_of_the_s16_gate():
    """A set cut into three parts (longest first): [250, 240, 230, 220, 210], [600], [250, 90].  With (64, -1, -1) a
    500-row read scores at most 64 * 250 = 16000 against the first and last parts (the biased s16 fill) and takes the
    wide path against the 600-base reference; the stitched arrays must be those of one set."""
    rnd = random.Random(31)
    refs = [_rand(rnd, n) for n in (250, 240, 230, 220, 210, 600, 250, 90)]
    scores = (64, -1, -1)
    reads = [_rand(rnd, 125) + refs[0] + _rand(rnd, 125), refs[5][50:550], (_mutate(rnd, refs[5][:520]) + _rand(rnd, 500))[:500],
             _rand(rnd, 500), ("AC" * 250)]
    eng = swb.Engine(0, workspace_bytes=parts_workspace(refs, 3))
    try:
        rs, res, kernels = _run(eng, refs, reads, scores)
        assert len(launches(kernels, r"\bfold_best_kernel\b")) == 3
        assert launches(kernels, r"\bfill_bias_kernel<64, true>") and launches(kernels, r"\bwide_fill_kernel<16, 4>")
        assert res.scores[0, 0] == 16000 and res.scores[5, 1] == 32000
        _check(res, refs, reads, scores, max_cells=300)
        res.free(); rs.free()
    finally:
        eng.close()
