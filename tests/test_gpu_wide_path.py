"""GPU parity of the int32 wide path (swb_wide.cu): long reads / long pairs (bands coupled through
HBM), scores outside the s16x2 domain (gap >= 0, non-negative mismatch, ...), alphabets with
more than four symbols.  Bit-exact vs the oracle."""
import random

import pytest

import oracle
from tests.helpers import check_pairs
from tests.wide_trace_cases import wide_shape

pytestmark = pytest.mark.gpu


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


def test_long_reads_multi_band(engine):
    rnd = random.Random(21)
    refs = [_rand(rnd, n) for n in (1, 31, 32, 33, 64, 65, 300, 1000, 2500)]
    base = refs[-1]
    reads = [_rand(rnd, m) for m in (257, 300, 511, 512, 513, 700)] + [_mutate(rnd, base[200:1100]), base[0:300]]
    check_pairs(engine, refs, reads)


@pytest.mark.parametrize("scores", [(5, -3, 0), (1, 0, 0), (2, 1, -1), (-1, -2, -3), (0, 0, 0), (1, -1, 1),
                                    (9000, -3, -4), (5, -9000, -4)])
def test_scores_outside_short_domain(engine, scores):
    rnd = random.Random(31)
    refs = [_rand(rnd, rnd.randint(5, 60)) for _ in range(4)] + ["ATATATAT", "AAAA"]
    reads = [_rand(rnd, rnd.randint(3, 40)) for _ in range(4)] + ["ATAT", "CCCC", ""]
    check_pairs(engine, refs, reads, scores, max_cells=400)


def test_alphabet_larger_than_four(engine):
    rnd = random.Random(41)
    refs = [_rand(rnd, 200, "ACGTN"), _rand(rnd, 150, "ACGTNRYKM"), "acgtnNNNacgtRYKM", "ACGT-ACGT*ACGT"]
    reads = [_rand(rnd, 40, "ACGTN"), "NNNN", "acgtn", "RYKM", "T-ACGT*A", _rand(rnd, 300, "ACGTNRY")]
    check_pairs(engine, refs, reads)


def test_mixed_short_and_long_reads_in_one_call(engine):
    rnd = random.Random(51)
    refs = [_rand(rnd, rnd.randint(100, 1500)) for _ in range(12)]
    reads = [_rand(rnd, m) for m in (50, 150, 256, 257, 400, 100, 1000)]
    reads.append(_mutate(rnd, refs[3][:600]))
    check_pairs(engine, refs, reads)


def test_long_pair_homologous(engine):
    """cfg3 shape at reduced size: long homologous pair (90 % identity with indels) + a random pair."""
    rnd = random.Random(61)
    a = _rand(rnd, 6000)
    b = _mutate(rnd, a, sub=0.07, indel=0.03)
    c = _rand(rnd, 5000)
    rs = engine.load_refset([a, c])
    res = rs.align([b]).cache()
    for r, ref in enumerate([a, c]):
        exp = oracle.align(ref, b, lowmem=True)
        got = res.pair(r, 0)
        assert got[0] == exp.score and got[1] == exp.cells and got[2] == exp.sites
    res.free(); rs.free()


@pytest.mark.parametrize("tie_gt", [False, True])
@pytest.mark.parametrize("scores", [(5, -3, -4), (2, -1, -2)])
def test_few_long_walks_cluster_traceback(engine, tie_gt, scores):
    """Few max cells with long paths take the pipelined CTA-wide traceback (cluster of CTAs per cell, per-tile exit
    tables, table chain + parallel re-walk): a homologous pair, a gappy one (low score density: the 16 x 8 corridor,
    except for the pair of the '>' rule's seed with (5, -3, -4), which scores just enough for 32 x 4), a low-complexity
    one where directions tie all along the path, under both tie rules (SmithWaterman.java:227-249
    '>=' cascade, DistributedSW.java:310-326 strict '>': there the host layer re-orders the cells diagonal-major and
    stably by beginning, sw.distributed_order)."""
    from sparksmithwaterman_b200 import sw
    rnd = random.Random(71 + int(tie_gt))
    a = _rand(rnd, 3300)
    b = _mutate(rnd, a, sub=0.06, indel=0.03)
    g = _mutate(rnd, a[500:2900], sub=0.25, indel=0.30)                  # gappy: wanders off the diagonal
    lc = _mutate(rnd, "AC" * 1600, sub=0.03, indel=0.0)
    lc_read = _mutate(rnd, lc[200:2400], sub=0.02, indel=0.01)
    refs, reads = [a, lc], [b, g, lc_read]
    rs = engine.load_refset(refs)
    res = rs.align(reads, scores, tie_gt=tie_gt).cache()
    assert res.total_cells <= 100, res.total_cells                       # else another traceback mode would run
    for r in range(len(refs)):
        for q in range(len(reads)):
            exp = oracle.align(refs[r], reads[q], *scores, tie_gt=tie_gt)
            score, cells, sites = res.pair(r, q)
            if tie_gt:
                cells, sites = sw.distributed_order(cells, sites)
            assert score == exp.score, (r, q)
            assert cells == exp.cells, (r, q)
            assert sites == exp.sites, (r, q)
            if (r, q) == (0, 1):                                        # the gappy pair's corridor shape
                wide = not (tie_gt and scores == (5, -3, -4))
                assert all(wide_shape(exp.score, scores[0], i, j) == wide for i, j in exp.cells), exp.cells
    res.free(); rs.free()


@pytest.mark.parametrize("scores", [(2, 200, -1), (-1, 200, -1), (3, 7, -2)])
def test_mismatch_above_match_leaves_the_s16_path(engine, scores):
    """A positive mismatch above the match score makes the maximum about max(match, mismatch) * min(m, n): with
    200-256 bp reads that leaves int16 although every single score is small, so these inputs must take the int32
    wide path (the s16x2 gate bounds the score with max(match, mismatch, 0), swb_align.cu)."""
    rnd = random.Random(81)
    refs = [_rand(rnd, n) for n in (240, 300, 520, 257)]
    reads = [_rand(rnd, m) for m in (200, 230, 256)] + [refs[2][100:350]]
    check_pairs(engine, refs, reads, scores, max_cells=200)
