"""GPU parity of the LONG rows-per-lane classes of the s16x2 path (K = 40, 48, 56, 64: reads of 257 .. 511 rows;
the reference's own read-length sweep goes to 500 bp, EngineerData.java:87-104).  Same kernels as the 150 bp
path (biased fill, tile locate, tile traceback) at larger K: bit-exact against the oracle at every class
boundary, for homologous / gappy / tie-heavy reads, both tie rules, segments of long references and
half-filled read pairs.  Reads of 512 rows and more still take the int32 wide path."""
import random

import pytest

import oracle
from tests.helpers import check_pairs

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


# (K class, read lengths at its edges): 8 * K rows per class
BOUNDARIES = [(40, (257, 300, 319, 320)), (48, (321, 350, 383, 384)), (56, (385, 420, 447, 448)),
              (64, (449, 480, 500, 510, 511))]


@pytest.mark.parametrize("k_class,lengths", BOUNDARIES)
def test_class_boundaries(engine, k_class, lengths):
    rnd = random.Random(100 + k_class)
    base = _rand(rnd, 2600)
    refs = [_rand(rnd, n) for n in (1, 7, 15, 16, 17, 40, 333, 1200)] + [base]
    reads = []
    for m in lengths:
        reads.append(_rand(rnd, m))                                   # random: short local hits anywhere
        s = rnd.randint(0, len(base) - m - 40)
        reads.append(_mutate(rnd, base[s:s + m + 30])[:m])            # homologous: a path across every lane
    check_pairs(engine, refs, reads)


def test_every_class_in_one_call_with_odd_counts(engine):
    """Reads of all four long classes, the 256-row class and a wide one in one call; odd read counts per class
    leave a read pair half empty."""
    rnd = random.Random(7)
    base = _rand(rnd, 1800)
    refs = [base, _rand(rnd, 900), _rand(rnd, 64), "ACGT" * 120]
    reads = [_mutate(rnd, base[100:100 + m])[:m] for m in (256, 258, 322, 330, 390, 470, 505, 511, 512, 600)]
    reads += [_rand(rnd, 301), ("ACGT" * 130)[:499]]
    check_pairs(engine, refs, reads)


@pytest.mark.parametrize("tie_gt", [False, True])
def test_tie_heavy_long_reads(engine, tie_gt):
    """Low-complexity reads: thousands of maximum cells per pair and direction ties all along the paths, under both
    tie rules (SmithWaterman.java:227-249, DistributedSW.java:310-326)."""
    from sparksmithwaterman_b200 import sw
    rnd = random.Random(17 + int(tie_gt))
    refs = ["AT" * 400, _mutate(rnd, "AC" * 600, sub=0.03, indel=0.0), "A" * 300, _rand(rnd, 700)]
    reads = [("AT" * 200)[:m] for m in (300, 401)] + [_mutate(rnd, "AC" * 230, sub=0.02, indel=0.01)[:450], "A" * 260]
    rs = engine.load_refset(refs)
    res = rs.align(reads, (5, -3, -4), tie_gt=tie_gt).cache()
    for r in range(len(refs)):
        for q in range(len(reads)):
            exp = oracle.align(refs[r], reads[q], 5, -3, -4, tie_gt=tie_gt)
            score, cells, sites = res.pair(r, q)
            if tie_gt:
                cells, sites = sw.distributed_order(cells, sites)
            assert score == exp.score, (r, q)
            assert cells == exp.cells, (r, q, len(cells), len(exp.cells))
            assert sites == exp.sites, (r, q)
    res.free(); rs.free()


@pytest.mark.parametrize("scores", [(2, -1, -2), (1, -1, -1), (3, 1, -2), (10, -9, -10)])
def test_other_score_sets(engine, scores):
    rnd = random.Random(sum(scores) + 50)
    base = _rand(rnd, 1500)
    refs = [base, _rand(rnd, 500), _rand(rnd, 90)]
    reads = [_mutate(rnd, base[50:50 + m], sub=0.1, indel=0.05)[:m] for m in (280, 400, 511)] + [_rand(rnd, 360)]
    check_pairs(engine, refs, reads, scores)


def test_long_reference_in_segments(engine):
    """References of 40 and 20 kbp, both longer than two fill segments.  The call has few items, so the warm-up window
    (W_al, from m + match * m / |gap| + 1) sets the segment length: 2 * W_al = 1,472 columns for the K = 40 read and
    2,336 for the K = 64 reads.  Copies of the reads are planted at multiples of 8,192 columns; the cuts of the other
    regimes are covered in test_gpu_long_refs.py."""
    rnd = random.Random(3)
    ref = list(_rand(rnd, 40000))
    r1, r2 = _rand(rnd, 480), _rand(rnd, 300)
    for pos, r in ((8192 - 240, r1), (16384 - 10, r2), (24576 - 479, r1), (39400, r2)):
        ref[pos:pos + len(r)] = list(_mutate(rnd, r, sub=0.03, indel=0.01))
    ref = "".join(ref[:40000])
    check_pairs(engine, [ref, _rand(rnd, 20000)], [r1, r2, _rand(rnd, 511)])


def test_gappy_paths(engine):
    """Paths that wander off the diagonal cross tiles through their top / left edges at odd places."""
    rnd = random.Random(29)
    base = _rand(rnd, 2000)
    reads = [_mutate(rnd, base[300:300 + 2 * m], sub=0.2, indel=0.25)[:m] for m in (270, 340, 430, 500)]
    check_pairs(engine, [base, base[::-1]], reads)


def test_scores_only_and_resident_reads(engine):
    """SWB_F_SCORES_ONLY (the locate scan makes the subsampled fill's scores exact) and the device-resident reads
    handle (swb_align_resident) with reads of every long class."""
    import numpy as np
    rnd = random.Random(61)
    base = _rand(rnd, 2400)
    refs = [base, _rand(rnd, 1000), "AT" * 300]
    reads = [_mutate(rnd, base[m:2 * m])[:m] for m in (260, 333, 401, 470)] + [_rand(rnd, 511), ("AT" * 200)[:385]]
    rs = engine.load_refset(refs)
    exp = np.array([[oracle.align(r, q, 5, -3, -4, max_cells=1).score for q in reads] for r in refs], dtype=np.int32)
    so = rs.align(reads, scores_only=True)
    assert (so.scores == exp).all()
    up = rs.upload_reads(reads)
    res = up.align()
    assert (res.scores == exp).all()
    assert (res.ref_totals == so.ref_totals).all()
    res.free(); up.free()
    so.free(); rs.free()


LONG_SCORE_SETS = [(5, -3, -4), (1, -1, -1), (2, -2, -2), (3, -3, -1), (2, -1, -3), (7, -5, -2), (10, -2, -7), (3, 1, -2)]


def _fuzz_workload(rnd):
    alphabet = rnd.choice(["ACGT", "ACGT", "AT", "acgtACGT"])

    def seq(n):
        if rnd.random() < 0.15 and n >= 4:                           # tandem repeat
            unit = "".join(rnd.choice(alphabet) for _ in range(rnd.randint(1, 5)))
            return (unit * (n // len(unit) + 1))[:n]
        return "".join(rnd.choice(alphabet) for _ in range(n))

    refs = [seq(rnd.choice([1, 16, 17, 100, 511, 512, 1023, 1500, 2600, 4000])) for _ in range(rnd.randint(1, 5))]
    if rnd.random() < 0.2:
        refs.append(seq(rnd.randint(9000, 22000)))                    # segmented fill
    reads = [seq(rnd.randint(257, 511)) for _ in range(rnd.randint(1, 5))]
    for _ in range(rnd.randint(1, 3)):                                # planted, mutated substrings
        r = rnd.choice(refs)
        if len(r) > 300:
            m = rnd.randint(257, min(511, len(r)))
            a = rnd.randrange(0, len(r) - m + 1)
            reads.append(_mutate(rnd, r[a:a + m], sub=rnd.choice([0.02, 0.1, 0.25]), indel=rnd.choice([0.0, 0.02, 0.2]))[:511])
    if rnd.random() < 0.3:
        reads.append(seq(rnd.choice([150, 256, 600])))                # a neighbour class / the wide path in the same call
    return refs, [q for q in reads if q]


@pytest.mark.parametrize("seed", range(24))
def test_fuzz_long_classes(engine, seed):
    rnd = random.Random(5000 + seed)
    refs, reads = _fuzz_workload(rnd)
    check_pairs(engine, refs, reads, LONG_SCORE_SETS[seed % len(LONG_SCORE_SETS)], max_cells=300)
