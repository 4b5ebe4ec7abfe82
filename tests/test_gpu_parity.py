"""GPU parity tests: CUDA path through the C ABI vs the CPU oracle, bit-exact
(scores, max-cell lists in list order, beginnings, both alignment strings)."""
import random

import pytest

import oracle
from sparksmithwaterman_b200 import synth
from tests.helpers import check_pairs

pytestmark = pytest.mark.gpu

REF = "CCTGGGTCCTGCCTCGCATCTGACCAGGGCAGGTGGCCTCCTCATCACACTGCTGCCTCTGCTGTTGGCCCTGCTCATGA"
READ_80 = "AATTTTAGTCTCTCCCTACCCTTTTGGACAGAGCTTCCTGTCCTCTCATTTCACAGGTTATGCAACAGAGGGTTCTGTGT"
READ_20 = "ACTGACTGACTGACTGACTG"


def test_kat_small(engine):
    kats = [("ACGT", "ACGT"), ("AAAA", "CCCC"), ("ACGTACGT", ""), ("AC", "ACGTT"), ("ATATATAT", "ATAT"),
            ("acgtTTacgt", "ACGT"), ("GATTACA", "GCATGCU"), ("CGTGAATTCAT", "GACTTAC"), ("AAGGAA", "AAA"),
            ("GTTCA", "CTA"), ("CCAAT", "CAT"), ("ATCAA", "TAC"), ("TGGTC", "TGT")]
    for ref, read in kats:
        check_pairs(engine, [ref], [read])


def test_engineer_data_constants(engine):
    refs = [REF * 5, REF, REF * 2]
    reads = [READ_80, READ_20, READ_20 * 2, READ_20 * 5]
    check_pairs(engine, refs, reads)


def test_tie_heavy(engine):
    refs = ["AT" * 400, "A" * 300, "ACG" * 100, "TA" * 37 + "G" + "AT" * 50]
    reads = ["AT" * 75, "TA" * 75, "A" * 50, "A" * 150, "ACG" * 40, "AT" * 30 + "C" + "AT" * 30]
    check_pairs(engine, refs, reads)


def test_random_small_all_lengths(engine):
    rnd = random.Random(7)
    refs = ["".join(rnd.choice("ACGT") for _ in range(n)) for n in (1, 2, 7, 8, 9, 31, 32, 33, 63, 64, 65, 127, 128, 129, 300, 0)]
    reads = ["".join(rnd.choice("ACGT") for _ in range(m)) for m in (1, 2, 3, 8, 9, 31, 32, 33, 63, 64, 65, 100, 104, 105, 127, 128, 129, 150, 152, 153, 200, 255, 256, 0)]
    check_pairs(engine, refs, reads)


def test_mixed_case_and_foreign_symbols(engine):
    refs = ["acgtACGTacgtTTGACA", "ACGTNNNN".replace("N", "A"), "ggggCCCC"]
    reads = ["ACGTacgt", "nnACGTnn", "GGGGcccc", "TTgaca"]
    check_pairs(engine, refs, reads)


@pytest.mark.parametrize("scores", [(5, -3, -4), (1, -1, -1), (2, -2, -2), (3, -3, -1), (2, -1, -3), (1, 0, -1), (7, -5, -2)])
def test_custom_scores(engine, scores):
    rnd = random.Random(11)
    refs = ["".join(rnd.choice("ACGT") for _ in range(rnd.randint(20, 200))) for _ in range(6)]
    reads = ["".join(rnd.choice("ACGT") for _ in range(rnd.randint(5, 120))) for _ in range(7)]
    reads.append(refs[0][10:60])
    check_pairs(engine, refs, reads, scores)


def test_cfg1_shape(engine):
    """BASELINE config 1: one 100 bp read vs 1,000 RefSeq-shaped refs, every pair, every string."""
    refs, reads = synth.workload(1, 100, 1000)
    n = check_pairs(engine, [r.decode() for r in refs], [q.decode() for q in reads])
    assert n == 1000


def test_cfg2_sample(engine):
    """BASELINE config 2 shape at reduced count: 150 bp reads vs RefSeq-shaped refs."""
    refs, reads = synth.workload(24, 150, 60)
    check_pairs(engine, [r.decode() for r in refs], [q.decode() for q in reads])


def test_long_references_are_segmented_exactly(engine):
    """References longer than two fill segments are cut into overlapping windows (swb_align.cu
    make_segments); results must not depend on it: reads planted across segment boundaries,
    a tie-heavy long repeat (max cells in every segment), scores with long gap runs."""
    rnd = random.Random(77)
    base = "".join(rnd.choice("ACGT") for _ in range(9000))
    refs = [base, "AT" * 3000, "".join(rnd.choice("ACGT") for _ in range(2500)), base[:2049], base[100:4300]]
    reads = [base[k - 70:k + 80] for k in (1024, 2048, 3072, 8192 - 40)]            # straddle 1024-column cuts
    reads += [base[950:1010] + base[1030:1100], "AT" * 75, base[2000:2100] + "ACGTACGT" + base[2100:2140]]
    check_pairs(engine, refs, reads)
    check_pairs(engine, refs[:2], reads[:5], (2, -1, -1))                           # wide windows: W = m + 2m


def test_long_gap_runs_leave_the_trace_window(engine):
    """Cheap gaps give alignments with long vertical / horizontal runs: the walk leaves the lanes a
    traceback block keeps (re-anchoring) and crosses many blocks without a diagonal step."""
    rnd = random.Random(91)
    base = "".join(rnd.choice("ACGT") for _ in range(1500))
    ins = "".join(rnd.choice("ACGT") for _ in range(60))
    reads = [base[100:170] + ins + base[170:240],                    # 60-row insertion run
             base[400:460] + base[560:640],                          # 100-column deletion run
             base[700:730] + ins[:45] + base[730:760] + ins[10:50] + base[760:800],
             ("ACGT" * 60)[:230], "A" * 40 + base[900:1000] + "T" * 60]
    refs = [base, base[50:900], "ACGT" * 300, base[::-1]]
    for scores in ((5, -4, -1), (4, -6, -1), (3, -2, -1), (10, -9, -1)):
        check_pairs(engine, refs, reads, scores, max_cells=200)


def test_large_scores_fall_back_to_the_group_traceback(engine):
    """Byte tiles need every candidate within 250 of H (tile_trace_ok); larger score sets take the
    group-based traceback kernel (swb_trace.cu), which keeps full s16 tiles."""
    rnd = random.Random(92)
    base = "".join(rnd.choice("ACGT") for _ in range(900))
    refs = [base, base[200:700], "ACGT" * 100, "".join(rnd.choice("ACGT") for _ in range(333))]
    reads = [base[50:200], base[300:380] + "TT" + base[380:440], "ACGT" * 30, base[600:700][::-1], "A" * 20]
    for scores in ((100, -90, -30), (60, -50, -40), (90, 10, -80)):
        check_pairs(engine, refs, reads, scores, max_cells=200)


def test_max_cell_at_every_tile_position(engine):
    """The fill's tile maxima are subsampled (even rows x even steps + the tile's last row / step); the locate
    stage must still find the exact score and every maximum cell.  Exact-substring reads put the unique maximum at
    (m, j) for every j mod 16 and row parities / lane-final rows of the K = 4, 8, 13, 19 classes."""
    rnd = random.Random(93)
    base = "".join(rnd.choice("ACGT") for _ in range(420))
    refs = [base, base[3:400]]
    reads = []
    for m in (3, 4, 5, 8, 9, 31, 32, 33, 37, 64, 65, 97, 104, 105, 149, 150, 151, 152):
        for k in range(3):
            j = 160 + ((7 * m + 5 * k) % 19)                   # end column: all residues mod 16 over the set
            reads.append(base[j - m:j])
    for scores in ((5, -3, -4), (10, -2, -7), (3, 1, -2)):     # the three fuzz score sets that take the subsampled fill
        check_pairs(engine, refs, reads, scores, max_cells=50)
