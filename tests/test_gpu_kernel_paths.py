"""GPU: the fill and traceback kernels the selection rules choose between, reached the way a caller reaches them --
through the score set, the alphabet, the read length, the number of max cells or the workspace size -- in one process.  Each case checks
every pair against the oracle and asserts, from a profile of the same call, that the kernel it covers ran, so that a
change to a selection rule cannot silently drop the coverage."""
import random

import numpy as np
import pytest
import torch

import sparksmithwaterman_b200 as swb
from tests.helpers import check_pairs, launched_kernels, launches, parts_workspace

pytestmark = pytest.mark.gpu

rnd = random.Random(77)
BASE = "".join(rnd.choice("ACGT") for _ in range(2600))
REFS = [BASE, BASE[300:1500], "".join(rnd.choice("ACGT") for _ in range(900)), "AT" * 220, BASE[::-1][:1300], "ACG" * 150]
READS = [BASE[100:250], BASE[700:760] + "GG" + BASE[760:840], BASE[2000:2104][::-1], "AT" * 75, BASE[1200:1233],
         "".join(rnd.choice("ACGT") for _ in range(150)), BASE[40:290], "ACG" * 40, BASE[5:12]]
LONG_READS = [BASE[50:50 + m] for m in (300, 700, 1100)] + ["".join(rnd.choice("ACGT") for _ in range(400))]


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _kernels(eng, refs, reads, scores=(5, -3, -4)):
    """The kernels of one plain, fetched call."""
    rs = eng.load_refset(refs)
    res, kernels = launched_kernels(lambda: rs.align(reads, scores))
    res.free(); rs.free()
    return kernels


# scores -> the short-path kernels they select (reads <= 256 bp; the 150 bp reads are class K = 19)
@pytest.mark.parametrize("scores, expect", [
    # fill_sub_slack = 0 (one match does not exceed |gap|): exact tile maxima; byte-tile traceback
    ((2, -1, -2), [r"\bfill_bias_kernel<19, false>", r"\btile_trace_kernel<19, false>"]),
    # mismatch + |gap| < 0: no biased fill
    ((5, -10, -4), [r"\bfill_kernel<19>", r"\btile_trace_kernel<19, false>"]),
    # 2 (max score + |gap|) + max |score| >= 250: no byte tiles, the group traceback
    ((60, -30, -40), [r"\bfill_bias_kernel<19, true>", r"\btrace_kernel<19>"]),
    ((60, -100, -40), [r"\bfill_kernel<19>", r"\btrace_kernel<19>"]),
], ids=["exact-tile-maxima", "unbiased-fill", "group-trace", "unbiased-fill-group-trace"])
def test_short_path_kernels(engine, scores, expect):
    kernels = _kernels(engine, REFS, READS, scores)
    for pattern in expect:
        assert launches(kernels, pattern), pattern
    assert check_pairs(engine, REFS, READS, scores, max_cells=400)
    assert check_pairs(engine, REFS[:3], READS[:5], scores)


# REFS cut at reference boundaries by weights parts .. 1 gives exactly `parts` parts for these two counts
@pytest.mark.parametrize("parts, scores", [(3, (5, -3, -4)), (4, (60, -30, -40))])
def test_reference_set_in_parts(parts, scores):
    """A workspace small against the set cuts it into parts (part k's results cross PCIe while part k + 1 computes):
    the stitched arrays must be the single-set ones."""
    eng = swb.Engine(0, workspace_bytes=parts_workspace(REFS, parts))
    try:
        assert len(launches(_kernels(eng, REFS, READS, scores), r"\bfold_best_kernel\b")) == parts   # once per part
        assert check_pairs(eng, REFS, READS + LONG_READS, scores, max_cells=200)
    finally:
        eng.close()


def test_scores_only_late_fetch_and_best_hits(engine):
    rs = engine.load_refset(REFS)
    full = rs.align(READS)
    so = rs.align(READS, scores_only=True)
    late = rs.align(READS, fetch=False)
    late.fetch()
    assert (so.scores == full.scores).all() and (late.scores == full.scores).all()
    assert (so.best_hits[:, :2] == full.best_hits[:, :2]).all() and (late.best_hits == full.best_hits).all()
    assert (late.cell_offsets == full.cell_offsets).all() and (late.cells == full.cells).all()
    assert (late.op_lens == full.op_lens).all()
    best = full.best_hits
    for q in range(len(READS)):
        col = full.scores[:, q]
        assert best[q, 0] == col.max() and best[q, 1] == int(np.argmax(col))
    full.free(); so.free(); late.free(); rs.free()


# a fifth symbol in the set sends every read through the wide path; rows per lane from the read length (pick_kl)
@pytest.mark.parametrize("kl, m", [(8, 200), (16, 400), (32, 700)])
def test_wide_rows_per_lane(engine, kl, m):
    refs = REFS[:3] + [BASE[:600] + "N" + BASE[600:1200]]
    reads = [BASE[90:90 + m], BASE[1000:1000 + m][::-1], BASE[400:400 + m // 2] + "N" + BASE[400 + m // 2:400 + m]]
    kernels = _kernels(engine, refs, reads)
    assert launches(kernels, rf"\bwide_fill_kernel<{kl}, 8>") and launches(kernels, rf"\bwide_trace_kernel<{kl}, ")
    assert check_pairs(engine, refs, reads, max_cells=200)


# nine symbols or more: no score profile in shared memory, the compare-and-select fill
@pytest.mark.parametrize("kl, m", [(8, 200), (16, 400), (32, 700)])
def test_wide_fill_without_profile(engine, kl, m):
    r = random.Random(kl)
    ref = "".join(r.choice("ACGTNRYKM") for _ in range(2000))
    mutated = "".join(c if r.random() > 0.05 else r.choice("ACGTNRYKM") for c in ref[300:300 + m])
    refs, reads = [ref, ref[::-1], ref[500:1400]], [mutated, ref[1000:1000 + m]]
    kernels = _kernels(engine, refs, reads)
    assert launches(kernels, rf"\bwide_fill_kernel<{kl}, 0>")
    assert check_pairs(engine, refs, reads, max_cells=200)


def test_wide_trace_without_byte_tiles(engine):
    """2 (max score + |gap|) + max |score| >= 250 rules out byte tiles: the int32 tiles of the wide traceback."""
    reads = [BASE[50:450], LONG_READS[3]]                           # 400 rows: KL = 16; 60 x 400 is past the s16 range
    kernels = _kernels(engine, REFS, reads, (60, -30, -40))
    assert launches(kernels, r"\bwide_trace_kernel<16, 32, 32, false>")
    assert check_pairs(engine, REFS, reads, (60, -30, -40), max_cells=200)


# read lengths of the tie sets: one band of KL = 8, 16 and 32 rows per lane (pick_kl)
KL_OF_READ = {200: 8, 400: 16, 700: 32}


def _tie_set(m, n_cells, copies=1):
    """read A x m against `copies` references of A's with n_cells max cells each (row m, every column from m on), in
    a set with C, G, T and N: every read takes the wide path, the last reference scores 0."""
    return ["A" * (m - 1 + n_cells)] * copies + ["CGTN" * 50], ["A" * m]


# the traceback's lanes per max cell follow the cell count of the launch: a thread or a warp; byte tiles of NTB slots
@pytest.mark.parametrize("m", sorted(KL_OF_READ))
@pytest.mark.parametrize("grouping", ["thread", "warp"])
def test_wide_trace_grouping(engine, grouping, m):
    sm, kl = _sm_count(), KL_OF_READ[m]
    ntb = 64 if kl >= 32 else 128
    if grouping == "thread":                                        # >= 256 cells per SM
        per_ref = 20000 - m + 1
        refs, reads = _tie_set(m, per_ref, copies=-(-256 * sm // per_ref) + 1)
        pattern = rf"\bwide_trace_kernel<{kl}, {ntb}, 1, true>"
    else:                                                           # more cells than SMs, fewer than 256 per SM
        refs, reads = _tie_set(m, 8 * sm)
        pattern = rf"\bwide_trace_kernel<{kl}, {ntb}, 32, true>"
    assert launches(_kernels(engine, refs, reads), pattern)
    assert check_pairs(engine, refs, reads, max_cells=100)


@pytest.mark.parametrize("m", sorted(KL_OF_READ))
@pytest.mark.parametrize("c", [3, 2, 1])
def test_wide_trace_cluster(engine, c, m):
    """No more cells than SMs: one cluster of c CTAs per cell, c = 3 while every cluster is resident at once, fewer
    for more cells.  The kernel's grid is c times the cell count."""
    sm, kl = _sm_count(), KL_OF_READ[m]
    n_cells = {3: sm // 3, 2: sm // 2, 1: sm}[c]
    refs, reads = _tie_set(m, n_cells)
    grids = launches(_kernels(engine, refs, reads), rf"\bwide_trace_kernel<{kl}, 256, 256, true>")
    assert grids == [c * n_cells], grids
    assert check_pairs(engine, refs, reads, max_cells=100)
