"""GPU: the wide traceback (swb_wide.cu, wide_trace_kernel) on planted pairs (tests/wide_trace_cases.py) -- gaps, path
ends and max cells on tile, lane-row, band and round edges -- under every grouping of its walkers: a cluster of 3, 2 or
1 CTAs per max cell, a warp, a thread.  Between the five calls of a group only a filler tie set changes, sized from the
SM count so that the launch's max-cell count lands in each grouping's range; every planted pair must equal the oracle
in each of them (so the five calls agree with each other), under both tie rules.  Each case's geometry is asserted on
the oracle's own path before the first call."""
import re

import pytest
import torch

from tests import wide_trace_cases as W
from tests.helpers import check_pairs, launches, oracle_arrays, oracle_key

pytestmark = pytest.mark.gpu

GROUPS = W.all_groups()
ROWS = ["c3", "c2", "c1", "warp", "thread"]


@pytest.fixture(scope="module")
def sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _target(row, sm):
    """Max cells of a launch that lands in this row of the grouping matrix."""
    return {"c3": sm // 3, "c2": sm // 2, "c1": sm, "warp": 8 * sm, "thread": 256 * sm}[row]


def _oracle(g, tie_gt):
    """Oracle arrays of every case of the group, its geometry asserted first; memo keyed for check_pairs."""
    memo, counts = {}, []
    for c in g.cases:
        exp = oracle_arrays(g.ref, c.read, g.scores, tie_gt=tie_gt)
        c.assert_geometry(exp, g.scores, g.ref, g.kl)
        memo[oracle_key(g.ref, c.read, g.scores, tie_gt)] = exp
        counts.append(exp["count"])
    return memo, counts


def _chunks(counts, budget):
    """Cases cut into calls of at most `budget` max cells."""
    out, cur, n = [], [], 0
    for k, c in enumerate(counts):
        assert c < budget, f"case {k} has {c} max cells"
        if n + c > budget:
            out.append(cur)
            cur, n = [], 0
        cur.append(k)
        n += c
    return out + [cur] if cur else out


@pytest.mark.parametrize("tie_gt", [False, True], ids=["ge", "gt"])
@pytest.mark.parametrize("gi", range(len(GROUPS)), ids=[g.name for g in GROUPS])
def test_planted_pairs_every_grouping(engine, sm, gi, tie_gt):
    g = GROUPS[gi]
    memo, counts = _oracle(g, tie_gt)
    byte = W.tile_trace_ok(*g.scores)
    for chunk in _chunks(counts, sm // 3 - 1):
        reads = [g.cases[k].read for k in chunk]
        planted = sum(counts[k] for k in chunk)
        m_f = len(reads[0])                                 # the filler read: same rows-per-lane class
        for row in ROWS:
            total = _target(row, sm)
            refs = [g.ref, W.FILLER * (m_f - 1 + total - planted)]
            pairs = [(0, q) for q in range(len(reads))] + ([(1, len(reads))] if row == "c3" else [])
            kernels = []
            try:
                check_pairs(engine, refs, reads + [W.FILLER * m_f], g.scores, pairs=pairs, max_cells=40, tie_gt=tie_gt,
                            memo=memo, kernels=kernels)
            except AssertionError as e:
                q = re.search(r"ref=0 read=(\d+)", str(e))
                raise AssertionError(f"{row}, case {g.cases[chunk[int(q.group(1))]].name if q else '-'}: {e}") from None
            # one traceback launch of this class holds every max cell, planted and filler, in the expected mode
            group = W.grouping(total, sm)
            assert len(launches(kernels, rf"\bwide_trace_kernel<{g.kl}, ")) == 1, (row, kernels)
            grids = launches(kernels, W.trace_kernel(g.kl, group, byte))
            assert len(grids) == 1, (row, W.trace_kernel(g.kl, group, byte), sorted({k for k, _ in kernels}))
            if group == "cluster" and byte:
                assert grids == [W.cluster_c(total, sm) * total] and W.cluster_c(total, sm) == int(row[1]), (row, grids)


@pytest.mark.parametrize("tie_gt", [False, True], ids=["ge", "gt"])
def test_positive_mismatch_byte_tiles(engine, sm, tie_gt):
    """A positive mismatch above the match score on byte tiles: every pair scores more than 32 * max(|match|, |mismatch|),
    so the walker takes whole 32-step diagonal ballots, in the grouping its max-cell count selects (some thousand cells:
    the warp walker).  The filler symbol in a second reference sends the reads of up to 256 rows through the wide
    path."""
    scores = (3, 7, -2)
    assert W.tile_trace_ok(*scores)
    g = W.ends_group(8, (5, -3, -1))
    refs, reads = [g.ref, W.FILLER * 40], [c.read for c in g.cases[:12]]
    memo, total = {}, 0
    for r in range(len(refs)):
        for q, read in enumerate(reads):
            exp = oracle_arrays(refs[r], read, scores, tie_gt=tie_gt)
            memo[oracle_key(refs[r], read, scores, tie_gt)] = exp
            total += exp["count"]
            if r == 0:
                assert exp["score"] > 32 * 7, f"wrong geometry: read {q} scores {exp['score']}"
    kernels = []
    check_pairs(engine, refs, reads, scores, pairs=[(0, q) for q in range(len(reads))], max_cells=20, tie_gt=tie_gt,
                memo=memo, kernels=kernels)
    assert len(launches(kernels, r"\bwide_trace_kernel<8, ")) == 1
    assert len(launches(kernels, W.trace_kernel(8, W.grouping(total, sm), True))) == 1, (total, kernels)
