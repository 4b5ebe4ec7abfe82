"""CPU: the whole-result comparator of tests/helpers.py.  oracle_arrays must say what the list form of the oracle says,
the one-lexsort re-order must be DistributedSW's order, and assert_pair_equal must accept the oracle's own result fed
back as the engine's and reject each way an engine could get a cell list subtly wrong."""
import random

import numpy as np
import pytest

import oracle
from sparksmithwaterman_b200 import sw
from tests.helpers import OP_ALIGN, OP_DEL, OP_INS, _segments, assert_pair_equal, distributed_permutation, oracle_arrays

# small tie-heavy pairs: repeats, low-complexity sequence, indels inside repeats, zero and cheap gaps
PAIRS = [("AT" * 30, "AT" * 8), ("A" * 40, "A" * 12), ("ACG" * 20, "ACGACGTACGACG"), ("AC" * 25, "ACACACCACAC"),
         ("GATTACA" * 4, "TTACAGATT"), ("CCAAT", "CAT"), ("GTTCA", "CTA"), ("AAAA", "CC"), ("ACGT", ""),
         ("acgtACGTac", "ACGTacgT")]
SCORES = [(5, -3, -4), (1, -1, -1), (2, -2, 0), (3, 1, -2)]
CASES = [(r, q, s) for r, q in PAIRS for s in SCORES]


def _ops_of(ref_aln, read_aln):
    return [OP_INS if a == "_" else (OP_DEL if b == "_" else OP_ALIGN) for a, b in zip(ref_aln, read_aln)]


def _as_result(exp, tie_gt):
    """The oracle's arrays laid out as the engine lists them: cells row-major under both tie rules, score-0 pairs
    with no materialised cells and the closed form at a few probe indices."""
    got = {k: exp[k] for k in ("score", "count", "m", "n")}
    if exp["score"] == 0:
        mn = exp["m"] * exp["n"]
        ks = np.array(sorted({0, max(mn - 1, 0), mn // 2}), np.int64)
        got.update(cells=np.zeros((0, 2), np.int32), beginnings=np.zeros(0, np.int32), op_lens=np.zeros(0, np.int64),
                   ops=np.zeros(0, np.uint8), count=mn,
                   probe=np.stack([ks, ks // max(exp["n"], 1) + 1, ks % max(exp["n"], 1) + 1, 0 * ks, 0 * ks], axis=1))
        return got
    order = np.arange(exp["count"])
    if tie_gt:
        order = np.lexsort((exp["cells"][:, 1], exp["cells"][:, 0]))        # back to row-major
    got.update(cells=exp["cells"][order], beginnings=exp["beginnings"][order], op_lens=exp["op_lens"][order],
               ops=exp["ops"][_segments(exp["op_lens"], order)])
    return got


@pytest.mark.parametrize("tie_gt", [False, True])
@pytest.mark.parametrize("ref,read,scores", CASES)
def test_oracle_arrays_equal_the_list_form(ref, read, scores, tie_gt):
    exp = oracle.align(ref, read, *scores, tie_gt=tie_gt)
    a = oracle_arrays(ref, read, scores, tie_gt=tie_gt)
    assert a["score"] == exp.score and a["count"] == len(exp.cells) and (a["m"], a["n"]) == (len(read), len(ref))
    assert [tuple(c) for c in a["cells"].tolist()] == exp.cells
    assert a["beginnings"].tolist() == [s[0] for s in exp.sites]
    assert a["op_lens"].tolist() == [len(s[1]) for s in exp.sites]
    assert a["ops"].tolist() == [op for s in exp.sites for op in _ops_of(s[1], s[2])]


def test_oracle_arrays_refuse_the_gap_symbol():
    with pytest.raises(AssertionError):
        oracle_arrays("AC_GT", "ACGT")
    with pytest.raises(AssertionError):
        oracle_arrays("ACGT", "A_C")


@pytest.mark.parametrize("seed", range(20))
def test_lexsort_is_distributed_order(seed):
    rnd = random.Random(seed)
    n = rnd.randint(0, 400)
    cells = sorted({(rnd.randint(1, 30), rnd.randint(1, 60)) for _ in range(n)})          # row-major, unique
    sites = [(rnd.randint(0, 8), f"r{k}", f"q{k}") for k in range(len(cells))]          # many equal beginnings
    exp_cells, exp_sites = sw.distributed_order(cells, sites)
    arr = np.array(cells, np.int32).reshape(-1, 2)
    order = distributed_permutation(arr, np.array([s[0] for s in sites], np.int32))
    assert [cells[k] for k in order] == exp_cells and [sites[k] for k in order] == exp_sites


@pytest.mark.parametrize("tie_gt", [False, True])
@pytest.mark.parametrize("ref,read,scores", CASES)
def test_comparator_accepts_the_oracle_fed_back(ref, read, scores, tie_gt):
    exp = oracle_arrays(ref, read, scores, tie_gt=tie_gt)
    assert_pair_equal(_as_result(exp, tie_gt), exp, tie_gt)


def _copy(got):
    return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in got.items()}


def _drop_last(g):
    g["cells"], g["beginnings"] = g["cells"][:-1], g["beginnings"][:-1]
    g["ops"], g["op_lens"] = g["ops"][:len(g["ops"]) - int(g["op_lens"][-1])], g["op_lens"][:-1]
    g["count"] -= 1


def _duplicate(g):                                   # the second-to-last cell written twice, the last one lost
    c = len(g["cells"])
    keep = list(range(c - 1)) + [c - 2]
    g["ops"] = g["ops"][_segments(g["op_lens"], np.array(keep))]
    g["cells"], g["beginnings"], g["op_lens"] = g["cells"][keep], g["beginnings"][keep], g["op_lens"][keep]


def _swap(g):
    c = len(g["cells"])
    order = np.arange(c)
    order[[c // 2, c // 2 + 1]] = order[[c // 2 + 1, c // 2]]
    g["ops"] = g["ops"][_segments(g["op_lens"], order)]
    g["cells"], g["beginnings"], g["op_lens"] = g["cells"][order], g["beginnings"][order], g["op_lens"][order]


def _beginning(g):
    g["beginnings"][len(g["beginnings"]) // 2] += 1


def _op(g):
    k = len(g["ops"]) // 2
    g["ops"][k] = OP_ALIGN if g["ops"][k] != OP_ALIGN else OP_DEL


def _op_len(g):                                      # one op length one longer, the next one shorter: same ops
    k = int(np.nonzero(g["op_lens"][1:] > 0)[0][-1])
    g["op_lens"][k] += 1
    g["op_lens"][k + 1] -= 1


PERTURB = {"last-cell-missing": _drop_last, "cell-duplicated": _duplicate, "cells-swapped": _swap,
           "beginning+1": _beginning, "op-changed": _op, "op-length-moved": _op_len}

# tie-heavy pairs with enough cells for every perturbation, and a beginning that differs between neighbours
# (the last two list max cells on several rows, so that DistributedSW's order is not the row-major one)
RICH = [("ACG" * 20, "ACGACGTACGACG", (5, -3, -4)), ("AT" * 30, "AT" * 8, (1, -1, -1)), ("AC" * 25, "ACACACCACAC", (2, -2, 0)),
        ("CACCCCACACACAC", "CAAAAAC", (2, -3, -3)), ("AAACACACAACCAA", "ACACCCC", (1, -1, -1))]


@pytest.mark.parametrize("tie_gt", [False, True])
@pytest.mark.parametrize("how", sorted(PERTURB))
@pytest.mark.parametrize("ref,read,scores", RICH)
def test_comparator_rejects(ref, read, scores, how, tie_gt):
    exp = oracle_arrays(ref, read, scores, tie_gt=tie_gt)
    assert exp["count"] >= 4 and exp["score"] > 0
    got = _copy(_as_result(exp, tie_gt))
    PERTURB[how](got)
    with pytest.raises(AssertionError):
        assert_pair_equal(got, exp, tie_gt)


@pytest.mark.parametrize("ref,read,scores", RICH[3:])
def test_comparator_rejects_a_wrong_order_under_tie_gt(ref, read, scores):
    exp = oracle_arrays(ref, read, scores, tie_gt=True)
    assert (np.lexsort((exp["cells"][:, 1], exp["cells"][:, 0])) != np.arange(exp["count"])).any()
    # the engine must list row-major: DistributedSW's own order handed over as the list is wrong ...
    with pytest.raises(AssertionError):
        assert_pair_equal(_copy(exp), exp, tie_gt=True)
    # ... and a row-major list compared without the re-order is too
    with pytest.raises(AssertionError):
        assert_pair_equal(_as_result(exp, True), exp, tie_gt=False)


def test_comparator_rejects_a_wrong_score0_count():
    exp = oracle_arrays("AAAA", "CCC")
    assert exp["score"] == 0 and exp["count"] == 12
    got = _as_result(exp, False)
    assert_pair_equal(got, exp)
    for bad in (11, 13, 0):
        g = _copy(got)
        g["count"] = bad
        with pytest.raises(AssertionError):
            assert_pair_equal(g, exp)
    g = _copy(got)
    g["probe"][-1, 2] += 1                           # pair_cell's closed form off by one column
    with pytest.raises(AssertionError):
        assert_pair_equal(g, exp)
