"""GPU: every max cell of every pair against the oracle, at the cell counts tie-heavy genomic input produces.  Each
large row sizes its workload from the device's SM count, asserts from a profile of the call which traceback kernel ran
and with which grid, and compares every cell, beginning, op length and op through check_pairs:
  - the short tile traceback (launch_tile_trace_k) and the group traceback (launch_trace) with chunks of the sorted
    cell list longer than 256 cells, which they take only above sm_count * 16 * 256 and sm_count * 4 * 256 cells;
  - the locate stage's second attempt after its first cell list overflowed (short and wide path);
  - the strict '>' tie rule (SWB_F_TIE_GT) over both fuzz generators;
  - short, long-class and wide reads in one call, whole and with the reference set cut into parts."""
import random

import pytest
import torch

import oracle
import sparksmithwaterman_b200 as swb
from tests.helpers import check_pairs, launched_kernels, launches, parts_workspace
from tests.test_gpu_fuzz import SCORE_SETS, _workload
from tests.test_gpu_long_classes import LONG_SCORE_SETS, _fuzz_workload

pytestmark = pytest.mark.gpu

MARGIN = 1.08                                   # cell counts this far above each threshold


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _tandem(rnd, unit, n, subs, indels):
    """A tandem repeat of `unit`, n bases, with a few substitutions and single-base indels."""
    s = list((unit * (n // len(unit) + 2))[:n])
    for _ in range(subs):
        p = rnd.randrange(len(s))
        s[p] = rnd.choice("ACGT".replace(s[p], ""))
    for _ in range(indels):
        p = rnd.randrange(len(s))
        if rnd.random() < 0.5:
            del s[p]
        else:
            s.insert(p, rnd.choice("ACGT"))
    return "".join(s)


def _tie_reads(m, at):
    """Reads of m rows whose best paths carry a gap inside a repeat, where its position ties: an ACG repeat with one
    inserted base and an AC repeat with one deleted base, the gap near row `at`."""
    acg, ac = "ACG" * (m // 3 + 2), "AC" * (m // 2 + 2)
    return [acg[:at] + "T" + acg[at:m - 1], ac[:at] + ac[at + 1:m + 1]]


def _grow(rnd, reads, make_ref, scores, target, refs=()):
    """References from make_ref(rnd) until the call's max cells (counted by the oracle) exceed `target`.  Returns
    (refs, max cells per read)."""
    refs = list(refs)
    per_read = [sum(oracle.score(r, q, *scores)[1] for r in refs) for q in reads]
    while sum(per_read) <= target:
        r = make_ref(rnd)
        refs.append(r)
        for k, q in enumerate(reads):
            per_read[k] += oracle.score(r, q, *scores)[1]
    return refs, per_read


def _short_tie_set(m, scores, target, seed):
    """Reads of m rows (one rows-per-lane class): a run of A and the two gapped repeats; references: runs of A and
    ACG / AC tandem repeats with substitutions and indels."""
    rnd = random.Random(seed)
    reads = ["A" * m] + _tie_reads(m, m // 2) + _tie_reads(m, m // 3)

    def ref(rnd):
        unit = rnd.choice(["A", "ACG", "ACG", "AC", "AC"])
        return _tandem(rnd, unit, rnd.randrange(1500, 3500), rnd.randint(1, 4), rnd.randint(0, 3))
    refs, per_read = _grow(rnd, reads, ref, scores, target)
    return refs, reads, sum(per_read)


def _call_profile(eng, refs, reads, scores, tie_gt=False):
    rs = eng.load_refset(refs)
    res, kernels = launched_kernels(lambda: rs.align(reads, scores, tie_gt=tie_gt))
    n = int(res.stats["max_cells"])
    res.free(); rs.free()
    return kernels, n


def _assert_locate_retried(kernels, k, n_cells, n_refs, n_reads):
    """The short path's first cell list holds 2 * pairs + 4096 cells (swb_align.cu locate_cells): past it the flag and
    locate kernels run again, once per attempt (a third attempt when the first one's task list overflowed too and
    undercounted the cells)."""
    pairs = (n_reads + 1) // 2 * 2 * n_refs
    assert n_cells > 2 * pairs + 4096
    attempts = len(launches(kernels, r"\bflag_tiles_kernel\b"))
    assert attempts in (2, 3)
    assert len(launches(kernels, rf"\btile_scan_kernel<{k}>")) == attempts
    assert len(launches(kernels, rf"\btile_emit_kernel<{k}, false>")) == attempts


def _cdiv(a, b):
    return -(-a // b)


@pytest.mark.parametrize("k,m,tie_gt", [(19, 150, False), (19, 150, True), (40, 300, False)],
                         ids=["K19-ge", "K19-gt", "K40-ge"])
def test_tile_trace_long_chunks(engine, k, m, tie_gt):
    """launch_tile_trace_k: chunk = ceil(n / (sm_count * 16)) cells, past 2 * NT = 256 above sm_count * 16 * 256."""
    sm = _sm_count()
    scores = (5, -3, -4)
    refs, reads, n = _short_tie_set(m, scores, int(sm * 16 * 256 * MARGIN), seed=k + int(tie_gt))
    kernels, n_call = _call_profile(engine, refs, reads, scores, tie_gt)
    assert n_call == n
    chunk = _cdiv(n, sm * 16)
    assert chunk > 256
    assert launches(kernels, rf"\btile_trace_kernel<{k}, {'true' if tie_gt else 'false'}>") == [_cdiv(n, chunk)]
    _assert_locate_retried(kernels, k, n, len(refs), len(reads))
    check_pairs(engine, refs, reads, scores, max_cells=20, tie_gt=tie_gt)


@pytest.mark.parametrize("tie_gt", [False, True], ids=["ge", "gt"])
def test_group_trace_long_chunks(engine, tie_gt):
    """launch_trace (no byte tiles for these scores): chunk = max(256, ceil(n / (sm_count * 4))) cells."""
    sm = _sm_count()
    scores = (60, -30, -40)
    refs, reads, n = _short_tie_set(150, scores, int(sm * 4 * 256 * MARGIN), seed=60 + int(tie_gt))
    kernels, n_call = _call_profile(engine, refs, reads, scores, tie_gt)
    assert n_call == n
    chunk = _cdiv(n, sm * 4)
    assert chunk > 256
    assert launches(kernels, r"\btrace_kernel<19>") == [_cdiv(n, chunk)]
    assert not launches(kernels, r"\btile_trace_kernel<")
    _assert_locate_retried(kernels, 19, n, len(refs), len(reads))
    check_pairs(engine, refs, reads, scores, max_cells=20, tie_gt=tie_gt)


def test_wide_locate_retry_thread_grouping(engine):
    """The wide path (a fifth symbol in the set sends the 300-row reads there too): per rows-per-lane batch more cells
    than its first list of 4 * pairs + 4096 and at least 256 per SM, so one thread walks each cell."""
    sm = _sm_count()
    scores = (5, -3, -4)
    rnd = random.Random(71)
    reads = {16: _tie_reads(300, 150) + _tie_reads(300, 101), 32: _tie_reads(700, 350) + _tie_reads(700, 233)}

    def ref(rnd):
        return _tandem(rnd, rnd.choice(["ACG", "AC"]), rnd.randrange(3000, 6000), rnd.randint(2, 6), rnd.randint(2, 6))
    refs = ["CGTN" * 50]
    all_reads = reads[16] + reads[32]
    per_kl = {kl: sum(oracle.score(refs[0], q, *scores)[1] for q in rd) for kl, rd in reads.items()}

    def short(kl):
        return per_kl[kl] <= max(sm * 256, 4 * len(reads[kl]) * len(refs) + 4096) * MARGIN
    while short(16) or short(32):
        r = ref(rnd)
        refs.append(r)
        for kl, rd in reads.items():
            per_kl[kl] += sum(oracle.score(r, q, *scores)[1] for q in rd)
    kernels, n_call = _call_profile(engine, refs, all_reads, scores)
    assert n_call == sum(per_kl.values())
    for kl, rd in reads.items():
        pairs = len(rd) * len(refs)
        assert per_kl[kl] > 4 * pairs + 4096 and per_kl[kl] >= sm * 256, (kl, per_kl[kl], pairs)
        ntb = 64 if kl >= 32 else 128
        grids = launches(kernels, rf"\bwide_trace_kernel<{kl}, {ntb}, 1, true>")
        groups = _cdiv(per_kl[kl], ntb)
        assert len(grids) == 1 and (grids[0] == groups or (grids[0] % sm == 0 and sm <= grids[0] < groups)), (kl, grids)
        assert len(launches(kernels, rf"\bwide_locate_kernel<{kl}>")) in (2, 3)     # the first list overflowed
    assert len(launches(kernels, r"\bwide_flag_kernel\b")) == len(launches(kernels, r"\bwide_locate_kernel<"))
    check_pairs(engine, refs, all_reads, scores, max_cells=20)


@pytest.mark.parametrize("seed", range(60))
def test_fuzz_tie_gt(engine, seed):
    rnd = random.Random(1000 + seed)
    refs, reads = _workload(rnd)
    check_pairs(engine, refs, reads, SCORE_SETS[seed % len(SCORE_SETS)], max_cells=300, tie_gt=True)


@pytest.mark.parametrize("seed", range(24))
def test_fuzz_long_classes_tie_gt(engine, seed):
    rnd = random.Random(5000 + seed)
    refs, reads = _fuzz_workload(rnd)
    check_pairs(engine, refs, reads, LONG_SCORE_SETS[seed % len(LONG_SCORE_SETS)], max_cells=300, tie_gt=True)


def _mixed_tie_set():
    rnd = random.Random(91)
    refs = [_tandem(rnd, u, n, 3, 3) for u, n in (("A", 900), ("ACG", 2400), ("AC", 1800), ("ACG", 1200), ("AC", 3000),
                                                   ("A", 400))]
    refs += ["".join(rnd.choice("ACGT") for _ in range(1500))]
    reads = ["A" * 150] + _tie_reads(150, 70) + _tie_reads(300, 140) + _tie_reads(700, 300) + ["A" * 300, "AC" * 50]
    return refs, reads


@pytest.mark.parametrize("tie_gt", [False, True], ids=["ge", "gt"])
def test_assembly_across_batches_and_parts(tie_gt):
    """Short, long-class and wide reads in one call (one batch per class, the wide path's own batches), assembled into
    one result: whole, and with the reference set cut into 3 parts."""
    refs, reads = _mixed_tie_set()
    eng = swb.Engine(0)
    try:
        check_pairs(eng, refs, reads, max_cells=50, tie_gt=tie_gt)
    finally:
        eng.close()
    eng = swb.Engine(0, workspace_bytes=parts_workspace(refs, 3))
    try:
        kernels, _ = _call_profile(eng, refs, reads, (5, -3, -4), tie_gt)
        assert len(launches(kernels, r"\bfold_best_kernel\b")) >= 3                   # part by part
        check_pairs(eng, refs, reads, max_cells=50, tie_gt=tie_gt)
    finally:
        eng.close()
