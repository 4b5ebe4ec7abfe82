"""GPU: all-hits mode (swb_align_all_hits).  Every case runs the plain call and the all-hits call on the same inputs:
scores, totals and best hits must be the plain ones, the lists the numpy rule on the plain scores, every listed pair's
cells / beginnings / op lengths / alignments the plain ones, and every other pair must have no cells."""
import random
import re

import numpy as np
import pytest

import oracle
import sparksmithwaterman_b200 as swb
from sparksmithwaterman_b200 import synth
from sparksmithwaterman_b200.engine import reverse_complement
from tests.helpers import assert_ranges_equal, launched_kernels, launches, parts_workspace, result_range
from tests.test_all_hits_host import all_hits_ref

pytestmark = pytest.mark.gpu

BIG = 2**31 - 1


def _rand(rnd, n, alphabet="ACGT"):
    return "".join(rnd.choice(alphabet) for _ in range(n))


def check_all_hits(eng, refs, reads, scores=(5, -3, -4), min_score=1, margin=0, scores_only=False, tie_gt=False, fetch=True,
                   both_strands=False):
    rs = eng.load_refset(refs)
    plain = rs.align(reads, scores, scores_only=scores_only, tie_gt=tie_gt, both_strands=both_strands).cache()
    ar = rs.align(reads, scores, scores_only, fetch, tie_gt, min_score=min_score, margin=margin, both_strands=both_strands)
    if not fetch:
        assert len(ar.hit_offsets) == 0                          # nothing on the host before the fetch
        ar.fetch()
    ar.cache()
    assert (ar.scores == plain.scores).all()
    assert (ar.ref_totals == plain.ref_totals).all()
    assert (ar.best_hits == plain.best_hits).all()
    off, lst = ar.hit_offsets, ar.hit_list
    exp_o, exp_l = all_hits_ref(plain.scores, min_score, margin)
    assert (off == exp_o).all()
    assert (lst[:, :2] == exp_l[:, :2]).all()
    if scores_only:
        assert (lst[:, 2:] == 0).all()
        plain.free(); ar.free(); rs.free()
        return off, lst
    n_refs, n_reads = plain.n_refs, plain.n_reads
    cnt_a = np.diff(ar.cell_offsets).reshape(n_refs, n_reads)
    cnt_p = np.diff(plain.cell_offsets).reshape(n_refs, n_reads)
    mask = np.zeros((n_refs, n_reads), bool)
    for q in range(n_reads):
        for score, ref, i, j in lst[off[q]:off[q + 1]]:
            mask[ref, q] = True
            assert cnt_a[ref, q] == cnt_p[ref, q] > 0
            assert ar.pair_cell_count(int(ref), q) == plain.pair_cell_count(int(ref), q)
            want = result_range(plain, ref * n_reads + q)
            assert_ranges_equal(result_range(ar, ref * n_reads + q), want, (ref, q))
            assert (i, j) == tuple(want["cells"][0])
            assert ar.pair(int(ref), q, 20) == plain.pair(int(ref), q, 20), (ref, q)  # the string builder
    assert (cnt_a[~mask] == 0).all()
    assert ar.total_cells == int(cnt_p[mask].sum())
    for ref, q in list(zip(*np.nonzero(~mask)))[:20]:
        assert ar.pair_cell_count(int(ref), int(q)) == 0
    plain.free(); ar.free(); rs.free()
    return off, lst


@pytest.mark.parametrize("lengths", [(36, 100, 150, 250), (300, 500)])
@pytest.mark.parametrize("min_score,margin", [(1, 0), (40, 10), (1, BIG)])
def test_read_length_classes(engine, lengths, min_score, margin):
    refs = synth.make_refs(60, lo=50, hi=3000)
    reads = []
    for m in lengths:
        reads += synth.make_reads(6, m, refs, seed=m)
    check_all_hits(engine, refs, reads, min_score=min_score, margin=margin)


def test_wide_path_long_reads_and_alphabet(engine):
    rnd = random.Random(3)
    refs = [_rand(rnd, n) for n in (400, 900, 1500, 2500, 700)]
    reads = [refs[3][100:700], refs[2][0:650], _rand(rnd, 600), refs[1][10:160]]
    for ms, margin in ((1, 0), (60, 20), (1, BIG)):
        check_all_hits(engine, refs, reads, min_score=ms, margin=margin)
    refs5 = [_rand(rnd, n, "ACGTN") for n in (300, 800, 120)]
    reads5 = [refs5[1][50:200], _rand(rnd, 90, "ACGTN"), refs5[0][:60]]
    check_all_hits(engine, refs5, reads5, min_score=1, margin=5)
    check_all_hits(engine, refs5, reads5, min_score=100, margin=BIG)


def test_unbiased_fill_and_group_traceback(engine):
    refs = synth.make_refs(40, lo=50, hi=2000)
    reads = synth.make_reads(10, 150, refs, seed=9)
    check_all_hits(engine, refs, reads, scores=(60, -30, -60), min_score=1, margin=300)
    check_all_hits(engine, refs, reads, scores=(60, -30, -60), min_score=2000, margin=BIG)


def test_cfg5_and_a_repeat_family_beyond_32(engine):
    """Tie-heavy cfg5 at margin 0 lists each read's co-optimal set; a repeat family of 48 references that share a
    segment gives reads with more co-optimal references than hits mode's cap of 32, and all of them are listed."""
    from tests.test_gpu_cfg_sizes import _cfg5_workload
    refs, reads = _cfg5_workload()
    off, _ = check_all_hits(engine, refs, reads, min_score=1, margin=0)
    assert (np.diff(off) > 1).any()
    rnd = random.Random(5)
    segment = _rand(rnd, 300)
    family = [_rand(rnd, rnd.randrange(50, 400)) + segment + _rand(rnd, rnd.randrange(50, 400)) for _ in range(48)]
    refs = [_rand(rnd, rnd.randrange(300, 1200)) for _ in range(30)] + family
    rnd.shuffle(refs)
    reads = [segment[10:160], segment[120:270], _rand(rnd, 150)]
    off, lst = check_all_hits(engine, refs, reads, min_score=1, margin=0)
    assert off[1] - off[0] >= 48 and off[2] - off[1] >= 48
    fam = sorted(k for k, r in enumerate(refs) if segment in r)
    assert sorted(lst[off[0]:off[1], 1]) == fam


def test_min_score_high_enough_that_some_reads_list_nothing(engine):
    refs = synth.make_refs(40, lo=50, hi=2500)
    reads = synth.make_reads(8, 150, refs, seed=14) + [b"GATTACA", b"CCCCCCCCCCCC"]
    off, _ = check_all_hits(engine, refs, reads, min_score=200, margin=BIG)
    assert (np.diff(off) == 0).any() and (np.diff(off) > 0).any()


@pytest.mark.parametrize("mode", ["scores_only", "tie_gt", "no_fetch"])
def test_flags(engine, mode):
    refs = synth.make_refs(50, lo=50, hi=2500)
    reads = synth.make_reads(8, 150, refs, seed=4) + synth.make_reads(4, 600, refs, seed=5)
    kw = {"scores_only": mode == "scores_only", "tie_gt": mode == "tie_gt", "fetch": mode != "no_fetch"}
    check_all_hits(engine, refs, reads, min_score=1, margin=0, **kw)
    check_all_hits(engine, refs, reads, min_score=50, margin=30, **kw)


@pytest.mark.parametrize("margin", [0, 25, BIG])
def test_both_strands(engine, margin):
    refs = synth.make_refs(40, lo=50, hi=2500)
    fwd = synth.make_reads(6, 150, refs, seed=31)
    reads = fwd[:3] + [reverse_complement(q) for q in fwd[3:]] + synth.make_reads(2, 600, refs, seed=32)
    check_all_hits(engine, refs, reads, min_score=30, margin=margin, both_strands=True)


def test_resident_reads_and_a_set_in_three_parts():
    refs = synth.make_refs(90, lo=50, hi=3000)
    reads = synth.make_reads(10, 150, refs, seed=3) + synth.make_reads(3, 600, refs, seed=6)
    eng = swb.Engine(0, workspace_bytes=parts_workspace(refs, 3))
    try:
        rs = eng.load_refset(refs)
        res, kernels = launched_kernels(lambda: rs.align(reads))
        assert len(launches(kernels, r"\bfold_best_kernel\b")) >= 2          # the plain call ran part by part
        res.free()
        rd = rs.upload_reads(reads)
        a = rs.align(reads, margin=5, min_score=20)
        b = rd.align(margin=5, min_score=20)
        assert (a.hit_offsets == b.hit_offsets).all() and (a.hit_list == b.hit_list).all()
        assert (a.cells == b.cells).all() and (a.cell_offsets == b.cell_offsets).all()
        a.free(); b.free(); rd.free(); rs.free()
        for ms, margin in ((1, 0), (60, 40)):
            check_all_hits(eng, refs, reads, min_score=ms, margin=margin)
        check_all_hits(eng, refs, reads, min_score=1, margin=3, fetch=False)
    finally:
        eng.close()


def test_hits_mode_is_a_prefix(engine):
    refs = synth.make_refs(60, lo=50, hi=2500)
    reads = synth.make_reads(10, 150, refs, seed=17) + synth.make_reads(2, 600, refs, seed=18)
    rs = engine.load_refset(refs)
    for ms in (1, 30):
        ar = rs.align(reads, min_score=ms, margin=BIG)
        off, lst = ar.hit_offsets, ar.hit_list
        for k in (1, 5, 32):
            hr = rs.align(reads, top_k=k, min_score=ms)
            h = hr.hits
            for q in range(len(reads)):
                n = int((h[q, :, 1] >= 0).sum())
                assert n == min(k, int(off[q + 1] - off[q]))
                assert (h[q, :n] == lst[off[q]:off[q] + n]).all()
            hr.free()
        ar.free()
    rs.free()


def test_invalid_arguments(engine):
    rs = engine.load_refset(["ACGTACGT"])
    for ms, margin in ((0, 0), (-3, 5), (1, -1), (5, -100)):
        with pytest.raises(swb.SwbError) as ei:
            rs.align(["ACGT"], min_score=ms, margin=margin)
        assert ei.value.code == -1
    with pytest.raises(ValueError):
        rs.align(["ACGT"], top_k=3, margin=0)
    rs.free()


def test_listed_pairs_against_the_oracle(engine):
    refs = [r.decode() for r in synth.make_refs(25, lo=50, hi=1500)]
    reads = [q.decode() for q in synth.make_reads(8, 150, [r.encode() for r in refs], seed=11)]
    rs = engine.load_refset(refs)
    ar = rs.align(reads, min_score=20, margin=60).cache()
    n = 0
    for q in range(len(reads)):
        for ref, score, cells, sites in ar.read_hits(q):
            exp = oracle.align(refs[ref], reads[q])
            assert (score, cells, sites) == (exp.score, exp.cells, exp.sites)
            n += 1
    assert n >= 8
    ar.free(); rs.free()


def test_selection_kernels_run_and_the_emit_is_the_hits_one(engine):
    refs = synth.make_refs(40, lo=50, hi=2500)
    reads = synth.make_reads(8, 150, refs, seed=41)
    rs = engine.load_refset(refs)
    res, kernels = launched_kernels(lambda: rs.align(reads, min_score=1, margin=0))
    for name in ("margin_best_kernel", "margin_mark_kernel", "margin_count_kernel", "margin_write_kernel", "list_cells_kernel"):
        assert launches(kernels, name), name
    names = [n for n, _ in kernels if "tile_emit_kernel" in n]
    assert names and all(re.search(r"\btile_emit_kernel<\d+, true>", n) for n in names), names
    assert not launches(kernels, r"hits_partial_kernel")
    res.free(); rs.free()


def _device_count():
    from sparksmithwaterman_b200 import _ffi
    return int(_ffi.load().swb_device_count())


@pytest.mark.parametrize("n_gpus", [1, 2, 4, 8])
def test_multi_gpu_merged_lists(engine, n_gpus):
    if _device_count() < n_gpus:
        pytest.skip(f"needs {n_gpus} GPUs")
    from sparksmithwaterman_b200 import multigpu
    refs = synth.make_refs(70, lo=50, hi=3000)
    reads = synth.make_reads(12, 150, refs, seed=12) + synth.make_reads(2, 600, refs, seed=13) + [b"", b"GGGG"]
    rs = engine.load_refset(refs)
    for ms, margin, both in ((1, 0, False), (1, 20, False), (60, BIG, False), (1, 10, True)):
        one = rs.align(reads, min_score=ms, margin=margin, both_strands=both).cache()
        me = multigpu.MultiEngine(list(range(n_gpus)))
        me.load_refset(refs)
        mr = me.align(reads, min_score=ms, margin=margin, both_strands=both)
        assert (mr.hit_offsets == one.hit_offsets).all(), (n_gpus, ms, margin)
        assert (mr.hit_list == one.hit_list).all(), (n_gpus, ms, margin)
        assert (mr.best_hits == one.best_hits).all()
        off, lst = mr.hit_offsets, mr.hit_list
        for q in range(len(reads)):
            for score, ref, i, j in lst[off[q]:off[q + 1]][:5]:
                assert mr.pair(int(ref), q, 100) == one.pair(int(ref), q, 100)
        mr.free(); me.close(); one.free()
    rs.free()


def test_comm_allgather_all_hits_world1(engine):
    """The one-process-per-device form at world 1 (no NCCL): the merged lists are the result's own with the reference
    indices moved through global_ids."""
    from sparksmithwaterman_b200 import multigpu
    refs = synth.make_refs(40, lo=50, hi=2500)
    reads = synth.make_reads(10, 150, refs, seed=21) + [b"", b"CCCC"]
    rs = engine.load_refset(refs)
    res = rs.align(reads, min_score=1, margin=15)
    ids = np.arange(len(refs), dtype=np.int64) * 3 + 7                 # any ascending global numbering
    comm = multigpu.Comm(engine, b"\0" * 128, 0, 1)
    off, lst = comm.allgather_all_hits(res, ids)
    exp = res.hit_list.copy()
    exp[:, 1] = ids[exp[:, 1]]
    assert (off == res.hit_offsets).all() and (lst == exp).all()
    with pytest.raises(swb.SwbError):
        comm.allgather_all_hits(rs.align(reads), ids)                  # a plain result has no lists
    comm.close(); res.free(); rs.free()
