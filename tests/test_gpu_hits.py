"""GPU: hits mode (swb_align_hits).  Every case runs the plain call and the hits call on the same inputs: scores,
totals and best hits must be the plain ones, the hit lists the numpy top k of the plain scores, every hit pair's
cells / beginnings / op lengths / alignments the plain ones, and every other pair must have no cells."""
import random

import numpy as np
import pytest

import oracle
import sparksmithwaterman_b200 as swb
from sparksmithwaterman_b200 import synth
from tests.helpers import assert_ranges_equal, launched_kernels, launches, parts_workspace, result_range
from tests.test_hits_host import top_hits_ref

pytestmark = pytest.mark.gpu


def _rand(rnd, n, alphabet="ACGT"):
    return "".join(rnd.choice(alphabet) for _ in range(n))


def check_hits(eng, refs, reads, scores=(5, -3, -4), k=3, min_score=1, scores_only=False, tie_gt=False, fetch=True):
    rs = eng.load_refset(refs)
    plain = rs.align(reads, scores, scores_only=scores_only, tie_gt=tie_gt).cache()
    hr = rs.align(reads, scores, scores_only, fetch, tie_gt, top_k=k, min_score=min_score)
    if not fetch:
        assert hr.hits.shape == (len(reads), 0, 4)               # nothing on the host before the fetch
        hr.fetch()
    hr.cache()
    assert (hr.scores == plain.scores).all()
    assert (hr.ref_totals == plain.ref_totals).all()
    assert (hr.best_hits == plain.best_hits).all()
    hits = hr.hits
    exp = top_hits_ref(plain.scores, k, min_score)
    assert hits.shape == exp.shape
    assert (hits[:, :, :2] == exp[:, :, :2]).all()
    best = plain.best_hits
    has = best[:, 0] >= min_score
    assert (hits[has, 0] == best[has]).all() or scores_only
    if scores_only:
        assert (hits[:, :, 2:] == 0).all()
        plain.free(); hr.free(); rs.free()
        return hits
    n_refs, n_reads = len(refs), len(reads)
    cnt_h = np.diff(hr.cell_offsets).reshape(n_refs, n_reads)
    cnt_p = np.diff(plain.cell_offsets).reshape(n_refs, n_reads)
    mask = np.zeros((n_refs, n_reads), bool)
    for q in range(n_reads):
        for score, ref, i, j in hits[q]:
            if ref < 0:
                assert score == 0 and i == 0 and j == 0
                continue
            mask[ref, q] = True
            assert cnt_h[ref, q] == cnt_p[ref, q] > 0
            assert hr.pair_cell_count(ref, q) == plain.pair_cell_count(ref, q)
            want = result_range(plain, ref * n_reads + q)
            assert_ranges_equal(result_range(hr, ref * n_reads + q), want, (ref, q))
            assert (i, j) == tuple(want["cells"][0])
            assert hr.pair(ref, q, 20) == plain.pair(ref, q, 20), (ref, q)          # the string builder
    assert (cnt_h[~mask] == 0).all()
    assert hr.total_cells == int(cnt_p[mask].sum())
    for ref, q in list(zip(*np.nonzero(~mask)))[:20]:
        assert hr.pair_cell_count(int(ref), int(q)) == 0
    plain.free(); hr.free(); rs.free()
    return hits


@pytest.mark.parametrize("lengths", [(36, 100, 150, 250), (300, 500)])
@pytest.mark.parametrize("k,min_score", [(1, 1), (3, 40), (32, 1)])
def test_read_length_classes(engine, lengths, k, min_score):
    refs = synth.make_refs(60, lo=50, hi=3000)
    reads = []
    for m in lengths:
        reads += synth.make_reads(6, m, refs, seed=m)
    check_hits(engine, refs, reads, k=k, min_score=min_score)


def test_wide_path_long_reads_and_alphabet(engine):
    rnd = random.Random(3)
    refs = [_rand(rnd, n) for n in (400, 900, 1500, 2500, 700)]
    reads = [refs[3][100:700], refs[2][0:650], _rand(rnd, 600), refs[1][10:160]]
    for k, ms in ((1, 1), (3, 60), (32, 1)):
        check_hits(engine, refs, reads, k=k, min_score=ms)
    refs5 = [_rand(rnd, n, "ACGTN") for n in (300, 800, 120)]
    reads5 = [refs5[1][50:200], _rand(rnd, 90, "ACGTN"), refs5[0][:60]]
    check_hits(engine, refs5, reads5, k=2, min_score=1)
    check_hits(engine, refs5, reads5, k=2, min_score=100)


def test_unbiased_fill_and_group_traceback(engine):
    # |scores| this large leave the byte-tile traceback and the biased fill: unbiased fill + group traceback
    refs = synth.make_refs(40, lo=50, hi=2000)
    reads = synth.make_reads(10, 150, refs, seed=9)
    check_hits(engine, refs, reads, scores=(60, -30, -60), k=3, min_score=1)
    check_hits(engine, refs, reads, scores=(60, -30, -60), k=5, min_score=2000)


def test_cfg5_tie_heavy_cut_through_a_tie(engine):
    from tests.test_gpu_cfg_sizes import _cfg5_workload
    refs, reads = _cfg5_workload()
    for k in (1, 3, 32):
        hits = check_hits(engine, refs, reads, k=k, min_score=1)
    # a read whose top k is cut inside a run of equal scores (lowest reference indices win)
    rs = engine.load_refset(refs)
    sc = rs.align(reads, scores_only=True).scores
    assert any((sc[:, q] == sc[:, q].max()).sum() > 3 for q in range(len(reads)))
    rs.free()


@pytest.mark.parametrize("mode", ["scores_only", "tie_gt", "no_fetch"])
def test_flags(engine, mode):
    refs = synth.make_refs(50, lo=50, hi=2500)
    reads = synth.make_reads(8, 150, refs, seed=4) + synth.make_reads(4, 600, refs, seed=5)
    kw = {"scores_only": mode == "scores_only", "tie_gt": mode == "tie_gt", "fetch": mode != "no_fetch"}
    check_hits(engine, refs, reads, k=4, min_score=1, **kw)
    check_hits(engine, refs, reads, k=4, min_score=50, **kw)


def test_resident_reads(engine):
    refs = synth.make_refs(30, lo=50, hi=2000)
    reads = synth.make_reads(8, 100, refs, seed=8)
    rs = engine.load_refset(refs)
    rd = rs.upload_reads(reads)
    a = rs.align(reads, top_k=4)
    b = rd.align(top_k=4)
    assert (a.hits == b.hits).all() and (a.cells == b.cells).all() and (a.cell_offsets == b.cell_offsets).all()
    a.free(); b.free(); rd.free(); rs.free()


def test_invalid_arguments(engine):
    rs = engine.load_refset(["ACGTACGT"])
    for k, ms in ((0, 1), (33, 1), (-1, 1), (1, 0), (4, -5)):
        with pytest.raises(swb.SwbError) as ei:
            rs.align(["ACGT"], top_k=k, min_score=ms)
        assert ei.value.code == -1
    rs.free()


def test_hit_pairs_against_the_oracle(engine):
    refs = [r.decode() for r in synth.make_refs(25, lo=50, hi=1500)]
    reads = [q.decode() for q in synth.make_reads(8, 150, [r.encode() for r in refs], seed=11)]
    rs = engine.load_refset(refs)
    hr = rs.align(reads, top_k=3, min_score=20).cache()
    n = 0
    for q in range(len(reads)):
        for res in hr.read_hits(q):
            ref, score, cells, sites = res
            exp = oracle.align(refs[ref], reads[q])
            assert (score, cells, sites) == (exp.score, exp.cells, exp.sites)
            n += 1
    assert n >= 8
    hr.free(); rs.free()


def test_reference_set_in_three_parts():
    """A set cut into parts is aligned as one set in hits mode: this checks that a parted set gives the whole-set
    answer (the same hits and cells as the plain call on the parted set), not any per-part selection."""
    refs = synth.make_refs(90, lo=50, hi=3000)
    reads = synth.make_reads(10, 150, refs, seed=3) + synth.make_reads(3, 600, refs, seed=6)
    eng = swb.Engine(0, workspace_bytes=parts_workspace(refs, 3))
    try:
        rs = eng.load_refset(refs)
        res, kernels = launched_kernels(lambda: rs.align(reads))
        assert len(launches(kernels, r"\bfold_best_kernel\b")) >= 2          # the plain call ran part by part
        res.free(); rs.free()
        for k, ms in ((1, 1), (3, 1), (5, 60)):
            check_hits(eng, refs, reads, k=k, min_score=ms)
        check_hits(eng, refs, reads, k=3, min_score=1, fetch=False)
    finally:
        eng.close()


def _device_count():
    from sparksmithwaterman_b200 import _ffi
    return int(_ffi.load().swb_device_count())


@pytest.mark.parametrize("n_gpus", [1, 2, 4, 8])
def test_multi_gpu_merged_hits(engine, n_gpus):
    if _device_count() < n_gpus:
        pytest.skip(f"needs {n_gpus} GPUs")
    from sparksmithwaterman_b200 import multigpu
    refs = synth.make_refs(70, lo=50, hi=3000)
    reads = synth.make_reads(12, 150, refs, seed=12) + synth.make_reads(2, 600, refs, seed=13) + [b"", b"GGGG"]
    rs = engine.load_refset(refs)
    for k, ms in ((1, 1), (5, 1), (5, 60)):
        one = rs.align(reads, top_k=k, min_score=ms).cache()
        me = multigpu.MultiEngine(list(range(n_gpus)))
        me.load_refset(refs)
        mr = me.align(reads, top_k=k, min_score=ms)
        assert (mr.hits == one.hits).all(), (n_gpus, k, ms)
        assert (mr.best_hits == one.best_hits).all()
        for q in range(len(reads)):
            for score, ref, i, j in mr.hits[q]:
                if ref < 0:
                    continue
                assert mr.pair(int(ref), q, 200) == one.pair(int(ref), q, 200)
        mr.free(); me.close(); one.free()
    rs.free()


def test_comm_allgather_hits_world1(engine):
    """The one-process-per-device form at world 1 (no NCCL): the merged lists are the result's own hits with the
    reference indices moved through global_ids."""
    from sparksmithwaterman_b200 import multigpu
    refs = synth.make_refs(40, lo=50, hi=2500)
    reads = synth.make_reads(10, 150, refs, seed=21) + [b"", b"CCCC"]
    rs = engine.load_refset(refs)
    res = rs.align(reads, top_k=4, min_score=1)
    ids = np.arange(len(refs), dtype=np.int64) * 3 + 7                 # any global numbering
    comm = multigpu.Comm(engine, b"\0" * 128, 0, 1)
    merged = comm.allgather_hits(res, ids)
    exp = res.hits.copy()
    ok = exp[:, :, 1] >= 0
    exp[ok, 1] = ids[exp[ok, 1]]
    assert (merged == exp).all()
    with pytest.raises(swb.SwbError):
        comm.allgather_hits(rs.align(reads), ids)                      # a plain result has no hit lists
    comm.close(); res.free(); rs.free()
