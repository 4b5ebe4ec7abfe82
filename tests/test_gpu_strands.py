"""GPU: the both-strands mode (SWB_F_BOTH_STRANDS).  A both-strands call over reads must equal, array for array, the
plain call over reads + rc(reads) after the index map [2r + s, q] <-> [r, s * n + q] -- which is the same memory, so
scores, cell offsets, cells, beginnings, op lengths and ops compare as whole arrays.  Totals, best hits and hit lists
are recomputed from the plain scores by the oriented rule."""
import ctypes as C
import random

import numpy as np
import pytest

import oracle
import sparksmithwaterman_b200 as swb
from sparksmithwaterman_b200 import synth
from sparksmithwaterman_b200.engine import reverse_complement
from tests.helpers import launched_kernels, launches, parts_workspace, result_ops
from tests.test_hits_host import top_hits_ref

pytestmark = pytest.mark.gpu


def _rand(rnd, n, alphabet="ACGT"):
    return "".join(rnd.choice(alphabet) for _ in range(n))


def _wrap_sum(a):
    return (a.astype(np.int64).sum(axis=1) & 0xFFFFFFFF).astype(np.uint32).view(np.int32)


def check_strands(eng, refs, reads, scores=(5, -3, -4), k=None, min_score=1, **kw):
    """The both-strands call against the plain call over reads + rc(reads)."""
    rs = eng.load_refset(refs)
    try:
        _check(rs, refs, reads, scores, k, min_score, **kw)
    finally:
        rs.free()


def _check(rs, refs, reads, scores, k, min_score, scores_only=False, tie_gt=False, fetch=True, resident=False,
           rc=reverse_complement):
    n, R = len(reads), len(refs)
    plain = rs.align(list(reads) + [rc(q) for q in reads], scores, scores_only=scores_only, tie_gt=tie_gt).cache()
    if resident:
        rd = rs.upload_reads(reads)
        res = rd.align(scores, scores_only, fetch, tie_gt, top_k=k, min_score=min_score, both_strands=True)
    else:
        res = rs.align(reads, scores, scores_only, fetch, tie_gt, top_k=k, min_score=min_score, both_strands=True)
    if not fetch:
        assert not res.lib.swb_result_scores(res.h)        # nothing on the host before the fetch
        res.fetch()
    res.cache()
    assert (res.n_refs, res.n_reads) == (2 * R, n)
    exp = plain.scores.reshape(2 * R, n)
    assert (res.scores == exp).all()
    assert (res.ref_totals == _wrap_sum(exp)).all()
    st_b, st_p = res.stats, plain.stats
    assert st_b["cells"] == st_p["cells"] and st_b["pairs"] == st_p["pairs"]
    best = res.best_hits
    assert (best[:, 0] == exp.max(axis=0)).all() if n and R else True
    if n and R:
        assert (best[:, 1] == exp.argmax(axis=0)).all()          # lowest oriented index on ties: forward first
    if scores_only:
        assert (best[:, 2:] == 0).all()
        if k:
            assert (res.hits[:, :, :2] == top_hits_ref(exp, k, min_score)[:, :, :2]).all()
        return res
    off_p = plain.cell_offsets
    cells_p = plain.cells
    for q in range(n):
        o = int(best[q, 1])
        if best[q, 0] > 0:
            assert tuple(best[q, 2:]) == tuple(cells_p[off_p[o * n + q]]), q
    if k is None:
        assert (res.cell_offsets == off_p).all()
        assert (res.cells == cells_p).all()
        assert (res.beginnings == plain.beginnings).all() and (res.op_lens == plain.op_lens).all()
        assert np.array_equal(result_ops(res, 0, res.total_cells), result_ops(plain, 0, plain.total_cells))
        return res
    hits = res.hits
    assert (hits[:, :, :2] == top_hits_ref(exp, k, min_score)[:, :, :2]).all()
    cnt_b = np.diff(res.cell_offsets).reshape(2 * R, n)
    cnt_p = np.diff(off_p).reshape(2 * R, n)
    mask = np.zeros((2 * R, n), bool)
    off_b = res.cell_offsets
    for q in range(n):
        for score, o, i, j in hits[q]:
            if o < 0:
                continue
            mask[o, q] = True
            p = o * n + q
            assert cnt_b[o, q] == cnt_p[o, q] > 0
            b0, p0, c = int(off_b[p]), int(off_p[p]), int(cnt_p[o, q])
            assert (i, j) == tuple(cells_p[p0])
            assert (res.cells[b0:b0 + c] == cells_p[p0:p0 + c]).all()
            assert (res.beginnings[b0:b0 + c] == plain.beginnings[p0:p0 + c]).all()
            assert (res.op_lens[b0:b0 + c] == plain.op_lens[p0:p0 + c]).all()
            assert np.array_equal(result_ops(res, b0, b0 + c), result_ops(plain, p0, p0 + c))
    assert (cnt_b[~mask] == 0).all()
    return res


@pytest.mark.parametrize("lengths", [(36, 100, 150, 250), (300, 500), (600,)], ids=["K-classes", "long", "wide"])
def test_read_length_classes(engine, lengths):
    refs = synth.make_refs(40, lo=50, hi=2500)
    reads = []
    for m in lengths:
        fw = synth.make_reads(4, m, refs, seed=m)
        reads += fw + [reverse_complement(q) for q in fw[:2]]         # reads that align to the reverse strand
    check_strands(engine, refs, reads)
    check_strands(engine, refs, reads, k=3, min_score=40)


def test_five_symbol_alphabet(engine):
    rnd = random.Random(5)
    refs = [_rand(rnd, n, "ACGTN") for n in (300, 800, 120, 1000)]
    reads = [refs[1][50:200], reverse_complement(refs[3][100:220]).decode(), _rand(rnd, 90, "ACGTN"), refs[0][:60]]
    check_strands(engine, refs, reads)
    check_strands(engine, refs, reads, k=2, min_score=1)


@pytest.mark.parametrize("scores", [(60, -100, -40), (60, -30, -40)], ids=["unbiased-fill-group-trace", "group-trace"])
def test_unbiased_fill_and_group_traceback(engine, scores):
    refs = synth.make_refs(30, lo=50, hi=2000)
    reads = synth.make_reads(8, 150, refs, seed=9)
    check_strands(engine, refs, reads, scores)


@pytest.mark.parametrize("mode", ["scores_only", "tie_gt", "no_fetch"])
def test_flags(engine, mode):
    refs = synth.make_refs(40, lo=50, hi=2500)
    reads = synth.make_reads(8, 150, refs, seed=4) + synth.make_reads(2, 600, refs, seed=5)
    kw = {"scores_only": mode == "scores_only", "tie_gt": mode == "tie_gt", "fetch": mode != "no_fetch"}
    check_strands(engine, refs, reads, **kw)
    check_strands(engine, refs, reads, k=4, min_score=1, **kw)


def test_resident_reads(engine):
    refs = synth.make_refs(30, lo=50, hi=2000)
    reads = synth.make_reads(8, 100, refs, seed=8) + synth.make_reads(2, 600, refs, seed=18)
    check_strands(engine, refs, reads, resident=True)
    check_strands(engine, refs, reads, k=2, resident=True)


def test_reference_set_in_three_parts():
    refs = synth.make_refs(90, lo=50, hi=3000)
    reads = synth.make_reads(8, 150, refs, seed=3) + synth.make_reads(2, 600, refs, seed=6)
    eng = swb.Engine(0, workspace_bytes=parts_workspace(refs, 3))
    try:
        check_strands(eng, refs, reads)
        check_strands(eng, refs, reads, k=3, min_score=1)
        check_strands(eng, refs, reads, fetch=False)
    finally:
        eng.close()


@pytest.mark.parametrize("k,min_score", [(1, 1), (5, 1), (32, 1), (5, 60)])
def test_hits_mode(engine, k, min_score):
    refs = synth.make_refs(60, lo=50, hi=3000)
    fw = synth.make_reads(10, 150, refs, seed=12) + synth.make_reads(2, 600, refs, seed=13)
    reads = fw + [reverse_complement(q) for q in fw[::3]] + [b"", b"GGGG"]
    check_strands(engine, refs, reads, k=k, min_score=min_score)


def test_every_pair_against_the_oracle(engine):
    rnd = random.Random(31)
    refs = [_rand(rnd, n) for n in (400, 250, 700)]
    mixed = "".join(c.lower() if rnd.random() < 0.5 else c for c in reverse_complement(refs[2][200:300]).decode())
    reads = [refs[0][50:170], reverse_complement(refs[1][20:110]).decode(), mixed, _rand(rnd, 60)]
    rs = engine.load_refset(refs)
    res = rs.align(reads, both_strands=True).cache()
    for o in range(2 * len(refs)):
        r, s = res.oriented(o)
        assert (r, s) == (o >> 1, o & 1)
        for q, read in enumerate(reads):
            strand = reverse_complement(read).decode() if s else read
            exp = oracle.align(refs[r], strand)
            assert res.pair(o, q, 50) == (exp.score, exp.cells[:50], exp.sites[:50]), (o, q)
    # the mixed-case read: both materialized strings keep case, the reverse one complemented (a -> t)
    _, _, fwd_sites = res.pair(4, 2, 1)
    _, _, rev_sites = res.pair(5, 2, 1)
    assert any(c.islower() for c in rev_sites[0][2]) and rev_sites[0][2].replace("_", "") in reverse_complement(mixed).decode()
    assert fwd_sites[0][2].replace("_", "") in mixed
    res.free(); rs.free()


def test_reads_planted_on_the_reverse_strand(engine):
    """The user story: a read taken from the reverse strand of reference r reports 2r + 1, with the score of the same
    read planted forward; a palindromic read reports its forward hit."""
    rnd = random.Random(41)
    refs = [_rand(rnd, 2000) for _ in range(12)]
    fwd, rev, sites = [], [], []
    for k in range(12):
        r = (5 * k) % 12
        a = rnd.randrange(0, 1800)
        piece = refs[r][a:a + 150]
        fwd.append(piece); rev.append(reverse_complement(piece).decode()); sites.append(r)
    pal = "ACGT" * 10 + "AATT" + "ACGT" * 10                           # its own reverse complement
    assert reverse_complement(pal).decode() == pal
    refs.append("GGCC" * 20 + pal + "TTGA" * 20)
    rs = engine.load_refset(refs)
    res = rs.align(rev + fwd + [pal], both_strands=True)
    best = res.best_hits
    for k, r in enumerate(sites):
        assert best[k, 1] == 2 * r + 1 and best[12 + k, 1] == 2 * r
        assert best[k, 0] == best[12 + k, 0] == 150 * 5
    assert best[24, 1] == 2 * 12 and best[24, 0] == len(pal) * 5
    res.free(); rs.free()


def _rcx(present):
    """The host rule for a set lacking some symbols: a reverse-strand position whose base or complement is absent from
    the set matches nothing -- here the absent byte 'X'."""
    def f(read):
        out = []
        for c in reverse_complement(read).decode():
            base = reverse_complement(c).decode()                  # the read's own base at this position
            out.append(c if c.upper() in present and base.upper() in present else "X")
        return "".join(out)
    return f


def test_alphabet_edges(engine):
    rnd = random.Random(51)
    refs = [_rand(rnd, n, "ACG") for n in (300, 500, 200)]
    reads = [refs[1][40:160], _rand(rnd, 100, "ACGT"), "TTTT" + refs[0][10:80]]
    check_strands(engine, refs, reads, rc=_rcx("ACG"))
    rs = engine.load_refset(["ACGTX" * 20])
    with pytest.raises(swb.SwbError) as ei:
        rs.align(["ACGT"], both_strands=True)
    assert ei.value.code == -3 and "IUPAC" in str(ei.value)
    rs.free()
    h = C.c_void_p()
    rc = engine.lib.swb_align_pair(engine.h, b"ACGTACGT", 8, b"ACGT", 4, 5, -3, -4, swb._ffi.SWB_F_BOTH_STRANDS, C.byref(h))
    assert rc == -1 and not h.value


def test_kernels_launched(engine):
    refs = synth.make_refs(30, lo=50, hi=2000)
    reads = synth.make_reads(8, 150, refs, seed=2)
    rs = engine.load_refset(refs)
    res_p, kp = launched_kernels(lambda: rs.align(reads))
    res_b, kb = launched_kernels(lambda: rs.align(reads, both_strands=True))
    assert launches(kb, r"\brc_reads_kernel\b") and not launches(kp, r"\brc_reads_kernel\b")
    fill = r"\bfill(_bias)?_kernel<"
    assert {n for n, _ in kb if launches([(n, 0)], fill)} == {n for n, _ in kp if launches([(n, 0)], fill)} != set()
    res_p.free(); res_b.free(); rs.free()


def _device_count():
    return int(swb._ffi.load().swb_device_count())


@pytest.mark.parametrize("n_gpus", [1, 2, 4, 8])
def test_multi_gpu(engine, n_gpus):
    if _device_count() < n_gpus:
        pytest.skip(f"needs {n_gpus} GPUs")
    from sparksmithwaterman_b200 import multigpu
    refs = synth.make_refs(70, lo=50, hi=3000)
    fw = synth.make_reads(10, 150, refs, seed=22) + synth.make_reads(2, 600, refs, seed=23)
    reads = fw + [reverse_complement(q) for q in fw[::2]] + [b"", b"GGGG"]
    rs = engine.load_refset(refs)
    me = multigpu.MultiEngine(list(range(n_gpus)))
    me.load_refset(refs)
    for k, ms in ((None, 1), (1, 1), (5, 60)):
        one = rs.align(reads, top_k=k, min_score=ms, both_strands=True).cache()
        mr = me.align(reads, top_k=k, min_score=ms, both_strands=True)
        assert (mr.best_hits == one.best_hits).all(), (n_gpus, k)
        if k:
            assert (mr.hits == one.hits).all(), (n_gpus, k, ms)
            for q in range(len(reads)):
                for score, o, i, j in mr.hits[q]:
                    if o >= 0:
                        assert mr.pair(int(o), q, 100) == one.pair(int(o), q, 100)
        else:
            for q in range(len(reads)):
                o = int(one.best_hits[q, 1])
                assert mr.pair(o, q, 100) == one.pair(o, q, 100)
        mr.free(); one.free()
    me.close(); rs.free()


def test_comm_allgather_world1(engine):
    from sparksmithwaterman_b200 import multigpu
    refs = synth.make_refs(40, lo=50, hi=2500)
    reads = synth.make_reads(10, 150, refs, seed=21) + [b"", b"CCCC"]
    rs = engine.load_refset(refs)
    res = rs.align(reads, top_k=4, min_score=1, both_strands=True)
    ids = np.arange(len(refs), dtype=np.int64) * 3 + 7
    oids = multigpu.oriented_ids(ids)
    comm = multigpu.Comm(engine, b"\0" * 128, 0, 1)
    exp = res.hits.copy()
    ok = exp[:, :, 1] >= 0
    exp[ok, 1] = oids[exp[ok, 1]]
    assert (comm.allgather_hits(res, oids) == exp).all()
    eb = res.best_hits.copy()
    eb[:, 1] = oids[eb[:, 1]]
    assert (comm.allgather_best(res, oids) == eb).all()
    with pytest.raises(swb.SwbError):
        comm.allgather_best(res, ids)                       # a both-strands result needs the oriented ids
    comm.close(); res.free(); rs.free()
