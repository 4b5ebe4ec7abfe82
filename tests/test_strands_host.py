"""CPU: the both-strands mode's host-side pieces -- the complement table and reverse_complement, the oriented index
helpers, the best-hit and top-k merges over oriented global ids, and the flag constant across the bindings."""
import os
import re

import numpy as np

from sparksmithwaterman_b200 import _ffi, multigpu
from sparksmithwaterman_b200.engine import COMPLEMENT, AlignResult, reverse_complement
from tests.test_hits_host import top_hits_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
IUPAC = b"ACGTRYKMBVDHSWN"


def test_complement_is_an_involution_that_keeps_case():
    table = bytes(range(256))
    once = table.translate(COMPLEMENT)
    assert once.translate(COMPLEMENT) == table
    for c in IUPAC:
        up, lo = bytes([c]), bytes([c]).lower()
        assert up.translate(COMPLEMENT).isupper() and lo.translate(COMPLEMENT) == up.translate(COMPLEMENT).lower()
    assert b"ACGTRYKMBVDHSWN".translate(COMPLEMENT) == b"TGCAYRMKVBHDSWN"
    for c in b"XU-*. 0z":                                   # outside the table: the byte stays itself
        assert bytes([c]).translate(COMPLEMENT) == bytes([c])


def test_reverse_complement_of_mixed_case_and_iupac():
    assert reverse_complement("ACGTacgt") == b"acgtACGT"
    assert reverse_complement(b"AAcGtN") == b"NaCgTT"
    assert reverse_complement("RYKMBVDHSWN") == b"NWSDHBVKMRY"
    assert reverse_complement("gattacaX") == b"Xtgtaatc"
    assert reverse_complement("") == b""
    rng = np.random.default_rng(1)
    for _ in range(20):
        s = bytes(rng.choice(list(IUPAC + IUPAC.lower()), size=int(rng.integers(0, 80))))
        assert reverse_complement(reverse_complement(s)) == s
        assert len(reverse_complement(s)) == len(s)


def test_oriented_index_helpers():
    res = AlignResult.__new__(AlignResult)                      # the helper needs no result handle
    for o in range(12):
        r, s = res.oriented(o)
        assert (r, s) == (o // 2, o % 2) and 2 * r + s == o
    ids = np.array([4, 9, 17], dtype=np.int64)
    assert multigpu.oriented_ids(ids).tolist() == [8, 9, 18, 19, 34, 35]
    assert multigpu.oriented_ids(np.zeros(0, np.int64)).tolist() == []


def _shard_records(scores, world, k):
    """Per rank: the oriented best hit and top k of its shard, localized to oriented global ids."""
    n_refs = scores.shape[0] // 2
    lengths = np.random.default_rng(7).integers(50, 5000, n_refs)
    best, hits = [], []
    for rank in range(world):
        mine = multigpu.shard_refs(lengths, rank, world)
        oids = multigpu.oriented_ids(mine)
        local = scores[oids] if len(oids) else np.zeros((0, scores.shape[1]), scores.dtype)
        b = np.zeros((scores.shape[1], 4), np.int32)
        b[:, 1] = -1
        if len(oids):
            b[:, 0] = local.max(axis=0)
            b[:, 1] = local.argmax(axis=0)
        best.append(multigpu.localize(b, oids))
        h = top_hits_ref(local, k) if len(oids) else np.tile(np.array([0, -1, 0, 0], np.int32), (scores.shape[1], k, 1))
        ok = h[:, :, 1] >= 0
        h[ok, 1] = oids[h[ok, 1]]
        hits.append(h)
    return np.stack(best), np.stack(hits)


def test_merges_over_oriented_global_ids_are_shard_invariant():
    rng = np.random.default_rng(3)
    n_refs, n_reads = 23, 40
    scores = rng.integers(0, 12, (2 * n_refs, n_reads)).astype(np.int32)       # many ties, across strands too
    scores[:, 5] = 7                                                              # a read tied everywhere: o = 0 wins
    exp_best = np.stack([scores.max(axis=0), scores.argmax(axis=0)], axis=1)
    for k in (1, 5):
        exp_hits = top_hits_ref(scores, k)
        for world in (2, 4, 8):
            best, hits = _shard_records(scores, world, k)
            merged = multigpu.merge_best_hits(best)
            assert (merged[:, :2] == exp_best).all(), world
            assert (multigpu.merge_top_hits(hits)[:, :, :2] == exp_hits[:, :, :2]).all(), (world, k)
    assert exp_best[5, 1] == 0


def test_flag_constant_agrees_across_bindings():
    with open(os.path.join(ROOT, "include", "swb200.h")) as f:
        m = re.search(r"#define\s+SWB_F_BOTH_STRANDS\s+(\d+)u", f.read())
    assert m and int(m.group(1)) == _ffi.SWB_F_BOTH_STRANDS == 8
    for path in ("java/sw/NativeSW.java", "java/ffm/sw/NativeSW.java"):
        with open(os.path.join(ROOT, path)) as f:
            m = re.search(r"F_BOTH_STRANDS\s*=\s*(\d+)", f.read())
        assert m and int(m.group(1)) == 8, path
