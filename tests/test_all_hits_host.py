"""CPU: the all-hits mode's host-side pieces -- the numpy rule every GPU all-hits test compares against, and the merge
of per-shard lists (multigpu.merge_all_hits) at world 2/4/8 over random shard splits, with oriented ids."""
import ctypes as C

import numpy as np
import pytest

from sparksmithwaterman_b200 import _ffi, multigpu
from sparksmithwaterman_b200.engine import _mode
from tests.test_hits_host import top_hits_ref


def all_hits_ref(scores: np.ndarray, min_score: int = 1, margin: int = 0):
    """scores [n_refs, n_reads] -> (offsets [n_reads + 1], list [n, 4] (score, ref, 0, 0)): per read every ref with
    score >= min_score and score >= best - margin (best over the read's refs, in 64 bits), score descending then ref
    ascending."""
    scores = np.asarray(scores, dtype=np.int64)
    n_refs, n_reads = scores.shape
    off, out = [0], []
    for q in range(n_reads):
        col = scores[:, q]
        best = int(col.max()) if n_refs else 0
        bar = max(int(min_score), best - int(margin))
        order = np.lexsort((np.arange(n_refs), -col))
        order = order[col[order] >= bar]
        e = np.zeros((len(order), 4), np.int64)
        e[:, 0], e[:, 1] = col[order], order
        out.append(e)
        off.append(off[-1] + len(order))
    lst = np.concatenate(out) if out else np.zeros((0, 4), np.int64)
    return np.asarray(off, np.int64), lst.astype(np.int32).reshape(-1, 4)


def _brute(scores, min_score, margin):
    n_refs, n_reads = scores.shape
    off, out = [0], []
    for q in range(n_reads):
        best = max([int(scores[r, q]) for r in range(n_refs)] + [0])
        cand = sorted((-int(scores[r, q]), r) for r in range(n_refs)
                      if scores[r, q] >= min_score and scores[r, q] >= best - margin)
        out += [(-s, r, 0, 0) for s, r in cand]
        off.append(len(out))
    return np.asarray(off, np.int64), np.asarray(out, np.int32).reshape(-1, 4)


@pytest.mark.parametrize("seed", range(6))
def test_numpy_rule_matches_brute_force(seed):
    rng = np.random.default_rng(seed)
    sc = rng.integers(0, 12, size=(rng.integers(1, 40), rng.integers(1, 15)))
    sc[:, 0] = 0                                                         # a read with no hits
    for ms, margin in ((1, 0), (1, 3), (5, 0), (5, 2**31 - 1), (12, 0), (3, 100)):
        o, l = all_hits_ref(sc, ms, margin)
        ob, lb = _brute(sc, ms, margin)
        assert (o == ob).all() and (l == lb).all()
        assert o[1] == 0


def test_hits_mode_is_a_prefix_of_the_list():
    rng = np.random.default_rng(7)
    sc = rng.integers(0, 9, size=(60, 20))
    for ms in (1, 4):
        o, l = all_hits_ref(sc, ms, 2**31 - 1)
        for k in (1, 5, 32):
            top = top_hits_ref(sc, k, ms)
            for q in range(sc.shape[1]):
                mine = l[o[q]:o[q + 1]]
                n = int((top[q, :, 1] >= 0).sum())
                assert (top[q, :n, :2] == mine[:n, :2]).all()
                assert n == min(k, len(mine))


def test_margin_0_is_the_co_optimal_set_and_a_large_margin_is_a_threshold():
    rng = np.random.default_rng(3)
    sc = rng.integers(0, 6, size=(50, 12))
    o, l = all_hits_ref(sc, 1, 0)
    for q in range(12):
        best = sc[:, q].max()
        assert sorted(l[o[q]:o[q + 1], 1]) == (list(np.nonzero(sc[:, q] == best)[0]) if best >= 1 else [])
    o, l = all_hits_ref(sc, 3, 2**31 - 1)                               # best - INT32_MAX does not wrap
    for q in range(12):
        assert sorted(l[o[q]:o[q + 1], 1]) == list(np.nonzero(sc[:, q] >= 3)[0])


def _shard_lists(sc, shards, min_score, margin, oriented=False):
    """Each rank selects against its LOCAL best (as a shard's swb_align_all_hits does), then localizes to global ids."""
    offs, lists = [], []
    for ids in shards:
        ids = np.asarray(ids, dtype=np.int64)
        rows = multigpu.oriented_ids(ids) if oriented else ids
        o, l = all_hits_ref(sc[rows] if len(rows) else np.zeros((0, sc.shape[1]), np.int64), min_score, margin)
        l = l.astype(np.int64)
        if len(l):
            l[:, 1] = rows[l[:, 1]]
        offs.append(o)
        lists.append(l.astype(np.int32))
    return offs, lists


@pytest.mark.parametrize("world", [2, 4, 8])
def test_merge_equals_one_rank_over_random_splits(world):
    rng = np.random.default_rng(world)
    n_refs, n_reads = 70, 16
    sc = rng.integers(0, 10, size=(n_refs, n_reads))
    sc[:, 3] = 0                                                         # a read with no hits anywhere
    sc[:, 5] = 4                                                         # ties that span every shard
    for trial in range(4):
        owner = rng.integers(0, world, size=n_refs)
        owner[owner == world - 1] = 0                                    # the last rank holds an empty shard
        shards = [np.nonzero(owner == w)[0] for w in range(world)]
        # read 7: one shard's local best lies below the global best minus the margin
        sc[:, 7] = 1
        sc[shards[0][0], 7] = 9
        for ms, margin in ((1, 0), (1, 2), (4, 1), (2, 2**31 - 1), (9, 0)):
            offs, lists = _shard_lists(sc, shards, ms, margin)
            got_o, got_l = multigpu.merge_all_hits(offs, lists, ms, margin)
            exp_o, exp_l = all_hits_ref(sc, ms, margin)
            assert (got_o == exp_o).all() and (got_l == exp_l).all(), (world, trial, ms, margin)
            assert got_o[4] - got_o[3] == 0
            if margin < 8 and ms == 1:
                assert got_o[8] - got_o[7] == 1                          # only the global best survives


@pytest.mark.parametrize("world", [2, 4, 8])
def test_merge_with_oriented_ids(world):
    """Both strands: each rank's lists hold oriented global ids 2 * ref + strand; the merge orders them like one
    context over the 2R oriented references."""
    rng = np.random.default_rng(10 + world)
    n_refs, n_reads = 40, 9
    sc = rng.integers(0, 8, size=(2 * n_refs, n_reads))                 # row o = 2r + s
    sc[0::2, 2] = sc[1::2, 2]                                            # both strands tie on read 2
    shards = [multigpu.shard_refs(np.ones(n_refs), w, world) for w in range(world)]
    for ms, margin in ((1, 0), (2, 3), (1, 2**31 - 1)):
        offs, lists = _shard_lists(sc, shards, ms, margin, oriented=True)
        got_o, got_l = multigpu.merge_all_hits(offs, lists, ms, margin)
        exp_o, exp_l = all_hits_ref(sc, ms, margin)
        assert (got_o == exp_o).all() and (got_l == exp_l).all()


def test_top_k_and_margin_are_exclusive():
    assert _mode(None, None) == "plain" and _mode(3, None) == "hits" and _mode(None, 0) == "all_hits"
    with pytest.raises(ValueError):
        _mode(3, 0)


def test_all_hits_signatures():
    s = _ffi.SIGNATURES
    assert s["swb_align_all_hits"][1][-3:] == [C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
    assert s["swb_result_hit_offsets"][0] is not None and s["swb_result_hit_list"][0] is not None
    for name in ("swb_multi_align_all_hits", "swb_multi_result_hit_offsets", "swb_multi_result_hit_list",
                 "swb_comm_allgather_all_hits", "swb_align_resident_all_hits"):
        assert name in s
