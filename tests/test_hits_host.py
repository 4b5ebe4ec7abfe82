"""CPU: the hits mode's host-side pieces -- the numpy top-k rule every GPU hits test compares against, and the
merge of per-shard hit lists (multigpu.merge_top_hits) at world 2/4/8 and over gloo at world 2."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from sparksmithwaterman_b200 import multigpu


def top_hits_ref(scores: np.ndarray, k: int, min_score: int = 1) -> np.ndarray:
    """scores [n_refs, n_reads] -> [n_reads, k, 4] (score, ref, 0, 0): per read the k best refs with score >=
    min_score, score descending then ref ascending, padded with (0, -1, 0, 0)."""
    scores = np.asarray(scores, dtype=np.int64)
    n_refs, n_reads = scores.shape
    out = np.zeros((n_reads, k, 4), np.int32)
    out[:, :, 1] = -1
    for q in range(n_reads):
        col = scores[:, q]
        order = np.lexsort((np.arange(n_refs), -col))           # score descending, then ref ascending
        order = order[col[order] >= min_score][:k]
        out[q, :len(order), 0] = col[order]
        out[q, :len(order), 1] = order
    return out


def _brute(scores, k, min_score):
    n_refs, n_reads = scores.shape
    out = np.zeros((n_reads, k, 4), np.int32)
    out[:, :, 1] = -1
    for q in range(n_reads):
        cand = sorted((-int(scores[r, q]), r) for r in range(n_refs) if scores[r, q] >= min_score)[:k]
        for h, (s, r) in enumerate(cand):
            out[q, h, :2] = (-s, r)
    return out


def test_top_hits_reference_order_ties_and_cut():
    rng = np.random.default_rng(1)
    for n_refs, n_reads, hi in ((50, 9, 40), (300, 5, 4), (3, 7, 10)):     # wide spread, heavy ties, k > n_refs
        scores = rng.integers(0, hi, size=(n_refs, n_reads))
        for k in (1, 3, 32):
            for ms in (1, hi // 2 + 1):
                got = top_hits_ref(scores, k, ms)
                assert (got == _brute(scores, k, ms)).all(), (n_refs, k, ms)
                assert (np.diff(got[:, :, 0].astype(np.int64), axis=1) <= 0).all()
    # a tie across many refs is cut by reference index, and score 0 is never a hit
    s = np.array([[7], [9], [9], [9], [0], [9]])
    assert top_hits_ref(s, 3)[0, :, :2].tolist() == [[9, 1], [9, 2], [9, 3]]
    assert top_hits_ref(s * 0, 2)[0].tolist() == [[0, -1, 0, 0], [0, -1, 0, 0]]


def _with_cells(hits, cells):
    out = hits.copy()
    for q in range(hits.shape[0]):
        for h in range(hits.shape[1]):
            if hits[q, h, 1] >= 0:
                out[q, h, 2:] = cells[hits[q, h, 1], q]
    return out


def _shard_lists(scores, cells, lengths, k, min_score, world):
    recs = []
    for r in range(world):
        ids = multigpu.shard_refs(lengths, r, world)
        loc = top_hits_ref(scores[ids], k, min_score) if ids else top_hits_ref(np.zeros((0, scores.shape[1])), k, min_score)
        ok = loc[:, :, 1] >= 0
        loc[ok, 1] = np.asarray(ids, np.int32)[loc[ok, 1]] if ids else 0
        recs.append(_with_cells(loc, cells))
    return np.stack(recs)


def test_merge_top_hits_is_shard_invariant():
    rng = np.random.default_rng(2)
    for n_refs, hi in ((64, 30), (5, 6)):                       # 5 refs: empty shards at world 8
        n_reads = 21
        scores = rng.integers(0, hi, size=(n_refs, n_reads))
        scores[:, 0] = 0                                        # a read without hits
        scores[:, 1] = 0
        scores[0, 1] = hi                                       # a read with one hit
        cells = rng.integers(1, 100, size=(n_refs, n_reads, 2))
        lengths = rng.integers(50, 500, size=n_refs)
        for k in (1, 4, 32):
            for ms in (1, hi // 2):
                single = _with_cells(top_hits_ref(scores, k, ms), cells)
                for world in (2, 4, 8):
                    merged = multigpu.merge_top_hits(_shard_lists(scores, cells, lengths, k, ms, world))
                    assert (merged == single).all(), (n_refs, k, ms, world)


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, scores, cells, lengths, k, expect):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mine = _shard_lists(scores, cells, lengths, k, 1, world)[rank]
    out = [torch.empty_like(torch.from_numpy(mine)) for _ in range(world)]
    dist.all_gather(out, torch.from_numpy(mine))
    merged = multigpu.merge_top_hits(torch.stack(out).numpy())
    assert (merged == expect).all(), rank
    dist.destroy_process_group()


def test_allgather_merge_top_hits_world2():
    rng = np.random.default_rng(6)
    n_refs, n_reads, k = 40, 13, 5
    scores = rng.integers(0, 12, size=(n_refs, n_reads))
    cells = rng.integers(1, 200, size=(n_refs, n_reads, 2))
    lengths = rng.integers(50, 3000, size=n_refs)
    expect = _with_cells(top_hits_ref(scores, k, 1), cells)
    mp.spawn(_worker, args=(2, _free_port(), scores, cells, lengths, k, expect), nprocs=2, join=True)
