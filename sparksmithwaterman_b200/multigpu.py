"""Reference-set sharding and the best-hit merge (SURVEY.md 8e).

The pair set is refs x reads and pairs are independent (the reference itself partitions by
reference, Distribution.java:337), so each rank keeps a length-balanced shard of the
references resident in its HBM, aligns ALL reads against it, and only the per-read
best-hit records (score, global ref id, i, j) cross NVLink: one all_gather, then every rank
applies the same deterministic merge.  Works with torch.distributed on nccl (CUDA tensors)
and gloo (CPU tensors; used by the world_size-2 tests)."""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np


def shard_refs(lengths: Sequence[int], rank: int, world: int) -> List[int]:
    """Indices of the references rank `rank` owns: sort by descending length (stable), deal
    in snake order (0..w-1, w-1..0, ...) so no rank always gets the longest of a round;
    return ascending ids.  Every ref belongs to exactly one rank."""
    order = sorted(range(len(lengths)), key=lambda k: -int(lengths[k]))
    mine = []
    for pos, k in enumerate(order):
        rnd, slot = divmod(pos, world)
        if (slot if rnd % 2 == 0 else world - 1 - slot) == rank:
            mine.append(k)
    return sorted(mine)


def merge_best_hits(records: np.ndarray) -> np.ndarray:
    """records: [world, n_reads, 4] int (score, global ref id, i, j).  Winner per read =
    highest score, then lowest global ref id (the running-max-with-first-wins order of a
    single-GPU scan over refs in index order).  Returns [n_reads, 4]."""
    rec = np.asarray(records).astype(np.int64)
    # a record without a reference (ref < 0: a rank whose shard is empty) loses against every real one
    key = rec[:, :, 0] * (1 << 32) - np.where(rec[:, :, 1] < 0, 1 << 31, rec[:, :, 1])
    key = np.where(rec[:, :, 1] < 0, -(1 << 62), key)
    win = key.argmax(axis=0)
    return rec[win, np.arange(rec.shape[1])].astype(np.int32)


def merge_top_hits(records: np.ndarray) -> np.ndarray:
    """records: [world, n_reads, k, 4] int (score, global ref id, i, j), each rank's hit list in hit order (score
    descending, then ref ascending), padded with (0, -1, 0, 0).  Returns the top k of the union per read in the same
    order, [n_reads, k, 4] -- exact, since the global top k lies in the union of the ranks' top k's.  Entries without
    a reference (padding, an empty shard) never win."""
    rec = np.asarray(records).astype(np.int64)
    world, n_reads, k = rec.shape[:3]
    allr = rec.transpose(1, 0, 2, 3).reshape(n_reads, world * k, 4)
    ok = allr[:, :, 1] >= 0
    # sort key: score descending, then ref ascending; padding last
    key = np.where(ok, -(allr[:, :, 0] * (1 << 32)) + allr[:, :, 1], np.iinfo(np.int64).max)
    order = np.argsort(key, axis=1, kind="stable")[:, :k]
    out = np.take_along_axis(allr, order[:, :, None], axis=1)
    out[~np.take_along_axis(ok, order, axis=1)] = (0, -1, 0, 0)
    return out.astype(np.int32)


def merge_all_hits(offsets: Sequence[np.ndarray], lists: Sequence[np.ndarray], min_score: int, margin: int):
    """All-hits merge over ranks.  Rank w's lists: offsets[w] [n_reads + 1] and lists[w] [n_w, 4] (score, global ref
    id, i, j), each read's entries in list order (score descending, then ref ascending), selected against the rank's
    LOCAL best.  The global best of read q is the largest head; its entries with score >= max(min_score, best - margin)
    over all ranks, in list order, are read q's merged list.  Returns (offsets [n_reads + 1] int64, list [n, 4] int32)."""
    n_reads = len(offsets[0]) - 1
    out_off, out = [0], []
    for q in range(n_reads):
        parts = [np.asarray(l, dtype=np.int64).reshape(-1, 4)[o[q]:o[q + 1]] for o, l in zip(offsets, lists)]
        parts = [p for p in parts if len(p)]
        if parts:
            e = np.concatenate(parts)
            bar = max(int(min_score), int(e[:, 0].max()) - int(margin))
            e = e[e[:, 0] >= bar]
            e = e[np.lexsort((e[:, 1], -e[:, 0]))]
            out.append(e)
            out_off.append(out_off[-1] + len(e))
        else:
            out_off.append(out_off[-1])
    lst = np.concatenate(out).astype(np.int32) if out else np.zeros((0, 4), np.int32)
    return np.asarray(out_off, dtype=np.int64), lst.reshape(-1, 4)


def oriented_ids(global_ids: Sequence[int]) -> np.ndarray:
    """A shard's global reference ids -> the oriented ids a both-strands result needs (Comm.allgather_best / _hits):
    entry 2r + s is 2 * global_ids[r] + s."""
    g = np.asarray(global_ids, dtype=np.int64)
    return (2 * g[:, None] + np.arange(2, dtype=np.int64)[None, :]).reshape(-1)


def localize(best_local: np.ndarray, my_ids: Sequence[int]) -> np.ndarray:
    """Shard-local ref indices -> global ref ids."""
    out = np.array(best_local, dtype=np.int32, copy=True)
    ids = np.asarray(my_ids, dtype=np.int32)
    ok = out[:, 1] >= 0
    out[ok, 1] = ids[out[ok, 1]]
    return out


def allgather_best_hits(best_global, group=None):
    """torch tensor [n_reads, 4] int32 (already global ref ids) -> merged [n_reads, 4] on every rank."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    out = [torch.empty_like(best_global) for _ in range(world)]
    dist.all_gather(out, best_global.contiguous(), group=group)
    allb = torch.stack(out).long()
    key = allb[:, :, 0] * (1 << 32) - allb[:, :, 1]
    key = torch.where(allb[:, :, 1] < 0, torch.full_like(key, -(1 << 62)), key)      # empty shard: never the winner
    win = key.argmax(dim=0)
    return allb[win, torch.arange(allb.shape[1], device=allb.device)].to(torch.int32)


# ---------------------------------------------------------------------------------------------------
# The same sharding + merge INSIDE the C ABI (include/swb200.h, "multi-GPU"): what a JVM host binds.
import ctypes as _C

from . import _ffi
from .engine import AlignResult, DEFAULT_SCORES, concat, _entry, _flags, _i64p
from ._ffi import SWB_F_NO_FETCH, SWB_F_SCORES_ONLY, SWB_F_TIE_GT, check  # noqa: F401


class _Lib:
    def __init__(self, lib):
        self.lib = lib


class _ShardRefs:
    """What AlignResult needs from a RefSet: the library and the shard's sequences."""

    def __init__(self, lib, seqs):
        self.eng = _Lib(lib)
        self.seqs = seqs


class MultiEngine:
    """One process, several devices (swb_multi_*): reference set sharded by length-balanced snake deal,
    every device aligns all reads against its shard on its own host thread, best hits merged with one
    ncclAllGather + a merge kernel."""

    def __init__(self, devices, workspace_bytes: int = 0):
        self.lib = _ffi.load()
        arr = (_C.c_int32 * len(devices))(*devices)
        h = _C.c_void_p()
        check(self.lib.swb_multi_create(arr, len(devices), workspace_bytes, _C.byref(h)))
        self.h, self.n = h, len(devices)
        self.seqs = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.swb_multi_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_refset(self, refs):
        data, off, bs = concat(refs)
        check(self.lib.swb_multi_refset_load(self.h, len(bs), data, _i64p(off)))
        self.seqs = bs
        return self

    def shard_refs(self, d: int) -> np.ndarray:
        n = _C.c_int64()
        p = self.lib.swb_multi_shard_refs(self.h, d, _C.byref(n))
        return np.ctypeslib.as_array(p, shape=(n.value,)).copy() if n.value else np.zeros(0, np.int64)

    def ref_location(self, g: int):
        sh, loc = _C.c_int32(), _C.c_int64()
        check(self.lib.swb_multi_ref_location(self.h, g, _C.byref(sh), _C.byref(loc)))
        return sh.value, loc.value

    def align(self, reads, scores=DEFAULT_SCORES, scores_only: bool = False, fetch: bool = True, tie_gt: bool = False,
              *, top_k: int | None = None, min_score: int = 1, both_strands: bool = False, margin: int | None = None):
        """top_k: hits mode (swb_multi_align_hits), every shard in hits mode and the hit lists merged (MultiResult.hits).
        margin: all-hits mode (swb_multi_align_all_hits), the lists merged (MultiResult.hit_offsets / hit_list).
        both_strands: SWB_F_BOTH_STRANDS; merged records and MultiResult.pair use oriented global ids 2 * ref + strand."""
        fn, sel = _entry(self.lib, "swb_multi_align", top_k, min_score, margin)
        data, off, bs = concat(reads)
        flags = _flags(scores_only, fetch, tie_gt, both_strands)
        h = _C.c_void_p()
        check(fn(self.h, len(bs), data, _i64p(off), scores[0], scores[1], scores[2], flags, *sel, _C.byref(h)))
        return MultiResult(self, bs, h, scores_only, both_strands)


class MultiResult:
    def __init__(self, eng: MultiEngine, reads, h, scores_only, both_strands: bool = False):
        self.eng, self.reads, self.h, self.scores_only = eng, reads, h, scores_only
        self.both_strands = both_strands
        self.lib = eng.lib
        self._shards = {}

    def free(self):
        for r in self._shards.values():
            r.h = None
        self._shards = {}
        if getattr(self, "h", None):
            self.lib.swb_multi_result_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    @property
    def best_hits(self) -> np.ndarray:
        n = len(self.reads)
        p = self.lib.swb_multi_result_best_hits(self.h)
        return np.ctypeslib.as_array(p, shape=(n * 4,)).copy().reshape(n, 4) if n else np.zeros((0, 4), np.int32)

    @property
    def hits(self) -> np.ndarray:
        """Hits mode: merged [n_reads, k, 4] (score, GLOBAL ref id, i, j); [n_reads, 0, 4] for a plain result."""
        n, k = len(self.reads), _C.c_int32()
        p = self.lib.swb_multi_result_hits(self.h, _C.byref(k))
        if not p or n == 0:
            return np.zeros((n, k.value, 4), np.int32)
        return np.ctypeslib.as_array(p, shape=(n * k.value * 4,)).copy().reshape(n, k.value, 4)

    @property
    def hit_offsets(self) -> np.ndarray:
        """All-hits mode: merged [n_reads + 1] offsets into hit_list; empty for any other result."""
        n = _C.c_int64()
        p = self.lib.swb_multi_result_hit_offsets(self.h, _C.byref(n))
        return np.ctypeslib.as_array(p, shape=(len(self.reads) + 1,)).copy() if p else np.zeros(0, np.int64)

    @property
    def hit_list(self) -> np.ndarray:
        """All-hits mode: merged [n_hits, 4] (score, GLOBAL ref id, i, j)."""
        n = _C.c_int64()
        self.lib.swb_multi_result_hit_offsets(self.h, _C.byref(n))
        p = self.lib.swb_multi_result_hit_list(self.h)
        if not p or n.value == 0:
            return np.zeros((0, 4), np.int32)
        return np.ctypeslib.as_array(p, shape=(n.value * 4,)).copy().reshape(-1, 4)

    @property
    def stats(self) -> dict:
        out = (_C.c_double * 3)()
        check(self.lib.swb_multi_result_stats(self.h, out, 3))
        return {"wall_ms": out[0], "align_ms": out[1], "allgather_merge_ms": out[2]}

    def shard(self, d: int) -> AlignResult:
        """Shard d's own AlignResult (borrowed): local ref index = position in MultiEngine.shard_refs(d)."""
        if d not in self._shards:
            ids = self.eng.shard_refs(d)
            seqs = [self.eng.seqs[int(g)] for g in ids]
            hp = _C.c_void_p(self.lib.swb_multi_result_shard(self.h, d))
            self._shards[d] = AlignResult(_ShardRefs(self.lib, seqs), self.reads, hp, self.scores_only, owned=False,
                                          both_strands=self.both_strands).cache()
        return self._shards[d]

    def pair(self, global_ref: int, read: int, max_cells=None):
        """A both-strands result takes the oriented global id 2 * ref + strand."""
        if self.both_strands:
            sh, loc = self.eng.ref_location(global_ref >> 1)
            return self.shard(sh).pair(2 * loc + (global_ref & 1), read, max_cells)
        sh, loc = self.eng.ref_location(global_ref)
        return self.shard(sh).pair(loc, read, max_cells)


class Comm:
    """One rank of a multi-process job (swb_comm_*): NCCL communicator over this rank's Engine."""

    @staticmethod
    def unique_id() -> bytes:
        buf = _C.create_string_buffer(128)
        check(_ffi.load().swb_comm_unique_id(buf))
        return buf.raw

    def __init__(self, eng, id128: bytes, rank: int, world: int):
        self.lib = _ffi.load()
        h = _C.c_void_p()
        check(self.lib.swb_comm_create(eng.h, id128, rank, world, _C.byref(h)))
        self.h, self.eng = h, eng

    def close(self):
        if getattr(self, "h", None):
            self.lib.swb_comm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def allgather_best(self, res: AlignResult, global_ids, want_host: bool = True):
        ids = np.ascontiguousarray(global_ids, dtype=np.int64)
        out = np.empty((res.n_reads, 4), dtype=np.int32) if want_host else None
        check(self.lib.swb_comm_allgather_best(self.h, res.h, _i64p(ids), len(ids),
                                               out.ctypes.data_as(_C.POINTER(_C.c_int32)) if want_host else None))
        return out

    def allgather_hits(self, res: AlignResult, global_ids) -> np.ndarray:
        """Hit lists of a hits-mode result of this rank's shard -> merged [n_reads, k, 4] with global ref ids."""
        ids = np.ascontiguousarray(global_ids, dtype=np.int64)
        k = _C.c_int32()
        self.lib.swb_result_hits(res.h, _C.byref(k))
        out = np.empty((res.n_reads, k.value, 4), dtype=np.int32)
        check(self.lib.swb_comm_allgather_hits(self.h, res.h, _i64p(ids), len(ids),
                                               out.ctypes.data_as(_C.POINTER(_C.c_int32)) if out.size else None))
        return out

    def allgather_all_hits(self, res: AlignResult, global_ids):
        """Lists of an all-hits result of this rank's shard -> merged (offsets [n_reads + 1], list [n, 4]) with global
        ref ids."""
        ids = np.ascontiguousarray(global_ids, dtype=np.int64)
        po, pl, n = _C.POINTER(_C.c_int64)(), _C.POINTER(_C.c_int32)(), _C.c_int64()
        check(self.lib.swb_comm_allgather_all_hits(self.h, res.h, _i64p(ids), len(ids), _C.byref(po), _C.byref(pl), _C.byref(n)))
        off = np.ctypeslib.as_array(po, shape=(res.n_reads + 1,)).copy()
        lst = np.ctypeslib.as_array(pl, shape=(n.value * 4,)).copy().reshape(-1, 4) if n.value else np.zeros((0, 4), np.int32)
        return off, lst
