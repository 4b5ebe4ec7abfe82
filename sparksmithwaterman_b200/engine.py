"""Python host layer over the C ABI: Engine (context), RefSet (HBM-resident packed
references), AlignResult (scores, max-cell lists, alignments)."""
from __future__ import annotations

import ctypes as C
from typing import List, Sequence, Tuple

import numpy as np

from . import _ffi
from ._ffi import SWB_F_BOTH_STRANDS, SWB_F_NO_FETCH, SWB_F_SCORES_ONLY, SWB_F_TIE_GT, check

DEFAULT_SCORES = (5, -3, -4)          # Distribution.java:36 of the reference: match, mismatch, gap


def _b(s) -> bytes:
    return bytes(s) if isinstance(s, (bytes, bytearray, memoryview)) else s.encode("latin-1")


def concat(seqs: Sequence) -> Tuple[bytes, np.ndarray, List[bytes]]:
    bs = [_b(s) for s in seqs]
    off = np.zeros(len(bs) + 1, dtype=np.int64)
    if bs:
        np.cumsum([len(x) for x in bs], out=off[1:])
    return b"".join(bs), off, bs


def _i64p(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_int64))


# IUPAC DNA complement (the library's table for SWB_F_BOTH_STRANDS): an involution that keeps case; S, W and N map to
# themselves, and any other byte stays itself
_COMP_FROM, _COMP_TO = b"ACGTRYKMBVDHSWN", b"TGCAYRMKVBHDSWN"
COMPLEMENT = bytes.maketrans(_COMP_FROM + _COMP_FROM.lower(), _COMP_TO + _COMP_TO.lower())


def reverse_complement(seq) -> bytes:
    """The reverse complement of a read, as a both-strands call aligns it (o = 2r + 1), case kept."""
    return _b(seq).translate(COMPLEMENT)[::-1]


def _mode(top_k, margin) -> str:
    """Which entry a call takes: "plain", "hits" (top_k) or "all_hits" (margin); both at once is a ValueError."""
    if top_k is not None and margin is not None:
        raise ValueError("top_k (hits mode) and margin (all-hits mode) select different modes: pass one of them")
    return "plain" if top_k is None and margin is None else ("hits" if margin is None else "all_hits")


def _entry(lib, name: str, top_k, min_score, margin):
    """The C entry point of a call's mode (_mode): `name`, name + "_hits" or name + "_all_hits", and the selection
    arguments it takes after the flags."""
    mode = _mode(top_k, margin)
    if mode == "plain":
        return getattr(lib, name), ()
    if mode == "hits":
        return getattr(lib, name + "_hits"), (top_k, min_score)
    return getattr(lib, name + "_all_hits"), (min_score, margin)


def _flags(scores_only: bool, fetch: bool, tie_gt: bool, both_strands: bool) -> int:
    return ((SWB_F_SCORES_ONLY if scores_only else 0) | (0 if fetch else SWB_F_NO_FETCH) | (SWB_F_TIE_GT if tie_gt else 0)
            | (SWB_F_BOTH_STRANDS if both_strands else 0))


class Engine:
    """One CUDA device.  Raises if no device / library is present (no CPU fallback)."""

    def __init__(self, device: int = 0, workspace_bytes: int = 0):
        self.lib = _ffi.load()
        h = C.c_void_p()
        check(self.lib.swb_create(device, workspace_bytes, C.byref(h)))
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.swb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream_ptr(self) -> int:
        """cudaStream_t the engine launches on (for external event timing)."""
        p = C.c_void_p()
        check(self.lib.swb_get_stream(self.h, C.byref(p)))
        return int(p.value or 0)

    def load_refset(self, refs: Sequence) -> "RefSet":
        return RefSet(self, refs)

    def align_pair(self, ref, read, scores=DEFAULT_SCORES, scores_only: bool = False, tie_gt: bool = False) -> "AlignResult":
        """ONE pair through the context's submission queue (swb_align_pair): what the unchanged driver's per-pair
        `OptAlignments.call` becomes.  Safe to call from many threads; concurrent calls are coalesced natively."""
        rb, qb = _b(ref), _b(read)
        flags = (SWB_F_SCORES_ONLY if scores_only else 0) | (SWB_F_TIE_GT if tie_gt else 0)
        h = C.c_void_p()
        check(self.lib.swb_align_pair(self.h, rb, len(rb), qb, len(qb), scores[0], scores[1], scores[2], flags, C.byref(h)))
        return AlignResult(_PairRefs(self, rb), [qb], h, scores_only)

    def queue_stats(self) -> dict:
        out = (C.c_int64 * 3)()
        check(self.lib.swb_queue_stats(self.h, out, 3))
        return {"calls": int(out[0]), "batches": int(out[1]), "largest_batch": int(out[2])}

    def microbench(self, iters: int = 4000) -> dict:
        import json
        buf = C.create_string_buffer(1 << 15)
        check(self.lib.swb_microbench_json(self.device, iters, buf, len(buf)))
        return json.loads(buf.value.decode())


class _PairRefs:
    """What an AlignResult needs from its reference set, for the 1 x 1 results of Engine.align_pair."""

    def __init__(self, eng: Engine, ref: bytes):
        self.eng, self.seqs, self.n = eng, [ref], 1


class RefSet:
    def __init__(self, eng: Engine, refs: Sequence, keep_host: bool = True):
        self.eng = eng
        data, off, bs = concat(refs)
        h = C.c_void_p()
        check(eng.lib.swb_refset_load(eng.h, len(bs), data, _i64p(off), C.byref(h)))
        self.h = h
        self.seqs = bs if keep_host else None
        self.n = len(bs)
        self.total_bases = int(off[-1])

    def free(self):
        if getattr(self, "h", None):
            self.eng.lib.swb_refset_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def upload_reads(self, reads: Sequence) -> "Reads":
        return Reads(self, reads)

    def align(self, reads, scores=DEFAULT_SCORES, scores_only: bool = False, fetch: bool = True,
              tie_gt: bool = False, *, top_k: int | None = None, min_score: int = 1,
              both_strands: bool = False, margin: int | None = None) -> "AlignResult":
        """Host-buffer path (swb_align): H2D of the reads, compute, D2H of the results.
        tie_gt: DistributedSW's strict-'>' tie rule in the traceback (SWB_F_TIE_GT).
        top_k: hits mode (swb_align_hits) -- every pair is scored, but only each read's top_k best pairs with
        score >= min_score are traced (AlignResult.hits / read_hits).
        margin: all-hits mode (swb_align_all_hits) -- every pair with score >= min_score and score >= the read's best
        score - margin is listed and traced, with no cap on the count (AlignResult.hit_offsets / hit_list / read_hits).
        margin=0 gives each read's co-optimal references.  Passing both top_k and margin is a ValueError.
        both_strands: every read and its reverse complement (SWB_F_BOTH_STRANDS); the result has 2 * n_refs oriented
        references, o = 2r (read as given) and o = 2r + 1 (reverse complement) -- AlignResult.oriented."""
        if isinstance(reads, Reads):
            return reads.align(scores, scores_only, fetch, tie_gt, top_k=top_k, min_score=min_score, both_strands=both_strands,
                               margin=margin)
        fn, sel = _entry(self.eng.lib, "swb_align", top_k, min_score, margin)
        data, off, bs = concat(reads)
        flags = _flags(scores_only, fetch, tie_gt, both_strands)
        h = C.c_void_p()
        check(fn(self.eng.h, self.h, len(bs), data, _i64p(off), scores[0], scores[1], scores[2], flags, *sel, C.byref(h)))
        return AlignResult(self, bs, h, scores_only, both_strands=both_strands)


class Reads:
    """A read batch encoded and resident in HBM (swb_reads_upload)."""

    def __init__(self, rs: RefSet, reads: Sequence):
        self.rs = rs
        data, off, bs = concat(reads)
        h = C.c_void_p()
        check(rs.eng.lib.swb_reads_upload(rs.eng.h, rs.h, len(bs), data, _i64p(off), C.byref(h)))
        self.h = h
        self.seqs = bs
        self.nbytes = len(data) + off.nbytes

    def free(self):
        if getattr(self, "h", None):
            self.rs.eng.lib.swb_reads_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def align(self, scores=DEFAULT_SCORES, scores_only: bool = False, fetch: bool = True,
              tie_gt: bool = False, *, top_k: int | None = None, min_score: int = 1,
              both_strands: bool = False, margin: int | None = None) -> "AlignResult":
        fn, sel = _entry(self.rs.eng.lib, "swb_align_resident", top_k, min_score, margin)
        flags = _flags(scores_only, fetch, tie_gt, both_strands)
        h = C.c_void_p()
        check(fn(self.rs.eng.h, self.rs.h, self.h, scores[0], scores[1], scores[2], flags, *sel, C.byref(h)))
        return AlignResult(self.rs, self.seqs, h, scores_only, both_strands=both_strands)


STAT_NAMES = ("h2d_ms", "fill_ms", "locate_ms", "trace_ms", "d2h_ms", "device_ms", "cells", "pairs",
              "max_cells", "launches", "checkpoint_bytes", "batches", "select_ms")


class AlignResult:
    def __init__(self, rs: RefSet, reads: List[bytes], h, scores_only: bool, owned: bool = True, both_strands: bool = False):
        self.rs, self.reads, self.h, self.scores_only = rs, reads, h, scores_only
        self.both_strands = both_strands        # n_refs counts oriented references o = 2r + strand
        self._owned = owned                     # False: a shard of a MultiResult, freed with it
        self.lib = rs.eng.lib
        self.n_refs = int(self.lib.swb_result_n_refs(h))
        self.n_reads = int(self.lib.swb_result_n_reads(h))

    def free(self):
        if getattr(self, "h", None):
            if self._owned:
                self.lib.swb_result_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def fetch(self):
        check(self.lib.swb_result_fetch(self.h))
        return self

    def _arr(self, ptr, n, dtype):
        if n == 0 or not ptr:
            return np.zeros(0, dtype=dtype)
        return np.ctypeslib.as_array(ptr, shape=(n,)).copy()

    @property
    def stats(self) -> dict:
        out = (C.c_double * len(STAT_NAMES))()
        check(self.lib.swb_result_stats(self.h, out, len(STAT_NAMES)))
        return dict(zip(STAT_NAMES, list(out)))

    @property
    def scores(self) -> np.ndarray:
        """[n_refs, n_reads] int32 maximum scores."""
        a = self._arr(self.lib.swb_result_scores(self.h), self.n_refs * self.n_reads, np.int32)
        return a.reshape(self.n_refs, self.n_reads)

    @property
    def ref_totals(self) -> np.ndarray:
        return self._arr(self.lib.swb_result_ref_totals(self.h), self.n_refs, np.int32)

    @property
    def best_hits(self) -> np.ndarray:
        return self._arr(self.lib.swb_result_best_hits(self.h), self.n_reads * 4, np.int32).reshape(self.n_reads, 4)

    @property
    def hits(self) -> np.ndarray:
        """Hits mode: [n_reads, k, 4] int32 (score, ref, i, j), each read's k best pairs with score >= min_score,
        score descending then ref ascending, padded with (0, -1, 0, 0).  [n_reads, 0, 4] for a plain result."""
        k = C.c_int32()
        p = self.lib.swb_result_hits(self.h, C.byref(k))
        if not p:                                 # a plain result, or not fetched yet
            return np.zeros((self.n_reads, 0, 4), np.int32)
        return self._arr(p, self.n_reads * k.value * 4, np.int32).reshape(self.n_reads, k.value, 4)

    @property
    def hit_offsets(self) -> np.ndarray:
        """All-hits mode: [n_reads + 1] int64, read q's entries are hit_list[hit_offsets[q]:hit_offsets[q + 1]].
        Empty for any other result (or before the fetch)."""
        n = C.c_int64()
        p = self.lib.swb_result_hit_offsets(self.h, C.byref(n))
        return self._arr(p, self.n_reads + 1, np.int64) if p else np.zeros(0, np.int64)

    @property
    def hit_list(self) -> np.ndarray:
        """All-hits mode: [n_hits, 4] int32 (score, ref, i, j), per read score descending then ref ascending."""
        n = C.c_int64()
        self.lib.swb_result_hit_offsets(self.h, C.byref(n))
        return self._arr(self.lib.swb_result_hit_list(self.h), n.value * 4, np.int32).reshape(-1, 4)

    def _read_entries(self, read: int) -> np.ndarray:
        off = self.hit_offsets
        if len(off):
            return self.hit_list[off[read]:off[read + 1]]
        return self.hits[read]

    def read_hits(self, read: int):
        """Hits or all-hits mode: [(ref, score, cells, sites)] of read `read`'s hits in hit order; cells / sites as
        pair().  A both-strands result gives [(ref, strand, score, cells, sites)], ref the reference's own index."""
        out = []
        for score, ref, _, _ in self._read_entries(read):
            if ref < 0:
                break
            _, cells, sites = self.pair(int(ref), read)
            if self.both_strands:
                out.append(self.oriented(int(ref)) + (int(score), cells, sites))
            else:
                out.append((int(ref), int(score), cells, sites))
        return out

    def oriented(self, o: int) -> Tuple[int, int]:
        """Oriented reference o of a both-strands result -> (reference index, strand): 0 = read as given, 1 = its
        reverse complement."""
        return o >> 1, o & 1

    @property
    def cell_offsets(self) -> np.ndarray:
        return self._arr(self.lib.swb_result_cell_offsets(self.h), self.n_refs * self.n_reads + 1, np.int64)

    @property
    def total_cells(self) -> int:
        return int(self.lib.swb_result_total_cells(self.h))

    @property
    def cells(self) -> np.ndarray:
        return self._arr(self.lib.swb_result_cells(self.h), self.total_cells * 2, np.int32).reshape(-1, 2)

    @property
    def beginnings(self) -> np.ndarray:
        return self._arr(self.lib.swb_result_beginnings(self.h), self.total_cells, np.int32)

    @property
    def op_lens(self) -> np.ndarray:
        return self._arr(self.lib.swb_result_op_lens(self.h), self.total_cells, np.int32)

    def device_array(self, which: int, shape, typestr: str = "<i4"):
        """Zero-copy view of an HBM-resident output (0 scores, 1 ref_totals, 2 best_hits) as an
        object with __cuda_array_interface__ (torch.as_tensor(..., device="cuda") wraps it)."""
        ptr = C.c_void_p(); n = C.c_int64()
        check(self.lib.swb_result_device_ptr(self.h, which, C.byref(ptr), C.byref(n)))

        class _View:
            pass
        v = _View()
        v.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr.value or 0), False),
                                      "version": 2, "strides": None}
        v._keepalive = self
        return v

    def pair_index(self, ref: int, read: int) -> int:
        return ref * self.n_reads + read

    def pair_cell_count(self, ref: int, read: int) -> int:
        return int(self.lib.swb_result_pair_cell_count(self.h, self.pair_index(ref, read)))

    def ops(self, cell: int) -> np.ndarray:
        n = int(self.op_lens[cell]) if not hasattr(self, "_oplens") else int(self._oplens[cell])
        buf = (C.c_uint8 * max(n, 1))()
        check(self.lib.swb_result_ops(self.h, cell, buf, n))
        return np.frombuffer(buf, dtype=np.uint8, count=n).copy()

    def materialize(self, cell: int, ref: bytes, read: bytes, op_len: int) -> Tuple[str, str]:
        a = C.create_string_buffer(op_len + 1)
        b = C.create_string_buffer(op_len + 1)
        check(self.lib.swb_result_materialize(self.h, cell, ref, len(ref), read, len(read), a, b, op_len + 1))
        return a.value.decode("latin-1"), b.value.decode("latin-1")

    def pair(self, ref: int, read: int, max_cells: int | None = None):
        """(score, [(i, j)], [(beginning, ref_aln, read_aln)]) of one pair, in the reference's
        list order -- the value OptAlignments.call returns (SmithWaterman.java:91).  A both-strands result takes the
        oriented reference o as `ref`; for odd o the read string is the reverse complement of the read."""
        p = self.pair_index(ref, read)
        score = int(self.scores[ref, read]) if not hasattr(self, "_scores") else int(self._scores[ref, read])
        cnt = int(self.lib.swb_result_pair_cell_count(self.h, p))
        k_max = cnt if max_cells is None else min(cnt, max_cells)
        cells, sites = [], []
        i, j, bg, ln = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        base = int(self._celloff[p]) if hasattr(self, "_celloff") else int(self.cell_offsets[p])
        for k in range(k_max):
            check(self.lib.swb_result_pair_cell(self.h, p, k, C.byref(i), C.byref(j), C.byref(bg), C.byref(ln)))
            cells.append((i.value, j.value))
            if score == 0:
                sites.append((0, "", ""))
            else:
                seq = self.rs.seqs[ref >> 1] if self.both_strands else self.rs.seqs[ref]
                ra, qa = self.materialize(base + k, seq, self.reads[read], ln.value)
                sites.append((bg.value, ra, qa))
        return score, cells, sites

    def cache(self):
        """Pull the flat arrays once (avoids re-copying in loops over pairs)."""
        self._scores = self.scores
        self._celloff = self.cell_offsets
        self._oplens = self.op_lens
        return self
