"""oracle -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

ctypes front-end of the plain-C oracle (oracle/sw_oracle.c) and the CPU baseline
harness (oracle/cpu_baseline.c).  Importable only from tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs; the
product package sparksmithwaterman_b200 never imports it.

Parity status: the Java reference cannot run here (no JVM) and ships no golden
vectors, so this oracle is "parity unpinned" by reference outputs; it is pinned by
the hand-derivable known answers of SURVEY.md section 8c (tests/golden/kat.json)
and by agreement with the independent twin oracle/sw_twin.py.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass
from typing import List, Sequence, Tuple

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libsw_oracle.so")
_lib = None


class _Result(C.Structure):
    _fields_ = [
        ("score", C.c_int32),
        ("n_cells", C.c_int64),
        ("cells", C.POINTER(C.c_int32)),
        ("beginning", C.POINTER(C.c_int32)),
        ("aln_off", C.POINTER(C.c_int64)),
        ("ref_aln", C.POINTER(C.c_char)),
        ("read_aln", C.POINTER(C.c_char)),
    ]


def build(force: bool = False) -> str:
    """Compile the oracle with gcc (no-op when up to date)."""
    srcs = [os.path.join(_HERE, f) for f in ("sw_oracle.c", "cpu_baseline.c", "sw_oracle.h")]
    if not force and os.path.exists(_LIB_PATH):
        if all(os.path.getmtime(s) <= os.path.getmtime(_LIB_PATH) for s in srcs):
            return _LIB_PATH
    subprocess.check_call(["make", "-s", "-C", _HERE])
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        sig = [C.c_char_p, C.c_int64, C.c_char_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
               C.POINTER(_Result)]
        for name in ("sw_oracle_align", "sw_oracle_align_lowmem", "sw_oracle_align_gt"):
            getattr(L, name).argtypes = sig
            getattr(L, name).restype = C.c_int
        L.sw_oracle_score.argtypes = [C.c_char_p, C.c_int64, C.c_char_p, C.c_int64, C.c_int32,
                                      C.c_int32, C.c_int32, C.POINTER(C.c_int32),
                                      C.POINTER(C.c_int64)]
        L.sw_oracle_score.restype = C.c_int
        L.sw_oracle_free.argtypes = [C.POINTER(_Result)]
        L.sw_oracle_free.restype = None
        L.sw_oracle_digest.argtypes = [C.POINTER(_Result)]
        L.sw_oracle_digest.restype = C.c_uint64
        L.sw_cpu_baseline_run.argtypes = [
            C.c_char_p, C.POINTER(C.c_int64), C.c_int64,
            C.c_char_p, C.POINTER(C.c_int64), C.c_int64,
            C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
            C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_uint64)]
        L.sw_cpu_baseline_run.restype = C.c_double
        _lib = L
    return _lib


@dataclass
class PairResult:
    score: int
    cells: List[Tuple[int, int]]                 # (i, j), 1-based, reference list order
    sites: List[Tuple[int, str, str]]            # (beginning, ref_aln, read_aln)
    digest: int


def _b(s) -> bytes:
    return s if isinstance(s, (bytes, bytearray)) else s.encode("latin-1")


def align(ref, read, match: int = 5, mismatch: int = -3, gap: int = -4,
          lowmem: bool = False, max_cells: int | None = None, tie_gt: bool = False) -> PairResult:
    """One pair through the C oracle (SmithWaterman.java:62-92; tie_gt: DistributedSW.java semantics)."""
    L = lib()
    ref_b, read_b = _b(ref), _b(read)
    r = _Result()
    fn = L.sw_oracle_align_gt if tie_gt else (L.sw_oracle_align_lowmem if lowmem else L.sw_oracle_align)
    rc = fn(ref_b, len(ref_b), read_b, len(read_b), match, mismatch, gap, C.byref(r))
    if rc != 0:
        raise MemoryError("oracle allocation failed")
    try:
        n = r.n_cells
        k = n if max_cells is None else min(n, max_cells)
        cells = [(r.cells[2 * c], r.cells[2 * c + 1]) for c in range(k)]
        sites = []
        for c in range(k):
            a, b = r.aln_off[c], r.aln_off[c + 1]
            sites.append((r.beginning[c],
                          C.string_at(C.addressof(r.ref_aln.contents) + a, b - a).decode("latin-1"),
                          C.string_at(C.addressof(r.read_aln.contents) + a, b - a).decode("latin-1")))
        return PairResult(r.score, cells, sites, L.sw_oracle_digest(C.byref(r)))
    finally:
        L.sw_oracle_free(C.byref(r))


def align_raw(ref, read, match: int = 5, mismatch: int = -3, gap: int = -4, lowmem: bool = False,
              tie_gt: bool = False) -> dict:
    """One pair through the C oracle as numpy arrays, copied in bulk: score, cells [n, 2] int32, beginnings [n] int32,
    aln_off [n + 1] int64, and the concatenated aligned strings ref_aln / read_aln as uint8.  Same order as align()."""
    import numpy as np
    L = lib()
    ref_b, read_b = _b(ref), _b(read)
    r = _Result()
    fn = L.sw_oracle_align_gt if tie_gt else (L.sw_oracle_align_lowmem if lowmem else L.sw_oracle_align)
    if fn(ref_b, len(ref_b), read_b, len(read_b), match, mismatch, gap, C.byref(r)) != 0:
        raise MemoryError("oracle allocation failed")
    try:
        n = int(r.n_cells)

        def arr(ptr, k, dtype):
            return np.ctypeslib.as_array(ptr, shape=(k,)).copy() if k else np.zeros(0, dtype)
        aln_off = arr(r.aln_off, n + 1, np.int64) if n else np.zeros(1, np.int64)
        total = int(aln_off[-1])
        return {"score": int(r.score),
                "cells": arr(r.cells, 2 * n, np.int32).reshape(n, 2),
                "beginnings": arr(r.beginning, n, np.int32),
                "aln_off": aln_off,
                "ref_aln": np.frombuffer(C.string_at(C.addressof(r.ref_aln.contents), total), np.uint8) if total else np.zeros(0, np.uint8),
                "read_aln": np.frombuffer(C.string_at(C.addressof(r.read_aln.contents), total), np.uint8) if total else np.zeros(0, np.uint8)}
    finally:
        L.sw_oracle_free(C.byref(r))


def score(ref, read, match: int = 5, mismatch: int = -3, gap: int = -4) -> Tuple[int, int]:
    """(max score, number of max cells), two-row memory."""
    L = lib()
    ref_b, read_b = _b(ref), _b(read)
    s = C.c_int32(); n = C.c_int64()
    if L.sw_oracle_score(ref_b, len(ref_b), read_b, len(read_b), match, mismatch, gap,
                         C.byref(s), C.byref(n)) != 0:
        raise MemoryError
    return s.value, n.value


def _concat(seqs: Sequence) -> Tuple[bytes, "C.Array"]:
    bs = [_b(s) for s in seqs]
    off = (C.c_int64 * (len(bs) + 1))()
    t = 0
    for k, s in enumerate(bs):
        off[k] = t
        t += len(s)
    off[len(bs)] = t
    return b"".join(bs), off


def cpu_baseline(refs: Sequence, reads: Sequence, match: int = 5, mismatch: int = -3,
                 gap: int = -4, threads: int = 1, mode: int = 0, want_scores: bool = False):
    """Run reads x refs on host cores. mode 0 = spark-local[N]-shaped slices,
    mode 1 = dynamic queue ("threadedMetrics"-shaped). Returns dict."""
    L = lib()
    rb, roff = _concat(refs)
    qb, qoff = _concat(reads)
    totals = (C.c_int32 * max(1, len(refs)))()
    scores = (C.c_int32 * max(1, len(refs) * len(reads)))() if want_scores else None
    cs = C.c_uint64()
    secs = L.sw_cpu_baseline_run(rb, roff, len(refs), qb, qoff, len(reads), match, mismatch, gap,
                                 threads, mode, totals, scores, C.byref(cs))
    cells = sum(len(_b(r)) for r in refs) * sum(len(_b(q)) for q in reads)
    out = {"seconds": secs, "cells": cells, "gcups": cells / 1e9 / secs if secs > 0 else 0.0,
           "ref_totals": list(totals)[:len(refs)], "checksum": cs.value, "threads": threads,
           "mode": "spark-local" if mode == 0 else "threaded-queue"}
    if want_scores:
        out["pair_scores"] = list(scores)
    return out
