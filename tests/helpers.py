"""Shared test helpers: the CUDA path (through the C ABI) against the C oracle, and which kernels a call ran."""
import ctypes as C
import json
import os
import re
import tempfile

import numpy as np

import oracle


OP_ALIGN, OP_INS, OP_DEL = 1, 2, 3         # swb_result_ops codes: aligned pair, gap in the reference, gap in the read


def oracle_arrays(ref, read, scores=(5, -3, -4), tie_gt=False, lowmem=False):
    """One pair through the C oracle as whole arrays, in its list order (row-major; under tie_gt DistributedSW's
    order): score, count, m, n, cells [c, 2], beginnings [c], op_lens [c], ops (all cells' ops concatenated, the
    result's codes), and the raw aligned strings (aln_off, ref_aln, read_aln) for checks of the string builder.  A
    score-0 pair lists all m * n cells with empty alignments, as the reference does."""
    rb, qb = oracle._b(ref), oracle._b(read)
    assert b"_" not in rb and b"_" not in qb, "'_' is the oracle's gap symbol: ops could not be told apart"
    r = oracle.align_raw(rb, qb, *scores, lowmem=lowmem, tie_gt=tie_gt)
    ops = np.where(r["ref_aln"] == ord("_"), OP_INS, np.where(r["read_aln"] == ord("_"), OP_DEL, OP_ALIGN)).astype(np.uint8)
    r.update(count=len(r["beginnings"]), m=len(qb), n=len(rb), op_lens=np.diff(r["aln_off"]), ops=ops)
    return r


def _flat(res):
    """The fetched result's flat arrays, pulled once per result."""
    f = getattr(res, "_every_cell_flat", None)
    if f is None:
        f = {"scores": res.scores, "offsets": res.cell_offsets, "cells": res.cells, "beginnings": res.beginnings,
             "op_lens": res.op_lens.astype(np.int64)}
        res._every_cell_flat = f
    return f


def result_ops(res, lo, hi):
    """The ops of materialised cells lo .. hi - 1 of a fetched result, concatenated: one swb_result_ops call per cell
    (the C ABI has no bulk accessor) into one buffer."""
    lens = _flat(res)["op_lens"][lo:hi]
    starts = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=starts[1:])
    buf = np.zeros(max(int(starts[-1]), 1), np.uint8)
    base, fn, h = buf.ctypes.data, res.lib.swb_result_ops, res.h
    u8 = C.c_uint8
    for k in range(hi - lo):
        n = int(lens[k])
        if n:
            assert fn(h, lo + k, (u8 * n).from_address(base + int(starts[k])), n) == 0
    return buf[:int(starts[-1])]


def result_range(res, p):
    """cells, beginnings, op lengths and ops of pair index p's materialised range, as whole arrays."""
    f = _flat(res)
    lo, hi = int(f["offsets"][p]), int(f["offsets"][p + 1])
    return {"cells": f["cells"][lo:hi], "beginnings": f["beginnings"][lo:hi], "op_lens": f["op_lens"][lo:hi],
            "ops": result_ops(res, lo, hi), "lo": lo}


def assert_ranges_equal(a, b, where=""):
    """Two results' ranges of one pair (result_range) hold the same cells, beginnings, op lengths and ops."""
    for key in ("cells", "beginnings", "op_lens", "ops"):
        assert a[key].shape == b[key].shape and np.array_equal(a[key], b[key]), f"{key} {where}"


def result_arrays(res, ref, read, probes=4, seed=0):
    """The arrays of oracle_arrays from a fetched AlignResult for pair (ref, read), in the result's (row-major) order.
    A score-0 pair has no materialised cells: `probe` holds swb_result_pair_cell's (k, i, j) at k = 0, m * n - 1 and
    a few seeded k, for the closed form of its implicit cells."""
    f = _flat(res)
    p = res.pair_index(ref, read)
    out = result_range(res, p)
    m, n = len(res.reads[read]), len(res.rs.seqs[ref >> 1] if res.both_strands else res.rs.seqs[ref])
    out.update(score=int(f["scores"][ref, read]), count=res.pair_cell_count(ref, read), m=m, n=n)
    if out["score"] == 0 and m * n:
        ks = sorted({0, m * n - 1} | set(np.random.default_rng(seed + p).integers(0, m * n, probes).tolist()))
        i, j, bg, ln = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        probe = []
        for k in ks:
            assert res.lib.swb_result_pair_cell(res.h, p, k, C.byref(i), C.byref(j), C.byref(bg), C.byref(ln)) == 0
            probe.append((k, i.value, j.value, bg.value, ln.value))
        out["probe"] = np.array(probe, np.int64).reshape(-1, 5)
    return out


def distributed_permutation(cells, beginnings):
    """DistributedSW's order of a row-major cell list (sw.distributed_order): beginning, then anti-diagonal i + j,
    then j -- one lexsort, since (i + j, j) is unique per cell."""
    i, j = cells[:, 0].astype(np.int64), cells[:, 1].astype(np.int64)
    return np.lexsort((j, i + j, beginnings))


def _segments(op_lens, order):
    """Indices that gather the concatenated ops of cells `order` from ops laid out in op_lens order."""
    starts = np.zeros(len(op_lens) + 1, np.int64)
    np.cumsum(op_lens, out=starts[1:])
    lens = op_lens[order]
    if not len(lens) or not lens.sum():
        return np.zeros(0, np.int64)
    out_starts = np.zeros(len(lens), np.int64)
    np.cumsum(lens[:-1], out=out_starts[1:])
    return np.repeat(starts[:-1][order] - out_starts, lens) + np.arange(int(lens.sum()))


def assert_pair_equal(got, exp, tie_gt=False, where=""):
    """A pair of the result (result_arrays) against the oracle (oracle_arrays): the score, the cell count (the implicit
    m * n cells of a score-0 pair too), every cell in list order, every beginning, op length and op.  The result
    lists cells row-major under both tie rules; under tie_gt it is re-ordered the way the host layer does before
    the comparison."""
    assert got["score"] == exp["score"], f"score {where}: {got['score']} != {exp['score']}"
    if exp["score"] == 0:
        mn = exp["m"] * exp["n"]
        assert got["count"] == mn == exp["count"], f"score-0 count {where}: {got['count']}, m * n = {mn}"
        assert len(got["cells"]) == 0 and len(got["ops"]) == 0, f"score-0 pair materialised cells {where}"
        if mn:
            k, i, j, bg, ln = got["probe"].T
            assert (i == k // exp["n"] + 1).all() and (j == k % exp["n"] + 1).all(), f"score-0 cells {where}"
            assert (bg == 0).all() and (ln == 0).all(), f"score-0 alignments {where}"
        return
    cells, beg, lens, ops = got["cells"], got["beginnings"], got["op_lens"], got["ops"]
    c = len(cells)
    assert got["count"] == c == exp["count"], f"cell count {where}: {got['count']} / {c} != {exp['count']}"
    assert len(ops) == int(lens.sum()), f"ops {where}: {len(ops)} ops for op lengths summing to {int(lens.sum())}"
    key = cells[:, 0].astype(np.int64) * (exp["n"] + 1) + cells[:, 1]
    assert (np.diff(key) > 0).all(), f"cells not row-major {where}"
    if tie_gt:
        order = distributed_permutation(cells, beg)
        ops = ops[_segments(lens, order)]
        cells, beg, lens = cells[order], beg[order], lens[order]
    bad = np.nonzero((cells != exp["cells"]).any(axis=1))[0]
    assert not len(bad), f"cell {bad[0]} of {c} {where}: {tuple(cells[bad[0]])} != {tuple(exp['cells'][bad[0]])}"
    bad = np.nonzero(beg != exp["beginnings"])[0]
    assert not len(bad), f"beginning of cell {bad[0]} {where}: {beg[bad[0]]} != {exp['beginnings'][bad[0]]}"
    bad = np.nonzero(lens != exp["op_lens"])[0]
    assert not len(bad), f"op length of cell {bad[0]} {where}: {lens[bad[0]]} != {exp['op_lens'][bad[0]]}"
    if not np.array_equal(ops, exp["ops"]):
        at = int(np.nonzero(ops != exp["ops"])[0][0])
        cell = int(np.searchsorted(np.cumsum(lens), at, side="right"))
        raise AssertionError(f"op {at} (cell {cell}) {where}: {ops[at]} != {exp['ops'][at]}")


def oracle_key(ref, read, scores, tie_gt):
    return ref, read, tuple(scores), bool(tie_gt)


def check_pairs(eng, refs, reads, scores=(5, -3, -4), pairs=None, max_cells=None, tie_gt=False, lowmem=False,
                memo=None, kernels=None):
    """Every pair (or `pairs`) of one plain call against the oracle, every max cell: assert_pair_equal.  max_cells
    limits only the check of the host string builder (swb_result_materialize) to each pair's first max_cells cells.
    Identical (reference, read) pairs share one oracle run.  lowmem: the oracle's low-memory form (a 4 Mbp x 150
    pair needs about 3 GB with full matrices); the tie_gt oracle has no such form.  memo: a dict of oracle results
    (keyed by oracle_key) shared between calls.  kernels: a list that receives the call's launches
    (launched_kernels)."""
    rs = eng.load_refset(refs)
    if kernels is None:
        res = rs.align(reads, scores, tie_gt=tie_gt).cache()
    else:
        res, launched = launched_kernels(lambda: rs.align(reads, scores, tie_gt=tie_gt).cache())
        kernels.extend(launched)
    n_checked = 0
    memo = {} if memo is None else memo
    it = pairs if pairs is not None else [(r, q) for r in range(len(refs)) for q in range(len(reads))]
    for (r, q) in it:
        k = oracle_key(refs[r], reads[q], scores, tie_gt)
        if k not in memo:
            memo[k] = oracle_arrays(refs[r], reads[q], scores, tie_gt=tie_gt, lowmem=lowmem)
        exp = memo[k]
        got = result_arrays(res, r, q)
        assert_pair_equal(got, exp, tie_gt, where=f"ref={r} read={q}")
        if exp["score"] > 0:
            _check_strings(res, got, exp, oracle._b(refs[r]), oracle._b(reads[q]), max_cells, tie_gt, f"ref={r} read={q}")
        n_checked += 1
    # per-ref wrapping totals (Distribution.java:424)
    sc = res.scores.astype(np.int64)
    tot = (sc.sum(axis=1) & 0xFFFFFFFF).astype(np.uint32).view(np.int32) if sc.size else np.zeros(len(refs), np.int32)
    assert (res.ref_totals == tot).all()
    res.free(); rs.free()
    return n_checked


def _check_strings(res, got, exp, ref, read, max_cells, tie_gt, where):
    """swb_result_materialize of the pair's first max_cells cells (row-major) against the oracle's strings."""
    c = len(got["cells"])
    k_max = c if max_cells is None else min(c, max_cells)
    pos = np.arange(c)
    if tie_gt:
        pos[distributed_permutation(got["cells"], got["beginnings"])] = np.arange(c)
    off = exp["aln_off"]
    for k in range(k_max):
        e = int(pos[k])
        a, b = int(off[e]), int(off[e + 1])
        ra, qa = res.materialize(got["lo"] + k, ref, read, b - a)
        assert ra == exp["ref_aln"][a:b].tobytes().decode("latin-1") and qa == exp["read_aln"][a:b].tobytes().decode("latin-1"), \
            f"strings of cell {k} {where}"


def launched_kernels(fn):
    """Runs fn() under torch.profiler with CUDA activities.  Returns fn's result and the kernels the device ran, as
    (demangled name, grid x) in launch order."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    return out, [(e["name"], e["args"]["grid"][0]) for e in events if e.get("cat") == "kernel"]


def launches(kernels, pattern):
    """The grids of the launches whose name matches the regular expression.  Match unqualified names with a word
    boundary in front: r"\\btrace_kernel<" does not match tile_trace_kernel or wide_trace_kernel."""
    return [grid for name, grid in kernels if re.search(pattern, name)]


def parts_workspace(refs, parts):
    """Workspace bytes at which a set of these references is cut into `parts` (>= 3) parts: a part holds about
    96 read pairs' block records of 74 bytes per base, and the count rounds to the nearest, plus one smaller part."""
    total = sum(len(r) for r in refs)
    return 74 * 96 * total // (parts - 1)
