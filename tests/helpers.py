"""Shared test helpers: the CUDA path (through the C ABI) against the C oracle, and which kernels a call ran."""
import json
import os
import re
import tempfile

import oracle


def check_pairs(eng, refs, reads, scores=(5, -3, -4), pairs=None, max_cells=None):
    rs = eng.load_refset(refs)
    res = rs.align(reads, scores).cache()
    n_checked = 0
    it = pairs if pairs is not None else [(r, q) for r in range(len(refs)) for q in range(len(reads))]
    for (r, q) in it:
        exp = oracle.align(refs[r], reads[q], *scores, max_cells=max_cells)
        got = res.pair(r, q, max_cells=max_cells)
        assert got[0] == exp.score, f"score ref={r} read={q}: {got[0]} != {exp.score}"
        exp_n = len(refs[r]) * len(reads[q]) if exp.score == 0 else None
        if exp_n is not None:
            assert res.pair_cell_count(r, q) == exp_n
        elif max_cells is None:
            assert res.pair_cell_count(r, q) == len(exp.cells)
        assert got[1] == exp.cells, f"cells ref={r} read={q}: {got[1][:5]} != {exp.cells[:5]}"
        assert got[2] == exp.sites, f"sites ref={r} read={q}: {got[2][:2]} != {exp.sites[:2]}"
        n_checked += 1
    # per-ref wrapping totals (Distribution.java:424)
    import numpy as np
    sc = res.scores.astype(np.int64)
    tot = (sc.sum(axis=1) & 0xFFFFFFFF).astype(np.uint32).view(np.int32) if sc.size else np.zeros(len(refs), np.int32)
    assert (res.ref_totals == tot).all()
    res.free(); rs.free()
    return n_checked


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
