#!/usr/bin/env python
"""All-hits mode against the plain call and hits mode on bench.py's default workload (128 x 150 bp reads per step
against 10,000 RefSeq-shaped references, synth seeds as in bench.py, scores 5/-3/-4), in one process on one GPU.

Per step, alternating: plain swb_align, swb_align_hits with k = 1, swb_align_all_hits with margin 0 (the co-optimal
set) and with a threshold (min_score 100, no margin), all through host buffers (H2D of the reads, compute, D2H of every
result array).  Every mode's lists are checked against the plain call's filtered scores.  Reported per mode: median
e2e ms over the steps, the engine's phase times (fill, locate, select, trace), the max cells kept and the bytes of
the result arrays copied to the host; the card's name and power limit are read in the same run.

    python tests/checks/run_all_hits.py [--steps 12] [--warmup 3] [--out profiles/all_hits_r03.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))


def result_bytes(res, k):
    """bytes of the arrays a fetch copies to the host (scores, totals, best hits, hits or lists, cell offsets, cells,
    beginnings, op lengths, ops offsets, ops)"""
    import numpy as np
    n_pairs, n = res.n_refs * res.n_reads, res.total_cells
    words = int(((res.op_lens.astype(np.int64) + 15) // 16).sum()) if n else 0
    lists = 8 * (res.n_reads + 1) + 16 * len(res.hit_list) if len(res.hit_offsets) else 0
    return (4 * n_pairs + 4 * res.n_refs + 16 * res.n_reads + 16 * res.n_reads * k + lists + 8 * (n_pairs + 1) + 16 * n
            + 8 * (n + 1) + 4 * words)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reads-per-step", type=int, default=128)
    ap.add_argument("--refs", type=int, default=10_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    import sparksmithwaterman_b200 as swb
    from sparksmithwaterman_b200 import synth
    from tests.test_all_hits_host import all_hits_ref
    from tests.test_hits_host import top_hits_ref
    try:
        card = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                                        "--format=csv,noheader"], text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        card = "unknown (nvidia-smi unavailable)"
    B, W, K = a.reads_per_step, a.warmup, a.steps
    refs = synth.make_refs(a.refs)
    pool = synth.make_reads(B * (W + K), 150, refs)
    steps = [pool[s * B:(s + 1) * B] for s in range(W + K)]
    eng = swb.Engine(0, 64 << 30)
    rs = eng.load_refset(refs)
    modes = {"plain": {}, "hits_k1": {"top_k": 1}, "all_hits_margin0": {"margin": 0},
             "all_hits_threshold100": {"margin": 2**31 - 1, "min_score": 100}}
    rows = {m: [] for m in modes}
    for s in range(W + K):
        for m, kw in modes.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = rs.align(steps[s], (5, -3, -4), **kw)
            ms = (time.perf_counter() - t0) * 1e3
            k = kw.get("top_k", 0)
            if s >= W:
                st = res.stats
                rows[m].append({"e2e_ms": ms, "fill_ms": st["fill_ms"], "locate_ms": st["locate_ms"], "select_ms": st["select_ms"],
                                "trace_ms": st["trace_ms"], "d2h_ms": st["d2h_ms"], "max_cells": int(st["max_cells"]),
                                "d2h_bytes": result_bytes(res, k), "listed": int(len(res.hit_list)) if "margin" in kw else k * B})
                if m == "plain":
                    plain_scores, plain_best = res.scores, res.best_hits
                else:
                    assert (res.scores == plain_scores).all() and (res.best_hits == plain_best).all(), (m, s)
                if k:
                    assert (res.hits[:, :, :2] == top_hits_ref(plain_scores, k)[:, :, :2]).all(), (m, s)
                if "margin" in kw:
                    eo, el = all_hits_ref(plain_scores, kw.get("min_score", 1), kw["margin"])
                    assert (res.hit_offsets == eo).all() and (res.hit_list[:, :2] == el[:, :2]).all(), (m, s)
            res.free()
    summary = {}
    for m, r in rows.items():
        summary[m] = {key: float(np.median([x[key] for x in r])) for key in r[0]}
        summary[m]["e2e_ms_min"] = float(min(x["e2e_ms"] for x in r))
        summary[m]["e2e_ms_max"] = float(max(x["e2e_ms"] for x in r))
    out = {"card": card, "workload": f"{B} x 150 bp reads x {a.refs} refs per step (bench.py default seeds), scores 5/-3/-4",
           "steps": K, "warmup": W, "order": "per step: plain, hits k=1, all-hits margin 0, all-hits min_score 100 without margin",
           "median": summary, "per_step": rows}
    text = json.dumps(out, indent=1)
    print(json.dumps({"card": card, "median": summary}, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    rs.free(); eng.close()


if __name__ == "__main__":
    main()
