#!/usr/bin/env python
"""Both-strands mode (SWB_F_BOTH_STRANDS) against the plain call on bench.py's default workload (128 x 150 bp reads
per step against 10,000 RefSeq-shaped references, synth seeds as in bench.py, scores 5/-3/-4), in one process on one
GPU.

Per step, alternating: the plain call, the plain call in hits mode at k = 1, the both-strands call and the
both-strands call in hits mode at k = 1, all through host buffers (H2D of the reads, compute, D2H of every result
array).  Reported per mode: median e2e ms over the steps, the engine's phase times (fill, locate = tile flag + scan +
emit + sort, select = top-k selection, inside the locate span on the short path, trace), the max cells kept and the
bytes of the result arrays copied to the host, and the both-strands / plain ratios; the card's name and power limit
are read in the same run.  Every both-strands step is checked against the plain step: its even oriented rows are the
plain scores.

    python tests/checks/run_strands.py [--steps 12] [--warmup 3] [--out profiles/strands_r03.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

from tests.checks.run_hits import result_bytes  # noqa: E402


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
    modes = {"plain": (None, False), "plain_hits_k1": (1, False), "both": (None, True), "both_hits_k1": (1, True)}
    rows = {m: [] for m in modes}
    for s in range(W + K):
        for m, (k, both) in modes.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = rs.align(steps[s], (5, -3, -4), top_k=k, both_strands=both)
            ms = (time.perf_counter() - t0) * 1e3
            if s >= W:
                st = res.stats
                rows[m].append({"e2e_ms": ms, "fill_ms": st["fill_ms"], "locate_ms": st["locate_ms"], "select_ms": st["select_ms"],
                                "trace_ms": st["trace_ms"], "d2h_ms": st["d2h_ms"], "max_cells": int(st["max_cells"]),
                                "d2h_bytes": result_bytes(res, k or 0)})
                if m == "plain":
                    plain_scores = res.scores
                elif both:
                    assert (res.scores[0::2] == plain_scores).all(), (m, s)
            res.free()
    summary = {}
    for m, r in rows.items():
        summary[m] = {key: float(np.median([x[key] for x in r])) for key in r[0]}
        summary[m]["e2e_ms_min"] = float(min(x["e2e_ms"] for x in r))
        summary[m]["e2e_ms_max"] = float(max(x["e2e_ms"] for x in r))
    ratios = {f"{b}/{p}": {key: summary[b][key] / summary[p][key] for key in ("e2e_ms", "fill_ms", "locate_ms", "trace_ms", "d2h_bytes")
                           if summary[p][key] > 0}
              for b, p in (("both", "plain"), ("both_hits_k1", "plain_hits_k1"), ("both_hits_k1", "plain"))}
    out = {"card": card, "workload": f"{B} x 150 bp reads x {a.refs} refs per step (bench.py default seeds), scores 5/-3/-4",
           "steps": K, "warmup": W, "order": "per step: plain, plain hits k=1, both strands, both strands hits k=1",
           "median": summary, "ratios": ratios, "per_step": rows}
    text = json.dumps(out, indent=1)
    print(json.dumps({"card": card, "median": summary, "ratios": ratios}, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    rs.free(); eng.close()


if __name__ == "__main__":
    main()
