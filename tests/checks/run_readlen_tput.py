#!/usr/bin/env python
"""Throughput of whole batches of reads of one length against the cfg2-shaped reference set (10,000 lognormal
references, 21.3 Mbp): where does the s16x2 path end?  Reads up to 256 rows use the classes K <= 32, reads of
257 .. 511 rows the LONG classes K = 40 .. 64 (same kernels), longer reads the int32 wide path.  The wide path's
numbers for 257 .. 511 rows, from before the long classes, are kept in profiles/readlen_tput_r02.json.

    python tests/checks/run_readlen_tput.py --out profiles/readlen_tput_r02.json
"""
import argparse, json, os, sys, time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

CASES = [(36, 256), (50, 256), (75, 256), (100, 128), (125, 128), (150, 128), (200, 128), (250, 128), (260, 64), (300, 64), (400, 64), (500, 64), (511, 64), (512, 32), (1000, 32), (2000, 16)]


def run(cases):
    import sparksmithwaterman_b200 as swb
    from sparksmithwaterman_b200 import synth
    refs = synth.make_refs(10000)
    tot = sum(len(r) for r in refs)
    eng = swb.Engine(0, 64 << 30)
    rs = eng.load_refset(refs)
    rows = []
    for m, n in cases:
        reads = synth.make_reads(n, m, refs)
        for _ in range(2):
            rs.align(reads).free()
        t0 = time.perf_counter(); res = rs.align(reads); dt = (time.perf_counter() - t0) * 1e3
        st = res.stats; res.free()
        cells = m * n * tot
        rows.append({"read_len": m, "reads": n, "refs": len(refs), "cells": cells, "wall_ms": round(dt, 2),
                     "gcups_e2e": round(cells / 1e9 / (dt * 1e-3), 1), "gcups_fill": round(cells / 1e9 / (st["fill_ms"] * 1e-3), 1),
                     "fill_ms": round(st["fill_ms"], 2), "locate_ms": round(st["locate_ms"], 2), "trace_ms": round(st["trace_ms"], 2),
                     "batches": int(st["batches"])})
        print(rows[-1], flush=True)
    rs.free(); eng.close()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rows = run(CASES)
    doc = {"what": "whole batches of one read length x 10,000 references through swb_align (host buffers, incl. traceback)",
           "rows": rows}
    if a.out:
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
