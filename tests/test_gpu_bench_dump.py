"""GPU: bench.py --dump-outputs on a small workload writes the results of the last timed step, and they are the
oracle's answers for that step's seeded inputs (scores, max-cell lists, beginnings, alignment columns, totals,
best hits)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from bench import READ_LEN
from sparksmithwaterman_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_match_the_oracle(tmp_path):
    B, K, W, n_refs = 4, 2, 1, 40
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(K), "--warmup", str(W),
                        "--reads-per-step", str(B), "--refs-per-gpu", str(n_refs), "--workspace-gb", "2",
                        "--no-cpu-baseline", "--dump-outputs", str(out)],
                       cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype == np.float64 for a in d.values())

    refs = synth.make_refs(n_refs)
    reads = synth.make_reads(B * (W + K), READ_LEN, refs)[B * (W + K - 1):]     # the last timed step
    exp = [oracle.align(r, q) for r in refs for q in reads]                              # pair p = ref * B + read
    assert d["pair_index"].tolist() == list(range(n_refs * B))                           # small: nothing sampled
    assert d["scores"].tolist() == [e.score for e in exp]
    assert d["cell_counts"].tolist() == [len(e.cells) if e.score else 0 for e in exp]
    sc = np.array([e.score for e in exp], np.int64).reshape(n_refs, B)
    assert d["ref_totals"].tolist() == [int(t) for t in (sc.sum(axis=1) & 0xFFFFFFFF).astype(np.uint32).view(np.int32)]
    for q in range(B):
        k = int(np.argmax(sc[:, q]))                                                      # lowest ref on ties
        assert d["best_hits"][q].tolist() == [sc[k, q], k, *exp[k * B + q].cells[0]]

    cells = [c for e in exp if e.score for c in e.cells]
    sites = [s for e in exp if e.score for s in e.sites]
    assert d["cell_index"].tolist() == list(range(len(cells)))
    assert d["cells"].tolist() == [list(c) for c in cells]
    assert d["beginnings"].tolist() == [s[0] for s in sites]
    assert d["op_lens"].tolist() == [len(s[1]) for s in sites]
    ops = [2 if a == "_" else 3 if b == "_" else 1 for (_, ra, qa) in sites[:4096] for a, b in zip(ra, qa)]
    assert d["ops"].tolist() == ops
