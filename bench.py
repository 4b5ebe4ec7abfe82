#!/usr/bin/env python
"""bench.py -- GCUPS (including traceback) of the Smith-Waterman hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--reads-per-step B] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload = BASELINE.json configs[1]: 150 bp reads vs 10,000 RefSeq-shaped references
(lognormal lengths, mean 2,160 / median 1,609 bp), default scores 5/-3/-4.  A STEP is one
batch of B reads (a slice of the 100k-read job) aligned against ALL references resident in
HBM: fill, every max cell, every traceback.  GCUPS = sum(m*n) / 1e9 / seconds.

  value : reads already resident in HBM, results left in HBM (swb_align_resident)
  e2e   : the reference-facing C-ABI call with HOST buffers (swb_align): H2D of the reads
          and D2H of scores, max-cell lists and packed alignments inside the timed region
  N > 1 : the reference set is sharded over the ranks (balanced by length), every rank
          aligns the same reads against its shard, and the per-read best-hit records are
          merged with one ncclAllGather + a merge kernel per step, issued by libswb200 itself
          on the engine's stream (swb_comm_*, the C ABI a JVM host binds; torch.distributed only
          carries the 128-byte NCCL id and the timing reductions).  Weak scaling: 10k refs per GPU.
          After the timed region the merged records of the last step are checked against an
          independent torch reduction (max score, lowest global ref id).

`--impl reference` times the reference's CPU path instead: the C restatement of
SmithWaterman.java under oracle/ (no JVM exists in this image) on all host cores.

`--dump-outputs DIR` writes the results of the last timed step to DIR/<name>.npy (see dump_outputs), so that
two builds can be compared output for output on identical, seeded inputs.

bench.py compiles nothing: it runs from a tree built by `python __graft_entry__.py` (libswb200 and the CPU oracle).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCORES = (5, -3, -4)
METRIC = "GCUPS incl. traceback (150 bp reads x 10k RefSeq-shaped refs per B200)"
UNIT = "GCUPS"
READ_LEN = 150
N_REFS_PER_GPU = 10_000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reads-per-step", type=int, default=128)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workspace-gb", type=float, default=64.0)
    ap.add_argument("--refs-per-gpu", type=int, default=N_REFS_PER_GPU,
                    help="10000 = BASELINE config 2 per GPU; 15402 x 8 GPUs = config 4 (123,212 refs, ~266 Mbp)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results to DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("sm_max_mhz", 1965.0), "measured"
    return 6650.0, 1965.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        # samples under load = upper half (the sampler also sees the idle edges)
        load = sm[len(sm) // 2:] if sm else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


def bind_to_gpu_numa_node(index: int):
    """Run this rank (and the pinned result buffers it allocates: first touch) on the CPU cores of the NUMA node the GPU
    hangs off, so that 8 ranks pulling their results over PCIe do not cross the socket interconnect.  Best effort."""
    try:
        bus = subprocess.check_output(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                      text=True).strip().lower()
        bus = bus[-12:] if len(bus) > 12 else bus                      # 00000000:1B:00.0 -> 0000:1b:00.0
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return {"numa_node": node, "cpus": len(allowed)}
    except Exception:
        pass
    return None


def shard_refs(refs, rank: int, world: int):
    """Length-balanced shard of the reference set (SURVEY.md 8e)."""
    from sparksmithwaterman_b200 import multigpu
    mine = multigpu.shard_refs([len(r) for r in refs], rank, world)
    return [refs[k] for k in mine], mine


def cpu_baseline_leg(refs, reads, threads, target_cells=2.0e10):
    """Oracle CPU harness (C restatement of the Java path) on a bounded sample."""
    import oracle
    n_refs = min(len(refs), 1000)
    sub_refs = refs[:n_refs]
    ref_bases = sum(len(r) for r in sub_refs)
    n_reads = max(1, min(len(reads), int(target_cells / (ref_bases * READ_LEN))))
    r = oracle.cpu_baseline(sub_refs, reads[:n_reads], *SCORES, threads=threads, mode=1)
    # the same sample, sliced like ParallelCollectionRDD (contiguous ref slices, one thread each)
    r0 = oracle.cpu_baseline(sub_refs, reads[:max(1, n_reads // 4)], *SCORES, threads=threads, mode=0)
    return {"value": round(r["gcups"], 4), "unit": UNIT, "cores": threads, "kind": "port",
            "spark_local_shaped_gcups": round(r0["gcups"], 4),
            "spark_local_as_written_gcups": round(r0["gcups"] / 2.0, 4),
            "spark_local_note": "contiguous ref slices, one thread per slice; 'as written' halves it because the un-cached "
                                "map is evaluated again by lookup() after first() (Distribution.java:341-352)",
            "sample": f"{n_reads} x {READ_LEN} bp reads vs first {n_refs} refs of the workload "
                      f"({r['cells']:.3g} cells, {r['seconds']:.1f} s), dynamic ref queue over {threads} threads, "
                      "C restatement of SmithWaterman.java (no JVM in this image)",
            "reads_per_s": round(n_reads / r["seconds"] * (n_refs / len(refs)), 4),
            "seconds": round(r["seconds"], 3)}


def workload_config(B, refs_per_gpu, world, n_refs_local, ref_bases_local):
    return {"workload": f"cfg2: 150 bp reads vs {refs_per_gpu:,} RefSeq-shaped refs per GPU, scores 5/-3/-4; "
                        f"step = {B} reads of the 100k-read job x all refs, fill + all max cells + traceback",
            "reads_per_step": B, "refs_per_gpu": n_refs_local, "ref_bases_per_gpu": int(ref_bases_local),
            "pairs_per_step": B * n_refs_local * world,
            "l2": "per-step working set (block records, tens of GB) exceeds the 126 MB L2; no explicit flush",
            "parallelism": f"refshard{world}" if world > 1 else "single"}


DUMP_MAX_BYTES = 64 * 10**6
DUMP_MAX_PAIRS = 1 << 20
DUMP_MAX_CELLS = 1 << 19
DUMP_OPS_CELLS = 4096


def dump_outputs(res, out_dir):
    """What a caller of the timed path receives once it fetches the step's results, as out_dir/<name>.npy in float64
    (exact for every int32 and int64 value the arrays hold).  Per-pair and per-cell arrays larger than the caps
    above are cut to a fixed-seed sample; its indices go to pair_index / cell_index.  Pair p is (ref p // n_reads,
    read p % n_reads); cells are numbered across pairs in the order of the result's flat arrays."""
    import numpy as np

    def sample(n, cap, seed):
        if n <= cap:
            return np.arange(n)
        return np.sort(np.random.Generator(np.random.PCG64(seed)).choice(n, cap, replace=False))

    res.fetch().cache()
    pairs = sample(res.n_refs * res.n_reads, DUMP_MAX_PAIRS, 1)
    cells = sample(res.total_cells, DUMP_MAX_CELLS, 2)
    out = {"pair_index": pairs,
           "scores": res.scores.reshape(-1)[pairs],
           "cell_counts": np.diff(res.cell_offsets)[pairs],       # materialised max cells (none for score-0 pairs)
           "ref_totals": res.ref_totals,
           "best_hits": res.best_hits,                            # per read: score, ref, i, j
           "cell_index": cells,
           "cells": res.cells[cells],                             # (i, j), 1-based
           "beginnings": res.beginnings[cells],
           "op_lens": res.op_lens[cells],
           # alignment columns (1 aligned, 2 insertion, 3 deletion) of the first sampled cells, concatenated;
           # op_lens[:DUMP_OPS_CELLS] splits them
           "ops": np.concatenate([np.zeros(0)] + [res.ops(int(c)) for c in cells[:DUMP_OPS_CELLS]])}
    out = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in out.items()}
    total = sum(a.nbytes + 128 for a in out.values())             # + the .npy header
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_MAX_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path, all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from sparksmithwaterman_b200 import synth
    oracle.build()
    threads = os.cpu_count() or 1
    refs = synth.make_refs(1000)
    ref_bases = sum(len(r) for r in refs)
    pool = synth.make_reads(64 * (args.steps + 1), READ_LEN, refs)
    # size one step to ~8 s of host time from a 2-read probe over the same references
    probe = oracle.cpu_baseline(refs, pool[:2], *SCORES, threads=threads, mode=1)
    rate = probe["cells"] / probe["seconds"]
    per = max(1, min(64, int(8.0 * rate / (ref_bases * READ_LEN))))
    reads = pool[2:]
    for w in range(args.warmup):
        oracle.cpu_baseline(refs[:100], reads[:1], *SCORES, threads=threads, mode=1)
    t0 = time.perf_counter()
    cells = 0
    for k in range(args.steps):
        r = oracle.cpu_baseline(refs, reads[k * per:(k + 1) * per], *SCORES, threads=threads, mode=1)
        cells += r["cells"]
    dt = time.perf_counter() - t0
    v = cells / 1e9 / dt
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic",
            "config": dict(workload_config(args.reads_per_step, args.refs_per_gpu, 1, args.refs_per_gpu,
                                           sum(len(r) for r in synth.make_refs(args.refs_per_gpu))),
                           sample=f"each timed step = {per} reads x the first {len(refs)} refs of that workload "
                                  f"({ref_bases * READ_LEN * per:.3g} cells), rate is size-invariant"),
            "cpu_baseline": {"value": round(v, 4), "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"{per} reads x {len(refs)} refs per step, {args.steps} steps; "
                                       "C restatement of SmithWaterman.java + MapRef loop (no JVM in this image), "
                                       "dynamic ref queue over all host threads"},
            "e2e": {"value": round(v, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import sparksmithwaterman_b200 as swb
    from sparksmithwaterman_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs writes one GPU's results; run it with --gpus 1")
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None

    B, K, W = args.reads_per_step, args.steps, args.warmup
    # weak scaling: 10k refs per GPU; every rank generates the same global set and keeps its shard
    all_refs = synth.make_refs(args.refs_per_gpu * world)
    refs, my_ids = shard_refs(all_refs, rank, world)
    reads_pool = synth.make_reads(B * (W + K), READ_LEN, all_refs)
    step_reads = [reads_pool[k * B:(k + 1) * B] for k in range(W + K)]

    eng = swb.Engine(local_rank, int(args.workspace_gb * (1 << 30)))
    t0 = time.perf_counter()
    rs = eng.load_refset(refs)
    torch.cuda.synchronize()
    refset_load_ms = (time.perf_counter() - t0) * 1e3
    ref_bases = rs.total_bases
    cells_per_step_local = ref_bases * READ_LEN * B
    stream = torch.cuda.ExternalStream(eng.stream_ptr, device=torch.device("cuda", local_rank))
    my_ids_np = np.asarray(my_ids, dtype=np.int64)
    comm = None
    if dist:
        # the data-path collective lives in libswb200 (swb_comm_*): NCCL id from rank 0, one communicator per rank
        from sparksmithwaterman_b200 import multigpu
        box = [multigpu.Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        comm = multigpu.Comm(eng, box[0], rank, world)

    def step_resident(rd, fetch=False):
        return rd.align(SCORES, scores_only=False, fetch=fetch)

    def allgather_best(res, want_host=False):
        """best hits -> global ref ids -> ncclAllGather -> merge kernel, all on the engine's stream (C ABI)."""
        if not comm:
            return None
        return comm.allgather_best(res, my_ids_np, want_host=want_host)

    def check_merge(res, merged):
        """Independent check of the merged records of one step with torch collectives: score = max over ranks of
        the local best score; ref = lowest global id among the ranks that reach it."""
        if not dist:
            return True
        local = torch.from_numpy(res.best_hits.astype(np.int64)).cuda()
        gid = torch.from_numpy(my_ids_np).cuda()[local[:, 1].clamp(min=0)]
        smax = local[:, 0].clone()
        dist.all_reduce(smax, op=dist.ReduceOp.MAX)
        cand = torch.where(local[:, 0] == smax, gid, torch.full_like(gid, 1 << 40))
        dist.all_reduce(cand, op=dist.ReduceOp.MIN)
        m = torch.from_numpy(merged.astype(np.int64)).cuda()
        mine = (local[:, 0] == smax) & (gid == cand)                  # the winning rank also checks (i, j)
        ok = bool((m[:, 0] == smax).all() and (m[:, 1] == cand).all() and (m[mine][:, 2:] == local[mine][:, 2:]).all())
        t = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    # resident read batches (inputs in HBM before the timed region)
    resident = [rs.upload_reads(r) for r in step_reads]
    # nvidia-smi takes ~0.1 s to start: launch the sampler before the warm-up so it is sampling (every 20 ms)
    # throughout the timed region; warm-up samples are under the same load
    sampler = ClockSampler(local_rank)
    sampler.start()
    for k in range(W):
        res = step_resident(resident[k]); allgather_best(res); res.free()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    t_wall0 = time.perf_counter()
    ev0.record(stream)
    agg = {"fill_ms": 0.0, "locate_ms": 0.0, "trace_ms": 0.0, "launches": 0.0, "checkpoint_bytes": 0.0,
           "max_cells": 0.0, "batches": 0.0}
    for k in range(W, W + K):
        res = step_resident(resident[k])
        st = res.stats
        for key in agg:
            agg[key] += st[key]
        allgather_best(res)
        if k < W + K - 1:
            res.free()                                            # the last step's results are freed after the clock
    ev1.record(stream)
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    if dist:
        dist.barrier()
    clocks = sampler.stop()
    dev_ms = ev0.elapsed_time(ev1)
    step_ms = max(dev_ms, t_wall * 1e3) / K          # events and wall agree unless the host lags
    if dist:
        t = torch.tensor([step_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        step_ms = float(t.item())
        c = torch.tensor([float(cells_per_step_local)], device="cuda", dtype=torch.float64)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        cells_per_step = float(c.item())
    else:
        cells_per_step = float(cells_per_step_local)
    value = cells_per_step / 1e9 / (step_ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(res, args.dump_outputs)
    res.free()

    # ---- e2e: host buffers through swb_align, H2D + D2H inside the timed region ----------
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    h2d = d2h = 0
    for k in range(min(W, 2)):                                    # untimed: pinned-buffer pool, allocator
        res = rs.align(step_reads[k], SCORES); allgather_best(res); res.free()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    t0 = time.perf_counter()
    merged_last = None
    for k in range(W, W + K):
        res = rs.align(step_reads[k], SCORES)                     # H2D reads + compute + D2H of every result array
        if k == W + K - 1:
            last = res
        merged_last = allgather_best(res, want_host=True)         # merged best hits land on the host too
        if k != W + K - 1:
            res.free()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / K
    merge_ok = check_merge(last, merged_last) if dist else None
    if dist and not merge_ok:
        raise SystemExit("bench.py: merged best hits of the last step differ from the independent reduction")
    if dist:
        t = torch.tensor([e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = cells_per_step / 1e9 / (e2e_ms * 1e-3)
    # bytes that crossed PCIe in one e2e step (counted from the arrays of the last step, after the clock)
    sc = last.scores
    nc = last.total_cells
    words = int(((last.op_lens.astype(np.int64) + 15) >> 4).sum())
    h2d = sum(len(r) for r in step_reads[W + K - 1]) + 8 * (B + 1)
    d2h = sc.nbytes + 4 * len(refs) + 16 * B + 8 * (sc.size + 1) + nc * (8 + 4 + 4 + 8) + 8 + 4 * words
    last.free()

    if comm:
        comm.close()
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    hbm_peak, sm_max, peak_kind = peaks()
    sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
    # DPX roofline (SURVEY.md 8d): 64 integer-pipe lane-ops/clk/SM (measured, profiles/dpx_microbench_r01.json),
    # 2 lane-ops per cell at the s16x2 minimum
    peak_gcups = sms * sm_max * 1e6 * 64 / 2 / 1e9
    # what this kernel can reach at most on the integer pipe: 2 DPX ops per s16x2 cell PAIR (VIMNMX3 + VIADDMNMX,
    # the add runs as IMAD on the FMA pipe) -> twice the SURVEY figure
    alu_bound_gcups = sms * sm_max * 1e6 * 64 / 1e9
    fill_gcups = cells_per_step_local * K / 1e9 / (agg["fill_ms"] * 1e-3) if agg["fill_ms"] > 0 else 0.0
    run_clock = clocks.get("sm_mhz") or sm_max
    # DRAM bytes of the fill kernel per launch: NOT measured in this run -- scaled from the committed ncu --set full
    # capture (one fill launch over `read_pairs_per_launch` read pairs of this refset) to this run's launch size
    traffic, traffic_src = None, None
    for prof_name in ("ncu_kernels_r02.json", "ncu_kernels_r01.json"):
        try:
            with open(os.path.join(ROOT, "profiles", prof_name)) as f:
                prof = json.load(f)
            cap = next(k for k in prof["kernels"] if "fill_bias_kernel" in k["kernel"])
            gb = float(cap["dram__bytes_read.sum"].split()[0]) + float(cap["dram__bytes_write.sum"].split()[0])
            # a launch covers (read pairs) x (reference bases of one part); the step's read-pair x base product is
            # spread over its launches
            launches_per_step = max(agg["batches"] / K, 1)
            cap_rp_bases = float(prof["meta"].get("rp_bases_per_launch") or prof["meta"]["read_pairs_per_launch"] * ref_bases)
            traffic = round(gb * 1e9 / cap_rp_bases * (B / 2.0) * ref_bases / launches_per_step)
            traffic_src = f"scaled from profiles/{prof_name} (ncu --set full of the same kernel and refset), not measured in this run"
            break
        except Exception:
            continue
    roofline = {"bound": "int_dpx", "kernel": "fill_bias_kernel<19>",
                "note": "frac uses SURVEY 8d's unit (2 integer-pipe lane-ops per cell) and exceeds 1 because the kernel needs "
                        "2.16 DPX ops per s16x2 cell PAIR; frac_alu_bound is the honest ceiling of this kernel design "
                        "(2 DPX ops per cell pair, 64 lane-ops/clk/SM)",
                "achieved": round(fill_gcups, 1),
                "peak": round(peak_gcups, 1), "unit": "GCUPS", "frac": round(fill_gcups / peak_gcups, 4),
                "frac_alu_bound": round(fill_gcups / alu_bound_gcups, 4), "alu_bound_peak": round(alu_bound_gcups, 1),
                "peak_def": f"{sms} SMs x {sm_max:.0f} MHz ({peak_kind} sm_max_mhz) x 64 int lane-ops/clk/SM "
                            "(measured: profiles/dpx_microbench_r01.json) / 2 ops per s16x2 cell",
                "frac_at_run_clock": round(fill_gcups / (peak_gcups * run_clock / sm_max), 4),
                "traffic": traffic, "traffic_source": traffic_src,
                "hbm": {"algorithmic_bytes_per_launch": agg["checkpoint_bytes"] / max(agg["batches"], 1),
                        "achieved_gbs": round(agg["checkpoint_bytes"] / 1e9 / (agg["fill_ms"] * 1e-3), 1)
                        if agg["fill_ms"] > 0 else 0.0,
                        "peak_gbs": hbm_peak, "peak_kind": peak_kind,
                        "note": "block records (checkpoints + seams) + tile maxima written by the fill; HBM is the secondary bound"},
                "fill_ms_per_step": round(agg["fill_ms"] / K, 3), "locate_ms_per_step": round(agg["locate_ms"] / K, 3),
                "trace_ms_per_step": round(agg["trace_ms"] / K, 3)}
    line = {"metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(step_ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "s16x2", "data": "synthetic",
            "config": workload_config(B, args.refs_per_gpu, world, len(refs), ref_bases),
            "reads_per_s": round(B / (step_ms * 1e-3), 1),
            "refset_load_ms": round(refset_load_ms, 1),
            "roofline": roofline, "clocks": clocks,
            "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "ms_per_step": round(e2e_ms, 3),
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(agg["launches"]), "max_cells_per_step": int(agg["max_cells"] / K)}
    if world > 1:
        line["host_affinity"] = numa
        line["collective"] = {"impl": "libswb200 swb_comm_allgather_best: ncclAllGather + merge kernel on the engine stream",
                              "bytes_per_rank_per_step": 16 * B, "merged_equals_independent_reduction": merge_ok}
    if not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline_leg(all_refs, reads_pool, os.cpu_count() or 1)
        except Exception as e:  # the baseline is a report, never a reason to lose the GPU numbers
            line["cpu_baseline"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
