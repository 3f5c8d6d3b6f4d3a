#!/usr/bin/env python
"""bench.py -- variant clusters/sec and whole-genome compare time through the solve phase (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --config chr20|sv|wgs [--scale F]        (default: wgs, scale 1.0)

A "step" is one pass of the hot path (alt_ed + cluster digests + per-cluster solve + summary counters) over ONE batch:
the synthetic whole-genome HG002-like compare of BASELINE.json configs[2] -- 24 contigs with GRCh38 lengths (3.09 Gbp),
~4.95 M variants per side, ~3.95 M clusters (the phase the reference times as "Comparing regions", src/main.rs:250-272).
STRONG scaling: the same genome at every N; the region_id-ordered cluster list is cut into N contiguous bins
(avk_partition_regions) and rank r solves bin r with no data-path collective; one NCCL gather (grouped send/recv over
NVLink) brings the per-region / per-variant result arrays and the summary counters to rank 0.

  value  clusters/s with the batch already resident in HBM: K passes, --in-flight M of them at a time on every GPU (one
         context = lane + one host thread per pass in flight, avk_create_lane; each lane holds its own copy of the bin, the
         reference is shared) -- a pass ends with its slowest clusters, and passes in flight fill each other's tails.
         Device time of the slowest rank between CUDA events around the K passes.
  single_pass  the same with ONE pass at a time, L2 flushed between steps (CUDA events on the library's stream): the
         latency of one batch, and the figure phases_ms / roofline / int_roofline describe
  e2e    clusters/s through the C ABI with HOST (pinned) buffers, wall clock: H2D of the bin, kernels, the gather
         (N > 1) and the D2H of status / ed / per-variant labels / summary counters inside the timed region; at N = 1
         M calls are in flight (one lane each), e2e.single_call_ms is one call at a time
         => e2e.seconds_per_genome (single call) is the "WGS compare wall-time" half of the metric
  --impl reference: the CPU restatement of the reference path (oracle "port"; the reference is Rust and cannot be
         built here) on the SAME whole batch, OpenMP over clusters on ALL host cores, whatever N is.

  --dump-outputs DIR  after the timed steps, write what the last step returned to its caller as DIR/<name>.npy (see
         dump_outputs); the workload is seeded, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "variant_clusters_per_sec"
UNIT = "clusters/s"


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def workload(config, scale, workers):
    """([contig arrays], RegionBatch, description).  Called before CUDA is initialised (forks workers)."""
    from aardvark_b200 import synth
    if config == "wgs":
        refs, batch = synth.workload_wgs(scale=scale, seed=38, workers=workers)
        return refs, batch, (f"WGS HG002-like synthetic compare (BASELINE configs[2]): 24 contigs with GRCh38 lengths, "
                             f"{sum(r.size for r in refs) / 1e9:.2f} Gbp, scale={scale}, seed=38+contig")
    if config == "chr20":
        ref, batch = synth.workload_chr20(scale=scale, seed=20)
        return [ref], batch, f"chr20-scale synthetic compare (BASELINE configs[1]), scale={scale}, seed=20"
    if config == "sv":
        ref, batch = synth.workload_sv(scale=scale, seed=4)
        return [ref], batch, f"SV / long-indel heavy synthetic compare (BASELINE configs[3]), scale={scale}, seed=4"
    raise SystemExit(f"unknown --config {config}")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(prefix="avk_clocks_", suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def pinned_copy(arr):
    import torch
    t = torch.from_numpy(np.array(arr, copy=True)).pin_memory()
    return t.numpy()


def pin_batch(batch):
    from aardvark_b200.batch import RegionBatch
    f = lambda a: pinned_copy(a)
    return RegionBatch(batch.n_inputs, f(batch.region_id), f(batch.contig), f(batch.start), f(batch.end), f(batch.var_off),
                       f(batch.position), f(batch.variant_type), f(batch.zygosity), f(batch.raw_allele_space),
                       f(batch.allele_off), f(batch.a0_len), f(batch.a1_len), f(batch.allele_pool))


def bin_h2d_bytes(batch, lo, hi):
    """Bytes the library uploads for bin [lo, hi) (region_id stays on the host)."""
    k = batch.n_inputs
    v0, v1 = int(batch.var_off[lo * k]), int(batch.var_off[hi * k])
    pool = 0
    if v1 > v0:
        pool = int(batch.allele_off[v1 - 1]) + int(batch.a0_len[v1 - 1]) + int(batch.a1_len[v1 - 1]) - int(batch.allele_off[v0])
    return (hi - lo) * 12 + ((hi - lo) * k + 1) * 8 + (v1 - v0) * 22 + pool


DUMP_SAMPLE = 1 << 20        # indices kept per axis (regions, variants): the dump stays below 64 MB at any scale


def dump_outputs(out_dir, arrays, n_regions, n_variants):
    """Write a compare call's outputs as <out_dir>/<name>.npy.  `arrays`: name -> array over regions, over variants or
    whole-batch (totals, block counts).  An axis longer than DUMP_SAMPLE keeps a fixed, seeded sample of its indices,
    written as region_index / variant_index.  Small codes are stored as float32, edit distances, counters and indices as
    float64 (both exact for the integers they hold)."""
    os.makedirs(out_dir, exist_ok=True)
    idx = {}
    for axis, n in (("region", n_regions), ("variant", n_variants)):
        ix = np.arange(n) if n <= DUMP_SAMPLE else np.sort(np.random.default_rng(12345).choice(n, DUMP_SAMPLE, replace=False))
        idx[axis] = ix
        np.save(os.path.join(out_dir, f"{axis}_index.npy"), ix.astype(np.float64))
    for name, a in arrays.items():
        a = np.asarray(a)
        axis = "region" if name in ("status", "ed1", "ed2", "type_mask") else "variant" if name.startswith("var_") else None
        if axis is not None:
            a = a[:n_regions if axis == "region" else n_variants][idx[axis]]
        dt = np.float32 if name in ("status", "type_mask", "totals_mask") or name.startswith("var_") else np.float64
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(dt))


def compare_out_arrays(out):
    """The arrays of a CompareOutputs (region_metrics=False) that bench.py dumps."""
    return {f: getattr(out, f) for f in ("status", "ed1", "ed2", "type_mask", "var_expected", "var_observed", "var_class",
                                         "totals", "totals_mask", "solved_blocks", "error_blocks")}


def run_reference(args, rank):
    """--impl reference: the reference's CPU path (oracle port; the Rust crate cannot be built here) on the SAME whole
    batch the GPU arm solves, on all host cores (torchrun's OMP_NUM_THREADS=1 is overridden explicitly)."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as orc
    from aardvark_b200 import abi
    cores = host_cores()
    refs, batch, desc = workload(args.config, args.scale, cores)
    cfg = abi.CompareCfg(50, 0, 0, 0)
    for _ in range(min(args.warmup, 1)):
        orc.compare_batch(batch, refs, cfg, n_threads=cores, region_metrics=False)
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        out = orc.compare_batch(batch, refs, cfg, n_threads=cores, region_metrics=False)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, compare_out_arrays(out), batch.n_regions, batch.n_variants)
    v = batch.n_regions * steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": desc, "regions_per_step": batch.n_regions, "variants_per_step": batch.n_variants, "max_branch_factor": 50},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"the whole batch ({batch.n_regions} clusters) x {steps} steps, OpenMP dynamic over clusters, "
                                   "solve phase only; oracle built -O3 -march=native -flto on this host"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "seconds_per_genome": dt / steps},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="wgs", choices=["wgs", "chr20", "sv"])
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the named workload (tests only; default = full)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--in-flight", type=int, default=4,
                    help="passes in flight per GPU (one context + host thread each, avk_create_lane); 1 = one pass at a time")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, a seeded sample of "
                         "regions and variants when there are more than 2^20 of either)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    # ---------------- workload: generated before CUDA is touched (forked workers), identical on every rank --------------
    t_gen = time.perf_counter()
    refs, batch, desc = workload(args.config, args.scale, max(1, host_cores() // world))
    t_gen = time.perf_counter() - t_gen

    import torch
    import torch.distributed as dist
    from aardvark_b200.batch import CompareOutputs
    from aardvark_b200.dist import DeviceGather, partition_regions
    from aardvark_b200.lib import Solver
    from aardvark_b200.types import CompareConfig

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: aardvark_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # stdout carries ONE JSON line: NCCL's version banner (NCCL_DEBUG=VERSION) would land there too
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    k = batch.n_inputs
    bins = partition_regions(batch, world)
    var_bins = [(int(batch.var_off[lo * k]), int(batch.var_off[hi * k])) for lo, hi in bins]
    lo, hi = bins[rank]
    n_bin = hi - lo
    solver = Solver(local_rank)
    # this rank's GPU holds the contigs its bin touches (all of them at N = 1)
    used = set(np.unique(batch.contig[lo:hi]).tolist())
    solver.set_reference([r if i in used else r[:0] for i, r in enumerate(refs)])
    cfg = CompareConfig(enable_sequences=False)
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- resident leg: `value` -------------------------------------------------------
    solver.upload(batch, lo, hi)
    for _ in range(args.warmup):
        solver.run_resident(cfg)
    launches0 = solver.launch_count()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    dev_ms, pipe_ms = 0.0, 0.0
    tier_ms = np.zeros(3)
    for _ in range(args.steps):
        l2_flush.zero_()
        torch.cuda.synchronize()
        solver.run_resident(cfg)           # returns after its CUDA events (own stream) have completed
        tm = solver.last_timings_ms()
        dev_ms += tm["total"]
        pipe_ms += tm["search"]
        tier_ms += np.array(solver.last_tier_ms())
    barrier()
    launches = solver.launch_count() - launches0
    work = solver.last_work()
    resident_out = CompareOutputs(batch, region_metrics=False)
    solver.download(resident_out)

    # ---------------- in-flight leg: M passes over the resident bin at the same time -------------------
    # One context (lane) and one host thread per pass; the lanes share the owner's resident reference and hold their own copy
    # of the bin, so what the passes in flight read is M x the bin: the count is raised until that is twice the L2, and a
    # bin too small for it keeps the single, L2-flushed pass above as its number.
    import threading
    bin_bytes = bin_h2d_bytes(batch, lo, hi)
    L2_BYTES = 126 << 20
    m_req = max(1, args.in_flight)
    M = m_req if m_req == 1 else min(8, max(m_req, -(-2 * L2_BYTES // max(bin_bytes, 1))))
    if M > 1 and M * bin_bytes < 2 * L2_BYTES:
        M = 1
    if world > 1:                                  # the same M on every rank
        mt = torch.tensor([M], dtype=torch.int64, device="cuda")
        dist.all_reduce(mt, op=dist.ReduceOp.MIN)
        M = int(mt.item())
    lanes = [solver] + [solver.lane() for _ in range(M - 1)]
    flight_ms = None

    def in_flight(fn, total):
        """`total` calls of fn(lane index) spread over the lanes' threads; returns device milliseconds (CUDA events around it)."""
        counts = [total // M + (1 if i < total % M else 0) for i in range(M)]
        errs = []

        def work(i):
            try:
                for _ in range(counts[i]):
                    fn(i)
            except Exception as e:      # noqa: BLE001
                errs.append(e)
        th = [threading.Thread(target=work, args=(i,)) for i in range(M)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for t in th:
            t.start()
        for t in th:
            t.join()
        torch.cuda.synchronize()
        e1.record()
        e1.synchronize()
        barrier()
        if errs:
            raise errs[0]
        return e0.elapsed_time(e1)

    if M > 1:
        for ln in lanes[1:]:
            ln.upload(batch, lo, hi)
            ln.run_resident(cfg)
        in_flight(lambda i: lanes[i].run_resident(cfg), max(args.warmup, M))
        l0 = sum(ln.launch_count() for ln in lanes)
        flight_ms = in_flight(lambda i: lanes[i].run_resident(cfg), args.steps)
        launches = sum(ln.launch_count() for ln in lanes) - l0
        for ln in lanes[1:]:
            o = CompareOutputs(batch, region_metrics=False)
            ln.download(o)
            assert o.diff(resident_out) == [], "a lane's resident result differs from the owner's"

    # ---------------- e2e leg: host buffers through the C ABI ----------------------------------------
    pbatch = pin_batch(batch)
    out = CompareOutputs(pbatch, region_metrics=False)
    OUT_FIELDS = ("status", "ed1", "ed2", "type_mask", "var_expected", "var_observed", "var_class")
    for f in OUT_FIELDS:
        setattr(out, f, pinned_copy(getattr(out, f)))
    gather = DeviceGather(bins, var_bins, rank) if world > 1 else None
    merged = None

    def e2e_step():
        nonlocal merged
        if world == 1:
            solver.compare_batch(pbatch, cfg, out=out)                 # H2D + kernels + D2H in one C-ABI call
        else:
            solver.upload(pbatch, lo, hi)                              # H2D of this rank's bin
            solver.run_resident(cfg)
            merged = gather.gather(solver.result_device_view())        # ONE NCCL gather to rank 0 + its D2H

    for _ in range(3):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    e2e_single_s = e2e_s
    if world == 1 and M > 1:
        # the same C-ABI call with M call sets in flight (one context + host thread each; every call copies its inputs
        # from pinned host memory and its results back); the serial figure above stays as the single-call wall time
        outs = [out]
        for _ in lanes[1:]:
            o = CompareOutputs(pbatch, region_metrics=False)
            for f in OUT_FIELDS:
                setattr(o, f, pinned_copy(getattr(o, f)))
            outs.append(o)
        in_flight(lambda i: lanes[i].compare_batch(pbatch, cfg, out=outs[i]), 2 * M)
        t0 = time.perf_counter()
        in_flight(lambda i: lanes[i].compare_batch(pbatch, cfg, out=outs[i]), args.steps)
        e2e_s = time.perf_counter() - t0
        for o in outs[1:]:
            assert o.diff(resident_out) == [], "an in-flight e2e result differs from the resident one"
    clocks = sampler.stop() if sampler else None
    h2d = bin_h2d_bytes(batch, lo, hi)
    if world == 1:
        assert out.diff(resident_out) == [], "e2e and resident outputs differ"
        d2h = sum(getattr(out, f).nbytes for f in OUT_FIELDS) + out.totals.nbytes + 24
        solved, errors = int(out.solved_blocks[0]), int(out.error_blocks[0])
    else:
        d2h = gather.d2h_bytes() if rank == 0 else 0
        solved = errors = 0
        if rank == 0:
            solved, errors = merged["solved"], merged["errors"]
            for f in OUT_FIELDS:       # this rank's bin of the gathered arrays == its own resident result
                a, b = ((var_bins[0][0], var_bins[0][1]) if f.startswith("var_") else (lo, hi))
                assert np.array_equal(merged[f][a:b], getattr(resident_out, f)[a:b]), f"gathered {f} differs from the resident result"
    if args.dump_outputs and rank == 0:
        # the last e2e step's results as its caller receives them (N > 1: the arrays gathered on rank 0)
        if world == 1:
            dumped = compare_out_arrays(out)
        else:
            dumped = {f: merged[f] for f in OUT_FIELDS}
            dumped.update(totals=merged["totals"], totals_mask=np.array([merged["totals_mask"]]),
                          solved_blocks=np.array([merged["solved"]]), error_blocks=np.array([merged["errors"]]))
        dump_outputs(args.dump_outputs, dumped, batch.n_regions, batch.n_variants)

    # ---------------- aggregate over ranks: max time, summed bytes --------------------------------
    stats = torch.tensor([dev_ms, e2e_s * 1e3, pipe_ms, flight_ms if flight_ms is not None else dev_ms, e2e_single_s * 1e3],
                         dtype=torch.float64, device="cuda")
    counts = torch.tensor([n_bin, h2d, d2h, launches], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    dev_ms_max, e2e_ms_max, pipe_ms_max, flight_ms_max, e2e_single_ms_max = (float(x) for x in stats.tolist())
    n_solved_regions, h2d_all, d2h_all, launches_all = (int(x) for x in counts.tolist())
    assert n_solved_regions == batch.n_regions

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        k_ms = pipe_ms / args.steps                        # rank 0's compare pipeline (all solver kernels between prepare and fold)
        int_peak = solver.int_peak_ops_per_s()
        int_ops = 6 * work["cells"] + 4 * ((work["matched_bases"] + 15) // 16)
        line = {
            "metric": METRIC, "value": batch.n_regions * args.steps / (flight_ms_max * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": flight_ms_max / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": desc, "regions_per_step": batch.n_regions, "variants_per_step": batch.n_variants,
                       "max_branch_factor": 50,
                       "passes_in_flight": M,
                       "l2": (f"{M} passes in flight per GPU, each on its own copy of the bin ({bin_bytes >> 20} MiB) + the shared reference: "
                              f"{M * bin_bytes >> 20} MiB of inputs in flight, larger than the 126 MiB L2; single_pass is flushed (256 MiB write) between steps")
                             if M > 1 else "flushed between timed steps (256 MiB write)",
                       "solved_blocks": solved, "error_blocks": errors,
                       "partition": f"{world} contiguous region bin(s) balanced by the cost proxy, no data-path collective; "
                                    "single NCCL gather of results to rank 0 in e2e",
                       "regions_per_rank": [b - a for a, b in bins], "generation_s": round(t_gen, 1)},
            # value / ms_per_step: `steps` passes, M at a time; single_pass: one pass at a time (the latency of one batch)
            "single_pass": {"value": batch.n_regions * args.steps / (dev_ms_max * 1e-3), "unit": UNIT, "ms_per_step": dev_ms_max / args.steps},
            "e2e": {"value": batch.n_regions * args.steps / (e2e_ms_max * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": h2d_all, "d2h_bytes_per_step": d2h_all, "ms_per_step": e2e_ms_max / args.steps,
                    "calls_in_flight": M if world == 1 else 1,
                    "single_call_ms": e2e_single_ms_max / args.steps,
                    "seconds_per_genome": e2e_single_ms_max / args.steps / 1e3},
            "gpu_launches": launches_all,
            # executed on the device (closed forms and pruned searches do less than the reference algorithm);
            # replaced below by the reference algorithm's own counts when the CPU leg runs
            "int_roofline": {"achieved_gops": int_ops / (k_ms * 1e-3) / 1e9, "peak_gops": int_peak / 1e9,
                             "frac": int_ops / (k_ms * 1e-3) / int_peak, "algorithmic_int_ops": int_ops,
                             "ops_counted_by": "device counters (work actually executed by rank 0's bin)",
                             "cells": work["cells"], "matched_bases": work["matched_bases"],
                             "search_pops": work["search_pops"], "exact_pops": work["exact_pops"],
                             "peak_source": "measured live (avk_int_peak: add/max/xor chains)"},
            "phases_ms": {"alt_ed+digests": (dev_ms - pipe_ms) / args.steps, "solver_pipeline": k_ms,
                          "closed_form+dense_stage": float(tier_ms[0]) / args.steps,
                          "search+score+27KB_stage": float(tier_ms[1]) / args.steps, "2MB_stage": float(tier_ms[2]) / args.steps},
            "clocks": clocks,
        }
        alg_bytes = None
        if not args.no_cpu_baseline and world == 1:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import oracle_py as orc
            from aardvark_b200.lib import compare_cfg
            threads = host_cores()
            best = None
            cpu_out = None
            reps = 3
            for _ in range(reps):
                t0 = time.perf_counter()
                cpu_out = orc.compare_batch(batch, refs, compare_cfg(cfg), n_threads=threads, region_metrics=False)
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            # SURVEY 8(d): algorithmic work = what the reference algorithm computes, counted by the CPU restatement
            _, cw = orc.compare_batch(batch, refs, compare_cfg(cfg), n_threads=threads, region_metrics=False, work=True)
            ref_ops = 6 * cw["cells"] + 4 * ((cw["matched_bases"] + 15) // 16)
            alg_bytes = cw["alg_bytes"]
            ir = line["int_roofline"]
            ir.update({"device_executed": {kk: ir[kk] for kk in ("algorithmic_int_ops", "cells", "matched_bases", "search_pops", "exact_pops")},
                       "achieved_gops": ref_ops / (k_ms * 1e-3) / 1e9, "frac": ref_ops / (k_ms * 1e-3) / int_peak,
                       "frac_passes_in_flight": ref_ops / (flight_ms_max / args.steps * 1e-3) / int_peak,
                       "algorithmic_int_ops": ref_ops, "cells": cw["cells"], "matched_bases": cw["matched_bases"],
                       "search_pops": cw["search_pops"], "exact_pops": cw["exact_pops"], "alignments": cw["alignments"],
                       "ops_counted_by": "CPU restatement of the reference algorithm (6*cells + 4*ceil(matched/16))"})
            line["cpu_baseline"] = {"value": batch.n_regions / best, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"the whole batch ({batch.n_regions} clusters), best of {reps}, "
                                              "OpenMP dynamic over clusters, solve phase only",
                                    "seconds_per_genome": best,
                                    "matches_gpu_bit_exact": out.diff(cpu_out) == []}
        traffic, traffic_src = None, None
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "r2_pipeline_traffic.json")))
            if prof.get("config") == args.config and abs(prof.get("scale", -1) - args.scale) < 1e-9:
                traffic, traffic_src = prof.get("dram_bytes_per_step"), prof.get("source")
        except (OSError, ValueError):
            pass
        if alg_bytes is not None:
            achieved = alg_bytes / (k_ms * 1e-3) / 1e9
            line["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                                "traffic": traffic, "traffic_source": traffic_src, "kernel": "compare pipeline (solver kernels of one pass)",
                                "kernel_ms": k_ms, "measured_in": "single_pass leg: one pass at a time, CUDA events on the library's stream",
                                "achieved_passes_in_flight": alg_bytes / (flight_ms_max / args.steps * 1e-3) / 1e9,
                                "frac_passes_in_flight": alg_bytes / (flight_ms_max / args.steps * 1e-3) / 1e9 / hbm_peak,
                                "algorithmic_bytes": alg_bytes,
                                "algorithmic_bytes_definition": "SURVEY 8(d): sum over the reference algorithm's global alignments of "
                                                                "ceil(|a|/4) + ceil(|b|/4) + 8, counted by the CPU restatement",
                                "peak_source": peak_src,
                                "note": "integer DP: the binding roof is the INT32 ALU pipe / latency, see int_roofline"}
        else:
            line["roofline"] = {"bound": "hbm", "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None, "traffic": traffic,
                                "kernel": "compare pipeline", "kernel_ms": k_ms, "peak_source": peak_src,
                                "note": "algorithmic bytes are counted by the CPU leg, which runs at N = 1 only"}
        print(json.dumps(line))
    for ln in reversed(lanes):
        ln.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
