#!/usr/bin/env python
"""Stratified compare passes on the WGS workload (BASELINE configs[2], seed 38) with seeded GIAB-like strata of 8, 32 and 64
strata per set: this build against an earlier build of the library (--parent-lib), alternated in one process on one GPU.

Per strata set:
  resident_plain_ms    avk_compare_run_resident, no flag                               (this build)
  resident_strata_ms   avk_compare_run_resident with AVK_CMP_STRATA                   (this build)
  batch_lookup_ms      avk_compare_batch, strata through the device lookup            (this build and the parent)
  batch_list_ms        avk_compare_batch, strata from a membership list              (this build and the parent)
Times are device time of the pass (CUDA events from the first kernel to the end of the summary folds, avk_last_timings
[4], cooperative tiers included), medians over --reps passes after a warm-up pass; the batch calls alternate the two builds
call by call.  Both batch calls ask for no per-region rows (region_metrics NULL), as summary.tsv needs none.
Memory: device memory a fresh context holds after one stratified avk_compare_batch (its buffers only grow, so this is the
peak of the call), read with cudaMemGetInfo before and after, for both builds.
Exactness, in the same run: strat_totals of the resident pass, of the batch call with the lookup and of the batch call with
the list built from the resident pass's masks are equal, for both builds; on the 64-stratum set they equal the CPU oracle
(OpenMP, membership list from the same masks).  The card's name and power limit are read in the same run.

    python tools/strata_bench.py --parent-lib PATH [--scale 1.0] [--reps 5] [--out profiles/r3_strata_bench.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import numpy as np  # noqa: E402

NAMES = [f"chr{i}" for i in range(1, 23)] + ["chrX", "chrY"]


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def giab_like(lens, n_strata, seed):
    """per stratum, per contig: (first, last) 0-based inclusive.  Mix: n/8 dense sets (1 Mbp blocks covering ~90 % of each
    contig), n/8 sparse sets (~1 interval per 2 Mbp, 1-20 kbp long), the rest many short intervals (50 bp - 5 kbp, ~8 per
    100 kbp, like repeat or low-complexity sets).  Most clusters lie in every dense set and in some short ones."""
    rng = np.random.default_rng(seed)
    n_dense = max(1, n_strata // 8)
    n_sparse = max(1, n_strata // 8)
    strata = []
    for s in range(n_strata):
        per = []
        for L in lens:
            if s < n_dense:
                b = np.arange(0, L, 1_000_000, dtype=np.int64)
                keep = rng.random(b.size) < 0.9
                f, e = b[keep] + rng.integers(0, 20_000, keep.sum()), np.minimum(b[keep] + 1_000_000, L)
            else:
                k = max(1, int(L / (2_000_000 if s < n_dense + n_sparse else 12_500)))
                lo_len, hi_len = (1_000, 20_000) if s < n_dense + n_sparse else (50, 5_000)
                f = rng.integers(0, L, k)
                e = np.minimum(f + np.exp(rng.uniform(np.log(lo_len), np.log(hi_len), k)).astype(np.int64), L)
            per.append((f.astype(np.uint32), (e - 1).astype(np.uint32)))
        strata.append(per)
    return strata


def strat_intervals(strata, n_contigs):
    from aardvark_b200.batch import StratIntervals
    st = StratIntervals.__new__(StratIntervals)
    st.n_strata, st.n_contigs = len(strata), n_contigs
    sizes = [f.size for per in strata for (f, _) in per]
    st.off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    st.first = np.concatenate([f for per in strata for (f, _) in per]).astype(np.uint32)
    st.last = np.concatenate([la for per in strata for (_, la) in per]).astype(np.uint32)
    return st


def membership(masks):
    bits = ((masks[:, None] >> np.arange(64, dtype=np.uint64)) & np.uint64(1)).astype(bool)
    r, s = np.nonzero(bits)
    off = np.zeros(masks.size + 1, dtype=np.uint64)
    np.add.at(off, r + 1, 1)
    return np.cumsum(off).astype(np.uint64), (s.astype(np.uint32) if s.size else np.zeros(1, np.uint32))


def open_solver(libh):
    from aardvark_b200.lib import AvkError, Solver
    s = Solver.__new__(Solver)
    s._lib, s._ctx, s.contig_index, s._contigs = libh, C.c_void_p(), {}, []
    if libh.avk_create(0, C.byref(s._ctx)) != 0:
        raise AvkError("avk_create failed")
    return s


def load_parent(path):
    from aardvark_b200 import lib as L
    saved = L._LIB, L.SO_PATH
    L._LIB, L.SO_PATH = None, os.path.abspath(path)
    try:
        return L.load()
    finally:
        L._LIB, L.SO_PATH = saved


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True, help="libaardvark_b200.so built from the parent commit")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sets", default="8,32,64")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from aardvark_b200 import synth
    workers = min(24, os.cpu_count() or 1)
    refs, batch = synth.workload_wgs(scale=args.scale, seed=38, workers=workers)     # before CUDA is initialised (forks)

    import torch
    import oracle_py as orc
    from aardvark_b200.batch import CompareOutputs
    from aardvark_b200.lib import compare_cfg, load
    from aardvark_b200.types import CompareConfig
    cfg = CompareConfig(enable_sequences=False)
    gpu = card()
    libs = {"this": load(), "parent": load_parent(args.parent_lib)}
    lens = [r.size for r in refs]
    n = batch.n_regions

    def device_ms(s):
        return s.last_timings_ms()["total"]

    def mem_of_call(name, st, kw):
        torch.cuda.synchronize()
        s = open_solver(libs[name])
        s.set_reference(refs, NAMES)
        s.set_stratifications(st)
        free0, _ = torch.cuda.mem_get_info(0)
        s.compare_batch(batch, cfg, region_metrics=False, **kw)
        free1, _ = torch.cuda.mem_get_info(0)
        s.close()
        return (free0 - free1) / 2**20

    res_sets = {}
    for k in [int(x) for x in args.sets.split(",")]:
        strata = giab_like(lens, k, seed=1000 + k)
        st = strat_intervals(strata, len(refs))
        mem = {name: mem_of_call(name, st, dict(n_strata=k, device_strata=True)) for name in ("parent", "this")}
        sol = {name: open_solver(libs[name]) for name in libs}
        for s in sol.values():
            s.set_reference(refs, NAMES)
            s.set_stratifications(st)
        this = sol["this"]
        # resident passes (this build)
        this.upload(batch)
        plain, strat = [], []
        for rep in range(args.reps + 1):
            this.run_resident(cfg)
            t0 = device_ms(this)
            this.run_resident(cfg, strata=True)
            t1 = device_ms(this)
            if rep:
                plain.append(t0)
                strat.append(t1)
        res_out = this.download(CompareOutputs(batch, region_metrics=False, n_strata=k, device_strata=True, containment=True))
        masks = res_out.containment[:n].copy()
        so, si = membership(masks)
        per_region = np.diff(so.astype(np.int64))
        kw = {"lookup": dict(n_strata=k, device_strata=True), "list": dict(strat_off=so, strat_idx=si, n_strata=k)}
        times = {(name, mode): [] for name in libs for mode in kw}
        outs = {}
        for rep in range(args.reps + 1):                      # alternate the builds call by call
            for mode in kw:
                for name in (("parent", "this") if rep % 2 == 0 else ("this", "parent")):
                    o = sol[name].compare_batch(batch, cfg, region_metrics=False, **kw[mode])
                    if rep:
                        times[(name, mode)].append(device_ms(sol[name]))
                    outs[(name, mode)] = o
        for s in sol.values():
            s.close()
        exact = all(np.array_equal(o.strat_totals, res_out.strat_totals) and np.array_equal(o.totals, res_out.totals) for o in outs.values())
        exact = exact and all(np.array_equal(o.status, outs[("parent", "lookup")].status) for o in outs.values())
        row = {
            "n_strata": k, "intervals": int(st.off[-1]),
            "regions_in_0_1_2_3_4plus_strata": [int((per_region == c).sum()) for c in range(4)] + [int((per_region >= 4).sum())],
            "mean_strata_per_region": float(per_region.mean()),
            "resident_plain_ms": statistics.median(plain), "resident_strata_ms": statistics.median(strat),
            "batch_lookup_ms": {"this": statistics.median(times[("this", "lookup")]), "parent": statistics.median(times[("parent", "lookup")])},
            "batch_list_ms": {"this": statistics.median(times[("this", "list")]), "parent": statistics.median(times[("parent", "list")])},
            "batch_lookup_peak_device_mib": mem,
            "strat_totals_equal_resident_lookup_list_both_builds": bool(exact),
            "samples_ms": {"resident_plain": plain, "resident_strata": strat, **{f"batch_{m}_{b}": v for (b, m), v in times.items()}},
        }
        if k == 64:
            cpu = orc.compare_batch(batch, refs, compare_cfg(cfg), region_metrics=False, strat_off=so, strat_idx=si, n_strata=k)
            row["strat_totals_equal_oracle"] = bool(np.array_equal(cpu.strat_totals, res_out.strat_totals) and np.array_equal(cpu.totals, res_out.totals))
        res_sets[str(k)] = row
        print(json.dumps({k2: v for k2, v in row.items() if k2 != "samples_ms"}), file=sys.stderr, flush=True)

    res = {"workload": f"WGS HG002-like synthetic compare (BASELINE configs[2]), scale={args.scale}, seed=38+contig; "
                       "GIAB-like strata seeded 1000 + n_strata (tools/strata_bench.py giab_like)",
           "regions": n, "variants": batch.n_variants, "gpu": gpu, "reps": args.reps, "sets": res_sets,
           "note": "device time per pass (avk_last_timings total), medians; batch calls alternate this build and the parent "
                   "call by call on the same GPU; memory = cudaMemGetInfo delta of a fresh context over one stratified batch call"}
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
