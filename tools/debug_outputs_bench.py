#!/usr/bin/env python
"""The debug folder of a resident compare -- region_summary.tsv.gz and region_sequences.tsv.gz -- and what keeping its inputs
costs the pass, on the chr20-shaped workload (BASELINE configs[2], synth.workload_chr20, seed 20) and, with --wgs, on the
whole-genome workload for region_summary only (configs[3], synth.workload_wgs, seed 38).

  passes:      avk_compare_run_resident plain, with AVK_CMP_KEEP_REGION_ROWS, and with rows and AVK_CMP_KEEP_SEQUENCES
               (enable_sequences: the bundle routes every cluster through the team stage);
  summary:     device = avk_compare_region_summary_bgzf; host = avk_compare_download of the rows (with the other per-region and
               per-variant outputs), avk_region_summary_write, avk_bgzf_compress;
  sequences:   device = avk_compare_region_sequences_bgzf; host = avk_region_sequences_write + avk_bgzf_compress over the bundle of
               an avk_compare_batch call with the seq_* outputs (the resident download does not return the bundle, so the
               host path's bundle download is inside that call, whose time is reported beside it).

Both ways must give the same bytes.  After a warm-up of everything, --reps repetitions alternate the device and host paths;
times are wall clock through the Python binding around calls that end in a device synchronise.  The card's name, power
limit and maximum SM clock are read in the same run.

    python tools/debug_outputs_bench.py [--scale 1.0] [--reps 3] [--wgs] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from merge_writers_bench import card, timed  # noqa: E402


def med(rows):
    return {k: statistics.median(r[k] for r in rows) for k in rows[0]}


def run(s, refs, batch, names, reps, sequences):
    from aardvark_b200.batch import CompareOutputs, seq_offsets
    from aardvark_b200.types import CompareConfig
    from aardvark_b200.writers import bgzf_compress, region_sequence_lines, region_sequences_bgzf, region_summary_bgzf, region_summary_lines
    plain, seq_cfg = CompareConfig(enable_sequences=False), CompareConfig(enable_sequences=True)
    s.set_reference(refs)
    s.upload(batch)
    bundle = None
    if sequences:
        off, plen = seq_offsets(batch)
        bundle_out = CompareOutputs(batch, region_metrics=False, seq_off=off, seq_pool_len=plen)

    def passes():
        t = {}
        _, t["pass_plain"] = timed(lambda: s.run_resident(plain))
        _, t["pass_rows"] = timed(lambda: s.run_resident(plain, region_metrics=True))
        if sequences:
            _, t["pass_rows_sequences"] = timed(lambda: s.run_resident(seq_cfg, region_metrics=True, sequences=True))
        return t

    def device():
        t = {}
        summ, t["summary_bgzf"] = timed(lambda: region_summary_bgzf(s, names, region_ids=batch.region_id))
        seqs = None
        if sequences:
            seqs, t["sequences_bgzf"] = timed(lambda: region_sequences_bgzf(s, names, region_ids=batch.region_id))
        return (summ, seqs), t

    def host():
        t = {}
        out, t["summary_download"] = timed(lambda: s.download(CompareOutputs(batch)))
        text, t["summary_format"] = timed(lambda: region_summary_lines(batch, names, out).encode())
        summ, t["summary_bgzf_compress"] = timed(lambda: bgzf_compress(s, text))
        t["summary_total"] = t["summary_download"] + t["summary_format"] + t["summary_bgzf_compress"]
        seqs = None
        if sequences:
            stext, t["sequences_format"] = timed(lambda: region_sequence_lines(batch, names, bundle))
            seqs, t["sequences_bgzf_compress"] = timed(lambda: bgzf_compress(s, stext))
            t["sequences_total"] = t["sequences_format"] + t["sequences_bgzf_compress"]
        return (summ, seqs), t, (len(text), len(stext) if sequences else 0)

    def bundle_call():
        t = {}
        _, t["compare_batch_with_bundle"] = timed(lambda: s.compare_batch(batch, seq_cfg, out=bundle_out))
        s.upload(batch)
        return t

    # warm-up of every shape; the host path reads the rows / bundle of the pass before it
    if sequences:
        bundle_call()
        bundle = bundle_out
    passes()
    want, _, text_bytes = host()
    got, _ = device()
    assert got == want, "device and host outputs differ"
    rows = []
    for _ in range(reps):
        t = bundle_call() if sequences else {}
        t.update(passes())
        d, td = device()
        h, th, _ = host()
        assert d == want and h == want, "device and host outputs differ"
        t.update({"device_" + k: v for k, v in td.items()})
        t.update({"host_" + k: v for k, v in th.items()})
        rows.append(t)
    return {"regions": batch.n_regions, "variants": batch.n_variants,
            "text_bytes": {"region_summary": text_bytes[0], "region_sequences": text_bytes[1]},
            "bgzf_bytes": {"region_summary": len(want[0]), "region_sequences": len(want[1]) if sequences else 0},
            "median_ms": med(rows), "samples_ms": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--wgs", action="store_true", help="also time region_summary on the whole-genome workload")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    from aardvark_b200 import synth
    from aardvark_b200.lib import Solver
    wgs = synth.workload_wgs(scale=args.scale, seed=38, workers=min(16, os.cpu_count() or 1)) if args.wgs else None   # (forks: before CUDA)
    gpu = card()
    s = Solver(0)
    res = {"gpu": gpu, "host_cpus": os.cpu_count(), "reps": args.reps}
    ref, batch = synth.workload_chr20(scale=args.scale, seed=20)
    res["chr20"] = dict(workload=f"chr20-shaped (BASELINE configs[2]) x {args.scale}, seed 20", **run(s, [ref], batch, ["chr20"], args.reps, True))
    if wgs:
        refs, batch = wgs
        res["wgs"] = dict(workload=f"whole genome (BASELINE configs[3]) x {args.scale}, seed 38, region_summary only",
                          **run(s, refs, batch, [f"chr{i + 1}" for i in range(len(refs))], args.reps, False))
    res["note"] = ("wall clock through the Python binding, medians of alternating repetitions after one warm-up; the host path formats "
                   "on one host core and its bgzf_compress includes the text upload and the file download")
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")
    s.close()


if __name__ == "__main__":
    main()
