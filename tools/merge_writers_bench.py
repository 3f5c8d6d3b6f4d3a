#!/usr/bin/env python
"""passing.vcf.gz, regions.bed.gz, failed_regions.bed.gz and the merge summary of a resident merge result, two ways, on the
tools/merge_timing.py workload (BASELINE configs[4]: K = 5 call sets on one chr20-length contig, majority voting, seed 38):

  host path:   avk_merge_download of the result (the batch is already on the host, as after an upload), then
               avk_merge_records_write / avk_merge_regions_write (passing and failed) / avk_merge_summary_write (size query +
               write each, one host core) and avk_bgzf_compress of the three files (text up, deflate on the device, file down);
  device path: avk_merge_records_bgzf, avk_merge_regions_bgzf (passing and failed), avk_merge_summary_counts +
               avk_merge_summary_rows_write (format and deflate on the device, only the files and the distinct keys come down).

Both paths must give the same bytes.  After a warm-up call of each, the two paths alternate for --reps repetitions; each time
is wall clock through the Python binding around calls that end in a device synchronise.  The card's name, power limit and
maximum SM clock are read in the same run.

    python tools/merge_writers_bench.py [--scale 1.0] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LABELS = ["pb", "ilmn", "ont", "hifi", "ul"]
HEADER = (b"##fileformat=VCFv4.2\n##contig=<ID=chr20,length=64444167>\n"
          b'##INFO=<ID=SOURCES,Number=.,Type=String,Description="Inputs the variant was copied from">\n'
          b'##INFO=<ID=MR,Number=1,Type=String,Description="Merge reason">\n'
          b'##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n'
          b'##FORMAT=<ID=RI,Number=1,Type=Integer,Description="Region index">\n'
          b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tSAMPLE\n")


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return r, (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    from aardvark_b200 import synth
    from aardvark_b200.batch import MergeOutputs
    from aardvark_b200.lib import Solver
    from aardvark_b200.types import MergeConfig
    from aardvark_b200.writers import (VariantMerger, bgzf_compress, merge_records_bgzf, merge_regions_bgzf, merge_summary_rows,
                                       merge_summary_text)
    ref, batch = synth.workload_merge(int(synth.CHR20_LEN * args.scale), int(150_000 * args.scale), n_sets=5, seed=38)
    gpu = card()
    s = Solver(0)
    s.set_reference([ref])
    s.merge_upload(batch)
    s.merge_run_resident(MergeConfig(majority_voting_enabled=True))
    names = ["chr20"]

    def host_path():
        t = {}
        out, t["download_result"] = timed(lambda: s.merge_download(MergeOutputs(batch)))
        vm = VariantMerger(batch, out, names, LABELS)
        rec, t["format_records"] = timed(lambda: HEADER + vm.passing_records().encode())
        bed, t["format_regions"] = timed(lambda: vm.regions_bed(True).encode())
        fbed, t["format_failed_regions"] = timed(lambda: vm.regions_bed(False).encode())
        summ, t["format_summary"] = timed(lambda: vm.summary_text())
        files, t["bgzf_compress"] = timed(lambda: [bgzf_compress(s, x) for x in (rec, bed, fbed)])
        t["total"] = sum(t.values())
        return files + [summ], t, [len(rec), len(bed), len(fbed)]

    def device_path():
        t = {}
        rec, t["records_bgzf"] = timed(lambda: merge_records_bgzf(s, names, LABELS, HEADER, batch.region_id))
        bed, t["regions_bgzf"] = timed(lambda: merge_regions_bgzf(s, names, True, batch.region_id))
        fbed, t["failed_regions_bgzf"] = timed(lambda: merge_regions_bgzf(s, names, False, batch.region_id))
        rows, t["summary_counts"] = timed(lambda: merge_summary_rows(s))
        summ, t["summary_rows_write"] = timed(lambda: merge_summary_text(rows, 5, LABELS))
        t["total"] = sum(t.values())
        return [rec, bed, fbed, summ], t, int(rows.size)

    want, _, text_bytes = host_path()                         # warm-up (buffers, module load)
    got, _, n_rows = device_path()
    assert got == want, "device and host outputs differ"
    host, dev = [], []
    for _ in range(args.reps):
        h, th, _ = host_path()
        d, td, _ = device_path()
        assert h == want and d == want, "device and host outputs differ"
        host.append(th)
        dev.append(td)
    med = lambda rows: {k: statistics.median(r[k] for r in rows) for k in rows[0]}
    res = {"workload": f"merge x5 (BASELINE configs[4]), chr20 length x {args.scale}, majority voting, seed 38",
           "regions": batch.n_regions, "variants": batch.n_variants, "gpu": gpu, "host_cpus": os.cpu_count(), "reps": args.reps,
           "text_bytes": {"passing_vcf": text_bytes[0], "regions_bed": text_bytes[1], "failed_regions_bed": text_bytes[2]},
           "bgzf_bytes": {"passing_vcf": len(want[0]), "regions_bed": len(want[1]), "failed_regions_bed": len(want[2])},
           "summary_rows": n_rows,
           "host_path_ms": med(host), "device_path_ms": med(dev), "host_samples_ms": host, "device_samples_ms": dev,
           "note": "wall clock through the Python binding, medians of alternating repetitions after one warm-up of each path; the host "
                   "path formats on one host core and its bgzf_compress includes the text upload and the file download"}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")
    s.close()


if __name__ == "__main__":
    main()
