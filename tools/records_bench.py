#!/usr/bin/env python
"""truth.vcf.gz / query.vcf.gz of a resident compare result, two ways, on the WGS workload (BASELINE configs[2], seed 38):

  host path:   avk_compare_download of the labels, avk_vcf_records_write (size query + write, one host core),
               avk_bgzf_compress (text up, deflate on the device, file down);
  device path: avk_compare_records_bgzf (format and deflate on the device, only the file comes down).

Both files must be byte-equal.  Wall-clock times per side are the median of --reps calls, each ending in a device synchronise
(every library call returns after its copy to the host).  A separate, untimed call per side under torch.profiler gives the
device time of each kernel of the device path: the format phase (count, length and write passes and their scans) and the
compress phase (k_bgzf_deflate, k_bgzf_pack).  The card's name and power limit are read in the same run.

    python tools/records_bench.py [--scale 1.0] [--reps 3] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

NAMES = [f"chr{i}" for i in range(1, 23)] + ["chrX", "chrY"]


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def header(refs):
    lines = [b"##fileformat=VCFv4.2"] + [b"##contig=<ID=%s,length=%d>" % (n.encode(), r.size) for n, r in zip(NAMES, refs)]
    lines += [b'##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">',
              b'##FORMAT=<ID=BD,Number=1,Type=String,Description="Benchmark classification">',
              b'##FORMAT=<ID=EA,Number=1,Type=Integer,Description="Expected alleles">',
              b'##FORMAT=<ID=OA,Number=1,Type=Integer,Description="Observed alleles">',
              b'##FORMAT=<ID=RI,Number=1,Type=Integer,Description="Region index">',
              b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tSAMPLE"]
    return b"\n".join(lines) + b"\n"


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
    from aardvark_b200 import abi, synth
    workers = min(24, os.cpu_count() or 1)
    refs, batch = synth.workload_wgs(scale=args.scale, seed=38, workers=workers)     # before CUDA is initialised (forks)

    from aardvark_b200.batch import CompareOutputs
    from aardvark_b200.lib import Solver
    from aardvark_b200.writers import _bind, bgzf_compress, vcf_records_bgzf
    gpu = card()
    s = Solver(0)
    s.set_reference(refs, NAMES)
    s.upload(batch)
    s.run_resident()
    hdr = header(refs)
    lib = _bind()
    cb = batch.to_c()
    names = (C.c_char_p * len(NAMES))(*[n.encode() for n in NAMES])

    def download():
        out = CompareOutputs(batch, region_metrics=False)
        s.download(out)
        return out

    def host_format(out, side):
        n = C.c_uint64(0)
        args_ = lambda buf, cap: (C.byref(cb), side, names, len(NAMES), abi.ptr(out.var_class), abi.ptr(out.var_expected),
                                  abi.ptr(out.var_observed), 0, batch.n_regions, buf, cap, C.byref(n))
        _, t_query = timed(lambda: lib.avk_vcf_records_write(*args_(None, 0)))
        buf = np.empty(len(hdr) + int(n.value), dtype=np.uint8)
        buf[:len(hdr)] = np.frombuffer(hdr, dtype=np.uint8)
        body = buf[len(hdr):]
        rc, t_write = timed(lambda: lib.avk_vcf_records_write(*args_(body.ctypes.data_as(C.c_char_p), body.size)))
        assert rc == 0
        return buf.tobytes(), t_query, t_write

    sides = {}
    for side in (0, 1):
        device_file = vcf_records_bgzf(s, side, NAMES, hdr, batch.region_id)                   # warm-up (buffers, module load)
        rows = []
        for _ in range(args.reps):
            out, t_dl = timed(download)
            text, t_q, t_w = host_format(out, side)
            host_file, t_gz = timed(lambda: bgzf_compress(s, text))
            dev, t_dev = timed(lambda: vcf_records_bgzf(s, side, NAMES, hdr, batch.region_id))
            assert dev == host_file == device_file, f"side {side}: device and host files differ"
            rows.append((t_dl, t_q, t_w, t_gz, t_dev))
        med = [statistics.median(r[k] for r in rows) for k in range(5)]
        sides["truth" if side == 0 else "query"] = {
            "records": int(text.count(b"\n") - hdr.count(b"\n")), "text_bytes": len(text), "bgzf_bytes": len(device_file),
            "host_path_ms": {"download_labels": med[0], "format_size_query": med[1], "format_write": med[2], "bgzf_compress": med[3],
                             "total": med[0] + med[1] + med[2] + med[3]},
            "device_path_ms": {"total": med[4]},
            "samples_ms": [list(r) for r in rows],
        }

    profile = {}
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile as tprofile
        for side in (0, 1):
            with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                vcf_records_bgzf(s, side, NAMES, hdr, batch.region_id)
                torch.cuda.synchronize()
            k = {}
            for ev in prof.key_averages():
                dt = getattr(ev, "device_time_total", None)
                if dt is None:
                    dt = getattr(ev, "cuda_time_total", 0)
                if dt:
                    k[ev.key] = k.get(ev.key, 0.0) + dt / 1e3
            fmt = sum(v for n, v in k.items() if "k_rw_" in n or "Scan" in n)
            gz = sum(v for n, v in k.items() if "k_bgzf_" in n)
            copies = sum(v for n, v in k.items() if "Memcpy" in n or "Memset" in n)
            profile["truth" if side == 0 else "query"] = {"format_kernels_ms": fmt, "compress_kernels_ms": gz, "copies_ms": copies, "by_name_ms": k}
    except Exception as e:                               # noqa: BLE001 - the wall-clock result above stands on its own
        profile = {"error": repr(e)}

    res = {"workload": f"WGS HG002-like synthetic compare (BASELINE configs[2]), scale={args.scale}, seed=38+contig",
           "regions": batch.n_regions, "variants": batch.n_variants, "gpu": gpu, "host_cpus": os.cpu_count(), "reps": args.reps,
           "sides": sides, "device_path_kernels": profile,
           "note": "wall clock through the Python binding, medians; the host path's format runs on one host core; "
                   "bgzf_compress includes the text upload and the file download, the device path the file download"}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")
    s.close()


if __name__ == "__main__":
    main()
