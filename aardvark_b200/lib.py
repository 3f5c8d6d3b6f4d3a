"""ctypes binding of libaardvark_b200.so (the CUDA product) + the host-side operator mirror.

`Solver` is the drop-in for the two call sites the reference parallelises with rayon:

    solve_compare_region(&CompareRegion, &ReferenceGenome, CompareConfig, ..)  src/waffle_solver.rs:122-124
    solve_merge_region(&MultiRegion, &ReferenceGenome, MergeConfig)            src/merge_solver.rs:110

Because the reference materialises all regions first (src/main.rs:217-232), the natural
unit here is the batch: `Solver.compare_batch(RegionBatch)`; the single-region calls
exist for parity with the reference's tests.  There is NO CPU fallback: if the shared
library is missing or no CUDA device is present, construction raises.
"""
import ctypes as C
import os
import shutil
import subprocess
from typing import List, Sequence

import numpy as np

from . import abi
from .batch import CompareOutputs, MergeOutputs, RegionBatch, seq_offsets
from .results import unpack_compare, unpack_merge
from .types import CompareConfig, CompareRegion, MergeConfig, MultiRegion, RegionError

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.path.join(CSRC, "libaardvark_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--shared", "-Xcompiler", "-fPIC"]

_LIB = None


class AvkError(RuntimeError):
    pass


def build(force=False, verbose=False):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, "avk_lib.cu")] + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h")))
    srcs.append(os.path.join(_HERE, "..", "include", "aardvark_b200.h"))
    if not force and os.path.exists(SO_PATH) and os.path.getmtime(SO_PATH) >= max(os.path.getmtime(s) for s in srcs):
        return SO_PATH
    # nvcc is often not on an ordinary user's PATH: fall back to the toolkit's usual locations
    nvcc = shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda", "bin", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO_PATH, srcs[0]]
    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    subprocess.check_call(cmd + ["-ccbin", "/usr/bin/g++"], env=env)
    return SO_PATH


def load():
    """Load the product library; raises loudly when it is not built (no fallback path exists)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(SO_PATH):
        raise AvkError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`; "
                       "aardvark_b200 has no CPU fallback")
    lib = C.CDLL(SO_PATH)
    vp = C.c_void_p
    lib.avk_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.avk_destroy.argtypes = [vp]
    lib.avk_create_lane.argtypes = [vp, C.POINTER(vp)]
    lib.avk_last_error.restype = C.c_char_p
    lib.avk_last_error.argtypes = [vp]
    lib.avk_launch_count.restype = C.c_uint64
    lib.avk_launch_count.argtypes = [vp]
    lib.avk_set_reference.argtypes = [vp, C.c_uint32, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_uint64)]
    lib.avk_compare_batch.argtypes = [vp, C.POINTER(abi.RegionBatch), C.POINTER(abi.CompareCfg), C.POINTER(abi.CompareOut)]
    lib.avk_merge_batch.argtypes = [vp, C.POINTER(abi.RegionBatch), C.POINTER(abi.MergeCfg), C.POINTER(abi.MergeOut)]
    lib.avk_wfa_ed_batch.argtypes = [vp, C.c_uint64, C.POINTER(C.c_uint8), C.c_uint64, C.POINTER(C.c_uint64),
                                     C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32),
                                     C.POINTER(C.c_uint32)]
    lib.avk_compare_seq_offsets.argtypes = [C.POINTER(abi.RegionBatch), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    if hasattr(lib, "avk_build_regions"):   # (older builds used for A/B timing do not have the region builder)
        lib.avk_build_regions.argtypes = [vp, C.POINTER(abi.CallSets), C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        lib.avk_regions_download.argtypes = [vp, C.POINTER(abi.RegionBatch)]
        lib.avk_build_regions_bed.argtypes = [vp, C.POINTER(abi.CallSets), C.POINTER(C.c_uint32), C.POINTER(abi.BedIntervals), C.c_uint32, C.c_uint64,
                                              C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.avk_compare_batch_range.argtypes = [vp, C.POINTER(abi.RegionBatch), C.c_uint64, C.c_uint64, C.POINTER(abi.CompareCfg),
                                            C.POINTER(abi.CompareOut)]
    lib.avk_compare_batch_multi.argtypes = [C.POINTER(vp), C.c_uint32, C.POINTER(abi.RegionBatch), C.POINTER(abi.CompareCfg),
                                            C.POINTER(abi.CompareOut)]
    lib.avk_merge_batch_multi.argtypes = [C.POINTER(vp), C.c_uint32, C.POINTER(abi.RegionBatch), C.POINTER(abi.MergeCfg),
                                          C.POINTER(abi.MergeOut)]
    lib.avk_partition_regions.argtypes = [C.POINTER(abi.RegionBatch), C.c_uint32, C.POINTER(C.c_uint64)]
    lib.avk_compare_upload_range.argtypes = [vp, C.POINTER(abi.RegionBatch), C.c_uint64, C.c_uint64]
    lib.avk_compare_result_device.argtypes = [vp, C.POINTER(abi.CompareDevView)]
    lib.avk_last_tier_overflow.argtypes = [vp, C.POINTER(C.c_uint32)]
    lib.avk_last_tier_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.avk_set_stratifications.argtypes = [vp, C.POINTER(abi.StratIntervals)]
    lib.avk_compare_upload.argtypes = [vp, C.POINTER(abi.RegionBatch)]
    lib.avk_compare_run_resident.argtypes = [vp, C.POINTER(abi.CompareCfg)]
    lib.avk_compare_download.argtypes = [vp, C.POINTER(abi.CompareOut)]
    lib.avk_merge_upload_range.argtypes = [vp, C.POINTER(abi.RegionBatch), C.c_uint64, C.c_uint64]
    lib.avk_merge_run_resident.argtypes = [vp, C.POINTER(abi.MergeCfg)]
    lib.avk_merge_download.argtypes = [vp, C.POINTER(abi.MergeOut)]
    lib.avk_last_timings.argtypes = [vp, C.POINTER(C.c_float)]
    lib.avk_last_work.argtypes = [vp, C.POINTER(abi.WorkCounters)]
    lib.avk_int_peak.argtypes = [vp, C.POINTER(C.c_double)]
    _LIB = lib
    return lib


EXPORTED_SYMBOLS = [
    "avk_create", "avk_destroy", "avk_last_error", "avk_set_reference", "avk_compare_batch", "avk_merge_batch",
    "avk_wfa_ed_batch", "avk_compare_seq_offsets", "avk_compare_upload", "avk_compare_run_resident",
    "avk_compare_download", "avk_build_regions", "avk_build_regions_bed", "avk_regions_download", "avk_summary_write", "avk_vcf_records_write", "avk_vcf_parse", "avk_last_timings", "avk_last_work", "avk_launch_count", "avk_int_peak", "avk_last_tier_overflow", "avk_last_tier_ms",
    "avk_compare_batch_range", "avk_compare_batch_multi", "avk_merge_batch_multi", "avk_partition_regions", "avk_compare_upload_range",
    "avk_compare_result_device", "avk_set_stratifications", "avk_create_lane",
    "avk_merge_records_write", "avk_merge_regions_write", "avk_merge_summary_write", "avk_bgzf_inflate", "avk_vcf_parse_bgzf", "avk_bgzf_compress", "avk_spec_profile",
    "avk_compare_records_bgzf",
    "avk_merge_upload_range", "avk_merge_run_resident", "avk_merge_download", "avk_merge_records_bgzf", "avk_merge_regions_bgzf",
    "avk_merge_summary_counts", "avk_merge_summary_rows_write",
    "avk_region_summary_write", "avk_region_sequences_write", "avk_compare_region_summary_bgzf", "avk_compare_region_sequences_bgzf",
]


def compare_cfg(cfg: CompareConfig, flags: int = 0) -> abi.CompareCfg:
    return abi.CompareCfg(cfg.max_branch_factor, int(cfg.enable_exact_shortcut), int(cfg.enable_sequences), flags,
                          int(getattr(cfg, "exact_gt_max_expansions", 0)))


def partition_regions(batch: RegionBatch, n_bins: int):
    """Contiguous bins [lo, hi) balanced by the library's cost proxy (avk_partition_regions; host only, no GPU needed)."""
    cuts = (C.c_uint64 * (n_bins + 1))()
    cb = batch.to_c()
    rc = load().avk_partition_regions(C.byref(cb), n_bins, cuts)
    if rc != 0:
        raise AvkError(f"avk_partition_regions failed ({rc})")
    return [(int(cuts[k]), int(cuts[k + 1])) for k in range(n_bins)]


def merge_cfg(cfg: MergeConfig) -> abi.MergeCfg:
    return abi.MergeCfg(cfg.max_branch_factor, int(cfg.no_conflict_enabled), int(cfg.majority_voting_enabled),
                        -1 if cfg.conflict_selection is None else int(cfg.conflict_selection))


class Solver:
    """One context per process / GPU.  The reference genome stays resident in HBM
    (ReferenceGenome::from_fasta once per run, src/main.rs:94)."""

    def __init__(self, device: int = 0):
        self._lib = load()
        self._ctx = C.c_void_p()
        rc = self._lib.avk_create(device, C.byref(self._ctx))
        if rc != 0:
            self._ctx = None
            raise AvkError(f"avk_create(device={device}) failed with {rc}: no usable CUDA device "
                           "(aardvark_b200 has no CPU fallback)")
        self.contig_index = {}
        self._contigs = []

    def lane(self) -> "Solver":
        """A second context on this solver's GPU that shares its resident reference and stratifications (avk_create_lane):
        use one per host thread to keep several batches in flight.  Close the lanes before this solver."""
        ln = Solver.__new__(Solver)
        ln._lib = self._lib
        ln._ctx = C.c_void_p()
        self._check(self._lib.avk_create_lane(self._ctx, C.byref(ln._ctx)), "avk_create_lane")
        ln.contig_index, ln._contigs, ln._owner = self.contig_index, self._contigs, self
        return ln

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.avk_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise AvkError(f"{what} failed ({rc}): {self._lib.avk_last_error(self._ctx).decode()}")

    # -- reference ---------------------------------------------------------------------
    def set_reference(self, contigs, names: Sequence[str] = None):
        """contigs: list of bytes / uint8 arrays (raw bases, compared as raw bytes)."""
        arrs = [np.frombuffer(c, dtype=np.uint8) if isinstance(c, (bytes, bytearray)) else np.ascontiguousarray(c, dtype=np.uint8)
                for c in contigs]
        self._contigs = arrs
        ptrs = (C.POINTER(C.c_uint8) * len(arrs))(*[a.ctypes.data_as(C.POINTER(C.c_uint8)) for a in arrs])
        lens = (C.c_uint64 * len(arrs))(*[a.size for a in arrs])
        self._check(self._lib.avk_set_reference(self._ctx, len(arrs), ptrs, lens), "avk_set_reference")
        names = list(names) if names is not None else [str(i) for i in range(len(arrs))]
        self.contig_index = {n: i for i, n in enumerate(names)}

    def set_stratifications(self, strat):
        """strat: batch.StratIntervals.  Replaces Stratifications::from_tsv_batch (stratifications.rs:23-80): the interval
        sets stay resident; CompareOutputs(containment=True / device_strata=True) use the device lookup."""
        cs = strat.to_c()
        self._check(self._lib.avk_set_stratifications(self._ctx, C.byref(cs)), "avk_set_stratifications")

    # -- batched operators --------------------------------------------------------------
    def compare_batch(self, batch: RegionBatch, cfg: CompareConfig = None, out: CompareOutputs = None, **out_kwargs):
        cfg = cfg or CompareConfig(enable_sequences=False)
        if out is None:
            if cfg.enable_sequences and "seq_off" not in out_kwargs:
                off, plen = seq_offsets(batch)
                out_kwargs.update(seq_off=off, seq_pool_len=plen)
            out = CompareOutputs(batch, **out_kwargs)
        cb, cc, co = batch.to_c(), compare_cfg(cfg), out.to_c()
        self._check(self._lib.avk_compare_batch(self._ctx, C.byref(cb), C.byref(cc), C.byref(co)), "avk_compare_batch")
        return out

    def compare_batch_range(self, batch: RegionBatch, lo: int, hi: int, cfg: CompareConfig = None, out: CompareOutputs = None, **out_kwargs):
        """One contiguous bin [lo, hi) of `batch`; results land in out[lo:hi] (totals = this bin's sums)."""
        cfg = cfg or CompareConfig(enable_sequences=False)
        if out is None:
            out = CompareOutputs(batch, **out_kwargs)
        cb, cc, co = batch.to_c(), compare_cfg(cfg), out.to_c()
        self._check(self._lib.avk_compare_batch_range(self._ctx, C.byref(cb), lo, hi, C.byref(cc), C.byref(co)), "avk_compare_batch_range")
        return out

    def merge_batch(self, batch: RegionBatch, cfg: MergeConfig = None) -> MergeOutputs:
        cfg = cfg or MergeConfig()
        out = MergeOutputs(batch)
        cb, cc, co = batch.to_c(), merge_cfg(cfg), out.to_c()
        self._check(self._lib.avk_merge_batch(self._ctx, C.byref(cb), C.byref(cc), C.byref(co)), "avk_merge_batch")
        return out

    def wfa_ed_batch(self, pairs) -> np.ndarray:
        """Batched wfa_ed (src/util/sequence_alignment.rs:9-13) over [(a, b)] byte pairs."""
        pool = bytearray()
        a_off, a_len, b_off, b_len = [], [], [], []
        for a, b in pairs:
            a_off.append(len(pool)); a_len.append(len(a)); pool += a
            b_off.append(len(pool)); b_len.append(len(b)); pool += b
        pool_a = np.frombuffer(bytes(pool) if pool else b"\0", dtype=np.uint8)
        ao, bo = np.array(a_off, dtype=np.uint64), np.array(b_off, dtype=np.uint64)
        al, bl = np.array(a_len, dtype=np.uint32), np.array(b_len, dtype=np.uint32)
        ed = np.zeros(max(len(a_off), 1), dtype=np.uint32)
        self._check(self._lib.avk_wfa_ed_batch(self._ctx, len(a_off), abi.ptr(pool_a), len(pool), abi.ptr(ao), abi.ptr(al),
                                                abi.ptr(bo), abi.ptr(bl), abi.ptr(ed)), "avk_wfa_ed_batch")
        return ed[:len(a_off)]

    # -- region builder on the device (SURVEY 8f N1) ------------------------------------------
    def build_regions(self, callsets, contig: int, flank: int, first_region_id: int = 0, download: bool = True, bed=None):
        """region_generation.rs:276-479 on the device: clusters K call sets (batch.CallSets) into a batch that stays
        resident (run_resident() can follow).  One contig spanned by one interval by default; with call sets that carry
        variant_contig (several contigs in one table) and / or bed (batch.BedIntervals) the whole per-contig, per-interval
        iteration runs in one call (avk_build_regions_bed).  Returns the RegionBatch (or (n_regions, n_variants) when
        download is False)."""
        import numpy as np
        cs = callsets.to_c()
        n, nv = C.c_uint64(0), C.c_uint64(0)
        if bed is not None or getattr(callsets, "variant_contig", None) is not None:
            vc = callsets.variant_contig if getattr(callsets, "variant_contig", None) is not None else np.full(callsets.n_variants, contig, dtype=np.uint32)
            vc = np.ascontiguousarray(vc if vc.size else np.zeros(1, np.uint32), dtype=np.uint32)
            cbed = bed.to_c() if bed is not None else None
            self._check(self._lib.avk_build_regions_bed(self._ctx, C.byref(cs), abi.ptr(vc), C.byref(cbed) if cbed is not None else None, flank,
                                                        first_region_id, C.byref(n), C.byref(nv)), "avk_build_regions_bed")
        else:
            self._check(self._lib.avk_build_regions(self._ctx, C.byref(cs), contig, flank, first_region_id, C.byref(n), C.byref(nv)),
                        "avk_build_regions")
        n, nv = int(n.value), int(nv.value)
        if not download:
            return n, nv
        k = callsets.n_inputs
        b = RegionBatch(k, np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.uint32),
                        np.zeros(n * k + 1, np.uint64), np.zeros(nv, np.uint32), np.zeros(nv, np.uint8), np.zeros(nv, np.uint8),
                        np.zeros(nv, np.uint32), np.zeros(nv, np.uint32), np.zeros(nv, np.uint32), np.zeros(nv, np.uint32),
                        np.zeros(max(callsets.pool_len, 1), np.uint8))
        cb = b.to_c()
        self._check(self._lib.avk_regions_download(self._ctx, C.byref(cb)), "avk_regions_download")
        b.allele_pool = b.allele_pool[:max(int(cb.variants.allele_pool_len), 1)]
        return b

    # -- resident mode (bench: inputs already in HBM) --------------------------------------
    def upload(self, batch: RegionBatch, lo: int = None, hi: int = None):
        cb = batch.to_c()
        if lo is None:
            self._check(self._lib.avk_compare_upload(self._ctx, C.byref(cb)), "avk_compare_upload")
        else:
            self._check(self._lib.avk_compare_upload_range(self._ctx, C.byref(cb), lo, hi), "avk_compare_upload_range")

    def run_resident(self, cfg: CompareConfig = None, region_metrics: bool = False, sequences: bool = False):
        """One pass over the resident batch.  region_metrics=True keeps the per-region metric rows on the device so
        that download() and writers.region_summary_bgzf can use them; sequences=True (needs cfg.enable_sequences) fills the
        sequence bundle on the device for writers.region_sequences_bgzf (AVK_CMP_KEEP_SEQUENCES; a slower pass)."""
        flags = (abi.CMP_KEEP_REGION_ROWS if region_metrics else 0) | (abi.CMP_KEEP_SEQUENCES if sequences else 0)
        cc = compare_cfg(cfg or CompareConfig(enable_sequences=False), flags)
        self._check(self._lib.avk_compare_run_resident(self._ctx, C.byref(cc)), "avk_compare_run_resident")

    def result_device_view(self) -> abi.CompareDevView:
        v = abi.CompareDevView()
        self._check(self._lib.avk_compare_result_device(self._ctx, C.byref(v)), "avk_compare_result_device")
        return v

    def download(self, out: CompareOutputs):
        co = out.to_c()
        self._check(self._lib.avk_compare_download(self._ctx, C.byref(co)), "avk_compare_download")
        return out

    # -- resident merge: upload (or build_regions), solve, and write the outputs where the batch lies -------------------
    def merge_upload(self, batch: RegionBatch, lo: int = None, hi: int = None):
        """Regions [lo, hi) of `batch` (all by default) become the resident batch of a merge (avk_merge_upload_range)."""
        cb = batch.to_c()
        lo, hi = (0, batch.n_regions) if lo is None else (lo, hi)
        self._check(self._lib.avk_merge_upload_range(self._ctx, C.byref(cb), lo, hi), "avk_merge_upload_range")

    def merge_run_resident(self, cfg: MergeConfig = None):
        """Solve the resident batch (merge_upload or build_regions); the result stays on the device for merge_download and the
        device writers (writers.merge_records_bgzf / merge_regions_bgzf / merge_summary_rows)."""
        cc = merge_cfg(cfg or MergeConfig())
        self._check(self._lib.avk_merge_run_resident(self._ctx, C.byref(cc)), "avk_merge_run_resident")

    def merge_download(self, out: MergeOutputs) -> MergeOutputs:
        """The resident bin's merge result into out[lo:hi] (out is sized for the whole batch)."""
        co = out.to_c()
        self._check(self._lib.avk_merge_download(self._ctx, C.byref(co)), "avk_merge_download")
        return out

    def last_timings_ms(self):
        buf = (C.c_float * 5)()
        self._lib.avk_last_timings(self._ctx, buf)
        return dict(zip(("alt_ed", "search", "heavy_ed", "reduce", "total"), (float(x) for x in buf)))

    def last_work(self):
        wc = abi.WorkCounters()
        self._lib.avk_last_work(self._ctx, C.byref(wc))
        return wc.as_dict()

    def int_peak_ops_per_s(self) -> float:
        v = C.c_double(0)
        self._check(self._lib.avk_int_peak(self._ctx, C.byref(v)), "avk_int_peak")
        return float(v.value)

    def last_tier_overflow(self):
        buf = (C.c_uint32 * 3)()
        self._lib.avk_last_tier_overflow(self._ctx, buf)
        return [int(x) for x in buf]

    def last_tier_ms(self):
        buf = (C.c_float * 3)()
        self._lib.avk_last_tier_ms(self._ctx, buf)
        return [float(x) for x in buf]

    def launch_count(self) -> int:
        return int(self._lib.avk_launch_count(self._ctx))

    # -- the reference's per-region operators ------------------------------------------------
    def solve_compare_regions(self, regions: Sequence[CompareRegion], cfg: CompareConfig = None) -> List:
        cfg = cfg or CompareConfig()
        batch = RegionBatch.from_compare_regions(regions, self.contig_index)
        out = self.compare_batch(batch, cfg)
        return unpack_compare(batch, out)

    def solve_compare_region(self, region: CompareRegion, cfg: CompareConfig = None):
        """Ok(CompareBenchmark) or raises RegionError (the reference's per-region Err)."""
        res = self.solve_compare_regions([region], cfg)[0]
        if isinstance(res, RegionError):
            raise res
        return res

    def solve_merge_regions(self, regions: Sequence[MultiRegion], cfg: MergeConfig = None) -> List:
        batch = RegionBatch.from_multi_regions(regions, self.contig_index)
        return unpack_merge(batch, self.merge_batch(batch, cfg))

    def solve_merge_region(self, region: MultiRegion, cfg: MergeConfig = None):
        res = self.solve_merge_regions([region], cfg)[0]
        if isinstance(res, RegionError):
            raise res
        return res


class SolverPool:
    """Several batches in flight on ONE GPU: the owner context plus `n - 1` lanes (avk_create_lane), one host thread each.
    `compare_batches` hands the batches to the contexts as they become free and returns the outputs in input order; the
    calls are plain avk_compare_batch calls (ctypes releases the GIL), so results are those of Solver.compare_batch."""

    def __init__(self, device: int = 0, n: int = 4):
        self.owner = Solver(device)
        self.solvers = [self.owner]
        self._n = max(1, int(n))

    def set_reference(self, contigs, names: Sequence[str] = None):
        self.owner.set_reference(contigs, names)
        for s in self.solvers[1:]:
            s.contig_index, s._contigs = self.owner.contig_index, self.owner._contigs

    def set_stratifications(self, strat):
        self.owner.set_stratifications(strat)

    def _grow(self):
        while len(self.solvers) < self._n:
            self.solvers.append(self.owner.lane())

    def launch_count(self) -> int:
        return sum(s.launch_count() for s in self.solvers)

    def compare_batches(self, batches, cfg: CompareConfig = None, outs=None, **out_kwargs):
        import threading
        self._grow()
        batches = list(batches)
        outs = list(outs) if outs is not None else [None] * len(batches)
        res, errs = [None] * len(batches), []
        nxt, lock = [0], threading.Lock()

        def work(s):
            while True:
                with lock:
                    i = nxt[0]
                    nxt[0] += 1
                if i >= len(batches) or errs:
                    return
                try:
                    res[i] = s.compare_batch(batches[i], cfg, out=outs[i], **out_kwargs)
                except Exception as e:          # noqa: BLE001 - re-raised below on the caller's thread
                    errs.append(e)
        th = [threading.Thread(target=work, args=(s,)) for s in self.solvers[:max(1, min(self._n, len(batches)))]]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]
        return res

    def close(self):
        for s in reversed(self.solvers):
            s.close()
        self.solvers = []


class MultiSolver:
    """Several GPUs of one node behind one call (avk_compare_batch_multi / avk_merge_batch_multi): one context per
    device, contiguous region bins, one host thread per device inside the library."""

    def __init__(self, devices: Sequence[int]):
        self.solvers = [Solver(d) for d in devices]
        self._lib = self.solvers[0]._lib
        self._ctxs = (C.c_void_p * len(self.solvers))(*[s._ctx for s in self.solvers])

    def close(self):
        for s in self.solvers:
            s.close()

    def set_reference(self, contigs, names: Sequence[str] = None):
        for s in self.solvers:
            s.set_reference(contigs, names)

    def set_stratifications(self, strat):
        for s in self.solvers:
            s.set_stratifications(strat)

    def compare_batch(self, batch: RegionBatch, cfg: CompareConfig = None, out: CompareOutputs = None, **out_kwargs):
        cfg = cfg or CompareConfig(enable_sequences=False)
        if out is None:
            if cfg.enable_sequences and "seq_off" not in out_kwargs:
                off, plen = seq_offsets(batch)
                out_kwargs.update(seq_off=off, seq_pool_len=plen)
            out = CompareOutputs(batch, **out_kwargs)
        cb, cc, co = batch.to_c(), compare_cfg(cfg), out.to_c()
        self.solvers[0]._check(self._lib.avk_compare_batch_multi(self._ctxs, len(self.solvers), C.byref(cb), C.byref(cc), C.byref(co)),
                               "avk_compare_batch_multi")
        return out

    def merge_batch(self, batch: RegionBatch, cfg: MergeConfig = None) -> MergeOutputs:
        cfg = cfg or MergeConfig()
        out = MergeOutputs(batch)
        cb, cc, co = batch.to_c(), merge_cfg(cfg), out.to_c()
        self.solvers[0]._check(self._lib.avk_merge_batch_multi(self._ctxs, len(self.solvers), C.byref(cb), C.byref(cc), C.byref(co)),
                               "avk_merge_batch_multi")
        return out
