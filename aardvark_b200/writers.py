"""Host-side mirrors of the reference's writers for the compare path's results (SURVEY 8f N3).

SummaryWriter follows src/writers/summary.rs (new / add_comparison totals / write_summary), VariantCategorizer's record
lines follow src/writers/variant_categorizer.rs:178-237.  Both only format counters and labels the CUDA kernels produced
(avk_compare_out::totals / strat_totals, var_class / var_expected / var_observed); the formatting itself is in the product
library (avk_summary_write / avk_vcf_records_write, host C++), so a Rust caller gets the same bytes."""
import ctypes as C

import numpy as np

from . import abi
from .lib import AvkError, load

METRICS = {"GT": 0, "HAP": 1, "WEIGHTED_HAP": 2, "BASEPAIR": 3, "RECORD_BP": 4}


def _bind():
    lib = load()
    lib.avk_summary_write.argtypes = [C.POINTER(C.c_uint64), C.POINTER(C.c_uint8), C.c_uint32, C.c_char_p, C.c_char_p, C.c_int, C.c_int,
                                      C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.avk_vcf_records_write.argtypes = [C.POINTER(abi.RegionBatch), C.c_uint32, C.POINTER(C.c_char_p), C.c_uint32, C.POINTER(C.c_uint8),
                                          C.POINTER(C.c_uint8), C.POINTER(C.c_uint8), C.c_uint64, C.c_uint64, C.c_char_p, C.c_uint64,
                                          C.POINTER(C.c_uint64)]
    t = [C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64)]
    names = C.POINTER(C.c_char_p)
    lib.avk_merge_records_write.argtypes = [C.POINTER(abi.RegionBatch), C.POINTER(abi.MergeOut), names, C.c_uint32, names, C.c_uint64, C.c_uint64] + t
    lib.avk_merge_regions_write.argtypes = [C.POINTER(abi.RegionBatch), C.POINTER(abi.MergeOut), names, C.c_uint32, C.c_int, C.c_uint64, C.c_uint64] + t
    lib.avk_merge_summary_write.argtypes = [C.POINTER(abi.RegionBatch), C.POINTER(abi.MergeOut), names, C.c_int, C.c_int] + t
    lib.avk_merge_summary_rows_write.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, names, C.c_int, C.c_int] + t
    return lib


def _text(call):
    n = C.c_uint64(0)
    rc = call(None, 0, C.byref(n))
    if rc != 0:
        raise AvkError(f"writer call failed: {rc}")
    buf = C.create_string_buffer(int(n.value) + 1)
    rc = call(buf, int(n.value), C.byref(n))
    if rc != 0:
        raise AvkError(f"writer call failed: {rc}")
    return buf.raw[:int(n.value)].decode()


class SummaryWriter:
    """summary.rs:14-30, 116-221: accumulates nothing itself -- the sums come from the device -- and writes the rows."""

    def __init__(self, compare_label, metrics_to_write=("GT", "HAP", "WEIGHTED_HAP", "BASEPAIR", "RECORD_BP"), strat_labels=None):
        self.compare_label = compare_label
        self.metrics = np.asarray([METRICS[m] for m in metrics_to_write], dtype=np.uint8)
        self.strat_labels = list(strat_labels or [])

    def _group(self, totals, region_label, csv, header):
        lib = _bind()
        t = np.ascontiguousarray(totals, dtype=np.uint64).reshape(-1)
        assert t.size == abi.N_GROUPS * abi.N_METRICS
        return _text(lambda buf, cap, n: lib.avk_summary_write(abi.ptr(t), abi.ptr(self.metrics), self.metrics.size, self.compare_label.encode(),
                                                               region_label.encode(), 1 if csv else 0, 1 if header else 0, buf, cap, n))

    def summary_text(self, totals, strat_totals=None, csv=False):
        """write_summary (:166-221): the ALL group, then one group per stratification label in order."""
        out = self._group(totals, "ALL", csv, True)
        if strat_totals is not None:
            st = np.asarray(strat_totals, dtype=np.uint64).reshape(len(self.strat_labels), -1)
            for label, row in zip(self.strat_labels, st):
                out += self._group(row, label, csv, False)
        return out

    def write_summary(self, filename, totals, strat_totals=None):
        with open(filename, "w") as f:
            f.write(self.summary_text(totals, strat_totals, csv=str(filename).endswith(".csv")))


def vcf_record_lines(batch, side, contig_names, outputs, lo=0, hi=None):
    """variant_categorizer.rs:178-237: the GT:BD:EA:OA:RI body lines of input `side` (0 truth, 1 query), regions [lo, hi)."""
    lib = _bind()
    hi = batch.n_regions if hi is None else hi
    cb = batch.to_c()
    names = (C.c_char_p * len(contig_names))(*[n.encode() for n in contig_names])
    return _text(lambda buf, cap, n: lib.avk_vcf_records_write(C.byref(cb), side, names, len(contig_names), abi.ptr(outputs.var_class),
                                                               abi.ptr(outputs.var_expected), abi.ptr(outputs.var_observed), lo, hi, buf, cap, n))


class VariantMerger:
    """src/writers/variant_merger.rs + merge_summary.rs over a solved merge batch (MergeOutputs): the body of passing.vcf.gz,
    regions.bed / failed_regions.bed and the merge summary table.  Formatting happens in the product library
    (avk_merge_records_write / avk_merge_regions_write / avk_merge_summary_write, host C++)."""

    def __init__(self, batch, outputs, contig_names, input_labels):
        assert len(input_labels) == batch.n_inputs
        self.batch, self.out = batch, outputs
        self._cb, self._co = batch.to_c(), outputs.to_c()
        self._names = (C.c_char_p * len(contig_names))(*[n.encode() for n in contig_names])
        self._labels = (C.c_char_p * len(input_labels))(*[n.encode() for n in input_labels])
        self._n_contigs = len(contig_names)

    def passing_records(self, lo=0, hi=None):
        lib = _bind()
        hi = self.batch.n_regions if hi is None else hi
        return _text(lambda buf, cap, n: lib.avk_merge_records_write(C.byref(self._cb), C.byref(self._co), self._names, self._n_contigs, self._labels,
                                                                     lo, hi, buf, cap, n))

    def regions_bed(self, passing=True, lo=0, hi=None):
        lib = _bind()
        hi = self.batch.n_regions if hi is None else hi
        return _text(lambda buf, cap, n: lib.avk_merge_regions_write(C.byref(self._cb), C.byref(self._co), self._names, self._n_contigs,
                                                                     1 if passing else 0, lo, hi, buf, cap, n))

    def summary_text(self, csv=False, header=True):
        lib = _bind()
        return _text(lambda buf, cap, n: lib.avk_merge_summary_write(C.byref(self._cb), C.byref(self._co), self._labels, 1 if csv else 0,
                                                                     1 if header else 0, buf, cap, n))


def bgzf_compress(solver, text: bytes) -> bytes:
    """avk_bgzf_compress: text -> a complete BGZF file (EOF marker included), compressed on the device."""
    lib = solver._lib
    lib.avk_bgzf_compress.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64)]
    n = C.c_uint64(0)
    solver._check(lib.avk_bgzf_compress(solver._ctx, text, len(text), None, 0, C.byref(n)), "avk_bgzf_compress")
    buf = C.create_string_buffer(int(n.value) + 1)
    solver._check(lib.avk_bgzf_compress(solver._ctx, text, len(text), buf, int(n.value), C.byref(n)), "avk_bgzf_compress")
    return buf.raw[:int(n.value)]


def _records_bgzf_fn(lib):
    lib.avk_compare_records_bgzf.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_char_p), C.c_uint32, C.POINTER(C.c_uint64), C.c_char_p,
                                             C.c_uint64, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    return lib.avk_compare_records_bgzf


def vcf_records_bgzf(solver, side, contig_names, header: bytes = b"", region_ids=None, eof=True) -> bytes:
    """avk_compare_records_bgzf: truth.vcf.gz (side 0) / query.vcf.gz (side 1) of the solver's resident compare result,
    formatted and compressed on the device -- the same bytes as bgzf_compress(solver, header + vcf_record_lines(...)).
    region_ids: the ids of the batch given to upload() (the whole batch's array; the resident bin's part is read), None
    after build_regions().  eof=False leaves out the EOF marker so that the next bin's file can be appended."""
    fn = _records_bgzf_fn(solver._lib)
    names = (C.c_char_p * max(len(contig_names), 1))(*[n.encode() for n in contig_names])
    rid = None if region_ids is None else np.ascontiguousarray(region_ids, dtype=np.uint64)
    rid_p = abi.ptr(rid)
    n = C.c_uint64(0)
    call = lambda buf, cap: fn(solver._ctx, side, names, len(contig_names), rid_p, header, len(header), 1 if eof else 0, buf, cap, C.byref(n))
    solver._check(call(None, 0), "avk_compare_records_bgzf")
    out = np.empty(int(n.value), dtype=np.uint8)                 # an upper bound; pages past the compressed size are never touched
    solver._check(call(out.ctypes.data, out.size), "avk_compare_records_bgzf")
    return out[:int(n.value)].tobytes()


def _bgzf_call(solver, what, call):
    """size query (an upper bound), then the call into a buffer of that size"""
    n = C.c_uint64(0)
    solver._check(call(None, 0, C.byref(n)), what)
    out = np.empty(int(n.value), dtype=np.uint8)                 # pages past the compressed size are never touched
    solver._check(call(out.ctypes.data, out.size, C.byref(n)), what)
    return out[:int(n.value)].tobytes()


def _merge_bgzf_fns(lib):
    names = C.POINTER(C.c_char_p)
    t = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.avk_merge_records_bgzf.argtypes = [C.c_void_p, names, C.c_uint32, names, C.POINTER(C.c_uint64), C.c_char_p, C.c_uint64, C.c_int] + t
    lib.avk_merge_regions_bgzf.argtypes = [C.c_void_p, names, C.c_uint32, C.c_int, C.POINTER(C.c_uint64), C.c_int] + t
    lib.avk_merge_summary_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    return lib.avk_merge_records_bgzf, lib.avk_merge_regions_bgzf, lib.avk_merge_summary_counts


def _c_names(names):
    return (C.c_char_p * max(len(names), 1))(*[n if isinstance(n, bytes) else n.encode() for n in names])


def merge_records_bgzf(solver, contig_names, input_labels, header: bytes = b"", region_ids=None, eof=True) -> bytes:
    """avk_merge_records_bgzf: passing.vcf.gz of the solver's resident merge result, formatted and compressed on the device -- the
    same bytes as bgzf_compress(solver, header + VariantMerger(...).passing_records(lo, hi)) over the resident bin.  region_ids:
    the ids of the batch given to merge_upload() / merge_batch() (the whole batch's array), None after build_regions().
    eof=False leaves out the EOF marker so that the next bin's file can be appended.  Labels are str or raw bytes."""
    fn = _merge_bgzf_fns(solver._lib)[0]
    names, labels = _c_names(contig_names), _c_names(input_labels)
    rid = None if region_ids is None else np.ascontiguousarray(region_ids, dtype=np.uint64)
    rid_p = abi.ptr(rid)
    return _bgzf_call(solver, "avk_merge_records_bgzf", lambda buf, cap, n: fn(solver._ctx, names, len(contig_names), labels, rid_p, header, len(header),
                                                                                1 if eof else 0, buf, cap, n))


def merge_regions_bgzf(solver, contig_names, passing=True, region_ids=None, eof=True) -> bytes:
    """avk_merge_regions_bgzf: regions.bed.gz (passing) / failed_regions.bed.gz of the resident merge result -- the same bytes as
    bgzf_compress(solver, VariantMerger(...).regions_bed(passing, lo, hi)) over the resident bin."""
    fn = _merge_bgzf_fns(solver._lib)[1]
    names = _c_names(contig_names)
    rid = None if region_ids is None else np.ascontiguousarray(region_ids, dtype=np.uint64)
    rid_p = abi.ptr(rid)
    return _bgzf_call(solver, "avk_merge_regions_bgzf", lambda buf, cap, n: fn(solver._ctx, names, len(contig_names), 1 if passing else 0, rid_p,
                                                                                1 if eof else 0, buf, cap, n))


# avk_merge_summary_row
SUMMARY_ROW = np.dtype([("indices", np.uint32), ("classification", np.uint8), ("variant_type", np.uint8), ("input", np.uint8), ("pad", np.uint8),
                        ("pass_variants", np.uint64), ("fail_variants", np.uint64)], align=True)


def merge_summary_rows(solver) -> np.ndarray:
    """avk_merge_summary_counts: the merge summary's per-key variant counts of the resident bin, counted on the device (a
    SUMMARY_ROW array in no particular order).  Rows of several bins or GPUs are simply concatenated for merge_summary_text."""
    fn = _merge_bgzf_fns(solver._lib)[2]
    n = C.c_uint64(0)
    solver._check(fn(solver._ctx, None, 0, C.byref(n)), "avk_merge_summary_counts")
    rows = np.zeros(max(int(n.value), 1), dtype=SUMMARY_ROW)
    solver._check(fn(solver._ctx, rows.ctypes.data, rows.size, C.byref(n)), "avk_merge_summary_counts")
    return rows[:int(n.value)]


def merge_summary_text(rows, n_inputs, labels, csv=False, header=True) -> str:
    """avk_merge_summary_rows_write (host): the merge summary of the rows -- the text VariantMerger.summary_text gives over the
    whole batch.  Rows that share a key add up."""
    lib = _bind()
    rows = np.ascontiguousarray(rows, dtype=SUMMARY_ROW)
    lab = _c_names(labels)
    return _text(lambda buf, cap, n: lib.avk_merge_summary_rows_write(rows.ctypes.data if rows.size else None, rows.size, n_inputs, lab,
                                                                      1 if csv else 0, 1 if header else 0, buf, cap, n))
