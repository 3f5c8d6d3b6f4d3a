"""ctypes mirror of include/aardvark_b200.h (struct layouts and enums).

Both the CUDA product library and the CPU oracle (tests only) take these
structs, so one Python-side batch can be handed to either and the outputs
compared bit for bit.
"""
import ctypes as C

import numpy as np

# --- enums (include/aardvark_b200.h) ---------------------------------------
VT_SNV, VT_INSERTION, VT_DELETION, VT_INDEL = 0, 1, 2, 3
VT_SV_INSERTION, VT_SV_DELETION, VT_SV_DUPLICATION, VT_SV_INVERSION = 4, 5, 6, 7
VT_SV_BREAKEND, VT_TR_CONTRACTION, VT_TR_EXPANSION, VT_UNKNOWN = 8, 9, 10, 11
N_VARIANT_TYPES = 12
VT_NAMES = ["Snv", "Insertion", "Deletion", "Indel", "SvInsertion", "SvDeletion", "SvDuplication",
            "SvInversion", "SvBreakend", "TrContraction", "TrExpansion", "Unknown"]

ZYG_UNKNOWN, ZYG_HOM_REF, ZYG_UNPHASED_HET, ZYG_PHASED_HET01, ZYG_PHASED_HET10, ZYG_HOM_ALT = range(6)

CLASS_UNKNOWN, CLASS_TP, CLASS_FN, CLASS_FP = range(4)

MERGE_DIFFERENT, MERGE_NO_CONFLICT, MERGE_MAJORITY_AGREE, MERGE_CONFLICT_SELECTION, MERGE_BASEPAIR_IDENTICAL = range(5)

M_GT, M_GT_TRUTH_FN_GT, M_GT_QUERY_FP_GT, M_HAP, M_WEIGHTED_HAP, M_BASEPAIR, M_RECORD_BP = 0, 4, 5, 6, 10, 14, 18
N_METRICS = 22
N_GROUPS = 1 + N_VARIANT_TYPES

ST_OK, ST_BAD_ZYGOSITY, ST_NO_RESULT, ST_TRUTH_FP, ST_TP_UNDERFLOW, ST_BAD_INPUT, ST_WORKSPACE, ST_TIMEOUT = range(8)
CMP_KEEP_REGION_ROWS = 1
CMP_KEEP_SEQUENCES = 2
CMP_STRATA = 4

AVK_OK, AVK_ERR_INVALID, AVK_ERR_CUDA, AVK_ERR_NO_REFERENCE, AVK_ERR_OOM = 0, -1, -2, -3, -4

_u8p = C.POINTER(C.c_uint8)
_u16p = C.POINTER(C.c_uint16)
_u32p = C.POINTER(C.c_uint32)
_i32p = C.POINTER(C.c_int32)
_u64p = C.POINTER(C.c_uint64)


class VariantTable(C.Structure):
    _fields_ = [
        ("n_variants", C.c_uint64),
        ("position", _u32p),
        ("variant_type", _u8p),
        ("zygosity", _u8p),
        ("raw_allele_space", _u32p),
        ("allele_off", _u32p),
        ("a0_len", _u32p),
        ("a1_len", _u32p),
        ("allele_pool", _u8p),
        ("allele_pool_len", C.c_uint64),
    ]


class RegionBatch(C.Structure):
    _fields_ = [
        ("n_regions", C.c_uint64),
        ("n_inputs", C.c_uint32),
        ("region_id", _u64p),
        ("contig", _u32p),
        ("start", _u32p),
        ("end", _u32p),
        ("var_off", _u64p),
        ("variants", VariantTable),
    ]


class CallSets(C.Structure):
    _fields_ = [
        ("n_inputs", C.c_uint32),
        ("input_off", _u64p),
        ("variants", VariantTable),
    ]


class BedIntervals(C.Structure):
    _fields_ = [
        ("n_contigs", C.c_uint32),
        ("first", _u64p),
        ("start", _u32p),
        ("end", _u32p),
    ]


class VcfOut(C.Structure):
    _fields_ = [
        ("n_variants", C.c_uint64), ("allele_pool_len", C.c_uint64), ("cap_variants", C.c_uint64), ("cap_pool", C.c_uint64),
        ("contig", _u32p), ("position", _u32p), ("variant_type", _u8p), ("zygosity", _u8p),
        ("raw_allele_space", _u32p), ("allele_off", _u32p), ("a0_len", _u32p), ("a1_len", _u32p), ("allele_pool", _u8p),
    ]


class CompareCfg(C.Structure):
    _fields_ = [
        ("max_branch_factor", C.c_uint32),
        ("enable_exact_shortcut", C.c_uint32),
        ("enable_sequences", C.c_uint32),
        ("flags", C.c_uint32),
        ("exact_gt_max_expansions", C.c_uint32),
    ]


class MergeCfg(C.Structure):
    _fields_ = [
        ("max_branch_factor", C.c_uint32),
        ("no_conflict_enabled", C.c_uint32),
        ("majority_voting_enabled", C.c_uint32),
        ("conflict_selection", C.c_int32),
    ]


class CompareOut(C.Structure):
    _fields_ = [
        ("status", _i32p),
        ("ed1", _u32p),
        ("ed2", _u32p),
        ("region_metrics", _u64p),
        ("type_mask", _u16p),
        ("var_expected", _u8p),
        ("var_observed", _u8p),
        ("var_class", _u8p),
        ("totals", _u64p),
        ("totals_mask", _u16p),
        ("solved_blocks", _u64p),
        ("error_blocks", _u64p),
        ("strat_off", _u64p),
        ("strat_idx", _u32p),
        ("n_strata", C.c_uint32),
        ("pad0", C.c_uint32),
        ("strat_totals", _u64p),
        ("seq_off", _u64p),
        ("seq_len", _u32p),
        ("seq_pool", _u8p),
        ("containment", _u64p),
    ]


class CompareDevView(C.Structure):
    _fields_ = [
        ("lo", C.c_uint64), ("n_regions", C.c_uint64), ("v_base", C.c_uint64), ("n_variants", C.c_uint64),
        ("status", C.c_void_p), ("ed1", C.c_void_p), ("ed2", C.c_void_p), ("type_mask", C.c_void_p),
        ("var_expected", C.c_void_p), ("var_observed", C.c_void_p), ("var_class", C.c_void_p), ("totals", C.c_void_p),
    ]


class StratIntervals(C.Structure):
    _fields_ = [
        ("n_strata", C.c_uint32), ("n_contigs", C.c_uint32),
        ("off", _u64p), ("first", _u32p), ("last", _u32p),
    ]


class MergeOut(C.Structure):
    _fields_ = [
        ("status", _i32p),
        ("classification", _u8p),
        ("n_indices", _u8p),
        ("indices", _u8p),
    ]


class WorkCounters(C.Structure):
    _fields_ = [
        ("alignments", C.c_uint64),
        ("cells", C.c_uint64),
        ("matched_bases", C.c_uint64),
        ("search_pops", C.c_uint64),
        ("exact_pops", C.c_uint64),
        ("alg_bytes", C.c_uint64),
    ]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


_CT = {
    np.dtype(np.uint8): C.c_uint8,
    np.dtype(np.uint16): C.c_uint16,
    np.dtype(np.uint32): C.c_uint32,
    np.dtype(np.int32): C.c_int32,
    np.dtype(np.uint64): C.c_uint64,
}


def ptr(arr):
    """ctypes pointer to a C-contiguous numpy array (None -> NULL)."""
    if arr is None:
        return None
    assert arr.flags["C_CONTIGUOUS"], "array must be C-contiguous"
    return arr.ctypes.data_as(C.POINTER(_CT[arr.dtype]))
