/*
 * aardvark_b200.h -- C ABI of the B200-native haplotype-comparison hot path.
 *
 * This header is the drop-in boundary for ONE path of PacificBiosciences/aardvark
 * (v0.10.5): the per-cluster solvers that `aardvark compare` / `aardvark merge`
 * call from their rayon loops.  The reference has no FFI today; the two pure
 * functions below are its de-facto operator interface, and each entry point here
 * names the reference interface it replaces (paths relative to the reference):
 *
 *   solve_compare_region(&CompareRegion, &ReferenceGenome, CompareConfig, ..)
 *       -> anyhow::Result<CompareBenchmark>          src/waffle_solver.rs:122-124
 *       call site (rayon par_iter)                   src/main.rs:251-268
 *   solve_merge_region(&MultiRegion, &ReferenceGenome, MergeConfig)
 *       -> anyhow::Result<MergeBenchmark>            src/merge_solver.rs:110
 *       call site (rayon par_iter)                   src/main.rs:463-478
 *   wfa_ed(&[u8], &[u8]) -> usize                    src/util/sequence_alignment.rs:9-13
 *
 * Because the reference materialises ALL regions before solving
 * (src/main.rs:217-232, :434-443), the per-region call is replaced by ONE
 * batched call over a flat SoA/CSR description of every region.
 *
 * Plain C: pointers + sizes only, no torch/CUDA types.  All pointers are HOST
 * pointers unless a function says otherwise; the library owns all device
 * memory.  Nothing allocated by the library is freed by the caller.
 *
 * Implemented by aardvark_b200/csrc -> libaardvark_b200.so (CUDA sm_100a).  The CPU
 * oracle used by the tests takes the same structs (oracle/oracle.h) so that outputs
 * can be compared bit for bit; it is not part of the product.
 */
#ifndef AARDVARK_B200_H
#define AARDVARK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ enums */

/* VariantType, same discriminants as src/data_types/variants.rs:6-31 */
enum {
    AVK_VT_SNV = 0,
    AVK_VT_INSERTION = 1,
    AVK_VT_DELETION = 2,
    AVK_VT_INDEL = 3,
    AVK_VT_SV_INSERTION = 4,
    AVK_VT_SV_DELETION = 5,
    AVK_VT_SV_DUPLICATION = 6,
    AVK_VT_SV_INVERSION = 7,
    AVK_VT_SV_BREAKEND = 8,
    AVK_VT_TR_CONTRACTION = 9,
    AVK_VT_TR_EXPANSION = 10,
    AVK_VT_UNKNOWN = 11,
    AVK_N_VARIANT_TYPES = 12
};

/* PhasedZygosity, declaration order of src/data_types/phase_enums.rs:33-46 */
enum {
    AVK_ZYG_UNKNOWN = 0,
    AVK_ZYG_HOM_REF = 1,
    AVK_ZYG_UNPHASED_HET = 2,
    AVK_ZYG_PHASED_HET01 = 3,
    AVK_ZYG_PHASED_HET10 = 4,
    AVK_ZYG_HOM_ALT = 5
};

/* Classification, src/data_types/variant_metrics.rs:11-22 */
enum {
    AVK_CLASS_UNKNOWN = 0,
    AVK_CLASS_TP = 1,
    AVK_CLASS_FN = 2,
    AVK_CLASS_FP = 3
};

/* MergeClassification, src/data_types/merge_benchmark.rs:7-20 */
enum {
    AVK_MERGE_DIFFERENT = 0,
    AVK_MERGE_NO_CONFLICT = 1,
    AVK_MERGE_MAJORITY_AGREE = 2,
    AVK_MERGE_CONFLICT_SELECTION = 3,
    AVK_MERGE_BASEPAIR_IDENTICAL = 4
};

/* GroupMetrics flattened to 22 u64 (src/data_types/grouped_metrics.rs:149-161,
 * summary_metrics.rs:5-14,82-91).  Each SummaryMetrics block is
 * {truth_tp, truth_fn, query_tp, query_fp}. */
enum {
    AVK_M_GT = 0,            /* +0 tp +1 fn +2 qtp +3 qfp */
    AVK_M_GT_TRUTH_FN_GT = 4,
    AVK_M_GT_QUERY_FP_GT = 5,
    AVK_M_HAP = 6,
    AVK_M_WEIGHTED_HAP = 10,
    AVK_M_BASEPAIR = 14,
    AVK_M_RECORD_BP = 18,
    AVK_N_METRICS = 22
};
/* group index into per-region metric rows: 0 = joint, 1 + VariantType = that type */
#define AVK_N_GROUPS (1 + AVK_N_VARIANT_TYPES)

/* Per-region status.  0 = Ok(..); anything else is the reference's Err(..)
 * (counted as an "error block", src/main.rs:259-262) or an input the reference
 * would panic on.  The GPU library adds AVK_ST_WORKSPACE for its own limits. */
enum {
    AVK_ST_OK = 0,
    AVK_ST_BAD_ZYGOSITY = 1,      /* HomRef/Unknown zygosity: reference panics (query_optimizer.rs:315) */
    AVK_ST_NO_RESULT = 2,         /* "no results found" / "No result found for problem" */
    AVK_ST_TRUTH_FP = 3,          /* expected < observed (waffle_solver.rs:322, grouped_metrics.rs:197) */
    AVK_ST_TP_UNDERFLOW = 4,      /* ensure!(truth_tp >= basepair tp) waffle_solver.rs:492-493 */
    AVK_ST_BAD_INPUT = 5,         /* malformed batch entry (window outside contig, empty allele, ...) */
    AVK_ST_WORKSPACE = 6,         /* GPU only: search exceeded the largest workspace tier */
    AVK_ST_TIMEOUT = 7            /* optimize_gt_alleles gave up: deterministic stand-in (node-expansion cap) for the
                                   * reference's 300 s wall-clock bail-out, exact_gt_optimizer.rs:165,174-176 */
};

/* Library-level return codes */
enum {
    AVK_OK = 0,
    AVK_ERR_INVALID = -1,
    AVK_ERR_CUDA = -2,
    AVK_ERR_NO_REFERENCE = -3,
    AVK_ERR_OOM = -4
};

/* ------------------------------------------------------------- input batch */

/* Variant fields read on the path (src/data_types/variants.rs:73-91): position,
 * allele0, allele1, variant_type, raw_allele_space; zygosity is the parallel
 * Vec<PhasedZygosity>.  allele0 is stored at allele_pool[allele_off ..+a0_len],
 * allele1 directly after it.  Alleles are raw bytes and compared as raw bytes
 * (src/dwfa/dynamic_wfa.rs:118). */
typedef struct avk_variant_table {
    uint64_t n_variants;
    const uint32_t *position;          /* 0-based, contigs < 2^32 bp */
    const uint8_t *variant_type;       /* AVK_VT_* */
    const uint8_t *zygosity;           /* AVK_ZYG_* */
    const uint32_t *raw_allele_space;  /* pre-trim max allele length (RECORD_BP) */
    const uint32_t *allele_off;
    const uint32_t *a0_len;
    const uint32_t *a1_len;
    const uint8_t *allele_pool;
    uint64_t allele_pool_len;
} avk_variant_table;

/* A batch of regions, each with n_inputs variant lists.  Compare uses
 * n_inputs == 2 (input 0 = truth, input 1 = query: compare_region.rs:102-118);
 * merge uses n_inputs >= 2 (multi_region.rs:9-18).  List (r, k) is the variant
 * index range [var_off[r*n_inputs+k], var_off[r*n_inputs+k+1]); every list is
 * position-sorted (region_generation.rs:373). */
typedef struct avk_region_batch {
    uint64_t n_regions;
    uint32_t n_inputs;
    const uint64_t *region_id;   /* [n_regions] */
    const uint32_t *contig;      /* [n_regions] index given to avk_set_reference */
    const uint32_t *start;       /* [n_regions] Coordinates.start (0-based) */
    const uint32_t *end;         /* [n_regions] Coordinates.end (exclusive) */
    const uint64_t *var_off;     /* [n_regions*n_inputs + 1] */
    avk_variant_table variants;
} avk_region_batch;

/* CompareConfig, src/waffle_solver.rs:94-115 */
typedef struct avk_compare_cfg {
    uint32_t max_branch_factor;      /* default 50 */
    uint32_t enable_exact_shortcut;  /* default 0 */
    uint32_t enable_sequences;       /* fill the sequence bundle outputs */
    uint32_t flags;                  /* AVK_CMP_* (GPU library only; 0 = defaults) */
    /* Deterministic stand-in for the reference's 300 s wall-clock bail-out of optimize_gt_alleles
     * (exact_gt_optimizer.rs:165,174-176): one call may expand at most this many queue nodes (nodes that pass the
     * `errors >= best` skip, where the reference looks at its clock), else the region ends with AVK_ST_TIMEOUT.
     * 0 = AVK_EXACT_GT_DEFAULT_MAX_EXPANSIONS.  The auto-fail heuristic (:160,309-339) bounds sane inputs far below it:
     * it never fires on the five BASELINE configs. */
    uint32_t exact_gt_max_expansions;
} avk_compare_cfg;
#define AVK_EXACT_GT_DEFAULT_MAX_EXPANSIONS (1u << 24)
/* avk_compare_run_resident: keep the per-region GroupTypeMetrics rows (2288 B per region) on the device so that
 * avk_compare_download can return out->region_metrics.  avk_compare_batch* decide from out->region_metrics != NULL. */
#define AVK_CMP_KEEP_REGION_ROWS 1u

/* MergeConfig, src/merge_solver.rs:62-84 */
typedef struct avk_merge_cfg {
    uint32_t max_branch_factor;
    uint32_t no_conflict_enabled;
    uint32_t majority_voting_enabled;
    int32_t conflict_selection;      /* -1 = None */
} avk_merge_cfg;

/* ------------------------------------------------------------ output (SoA) */

/* CompareBenchmark (src/data_types/compare_benchmark.rs:9-33) as caller-owned
 * arrays.  Any pointer may be NULL to skip that output, except status. */
typedef struct avk_compare_out {
    int32_t *status;          /* [n_regions] AVK_ST_* */
    uint32_t *ed1;            /* [n_regions] bm_edit_distance_h1 */
    uint32_t *ed2;            /* [n_regions] bm_edit_distance_h2 */
    uint64_t *region_metrics; /* [n_regions][AVK_N_GROUPS][AVK_N_METRICS] GroupTypeMetrics */
    uint16_t *type_mask;      /* [n_regions] bit t set <=> variant_metrics has key t */
    /* per variant, indexed like the variant table (VariantMetrics,
     * variant_metrics.rs:25-35): truth entries as computed, query entries
     * already toggled (compare_benchmark.rs:109-123) */
    uint8_t *var_expected;    /* [n_variants] */
    uint8_t *var_observed;    /* [n_variants] */
    uint8_t *var_class;       /* [n_variants] AVK_CLASS_* */
    /* reduction over all status==0 regions: what SummaryWriter::
     * add_comparison_benchmark accumulates (writers/summary.rs:146-158) */
    uint64_t *totals;         /* [AVK_N_GROUPS][AVK_N_METRICS] */
    uint16_t *totals_mask;    /* [1] */
    uint64_t *solved_blocks;  /* [1] */
    uint64_t *error_blocks;   /* [1] */
    /* optional stratified reduction: region r belongs to strata
     * strat_idx[strat_off[r] .. strat_off[r+1]) (containment_regions) */
    const uint64_t *strat_off;   /* [n_regions+1] or NULL */
    const uint32_t *strat_idx;
    uint32_t n_strata;
    uint32_t pad0;
    uint64_t *strat_totals;   /* [n_strata][AVK_N_GROUPS][AVK_N_METRICS] */
    /* optional SequenceBundle (compare_benchmark.rs:159-185): 5 strings per
     * region in the order ref, truth1, truth2, query1, query2.  String s of
     * region r is written at seq_pool[seq_off[r*5+s]] with length seq_len[r*5+s];
     * seq_off is an INPUT computed by avk_compare_seq_offsets. */
    const uint64_t *seq_off;  /* [n_regions*5 + 1] */
    uint32_t *seq_len;        /* [n_regions*5] */
    uint8_t *seq_pool;
    /* containment_regions (compare_benchmark.rs:28-30) by device lookup: bit s set <=> the region's var_coordinates()
     * (compare_region.rs:63-74) lie inside one interval of stratum s (waffle_solver.rs:151-166).  Needs
     * avk_set_stratifications.  May be NULL.  When strat_totals is set and strat_off is NULL, the stratified sums
     * use this lookup instead of a caller-provided membership list. */
    uint64_t *containment;    /* [n_regions] */
} avk_compare_out;

/* MergeBenchmark (src/data_types/merge_benchmark.rs:57-62) */
typedef struct avk_merge_out {
    int32_t *status;       /* [n_regions] */
    uint8_t *classification; /* [n_regions] AVK_MERGE_* */
    uint8_t *n_indices;    /* [n_regions] number of valid entries in indices row */
    uint8_t *indices;      /* [n_regions][n_inputs] ascending input indices (or the selected index) */
} avk_merge_out;

/* Work counters (DESIGN.md "algorithmic work"): filled by both libraries when
 * non-NULL so that roofline numerators come from the same definition. */
typedef struct avk_work_counters {
    uint64_t alignments;     /* finalize() calls (global EDs) */
    uint64_t cells;          /* sum over alignments/updates of wavefront entries touched */
    uint64_t matched_bases;  /* bases walked by extend() */
    uint64_t search_pops;    /* optimize_sequences pops */
    uint64_t exact_pops;     /* optimize_gt_alleles pops */
    uint64_t alg_bytes;      /* SURVEY 8(d): sum over alignments of ceil(|a|/4) + ceil(|b|/4) + 8 (CPU oracle only; GPU leaves 0) */
} avk_work_counters;

/* ------------------------------------------------------ GPU library (product) */

typedef struct avk_ctx avk_ctx;

/* Create a context bound to one CUDA device.  One process may hold one context per
 * GPU (avk_compare_batch_multi); a context is used by one host thread at a time. */
int avk_create(int device, avk_ctx **out);
void avk_destroy(avk_ctx *ctx);
/* A lane of `owner`: a context on the same device that reads the owner's resident reference and stratification tables
 * (avk_set_reference / avk_set_stratifications on a lane are errors) and has its own streams and buffers.  With one host
 * thread per context several batches -- e.g. the call sets of several samples against one truth set, the reference's
 * one-process-per-sample use of src/main.rs -- are in flight on one GPU: copies of one overlap kernels of another and the
 * passes fill each other's tails.  Destroy the lanes before the owner, and do not replace the owner's reference or
 * stratifications while a lane has a call in flight. */
int avk_create_lane(avk_ctx *owner, avk_ctx **out);
const char *avk_last_error(const avk_ctx *ctx);

/* Replaces ReferenceGenome::from_fasta + get_full_chromosome
 * (src/main.rs:94, src/waffle_solver.rs:131): uploads the contigs once; they
 * stay resident in HBM for every later batch. */
int avk_set_reference(avk_ctx *ctx, uint32_t n_contigs,
                      const uint8_t *const *seqs, const uint64_t *lens);

/* Stratification BED sets (SURVEY 8f N4).  Replaces Stratifications::from_tsv_batch + containments
 * (src/parsing/stratifications.rs:23-80, 108-118, 197-210): the intervals of every (stratum, contig) -- 0-based
 * INCLUSIVE [first, last], i.e. BED start and BED end - 1 (:158-163) -- stay resident on the device, sorted by first
 * with a running maximum of last, so that "is [a, b] inside one interval" is one binary search per (region, stratum).
 * Strata are numbered in the order given (the reference orders its labels alphabetically, :37,63). */
typedef struct avk_strat_intervals {
    uint32_t n_strata;      /* <= 64 */
    uint32_t n_contigs;     /* contig numbering of avk_set_reference */
    const uint64_t *off;    /* [n_strata * n_contigs + 1]: (stratum s, contig c) owns intervals [off[s*n_contigs+c], off[s*n_contigs+c+1]) */
    const uint32_t *first;
    const uint32_t *last;
} avk_strat_intervals;
int avk_set_stratifications(avk_ctx *ctx, const avk_strat_intervals *in);

/* Replaces the par_iter over solve_compare_region (src/main.rs:251-268). */
int avk_compare_batch(avk_ctx *ctx, const avk_region_batch *batch,
                      const avk_compare_cfg *cfg, avk_compare_out *out);

/* Replaces the par_iter over solve_merge_region (src/main.rs:463-478). */
int avk_merge_batch(avk_ctx *ctx, const avk_region_batch *batch,
                    const avk_merge_cfg *cfg, avk_merge_out *out);

/* ---- several GPUs of one node behind the same call (SURVEY 8e).  The reference host is ONE process
 * (src/main.rs:251-271): the region_id-ordered list is cut into contiguous bins balanced by a cost proxy
 * (avk_partition_regions), bin k is solved on ctxs[k] by its own host thread, every device copies its
 * slice of the results straight into the caller's arrays at its bin offset, and the bins' summary
 * counters are added on the host (wrapping u64, like SummaryWriter's AddAssign).  No collective is
 * needed on the data path; result order == region order (src/main.rs:271).  Every context must hold
 * the reference (avk_set_reference). */
int avk_compare_batch_multi(avk_ctx *const *ctxs, uint32_t n_ctx, const avk_region_batch *batch,
                            const avk_compare_cfg *cfg, avk_compare_out *out);
int avk_merge_batch_multi(avk_ctx *const *ctxs, uint32_t n_ctx, const avk_region_batch *batch,
                          const avk_merge_cfg *cfg, avk_merge_out *out);
/* cuts[0..n_bins]: bin k = regions [cuts[k], cuts[k+1]).  Cost per region: (variants + 1) * window +
 * sum of max(|allele0|, |allele1|)^2.  Host only. */
int avk_partition_regions(const avk_region_batch *batch, uint32_t n_bins, uint64_t *cuts);
/* One bin on one context (the building block of the calls above; also what a one-process-per-GPU
 * launcher calls with its own bin): regions [lo, hi) are solved and written to out->status[lo..hi) etc.;
 * totals / strat_totals receive this bin's sums only. */
int avk_compare_batch_range(avk_ctx *ctx, const avk_region_batch *batch, uint64_t lo, uint64_t hi,
                            const avk_compare_cfg *cfg, avk_compare_out *out);

/* Batched global edit distance == wfa_ed (src/util/sequence_alignment.rs:9-13).
 * Pair p aligns pool[a_off[p]..+a_len[p]] against pool[b_off[p]..+b_len[p]]. */
int avk_wfa_ed_batch(avk_ctx *ctx, uint64_t n_pairs, const uint8_t *pool, uint64_t pool_len,
                     const uint64_t *a_off, const uint32_t *a_len,
                     const uint64_t *b_off, const uint32_t *b_len, uint32_t *ed_out);

/* Upper-bound layout for the optional sequence bundle: fills
 * seq_off[n_regions*5+1]; returns the pool size in *pool_len. Host only. */
int avk_compare_seq_offsets(const avk_region_batch *batch, uint64_t *seq_off, uint64_t *pool_len);

/* Device-resident variants used by bench.py (`value`, inputs already in HBM):
 * upload once, run many times, download once. */
/* ---- region builder (SURVEY 8f N1): src/parsing/region_generation.rs:352-469 for ONE contig and one BED interval
 * spanning it.  K call sets in one variant table, input k = variants [input_off[k], input_off[k+1]), each range sorted
 * by position (VCF order).  Variants not fully inside the contig are dropped (:551); all inputs are concatenated in
 * input order and stable-sorted by position (:352-373); a variant with pos >= window_end closes the cluster, where
 * window_start = first pos - flank (saturating) and window_end = max(pos + ref_len + flank) clipped to the contig
 * (:396-433).  The batch is built ON THE DEVICE and stays resident exactly as after avk_compare_upload (region_id =
 * first_region_id + running index, n_inputs = K), so avk_compare_run_resident can follow without a host round trip;
 * avk_regions_download copies it out (caller-allocated arrays sized from *n_regions / *n_variants; allele pool
 * capacity >= the input pool length). */
typedef struct {
    uint32_t n_inputs;
    const uint64_t *input_off;   /* [n_inputs + 1] */
    avk_variant_table variants;
} avk_callsets;
int avk_build_regions(avk_ctx *ctx, const avk_callsets *in, uint32_t contig, uint32_t flank, uint64_t first_region_id,
                      uint64_t *n_regions, uint64_t *n_variants);
/* The whole iterator of src/parsing/region_generation.rs:276-479 in one call: call sets that span several contigs and a
 * BED of high-confidence intervals.  variant_contig[v] = contig of variant v (reference order; every input's list sorted
 * by (contig, position), i.e. VCF order).  Intervals are 0-based half-open, sorted and non-overlapping within a contig
 * (the reference assumes the latter, :438-441), contigs in reference order; bed == NULL means one interval spanning each
 * contig.  Per contig (:283-292) and per interval (:374-470) in order: a variant starting before the interval is dropped
 * (Containment::Before), one starting behind it is left for the next interval (After), one that starts inside but ends
 * outside is dropped (Overlapping), a contained one joins the open cluster or -- pos >= window_end -- closes it
 * (get_variant_containment :796-812).  Every interval starts with a fresh window, so clusters never span two intervals;
 * window_start = first pos - flank (saturating, NOT clipped to the interval), window_end clipped to the contig length only
 * (:411-429); region_id runs on across intervals and contigs from first_region_id (:403-409, :459-466). */
typedef struct {
    uint32_t n_contigs;          /* == contigs of avk_set_reference */
    const uint64_t *first;       /* [n_contigs + 1]: intervals of contig c are first[c] .. first[c + 1] */
    const uint32_t *start;       /* 0-based, inclusive */
    const uint32_t *end;         /* 0-based, exclusive */
} avk_bed_intervals;
int avk_build_regions_bed(avk_ctx *ctx, const avk_callsets *in, const uint32_t *variant_contig, const avk_bed_intervals *bed,
                          uint32_t flank, uint64_t first_region_id, uint64_t *n_regions, uint64_t *n_variants);
int avk_regions_download(avk_ctx *ctx, avk_region_batch *out);

/* ---- VCF ingest (SURVEY 8f N2): parse_variant / parse_genotype / get_variant_type (src/parsing/region_generation.rs:565-758) on
 * the device, one record line per thread.  `text` = inflated VCF record lines (header lines starting with '#' are skipped;
 * BGZF inflate and the tabix query stay on the host), sample_index = column of the sample, contig_names = the reference's
 * contigs.  Output: the variants in record order with multi-ALT genotypes split into one variant per ALT allele, '*' and
 * symbolic ALTs, alleles over 10 kbp and BND / DUP records dropped, trailing bases trimmed (enable_trimming), types
 * inferred from INFO SVTYPE / TRID / allele lengths, raw_allele_space taken before trimming -- i.e. one input of an
 * avk_callsets table plus its variant_contig array.  A record the reference would fail on (missing GT key, ploidy > 2,
 * unsupported SVTYPE, ALT index out of range, ...) fails the call: AVK_ERR_INVALID with its line number and a code.
 * AVK_ERR_OOM with n_variants / allele_pool_len set: the caller's arrays are too small (2 * lines and len always suffice). */
typedef struct {
    uint64_t n_variants, allele_pool_len;        /* out */
    uint64_t cap_variants, cap_pool;             /* in: capacity of the arrays below */
    uint32_t *contig, *position;
    uint8_t *variant_type, *zygosity;
    uint32_t *raw_allele_space, *allele_off, *a0_len, *a1_len;
    uint8_t *allele_pool;
} avk_vcf_out;
int avk_vcf_parse(avk_ctx *ctx, const uint8_t *text, uint64_t len, const char *const *contig_names, uint32_t n_contigs, uint32_t sample_index,
                  int enable_trimming, avk_vcf_out *out, uint64_t *error_line, int32_t *error_code);

/* ---- BGZF inflate (SURVEY 8f N2 "parallel block inflate"; replaces the bgzf reader behind noodles_helper.rs:14-97 for a
 * whole file).  BGZF members (SAM specification 4.1: gzip members of at most 64 KiB with a BC extra subfield) are independent:
 * the host walks the member headers, one device thread inflates one member (RFC 1951 restated in csrc/avk_inflate.cuh) and,
 * with verify_crc != 0, checks its CRC-32 against the trailer.  A plain gzip file, a truncated file or a member that does not
 * inflate fails the call (avk_last_error names the member).
 * avk_bgzf_inflate: out == NULL -> *out_len = inflated size (host walk only); else the text is copied to `out`.
 * avk_vcf_parse_bgzf = avk_bgzf_inflate + avk_vcf_parse without the text leaving the device ('#' lines are skipped). */
int avk_bgzf_inflate(avk_ctx *ctx, const uint8_t *gz, uint64_t gz_len, int verify_crc, uint8_t *out, uint64_t out_cap, uint64_t *out_len);
int avk_vcf_parse_bgzf(avk_ctx *ctx, const uint8_t *gz, uint64_t gz_len, int verify_crc, const char *const *contig_names, uint32_t n_contigs,
                       uint32_t sample_index, int enable_trimming, avk_vcf_out *out, uint64_t *error_line, int32_t *error_code);

/* avk_bgzf_compress (SURVEY 8f N3: the BGZF compression behind truth.vcf.gz / query.vcf.gz / passing.vcf.gz and the BED outputs,
 * src/writers/compare_parallel.rs:25-214, variant_merger.rs:124-147): text -> a complete BGZF file (members of 0xff00 input
 * bytes + the EOF marker), one warp per member: dynamic-Huffman DEFLATE over a greedy LZ77 parse, a stored block where that does
 * not pay.  The bytes differ from the reference's compressor's (any valid DEFLATE stream is a valid member); the inflated
 * content, member sizes and CRCs are what zlib / htslib expect.  out == NULL -> *out_len = an upper bound of the size. */
int avk_bgzf_compress(avk_ctx *ctx, const uint8_t *text, uint64_t len, uint8_t *out, uint64_t cap, uint64_t *out_len);

/* ---- writers (SURVEY 8f N3): host-side text of what the kernels counted.  buf == NULL: *len receives the size needed.
 * avk_summary_write: the rows SummaryWriter::write_summary (src/writers/summary.rs:166-221, :243-420) emits for ONE
 * GroupTypeMetrics table -- `totals` = avk_compare_out::totals for region_label "ALL", or row s of strat_totals for the
 * label of stratum s -- for the metrics listed (0 GT, 1 HAP, 2 WEIGHTED_HAP, 3 BASEPAIR, 4 RECORD_BP, in this order):
 * per metric the ALL row, the non-empty variant types, the non-empty JointIndel / JointStructuralVariant /
 * JointTandemRepeat rows; recall / precision / F1 as f64 in the csv crate's formatting (shortest round trip), empty when
 * undefined (src/data_types/summary_metrics.rs:48-74); filter column "ALL"; csv != 0 -> ',' instead of tab (:169-170). */
int avk_summary_write(const uint64_t *totals, const uint8_t *metrics, uint32_t n_metrics, const char *compare_label, const char *region_label,
                      int csv, int header, char *buf, uint64_t cap, uint64_t *len);
/* avk_vcf_records_write: the body lines VariantCategorizer::write_variants (src/writers/variant_categorizer.rs:178-237)
 * writes for input `side` (0 truth, 1 query) of regions [lo, hi): CHROM POS . REF ALT . . . GT:BD:EA:OA:RI and the
 * sample column built from the variant's zygosity, var_class / var_expected / var_observed and the region id. */
int avk_vcf_records_write(const avk_region_batch *batch, uint32_t side, const char *const *contig_names, uint32_t n_contigs,
                          const uint8_t *var_class, const uint8_t *var_expected, const uint8_t *var_observed, uint64_t lo, uint64_t hi,
                          char *buf, uint64_t cap, uint64_t *len);
/* The labelled records of input `side` (0 truth, 1 query) of the resident compare batch, formatted and BGZF-compressed
 * on the device: out = a BGZF file whose inflated text is header[0..header_len) followed by exactly the lines
 * avk_vcf_records_write(batch, side, contig_names, n_contigs, var_class, var_expected, var_observed, lo, lo + n) returns
 * for the resident bin [lo, lo + n) and the last result (valid wherever avk_compare_download would succeed).  With eof != 0
 * the file is byte for byte avk_bgzf_compress(header || those lines); eof == 0 leaves out the 28-byte EOF member, so that
 * the files of consecutive bins (the header on the first only, eof on the last only) concatenate into one valid file.
 * region_id: the caller's host array, indexed like the batch given to avk_compare_upload[_range] (elements lo .. lo+n-1
 * are read); NULL when the resident batch was built by avk_build_regions[_bed], whose ids are on the device.
 * A region whose contig is >= n_contigs fails the call (AVK_ERR_INVALID), as in avk_vcf_records_write.
 * out == NULL: *out_len = an upper bound of the size.  Otherwise cap < size -> AVK_ERR_OOM with *out_len = the exact size. */
int avk_compare_records_bgzf(avk_ctx *ctx, uint32_t side, const char *const *contig_names, uint32_t n_contigs,
                             const uint64_t *region_id, const uint8_t *header, uint64_t header_len, int eof,
                             uint8_t *out, uint64_t cap, uint64_t *out_len);

/* The outputs of `aardvark merge` that are functions of avk_merge_out (host only; regions with status != 0 are skipped as
 * src/main.rs:507-524 skips failed regions; `result->status` may be NULL = all solved):
 * avk_merge_records_write: body lines of passing.vcf.gz (VariantMerger::write_variants, src/writers/variant_merger.rs:198-287)
 *   for regions [lo, hi): the variants of the lowest passing input (input 0 for `identical`), INFO
 *   SOURCES=<labels of the passing inputs>;MR=<identical|no_conflict|majority|conflict_select>, FORMAT GT:RI;
 * avk_merge_regions_write: BED lines chrom, start, end, {reason}_{region_id} (write_region :294-309) of the passing
 *   (passing != 0: regions.bed) or failed (failed_regions.bed) regions of [lo, hi);
 * avk_merge_summary_write: MergeSummaryWriter (src/writers/merge_summary.rs:56-112): pass / fail variant counts per
 *   (merge reason with its indices, variant type, input) in the reference's key order, e.g. `majority_0_2 Snv 1 ilmn 0 37810`. */
int avk_merge_records_write(const avk_region_batch *batch, const avk_merge_out *result, const char *const *contig_names, uint32_t n_contigs,
                            const char *const *input_labels, uint64_t lo, uint64_t hi, char *buf, uint64_t cap, uint64_t *len);
int avk_merge_regions_write(const avk_region_batch *batch, const avk_merge_out *result, const char *const *contig_names, uint32_t n_contigs,
                            int passing, uint64_t lo, uint64_t hi, char *buf, uint64_t cap, uint64_t *len);
int avk_merge_summary_write(const avk_region_batch *batch, const avk_merge_out *result, const char *const *input_labels, int csv, int header,
                            char *buf, uint64_t cap, uint64_t *len);

/* ---- resident merge: the batch stays on the device between the merge and its outputs (the merge chain K BGZF VCFs ->
 * avk_vcf_parse_bgzf -> avk_build_regions_bed -> avk_merge_run_resident -> the writers below never sends the batch or the
 * result to the host).
 * avk_merge_upload_range: regions [lo, hi) of a host batch (1 <= n_inputs <= 32) become the resident batch.
 * avk_merge_run_resident: solves the resident batch (from avk_merge_upload_range or avk_build_regions[_bed]); the merge
 *   result stays on the device.  It overwrites the status array a compare result uses: after it avk_compare_download,
 *   avk_compare_result_device and avk_compare_records_bgzf are refused, and a compare run (or any upload, build,
 *   avk_set_reference or avk_wfa_ed_batch) in turn drops the merge result.  avk_merge_batch leaves its result resident as
 *   well, and so does every context of avk_merge_batch_multi for its own bin.
 * avk_merge_download: status / classification / n_indices / indices of the resident bin into out->...[lo, hi) (out->status
 *   required, the others may be NULL).
 * Every merge call below fails with AVK_ERR_INVALID (and a message) when no merge result is resident; the context stays usable. */
int avk_merge_upload_range(avk_ctx *ctx, const avk_region_batch *batch, uint64_t lo, uint64_t hi);
int avk_merge_run_resident(avk_ctx *ctx, const avk_merge_cfg *cfg);
int avk_merge_download(avk_ctx *ctx, avk_merge_out *out);
/* passing.vcf.gz and regions.bed.gz / failed_regions.bed.gz of the resident merge result, formatted and BGZF-compressed on the
 * device: out = byte for byte avk_bgzf_compress(header || avk_merge_records_write(batch, result, contig_names, n_contigs,
 * input_labels, lo, lo + n)), resp. avk_bgzf_compress(avk_merge_regions_write(batch, result, contig_names, n_contigs, passing,
 * lo, lo + n)), for the resident bin [lo, lo + n).  region_id, eof, out == NULL (an upper bound of the size) and cap < size
 * (AVK_ERR_OOM with *out_len = the exact size) behave as in avk_compare_records_bgzf.  A region whose contig is >= n_contigs,
 * a null contig name or a null label (input_labels has n_inputs entries) fails the call with AVK_ERR_INVALID. */
int avk_merge_records_bgzf(avk_ctx *ctx, const char *const *contig_names, uint32_t n_contigs, const char *const *input_labels,
                           const uint64_t *region_id, const uint8_t *header, uint64_t header_len, int eof,
                           uint8_t *out, uint64_t cap, uint64_t *out_len);
int avk_merge_regions_bgzf(avk_ctx *ctx, const char *const *contig_names, uint32_t n_contigs, int passing,
                           const uint64_t *region_id, int eof, uint8_t *out, uint64_t cap, uint64_t *out_len);
/* The merge summary without the batch on the host.  A row counts the variants of one key (classification, index list,
 * variant type, input) over the solved regions of the resident bin; the index list is a bit mask (bit k <=> input k; for
 * conflict selection the selected input), and a key's variants all pass or all fail.  avk_merge_summary_counts: the keys are
 * counted on the device (sort + run-length encoding), only the distinct ones are copied; rows == NULL: *n_rows = the number
 * of rows; cap < that number: AVK_ERR_OOM with *n_rows set.  Rows come in no particular order.
 * avk_merge_summary_rows_write (host only): rows of one or several bins / GPUs, simply concatenated (rows that share a key
 * add up) -> the text avk_merge_summary_write gives over the whole batch, in the same order and csv quoting. */
typedef struct avk_merge_summary_row {
    uint32_t indices;
    uint8_t classification, variant_type, input, pad;
    uint64_t pass_variants, fail_variants;
} avk_merge_summary_row;
int avk_merge_summary_counts(avk_ctx *ctx, avk_merge_summary_row *rows, uint64_t cap, uint64_t *n_rows);
int avk_merge_summary_rows_write(const avk_merge_summary_row *rows, uint64_t n_rows, uint32_t n_inputs, const char *const *input_labels,
                                 int csv, int header, char *buf, uint64_t cap, uint64_t *len);

int avk_compare_upload(avk_ctx *ctx, const avk_region_batch *batch);
int avk_compare_upload_range(avk_ctx *ctx, const avk_region_batch *batch, uint64_t lo, uint64_t hi);
int avk_compare_run_resident(avk_ctx *ctx, const avk_compare_cfg *cfg);
/* copies the resident bin's results into out->...[lo..hi) / [v_base..) of the caller's arrays.  AVK_ERR_INVALID when out
 * asks for what the last pass did not compute: region_metrics after a run without AVK_CMP_KEEP_REGION_ROWS, containment
 * after avk_compare_run_resident (which never computes it), and stratified sums (strat_totals with n_strata > 0) always:
 * request those from avk_compare_batch*. */
int avk_compare_download(avk_ctx *ctx, avk_compare_out *out);
/* DEVICE addresses of the resident bin's results (valid until the next call on the context): what a
 * one-process-per-GPU run hands to its single NCCL gather, so that results travel GPU -> root GPU over
 * NVLink and reach the host in one copy.  totals = [AVK_N_GROUPS*AVK_N_METRICS] sums, type mask, solved
 * blocks, error blocks (u64 each). */
typedef struct avk_compare_dev_view {
    uint64_t lo, n_regions;      /* resident bin = regions [lo, lo + n_regions) of the uploaded batch */
    uint64_t v_base, n_variants; /* = variants [v_base, v_base + n_variants) of its variant table */
    void *status;                /* int32  [n_regions] */
    void *ed1, *ed2;             /* uint32 [n_regions] */
    void *type_mask;             /* uint16 [n_regions] */
    void *var_expected, *var_observed, *var_class; /* uint8 [n_variants] */
    void *totals;                /* uint64 [AVK_N_GROUPS*AVK_N_METRICS + 3] */
} avk_compare_dev_view;
int avk_compare_result_device(avk_ctx *ctx, avk_compare_dev_view *view);
/* Milliseconds spent in the phases of the last resident run (CUDA events on the
 * library's stream): [0] alt_ed kernel, [1] search kernel(s), [2] heavy ED kernel,
 * [3] finalize/reduce, [4] total. */
int avk_last_timings(avk_ctx *ctx, float *ms5);
int avk_last_work(avk_ctx *ctx, avk_work_counters *out);
/* Diagnostics: with AVK_SPEC_PROFILE=1 in the environment k_search_spec records per-cluster phase clocks (64 bytes per
 * cluster, up to 65536 clusters); this copies the first n 64-bit words back (tools/spec_profile.py). */
int avk_spec_profile(avk_ctx *ctx, unsigned long long *out, uint32_t n);
/* Diagnostics: clusters that overflowed workspace tiers 0, 1, 2 in the last run. */
int avk_last_tier_overflow(avk_ctx *ctx, uint32_t *out3);
/* Diagnostics: device milliseconds spent in workspace tiers 0, 1, 2 in the last run. */
int avk_last_tier_ms(avk_ctx *ctx, float *out3);
/* INT32 ALU throughput probe (add/max/xor chains), integer ops per second: the measured
 * denominator of the integer roofline, obtained the way MEASURED_PEAKS.json obtains HBM GB/s. */
int avk_int_peak(avk_ctx *ctx, double *ops_per_s);
/* Number of kernel launches issued by the library since avk_create. */
uint64_t avk_launch_count(const avk_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* AARDVARK_B200_H */
