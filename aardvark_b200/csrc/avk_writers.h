// avk_writers.h -- host side of the two writers that consume the compare path's results (SURVEY 8f N3):
//   * avk_summary_write: SummaryWriter::write_summary (src/writers/summary.rs:166-221, write_group / write_category /
//     write_gt_category :243-420) over one GroupTypeMetrics table, i.e. the [AVK_N_GROUPS][AVK_N_METRICS] sums the kernels
//     accumulate (avk_compare_out::totals or one row of strat_totals);
//   * avk_vcf_records_write: VariantCategorizer::write_variants (src/writers/variant_categorizer.rs:178-237): the
//     GT:BD:EA:OA:RI record of every variant of one input, in region order;
//   * the three outputs of `aardvark merge` that are functions of the merge path's results (avk_merge_out):
//     avk_merge_records_write (VariantMerger::write_variants, src/writers/variant_merger.rs:198-287: body lines of
//     passing.vcf.gz), avk_merge_regions_write (write_region :294-309: regions.bed / failed_regions.bed) and
//     avk_merge_summary_write (MergeSummaryWriter, src/writers/merge_summary.rs:56-112), whose ordering and formatting
//     avk_merge_summary_rows_write shares for the per-key counts the device computes (avk_merge_summary_counts).
// Plain C++17, no CUDA: the counters and labels were computed on the device, these functions only format them.
#pragma once
#include <charconv>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/aardvark_b200.h"

namespace avk_writers {

// one field the way the csv crate writes it (QuoteStyle::Necessary): quoted, with doubled quotes, iff it contains the
// delimiter, a quote, CR or LF
static inline void csv_field(std::string &o, const char *f, char delim) {
    bool q = false;
    for (const char *c = f; *c; ++c) if (*c == delim || *c == '"' || *c == '\n' || *c == '\r') { q = true; break; }
    if (!q) { o += f; return; }
    o += '"';
    for (const char *c = f; *c; ++c) { if (*c == '"') o += '"'; o += *c; }
    o += '"';
}

// f64 -> text the way the csv crate serialises it (ryu::Buffer::format_finite -- shortest round-trip digits, then ryu's
// "pretty" layout: plain decimals while the decimal point lies within [-5, 16] digits of the first digit, a trailing ".0"
// for integers, otherwise d.ddde[-]x)
static inline std::string ryu_f64(double v) {
    if (v == 0.0) return "0.0";
    char sci[64];
    auto r = std::to_chars(sci, sci + sizeof(sci), v, std::chars_format::scientific);   // shortest round-trip, d[.ddd]e[+-]xx
    std::string s(sci, r.ptr);
    std::string out;
    size_t i = 0;
    if (s[0] == '-') { out = "-"; i = 1; }
    const size_t e = s.find('e');
    std::string digits;
    for (size_t k = i; k < e; ++k) if (s[k] != '.') digits.push_back(s[k]);
    const int exp10 = std::atoi(s.c_str() + e + 1);
    const int length = (int)digits.size();
    const int kk = exp10 + 1;                            // 10^(kk-1) <= |v| < 10^kk
    const int k = kk - length;                           // v = digits * 10^k
    if (0 <= k && kk <= 16) { out += digits; out.append((size_t)k, '0'); out += ".0"; }             // 1234e7 -> 12340000000.0
    else if (0 < kk && kk <= 16) { out += digits.substr(0, (size_t)kk); out += "."; out += digits.substr((size_t)kk); }   // 1234e-2 -> 12.34
    else if (-5 < kk && kk <= 0) { out += "0."; out.append((size_t)(-kk), '0'); out += digits; }     // 1234e-6 -> 0.001234
    else if (length == 1) { out += digits; out += "e"; out += std::to_string(kk - 1); }              // 1e30
    else { out += digits.substr(0, 1); out += "."; out += digits.substr(1); out += "e"; out += std::to_string(kk - 1); }   // 1234e30 -> 1.234e33
    return out;
}

static const char *const METRIC_NAMES[5] = {"GT", "HAP", "WEIGHTED_HAP", "BASEPAIR", "RECORD_BP"};          // grouped_metrics.rs:10-27 (serde renames)
static const int METRIC_COL[5] = {AVK_M_GT, AVK_M_HAP, AVK_M_WEIGHTED_HAP, AVK_M_BASEPAIR, AVK_M_RECORD_BP};
static const char *const TYPE_NAMES[AVK_N_VARIANT_TYPES] = {"Snv", "Insertion", "Deletion", "Indel", "SvInsertion", "SvDeletion", "SvDuplication",
                                                            "SvInversion", "SvBreakend", "TrContraction", "TrExpansion", "Unknown"};   // {variant_type:?}

struct Row4 { uint64_t tp, fn, qtp, qfp, fn_gt, fp_gt; };

static inline void emit_row(std::string &o, char d, const char *label, const char *comparison, const char *region_label, const char *variant_type,
                            const Row4 &m, bool gt) {
    // SummaryRow (summary.rs:33-114): compare_label comparison region_label filter variant_type truth_total truth_tp truth_fn
    // query_total query_tp query_fp metric_recall metric_precision metric_f1 truth_fn_gt query_fp_gt; None -> empty field
    csv_field(o, label, d); o += d; o += comparison; o += d; csv_field(o, region_label, d); o += d; o += "ALL"; o += d; o += variant_type; o += d;
    o += std::to_string(m.tp + m.fn); o += d; o += std::to_string(m.tp); o += d; o += std::to_string(m.fn); o += d;
    o += std::to_string(m.qtp + m.qfp); o += d; o += std::to_string(m.qtp); o += d; o += std::to_string(m.qfp); o += d;
    const bool hr = m.tp + m.fn > 0, hp = m.qtp + m.qfp > 0;                                        // summary_metrics.rs:48-74
    const double recall = hr ? (double)m.tp / (double)(m.tp + m.fn) : 0.0, precision = hp ? (double)m.qtp / (double)(m.qtp + m.qfp) : 0.0;
    if (hr) o += ryu_f64(recall);
    o += d;
    if (hp) o += ryu_f64(precision);
    o += d;
    if (hr && hp) {
        const double f1 = 2.0 * recall * precision / (recall + precision);
        if (f1 == f1) o += ryu_f64(f1); else o += "NaN";                                             // 0 / 0 when both are 0.0
    }
    o += d;
    if (gt) o += std::to_string(m.fn_gt);
    o += d;
    if (gt) o += std::to_string(m.fp_gt);
    o += '\n';
}

static inline Row4 row_of(const uint64_t *totals, int group, int metric) {
    const uint64_t *p = totals + (size_t)group * AVK_N_METRICS + METRIC_COL[metric];
    Row4 r = {p[0], p[1], p[2], p[3], 0, 0};
    if (metric == 0) { r.fn_gt = totals[(size_t)group * AVK_N_METRICS + AVK_M_GT_TRUTH_FN_GT]; r.fp_gt = totals[(size_t)group * AVK_N_METRICS + AVK_M_GT_QUERY_FP_GT]; }
    return r;
}
static inline bool empty4(const Row4 &r) { return r.tp + r.fn + r.qtp + r.qfp == 0; }                // SummaryMetrics::is_empty

// write_group (:243-274): for every requested metric the ALL row, the non-empty per-type rows in VariantType order (the
// BTreeMap's), then the non-empty joint rows JointIndel, JointStructuralVariant, JointTandemRepeat (:176-204)
static inline std::string summary_text(const uint64_t *totals, const uint8_t *metrics, uint32_t n_metrics, const char *compare_label,
                                       const char *region_label, char delim, bool header) {
    std::string o;
    if (header) {
        const char *cols[16] = {"compare_label", "comparison", "region_label", "filter", "variant_type", "truth_total", "truth_tp", "truth_fn", "query_total",
                                "query_tp", "query_fp", "metric_recall", "metric_precision", "metric_f1", "truth_fn_gt", "query_fp_gt"};
        for (int c = 0; c < 16; ++c) { o += cols[c]; o += c == 15 ? '\n' : delim; }
    }
    static const int joint_indel[] = {AVK_VT_INSERTION, AVK_VT_DELETION, AVK_VT_INDEL};
    static const int joint_sv[] = {AVK_VT_SV_INSERTION, AVK_VT_SV_DELETION, AVK_VT_SV_DUPLICATION, AVK_VT_SV_INVERSION, AVK_VT_SV_BREAKEND};
    static const int joint_tr[] = {AVK_VT_TR_EXPANSION, AVK_VT_TR_CONTRACTION};
    struct Joint { const char *label; const int *types; int n; };
    const Joint joints[3] = {{"JointIndel", joint_indel, 3}, {"JointStructuralVariant", joint_sv, 5}, {"JointTandemRepeat", joint_tr, 2}};
    for (uint32_t q = 0; q < n_metrics; ++q) {
        const int m = metrics[q];
        if (m < 0 || m > 4) continue;
        const bool gt = m == 0;
        emit_row(o, delim, compare_label, METRIC_NAMES[m], region_label, "ALL", row_of(totals, 0, m), gt);
        for (int t = 0; t < AVK_N_VARIANT_TYPES; ++t) {
            const Row4 r = row_of(totals, 1 + t, m);
            if (!empty4(r)) emit_row(o, delim, compare_label, METRIC_NAMES[m], region_label, TYPE_NAMES[t], r, gt);
        }
        for (const Joint &j : joints) {
            Row4 s = {0, 0, 0, 0, 0, 0};
            for (int k = 0; k < j.n; ++k) { const Row4 r = row_of(totals, 1 + j.types[k], m); s.tp += r.tp; s.fn += r.fn; s.qtp += r.qtp; s.qfp += r.qfp; s.fn_gt += r.fn_gt; s.fp_gt += r.fp_gt; }
            if (!empty4(s)) emit_row(o, delim, compare_label, METRIC_NAMES[m], region_label, j.label, s, gt);
        }
    }
    return o;
}

// write_variants (variant_categorizer.rs:178-237) for input `side` (0 truth, 1 query) of regions [lo, hi): one VCF body line per
// variant -- CHROM, 1-based POS, no ID / QUAL / FILTER / INFO, FORMAT GT:BD:EA:OA:RI and the sample column
static inline std::string vcf_records_text(const avk_region_batch *b, uint32_t side, const char *const *contig_names, const uint8_t *var_class,
                                           const uint8_t *var_expected, const uint8_t *var_observed, uint64_t lo, uint64_t hi) {
    static const char *const GT[6] = {".", "0/0", "0/1", "0|1", "1|0", "1/1"};                       // PhasedZygosity -> genotype string (:190-197)
    static const char *const BD[4] = {"UNK", "TP", "FN", "FP"};                                      // Classification (variant_metrics.rs:11-21)
    const avk_variant_table &t = b->variants;
    const uint64_t K = b->n_inputs;
    std::string o;
    for (uint64_t r = lo; r < hi; ++r)
        for (uint64_t v = b->var_off[r * K + side]; v < b->var_off[r * K + side + 1]; ++v) {
            o += contig_names[b->contig[r]]; o += '\t';
            o += std::to_string((uint64_t)t.position[v] + 1); o += "\t.\t";
            o.append((const char *)t.allele_pool + t.allele_off[v], t.a0_len[v]); o += '\t';
            o.append((const char *)t.allele_pool + t.allele_off[v] + t.a0_len[v], t.a1_len[v]);
            o += "\t.\t.\t.\tGT:BD:EA:OA:RI\t";
            o += GT[t.zygosity[v] <= AVK_ZYG_HOM_ALT ? t.zygosity[v] : 0]; o += ':';
            o += BD[var_class[v] <= AVK_CLASS_FP ? var_class[v] : 0]; o += ':';
            o += std::to_string((int)var_expected[v]); o += ':';
            o += std::to_string((int)var_observed[v]); o += ':';
            o += std::to_string((int32_t)b->region_id[r]);                                           // `region_id as i32` (:214)
            o += '\n';
        }
    return o;
}

// ---- aardvark merge ----------------------------------------------------------------------------------------------------
// MergeClassification::simplify (src/data_types/merge_benchmark.rs:47-55)
static inline const char *merge_simple(uint8_t c) {
    switch (c) {
        case AVK_MERGE_NO_CONFLICT: return "no_conflict";
        case AVK_MERGE_MAJORITY_AGREE: return "majority";
        case AVK_MERGE_CONFLICT_SELECTION: return "conflict_select";
        case AVK_MERGE_BASEPAIR_IDENTICAL: return "identical";
        default: return "different";
    }
}
// the input whose variants are copied (variant_merger.rs:172-178); -1: the region fails
static inline int merge_source(uint8_t c, uint8_t n, const uint8_t *idx) {
    if (c == AVK_MERGE_BASEPAIR_IDENTICAL) return 0;
    if (c == AVK_MERGE_DIFFERENT || n == 0) return -1;
    return idx[0];
}
struct MergeView {
    const int32_t *status;          // may be NULL (all solved); regions with status != 0 are skipped everywhere (src/main.rs:507-524)
    const uint8_t *cls, *n_idx, *idx;
};
static inline bool merge_solved(const MergeView &m, uint64_t r) { return !m.status || m.status[r] == 0; }

// write_variants (variant_merger.rs:198-287) for the passing regions of [lo, hi): CHROM, 1-based POS, ".", REF, ALT, ".", ".",
// SOURCES=<labels of the passing inputs -- all of them for `identical`>;MR=<simplify()>, GT:RI, <genotype>:<region_id as i32>
static inline std::string merge_records_text(const avk_region_batch *b, const char *const *contig_names, const char *const *labels, const MergeView &m,
                                             uint64_t lo, uint64_t hi) {
    static const char *const GT[6] = {".", "0/0", "0/1", "0|1", "1|0", "1/1"};
    const avk_variant_table &t = b->variants;
    const uint64_t K = b->n_inputs;
    std::string o, info;
    for (uint64_t r = lo; r < hi; ++r) {
        if (!merge_solved(m, r)) continue;
        const uint8_t c = m.cls[r], n = m.n_idx[r];
        const uint8_t *idx = m.idx + r * K;
        const int src = merge_source(c, n, idx);
        if (src < 0) continue;
        info = "SOURCES=";
        if (c == AVK_MERGE_BASEPAIR_IDENTICAL) for (uint64_t k = 0; k < K; ++k) { if (k) info += ','; info += labels[k]; }
        else for (uint8_t k = 0; k < n; ++k) { if (k) info += ','; info += labels[idx[k]]; }
        info += ";MR="; info += merge_simple(c);
        for (uint64_t v = b->var_off[r * K + src]; v < b->var_off[r * K + src + 1]; ++v) {
            o += contig_names[b->contig[r]]; o += '\t';
            o += std::to_string((uint64_t)t.position[v] + 1); o += "\t.\t";
            o.append((const char *)t.allele_pool + t.allele_off[v], t.a0_len[v]); o += '\t';
            o.append((const char *)t.allele_pool + t.allele_off[v] + t.a0_len[v], t.a1_len[v]);
            o += "\t.\t.\t"; o += info; o += "\tGT:RI\t";
            o += GT[t.zygosity[v] <= AVK_ZYG_HOM_ALT ? t.zygosity[v] : 0]; o += ':';
            o += std::to_string((int32_t)b->region_id[r]);
            o += '\n';
        }
    }
    return o;
}
// write_region (:294-309): BED4 lines chrom, start, end, {simplify()}_{region_id} of the passing (passing != 0) or the failed
// regions of [lo, hi) -- noodles writes the 1-based inclusive feature start back as the 0-based BED start
static inline std::string merge_regions_text(const avk_region_batch *b, const char *const *contig_names, const MergeView &m, uint64_t lo, uint64_t hi, bool passing) {
    const uint64_t K = b->n_inputs;
    std::string o;
    for (uint64_t r = lo; r < hi; ++r) {
        if (!merge_solved(m, r)) continue;
        const bool pass = merge_source(m.cls[r], m.n_idx[r], m.idx + r * K) >= 0;
        if (pass != passing) continue;
        o += contig_names[b->contig[r]]; o += '\t'; o += std::to_string(b->start[r]); o += '\t'; o += std::to_string(b->end[r]); o += '\t';
        o += merge_simple(m.cls[r]); o += '_'; o += std::to_string(b->region_id[r]); o += '\n';
    }
    return o;
}
// MergeSummaryWriter (merge_summary.rs:56-112): pass / fail variant counts keyed by (MergeClassification, VariantType, vcf index)
// in the derived Ord -- Different < NoConflict{indices} < MajorityAgree{indices} < ConflictSelection{index} <
// BasepairIdentical, index lists compared lexicographically -- one row per key: merge_reason (Display: simplify() + "_i" per
// index, merge_benchmark.rs:22-44), variant_type ({:?}), vcf_index, vcf_label, pass_variants, fail_variants.
// The counts of either source -- a batch and its result on the host, or the avk_merge_summary_row keys the device counted --
// go into one ordered map, and one function writes it.
typedef std::tuple<uint8_t, std::vector<uint8_t>, uint8_t, uint32_t> MergeSummaryKey;       // class, indices, variant type, vcf index
typedef std::map<MergeSummaryKey, std::pair<uint64_t, uint64_t>> MergeSummaryCounts;       // key -> (pass, fail)

static inline void merge_summary_count_batch(MergeSummaryCounts &counts, const avk_region_batch *b, const MergeView &m) {
    const avk_variant_table &t = b->variants;
    const uint64_t K = b->n_inputs;
    for (uint64_t r = 0; r < b->n_regions; ++r) {
        if (!merge_solved(m, r)) continue;
        const uint8_t c = m.cls[r];
        const uint8_t *idx = m.idx + r * K;
        std::vector<uint8_t> ind;
        if (c == AVK_MERGE_NO_CONFLICT || c == AVK_MERGE_MAJORITY_AGREE) ind.assign(idx, idx + m.n_idx[r]);
        else if (c == AVK_MERGE_CONFLICT_SELECTION) ind.assign(idx, idx + 1);
        for (uint64_t k = 0; k < K; ++k) {
            bool pass = c == AVK_MERGE_BASEPAIR_IDENTICAL;
            for (uint8_t i : ind) pass = pass || i == k;
            for (uint64_t v = b->var_off[r * K + k]; v < b->var_off[r * K + k + 1]; ++v) {
                auto &e = counts[MergeSummaryKey(c, ind, t.variant_type[v], (uint32_t)k)];
                if (pass) e.first += 1; else e.second += 1;
            }
        }
    }
}
// rows of one or several bins: the index list of a row is the ascending list of the bits of `indices`; rows that share a key
// add up
static inline void merge_summary_count_rows(MergeSummaryCounts &counts, const avk_merge_summary_row *rows, uint64_t n_rows) {
    for (uint64_t i = 0; i < n_rows; ++i) {
        const avk_merge_summary_row &w = rows[i];
        std::vector<uint8_t> ind;
        for (uint32_t k = 0; k < 32; ++k) if (w.indices >> k & 1u) ind.push_back((uint8_t)k);
        auto &e = counts[MergeSummaryKey(w.classification, ind, w.variant_type, w.input)];
        e.first += w.pass_variants; e.second += w.fail_variants;
    }
}
static inline std::string merge_summary_format(const MergeSummaryCounts &counts, const char *const *labels, char delim, bool header) {
    std::string o;
    if (header && !counts.empty()) {        // (the csv crate writes the header with the first serialised row)
        const char *cols[6] = {"merge_reason", "variant_type", "vcf_index", "vcf_label", "pass_variants", "fail_variants"};
        for (int c = 0; c < 6; ++c) { o += cols[c]; o += c == 5 ? '\n' : delim; }
    }
    for (const auto &kv : counts) {
        const uint8_t c = std::get<0>(kv.first), vt = std::get<2>(kv.first);
        o += merge_simple(c);
        for (uint8_t i : std::get<1>(kv.first)) { o += '_'; o += std::to_string((int)i); }
        o += delim; o += TYPE_NAMES[vt < AVK_N_VARIANT_TYPES ? vt : AVK_N_VARIANT_TYPES - 1]; o += delim;
        o += std::to_string(std::get<3>(kv.first)); o += delim; csv_field(o, labels[std::get<3>(kv.first)], delim); o += delim;
        o += std::to_string(kv.second.first); o += delim; o += std::to_string(kv.second.second); o += '\n';
    }
    return o;
}
static inline std::string merge_summary_text(const avk_region_batch *b, const char *const *labels, const MergeView &m, char delim, bool header) {
    MergeSummaryCounts counts;
    merge_summary_count_batch(counts, b, m);
    return merge_summary_format(counts, labels, delim, header);
}

}  // namespace avk_writers
