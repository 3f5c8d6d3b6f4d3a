"""The debug folder of `aardvark compare`: region_summary.tsv.gz and region_sequences.tsv.gz.

CPU: the host formatters (avk_region_summary_write / avk_region_sequences_write) against literal text on the golden clusters,
hand-made rows, and the oracle's rows and bundle on a seeded batch.  GPU: the device writers against avk_bgzf_compress of
the host formatters' text, the BGZF layout and zlib, and the rows / bundle behind them against the CPU oracle -- after a
resident pass with AVK_CMP_KEEP_REGION_ROWS | AVK_CMP_KEEP_SEQUENCES and after avk_compare_batch with the outputs."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import oracle_py as orc
from aardvark_b200 import abi, synth
from aardvark_b200.batch import CompareOutputs, RegionBatch, seq_offsets
from aardvark_b200.lib import compare_cfg
from aardvark_b200.types import CompareConfig, CompareRegion
from aardvark_b200.writers import METRICS, _bind, _c_names, region_sequence_lines, region_summary_lines
from golden_cases import COMPARE_CASES, MOCK_CHR1

AVK_ERR_INVALID, AVK_ERR_OOM = -1, -4
SUMMARY_HEADER = "region_id\tcoordinates\tcomparison\ttruth_tp\ttruth_fn\tquery_tp\tquery_fp\ttruth_fn_gt\tquery_fp_gt\n"
SEQUENCES_HEADER = b"region_id\tcoordinates\tref_seq\ttruth_seq1\ttruth_seq2\tquery_seq1\tquery_seq2\n"
ALL = tuple(METRICS)
IDS = [0, 1 << 31, (1 << 32) + 5]


def _oracle(batch, refs, cfg=CompareConfig(enable_sequences=True)):
    off, plen = seq_offsets(batch)
    return orc.compare_batch(batch, refs, compare_cfg(cfg), seq_off=off, seq_pool_len=plen)


def _golden():
    regions = [CompareRegion(IDS[i % 3], r.coordinates, r.truth_variants, r.truth_zygosity, r.query_variants, r.query_zygosity)
               for i, (_, r, _) in enumerate(COMPARE_CASES)]
    batch = RegionBatch.from_compare_regions(regions, {"mock_chr1": 0})
    return batch, _oracle(batch, [MOCK_CHR1])


def parse_summary(text, n_metrics):
    """region_summary.tsv -> {region_id: {metric: (tp, fn, qtp, qfp, fn_gt, fp_gt)}} (None for the empty GT-only fields)"""
    lines = text.split("\n")
    assert lines[0] + "\n" == SUMMARY_HEADER and lines[-1] == ""
    rows = {}
    for ln in lines[1:-1]:
        f = ln.split("\t")
        assert len(f) == 9
        c = tuple(int(x) for x in f[3:7]) + tuple(int(x) if x else None for x in f[7:9])
        assert (c[4] is None) == (f[2] != "GT")
        rows.setdefault(int(f[0]), {})[f[2]] = (f[1], c)
    assert all(len(v) == n_metrics for v in rows.values())
    return rows


def parse_sequences(text):
    lines = text.split(b"\n")
    assert lines[0] + b"\n" == SEQUENCES_HEADER and lines[-1] == b""
    out = {}
    for ln in lines[1:-1]:
        f = ln.split(b"\t")
        assert len(f) == 7
        out[int(f[0])] = (f[1].decode(), tuple(f[2:]))
    return out


def _joint(row, m):
    col = [abi.M_GT, abi.M_HAP, abi.M_WEIGHTED_HAP, abi.M_BASEPAIR, abi.M_RECORD_BP][m]
    c = tuple(int(x) for x in row[0, col:col + 4])
    return c + ((int(row[0, abi.M_GT_TRUTH_FN_GT]), int(row[0, abi.M_GT_QUERY_FP_GT])) if m == 0 else (None, None))


# ---- CPU: the host formatters ----------------------------------------------------------------------------------------------
GOLDEN_SUMMARY_3 = (
    "0\tmock_chr1:1-10\tGT\t1\t0\t1\t0\t0\t0\n"
    "0\tmock_chr1:1-10\tHAP\t1\t0\t1\t0\t\t\n"
    "0\tmock_chr1:1-10\tWEIGHTED_HAP\t1\t0\t1\t0\t\t\n"
    "0\tmock_chr1:1-10\tBASEPAIR\t2\t0\t2\t0\t\t\n"
    "0\tmock_chr1:1-10\tRECORD_BP\t2\t0\t2\t0\t\t\n"
    "2147483648\tmock_chr1:1-10\tGT\t2\t0\t1\t0\t0\t0\n"
    "2147483648\tmock_chr1:1-10\tHAP\t2\t0\t1\t0\t\t\n"
    "2147483648\tmock_chr1:1-10\tWEIGHTED_HAP\t2\t0\t2\t0\t\t\n"
    "2147483648\tmock_chr1:1-10\tBASEPAIR\t4\t0\t4\t0\t\t\n"
    "2147483648\tmock_chr1:1-10\tRECORD_BP\t4\t0\t4\t0\t\t\n"
    "4294967301\tmock_chr1:1-10\tGT\t1\t0\t2\t0\t0\t0\n"
    "4294967301\tmock_chr1:1-10\tHAP\t1\t0\t2\t0\t\t\n"
    "4294967301\tmock_chr1:1-10\tWEIGHTED_HAP\t2\t0\t2\t0\t\t\n"
    "4294967301\tmock_chr1:1-10\tBASEPAIR\t4\t0\t4\t0\t\t\n"
    "4294967301\tmock_chr1:1-10\tRECORD_BP\t4\t0\t4\t0\t\t\n")
GOLDEN_GT = (
    "0\tmock_chr1:1-10\tGT\t1\t0\t1\t0\t0\t0\n"
    "2147483648\tmock_chr1:1-10\tGT\t2\t0\t1\t0\t0\t0\n"
    "4294967301\tmock_chr1:1-10\tGT\t1\t0\t2\t0\t0\t0\n"
    "0\tmock_chr1:1-10\tGT\t1\t0\t1\t0\t0\t0\n"
    "2147483648\tmock_chr1:1-10\tGT\t0\t1\t0\t0\t0\t0\n"
    "4294967301\tmock_chr1:1-10\tGT\t2\t1\t1\t1\t0\t1\n"
    "0\tmock_chr1:1-10\tGT\t0\t1\t1\t1\t1\t0\n"
    "2147483648\tmock_chr1:1-10\tGT\t1\t1\t1\t1\t1\t1\n")
GOLDEN_SEQUENCES = (
    b"0\tmock_chr1:1-10\tACCGTTACCA\tACGGTTACCA\tACCGTTACCA\tACGGTTACCA\tACCGTTACCA\n"
    b"2147483648\tmock_chr1:1-10\tACCGTTACCA\tACGTTTACCA\tACCGTTACCA\tACGTTTACCA\tACCGTTACCA\n"
    b"4294967301\tmock_chr1:1-10\tACCGTTACCA\tACCGTTACCA\tACGTTTACCA\tACCGTTACCA\tACGTTTACCA\n"
    b"0\tmock_chr1:1-10\tACCGTTACCA\tACCCGTTACCA\tACCCGTTACCA\tACCCGTTACCA\tACCCGTTACCA\n"
    b"2147483648\tmock_chr1:1-10\tACCGTTACCA\tACGGTTACCA\tACCGTTACCA\tACCGTTACCA\tACCGTTACCA\n"
    b"4294967301\tmock_chr1:1-10\tACCGTTACCA\tACGGTTCCCA\tACCGCTACCA\tACGGTTCCCA\tACGGTTACCA\n"
    b"0\tmock_chr1:1-10\tACCGTTACCA\tACCGCTACCA\tACCGCTACCA\tACCGATACCA\tACCGCTACCA\n"
    b"2147483648\tmock_chr1:1-10\tACCGTTACCA\tACCGGTACCA\tACCGTACCA\tACCGGTACCA\tACCGTACCA\n")


def test_golden_clusters_literal_text():
    batch, out = _golden()
    assert (out.status[:8] == 0).all()
    names = ["mock_chr1"]
    assert region_summary_lines(batch, names, out, ALL, True, 0, 3) == SUMMARY_HEADER + GOLDEN_SUMMARY_3
    assert region_summary_lines(batch, names, out, ALL, False, 0, 3) == GOLDEN_SUMMARY_3
    assert region_summary_lines(batch, names, out, ("GT",)) == SUMMARY_HEADER + GOLDEN_GT
    assert region_summary_lines(batch, names, out, ("GT",), header=False) == GOLDEN_GT
    assert region_summary_lines(batch, names, out, ()) == SUMMARY_HEADER
    assert region_summary_lines(batch, names, out, (), header=False) == ""
    assert region_sequence_lines(batch, names, out) == SEQUENCES_HEADER + GOLDEN_SEQUENCES
    assert region_sequence_lines(batch, names, out, header=False) == GOLDEN_SEQUENCES
    assert region_sequence_lines(batch, names, out, lo=3, hi=3) == SEQUENCES_HEADER
    # the literal text agrees with the reference's own expectations of every case (golden_cases.py)
    for i, (_, _, exp) in enumerate(COMPARE_CASES):
        lines = region_summary_lines(batch, names, out, ALL, False, i, i + 1).split("\n")
        g, h, b = exp["gt"], exp["hap"], exp["basepair"]
        assert lines[0].split("\t")[3:] == [str(x) for x in (g.truth_tp, g.truth_fn, g.query_tp, g.query_fp, g.truth_fn_gt, g.query_fp_gt)]
        assert lines[1].split("\t")[3:7] == [str(x) for x in (h.truth_tp, h.truth_fn, h.query_tp, h.query_fp)]
        assert lines[3].split("\t")[3:7] == [str(x) for x in (b.truth_tp, b.truth_fn, b.query_tp, b.query_fp)]
        seq = region_sequence_lines(batch, names, out, False, i, i + 1)
        assert tuple(s.decode() for s in seq[:-1].split(b"\t")[2:]) == exp["seqs"]


def _hand_made():
    """three regions on two contigs with made-up rows and bundle; region 1 unsolved"""
    batch = RegionBatch(2, [7, 8, (1 << 64) - 1], [0, 1, 1], [100, 0, 4294967294], [250, 1, 4294967295], [0, 0, 0, 0, 0, 0, 0],
                        [], [], [], [], [], [], [], np.zeros(1, np.uint8))
    out = CompareOutputs(batch, seq_off=np.arange(16, dtype=np.uint64) * 3, seq_pool_len=45)
    out.status[:] = [0, abi.ST_BAD_INPUT, 0]
    out.region_metrics[:] = np.arange(out.region_metrics.size, dtype=np.uint64).reshape(out.region_metrics.shape)
    out.seq_len[:] = [0, 1, 2, 3, 0] * 3
    out.seq_pool[:] = np.frombuffer(b"\x00\x01\xff" * 15, dtype=np.uint8)
    return batch, out


def test_hand_made_rows_coordinates_and_raw_bytes():
    batch, out = _hand_made()
    names = ["chr1", "HLA-A*01:01"]
    rm = out.region_metrics
    want = "".join(f"{rid}\t{co}\t{name}\t{' '.join(str(int(x)) for x in rm[r, 0, col:col + 4])}\t{gt}\n".replace(" ", "\t")
                   for r, rid, co in ((0, 7, "chr1:101-250"), (2, (1 << 64) - 1, "HLA-A*01:01:4294967295-4294967295"))
                   for name, col, gt in (("RECORD_BP", abi.M_RECORD_BP, "\t"), ("GT", abi.M_GT, f"{int(rm[r, 0, 4])}\t{int(rm[r, 0, 5])}")))
    assert region_summary_lines(batch, names, out, ("RECORD_BP", "GT"), header=False) == want
    p = out.seq_pool.tobytes()
    seqs = lambda r: b"\t".join(p[3 * (r * 5 + s):3 * (r * 5 + s) + [0, 1, 2, 3, 0][s]] for s in range(5))
    assert region_sequence_lines(batch, names, out, header=False) == (b"7\tchr1:101-250\t" + seqs(0) + b"\n" +
                                                                      b"18446744073709551615\tHLA-A*01:01:4294967295-4294967295\t" + seqs(2) + b"\n")


@pytest.mark.parametrize("bad", ["tab", "quote", "cr", "lf", "null", "short", "metric"])
def test_host_formatters_refuse(bad):
    batch, out = _hand_made()
    lib = _bind()
    names = ["chr1", {"tab": "a\tb", "quote": 'a"b', "cr": "a\rb", "lf": "a\nb"}.get(bad, "chrB")]
    cn = _c_names(names)
    if bad == "null":
        cn[1] = None
    n_contigs = 1 if bad == "short" else 2
    metrics = np.asarray([0, 5 if bad == "metric" else 4], dtype=np.uint8)
    cb, n = batch.to_c(), C.c_uint64(0)
    rc_s = lib.avk_region_summary_write(C.byref(cb), out.status.ctypes.data, out.region_metrics.ctypes.data, cn, n_contigs, metrics.ctypes.data, 2, 1,
                                        0, 3, None, 0, C.byref(n))
    rc_q = lib.avk_region_sequences_write(C.byref(cb), out.status.ctypes.data, out.seq_off.ctypes.data, out.seq_len.ctypes.data, out.seq_pool.ctypes.data,
                                          cn, n_contigs, 1, 0, 3, None, 0, C.byref(n))
    assert rc_s == AVK_ERR_INVALID
    assert rc_q == (0 if bad == "metric" else AVK_ERR_INVALID)
    # a range holding only contig 0 is fine with one name
    if bad == "short":
        assert lib.avk_region_sequences_write(C.byref(cb), out.status.ctypes.data, out.seq_off.ctypes.data, out.seq_len.ctypes.data,
                                              out.seq_pool.ctypes.data, cn, 1, 1, 0, 1, None, 0, C.byref(n)) == 0


def test_seeded_batch_parses_back_to_the_oracle():
    ref, batch = synth.workload_chr20(scale=0.002, seed=31)
    end = batch.end.copy()
    end[::31] = len(ref) + 1                              # windows past the contig's end: bad-input regions are skipped
    batch.end = end
    out = _oracle(batch, [ref])
    n = batch.n_regions
    solved = out.status[:n] == 0
    assert solved.sum() > 100 and (~solved).sum() > 3
    names = ["chr20"]
    rows = parse_summary(region_summary_lines(batch, names, out), 5)
    seqs = parse_sequences(region_sequence_lines(batch, names, out))
    ids = [int(x) for x in batch.region_id[:n][solved]]
    assert list(rows) == ids and list(seqs) == ids
    total = {m: np.zeros(6, dtype=np.uint64) for m in METRICS}
    for r in np.flatnonzero(solved):
        rid = int(batch.region_id[r])
        co = f"chr20:{int(batch.start[r]) + 1}-{int(batch.end[r])}"
        for m, name in enumerate(METRICS):
            assert rows[rid][name] == (co, _joint(out.region_metrics[r], m))
            total[name] += np.asarray([x or 0 for x in rows[rid][name][1]], dtype=np.uint64)
        assert seqs[rid] == (co, tuple(out.sequence(r, s) for s in range(5)))
    for m, name in enumerate(METRICS):                    # summed over solved regions: the joint rows of the oracle's totals
        assert tuple(int(x) for x in total[name]) == tuple(x or 0 for x in _joint(out.totals, m))


# ---- GPU: the device writers -----------------------------------------------------------------------------------------------
def _gpu():
    import test_bgzf as B
    from aardvark_b200.writers import bgzf_compress, region_sequences_bgzf, region_summary_bgzf
    return B, bgzf_compress, region_summary_bgzf, region_sequences_bgzf


@pytest.fixture(scope="module")
def solver():
    from aardvark_b200.lib import Solver
    s = Solver(0)
    yield s
    s.close()


def _files(s, names, metrics=ALL, region_ids=None, header=True, eof=True):
    _, _, summ, seqs = _gpu()
    return summ(s, names, metrics, region_ids, header, eof), seqs(s, names, region_ids, header, eof)


def _check_files(s, files, batch, names, out, metrics=ALL, lo=0, hi=None, header=True):
    """device files == avk_bgzf_compress(host text over `out`); both inflate to that text with a valid member layout"""
    B, bgzf_compress, _, _ = _gpu()
    texts = (region_summary_lines(batch, names, out, metrics, header, lo, hi).encode(), region_sequence_lines(batch, names, out, header, lo, hi))
    for got, text in zip(files, texts):
        assert got == bgzf_compress(s, text)
        B.check_bgzf_layout(got, text)
        assert B.gunzip_members(got) == text
    return texts


def _resident(s, batch, cfg, lo=None, hi=None, region_ids="batch", names=("chr20",), metrics=ALL):
    s.upload(batch, lo, hi)
    s.run_resident(cfg, region_metrics=True, sequences=True)
    return _files(s, list(names), metrics, batch.region_id if region_ids == "batch" else region_ids)


def _dense_batch():
    p = synth.SynthParams(n_variants=1500, dense_frac=0.9, dense_mean=6.0, het_frac=0.95, phased_frac=0.2,
                          p_repr=0.05, p_gt_err=0.08, p_fn=0.08, p_fp=0.08)
    return synth.workload_compare(30_000, p, seed=17)


def _sv_batch():
    p = synth.SynthParams(n_variants=40, sv_events=4, sv_min=6_000, sv_max=10_000, flank=1000)
    return synth.workload_compare(120_000, p, seed=46)


WORKLOADS = {"chr20": lambda: synth.workload_chr20(scale=0.004, seed=40), "dense": _dense_batch, "sv": _sv_batch}
CASES = [("chr20", 50, 0), ("chr20", 4, 0), ("chr20", 50, 1), ("dense", 50, 0), ("dense", 4, 1), ("sv", 50, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("work,bf,shortcut", CASES, ids=[f"{w}-bf{b}-sc{s}" for w, b, s in CASES])
def test_resident_pass_equals_compare_batch_and_oracle(solver, work, bf, shortcut):
    ref, batch = WORKLOADS[work]()
    if work == "sv":
        assert int(np.maximum(batch.a0_len, batch.a1_len).max()) >= 6_000
    cfg = CompareConfig(max_branch_factor=bf, enable_exact_shortcut=bool(shortcut), enable_sequences=True)
    solver.set_reference([ref])
    cpu = _oracle(batch, [ref], cfg)
    off, plen = seq_offsets(batch)
    gpu = solver.compare_batch(batch, cfg, seq_off=off, seq_pool_len=plen)
    assert gpu.diff(cpu) == []
    names = ["chr20"]
    by_batch = _files(solver, names, ALL, batch.region_id)
    _check_files(solver, by_batch, batch, names, cpu)
    resident = _resident(solver, batch, cfg)
    assert resident == by_batch
    rows = solver.download(CompareOutputs(batch))
    assert rows.diff(cpu) == []


@pytest.mark.gpu
def test_chain_on_the_device(solver):
    B, _, _, _ = _gpu()
    from test_gpu_parity import _same_batch, _vcf_text
    from aardvark_b200.batch import BedIntervals, CallSets
    from aardvark_b200.ingest import parse_vcf_bgzf
    from aardvark_b200.writers import vcf_record_lines, vcf_records_bgzf
    names = ["chrA", "chrB"]
    refs, sides = [], [[], []]
    for c, L in enumerate((120_000, 60_000)):
        p = synth.SynthParams(n_variants=L // 120, sv_events=2 if c == 0 else 0, sv_min=60, sv_max=300)
        ref, (truth, query) = synth.callsets_compare(L, p, seed=910 + c)
        refs.append(np.frombuffer(ref, dtype=np.uint8).copy())
        for k, lst in enumerate((truth, query)):
            sides[k] += [(c, pos, a0, a1, z, t, raw) for (pos, a0, a1, z, t, raw) in lst]
    bed = BedIntervals([[(1_000, 50_000), (52_000, 118_000)], [(0, 59_000)]])
    texts = [_vcf_text(recs, names) for recs in sides]
    solver.set_reference(refs)
    parsed = [parse_vcf_bgzf(solver, B.bgzf_compress(t, 6, 0x4000), names, 0, True) for t in texts]
    cs = CallSets([[r[1:] for r in tab.records()] for tab in parsed], contigs=[[r[0] for r in tab.records()] for tab in parsed])
    first = (1 << 31) - 40
    built = solver.build_regions(cs, 0, 50, first_region_id=first, bed=bed)
    cfg = CompareConfig(enable_sequences=True)
    solver.run_resident(cfg, region_metrics=True, sequences=True)
    files = _files(solver, names)
    out = solver.download(CompareOutputs(built))
    truth_gz = vcf_records_bgzf(solver, 0, names, b"", None)
    # the oracle's chain: vcf_parse -> build_regions_bed -> compare_batch, and the host formatters over its results
    ptabs = [orc.vcf_parse(t, names, 0, True) for t in texts]
    assert all(err == 0 for _, err in ptabs)
    ocs = CallSets([[r[1:] for r in tab.records()] for tab, _ in ptabs], contigs=[[r[0] for r in tab.records()] for tab, _ in ptabs])
    obatch = orc.build_regions_bed(ocs, [r.size for r in refs], 50, bed, first)
    _same_batch(built, obatch)
    assert built.n_regions > 40 and int(built.region_id[-1]) >= 1 << 31 and int(built.region_id[0]) < 1 << 31
    cpu = _oracle(obatch, refs, cfg)
    assert out.diff(cpu) == []
    summary, _ = _check_files(solver, files, obatch, names, cpu)
    assert b"chrB:" in summary and str((1 << 31) + 1).encode() in summary
    assert B.gunzip_members(truth_gz) == vcf_record_lines(obatch, 0, names, cpu).encode()


@pytest.mark.gpu
def test_unsolved_regions_are_skipped(solver):
    from test_gpu_parity import _solver_with_env
    # bad-input regions
    ref, batch = synth.workload_chr20(scale=0.003, seed=41)
    end = batch.end.copy()
    end[::50] = len(ref) + 1
    batch.end = end
    solver.set_reference([ref])
    cfg = CompareConfig(enable_sequences=True)
    files = _resident(solver, batch, cfg)
    cpu = _oracle(batch, [ref], cfg)
    assert (cpu.status[:batch.n_regions] == abi.ST_BAD_INPUT).sum() >= batch.n_regions // 50
    _check_files(solver, files, batch, ["chr20"], cpu)
    # AVK_ST_TIMEOUT under a tiny expansion cap: the device's own rows and bundle, solved regions only
    ref, batch = _dense_batch()
    solver.set_reference([ref])
    cfg = CompareConfig(enable_sequences=True, exact_gt_max_expansions=3)
    off, plen = seq_offsets(batch)
    gpu = solver.compare_batch(batch, cfg, seq_off=off, seq_pool_len=plen)
    n = batch.n_regions
    assert (gpu.status[:n] == abi.ST_TIMEOUT).sum() > 0
    by_batch = _files(solver, ["chr1"], ALL, batch.region_id)
    files = _resident(solver, batch, cfg, names=("chr1",))
    assert files == by_batch and solver.download(CompareOutputs(batch)).diff(gpu) == []
    texts = _check_files(solver, files, batch, ["chr1"], gpu)
    assert len(parse_sequences(texts[1])) == int((gpu.status[:n] == 0).sum())
    # forced cooperative tiers: SV clusters through the last-resort tier
    p = synth.SynthParams(n_variants=120, sv_events=30, sv_min=60, sv_max=900, flank=1000)
    ref, batch = synth.workload_compare(250_000, p, seed=45)
    s = _solver_with_env(AVK_TEST_WIDE_B0=32, AVK_TEST_COOP_ARENA_MB=1, AVK_TEST_COOP_ARENA1_MB=256)
    try:
        s.set_reference([ref])
        cfg = CompareConfig(enable_sequences=True)
        files = _resident(s, batch, cfg, names=("chr1",))
        assert s.last_tier_overflow()[2] > 0
        _check_files(s, files, batch, ["chr1"], _oracle(batch, [ref], cfg))
    finally:
        s.close()
    # a last-resort tier as small as the first: the 6-10 kbp SV clusters that overflow it end with AVK_ST_WORKSPACE and have no
    # lines; every other region equals the default tiers' result (which the SV case above pins to the oracle)
    ref, batch = _sv_batch()
    solver.set_reference([ref])
    off, plen = seq_offsets(batch)
    dflt = solver.compare_batch(batch, cfg, seq_off=off, seq_pool_len=plen)
    s = _solver_with_env(AVK_TEST_WIDE_B0=32, AVK_TEST_COOP_ARENA_MB=1, AVK_TEST_COOP_ARENA1_MB=1)
    try:
        s.set_reference([ref])
        gpu = s.compare_batch(batch, cfg, seq_off=off, seq_pool_len=plen)
        n = batch.n_regions
        ws = gpu.status[:n] == abi.ST_WORKSPACE
        assert ws.any() and (~ws).any() and (gpu.status[:n][~ws] == dflt.status[:n][~ws]).all()
        assert (gpu.region_metrics[:n][~ws] == dflt.region_metrics[:n][~ws]).all()
        assert all(gpu.sequence(r, k) == dflt.sequence(r, k) for r in np.flatnonzero(~ws) for k in range(5))
        by_batch = _files(s, ["chr1"], ALL, batch.region_id)
        files = _resident(s, batch, cfg, names=("chr1",))
        assert files == by_batch
        summary, seqs = _check_files(s, files, batch, ["chr1"], gpu)
        want_ids = [int(x) for x in batch.region_id[:n][gpu.status[:n] == 0]]
        assert list(parse_summary(summary.decode(), 5)) == want_ids and list(parse_sequences(seqs)) == want_ids
        assert not {int(x) for x in batch.region_id[:n][ws]} & set(want_ids)
    finally:
        s.close()


def _rand_acgt(rng, n):
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n, dtype=np.uint8)].tobytes()


@pytest.mark.gpu
def test_edges_long_window_empty_batch_all_failing(solver):
    B, bgzf_compress, summ, seqs = _gpu()
    rng = np.random.default_rng(12)
    L = 200_000
    ref = _rand_acgt(rng, L)
    pos, n = 20_000, 70_000                               # a 70 kbp deletion: a window (and each string) past 64 kbp
    truth = [synth.make_rec(pos, ref[pos:pos + n + 1], ref[pos:pos + 1], abi.ZYG_UNPHASED_HET, sv=True)]
    query = [synth.make_rec(pos, ref[pos:pos + n + 1], ref[pos:pos + 1], abi.ZYG_UNPHASED_HET, sv=True),
             synth.make_rec(150_000, ref[150_000:150_001], b"A" if ref[150_000] != ord("A") else b"C", abi.ZYG_HOM_ALT)]
    batch = synth.cluster_regions([truth, query], L, 50)
    assert int((batch.end - batch.start).max()) > 65_536
    solver.set_reference([ref])
    cfg = CompareConfig(enable_sequences=True)
    off, plen = seq_offsets(batch)
    gpu = solver.compare_batch(batch, cfg, seq_off=off, seq_pool_len=plen)    # (the oracle needs minutes for this window)
    files = _resident(solver, batch, cfg, names=("chr1",))
    texts = _check_files(solver, files, batch, ["chr1"], gpu)
    assert (gpu.status[:batch.n_regions] == 0).all() and max(len(x) for x in texts[1].split(b"\n")) > 2 * 0xff00
    r = int(np.argmax(batch.end - batch.start))
    assert gpu.sequence(r, 0) == ref[int(batch.start[r]):int(batch.end[r])]
    assert sorted(gpu.sequence(r, s) for s in (1, 2)) == sorted(gpu.sequence(r, s) for s in (3, 4))
    # an empty batch: the header only, or an empty file
    empty = RegionBatch(2, [], [], [], [], [0], [], [], [], [], [], [], [], np.zeros(1, np.uint8))
    _resident(solver, empty, cfg)
    assert summ(solver, ["chr1"], ALL, empty.region_id) == bgzf_compress(solver, SUMMARY_HEADER.encode())
    assert seqs(solver, ["chr1"], empty.region_id) == bgzf_compress(solver, SEQUENCES_HEADER)
    assert summ(solver, ["chr1"], ALL, empty.region_id, header=False) == B.BGZF_EOF
    assert seqs(solver, ["chr1"], empty.region_id, header=False, eof=False) == b""
    # every region fails (HomRef genotypes)
    ref, batch = synth.workload_chr20(scale=0.002, seed=42)
    batch.zygosity = np.full(batch.n_variants, abi.ZYG_HOM_REF, dtype=np.uint8)
    solver.set_reference([ref])
    files = _resident(solver, batch, cfg)
    cpu = _oracle(batch, [ref], cfg)
    assert (cpu.status[:batch.n_regions] != 0).all()
    assert _check_files(solver, files, batch, ["chr20"], cpu) == (SUMMARY_HEADER.encode(), SEQUENCES_HEADER)


@pytest.mark.gpu
def test_bins_and_multi_solver_concatenate(solver):
    B, _, _, _ = _gpu()
    from aardvark_b200.lib import MultiSolver
    ref, batch = synth.workload_chr20(scale=0.004, seed=43)
    solver.set_reference([ref])
    cfg = CompareConfig(enable_sequences=True)
    names = ["chr20"]
    cpu = _oracle(batch, [ref], cfg)
    n = batch.n_regions
    whole = _check_files(solver, _resident(solver, batch, cfg), batch, names, cpu)
    cuts = [(0, n // 7), (n // 7, n // 7 + 3), (n // 7 + 3, n)]    # three uneven bins
    parts = ([], [])
    for lo, hi in cuts:
        solver.upload(batch, lo, hi)
        solver.run_resident(cfg, region_metrics=True, sequences=True)
        for k, f in enumerate(_files(solver, names, ALL, batch.region_id, header=lo == 0, eof=hi == n)):
            parts[k].append(f)
    for k in range(2):
        gz = b"".join(parts[k])
        assert B.gunzip_members(gz) == whole[k] and gz.endswith(B.BGZF_EOF) and gz.count(B.BGZF_EOF) == 1
    # the contexts of a multi-context call hold one bin each, bundle offsets biased by the bin's first offset
    ms = MultiSolver([0, 0])
    try:
        ms.set_reference([ref])
        off, plen = seq_offsets(batch)
        out = ms.compare_batch(batch, cfg, seq_off=off, seq_pool_len=plen)
        assert out.diff(cpu) == []
        got = ([], [])
        for i, s in enumerate(ms.solvers):
            for k, f in enumerate(_files(s, names, ALL, batch.region_id, header=i == 0, eof=i == len(ms.solvers) - 1)):
                got[k].append(f)
        for k in range(2):
            assert B.gunzip_members(b"".join(got[k])) == whole[k]
    finally:
        ms.close()
    # a lane keeps its own result while the owner runs another batch
    other_ref, other = synth.workload_chr20(scale=0.002, seed=44)
    lane = solver.lane()
    try:
        lane_files = _resident(lane, batch, cfg)
        _resident(solver, other, cfg)
        assert _files(lane, names, ALL, batch.region_id) == lane_files
        _check_files(lane, lane_files, batch, names, cpu)
    finally:
        lane.close()


@pytest.mark.gpu
def test_refusals_leave_the_context_usable(solver):
    from aardvark_b200.batch import MergeOutputs
    from aardvark_b200.types import MergeConfig
    from aardvark_b200.writers import _debug_bgzf_fns
    ref, batch = synth.workload_chr20(scale=0.003, seed=45)
    parts = [batch, synth.workload_chr20(scale=0.003, seed=46)[1]]
    batch = RegionBatch.concat(parts)
    refs = [ref, synth.workload_chr20(scale=0.003, seed=46)[0]]
    names = ["chr20", "chr21"]
    solver.set_reference(refs)
    fs, fq = _debug_bgzf_fns(solver._lib)
    n = C.c_uint64(0)
    metrics = np.arange(5, dtype=np.uint8)

    def raw(which, names_=names, n_contigs=2, ids=batch.region_id, m=metrics, buf=None, cap=0):
        cn = (C.c_char_p * 2)(b"chr20", None) if names_ is None else _c_names(names_)
        if which == "s":
            return fs(solver._ctx, cn, n_contigs, m.ctypes.data, m.size, abi.ptr(ids), 1, 1, buf, cap, C.byref(n))
        return fq(solver._ctx, cn, n_contigs, abi.ptr(ids), 1, 1, buf, cap, C.byref(n))

    cfg = CompareConfig(enable_sequences=True)
    solver.upload(batch)
    assert raw("s") == AVK_ERR_INVALID and raw("q") == AVK_ERR_INVALID        # uploaded, not solved
    with pytest.raises(Exception):                                             # the flag without enable_sequences
        solver.run_resident(CompareConfig(enable_sequences=False), region_metrics=True, sequences=True)
    good = _resident(solver, batch, cfg, names=names)
    cpu = _oracle(batch, refs, cfg)
    _check_files(solver, good, batch, names, cpu)
    for which in ("s", "q"):
        for kw in (dict(names_=["chr20", "chr\t21"]), dict(names_=["chr20", 'chr"21']), dict(names_=["chr20", "chr21\r"]),
                   dict(names_=["chr20", "chr\n21"]), dict(names_=None), dict(n_contigs=1), dict(ids=None)):
            assert raw(which, **kw) == AVK_ERR_INVALID, (which, kw)
            assert _files(solver, names, ALL, batch.region_id) == good
    assert raw("s", m=np.asarray([0, 5], dtype=np.uint8)) == AVK_ERR_INVALID
    assert _files(solver, names, ALL, batch.region_id) == good
    for k, which in enumerate(("s", "q")):                                     # capacity: the exact size comes back
        size = len(good[k])
        buf = C.create_string_buffer(size)
        assert raw(which, buf=buf, cap=size - 1) == AVK_ERR_OOM and n.value == size
        assert raw(which, buf=buf, cap=size) == 0 and buf.raw[:size] == good[k]
    # rows / bundle missing: a plain resident pass, a pass with rows only, a pass with the bundle only
    solver.run_resident(cfg)
    assert raw("s") == AVK_ERR_INVALID and raw("q") == AVK_ERR_INVALID
    solver.run_resident(cfg, region_metrics=True)
    assert raw("q") == AVK_ERR_INVALID and _gpu()[2](solver, names, ALL, batch.region_id) == good[0]
    solver.run_resident(cfg, sequences=True)
    assert raw("s") == AVK_ERR_INVALID and _gpu()[3](solver, names, batch.region_id) == good[1]
    # compare_batch without enable_sequences keeps no bundle, even with the outputs
    off, plen = seq_offsets(batch)
    solver.compare_batch(batch, CompareConfig(enable_sequences=False), seq_off=off, seq_pool_len=plen)
    assert raw("q") == AVK_ERR_INVALID and raw("s") == 0
    # a merge result is not a compare result
    solver.merge_upload(batch)
    solver.merge_run_resident(MergeConfig())
    solver.merge_download(MergeOutputs(batch))
    assert raw("s") == AVK_ERR_INVALID and raw("q") == AVK_ERR_INVALID
    assert "merge" in solver._lib.avk_last_error(solver._ctx).decode()
    assert _resident(solver, batch, cfg, names=names) == good
