"""The resident merge and its device writers: avk_merge_upload_range / avk_merge_run_resident / avk_merge_download against
avk_merge_batch and the CPU oracle, and passing.vcf.gz, regions.bed.gz, failed_regions.bed.gz and the merge summary written
from the resident result against the host writers they replace (avk_merge_records_write / avk_merge_regions_write /
avk_merge_summary_write, then avk_bgzf_compress) -- byte for byte.  Every file is also read back with zlib and its member
layout checked.  The first test feeds hand-made summary rows through the host formatter and needs no GPU."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_py as orc
from aardvark_b200 import abi, synth
from aardvark_b200.batch import MergeOutputs, RegionBatch
from aardvark_b200.lib import AvkError, merge_cfg
from aardvark_b200.types import MergeConfig
from aardvark_b200.writers import (SUMMARY_ROW, VariantMerger, _merge_bgzf_fns, bgzf_compress, merge_records_bgzf, merge_regions_bgzf,
                                   merge_summary_rows, merge_summary_text)

HERE = os.path.dirname(os.path.abspath(__file__))
AVK_ERR_INVALID, AVK_ERR_OOM = -1, -4
DIFFERENT, NO_CONFLICT, MAJORITY, CONFLICT_SELECT, IDENTICAL = range(5)
HEADER = b"##fileformat=VCFv4.2\n##source=aardvark\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tSAMPLE\n"
CONFIGS = (MergeConfig(majority_voting_enabled=True), MergeConfig(no_conflict_enabled=True), MergeConfig(conflict_selection=2), MergeConfig())
TYPES = ["Snv", "Insertion", "Deletion", "Indel", "SvInsertion", "SvDeletion", "SvDuplication", "SvInversion", "SvBreakend", "TrContraction",
         "TrExpansion", "Unknown"]


def _rows(keys):
    """[(class, [indices], variant type, input, pass, fail)] -> SUMMARY_ROW array"""
    r = np.zeros(len(keys), dtype=SUMMARY_ROW)
    for i, (c, ind, vt, k, p, f) in enumerate(keys):
        r[i] = (sum(1 << j for j in ind), c, vt, k, 0, p, f)
    return r


# ---- 0. the host formatter over hand-made rows (no GPU) -----------------------------------------------------------------------
def test_summary_rows_formatter_matches_the_docs_example():
    gold = open(os.path.join(HERE, "golden", "merge_summary_doc_example.tsv")).read()
    code = {"different": DIFFERENT, "no": NO_CONFLICT, "majority": MAJORITY, "conflict": CONFLICT_SELECT, "identical": IDENTICAL}
    keys = []
    for line in gold.splitlines()[1:]:
        f = line.split("\t")
        parts = f[0].split("_")
        key = (code[parts[0]], [int(x) for x in parts if x.isdigit()], TYPES.index(f[1]), int(f[2]))
        p, q = int(f[4]), int(f[5])
        keys += [key + (p // 3, q // 3), key + (p - p // 3, q - q // 3)]      # every key split over two rows: they add up
    rng = np.random.default_rng(1)
    rows = _rows([keys[i] for i in rng.permutation(len(keys))])             # in no particular order: the formatter sorts
    assert merge_summary_text(rows, 3, ["pb", "ilmn", "ont"]) == gold
    assert merge_summary_text(rows, 3, ["pb", "ilmn", "ont"], header=False) == gold.split("\n", 1)[1]
    assert merge_summary_text(rows[:0], 3, ["pb", "ilmn", "ont"]) == ""
    # index lists compared lexicographically (0_1_3 < 0_2), conflict selection after majority, input 31, csv quoting
    rows = _rows([(MAJORITY, [0, 2], 0, 1, 0, 4), (CONFLICT_SELECT, [31], 2, 31, 9, 0), (MAJORITY, [0, 1, 3], 0, 3, 5, 0),
                  (CONFLICT_SELECT, [31], 2, 31, 1, 0), (IDENTICAL, [], 11, 0, 2, 0), (DIFFERENT, [], 1, 5, 0, 3)])
    labels = [f"l{k}" for k in range(32)]
    labels[31], labels[3] = 'x,"y"', "a\tb"
    assert merge_summary_text(rows, 32, labels, csv=True).splitlines() == [
        "merge_reason,variant_type,vcf_index,vcf_label,pass_variants,fail_variants",
        "different,Insertion,5,l5,0,3", "majority_0_1_3,Snv,3,a\tb,5,0", "majority_0_2,Snv,1,l1,0,4",
        'conflict_select_31,Deletion,31,"x,""y""",10,0', "identical,Unknown,0,l0,2,0"]
    assert merge_summary_text(rows, 32, labels).splitlines()[2] == 'majority_0_1_3\tSnv\t3\t"a\tb"\t5\t0'
    with pytest.raises(AvkError):
        merge_summary_text(rows, 31, labels[:31])                           # input 31 of 31 inputs


# ---- GPU -----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def solver():
    from aardvark_b200.lib import Solver
    s = Solver(0)
    yield s
    s.close()


def _resident(s, batch, cfg, bins=None):
    """merge_upload -> merge_run_resident -> merge_download, over the whole batch or the given bins"""
    out = MergeOutputs(batch)
    for lo, hi in bins or [(0, batch.n_regions)]:
        s.merge_upload(batch, lo, hi)
        s.merge_run_resident(cfg)
        s.merge_download(out)
    return out


def _host_files(s, batch, out, names, labels, header=HEADER, lo=0, hi=None, eof=True):
    """what the host path writes: the three texts over [lo, hi), compressed on the device"""
    vm = VariantMerger(batch, out, names, [l if isinstance(l, str) else l.decode() for l in labels])
    texts = [header + vm.passing_records(lo, hi).encode(), vm.regions_bed(True, lo, hi).encode(), vm.regions_bed(False, lo, hi).encode()]
    files = [bgzf_compress(s, t) for t in texts]
    return texts, [f if eof else f[:-28] for f in files]


def _device_files(s, names, labels, header=HEADER, region_ids=None, eof=True):
    return [merge_records_bgzf(s, names, labels, header, region_ids, eof), merge_regions_bgzf(s, names, True, region_ids, eof),
            merge_regions_bgzf(s, names, False, region_ids, eof)]


def _check(s, batch, out, names, labels, header=HEADER, region_ids="batch"):
    """the resident (whole-batch) result: device files == host texts compressed; they read back; the summary in both forms"""
    import test_bgzf as B
    rid = batch.region_id if isinstance(region_ids, str) else region_ids
    texts, want = _host_files(s, batch, out, names, labels, header)
    got = _device_files(s, names, labels, header, rid)
    for g, w, t in zip(got, want, texts):
        assert g == w
        B.check_bgzf_layout(g, t)
        assert B.gunzip_members(g) == t
    rows = merge_summary_rows(s)
    vm = VariantMerger(batch, out, names, [l if isinstance(l, str) else l.decode() for l in labels])
    for csv in (False, True):
        assert merge_summary_text(rows, batch.n_inputs, labels, csv) == vm.summary_text(csv)
    return got, texts


# ---- 1. resident == batch call == oracle ----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_resident_bins_and_batch_call_equal_the_oracle(solver):
    ref, batch = synth.workload_merge(150_000, 400, n_sets=5, seed=38)
    solver.set_reference([ref])
    names, labels = ["chr1"], ["pb", "ilmn", "ont", "hifi", "ul"]
    n = batch.n_regions
    bins = [(0, n // 7), (n // 7, n // 7 + n // 2), (n // 7 + n // 2, n)]
    seen = set()
    for cfg in CONFIGS:
        a = solver.merge_batch(batch, cfg)
        _check(solver, batch, a, names, labels)                           # avk_merge_batch leaves its result resident
        b = _resident(solver, batch, cfg)
        _check(solver, batch, b, names, labels)
        c = _resident(solver, batch, cfg, bins)
        cpu = orc.merge_batch(batch, [ref], merge_cfg(cfg))
        assert a.diff(b) == [] and a.diff(c) == [] and a.diff(cpu) == [], cfg
        seen |= set(a.classification[a.status == 0].tolist())
    assert seen == {DIFFERENT, NO_CONFLICT, MAJORITY, CONFLICT_SELECT, IDENTICAL}


# ---- 2. the whole merge chain on the device -------------------------------------------------------------------------------
@pytest.mark.gpu
def test_merge_chain_on_the_device(solver):
    import test_bgzf as B
    from test_gpu_parity import _same_batch, _vcf_text
    from aardvark_b200.batch import BedIntervals, CallSets
    from aardvark_b200.ingest import parse_vcf_bgzf
    names, K = ["chrA", "chrB"], 4
    refs, sets, flank = [], [[] for _ in range(K)], 0
    for c, L in enumerate((150_000, 90_000)):
        ref, cs, flank = synth.callsets_merge(L, L // 400, n_sets=K, seed=300 + c)
        refs.append(np.frombuffer(ref, dtype=np.uint8).copy())
        for k in range(K):
            sets[k] += [(c, pos, a0, a1, z, t, raw) for (pos, a0, a1, z, t, raw) in cs[k]]
    bed = BedIntervals([[(500, 70_000), (72_000, 149_000)], [(0, 89_000)]])
    texts = [_vcf_text(recs, names) for recs in sets]
    solver.set_reference(refs)
    parsed = [parse_vcf_bgzf(solver, B.bgzf_compress(t, 6, 0x4000), names, 0, True) for t in texts]
    cs = CallSets([[r[1:] for r in tab.records()] for tab in parsed], contigs=[[r[0] for r in tab.records()] for tab in parsed])
    first = (1 << 31) - 60                                                # ids cross 2^31: RI turns negative, BED names stay u64
    built = solver.build_regions(cs, 0, flank, first_region_id=first, bed=bed)
    cfg = MergeConfig(majority_voting_enabled=True)
    solver.merge_run_resident(cfg)
    out = solver.merge_download(MergeOutputs(built))
    # the oracle's chain: vcf_parse -> build_regions_bed -> merge_batch, and the host writers over its results
    ptabs = [orc.vcf_parse(t, names, 0, True) for t in texts]
    assert all(err == 0 for _, err in ptabs)
    ocs = CallSets([[r[1:] for r in tab.records()] for tab, _ in ptabs], contigs=[[r[0] for r in tab.records()] for tab, _ in ptabs])
    obatch = orc.build_regions_bed(ocs, [r.size for r in refs], flank, bed, first)
    _same_batch(built, obatch)
    assert built.n_regions > 60 and int(built.region_id[-1]) >= 1 << 31
    cpu = orc.merge_batch(obatch, refs, merge_cfg(cfg))
    assert out.diff(cpu) == []
    labels = ["pb", "ilmn", "ont", "hifi"]
    got, host_texts = _check(solver, obatch, cpu, names, labels, region_ids=None)
    assert b":-" in host_texts[0] and str((1 << 31) + 5).encode() in host_texts[1] + host_texts[2]
    # an uploaded batch's ids are not on the device: NULL ids are refused, the ids give the same files
    solver.merge_upload(built)
    solver.merge_run_resident(cfg)
    with pytest.raises(AvkError):
        merge_records_bgzf(solver, names, labels, HEADER, None)
    with pytest.raises(AvkError):
        merge_regions_bgzf(solver, names, True, None)
    assert _device_files(solver, names, labels, HEADER, built.region_id) == got


# ---- 3. edges -------------------------------------------------------------------------------------------------------------
def _rand_acgt(rng, n):
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n, dtype=np.uint8)].tobytes()


@pytest.mark.gpu
def test_unsolved_regions_empty_source_and_long_records(solver):
    rng = np.random.default_rng(17)
    L = 300_000
    ref = _rand_acgt(rng, L)
    other = lambda p: b"A" if ref[p] != ord("A") else b"C"
    sets = [[], [], []]
    for j, p in enumerate(range(1_000, 200_000, 1_500)):
        rec = synth.make_rec(p, ref[p:p + 1], other(p), abi.ZYG_HOM_ALT)
        if j % 4 == 0:                                    # inputs 0 and 1 disagree, input 2 holds nothing: conflict selection of 2 passes empty
            sets[0].append(rec)
            sets[1].append(synth.make_rec(p, ref[p:p + 1], b"T" if other(p) != b"T" else b"G", abi.ZYG_HOM_ALT))
        else:
            for k in range(3):
                if j % 4 != 3 or k != 1:
                    sets[k].append(rec)
    huge = 0xff00 + 4_000                                 # an SV insertion longer than a BGZF member, in every input
    sv = synth.make_rec(250_000, ref[250_000:250_001], ref[250_000:250_001] + _rand_acgt(rng, huge), abi.ZYG_HOM_ALT, sv=True)
    for k in range(3):
        sets[k].append(sv)
    batch = synth.cluster_regions(sets, L, 50)
    end = batch.end.copy()                                # windows past the contig's end: status != 0, in no output
    end[rng.choice(batch.n_regions - 1, 6, replace=False)] = 0xfffffff0   # (not the last region: it holds the long SV)
    batch.end = end
    solver.set_reference([ref])
    names, labels = ["chr_" + "z" * 200], ["a", "b", "c"]
    long_header = b"".join(b"##contig=<ID=c%d,length=%d>\n" % (i, 1000 + i) for i in range(3_000))
    assert len(long_header) > 0xff00
    for cfg in (MergeConfig(conflict_selection=2), MergeConfig(majority_voting_enabled=True)):
        out = _resident(solver, batch, cfg)
        assert out.diff(orc.merge_batch(batch, [ref], merge_cfg(cfg))) == []
        assert (out.status != 0).sum() >= 6 and (out.status == 0).any()
        _check(solver, batch, out, names, labels)
        _check(solver, batch, out, names, labels, header=long_header)
    out = _resident(solver, batch, MergeConfig(conflict_selection=2))
    empty2 = np.asarray(batch.var_off[2:-1:3] == batch.var_off[3::3])    # input 2 of each region has no records
    assert ((out.classification == CONFLICT_SELECT) & (out.status == 0) & empty2).any()
    text = _check(solver, batch, out, names, labels)[1][0]
    assert max(len(l) for l in text.split(b"\n")) > 0xff00


@pytest.mark.gpu
def test_32_inputs_with_long_labels(solver):
    ref, batch = synth.workload_merge(60_000, 120, n_sets=32, seed=5)
    solver.set_reference([ref])
    labels = [f'in{k},"q"'.ljust(300, "x") for k in range(32)]
    assert all(len(l) == 300 for l in labels)
    longest = 0
    for cfg in (MergeConfig(majority_voting_enabled=True), MergeConfig(conflict_selection=31), MergeConfig(no_conflict_enabled=True)):
        out = _resident(solver, batch, cfg)
        assert out.diff(orc.merge_batch(batch, [ref], merge_cfg(cfg))) == []
        got, texts = _check(solver, batch, out, ["chr1"], labels)
        longest = max([longest] + [len(l) for l in texts[0].split(b"\n")])
        if cfg.conflict_selection == 31:
            rows = merge_summary_rows(solver)
            assert ((rows["input"] == 31) & (rows["pass_variants"] > 0)).any()
    assert longest > 17 * 300                                             # a majority lists at least 17 of the long labels


@pytest.mark.gpu
def test_empty_batch(solver):
    import test_bgzf as B
    solver.set_reference([b"ACGT" * 100])
    empty = RegionBatch(3, [], [], [], [], [0], [], [], [], [], [], [], [], np.zeros(1, np.uint8))
    _resident(solver, empty, MergeConfig())
    assert merge_records_bgzf(solver, ["c"], ["a", "b", "c"], HEADER, empty.region_id) == bgzf_compress(solver, HEADER)
    assert merge_records_bgzf(solver, ["c"], ["a", "b", "c"], b"", empty.region_id) == B.BGZF_EOF
    assert merge_records_bgzf(solver, ["c"], ["a", "b", "c"], b"", empty.region_id, eof=False) == b""
    for passing in (True, False):
        assert merge_regions_bgzf(solver, ["c"], passing, empty.region_id) == B.BGZF_EOF
    assert merge_summary_rows(solver).size == 0


# ---- 4. bins and GPUs -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_two_bins_and_two_contexts_concatenate(solver):
    import test_bgzf as B
    from aardvark_b200.lib import MultiSolver
    ref, batch = synth.workload_merge(200_000, 600, n_sets=5, seed=9)
    solver.set_reference([ref])
    names, labels = ["chr20"], ["a", "b", "c", "d", "e"]
    cfg = MergeConfig(majority_voting_enabled=True)
    whole = solver.merge_batch(batch, cfg)
    want, _ = _check(solver, batch, whole, names, labels)
    vm = VariantMerger(batch, whole, names, labels)

    def bin_files(s, lo, hi):
        first, last = lo == 0, hi == batch.n_regions
        got = _device_files(s, names, labels, HEADER if first else b"", batch.region_id, eof=last)
        host = _host_files(s, batch, whole, names, labels, HEADER if first else b"", lo, hi, eof=last)[1]
        assert got == host
        return got, merge_summary_rows(s)

    mid = batch.n_regions // 3
    parts = []
    for lo, hi in ((0, mid), (mid, batch.n_regions)):
        solver.merge_upload(batch, lo, hi)
        solver.merge_run_resident(cfg)
        parts.append(bin_files(solver, lo, hi))
    m = MultiSolver([0, 0])
    try:
        m.set_reference([ref])
        assert m.merge_batch(batch, cfg).diff(whole) == []
        from aardvark_b200.lib import partition_regions
        cuts = partition_regions(batch, 2)
        ctx_parts = [bin_files(s, lo, hi) for s, (lo, hi) in zip(m.solvers, cuts)]
    finally:
        m.close()
    for ps in (parts, ctx_parts):                        # (each bin's members are its own, so the bytes differ from the whole file's)
        for f in range(3):
            gz = b"".join(p[0][f] for p in ps)
            assert B.gunzip_members(gz) == B.gunzip_members(want[f])
            assert gz.endswith(B.BGZF_EOF) and gz.count(B.BGZF_EOF) == 1
        rows = np.concatenate([p[1] for p in ps])
        for csv in (False, True):
            assert merge_summary_text(rows, 5, labels, csv) == vm.summary_text(csv)


# ---- 6. state and errors --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals_leave_the_context_usable(solver):
    from aardvark_b200.batch import CompareOutputs
    ref, batch = synth.workload_merge(120_000, 300, n_sets=3, seed=21)
    ref2, b2 = synth.workload_merge(80_000, 200, n_sets=3, seed=22)
    batch = RegionBatch.concat([batch, b2])
    refs, names, labels = [ref, ref2], ["c1", "c2"], ["a", "b", "c"]
    solver.set_reference(refs)
    fr, fg, fs = _merge_bgzf_fns(solver._lib)
    cn = (C.c_char_p * 2)(*[x.encode() for x in names])
    cl = (C.c_char_p * 3)(*[x.encode() for x in labels])
    n = C.c_uint64(0)

    def rec(n_contigs=2, lab=cl, buf=None, cap=0):
        return fr(solver._ctx, cn, n_contigs, lab, abi.ptr(batch.region_id), HEADER, len(HEADER), 1, buf, cap, C.byref(n))

    def bed(n_contigs=2):
        return fg(solver._ctx, cn, n_contigs, 1, abi.ptr(batch.region_id), 1, None, 0, C.byref(n))

    def refused():
        assert rec() == AVK_ERR_INVALID and bed() == AVK_ERR_INVALID and fs(solver._ctx, None, 0, C.byref(n)) == AVK_ERR_INVALID
        assert solver._lib.avk_last_error(solver._ctx)
        with pytest.raises(AvkError):
            solver.merge_download(MergeOutputs(batch))

    solver.merge_upload(batch)
    refused()                                             # uploaded, not solved
    cfg = MergeConfig(majority_voting_enabled=True)
    solver.merge_run_resident(cfg)
    out = solver.merge_download(MergeOutputs(batch))
    good, _ = _check(solver, batch, out, names, labels)
    # a compare result is refused after a merge run
    with pytest.raises(AvkError):
        solver.download(CompareOutputs(RegionBatch(2, [], [], [], [], [0], [], [], [], [], [], [], [], np.zeros(1, np.uint8))))
    from aardvark_b200.writers import vcf_records_bgzf
    with pytest.raises(AvkError):
        vcf_records_bgzf(solver, 0, names, HEADER, batch.region_id)
    assert rec(n_contigs=1) == AVK_ERR_INVALID            # regions of contig 1 with one name
    assert _check(solver, batch, out, names, labels)[0] == good
    null_label = (C.c_char_p * 3)(b"a", None, b"c")
    assert rec(lab=null_label) == AVK_ERR_INVALID
    assert bed(n_contigs=1) == AVK_ERR_INVALID
    assert _check(solver, batch, out, names, labels)[0] == good
    size = len(good[0])
    buf = C.create_string_buffer(size)
    assert rec(buf=buf, cap=size - 1) == AVK_ERR_OOM and n.value == size
    assert rec(buf=buf, cap=size) == 0 and n.value == size and buf.raw[:size] == good[0]
    n_rows = C.c_uint64(0)
    assert fs(solver._ctx, None, 0, C.byref(n_rows)) == 0 and n_rows.value > 1
    rows = np.zeros(n_rows.value, dtype=SUMMARY_ROW)
    assert fs(solver._ctx, rows.ctypes.data, n_rows.value - 1, C.byref(n)) == AVK_ERR_OOM and n.value == n_rows.value
    assert _check(solver, batch, out, names, labels)[0] == good
    # a compare run drops the merge result; a merge run drops the compare result
    cref, cb = synth.workload_chr20(scale=0.002, seed=1)
    solver.set_reference([cref])
    solver.upload(cb)
    solver.run_resident()
    refused()
    solver.merge_upload(cb)
    solver.merge_run_resident(cfg)
    with pytest.raises(AvkError):
        solver.download(CompareOutputs(cb, region_metrics=False))
    with pytest.raises(AvkError):
        vcf_records_bgzf(solver, 0, ["chr20"], HEADER, cb.region_id)
    solver.set_reference(refs)                            # a new reference drops it too
    refused()
    solver.merge_upload(batch)
    solver.merge_run_resident(cfg)
    assert _check(solver, batch, out, names, labels)[0] == good


# ---- 7. lanes -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_lane_keeps_its_own_merge_result(solver):
    ref, batch = synth.workload_merge(150_000, 400, n_sets=4, seed=31)
    other = synth.workload_merge(150_000, 400, n_sets=4, seed=32)[1]
    solver.set_reference([ref])
    labels = ["a", "b", "c", "d"]
    cfg = MergeConfig(majority_voting_enabled=True)
    lane = solver.lane()
    try:
        out = _resident(solver, batch, cfg)
        _resident(lane, other, cfg)                       # a different result resident on the lane
        owner_files, _ = _check(solver, batch, out, ["chr1"], labels)
        _resident(lane, batch, cfg)
        assert _device_files(lane, ["chr1"], labels, HEADER, batch.region_id) == owner_files
        assert _device_files(solver, ["chr1"], labels, HEADER, batch.region_id) == owner_files
    finally:
        lane.close()
