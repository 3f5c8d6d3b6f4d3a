"""truth.vcf.gz / query.vcf.gz written on the device (avk_compare_records_bgzf) against the host path it replaces:
avk_vcf_records_write over the downloaded batch and labels, then avk_bgzf_compress -- byte for byte, both sides.  Every file
is also read back with zlib and its member layout (sizes, CRCs, EOF marker) checked."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import test_bgzf as B
from aardvark_b200 import abi, synth
from aardvark_b200.batch import CompareOutputs, RegionBatch
from aardvark_b200.lib import AvkError, Solver
from aardvark_b200.writers import _records_bgzf_fn, bgzf_compress, vcf_record_lines, vcf_records_bgzf

AVK_ERR_INVALID, AVK_ERR_OOM = -1, -4
HEADER = b"##fileformat=VCFv4.2\n##source=aardvark\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tSAMPLE\n"


@pytest.fixture(scope="module")
def solver():
    s = Solver(0)
    yield s
    s.close()


def _solve(s, batch, lo=None, hi=None, out=None):
    s.upload(batch, lo, hi)
    s.run_resident()
    out = out if out is not None else CompareOutputs(batch, region_metrics=False)
    s.download(out)
    return out


def _check(s, batch, names, out, header=HEADER, region_ids="batch"):
    """both sides of the resident result: device file == host text compressed on the device; the file reads back"""
    files = []
    for side in (0, 1):
        text = header + vcf_record_lines(batch, side, names, out).encode()
        got = vcf_records_bgzf(s, side, names, header, batch.region_id if isinstance(region_ids, str) else region_ids)
        assert got == bgzf_compress(s, text), f"side {side}"
        B.check_bgzf_layout(got, text)
        assert B.gunzip_members(got) == text
        files.append(got)
    return files


def _rand_acgt(rng, n):
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n, dtype=np.uint8)].tobytes()


def _batch_of(contigs):
    """[(reference, [truth records, query records])] -> one multi-contig batch (one contig per entry), refs"""
    parts = [synth.cluster_regions(recs, len(ref), 50) for ref, recs in contigs]
    batch = RegionBatch.concat(parts)
    return batch, [np.frombuffer(ref, dtype=np.uint8).copy() for ref, _ in contigs]


# ---- 1. uploaded batches -----------------------------------------------------------------------------------------------------
def test_chr20_scale_batch(solver):
    ref, batch = synth.workload_chr20(scale=0.03, seed=20)
    solver.set_reference([ref])
    out = _solve(solver, batch)
    truth, query = _check(solver, batch, ["chr20"], out)
    assert len(B.gunzip_members(truth)) > 0x20000 and len(B.gunzip_members(query)) > 0x20000      # several members per side


def test_adversarial_clusters_several_contigs(solver):
    from test_gpu_parity import _random_adversarial_batch
    refs, parts = [], []
    for k in range(3):
        ref, b = _random_adversarial_batch(400, seed=70 + k, maxv=6, maxl0=4, maxins=6)
        refs.append(ref)
        parts.append(b)
    batch = RegionBatch.concat(parts)
    rng = np.random.default_rng(5)
    z = batch.zygosity.copy()                            # every zygosity code, out-of-range ones included (printed as ".")
    for i, code in zip(rng.choice(batch.n_variants, 24, replace=False), [0, 1, 2, 3, 4, 5, 6, 9] * 3):
        z[i] = code
    batch.zygosity = z
    end = batch.end.copy()                               # windows past the contig's end: the region fails on the device
    end[rng.choice(batch.n_regions, 10, replace=False)] = 0xfffffff0
    batch.end = end
    names = ["chr1_KI270706v1_random", "HLA-A*01:01:01:01", "x" * 300]
    solver.set_reference(refs)
    out = _solve(solver, batch)
    assert (out.status[:batch.n_regions] != 0).any() and (out.status[:batch.n_regions] == 0).any()
    assert {1, 2, 3} <= set(out.var_class[:batch.n_variants].tolist())              # TP, FN, FP
    _check(solver, batch, names, out)


# ---- 2. batch built on the device -------------------------------------------------------------------------------------------
def test_device_built_batch_uses_the_device_region_ids(solver):
    from test_gpu_parity import _vcf_text
    from aardvark_b200.batch import BedIntervals, CallSets
    from aardvark_b200.ingest import parse_vcf_bgzf
    names = ["chrA", "chrB"]
    refs, sides = [], [[], []]
    for c, L in enumerate((120_000, 60_000)):
        p = synth.SynthParams(n_variants=L // 120, sv_events=2 if c == 0 else 0, sv_min=60, sv_max=300)
        ref, (truth, query) = synth.callsets_compare(L, p, seed=900 + c)
        refs.append(ref)
        for k, lst in enumerate((truth, query)):
            sides[k] += [(c, pos, a0, a1, z, t, raw) for (pos, a0, a1, z, t, raw) in lst]
    bed = BedIntervals([[(1_000, 50_000), (52_000, 118_000)], [(0, 59_000)]])
    solver.set_reference(refs)
    parsed = [parse_vcf_bgzf(solver, B.bgzf_compress(_vcf_text(recs, names), 6, 0x4000), names, 0, True) for recs in sides]
    cs = CallSets([[r[1:] for r in tab.records()] for tab in parsed], contigs=[[r[0] for r in tab.records()] for tab in parsed])
    first = (1 << 31) - 40                               # ids cross 2^31 inside the batch: RI turns negative
    built = solver.build_regions(cs, 0, 50, first_region_id=first, bed=bed)
    assert built.n_regions > 40 and int(built.region_id[-1]) >= 1 << 31
    solver.run_resident()
    out = CompareOutputs(built, region_metrics=False)
    solver.download(out)
    _check(solver, built, names, out, region_ids=None)
    solver.upload(built)
    solver.run_resident()
    with pytest.raises(AvkError):                        # an uploaded batch's ids are not on the device
        vcf_records_bgzf(solver, 0, names, HEADER, None)
    _check(solver, built, names, out)


# ---- 3. long records ---------------------------------------------------------------------------------------------------------
def test_sv_alleles_and_a_record_longer_than_a_member(solver):
    rng = np.random.default_rng(11)
    L = 400_000
    ref = _rand_acgt(rng, L)
    truth, query = [], []
    for k, pos in enumerate(range(2_000, 300_000, 25_000)):
        n = int(rng.integers(6_000, 10_001))
        if k % 2:                                        # deletion, called in both
            rec = synth.make_rec(pos, ref[pos:pos + n + 1], ref[pos:pos + 1], abi.ZYG_HOM_ALT, sv=True)
            truth.append(rec); query.append(rec)
        else:                                            # insertion, truth only
            truth.append(synth.make_rec(pos, ref[pos:pos + 1], ref[pos:pos + 1] + _rand_acgt(rng, n), abi.ZYG_UNPHASED_HET, sv=True))
        query.append(synth.make_rec(pos + 12_000, ref[pos + 12_000:pos + 12_001], b"T" if ref[pos + 12_000] != ord("T") else b"G", abi.ZYG_PHASED_HET01))
    huge = 0xff00 + 5_000                                # one allele longer than a BGZF member
    truth.append(synth.make_rec(330_000, ref[330_000:330_001], ref[330_000:330_001] + _rand_acgt(rng, huge), abi.ZYG_HOM_ALT, sv=True))
    truth.sort(key=lambda r: r[0]); query.sort(key=lambda r: r[0])
    batch, refs = _batch_of([(ref, [truth, query])])
    assert int(batch.a1_len.max()) > 0xff00 and int(np.sort(np.maximum(batch.a0_len, batch.a1_len))[-8]) >= 6_000
    solver.set_reference(refs)
    out = _solve(solver, batch)
    _check(solver, batch, ["chr1"], out)


# ---- 4. formatting edges ----------------------------------------------------------------------------------------------------
def test_region_ids_positions_and_label_values(solver):
    rng = np.random.default_rng(3)
    L = 100_000_100
    ref = _rand_acgt(rng, L)

    def snv(p):
        return ref[p:p + 1], (b"A" if ref[p] != ord("A") else b"C")
    truth, query = [], []
    cuts = [0] + [10 ** d - 2 for d in range(1, 9)] + [10 ** d - 1 for d in range(1, 9)]   # POS = pos + 1: 1 .. 9 digits
    spread = [5_000_000 * j for j in range(2, 8)]        # far-apart records: enough regions for every id below
    for k, p in enumerate(sorted(set(cuts + spread))):
        a0, a1 = snv(p)
        z = [abi.ZYG_HOM_ALT, abi.ZYG_UNPHASED_HET, abi.ZYG_PHASED_HET01, abi.ZYG_PHASED_HET10][k % 4]
        if k % 3 != 1:
            truth.append(synth.make_rec(p, a0, a1, z))
        if k % 3 != 2:
            query.append(synth.make_rec(p, a0, a1, z if k % 5 else abi.ZYG_HOM_ALT))
    batch, refs = _batch_of([(ref, [truth, query])])
    ids = [(1 << 31) - 2, (1 << 31) - 1, 1 << 31, (1 << 31) + 1, (1 << 32) - 1, 1 << 32, (1 << 32) + 1, (1 << 32) + (1 << 31), 0, 7]
    batch.region_id = np.asarray([ids[i % len(ids)] for i in range(batch.n_regions)], dtype=np.uint64)
    assert batch.n_regions >= len(ids)
    solver.set_reference(refs)
    out = _solve(solver, batch)
    labels = set(out.var_expected[:batch.n_variants].tolist()) | set(out.var_observed[:batch.n_variants].tolist())
    assert {0, 1, 2} <= labels
    text = b"".join(B.gunzip_members(f) for f in _check(solver, batch, ["chr1"], out))
    assert b"\t1\t.\t" in text and b"\t100000000\t.\t" in text and b":-2147483648\n" in text and b":-1\n" in text


def test_empty_side_empty_batch_and_a_long_header(solver):
    rng = np.random.default_rng(4)
    ref = _rand_acgt(rng, 50_000)
    truth = [synth.make_rec(p, ref[p:p + 1], b"A" if ref[p] != ord("A") else b"C", abi.ZYG_UNPHASED_HET) for p in range(1_000, 40_000, 700)]
    batch, refs = _batch_of([(ref, [truth, []])])
    long_header = b"".join(b"##contig=<ID=chr%d,length=%d>\n" % (i, 1000 + i) for i in range(3_000))
    assert len(long_header) > 0xff00
    solver.set_reference(refs)
    out = _solve(solver, batch)
    _, query = _check(solver, batch, ["chr1"], out, header=long_header)
    assert B.gunzip_members(query) == long_header
    empty = RegionBatch(2, [], [], [], [], [0], [], [], [], [], [], [], [], np.zeros(1, np.uint8))
    out = _solve(solver, empty)
    for side in (0, 1):
        assert vcf_records_bgzf(solver, side, ["chr1"], HEADER, empty.region_id) == bgzf_compress(solver, HEADER)
        assert vcf_records_bgzf(solver, side, ["chr1"], b"", empty.region_id) == B.BGZF_EOF
        assert vcf_records_bgzf(solver, side, ["chr1"], b"", empty.region_id, eof=False) == b""


# ---- 5. bins ----------------------------------------------------------------------------------------------------------------
def test_two_bins_concatenate_into_one_file(solver):
    ref, batch = synth.workload_chr20(scale=0.01, seed=21)
    solver.set_reference([ref])
    names = ["chr20"]
    mid = batch.n_regions // 2
    out = CompareOutputs(batch, region_metrics=False)
    files = {0: [], 1: []}
    for lo, hi in ((0, mid), (mid, batch.n_regions)):
        _solve(solver, batch, lo, hi, out)
        for side in (0, 1):
            first, last = lo == 0, hi == batch.n_regions
            got = vcf_records_bgzf(solver, side, names, HEADER if first else b"", batch.region_id, eof=last)
            text = (HEADER if first else b"") + vcf_record_lines(batch, side, names, out, lo, hi).encode()
            want = bgzf_compress(solver, text)
            assert got == (want if last else want[:-28])
            files[side].append(got)
    for side in (0, 1):
        gz = b"".join(files[side])
        assert B.gunzip_members(gz) == HEADER + vcf_record_lines(batch, side, names, out).encode()
        assert gz.endswith(B.BGZF_EOF) and gz.count(B.BGZF_EOF) == 1


# ---- 6. errors --------------------------------------------------------------------------------------------------------------
def test_errors_leave_the_context_usable(solver):
    ref, batch = synth.workload_chr20(scale=0.003, seed=22)
    parts = [batch, synth.workload_chr20(scale=0.003, seed=23)[1]]
    batch = RegionBatch.concat(parts)
    refs = [ref, synth.workload_chr20(scale=0.003, seed=23)[0]]
    names = ["chr20", "chr21"]
    solver.set_reference(refs)
    fn = _records_bgzf_fn(solver._lib)
    cnames = (C.c_char_p * 2)(*[n.encode() for n in names])
    n = C.c_uint64(0)

    def raw(side=0, n_contigs=2, ids=batch.region_id, buf=None, cap=0):
        return fn(solver._ctx, side, cnames, n_contigs, abi.ptr(ids), HEADER, len(HEADER), 1, buf, cap, C.byref(n))

    solver.upload(batch)
    assert raw() == AVK_ERR_INVALID                      # uploaded, not solved: no result
    out = _solve(solver, batch)
    good = _check(solver, batch, names, out)
    assert raw(side=2) == AVK_ERR_INVALID
    assert _check(solver, batch, names, out) == good
    assert raw(n_contigs=1) == AVK_ERR_INVALID           # regions of contig 1 with one name
    assert _check(solver, batch, names, out) == good
    assert raw(ids=None) == AVK_ERR_INVALID              # uploaded batch without its ids
    assert _check(solver, batch, names, out) == good
    size = len(good[0])
    buf = C.create_string_buffer(size)
    assert raw(buf=buf, cap=size - 1) == AVK_ERR_OOM and n.value == size
    assert raw(buf=buf, cap=size) == 0 and n.value == size and buf.raw[:size] == good[0]
    assert _check(solver, batch, names, out) == good


# ---- 7. lanes ---------------------------------------------------------------------------------------------------------------
def test_lane_writes_its_own_result(solver):
    ref, batch = synth.workload_chr20(scale=0.005, seed=24)
    other = synth.workload_chr20(scale=0.005, seed=25)[1]
    solver.set_reference([ref])
    lane = solver.lane()
    try:
        out = _solve(solver, batch)
        _solve(lane, other)                              # a different result resident on the lane
        owner_files = _check(solver, batch, ["chr20"], out)
        _solve(lane, batch)
        for side in (0, 1):
            assert vcf_records_bgzf(lane, side, ["chr20"], HEADER, batch.region_id) == owner_files[side]
    finally:
        lane.close()
