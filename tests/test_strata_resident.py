"""Stratified resident passes (AVK_CMP_STRATA) and stratified sums without per-region rows, against the CPU oracle.

The solver stages add every solved cluster's metrics to the per-stratum partial tables at the same places where they add
to the totals, so a resident pass returns containment masks and strat_totals with the batch never on the host, and
avk_compare_batch no longer needs the [n][13][22] rows to produce them.  Checked here:

  - resident passes over 2, 5 and 64 strata on the chr20-shaped SV workload of test_strata_parity: masks and sums equal
    the oracle, every other output equals a pass without the flag, the sums equal those of the pass's own rows;
  - avk_compare_batch with strata and no rows (list of 100 strata, 64-stratum lookup);
  - the cooperative tiers forced, uneven resident bins, a lane on its owner's tables;
  - the device-built chain (BGZF VCFs -> parse -> build -> stratified resident pass -> sums -> summary text);
  - refusals, each leaving the context usable, and sums that belong to the pass rather than to the current tables.
"""
import numpy as np
import pytest

import oracle_py as orc
from aardvark_b200 import abi, synth
from aardvark_b200.batch import CompareOutputs, StratIntervals, masks_to_membership
from aardvark_b200.lib import AvkError, Solver, compare_cfg
from aardvark_b200.types import CompareConfig
from test_strata_parity import FORCED_COOP, Workload, _solver_with_env

CFG = CompareConfig(enable_sequences=False)
PER_REGION = ("status", "ed1", "ed2", "region_metrics", "type_mask", "var_expected", "var_observed", "var_class")
COUNTERS = ("totals", "totals_mask", "solved_blocks", "error_blocks")


@pytest.fixture(scope="module")
def wl():
    return Workload()


@pytest.fixture(scope="module")
def solver(wl):
    s = Solver(0)
    s.set_reference([wl.ref])
    yield s
    s.close()


def _refused(call, what):
    with pytest.raises(AvkError, match=r"failed \(-1\): .*" + what):
        call()


def _dev_out(batch, k, rows=False, containment=True):
    return CompareOutputs(batch, region_metrics=rows, n_strata=k, device_strata=True, containment=containment)


def _resident(s, wl, k, rows=False):
    """a stratified resident pass over the whole workload and its download"""
    s.upload(wl.batch)
    s.run_resident(CFG, region_metrics=rows, strata=True)
    return s.download(_dev_out(wl.batch, k, rows))


def _check_no_rows(wl, gpu, kind, ns):
    for f in PER_REGION + COUNTERS:
        if getattr(gpu, f) is not None:
            assert np.array_equal(getattr(gpu, f), getattr(wl.cpu, f)), f
    assert np.array_equal(gpu.strat_totals[:ns], wl.want_sums(kind, ns))
    if gpu.containment is not None:
        assert np.array_equal(gpu.containment[:wl.batch.n_regions], wl.masks[ns])


@pytest.mark.gpu
@pytest.mark.parametrize("k", (2, 5, 64))
def test_resident_pass_vs_oracle_and_plain_pass(wl, solver, k):
    solver.set_stratifications(wl.strat[k])
    gpu = _resident(solver, wl, k, rows=True)
    wl.check(gpu, "dev", k, containment=True)            # every output, masks, sums == oracle; sums == the pass's own rows
    solver.run_resident(CFG, region_metrics=True)
    plain = solver.download(CompareOutputs(wl.batch))
    for f in PER_REGION + COUNTERS:
        assert np.array_equal(getattr(gpu, f), getattr(plain, f)), f
    # without the rows on the device
    solver.run_resident(CFG, strata=True)
    _check_no_rows(wl, solver.download(_dev_out(wl.batch, k)), "dev", k)
    totals, st, solved, errors = solver.resident_sums(k)
    assert np.array_equal(totals, wl.cpu.totals) and np.array_equal(st, wl.want_sums("dev", k))
    assert (solved, errors) == (int(wl.cpu.solved_blocks[0]), int(wl.cpu.error_blocks[0]))


@pytest.mark.gpu
def test_compare_batch_strata_without_rows(wl, solver):
    """the list path (100 strata, no cap) and the 64-stratum lookup with region_metrics=False: no per-region rows at all"""
    solver.set_stratifications(wl.strat[64])
    for kind, ns in (("list", 100), ("dev", 64)):
        gpu = solver.compare_batch(wl.batch, CFG, region_metrics=False, **wl.kw(kind, ns))
        assert gpu.region_metrics is None
        _check_no_rows(wl, gpu, kind, ns)


@pytest.mark.gpu
def test_forced_cooperative_tiers_resident(wl):
    """clusters that reach the cooperative tiers, some of them the last one, are counted exactly once"""
    s = _solver_with_env(**FORCED_COOP)
    try:
        s.set_reference([wl.ref])
        s.set_stratifications(wl.strat[64])
        gpu = _resident(s, wl, 64, rows=True)
        assert s.last_tier_overflow()[2] > 0, "no cluster reached the cooperative tiers"
        wl.check(gpu, "dev", 64, containment=True)
        gpu = s.compare_batch(wl.batch, CFG, region_metrics=False, **wl.kw("list", 100))
        assert s.last_tier_overflow()[2] > 0
        _check_no_rows(wl, gpu, "list", 100)
    finally:
        s.close()


@pytest.mark.gpu
def test_uneven_resident_bins_and_a_lane(wl, solver):
    solver.set_stratifications(wl.strat[64])
    n = wl.batch.n_regions
    cuts = [0, n // 11, n - 7, n]
    tot, st, solved, errors = 0, 0, 0, 0
    masks = np.zeros(n, dtype=np.uint64)
    for lo, hi in zip(cuts, cuts[1:]):
        solver.upload(wl.batch, lo, hi)
        solver.run_resident(CFG, strata=True)
        t, s, a, b = solver.resident_sums(64)
        tot, st, solved, errors = tot + t, st + s, solved + a, errors + b
        out = solver.download(_dev_out(wl.batch, 64))
        masks[lo:hi] = out.containment[lo:hi]
    assert np.array_equal(tot, wl.cpu.totals) and np.array_equal(st, wl.want_sums("dev", 64))
    assert (solved, errors) == (int(wl.cpu.solved_blocks[0]), int(wl.cpu.error_blocks[0]))
    assert np.array_equal(masks, wl.masks[64])
    lane = solver.lane()
    try:
        gpu = _resident(lane, wl, 64)
        _check_no_rows(wl, gpu, "dev", 64)
    finally:
        lane.close()


@pytest.mark.gpu
def test_device_built_chain_summary_text(solver):
    """BGZF VCFs -> avk_vcf_parse_bgzf -> avk_build_regions_bed -> stratified resident pass -> sums -> summary text, with no
    batch on the host; the labelled VCFs of that pass are those of a pass without the flag"""
    import test_bgzf as B
    from test_gpu_parity import _vcf_text
    from aardvark_b200.batch import BedIntervals, CallSets
    from aardvark_b200.ingest import parse_vcf_bgzf
    from aardvark_b200.writers import SummaryWriter, vcf_records_bgzf
    names = ["chrA", "chrB"]
    refs, sides = [], [[], []]
    for c, L in enumerate((120_000, 60_000)):
        p = synth.SynthParams(n_variants=L // 120, sv_events=2 if c == 0 else 0, sv_min=60, sv_max=300)
        ref, (truth, query) = synth.callsets_compare(L, p, seed=930 + c)
        refs.append(np.frombuffer(ref, dtype=np.uint8).copy())
        for k, lst in enumerate((truth, query)):
            sides[k] += [(c, pos, a0, a1, z, t, raw) for (pos, a0, a1, z, t, raw) in lst]
    texts = [_vcf_text(recs, names) for recs in sides]
    bed = BedIntervals([[(1_000, 50_000), (52_000, 118_000)], [(0, 59_000)]])
    strat = StratIntervals([[(0, 0, 40_000), (1, 10_000, 30_000)], [(0, 30_000, 120_000)]], 2)
    s = Solver(0)
    try:
        s.set_reference(refs)
        s.set_stratifications(strat)
        parsed = [parse_vcf_bgzf(s, B.bgzf_compress(t, 6, 0x4000), names, 0, True) for t in texts]
        cs = CallSets([[r[1:] for r in tab.records()] for tab in parsed], contigs=[[r[0] for r in tab.records()] for tab in parsed])
        n, _nv = s.build_regions(cs, 0, 50, bed=bed, download=False)
        s.run_resident(CFG, strata=True)
        totals, st, _, _ = s.resident_sums(2)
        vcfs = [vcf_records_bgzf(s, side, names, b"", None) for side in (0, 1)]
        s.run_resident(CFG)
        assert [vcf_records_bgzf(s, side, names, b"", None) for side in (0, 1)] == vcfs
    finally:
        s.close()
    o_tabs = [orc.vcf_parse(t, names, 0, True)[0] for t in texts]
    o_cs = CallSets([[r[1:] for r in tab.records()] for tab in o_tabs], contigs=[[r[0] for r in tab.records()] for tab in o_tabs])
    host = orc.build_regions_bed(o_cs, [r.size for r in refs], 50, bed)
    assert host.n_regions == n > 40
    masks = orc.containments(host, strat)
    assert (masks == 1).any() and (masks == 2).any()
    so, si = masks_to_membership(masks)
    cpu = orc.compare_batch(host, refs, compare_cfg(CFG), strat_off=so, strat_idx=si, n_strata=2)
    sw = SummaryWriter("chain", strat_labels=["low", "high"])
    assert sw.summary_text(totals, st) == sw.summary_text(cpu.totals, cpu.strat_totals)
    assert np.array_equal(st, cpu.strat_totals) and int(st.sum()) > 0


@pytest.mark.gpu
def test_refusals_leave_the_context_usable(wl):
    s = Solver(0)
    try:
        s.set_reference([wl.ref])
        s.upload(wl.batch)
        _refused(lambda: s.run_resident(CFG, strata=True), "device containment lookup needs avk_set_stratifications")
        s.run_resident(CFG)
        assert np.array_equal(s.resident_sums()[0], wl.cpu.totals)
        s.set_stratifications(wl.strat[5])
        s.set_reference([wl.ref, wl.ref[:5000]])                            # tables built for one contig, reference has two
        s.upload(wl.batch)
        _refused(lambda: s.run_resident(CFG, strata=True), "device containment lookup needs avk_set_stratifications")
        s.set_stratifications(StratIntervals(wl.strata[5], 2))
        s.run_resident(CFG, strata=True)
        assert np.array_equal(s.resident_sums(5)[1], wl.want_sums("dev", 5))
        # downloads the flagged pass cannot serve
        off, idx = wl.lists[3]
        _refused(lambda: s.download(CompareOutputs(wl.batch, region_metrics=False, strat_off=off, strat_idx=idx, n_strata=3)), "stratified sums")
        _refused(lambda: s.resident_sums(4), "stratified sums")
        _refused(lambda: s.download(CompareOutputs(wl.batch, region_metrics=True)), "per-region metric rows")
        _check_no_rows(wl, s.download(_dev_out(wl.batch, 5)), "dev", 5)
        # tables replaced after the pass: the download still gives the pass's masks and sums
        s.set_stratifications(StratIntervals(wl.strata[64], 2))
        _refused(lambda: s.resident_sums(64), "stratified sums")
        _check_no_rows(wl, s.download(_dev_out(wl.batch, 5)), "dev", 5)
        # a later pass without the flag
        s.run_resident(CFG)
        _refused(lambda: s.resident_sums(5), "stratified sums")
        _refused(lambda: s.download(_dev_out(wl.batch, 5, containment=False)), "stratified sums")
        _refused(lambda: s.download(CompareOutputs(wl.batch, region_metrics=False, containment=True)), "containment masks were not computed")
        assert np.array_equal(s.resident_sums()[0], wl.cpu.totals)
        s.run_resident(CFG, strata=True)
        _check_no_rows(wl, s.download(_dev_out(wl.batch, 64)), "dev", 64)
    finally:
        s.close()
