"""Stratified compare results on the device against the CPU oracle, bit for bit.

The device containment lookup (k_strat_contain) sorts each (stratum, contig) cell by `first`, keeps a running maximum of
`last` and does one binary search per region; the oracle (orc_containments) tests every interval.  k_reduce sums the
per-region metric rows into strat_totals from a caller-provided membership list or from the containment masks, and with
strata it is also what yields `totals`.  These tests pin both at their edges and through every entry point:

  A  a plain Python brute-force containment agrees with orc.containments (CPU, so the reference itself is pinned)
  B  hand-made regions at the lookup's edges: expected mask per region, device == oracle
  C  stratified sums on a chr20-shaped batch with SV events (every solver stage), lists of up to 100 strata and the
     64-stratum device lookup, with the cooperative tiers forced
  D  compare_batch_range, the multi-context call, the streamed call, lanes and SolverPool give the single call's result
  E  replacing the interval sets, the streamed sibling, a changed reference and every rejected input

References: orc.containments for masks; the oracle's strat_totals (membership lists from masks_to_membership) for sums;
and, independently, strat_totals[s] == the u64 sum of the GPU's own region_metrics rows over the OK regions in stratum s.
"""
import os

import numpy as np
import pytest

import oracle_py as orc
from aardvark_b200 import abi, synth
from aardvark_b200.batch import CompareOutputs, RegionBatch, StratIntervals, masks_to_membership
from aardvark_b200.lib import AvkError, Solver, compare_cfg
from aardvark_b200.types import CompareConfig, CompareRegion, Coordinates, PhasedZygosity as Z, Variant

CFG = CompareConfig(enable_sequences=False)
HOM = Z.HomozygousAlternate


# ------------------------------------------------------------------------------------------------ brute-force reference
def brute_containments(batch: RegionBatch, strata, n_contigs):
    """Stratifications::containments by testing every interval.  strata: per stratum, [(contig, BED start, BED end)].
    var_coordinates(): start = min(first truth pos, first query pos), end = max(end of the LAST truth variant, end of the
    LAST query variant); a stratum contains the region when one interval has first <= start && last >= end - 1."""
    cells = {}
    for s, ivs in enumerate(strata):
        for (c, b, e) in ivs:
            cells.setdefault((s, c), []).append((b, e - 1))
    cells = {k: (np.array([f for f, _ in v], dtype=np.int64), np.array([l for _, l in v], dtype=np.int64)) for k, v in cells.items()}
    vo, pos, l0 = batch.var_off.tolist(), batch.position.tolist(), batch.a0_len.tolist()
    out = np.zeros(batch.n_regions, dtype=np.uint64)
    for r in range(batch.n_regions):
        t0, q0, q1 = vo[2 * r], vo[2 * r + 1], vo[2 * r + 2]
        start, end = None, 0
        for lo, hi in ((t0, q0), (q0, q1)):
            if hi > lo:
                start = pos[lo] if start is None else min(start, pos[lo])
                end = max(end, pos[hi - 1] + l0[hi - 1])
        c = int(batch.contig[r])
        if start is None or start >= end or c >= n_contigs:
            continue
        m = 0
        for s in range(len(strata)):
            f, l = cells.get((s, c), (None, None))
            if f is not None and bool(np.any((f <= start) & (l >= end - 1))):
                m |= 1 << s
        out[r] = m
    return out


# ------------------------------------------------------------------------------------------------ hand-made edge batch
L0, L1, L2 = 120_000, 1_400_000, 20_000
TOP = (1 << 32) - 1                                  # largest BED end a u32 holds


def _edge_cases():
    """(refs, batch, strata (64 lists of (contig, BED start, BED end)), expected mask per region, labels, bad-input rows)."""
    rng = np.random.default_rng(63)
    refs = [synth.random_reference(L, rng, 0) for L in (L0, L1, L2)]
    S = [[] for _ in range(64)]
    cases = []                                       # (label, contig, truth, query, window or None, expected strata)

    def snv(c, p):
        b = int(refs[c][p])          # (positions past the contig only occur in deletions below)
        return Variant(0, abi.VT_SNV, p, bytes([b]), bytes([b"ACGT"[(b"ACGT".index(b) + 1) % 4]]), 1)

    def dele(c, p, n, sv=False):
        a0 = refs[c][p:p + n + 1].tobytes() if p + n < len(refs[c]) else b"A" * (n + 1)
        return Variant(0, abi.VT_SV_DELETION if sv else abi.VT_DELETION, p, a0, a0[:1], len(a0))

    def add(label, c, t, q, expect, window=None):
        cases.append((label, c, t, q, window, set(expect)))

    def probe(label, c, a, z, expect, window=None):
        """a TP region whose var_coordinates() are exactly [a, z] (0-based inclusive)"""
        v = snv(c, a) if a == z else dele(c, a, z - a)
        add(label, c, [v], [v], expect, window)

    # exact boundaries: the interval equals [a, z] of the probe, or is off by one at either end
    B = 1000
    S[1].append((0, B + 100, B + 200)); S[2].append((0, B + 101, B + 200)); S[3].append((0, B + 100, B + 199)); S[4].append((0, B + 99, B + 201))
    probe("exact [a,z]", 0, B + 100, B + 199, {1, 4})
    probe("exact a", 0, B + 100, B + 100, {1, 3, 4})
    probe("exact z", 0, B + 199, B + 199, {1, 2, 4})
    probe("exact [a-1,z+1]", 0, B + 99, B + 200, {4})
    probe("exact a-2", 0, B + 98, B + 150, set())
    probe("exact z+1", 0, B + 150, B + 200, {4})
    # prefix maximum: the search lands on the short interval, the long one before it contains the region ([5]); a union
    # covers it but no single interval does ([6])
    B = 5000
    S[5] += [(0, B, B + 1001), (0, B + 500, B + 511)]
    S[6] += [(0, B, B + 651), (0, B + 620, B + 801)]
    probe("pmax inside long", 0, B + 600, B + 700, {5})
    probe("pmax first of two", 0, B + 520, B + 640, {5, 6})
    probe("pmax second of two", 0, B + 620, B + 790, {5, 6})
    probe("pmax union only", 0, B + 550, B + 790, {5})
    probe("pmax inside short", 0, B + 505, B + 509, {5, 6})
    probe("pmax to the end", 0, B + 600, B + 1000, {5})
    probe("pmax past the end", 0, B + 600, B + 1001, set())
    # adjacent intervals [10,19] [20,29]
    B = 8000
    S[7] += [(0, B + 10, B + 20), (0, B + 20, B + 30)]
    probe("adjacent across", 0, B + 15, B + 25, set())
    probe("adjacent second", 0, B + 20, B + 29, {7})
    probe("adjacent first", 0, B + 10, B + 19, {7})
    probe("adjacent seam", 0, B + 19, B + 20, set())
    # nested, duplicate and unsorted intervals
    B = 10_000
    S[8] += [(0, B + 500, B + 600), (0, B + 100, B + 900), (0, B + 200, B + 300), (0, B + 100, B + 900), (0, B + 50, B + 60)]
    S[9] += [(0, B + 400, B + 500)] * 3
    probe("nested outer", 0, B + 150, B + 850, {8})
    probe("nested before outer", 0, B + 95, B + 150, set())
    probe("nested first", 0, B + 55, B + 59, {8})
    probe("nested straddles first", 0, B + 40, B + 55, set())
    probe("nested after inner", 0, B + 550, B + 890, {8})
    probe("duplicates", 0, B + 400, B + 499, {8, 9})
    probe("duplicates z+1", 0, B + 400, B + 500, {8})
    probe("nested outer exact", 0, B + 100, B + 899, {8})
    probe("nested outer z+1", 0, B + 100, B + 900, set())
    # zero-length BED intervals (start > 0): [s, s) is first = s, last = s - 1 and contains nothing
    B = 13_000
    S[10] += [(0, B + 100, B + 100), (0, B + 200, B + 200)]
    S[11] += [(0, B + 150, B + 150), (0, B + 100, B + 160)]
    probe("zero-length at a", 0, B + 100, B + 100, {11})
    probe("zero-length a-1", 0, B + 99, B + 99, set())
    probe("zero-length after long", 0, B + 150, B + 155, {11})
    probe("zero-length alone", 0, B + 200, B + 200, set())
    probe("zero-length a-1 inside long", 0, B + 149, B + 149, {11})
    # region shapes against [100, 299]
    B = 16_000
    S[16].append((0, B + 100, B + 300))
    add("truth only", 0, [snv(0, B + 150)], [], {16})
    add("query only", 0, [], [dele(0, B + 120, 10)], {16})
    add("query before truth, outside", 0, [snv(0, B + 200)], [snv(0, B + 90)], set())
    add("query before truth, inside", 0, [snv(0, B + 250)], [snv(0, B + 110)], {16})
    # the end comes from the last variant: the deletion reaches B+370, the region is [120, 140]
    add("truth last not furthest", 0, [dele(0, B + 120, 250), snv(0, B + 140)], [snv(0, B + 130)], {16})
    add("query last not furthest", 0, [snv(0, B + 130)], [dele(0, B + 120, 250), snv(0, B + 140)], {16})
    add("bad: unsorted truth", 0, [snv(0, B + 150), snv(0, B + 90), snv(0, B + 250)], [snv(0, B + 160)], {16})
    # multi-kbp SV deletions across several intervals ([17]) or inside one ([18])
    B = 20_000
    S[17] += [(0, B, B + 1000), (0, B + 1000, B + 2000), (0, B + 2000, B + 5000)]
    S[18].append((0, B, B + 5000))
    v = dele(0, B + 100, 3000, sv=True)
    add("SV TP spanning", 0, [v], [v], {18})
    add("SV FN spanning", 0, [dele(0, B + 500, 4000, sv=True)], [], {18})
    probe("SV block SNV", 0, B + 2100, B + 2100, {17, 18})
    # every stratum holds [30000, 31000)
    B = 30_000
    for s in range(64):
        S[s].append((0, B, B + 1000))
    probe("all 64", 0, B + 10, B + 500, range(64))
    probe("all 64 last base", 0, B + 999, B + 999, range(64))
    probe("all 64 z+1", 0, B + 999, B + 1000, set())
    # empty cells: stratum 12 only has intervals on contig 1; contig 2 has none in any stratum; 63 alone on contig 1
    S[12].append((1, 0, 200_000))
    S[63].append((1, 250_000, 250_100))
    probe("contig 0 outside every interval", 0, 50_000, 50_010, set())
    probe("other contig's stratum", 1, 100, 200, {12})
    probe("contig without intervals", 2, 1000, 1100, set())
    probe("stratum 63 only", 1, 250_010, 250_050, {63})
    # coordinates up to BED end 2^32 - 1 (windows past contig 0: AVK_ST_BAD_INPUT, masks still computed)
    S[13].append((0, TOP - 100, TOP))
    probe("bad: top inside", 0, TOP - 50, TOP - 1, {13}, window=(TOP - 60, TOP))
    probe("bad: top exact", 0, TOP - 100, TOP - 1, {13}, window=(TOP - 110, TOP))
    probe("bad: top before", 0, TOP - 101, TOP - 60, set(), window=(TOP - 110, TOP))
    # deep search: 10^5 short intervals (given shuffled) and one long one in a single cell
    D, N = 300_000, 100_000
    deep = [(1, D + 10 * i, D + 10 * i + 5) for i in range(N)] + [(1, 800_000, 802_000)]
    S[15] += [deep[i] for i in rng.permutation(len(deep))]
    probe("deep before", 1, D - 500, D - 400, set())
    probe("deep first", 1, D + 1, D + 4, {15})
    probe("deep second", 1, D + 10, D + 14, {15})
    probe("deep last", 1, D + 10 * (N - 1) + 1, D + 10 * (N - 1) + 4, {15})
    probe("deep between", 1, D + 10 * 12_345 + 5, D + 10 * 12_345 + 7, set())
    probe("deep across a gap", 1, D + 10 * 777 + 3, D + 10 * 777 + 12, set())
    probe("deep after", 1, D + 10 * N + 100, D + 10 * N + 110, set())
    probe("deep inside long", 1, 800_500, 800_600, {15})
    probe("deep long carried", 1, 801_500, 801_600, {15})
    probe("deep long z+1", 1, 801_990, 802_003, set())
    # a window past the end of contig 1
    S[19].append((1, L1 - 100, L1))
    probe("bad: window past contig end", 1, L1 - 10, L1 - 10, {19}, window=(L1 - 60, L1 + 40))

    regions = []
    for i, (label, c, t, q, window, _) in enumerate(cases):
        vs = t + q
        if window is None:
            a = min(v.position for v in vs)
            z = max(v.position + len(v.allele0) for v in vs)
            window = (max(0, a - 50), min((L0, L1, L2)[c], z + 50))
        regions.append(CompareRegion(i, Coordinates(c, *window), t, [HOM] * len(t), q, [HOM] * len(q)))
    batch = RegionBatch.from_compare_regions(regions, {0: 0, 1: 1, 2: 2})
    expect = np.array([sum(1 << s for s in e) for *_, e in cases], dtype=np.uint64)
    labels = [c[0] for c in cases]
    bad = np.array([lab.startswith("bad:") for lab in labels])
    return refs, batch, S, expect, labels, bad


@pytest.fixture(scope="module")
def edge():
    return _edge_cases()


def _masks_equal(got, want, labels):
    bad = [f"{labels[r]}: got {int(got[r]):#x}, want {int(want[r]):#x}" for r in range(len(labels)) if int(got[r]) != int(want[r])]
    assert bad == [], bad


# ---- A: the reference itself (CPU) ----------------------------------------------------------------------------------
def test_brute_force_matches_oracle_on_hand_made_cases(edge):
    refs, batch, S, expect, labels, _ = edge
    _masks_equal(brute_containments(batch, S, 3), expect, labels)
    _masks_equal(orc.containments(batch, StratIntervals(S, 3)), expect, labels)


def test_brute_force_matches_oracle_on_random_cases():
    """Random intervals (nested, overlapping, duplicate, zero-length, adjacent) and random lists (empty sides, unsorted,
    the last variant not the furthest-reaching) on a small coordinate range, so that every relation occurs often."""
    rng = np.random.default_rng(20)
    for trial in range(4):
        n_contigs, n_strata, span = 3, int(rng.integers(3, 10)), 400
        strata = []
        for s in range(n_strata):
            ivs = []
            for _ in range(int(rng.integers(0, 24))):
                c = int(rng.integers(0, n_contigs - (trial % 2)))          # odd trials: the last contig has no intervals
                b = int(rng.integers(1, span))
                e = b + int(rng.choice([0, 1, 2, 5, 20, 80, 200, 300, 400]))
                ivs.append((c, b, e))
                if rng.random() < 0.2:
                    ivs.append(ivs[-1])                                  # duplicate
                if rng.random() < 0.2:
                    ivs.append((c, e, e + int(rng.integers(1, 30))))      # adjacent
            strata.append(ivs)
        pos, l0, var_off, contig = [], [], [0], []
        for _ in range(1000):
            for _side in range(2):
                k = int(rng.choice([0, 0, 1, 1, 2, 3, 4]))
                p = sorted(rng.integers(0, span, size=k).tolist()) if rng.random() < 0.8 else rng.integers(0, span, size=k).tolist()
                pos += p
                l0 += rng.choice([1, 1, 1, 2, 5, 30, 120], size=k).tolist()
                var_off.append(len(pos))
            contig.append(int(rng.integers(0, n_contigs + 1)))           # contig n_contigs: outside the interval table
        nv, n = len(pos), len(contig)
        a0 = np.asarray(l0, dtype=np.uint32)
        pool_off = np.concatenate([[0], np.cumsum(a0.astype(np.int64) + 1)])
        batch = RegionBatch(2, np.arange(n), contig, np.zeros(n), np.full(n, span * 2), var_off, pos, np.zeros(nv), np.full(nv, int(HOM)),
                            a0, pool_off[:-1], a0, np.ones(nv), np.full(int(pool_off[-1]), ord("A"), dtype=np.uint8))
        want = brute_containments(batch, strata, n_contigs)
        got = orc.containments(batch, StratIntervals(strata, n_contigs))
        assert np.array_equal(got, want), trial
        assert int((want != 0).sum()) > 80 and int((want == 0).sum()) > 80, trial


# ---- GPU helpers --------------------------------------------------------------------------------------------------
def _solver_with_env(**env):
    """A context of its own created under test knobs (read once in avk_create)."""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return Solver(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _row_sums(out: CompareOutputs, off, idx, n_strata):
    """strat_totals recomputed from the run's own rows: u64 sum over the OK regions listed in each stratum"""
    n = out.n
    rows = out.region_metrics[:n].reshape(n, -1)
    counts = np.diff(off.astype(np.int64))
    reg = np.repeat(np.arange(n), counts)
    s = idx[:int(off[-1])].astype(np.int64)
    keep = out.status[:n][reg] == abi.ST_OK
    acc = np.zeros((n_strata, rows.shape[1]), dtype=np.uint64)
    np.add.at(acc, s[keep], rows[reg[keep]])
    return acc.reshape((n_strata,) + out.strat_totals.shape[1:])


def _check_row_sums(out, off, idx, n_strata):
    assert np.array_equal(out.strat_totals[:n_strata], _row_sums(out, off, idx, n_strata))


# ---- B: the containment kernel at its edges -----------------------------------------------------------------------
@pytest.mark.gpu
def test_device_containment_edges_vs_oracle(edge):
    refs, batch, S, expect, labels, bad = edge
    strat = StratIntervals(S, 3)
    s = Solver(0)
    try:
        s.set_reference(refs)
        s.set_stratifications(strat)
        gpu = s.compare_batch(batch, CFG, n_strata=64, device_strata=True, containment=True)
        _masks_equal(gpu.containment[:batch.n_regions], expect, labels)
        masks = orc.containments(batch, strat)
        so, si = masks_to_membership(masks)
        cpu = orc.compare_batch(batch, refs, compare_cfg(CFG), strat_off=so, strat_idx=si, n_strata=64)
        assert gpu.diff(cpu) == []
        _check_row_sums(gpu, so, si, 64)
        st = gpu.status[:batch.n_regions]
        assert (st[bad] == abi.ST_BAD_INPUT).all() and (st[~bad] == abi.ST_OK).all()
        assert int((expect[bad] != 0).sum()) >= 4            # their masks are set, their rows stay out of the sums
        # 13 and 19 hold the "all 64" probes (which alone make up 62) plus bad-input regions only
        assert np.array_equal(gpu.strat_totals[13], gpu.strat_totals[62]) and np.array_equal(gpu.strat_totals[19], gpu.strat_totals[62])
        assert int(gpu.strat_totals[63].sum()) > int(gpu.strat_totals[62].sum()) > 0
    finally:
        s.close()


# ---- C / D: stratified sums on a chr20-shaped batch with SV events -------------------------------------------------
LIST_STRATA = (1, 3, 64, 100)


def _random_membership(rng, n, n_strata):
    off, idx = [0], []
    for _ in range(n):
        u = rng.random()
        k = 0 if u < 0.2 else (n_strata if u > 0.95 else int(rng.integers(1, min(n_strata, 6) + 1)))
        idx += rng.choice(n_strata, size=k, replace=False).tolist()
        off.append(len(idx))
    return np.asarray(off, dtype=np.uint64), np.asarray(idx or [0], dtype=np.uint32)


def _random_strata(rng, L, n_strata, n_contigs=1):
    strata = []
    for s in range(n_strata):
        ivs = []
        for _ in range(int(rng.integers(0, 16))):
            b = int(rng.integers(0, L))
            ivs.append((int(rng.integers(0, n_contigs)), b, b + int(np.exp(rng.uniform(np.log(50), np.log(20_000))))))
        strata.append(ivs)
    strata[n_strata - 1] += [(0, L // 2, L // 2 + L // 5), (0, L // 2 + 1000, L // 2 + 3000)]
    return strata


class Workload:
    """chr20 at 1/50 scale plus SV events; the oracle is run ONCE with every membership list the tests use side by side
    (stratum indices offset per list), and each test reads its own block of the oracle's strat_totals."""

    def __init__(self):
        L = int(synth.CHR20_LEN * 0.02)
        p = synth.SynthParams(n_variants=3000, sv_events=25, sv_min=60, sv_max=2500)
        self.ref, self.batch = synth.workload_compare(L, p, seed=57)
        n = self.batch.n_regions
        rng = np.random.default_rng(57)
        self.lists = {ns: _random_membership(rng, n, ns) for ns in LIST_STRATA}
        self.strata = {k: _random_strata(rng, L, k) for k in (2, 5, 64)}
        self.strat = {k: StratIntervals(v, 1) for k, v in self.strata.items()}
        self.masks = {k: orc.containments(self.batch, st) for k, st in self.strat.items()}
        blocks = [self.lists[ns] for ns in LIST_STRATA] + [masks_to_membership(self.masks[k]) for k in (2, 5, 64)]
        sizes = list(LIST_STRATA) + [2, 5, 64]
        base = np.cumsum([0] + sizes)
        off, idx = [0], []
        for r in range(n):
            for (o, ix), b0 in zip(blocks, base):
                idx += (ix[int(o[r]):int(o[r + 1])].astype(np.int64) + b0).tolist()
            off.append(len(idx))
        self.cpu = orc.compare_batch(self.batch, [self.ref], compare_cfg(CFG), strat_off=np.asarray(off, np.uint64),
                                     strat_idx=np.asarray(idx, np.uint32), n_strata=int(base[-1]))
        self._blocks = {("list", ns): (int(b0), ns) for ns, b0 in zip(LIST_STRATA, base)}
        self._blocks.update({("dev", k): (int(b0), k) for k, b0 in zip((2, 5, 64), base[len(LIST_STRATA):])})

    def want_sums(self, kind, ns):
        b0, k = self._blocks[(kind, ns)]
        return self.cpu.strat_totals[b0:b0 + k]

    def check(self, gpu, kind, ns, containment=False):
        """every output array against the oracle; the sums against the oracle's block and against the run's own rows"""
        cpu = self.cpu
        for f in ("status", "ed1", "ed2", "region_metrics", "type_mask", "var_expected", "var_observed", "var_class", "totals",
                  "totals_mask", "solved_blocks", "error_blocks"):
            if getattr(gpu, f) is not None:
                assert np.array_equal(getattr(gpu, f), getattr(cpu, f)), f
        assert np.array_equal(gpu.strat_totals[:ns], self.want_sums(kind, ns))
        off, idx = self.lists[ns] if kind == "list" else masks_to_membership(self.masks[ns])
        _check_row_sums(gpu, off, idx, ns)
        if containment:
            assert np.array_equal(gpu.containment[:self.batch.n_regions], self.masks[ns])

    def kw(self, kind, ns):
        if kind == "list":
            off, idx = self.lists[ns]
            return dict(strat_off=off, strat_idx=idx, n_strata=ns)
        return dict(n_strata=ns, device_strata=True, containment=True)


@pytest.fixture(scope="module")
def wl():
    return Workload()


@pytest.fixture(scope="module")
def solver(wl):
    s = Solver(0)
    s.set_reference([wl.ref])
    s.set_stratifications(wl.strat[64])
    yield s
    s.close()


@pytest.fixture(scope="module")
def single(wl, solver):
    """the single call's results, each checked against the oracle"""
    res = {}
    for kind, ns in (("list", 100), ("dev", 64)):
        res[kind] = solver.compare_batch(wl.batch, CFG, **wl.kw(kind, ns))
        wl.check(res[kind], kind, ns, containment=kind == "dev")
    return res


def _multi_strata(masks):
    return int((np.array([bin(int(m)).count("1") for m in masks]) >= 2).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("ns", LIST_STRATA)
def test_list_sums_random_membership_vs_oracle(wl, solver, ns):
    """0 to all strata per region; the list path has no 64-stratum cap"""
    gpu = solver.compare_batch(wl.batch, CFG, **wl.kw("list", ns))
    wl.check(gpu, "list", ns)
    off = wl.lists[ns][0].astype(np.int64)
    k = np.diff(off)
    assert (k == 0).any() and (k == ns).any() and (ns == 1 or (k >= 2).any())


@pytest.mark.gpu
def test_device_lookup_sums_64_strata_vs_oracle(wl, solver):
    gpu = solver.compare_batch(wl.batch, CFG, **wl.kw("dev", 64))
    wl.check(gpu, "dev", 64, containment=True)
    m = wl.masks[64]
    assert (m >> np.uint64(63) & np.uint64(1)).any(), "no region in stratum 63"
    assert _multi_strata(m) > 10 and (m == 0).any()


@pytest.mark.gpu
def test_totals_with_and_without_strata(wl, solver):
    """with strata, k_reduce over the rows yields `totals`; without, the in-kernel tot_slots fold does"""
    with_strata = solver.compare_batch(wl.batch, CFG, **wl.kw("list", 3))
    plain = solver.compare_batch(wl.batch, CFG, region_metrics=False)
    rows = solver.compare_batch(wl.batch, CFG)
    for f in ("totals", "totals_mask", "solved_blocks", "error_blocks"):
        for g in (with_strata, plain, rows):
            assert np.array_equal(getattr(g, f), getattr(wl.cpu, f)), f
    assert int(plain.solved_blocks[0]) == wl.batch.n_regions


@pytest.mark.gpu
def test_forced_cooperative_tiers_sums_vs_oracle(wl):
    """Clusters with an edit-distance bound >= 32 go to the cooperative tiers, whose first arena is shrunk so that some
    overflow into the last one; k_reduce runs again after them and must count those clusters exactly once."""
    s = _solver_with_env(AVK_TEST_WIDE_B0=32, AVK_TEST_COOP_ARENA_MB=1, AVK_TEST_COOP_ARENA1_MB=256)
    try:
        s.set_reference([wl.ref])
        s.set_stratifications(wl.strat[64])
        for kind, ns in (("list", 100), ("dev", 64), ("list", 1)):
            gpu = s.compare_batch(wl.batch, CFG, **wl.kw(kind, ns))
            assert s.last_tier_overflow()[2] > 0, "no cluster reached the cooperative tiers"
            wl.check(gpu, kind, ns, containment=kind == "dev")
    finally:
        s.close()


# ---- D: every entry point gives the single call's result ----------------------------------------------------------
def _assemble(batch, parts, cuts, kw):
    """per-bin outputs -> one output set for the whole batch: arrays at the bins' offsets, counters added up"""
    out = CompareOutputs(batch, **kw)
    for f in ("totals", "solved_blocks", "error_blocks", "totals_mask"):
        getattr(out, f)[...] = 0
    if out.strat_totals is not None:
        out.strat_totals[...] = 0
    for (lo, hi), p in zip(cuts, parts):
        v0, v1 = int(batch.var_off[2 * lo]), int(batch.var_off[2 * hi])
        for f in ("status", "ed1", "ed2", "region_metrics", "type_mask", "containment"):
            if getattr(out, f) is not None:
                getattr(out, f)[lo:hi] = getattr(p, f)[:hi - lo]
        for f in ("var_expected", "var_observed", "var_class"):
            getattr(out, f)[v0:v1] = getattr(p, f)[:v1 - v0]
        for f in ("totals", "solved_blocks", "error_blocks"):
            getattr(out, f)[...] += getattr(p, f)
        out.totals_mask |= p.totals_mask
        if out.strat_totals is not None:
            out.strat_totals += p.strat_totals
    return out


def _check_entry(single, got):
    for kind in ("list", "dev"):
        assert got[kind].diff(single[kind]) == [], kind


@pytest.mark.gpu
def test_compare_batch_range_five_uneven_bins(wl, solver, single):
    n = wl.batch.n_regions
    cuts = [0, 1, n // 9, n // 2, n - 5, n]
    got = {}
    for kind, ns in (("list", 100), ("dev", 64)):
        out = CompareOutputs(wl.batch, **wl.kw(kind, ns))
        tot, st, solved, errs, mask = np.zeros_like(out.totals), np.zeros_like(out.strat_totals), 0, 0, 0
        for lo, hi in zip(cuts, cuts[1:]):
            solver.compare_batch_range(wl.batch, lo, hi, CFG, out=out)
            tot += out.totals; st += out.strat_totals
            solved += int(out.solved_blocks[0]); errs += int(out.error_blocks[0]); mask |= int(out.totals_mask[0])
        out.totals[...] = tot; out.strat_totals[...] = st
        out.solved_blocks[0] = solved; out.error_blocks[0] = errs; out.totals_mask[0] = mask
        got[kind] = out
    _check_entry(single, got)


@pytest.mark.gpu
def test_multi_context_call(wl, single):
    import torch
    from aardvark_b200.lib import MultiSolver
    nd = torch.cuda.device_count()
    m = MultiSolver(list(range(min(nd, 3))) if nd >= 2 else [0, 0, 0])
    try:
        m.set_reference([wl.ref])
        m.set_stratifications(wl.strat[64])
        _check_entry(single, {kind: m.compare_batch(wl.batch, CFG, **wl.kw(kind, ns)) for kind, ns in (("list", 100), ("dev", 64))})
    finally:
        m.close()


FORCED_COOP = dict(AVK_TEST_WIDE_B0="32", AVK_TEST_COOP_ARENA_MB="1", AVK_TEST_COOP_ARENA1_MB="256")


@pytest.mark.gpu
@pytest.mark.parametrize("env", [dict(AVK_PIPELINE_BINS="7", AVK_PIPELINE_MIN_REGIONS="100"), dict(AVK_LANES="3", AVK_LANE_MIN_REGIONS="100")],
                         ids=["streamed", "lanes"])
def test_single_gpu_bins_with_forced_cooperative_tiers(wl, single, monkeypatch, env):
    """The streamed call and the concurrent lanes cut the batch into bins solved by sibling contexts.  The knobs stay set
    for the context's whole life: the streamed sibling is created at the first streamed call and reads them then."""
    for k, v in {**env, **FORCED_COOP}.items():
        monkeypatch.setenv(k, v)
    s = Solver(0)
    try:
        s.set_reference([wl.ref])
        s.set_stratifications(wl.strat[64])
        got = {}
        for kind, ns in (("list", 100), ("dev", 64)):
            got[kind] = s.compare_batch(wl.batch, CFG, **wl.kw(kind, ns))
            assert s.last_tier_overflow()[2] > 0, "no cluster of the owner's bin reached the cooperative tiers"
        _check_entry(single, got)
    finally:
        s.close()


@pytest.mark.gpu
def test_solver_pool_over_slices(wl, single):
    from aardvark_b200.lib import SolverPool
    n = wl.batch.n_regions
    cuts = [0, n // 7, n // 3, n // 2, n - 3, n]
    bins = list(zip(cuts, cuts[1:]))
    parts = [wl.batch.slice_regions(lo, hi) for lo, hi in bins]
    pool = SolverPool(0, 3)
    try:
        pool.set_reference([wl.ref])
        pool.set_stratifications(wl.strat[64])
        off, idx = wl.lists[100]
        outs = [CompareOutputs(p, strat_off=off[lo:hi + 1] - off[lo], strat_idx=idx[int(off[lo]):int(off[hi])], n_strata=100)
                for p, (lo, hi) in zip(parts, bins)]
        got = {"list": _assemble(wl.batch, pool.compare_batches(parts, CFG, outs=outs), bins, wl.kw("list", 100)),
               "dev": _assemble(wl.batch, pool.compare_batches(parts, CFG, **wl.kw("dev", 64)), bins, wl.kw("dev", 64))}
        _check_entry(single, got)
    finally:
        pool.close()


# ---- E: lifecycle and errors --------------------------------------------------------------------------------------
def _dev_call(s, wl, k):
    gpu = s.compare_batch(wl.batch, CFG, **wl.kw("dev", k))
    wl.check(gpu, "dev", k, containment=True)


@pytest.mark.gpu
def test_replaced_interval_sets_are_followed(wl, solver):
    for k in (2, 64, 5):
        solver.set_stratifications(wl.strat[k])
        _dev_call(solver, wl, k)
    solver.set_stratifications(wl.strat[64])


@pytest.mark.gpu
def test_set_stratifications_after_a_streamed_call(wl, monkeypatch):
    """The streamed call creates a sibling context that reads the owner's tables; replacing the tables afterwards must
    succeed on the owner and be followed by the next streamed call."""
    monkeypatch.setenv("AVK_PIPELINE_BINS", "7")
    monkeypatch.setenv("AVK_PIPELINE_MIN_REGIONS", "100")
    s = Solver(0)
    try:
        s.set_reference([wl.ref])
        s.set_stratifications(wl.strat[2])
        _dev_call(s, wl, 2)
        s.set_stratifications(wl.strat[64])
        _dev_call(s, wl, 64)
        s.set_stratifications(wl.strat[5])
        _dev_call(s, wl, 5)
    finally:
        s.close()


def _refused(call, what):
    with pytest.raises(AvkError, match=r"failed \(-1\): .*" + what):
        call()


@pytest.mark.gpu
def test_changed_reference_refuses_the_lookup_until_strata_are_set(wl):
    s = Solver(0)
    try:
        s.set_reference([wl.ref])
        s.set_stratifications(wl.strat[5])
        _dev_call(s, wl, 5)
        s.set_reference([wl.ref, wl.ref[:5000]])
        _refused(lambda: s.compare_batch(wl.batch, CFG, **wl.kw("dev", 5)), "device containment lookup needs avk_set_stratifications")
        _refused(lambda: s.compare_batch(wl.batch, CFG, containment=True), "device containment lookup")
        gpu = s.compare_batch(wl.batch, CFG, **wl.kw("list", 3))            # the list path does not need the tables
        wl.check(gpu, "list", 3)
        s.set_stratifications(StratIntervals(wl.strata[5], 2))
        _dev_call(s, wl, 5)
    finally:
        s.close()


@pytest.mark.gpu
def test_rejected_inputs_leave_the_context_usable(wl, solver):
    b = wl.batch
    solver.set_stratifications(wl.strat[64])
    _refused(lambda: solver.compare_batch(b, CFG, n_strata=63, device_strata=True), "same number of strata")
    _dev_call(solver, wl, 64)
    _refused(lambda: solver.set_stratifications(StratIntervals([[(0, 0, 100)]] * 65, 1)), "at most 64 strata")
    _dev_call(solver, wl, 64)
    bad = StratIntervals(wl.strata[5], 1)
    bad.off = bad.off.copy()
    k = len(bad.off) - 2                                                     # the last stratum always has intervals
    bad.off[k], bad.off[k + 1] = bad.off[k + 1], bad.off[k]
    assert bad.off[k] > bad.off[k + 1]
    _refused(lambda: solver.set_stratifications(bad), "offsets are not monotone")
    _dev_call(solver, wl, 64)                                                # the previous tables are still in place
    off, idx = wl.lists[3]
    off_bad = off.copy()
    r = int(np.nonzero(np.diff(off.astype(np.int64)) > 0)[0][0])
    off_bad[r + 1] = off_bad[r + 2] + 1
    _refused(lambda: solver.compare_batch(b, CFG, strat_off=off_bad, strat_idx=idx, n_strata=3), "not monotone")
    wl.check(solver.compare_batch(b, CFG, **wl.kw("list", 3)), "list", 3)
    idx_bad = idx.copy()
    idx_bad[len(idx_bad) // 2] = 3
    _refused(lambda: solver.compare_batch(b, CFG, strat_off=off, strat_idx=idx_bad, n_strata=3), "stratum index >= n_strata")
    wl.check(solver.compare_batch(b, CFG, **wl.kw("list", 3)), "list", 3)
    _dev_call(solver, wl, 64)


@pytest.mark.gpu
def test_resident_download_refuses_containment_and_strata(wl, solver):
    """avk_compare_run_resident computes neither containment masks nor stratified sums.  The earlier containment call
    covers a batch at least as large as the resident one, so the mask buffer holds other regions' masks, never too few."""
    n = wl.batch.n_regions
    lo, hi = n // 4, n // 4 + 600
    part = wl.batch.slice_regions(lo, hi)
    _dev_call(solver, wl, 64)
    solver.upload(part)
    solver.run_resident(CFG)
    o = CompareOutputs(part, region_metrics=False, containment=True)
    try:
        solver.download(o)
    except AvkError as e:
        assert "containment" in str(e)
    else:
        pytest.fail(f"download returned containment masks the resident run never computed: {o.containment[:6]} "
                    f"(this slice's masks: {wl.masks[64][lo:lo + 6]})")
    one = CompareOutputs(part, region_metrics=False, strat_off=np.arange(hi - lo + 1, dtype=np.uint64), strat_idx=np.zeros(hi - lo, np.uint32), n_strata=1)
    _refused(lambda: solver.download(one), "stratified sums")
    plain = solver.download(CompareOutputs(part, region_metrics=False))
    for f in ("status", "ed1", "ed2", "type_mask"):
        assert np.array_equal(getattr(plain, f)[:hi - lo], getattr(wl.cpu, f)[lo:hi]), f
    v0, v1 = int(wl.batch.var_off[2 * lo]), int(wl.batch.var_off[2 * hi])
    assert np.array_equal(plain.var_class[:v1 - v0], wl.cpu.var_class[v0:v1])
    assert np.array_equal(plain.totals, wl.cpu.region_metrics[lo:hi].sum(axis=0))
