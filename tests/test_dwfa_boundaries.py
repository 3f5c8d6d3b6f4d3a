"""The edit-distance kernels at their routing and capacity boundaries, bit-exact against the CPU oracle.

The DWFA (incremental wavefront edit-distance alignment) has five implementations: the warp path (32-bit offsets), the
CTA-wide byte-staged path (16-bit wavefront in shared memory), the opt-in CTA-wide 2-bit packed path, the CTA-wide 32-bit
path, and the spill (a CTA-wide wavefront that outgrows shared memory is finished on the warp path).  Which one runs depends
on the lengths, the edit distance the alignment resumes at and the capacities.  The cases here sit on either side of each
of those boundaries: the k_wfa_split thresholds (512, 60000, 8 * cap_ints), the 16-bit bound 2 * (64000 - lb) and the
shared-memory bound of the staged and packed capacities, 64 kbp haplotypes in the compare path, and alignments that spill
and resume.  test_route_coverage restates the routing rules in Python and checks on the CPU that every route is aimed at."""
import functools
import os

import numpy as np
import pytest

import oracle_py as orc
from aardvark_b200 import abi, synth
from aardvark_b200.lib import Solver, compare_cfg
from aardvark_b200.types import CompareConfig

# ---- the routing rules, restated ---------------------------------------------------------------------------------------
COOP_CAP_INTS = 26000     # avk_lib.cu, avk_ctx::coop_cap_ints (default; AVK_TEST_COOP_CAP_INTS overrides it in avk_create)
COOP_MIN_ED = 48          # avk_device.cuh, enum COOP_*: dwfa_run hands a wavefront to the CTA from this edit distance on
WIDE_B0 = 256             # avk_lib.cu, avk_ctx::wide_b0: clusters with this edit-distance bound go to the cooperative tier
SHRUNK_CAP_INTS = 3000    # the shrunk wavefront of the AVK_TEST_COOP_CAP_INTS cases


def cta_route(la, lb, cap_ints):
    """avk_lib.cu k_wfa_split (long_min = 512, max_sum = 8 * cap_ints as avk_wfa_ed_batch launches it)."""
    return min(la, lb) >= 512 and la + lb + 4096 <= 8 * cap_ints and max(la, lb) < 60000


def staged_cap16(la, lb, cap_ints):
    """avk_device.cuh coop_staged_cap16."""
    seq = ((la + 8 + 3) & ~3) + ((lb + 8 + 3) & ~3)
    cap = (8 * cap_ints - seq) // 4 if 8 * cap_ints >= seq else -((seq - 8 * cap_ints) // 4)   # C division truncates
    return max(min(cap, 2 * (64000 - lb)), 0)


def staged_e_cap(la, lb, cap_ints):
    """avk_device.cuh coop_dwfa_body_staged_t: cap = (cap16 - 4) & ~1, e_cap = (cap - 3) / 2."""
    return (((staged_cap16(la, lb, cap_ints) - 4) & ~1) - 3) // 2


def packed_cap16(la, lb, cap_ints):
    """avk_device.cuh coop_packed_cap16."""
    num = 8 * cap_ints - 4 * (((la + 15) >> 4) + ((lb + 15) >> 4) + 4) - 64
    cap = (num // 4 if num >= 0 else -((-num) // 4)) - 16
    cap = min(cap, 2 * (64000 - lb)) & ~7
    return max(cap, 0)


def packed_e_cap(la, lb, cap_ints):
    return (packed_cap16(la, lb, cap_ints) - 3) // 2       # avk_device.cuh coop_dwfa_body_packed


def plain_acgt(s):
    return all(c in b"ACGT" for c in set(s))


def coop_path(la, lb, ed, cap_ints, packed, acgt):
    """avk_device.cuh coop_dwfa_body: the path an alignment resumed at edit distance `ed` takes."""
    if packed and 0 < la < 64000 and 0 < lb < 64000 and acgt and packed_cap16(la, lb, cap_ints) >= 2 * ed + 256:
        return "packed"
    if la < 64000 and lb < 64000 and staged_cap16(la, lb, cap_ints) >= 2 * ed + 256:
        return "staged"
    return "32bit"


def binding_bound(path, la, lb, cap_ints):
    """Which bound sets a 16-bit capacity: '16bit' when 2 * (64000 - lb) is the smaller one, else 'smem'."""
    if path == "staged":
        room = (8 * cap_ints - ((la + 8 + 3) & ~3) - ((lb + 8 + 3) & ~3)) // 4
    else:
        room = (8 * cap_ints - 4 * (((la + 15) >> 4) + ((lb + 15) >> 4) + 4) - 64) // 4 - 16
    return "16bit" if 2 * (64000 - lb) <= room else "smem"


def path_e_cap(path, la, lb, cap_ints):
    if path == "packed":
        return packed_e_cap(la, lb, cap_ints)
    if path == "staged":
        return staged_e_cap(la, lb, cap_ints)
    return (cap_ints - 3) // 2                              # avk_device.cuh coop_dwfa_body, the 32-bit tail


def wfa_routes(a, b, ed, cap_ints, packed):
    """Routes one avk_wfa_ed_batch pair takes: k_wfa_ed_cta starts every alignment at ED 0 and spills past e_cap."""
    la, lb = len(a), len(b)
    if not cta_route(la, lb, cap_ints):
        return {"warp"}
    path = coop_path(la, lb, 0, cap_ints, packed, plain_acgt(a) and plain_acgt(b))
    return {"cta", path, "spill" if ed > path_e_cap(path, la, lb, cap_ints) else "no_spill"}


# ---- sequence builders (every generator is seeded) ------------------------------------------------------------------------
def _rand(rng, n):
    return synth.ACGT[rng.integers(0, 4, size=n)].copy()


def _subs(x, lo, hi, k, rng, slots=0):
    """k substitutions on an even grid of max(k, slots) positions over [lo, hi), a few bases apart: each costs one edit."""
    x = x.copy()
    if k:
        step = (hi - lo) / max(k, slots)
        assert step >= 3, (lo, hi, k)
        pos = (lo + step * (np.arange(k) + 0.5)).astype(np.int64)
        code = np.searchsorted(synth.ACGT, x[pos])
        x[pos] = synth.ACGT[(code + rng.integers(1, 4, size=k)) % 4]
    return x


def _with_ed(rng, la, lb, ed, extra=0):
    """A pair of lengths la, lb at edit distance `ed` (>= |la - lb|): the length difference as one block deleted from or
    inserted into the longer side near its end, the rest as spaced substitutions before it (`extra` more or fewer, on the
    same grid)."""
    d = abs(la - lb)
    assert ed >= d
    n = max(la, lb)
    long_ = _rand(rng, n)
    c = n - d - 300 if n > d + 600 else n - d                # where the block starts
    short = np.concatenate([long_[:c], long_[c + d:]])
    short = _subs(short, 0, max(c - 50, 0), ed - d + extra, rng, slots=(ed - d) * 51 // 50 + 4)
    return (long_, short) if la >= lb else (short, long_)


def _kinds(rng, la, lb, unrelated=True):
    """Identical, substitutions, indel block, unrelated -- each at the lengths (la, lb) where the kind allows it."""
    out = []
    if la == lb:
        a = _rand(rng, la)
        out.append((a, a.copy()))
        if la:
            out.append((a, _subs(a, 0, la, min(12, la // 4), rng)))
        if la >= 64:
            k = min(400, la // 4); c = int(rng.integers(0, la - 2 * k))
            out.append((a, np.concatenate([a[:c], a[c + k:c + 2 * k], _rand(rng, k), a[c + 2 * k:]])))   # block moved
    else:
        a, b = _with_ed(rng, la, lb, abs(la - lb))
        out.append((a, b))                                                                             # one indel block
        if min(la, lb) >= 64:
            out.append(_with_ed(rng, la, lb, abs(la - lb) + 9))                                        # + substitutions
    if unrelated and max(la, lb) <= 12000:
        out.append((_rand(rng, la), _rand(rng, lb)))
    return [(bytes(x), bytes(y)) for x, y in out]


def routing_pairs():
    """Part 1: around the k_wfa_split thresholds at the default capacity."""
    rng = np.random.default_rng(1101)
    shapes = [(511, 511), (512, 512), (513, 513), (511, 700), (700, 511), (512, 700), (700, 512), (513, 701), (701, 513),
              (59999, 59999), (60000, 60000), (60001, 60001), (59999, 59000), (60000, 59000), (60001, 59000),
              (59000, 59999), (59000, 60000), (59000, 60001), (512, 9001), (9001, 512),
              (0, 0), (0, 5001), (5001, 0), (1, 513), (1023, 1021), (16383, 16385), (4099, 4099)]
    pairs = []
    for la, lb in shapes:
        pairs += _kinds(rng, la, lb)
    return pairs


def routing_pairs_shrunk():
    """Part 1 under AVK_TEST_COOP_CAP_INTS=SHRUNK_CAP_INTS: la + lb + 4096 on either side of 8 * cap_ints."""
    rng = np.random.default_rng(1102)
    s = 8 * SHRUNK_CAP_INTS - 4096
    shapes = [(s // 2, s // 2), (s // 2 + 1, s // 2 + 1), (s // 2 - 300, s // 2 + 300), (s // 2 - 300, s // 2 + 301),
              (s // 2 + 301, s // 2 - 300), (s // 2 + 300, s // 2 - 301), (512, s - 512), (512, s - 511)]
    pairs = []
    for la, lb in shapes:
        pairs += _kinds(rng, la, lb)
    return pairs


def _with_ed_exact(rng, la, lb, ed):
    """_with_ed, then more or fewer substitutions until the oracle's distance is `ed` (dense substitutions, and those next to
    the block, can share an edit).  Returns (a, b, the oracle's distance)."""
    seed, extra = int(rng.integers(1 << 30)), 0
    for _ in range(8):
        a, b = _with_ed(np.random.default_rng(seed), la, lb, ed, extra)
        got = orc.wfa_ed(bytes(a), bytes(b))
        if got == ed:
            break
        extra += ed - got
    return bytes(a), bytes(b), got


def _at_e_cap(rng, la_of, lb, e_cap_of, deltas):
    """Pairs whose edit distance is e_cap + delta for each delta.  la_of(ed) gives la for a distance (lb itself, or lb -/+
    the distance); where la moves e_cap the fixed point ed = e_cap(la_of(ed + delta)) is settled first."""
    out = []
    for dl in deltas:
        ed = e_cap_of(la_of(0), lb)
        for _ in range(30):
            ed = e_cap_of(la_of(ed + dl), lb)
        out.append(_with_ed_exact(rng, la_of(ed + dl), lb, ed + dl))
    return out


@functools.lru_cache(maxsize=None)
def spill_pairs():
    """Part 2 at the default capacity: edit distances just below, at and past the staged and the packed e_cap, where
    2 * (64000 - lb) binds (lb 59999, 58000, 55000) and where shared memory binds (la 59999 against lb 50000)."""
    rng = np.random.default_rng(1201)
    st = lambda la, lb: staged_e_cap(la, lb, COOP_CAP_INTS)
    pk = lambda la, lb: packed_e_cap(la, lb, COOP_CAP_INTS)
    pairs = []
    for lb in (59999, 58000, 55000):
        same = lambda ed, lb=lb: lb
        shorter = lambda ed, lb=lb: lb - ed                  # a = b with a block deleted: the distance is exactly the block
        pairs += _at_e_cap(rng, same, lb, st, (-1, 0, 1, 2))
        pairs += _at_e_cap(rng, same, lb, pk, (0, 1))
        pairs += _at_e_cap(rng, shorter, lb, st, (-1, 0, 1))
        pairs += _at_e_cap(rng, shorter, lb, pk, (0, 1))
    # la much longer than lb: la 59999 (the extra length inserted), substitutions up to the staged e_cap
    for lb in (55000, 50000):
        pairs += _at_e_cap(rng, lambda ed: 59999, lb, st, (-1, 0, 1))
    return pairs


@functools.lru_cache(maxsize=None)
def packed_edge_pairs():
    """Bytes the 2-bit packed path declines (N first, last and mid-sequence; a soft-masked run; an IUPAC code) and the
    16-base word boundary (16k +- 1), at the default capacity."""
    rng = np.random.default_rng(1202)
    out = []
    for la, lb in ((16383, 16384), (16384, 16384), (16385, 16383), (16385, 16385)):
        out.append(_with_ed(rng, la, lb, abs(la - lb) + 600))
    for where in ("first", "last", "mid", "soft", "iupac"):
        a, b = (x.copy() for x in _with_ed(rng, 16385, 16383, 2 + 700))
        if where == "first":
            a[0] = ord("N")
        elif where == "last":
            b[-1] = ord("N")
        elif where == "mid":
            a[8192] = ord("N"); b[5000] = ord("N")
        elif where == "soft":
            b[3000:3400] += 32                                    # lower case
        else:
            b[16000] = ord("R")
        out.append((a, b))
    return [(bytes(x), bytes(y), orc.wfa_ed(bytes(x), bytes(y))) for x, y in out]


@functools.lru_cache(maxsize=None)
def spill_pairs_shrunk():
    """Part 2 with the wavefront shrunk to SHRUNK_CAP_INTS: the same crossings at a few kbp, where shared memory binds."""
    rng = np.random.default_rng(1203)
    st = lambda la, lb: staged_e_cap(la, lb, SHRUNK_CAP_INTS)
    pk = lambda la, lb: packed_e_cap(la, lb, SHRUNK_CAP_INTS)
    pairs = []
    for lb in (8000, 7001):
        same = lambda ed, lb=lb: lb
        shorter = lambda ed, lb=lb: lb - ed
        pairs += _at_e_cap(rng, same, lb, st, (-1, 0, 1, 2))
        pairs += _at_e_cap(rng, shorter, lb, st, (-1, 0, 1))
        pairs += _at_e_cap(rng, shorter, lb, pk, (-1, 0, 1, 2))
    pairs += _at_e_cap(rng, lambda ed: 7000, 6000, st, (-1, 0, 1))
    for k in range(2):                                        # the packed path declines: N at both ends, a soft-masked run
        a, b = (x.copy() for x in _with_ed(rng, 8000, 7990, 1500))
        if k == 0:
            a[0] = ord("N"); b[-1] = ord("N")
        else:
            b[100:500] += 32
        pairs.append((bytes(a), bytes(b), orc.wfa_ed(bytes(a), bytes(b))))
    return pairs


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


def _oracle_eds(pairs):
    return np.array([orc.wfa_ed(a, b) for a, b in pairs], dtype=np.uint32)


@pytest.fixture(scope="module")
def solver():
    s = Solver(0)
    yield s
    s.close()


@pytest.mark.gpu
def test_wfa_ed_routing_thresholds_vs_oracle(solver):
    """k_wfa_split: min(la, lb) 511 / 512 / 513, max(la, lb) 59999 / 60000 / 60001, one length far below the other, an empty
    side, lengths off the 4- and 16-byte grid; then la + lb + 4096 on either side of 8 * cap_ints under a shrunk wavefront."""
    pairs = routing_pairs()
    assert np.array_equal(solver.wfa_ed_batch(pairs), _oracle_eds(pairs))
    pairs = routing_pairs_shrunk()
    cpu = _oracle_eds(pairs)
    s = _solver_with_env(AVK_TEST_COOP_CAP_INTS=SHRUNK_CAP_INTS)
    try:
        assert np.array_equal(s.wfa_ed_batch(pairs), cpu)
    finally:
        s.close()


@pytest.mark.gpu
def test_wfa_ed_staged_and_packed_spill_vs_oracle(solver):
    """The staged and packed paths just below, at and past their e_cap, where 2 * (64000 - lb) binds and where shared memory
    binds; past it the alignment is finished on the warp path from the state the CTA wrote back."""
    cases = spill_pairs() + packed_edge_pairs()              # (a, b, the oracle's distance)
    pairs, cpu = [c[:2] for c in cases], np.array([c[2] for c in cases], dtype=np.uint32)
    assert np.array_equal(solver.wfa_ed_batch(pairs), cpu)
    shrunk, cpu_shrunk = [c[:2] for c in spill_pairs_shrunk()], np.array([c[2] for c in spill_pairs_shrunk()], dtype=np.uint32)
    try:
        for env in (dict(AVK_PACKED_DWFA=1), dict(AVK_TEST_COOP_CAP_INTS=SHRUNK_CAP_INTS),
                    dict(AVK_PACKED_DWFA=1, AVK_TEST_COOP_CAP_INTS=SHRUNK_CAP_INTS)):
            s = _solver_with_env(**env)
            try:
                if "AVK_TEST_COOP_CAP_INTS" in env:
                    assert np.array_equal(s.wfa_ed_batch(shrunk), cpu_shrunk), env
                else:
                    assert np.array_equal(s.wfa_ed_batch(pairs), cpu), env
            finally:
                s.close()
    finally:
        Solver(0).close()                                      # AVK_PACKED_DWFA is device-wide: back to the default


# ---- compare path under default capacities ---------------------------------------------------------------------------------
FLANK = 1000
HOM, H01 = abi.ZYG_HOM_ALT, abi.ZYG_PHASED_HET01


def compare_clusters(seed=1301):
    """Hand-made clusters, mostly HOM records (small searches).  Returns the reference, the truth and query records and,
    per targeted cluster, (name, a position inside it, detail)."""
    rng = np.random.default_rng(seed)
    ref = synth.random_reference(760_000, rng)
    T, Q, named = [], [], []
    base = lambda p: bytes([int(ref[p])])

    def snv(p, z=HOM):
        alt = b"ACGT"[(b"ACGT".index(base(p)) + int(rng.integers(1, 4))) % 4:][:1]
        return synth.make_rec(p, base(p), alt, z)

    def ins(p, n, z=HOM):
        return synth.make_rec(p, base(p), base(p) + synth._rand_seq(rng, n), z)

    def dele(p, n, z=HOM):
        return synth.make_rec(p, ref[p:p + 1 + n].tobytes(), base(p), z)

    def both(r):
        T.append(r); Q.append(r)

    def snvs(lo, hi, step, skip=()):
        """SNVs on both sides every `step` bases, none inside the [s, e) ranges of `skip`."""
        for p in range(lo, hi, step):
            if not any(s <= p < e for s, e in skip):
                both(snv(p))

    def tail(a0, a1):
        """make_rec trims trailing bases the alleles share: shorten a1 until its last base differs."""
        while len(a1) > 1 and a1[-1] == a0[-1]:
            a1 = a1[:-1]
        return a1

    pos = 5000
    # (a) windows of 64 kbp and more with small truth / query edit distances: records 400-900 bp apart, a few 300-1000 bp
    # indels (the edit-distance bound sends the cluster to the cooperative tier, and the basepair metrics align the
    # reference window to haplotypes of 64 kbp and more), a few false negative and false positive SNVs
    for span in (66_000, 71_000):
        named.append(("long_window", pos, None))
        p, k = pos, 0
        while p < pos + span:
            if k % 23 == 5:
                both(ins(p, int(rng.integers(300, 1001))))
            elif k % 23 == 16:
                n = int(rng.integers(300, 1001)); both(dele(p, n)); p += n
            elif k % 31 == 7:
                T.append(snv(p))                                   # FN
            elif k % 37 == 11:
                Q.append(snv(p))                                   # FP
            else:
                both(snv(p))
            p += int(rng.integers(400, 900)); k += 1
        pos += span + 5000
    # (b) a haplotype of exactly 63999, 64000 and 64001 bp in a window below 64 kbp, set by the insertions
    for target in (63_999, 64_000, 64_001):
        named.append(("hap_%d" % target, pos + 600, None))
        recs = [snv(pos + 600 * i) for i in range(1, 95)]                                        # window ~ 58 kbp
        ins_pos = [pos + 600 * i + 300 for i in range(3, 90, 11)]
        last = max(r[0] + len(r[1]) for r in recs)
        window = (last + FLANK) - (pos + 600 - FLANK)
        total = target - window
        sizes = [total // len(ins_pos)] * len(ins_pos)
        sizes[-1] += total - sum(sizes)
        recs += [ins(p, n) for p, n in zip(ins_pos, sizes)]
        for r in sorted(recs, key=lambda r: r[0]):
            both(r)
        Q.append(snv(pos + 600 * 50 + 100))                        # one FP: the search has a choice to make
        pos = last + 5000
    # (c) truth-only deletions totalling 13.5-16 kbp: ED(truth hap, query hap) past the 12,998 that the 32-bit wavefront of
    # the default capacity holds in shared memory, on haplotypes of 22-54 kbp
    for dels, span in (((7000, 6600), 52_000), ((6900, 6700), 36_000)):
        named.append(("deep_ed", pos, None))
        starts = np.linspace(pos + 900, pos + span - 2000, len(dels) + 1).astype(int)[:len(dels)] + 10
        ranges = [(int(s), int(s) + n + 1) for s, n in zip(starts, dels)]
        snvs(pos, pos + span, 850, ranges)
        for (s, _), n in zip(ranges, dels):
            T.append(dele(s, n))
        pos = max(pos + span, ranges[-1][1]) + 5000
    # (d) a 4-6 kbp FN early in a 50-60 kbp window: the updates behind it resume the truth / query alignment at an edit
    # distance in the thousands -- on the staged path while the haplotypes are short, on the 32-bit path once
    # 2 * (64000 - lb) < 2 * ED + 256
    for n_fn, span, fn_ins in ((5000, 58_000, False), (4200, 60_000, True), (6000, 52_000, False)):
        fn = pos + 1210
        named.append(("resume", pos, fn - (pos - FLANK)))
        snvs(pos, pos + span, 800, [] if fn_ins else [(fn, fn + n_fn + 1)])
        T.append(ins(fn, n_fn) if fn_ins else dele(fn, n_fn))
        if fn_ins:
            Q.append(snv(pos + 30_410, H01))                        # a query het behind the insertion
        pos += span + 5000
    # (e) long complex records: both alleles 1-10 kbp and neither a prefix of the other, equal-length long replacements, an
    # allele that is a long prefix of the other (k_alt_ed's warp alignment and its prefix shortcut); one pair differs.  One
    # cluster each: the basepair metrics align the reference window to the haplotype, at a cost of about ED^2 on the CPU
    for l0, l1, kind in ((3000, 2500, "replace"), (1200, 9500, "replace"), (9000, 1100, "replace"), (2000, 2000, "replace"),
                         (6000, 6000, "similar"), (4000, 1500, "prefix"), (1500, 5200, "prefix")):
        named.append(("complex", pos, None))
        a0 = ref[pos:pos + l0].tobytes()
        if kind == "replace":
            a1 = a0[:1] + synth._rand_seq(rng, l1 - 1)
        elif kind == "similar":
            arr = np.frombuffer(a0, dtype=np.uint8).copy()
            idx = np.arange(5, l0 - 5, 37)
            arr[idx] = synth.ACGT[(np.searchsorted(synth.ACGT, arr[idx]) + 1) % 4]
            a1 = arr.tobytes()
        elif l1 < l0:
            a1 = a0[:l1]
        else:
            a1 = a0 + synth._rand_seq(rng, l1 - l0)
        a1 = tail(a0, a1)
        if kind == "similar":                                       # truth and query disagree by one base inside the ALT
            T.append(synth.make_rec(pos, a0, a1, HOM))
            q1 = a1[:3000] + (b"A" if a1[3000:3001] != b"A" else b"C") + a1[3001:]
            Q.append(synth.make_rec(pos, a0, q1, HOM))
        else:
            both(synth.make_rec(pos, a0, a1, HOM))
        both(snv(pos + l0 + 700))
        pos += l0 + 5000
    assert pos + 5000 < ref.size, pos
    return ref, T, Q, named


def compare_batch_cases():
    ref, T, Q, named = compare_clusters()
    return ref, synth.cluster_regions([T, Q], ref.size, FLANK), named


@pytest.mark.gpu
def test_compare_boundaries_vs_oracle():
    """Compare clusters under default capacities whose CTA-wide alignments reach the 32-bit body (sequences of 64 kbp and
    more), the spill and the resumption of a spilled alignment; every output array, then again with the packed path on."""
    ref, batch, _ = compare_batch_cases()
    cfg = CompareConfig(enable_sequences=False)
    cpu = orc.compare_batch(batch, [ref], compare_cfg(cfg), n_threads=orc.num_threads())
    assert int(max(cpu.ed1.max(), cpu.ed2.max())) > (COOP_CAP_INTS - 3) // 2
    try:
        for env in (dict(), dict(AVK_PACKED_DWFA=1)):
            s = _solver_with_env(**env)
            try:
                s.set_reference([ref])
                gpu = s.compare_batch(batch, cfg)
                assert gpu.diff(cpu) == [], env
                assert int(gpu.error_blocks[0]) == 0 and int(gpu.solved_blocks[0]) == batch.n_regions, env
                assert s.last_tier_overflow()[2] > 0, "no cluster reached the cooperative tier"
            finally:
                s.close()
    finally:
        Solver(0).close()                                      # AVK_PACKED_DWFA is device-wide: back to the default


# ---- route coverage (CPU) ------------------------------------------------------------------------------------------------
def _haplotypes(ref, batch, r):
    """Truth and query haplotype of region r when all its records are HOM (None otherwise)."""
    s, e = int(batch.start[r]), int(batch.end[r])
    out = []
    for side in (0, 1):
        v0, v1 = int(batch.var_off[2 * r + side]), int(batch.var_off[2 * r + side + 1])
        parts, cur = [], s
        for v in range(v0, v1):
            if int(batch.zygosity[v]) != HOM:
                return None
            p, o = int(batch.position[v]), int(batch.allele_off[v])
            l0, l1 = int(batch.a0_len[v]), int(batch.a1_len[v])
            parts += [ref[cur:p].tobytes(), batch.allele_pool[o + l0:o + l0 + l1].tobytes()]
            cur = p + l0
        parts.append(ref[cur:e].tobytes())
        out.append(b"".join(parts))
    return out


def test_route_coverage():
    """The case generators above aim at every route: warp / CTA, staged / packed / 32-bit, spill / no spill, for
    avk_wfa_ed_batch and for the compare path's CTA-wide alignments.  Edit distances are the oracle's."""
    got = set()
    for pairs, cap in ((routing_pairs(), COOP_CAP_INTS), (routing_pairs_shrunk(), SHRUNK_CAP_INTS)):
        for a, b in pairs:
            la, lb = len(a), len(b)
            got.add("cta" if cta_route(la, lb, cap) else "warp")
            if min(la, lb) in (511, 512, 513) and la and lb:
                got.add("min_%d_%s" % (min(la, lb), "cta" if cta_route(la, lb, cap) else "warp"))
            if max(la, lb) in (59999, 60000, 60001) and min(la, lb) >= 512:
                got.add("max_%d_%s" % (max(la, lb), "cta" if cta_route(la, lb, cap) else "warp"))
            if cap == SHRUNK_CAP_INTS and min(la, lb) >= 512:
                got.add("sum_%s" % ("cta" if cta_route(la, lb, cap) else "warp"))
    for name in ("min_511_warp", "min_512_cta", "min_513_cta", "max_59999_cta", "max_60000_warp", "max_60001_warp",
                 "sum_cta", "sum_warp"):
        assert name in got, name
    for pairs, cap in ((spill_pairs() + packed_edge_pairs(), COOP_CAP_INTS), (spill_pairs_shrunk(), SHRUNK_CAP_INTS)):
        tag = "default" if cap == COOP_CAP_INTS else "shrunk"
        for a, b, ed in pairs:
            la, lb = len(a), len(b)
            assert cta_route(la, lb, cap), (la, lb, cap)
            for packed in (False, True):
                path = coop_path(la, lb, 0, cap, packed, plain_acgt(a) and plain_acgt(b))
                e_cap = path_e_cap(path, la, lb, cap)
                if packed and path != "packed":
                    got.add("packed_declined_" + tag)
                rel = "below" if ed < e_cap else ("at" if ed == e_cap else "past")
                got.add("%s_%s_%s_%s" % (tag, path, binding_bound(path, la, lb, cap), rel))
    for tag, bounds in (("default", ("16bit", "smem")), ("shrunk", ("smem",))):
        for path in ("staged", "packed"):
            for bound in bounds:
                if (tag, path, bound) == ("default", "packed", "smem"):
                    continue                                   # (the packed layout's room exceeds 2 * (64000 - lb) from ~40.5 kbp)
                for rel in ("below", "at", "past"):
                    assert "%s_%s_%s_%s" % (tag, path, bound, rel) in got, (tag, path, bound, rel)
        assert "packed_declined_" + tag in got
    # avk_wfa_ed_batch cannot reach the 32-bit CTA body: every pair k_wfa_split admits fits the staged path at ED 0
    for cap in (64, 700, SHRUNK_CAP_INTS, 12000, COOP_CAP_INTS):
        for la in range(512, 60000, 331):
            for lb in (512, 513, 4099, 30000, 59999):
                if cta_route(la, lb, cap):
                    assert coop_path(la, lb, 0, cap, False, True) == "staged", (la, lb, cap)
    # compare path: haplotype lengths and the oracle's edit distances of the targeted clusters
    ref, batch, named = compare_batch_cases()
    cpu = orc.compare_batch(batch, [ref], compare_cfg(CompareConfig(enable_sequences=False)), n_threads=orc.num_threads())
    got = set()
    for name, p, detail in named:
        r = int(np.searchsorted(batch.start, p, side="right")) - 1
        assert batch.start[r] <= p < batch.end[r], name
        v0, v1 = int(batch.var_off[2 * r]), int(batch.var_off[2 * r + 2])
        if int(np.maximum(batch.a0_len[v0:v1], batch.a1_len[v0:v1]).sum()) >= WIDE_B0:
            got.add("coop_tier")
        ed = int(max(cpu.ed1[r], cpu.ed2[r]))
        haps = _haplotypes(ref, batch, r)
        win = ref[int(batch.start[r]):int(batch.end[r])].tobytes()
        if haps is not None:
            lt, lq = len(haps[0]), len(haps[1])
            for h in haps:                                     # the basepair metrics align the reference window to each haplotype
                if max(len(win), len(h)) >= 64000 and orc.wfa_ed(win, h) >= COOP_MIN_ED:
                    got.add("metrics_32bit_64kbp")
            if name.startswith("hap_") and lt == int(name[4:]):
                got.add(name)
        else:
            lt = lq = len(win)
        if ed >= COOP_MIN_ED:
            path = coop_path(lt, lq, COOP_MIN_ED, COOP_CAP_INTS, False, True)
            got.add("tq_%s_%s" % (path, "spill" if ed > path_e_cap(path, lt, lq, COOP_CAP_INTS) else "no_spill"))
            if path != "32bit" and ed > path_e_cap(path, lt, lq, COOP_CAP_INTS):
                # resumed past the staged e_cap: the 32-bit tail, and past its own e_cap the immediate spill
                e32 = (COOP_CAP_INTS - 3) // 2
                got.add("tq_resumed_32bit_%s" % ("spill" if ed > e32 else "no_spill"))
        if name == "resume":
            after = detail + 2000                              # the haplotypes a few records behind the FN event
            if coop_path(after, after, ed, COOP_CAP_INTS, False, True) == "staged":
                got.add("resume_staged")
            if coop_path(lt, lq, ed, COOP_CAP_INTS, False, True) == "32bit":
                got.add("resume_32bit")
    need = {"coop_tier", "metrics_32bit_64kbp", "hap_63999", "hap_64000", "hap_64001", "tq_staged_spill",
            "tq_staged_no_spill", "tq_resumed_32bit_spill", "tq_resumed_32bit_no_spill", "resume_staged", "resume_32bit"}
    assert not need - got, need - got
