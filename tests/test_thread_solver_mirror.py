"""Basepair metrics of clusters whose truth and query lists are the same records (avk_thread_solver.cuh, mirror_lists): the
thread solver runs one filter pass per type slot for both sides.  Host build of the thread solver against the oracle on
identical lists of 2..5 records per side -- every zygosity combination (truth unphased / 0|1 / 1|0 / hom, query with the same
ALT copies in either phase), substitutions, anchored insertions and deletions, windows that are random, homopolymer or di- /
tri-nucleotide repeats (non-additive edit distances, subsets that spell the same string) -- and neighbouring shapes that
break the identity (a different ALT, overlapping or no-op records, an extra record, different copies or allele space)."""
import itertools

import numpy as np
import pytest

from aardvark_b200 import abi, synth
from aardvark_b200.batch import RegionBatch
from aardvark_b200.types import CompareRegion, Coordinates, PhasedZygosity as Z, Variant, VariantType
from test_thread_solver_host import check

HETS = (Z.UnphasedHeterozygous, Z.PhasedHet01, Z.PhasedHet10)
# (truth, query) zygosity of one record pair: the same ALT copies, the query in either phase
PAIRS = [(t, q) for t in HETS for q in HETS] + [(Z.HomozygousAlternate, Z.HomozygousAlternate)]
SEG = 400        # bases of reference per cluster
WIN = 240        # window length


def _window(kind, rng):
    if kind == "random":
        return synth.ACGT[rng.integers(0, 4, size=SEG)].tobytes()
    if kind == "homopolymer":
        return bytes([synth.ACGT[rng.integers(0, 4)]]) * SEG
    unit = synth.ACGT[rng.permutation(4)[:2 if kind == "di" else 3]].tobytes()
    return (unit * SEG)[:SEG]


def _other(b, rng):
    return bytes([[x for x in b"ACGT" if x != b[0]][int(rng.integers(0, 3))]])


def _record(kind, ref, p, rng):
    """One variant at p: substitution, anchored insertion / deletion, or a shape the thread solver's metric pass must not mirror."""
    if kind == "snv":
        return Variant(0, VariantType.Snv, p, ref[p:p + 1], _other(ref[p:p + 1], rng))
    if kind == "ins":
        k = int(rng.integers(1, 7))
        ins = ref[p + 1:p + 1 + k] if rng.random() < 0.5 else synth.ACGT[rng.integers(0, 4, size=k)].tobytes()   # often a repeat copy
        return Variant(0, VariantType.Insertion, p, ref[p:p + 1], ref[p:p + 1] + ins)
    if kind == "del":
        k = int(rng.integers(1, 7))
        return Variant(0, VariantType.Deletion, p, ref[p:p + 1 + k], ref[p:p + 1])
    if kind == "noop":                                                  # ALT == reference base
        return Variant(0, VariantType.Snv, p, ref[p:p + 1], ref[p:p + 1])
    if kind == "unanchored":                                            # first ALT base differs from the reference
        return Variant(0, VariantType.Insertion, p, ref[p:p + 1], _other(ref[p:p + 1], rng) + b"T")
    raise ValueError(kind)


def make_batch(n_clusters, seed, m_range=(2, 5), enumerate_m=None, p_decline=0.15):
    """Clusters of M identical records per side; with probability p_decline one neighbouring shape that breaks the identity
    (a different query ALT, overlapping records, two indels, a no-op or unanchored record, an extra query record, different
    copies).  enumerate_m: every zygosity combination of M records, once each, instead of random draws."""
    rng = np.random.default_rng(seed)
    combos = list(itertools.product(PAIRS, repeat=enumerate_m)) if enumerate_m else None
    n = len(combos) if combos else n_clusters
    ref = bytearray()
    regions = []
    for i in range(n):
        seg = _window(("random", "homopolymer", "di", "tri")[i % 4], rng)
        off = len(ref)
        ref += seg
        M = enumerate_m or int(rng.integers(m_range[0], m_range[1] + 1))
        zy = combos[i] if combos else [PAIRS[int(rng.integers(0, len(PAIRS)))] for _ in range(M)]
        kinds = ["snv"] * M
        r = rng.random()
        if r < 0.6:
            kinds[int(rng.integers(0, M))] = ("ins", "del")[int(rng.integers(0, 2))]
        decline = rng.random() < p_decline
        shape = int(rng.integers(0, 7)) if decline else -1
        if shape == 0:
            kinds[0], kinds[-1] = "ins", "del"
        elif shape == 1:
            kinds[int(rng.integers(0, M))] = ("noop", "unanchored")[int(rng.integers(0, 2))]
        refb = bytes(ref)
        tv, p = [], off + 20
        for k in kinds:
            v = _record(k, refb, p, rng)
            tv.append(v)
            p += len(v.allele0) + int(rng.integers(0, 12))               # 0: the next record starts where this one ends
        qv = list(tv)
        tz, qz = [z[0] for z in zy], [z[1] for z in zy]
        if shape == 2:
            j = int(rng.integers(0, M))
            if len(qv[j].allele0) == 1 and len(qv[j].allele1) == 1:
                a = bytes([x for x in b"ACGT" if x not in (refb[qv[j].position], qv[j].allele1[0])][0:1])
                qv[j] = Variant(0, VariantType.Snv, qv[j].position, qv[j].allele0, a)
        elif shape == 3:                                                 # overlapping: the last record moves onto the previous one
            last = tv[-1]
            pp = tv[-2].position
            tv[-1] = qv[-1] = _record("snv", refb, pp, rng) if last.variant_type == VariantType.Snv else last
        elif shape == 4:
            qv = qv + [_record("snv", refb, p + 3, rng)]
            qz = qz + [Z.HomozygousAlternate]
        elif shape == 5:
            j = int(rng.integers(0, M))
            qz[j] = Z.HomozygousAlternate if qz[j] != Z.HomozygousAlternate else Z.PhasedHet01
        elif shape == 6:
            j = int(rng.integers(0, M))
            qv[j] = Variant(0, qv[j].variant_type, qv[j].position, qv[j].allele0, qv[j].allele1, qv[j].raw_allele_space + 3)
        regions.append(CompareRegion(i, Coordinates("c", off + 10, off + 10 + WIN), tv, tz, qv, qz))
    return bytes(ref), RegionBatch.from_compare_regions(regions, {"c": 0})


@pytest.mark.parametrize("m", [2, 3])
def test_thread_solver_identical_lists_every_zygosity(m):
    ref, batch = make_batch(0, seed=100 + m, enumerate_m=m, p_decline=0.0)
    for mbf in (50, 16, 8, 4):
        check(batch, [ref], abi.CompareCfg(mbf, 0, 0, 0))


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_thread_solver_identical_lists_random_shapes(seed):
    ref, batch = make_batch(4000, seed=seed)
    for mbf in (50, 8):
        check(batch, [ref], abi.CompareCfg(mbf, 0, 0, 0), min_accept=0.5)
