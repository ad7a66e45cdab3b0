"""The comparison helpers of tests/graph_scale.py are sensitive: fed the oracle's own graph they pass, and fed it with
one defect each -- two slots of a vertex swapped, one multiplicity off by one, two vertex ids exchanged in EDGE_V2, one
start off by one, two expanded edges swapped, one high key word flipped -- they raise."""
import numpy as np
import pytest

import _native as N
import oracle
from graph_scale import (Artifacts, assert_graph_canonical, assert_graph_label_free, assert_partitioned, derived_graph, owner,
                         partition_of, relabel, same)
from util import random_reads


def _graph(l):
    reads = random_reads(41, 400, genome_len=3000, lens=(64, 80, 100, 150), n_frac=0.1) + ["A" * 90, "ACGT" * 30]
    buf, off = oracle.pack_reads(reads)
    return oracle.graph_build(buf, off, l, expand=True)


def _vertex_with_two_slots(lc):
    rows = lc.reshape(-1, 4)
    i = int(np.flatnonzero((rows != rows[:, :1]).any(1))[0])
    a = 0
    b = int(np.flatnonzero(rows[i] != rows[i, 0])[0])
    return i, a, b


def _swap_slots(a):
    x = a[N.ART_LCOUNT]
    i, p, q = _vertex_with_two_slots(x)
    x[4 * i + p], x[4 * i + q] = x[4 * i + q], x[4 * i + p]


def _lval_plus_one(a):
    a[N.ART_LMER_VALUES][len(a[N.ART_LMER_VALUES]) // 2] += 1


def _swap_v2(a):
    v2 = a[N.ART_EDGE_V2]
    j = int(np.flatnonzero(v2 != v2[0])[0])
    v2[0], v2[j] = v2[j], v2[0]


def _lstart_off_by_one(a):
    a[N.ART_LSTART][len(a[N.ART_LSTART]) // 3] += 1


def _swap_ee(a):
    ee = a[N.ART_EE]
    j = int(np.flatnonzero(ee["v1"] != ee["v1"][0])[0])
    ee[[0, j]] = ee[[j, 0]]


def _flip_hi(a):
    a[N.ART_KMER_KEYS_HI][len(a[N.ART_KMER_KEYS_HI]) // 2] ^= np.uint64(1 << 5)


DEFECTS = {"slots swapped": _swap_slots, "lvals + 1": _lval_plus_one, "v2 ids exchanged": _swap_v2,
           "lstart off by one": _lstart_off_by_one, "EE rows swapped": _swap_ee, "hi word flipped": _flip_hi}


@pytest.mark.parametrize("l", [32, 48])
@pytest.mark.parametrize("defect", sorted(DEFECTS))
def test_canonical_helper_catches_each_defect(l, defect):
    g = _graph(l)
    wide = l > 32
    assert_graph_canonical(Artifacts(g), g, wide)
    if defect == "hi word flipped" and not wide:
        pytest.skip("one-word keys")
    art = Artifacts(g)
    DEFECTS[defect](art.a)
    with pytest.raises(AssertionError):
        assert_graph_canonical(art, g, wide)


@pytest.mark.parametrize("l", [32, 48])
@pytest.mark.parametrize("defect", sorted(set(DEFECTS) - {"EE rows swapped"}))   # slot-order runs do not expand edges
def test_label_free_helper_catches_each_defect(l, defect):
    g = _graph(l)
    wide = l > 32
    assert_graph_label_free(relabel(g, 1), g, wide)
    assert_graph_label_free(Artifacts(g), g, wide)
    if defect == "hi word flipped" and not wide:
        pytest.skip("one-word keys")
    art = relabel(g, 2)
    DEFECTS[defect](art.a)
    with pytest.raises(AssertionError):
        assert_graph_label_free(art, g, wide)


_PART_DEFECTS = {
    "slots swapped": lambda p: _swap_slots({N.ART_LCOUNT: p["LCOUNT"]}),
    "lvals + 1": lambda p: _lval_plus_one({N.ART_LMER_VALUES: p["LMER_VALUES"]}),
    "v2 ids exchanged": lambda p: _swap_v2({N.ART_EDGE_V2: p["EDGE_V2"]}),
    "lstart off by one": lambda p: _lstart_off_by_one({N.ART_LSTART: p["LSTART"]}),
    "hi word flipped": lambda p: _flip_hi({N.ART_KMER_KEYS_HI: p["KMER_KEYS_HI"]}),
}


@pytest.mark.parametrize("l", [22, 48])
@pytest.mark.parametrize("defect", sorted(_PART_DEFECTS))
def test_partition_helper_catches_each_defect(l, defect):
    g = _graph(l)
    world = 3
    parts, windows = partition_of(g, world)
    assert all(p["KMER_KEYS"].size for p in parts)
    assert_partitioned(parts, windows, g, world)
    if defect == "hi word flipped" and l <= 32:
        pytest.skip("one-word keys")
    _PART_DEFECTS[defect](parts[1])
    with pytest.raises(AssertionError):
        assert_partitioned(parts, windows, g, world)


def test_owner_restates_the_scalar_rule():
    """the array form of the ownership rule equals the scalar restatement in tests/test_gpu_dist.py"""
    from test_gpu_dist import owner_kmer
    g = _graph(22)
    for world in (2, 8):
        got = owner(g.vk_lo[:500], g.vk_hi[:500], 21, world)
        assert got.tolist() == [owner_kmer(int(v), 21, world) for v in g.vk_lo[:500]]


@pytest.mark.parametrize("l", [12, 22, 32])
def test_derived_graph_equals_the_oracle_graph(l):
    """derived_graph (the check of the graph too large for the oracle's graph build) on reads without N, every one at
    least l long: what the oracle builds"""
    reads = [r.replace("N", "A") for r in random_reads(43, 600, genome_len=4000, lens=(64, 100, 150), n_frac=0.0)]
    reads = [r for r in reads if len(r) >= l] + ["A" * 90, "ACGT" * 30]
    buf, off = oracle.pack_reads(reads)
    g = oracle.graph_build(buf, off, l, expand=False)
    assert np.array_equal(oracle.count_mers(buf, off, l - 1)[0], g.vk_lo)
    exp = Artifacts(g).a
    for name, a in derived_graph(g.lk_lo, g.lvals, g.vk_lo, l).items():
        same(name, a, exp[getattr(N, "ART_" + name)])
