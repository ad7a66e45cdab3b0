"""CPU tests of tests/unitig_np.py, the vectorised restatement behind the exact GPU checks at scale: it must agree
with the string restatements (clean_ref.path_unitigs, clean_ref.clean) on every shape of tests/unitig_shapes.py, and
`certify` must accept the reference's unitigs and reject every kind of wrong contig list."""
import numpy as np
import pytest

import unitig_np as U
import unitig_shapes as S
from clean_ref import clean, path_unitigs
from oracle import py_all_contigs, py_build, twin

KS = list(range(2, 41))
VARIANTS = [{}, {"isolated_len": 0, "bubble_len": 0}, {"tip_len": 0, "bubble_len": 0}, {"tip_len": 0, "isolated_len": 0},
            {"max_rounds": 1}]


def _case(name, K, limit):
    reads = S.shape(name, K)
    return py_build([r.upper() for r in reads], K, limit), U.from_reads(reads, K, limit)


def _nodes(g, mask):
    return {g.text(i) for i in np.nonzero(mask)[0]}


@pytest.mark.parametrize("name", S.SHAPES)
def test_graph_and_chains_match_strings(name):
    for K in KS:
        for limit in (0, 1, 2):
            d, g = _case(name, K, limit)
            assert {g.text(i): int(c) for i, c in enumerate(g.cnt)} == d, (K, limit)
            alive = np.ones(g.n, bool)
            paths, cycles = U.path_chains(g, alive)
            exp = path_unitigs(d)
            assert sorted([g.text(x) for x in c] for c in paths) == sorted(exp), (K, limit)
            on_path = {x for c in exp for x in c}
            assert {g.text(x) for c in cycles for x in c} == set(d) - on_path, (K, limit)


@pytest.mark.parametrize("name", S.SHAPES)
def test_clean_matches_strings(name):
    for K in KS:
        for limit in (0, 1, 2):
            d, g = _case(name, K, limit)
            for kw in VARIANTS:
                A, est = clean(d, K, **kw)
                alive, st = U.clean(g, **kw)
                assert st == est, (K, limit, kw)
                assert _nodes(g, alive) == set(A), (K, limit, kw)


def test_shapes_have_their_features():
    """the shapes reach what they are for: self-loops, self-twin cycles, palindromes at the count limit, hairpins,
    clean-up removals next to repeats"""
    g = U.from_reads(S.tandem(), 10, 1)
    _, cycles = U.path_chains(g, np.ones(g.n, bool))
    assert any(len(c) == 1 for c in cycles)                                     # A^10 -> A^10
    assert any(len(c) == 4 and set(c) == set(g.twin[c]) for c in cycles)        # ACGT^n
    for limit, kept in ((1, True), (2, False)):
        d = py_build(S.pal_once(), 10, limit)
        assert any(x == twin(x) for x in d) == kept
    d = py_build(S.inverted(), 15, 1)
    assert any(twin(x) in [x[1:] + b for b in "ACGT"] for x in d)              # fw(x) holds twin(x)
    tot = {"tips": 0, "bubble_branches": 0, "isolated": 0}
    for K in (15, 21, 31):
        _, st = U.clean(U.from_reads(S.repeats(), K, 1))
        for k in tot:
            tot[k] += st[k]
    assert all(tot.values()), tot


# ---- certify --------------------------------------------------------------------------------------------------------
def _ref(name, K, limit):
    reads = S.shape(name, K)
    d = py_build([r.upper() for r in reads], K, limit)
    g = U.from_reads(reads, K, limit)
    contigs = py_all_contigs(d, K)
    sums = [sum(d[c[i:i + K]] for i in range(len(c) - K + 1)) for c in contigs]
    return g, contigs, sums


def _self_twin(c, K):
    nodes = {c[i:i + K] for i in range(len(c) - K + 1)}
    return any(twin(x) in nodes for x in nodes)


@pytest.mark.parametrize("name", S.SHAPES)
def test_certify_accepts_the_reference(name):
    checked = 0
    for K in KS:
        for limit in (0, 1):
            g, contigs, sums = _ref(name, K, limit)
            if any(_self_twin(c, K) for c in contigs):
                continue   # the reference writes a self-twin unitig in part (see _canon_set)
            assert U.certify(contigs, sums, g, np.ones(g.n, bool)) == [], (K, limit)
            checked += 1
    assert checked >= 20


def _corruptions(contigs, sums, K):
    """(what, contigs, sums or None) of deliberate errors in a correct unitig list"""
    longest = max(range(len(contigs)), key=lambda i: len(contigs[i]))
    c = contigs[longest]
    rest = contigs[:longest] + contigs[longest + 1:]
    yield "cut", rest + [c[:K + 1], c[2:]], None
    # two unitigs joined across a branch node: y's first K-mer is a forward extension of x's last one
    ends = {}
    for j, y in enumerate(contigs):
        ends.setdefault(y[:K - 1], j)
    for i, x in enumerate(contigs):
        j = ends.get(x[-K + 1:])
        if j is not None and j != i and not (_self_twin(x, K) or _self_twin(contigs[j], K)):
            yield "joined", [z for t, z in enumerate(contigs) if t not in (i, j)] + [x + contigs[j][K - 1:]], None
            break
    yield "dropped K-mer", rest + [c[:-1]], None
    yield "written twice", contigs + [c], None
    yield "both orientations", contigs + [twin(c)], None
    ws = list(sums)
    ws[longest] += 1
    yield "wrong sum", contigs, ws


def test_certify_rejects_corruptions():
    K = 21
    g, contigs, sums = _ref("repeats", K, 1)
    alive = np.ones(g.n, bool)
    assert U.certify(contigs, sums, g, alive) == []
    seen = set()
    for what, bad, bad_sums in _corruptions(contigs, sums, K):
        assert U.certify(bad, bad_sums, g, alive), what
        seen.add(what)
    assert seen == {"cut", "joined", "dropped K-mer", "written twice", "both orientations", "wrong sum"}


def test_certify_rejects_a_cycle_from_the_wrong_node():
    K = 4
    g = U.from_reads(["ACGT" * 10], K, 1)        # the self-twin cycle ACGT -> CGTA -> GTAC -> TACG -> ACGT
    alive = np.ones(g.n, bool)
    sums = lambda cs: [sum(int(g.cnt[i]) for i in U.windows(g, [c])[0]) for c in cs]
    assert U.certify(["ACGTACG"], sums(["ACGTACG"]), g, alive) == []
    assert U.certify(["CGTACGT"], sums(["CGTACGT"]), g, alive) == []          # another rotation is fine
    for bad in (["ACGTACGT"], ["ACGTAC"], ["ACGTACG", "ACGTACG"]):               # first node repeated, cut, twice
        assert U.certify(bad, sums(bad), g, alive), bad
    # a path unitig is not a cycle: writing poly-A's self-loop twice over is wrong, once is right
    g = U.from_reads(["A" * 30], 5, 1)
    alive = np.ones(g.n, bool)
    assert U.certify(["AAAAA"], [int(g.cnt[0])], g, alive) == []
    assert U.certify(["AAAAAA"], [2 * int(g.cnt[0])], g, alive)


def test_certify_checks_the_alive_set():
    K = 21
    g, contigs, sums = _ref("repeats", K, 1)
    alive, _ = U.clean(g)
    assert U.certify(contigs, sums, g, alive)                   # the removed K-mers are still there
    kept = [c for c in contigs if all(alive[i] for i in U.windows(g, [c])[0])]
    assert U.certify(kept, None, g, alive)                      # the survivors' unitigs are longer than these
