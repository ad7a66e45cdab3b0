"""CPU tests of the string restatement of unitig clean-up (tests/clean_ref.py): hand-built reads whose answers are
known, and the 100 kbp rows of the published clean-up table (oracle.synth_reads, 150 bp, 30x, 1 % errors)."""
import random

import pytest

import oracle
from clean_ref import assembly_stats, clean, clean_contigs, path_unitigs
from oracle import py_all_contigs, py_build, twin

K = 21
ZERO = {"rounds": 0, "tips": 0, "isolated": 0, "bubble_branches": 0, "kmers_removed": 0}


def _genome(seed=5, n=300):
    rng = random.Random(seed)
    return "".join(rng.choice("ACGT") for _ in range(n))


def _tiling(g, n=30, L=100):
    return [g[s:s + L] for s in (round(i * (len(g) - L) / (n - 1)) for i in range(n))]


def _sub(s, i):
    return s[:i] + {"A": "C", "C": "G", "G": "T", "T": "A"}[s[i]] + s[i + 1:]


def _canon(contigs):
    return sorted(min(c, twin(c)) for c in contigs)


G = _genome()
BASE = _tiling(G)


def _clean_reads_output():
    return _canon(py_all_contigs(py_build(BASE, K, 1), K))


def test_error_free_tiling_is_one_contig_and_nothing_is_removed():
    contigs, sums, st, A = clean_contigs(BASE, K)
    assert len(contigs) == 1 and (contigs[0] in G or twin(contigs[0]) in G)
    assert st == ZERO
    assert sums == [sum(A[c[i:i + K]] for i in range(len(c) - K + 1)) for c in contigs]


def test_tip_is_clipped():
    err = _sub(G[100:200], 95)   # 5 bases from the read's end: a branch of 5 K-mers, seen twice
    reads = BASE + [err, err]
    assert len(py_all_contigs(py_build(reads, K, 1), K)) == 3
    contigs, _, st, _ = clean_contigs(reads, K)
    assert _canon(contigs) == _clean_reads_output()
    assert st == {"rounds": 1, "tips": 1, "isolated": 0, "bubble_branches": 0, "kmers_removed": 5}


def test_tip_longer_than_tip_len_stays():
    err = _sub(G[100:200], 95)
    reads = BASE + [err, err]
    contigs, _, st, _ = clean_contigs(reads, K, tip_len=4)
    assert _canon(contigs) == _canon(py_all_contigs(py_build(reads, K, 1), K))
    assert st == ZERO


def test_bubble_branch_is_popped():
    err = _sub(G[100:200], 50)   # mid-read: a branch of K K-mers from the genome back to it
    reads = BASE + [err, err]
    assert len(py_all_contigs(py_build(reads, K, 1), K)) == 4
    contigs, _, st, _ = clean_contigs(reads, K)
    assert _canon(contigs) == _clean_reads_output()
    assert st == {"rounds": 1, "tips": 0, "isolated": 0, "bubble_branches": 1, "kmers_removed": K}


def test_equal_haplotypes_keep_both_branches():
    h2 = _sub(G, 150)
    reads = BASE + _tiling(h2)
    before = _canon(py_all_contigs(py_build(reads, K, 1), K))
    assert len(before) == 4
    contigs, _, st, _ = clean_contigs(reads, K)
    assert _canon(contigs) == before and st == ZERO


def test_isolated_fragment():
    frag = _genome(seed=9, n=30)
    reads = BASE + [frag, frag]
    contigs, _, st, _ = clean_contigs(reads, K)
    assert _canon(contigs) == _clean_reads_output()
    assert st == {"rounds": 1, "tips": 0, "isolated": 1, "bubble_branches": 0, "kmers_removed": 30 - K + 1}
    contigs, _, st, _ = clean_contigs(reads, K, isolated_len=0)
    assert _canon(contigs) == _canon(py_all_contigs(py_build(reads, K, 1), K)) and st == ZERO


def test_all_rules_off_is_the_plain_unitigs():
    reads = BASE + [_sub(G[100:200], 95)] * 2 + [_sub(G[0:100], 50)] * 2 + [_genome(seed=9, n=30)] * 2
    d = py_build(reads, K, 1)
    contigs, _, st, A = clean_contigs(reads, K, tip_len=0, isolated_len=0, bubble_len=0)
    assert A == d and st == ZERO
    assert contigs == py_all_contigs(d, K)


def test_palindromic_fragment_even_k():
    k = 20
    x = _genome(seed=3, n=15)
    pal = x + twin(x)            # its own reverse complement: one self-twin unitig through a palindromic K-mer
    d = py_build([pal, pal], k, 1)
    assert any(y == twin(y) for y in d)
    chains = path_unitigs(d)
    assert len(chains) == 1 and len(chains[0]) == 11
    A, st = clean(d, k)
    assert A == {}
    assert st == {"rounds": 1, "tips": 0, "isolated": 1, "bubble_branches": 0, "kmers_removed": 6}
    A, st = clean(d, k, isolated_len=10)
    assert A == d and st == ZERO


# ---- the 100 kbp rows of the table: synth_reads, 150 bp, 30x, 1 % substitutions, limit 1 ---------------------------
TABLE_100K = {
    # K: (today, cleaned), each (contigs, N50, total bases, K-mers off the genome, genome K-mers kept), rounds
    31: ((1999, 121, 175545, 31282, 199868), (61, 11707, 102381, 1234, 199868), 2),
    63: ((828, 395, 160557, 18806, 199636), (11, 24543, 100497, 30, 199600), 1),
}


def synth_case(G, K, err_ppm=10000, L=150, cov=30):
    """(reads, genome K-mers of both strands) of the table's data sets"""
    n = G * cov // L
    r = bytes(oracle.synth_reads(G, L, err_ppm=err_ppm, first=0, count=n)).decode()
    reads = [r[i * L:(i + 1) * L] for i in range(n)]
    genome = bytes(oracle.synth_reads(G, G, err_ppm=0, first=0, count=1)).decode()
    gk = {s[i:i + K] for s in (genome, twin(genome)) for i in range(G - K + 1)}
    return reads, gk


@pytest.mark.parametrize("k", [31, 63])
def test_table_rows_100kbp(k):
    reads, gk = synth_case(100_000, k)
    today, cleaned, rounds = TABLE_100K[k]
    d = py_build(reads, k, 1)
    assert assembly_stats(py_all_contigs(d, k), k, gk) == today
    A, st = clean(d, k)
    assert st["rounds"] == rounds
    assert assembly_stats(py_all_contigs(A, k), k, gk) == cleaned
