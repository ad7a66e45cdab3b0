"""GPU tests of unitig mode on two-word (128-bit) keys: K = 33..63 for unitigs, 32..63 for the link graph, up to
64 for counting.  Checkers: the string restatements of the reference CPU assembler (the oracle's py_build and
py_all_contigs, unitig_ref's py_link_graph and py_get_contig; pinned to the unmodified reference by the CPU tests)
and the oracle's 128-bit count (held to py_build at 64 by test_cpu_oracle.py::test_wide_keys_k63)."""
import random

import numpy as np
import pytest

import oracle
from unitig_ref import py_get_contig, py_link_graph

pytestmark = pytest.mark.gpu


# ---- inputs (random with N's, lower case, repeats / palindromes / poly-A, short reads, one long read) --------
def _random_reads(seed, n, genome_len, lens, n_frac):
    rng = random.Random(seed)
    genome = "".join(rng.choice("ACGT") for _ in range(genome_len))
    comp = {"A": "T", "C": "G", "G": "C", "T": "A"}
    reads = []
    for _ in range(n):
        L = rng.choice(lens)
        s = rng.randrange(0, genome_len - L)
        r = genome[s:s + L]
        if rng.random() < 0.5:
            r = "".join(comp[c] for c in reversed(r))
        if rng.random() < n_frac:
            p = rng.randrange(L)
            r = r[:p] + "N" + r[p + 1:]
        if rng.random() < 0.02:
            r = r[:rng.randrange(1, 5)]
        reads.append(r)
    return reads


def _lower_some(reads, seed, frac=0.3):
    rng = random.Random(seed)
    return [r.lower() if rng.random() < frac else r for r in reads]


def _inputs():
    return {
        "rand": _random_reads(11, 300, genome_len=3000, lens=(64, 80, 100, 100, 150), n_frac=0.1),
        "lower": _lower_some(_random_reads(12, 200, genome_len=2500, lens=(70, 100, 150), n_frac=0.05), 3),
        "repeat": ["ACGT" * 40, "A" * 150, "T" * 150, "AC" * 75, "ACGTTGCA" * 20, "TGCAACGT" * 12] * 2,
        "short": ["ACGT" * 8, "ACGTACGTAC", "", "A" * 33, "ACGGTCA" * 9 + "A"],
        "one_long": ["".join("ACGT"[(i * 7 + i // 3 + i // 11) % 4] for i in range(4000))],
    }


INPUTS = ["rand", "lower", "repeat", "short", "one_long"]


def _upper(reads):
    return [r.upper() for r in reads]


# ---- orientation-free, cycle-rotation-free contig sets -------------------------------------------------------
def _min_rotation(s, k):
    nodes = [s[i:i + k] for i in range(len(s) - k + 1)]
    best = None
    for r in range(len(nodes)):
        rot = nodes[r:] + nodes[:r]
        t = rot[0] + "".join(x[-1] for x in rot[1:])
        best = t if best is None or t < best else best
    return best


def _canon_set(contigs, k, d):
    out = []
    for c in contigs:
        nodes = set(c[i:i + k] for i in range(len(c) - k + 1))
        if any(oracle.twin(x) in nodes for x in nodes):
            # a unitig that is its own reverse complement (it runs through palindromic K-mers, so even k only): the
            # reference walks it from a dict-order start and stops before twin(start); the GPU path (at every k)
            # writes it whole.  Both spell the same K-mers up to orientation: compare those.
            out.append("~" + ",".join(sorted({min(x, oracle.twin(x)) for x in nodes})))
            continue
        first, last = c[:k], c[-k:]
        forms = [c, oracle.twin(c)]
        if (last[1:] + first[-1]) == first and first in d:   # an isolated cycle closes on itself
            forms = [_min_rotation(f, k) for f in forms]
        out.append(min(forms))
    return sorted(out)


def _expected_unitigs(reads, k, limit):
    d = oracle.py_build(_upper(reads), k, limit)
    return _canon_set(oracle.py_all_contigs(d, k), k, d), d


# ---- 1. counting ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", INPUTS)
@pytest.mark.parametrize("length", [33, 40, 47, 63, 64])
def test_count_mers_wide_bit_exact(ctx, name, length):
    buf, off = oracle.pack_reads(_inputs()[name])
    lo, hi, vals = oracle.count_mers(buf, off, length)
    for limit in (0, 1):
        glo, ghi, gv = ctx.count_mers_wide(buf, off, length, limit)
        keep = vals > limit
        assert np.array_equal(glo, lo[keep]) and np.array_equal(ghi, hi[keep]) and np.array_equal(gv, vals[keep]), limit


@pytest.mark.parametrize("name", INPUTS)
@pytest.mark.parametrize("k", [33, 64])
def test_build_equals_reference_build(name, k):
    import referenceassembler as ra
    reads = _inputs()[name]
    for limit in (0, 1):
        assert ra.build(reads, k, limit) == oracle.py_build(_upper(reads), k, limit), limit


def test_count_mers_wide_up_to_32_is_count_mers(ctx):
    buf, off = oracle.pack_reads(_inputs()["rand"])
    for length in (1, 17, 31, 32):
        keys, vals = ctx.count_mers(buf, off, length, 1)
        lo, hi, v2 = ctx.count_mers_wide(buf, off, length, 1)
        assert np.array_equal(lo, keys) and np.array_equal(v2, vals) and not hi.any()


# ---- 2. unitigs from reads -----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", INPUTS)
@pytest.mark.parametrize("K", [33, 34, 48, 62, 63])
def test_unitigs_wide_match_reference(ctx, name, K):
    buf, off = oracle.pack_reads(_inputs()[name])
    for limit in (0, 1):
        exp, d = _expected_unitigs(_inputs()[name], K, limit)
        got = ctx.unitigs(buf, off, K, limit)
        assert _canon_set(got, K, d) == exp, limit


# ---- 3. referenceassembler drop-in: all_contigs, link_graph, get_contig ---------------------------------------
@pytest.mark.parametrize("k", [33, 63])
def test_all_contigs_and_get_contig(ctx, k):
    import referenceassembler as ra
    for name in ("rand", "repeat", "one_long"):
        d = oracle.py_build(_upper(_inputs()[name]), k, 1)
        G, r = ra.all_contigs(d, k)
        assert _canon_set(r, k, d) == _canon_set(oracle.py_all_contigs(d, k), k, d), name
        assert G == py_link_graph(r, k)
        for c in r:
            for km in (c[:k], c[(len(c) - k) // 2:(len(c) - k) // 2 + k]):
                assert ra.get_contig(d, km) == py_get_contig(d, km), (name, km)


@pytest.mark.parametrize("k", [32, 33, 50, 63])
def test_link_graph_exact(ctx, k):
    from referenceassembler import referenceAssembler as ram
    contigs = []
    for name in INPUTS:
        contigs += oracle.py_all_contigs(oracle.py_build(_upper(_inputs()[name]), k, 0), k)
    assert len(contigs) >= 10
    # repeated heads and tails: the later contig must win, as in the reference's dicts
    lists = [contigs, contigs + contigs[:5] + [oracle.twin(c) for c in contigs[3:9]] + ["A" * k, "T" * (k + 1)]]
    for lst in lists:
        assert ram.link_graph(lst, k) == py_link_graph(lst, k)


# ---- 4. command line and assemble2 -----------------------------------------------------------------------------
def test_assembler_cli_k63(ctx, tmp_path):
    import assembler
    from referenceassembler import referenceAssembler as ram
    reads = [r for r in _inputs()["rand"] if r]
    fq = tmp_path / "reads.fq"
    fq.write_text("".join("@r%d\n%s\n+\n%s\n" % (i, r, "I" * len(r)) for i, r in enumerate(reads)))
    out = tmp_path / "contigs.fa"
    assert assembler.main(["-i", str(fq), "-o", str(out), "-k", "63"]) == 0
    got = [x for x in out.read_text().split("\n") if x and x[0] != ">"]
    buf, off = oracle.pack_reads(reads)
    d = oracle.py_build(_upper(reads), 63, 1)
    assert got and _canon_set(got, 63, d) == _canon_set(ctx.unitigs(buf, off, 63, 1), 63, d)
    gfa = (tmp_path / "contigs.fa.gfa").read_text().splitlines()
    assert gfa[0] == "H\tVN:Z:1.0"
    assert [x.split("\t")[2] for x in gfa if x.startswith("S\t")] == got
    links = [x.split("\t") for x in gfa if x.startswith("L\t")]
    assert all(x[5] == "62M" for x in links)
    G = ram.link_graph(got, 63)
    exp = [[str(i), "+", str(j), o] for i in G for j, o in G[i][0]] + [[str(i), "-", str(j), o] for i in G for j, o in G[i][1]]
    assert sorted(x[1:5] for x in links) == sorted(exp)


def test_assemble2_k41(ctx, tmp_path):
    import eulercuda.eulercuda as ec
    reads = [r for r in _inputs()["rand"] if r]
    exp, d = _expected_unitigs(reads, 41, 1)
    assert _canon_set(ec.assemble2(41, buffer=reads), 41, d) == exp
    fa = tmp_path / "r.fa"
    fa.write_text("".join(">r%d\n%s\n" % (i, r) for i, r in enumerate(reads)))
    assert _canon_set(ec.assemble2(41, infile=str(fa)), 41, d) == exp


# ---- 5. ranges and errors --------------------------------------------------------------------------------------
def test_ranges_are_refused(ctx):
    import _native as N
    import referenceassembler as ra
    buf, off = oracle.pack_reads(["ACGT" * 40])
    with pytest.raises(N.EulerError):
        ctx.unitigs(buf, off, 64, 0)
    with pytest.raises(N.EulerError):
        ctx.unitig_links(["A" * 70], 64)
    with pytest.raises(N.EulerError):
        ctx.count_mers_wide(buf, off, 65, 0)
    lo, hi, vals = ctx.count_mers_wide(buf, off, 40, 0)
    assert lo.size
    with pytest.raises(N.EulerError):
        ctx.unitigs_from_kmers(lo, vals, 40)
    d = oracle.py_build(["ACGT" * 40], 40, 0)
    assert _canon_set(ctx.unitigs_from_kmers(lo, vals, 40, keys_hi=hi), 40, d) == _canon_set(oracle.py_all_contigs(d, 40), 40, d)
    with pytest.raises(N.EulerError):
        ra.all_contigs(ra.build(["ACGT" * 40], 64, 0), 64)


# ---- 6. size-independent properties at the shape of real reads --------------------------------------------------
def _kmer_words(seqs, k):
    """(lo, hi) of every k-window of every sequence (ACGT only)"""
    code = np.full(256, 255, np.uint8)
    code[np.frombuffer(b"ACGT", np.uint8)] = np.arange(4, dtype=np.uint8)
    wins = [np.lib.stride_tricks.sliding_window_view(code[np.frombuffer(s.encode("ascii"), np.uint8)], k) for s in seqs]
    w = np.concatenate(wins).astype(np.uint64)
    lo = np.zeros(len(w), np.uint64)
    hi = np.zeros(len(w), np.uint64)
    for j in range(k):
        s = 2 * (k - 1 - j)
        if s < 64:
            lo |= w[:, j] << np.uint64(s)
        else:
            hi |= w[:, j] << np.uint64(s - 64)
    return lo, hi


def test_unitigs_k63_partition_the_kept_kmers(ctx):
    G, L, cov, K = 500_000, 150, 30, 63
    nreads = G * cov // L
    reads = oracle.synth_reads(G, L, err_ppm=10000, first=0, count=nreads)
    off = oracle.fixed_offsets(nreads, L)
    contigs = ctx.unitigs(reads, off, K, 1)
    klo, khi, kv = ctx.count_mers_wide(reads, off, K, 1)   # both strands, count > 1, ascending (hi, lo)
    assert contigs and klo.size > 2 * G * 0.9
    lo, hi = _kmer_words(contigs + [oracle.twin(c) for c in contigs], K)
    o = np.lexsort((lo, hi))
    lo, hi = lo[o], hi[o]
    assert lo.size == klo.size                            # every K-mer occurs once over both orientations ...
    assert np.array_equal(lo, klo) and np.array_equal(hi, khi)   # ... and they are exactly the kept K-mers
    # odd K: no palindromes, so the canonical kept K-mers are half of the both-strand ones
    assert sum(len(c) - (K - 1) for c in contigs) == klo.size // 2
