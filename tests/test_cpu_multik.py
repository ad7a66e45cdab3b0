"""The multi-k rule of include/euler_b200.h (euler_unitigs_multik), on the CPU: the two restatements of
tests/multik_ref.py agree, hand-built cases show each clause of the rule, and the 100 kbp table of multi-k against one
K is pinned."""

import pytest

import oracle
import unitig_shapes
from clean_ref import assembly_stats
from multik_ref import arrays, canon_pairs, cyclic_windows, raise_counts, strings
from oracle import py_build, twin
from test_cpu_clean import _genome

LISTS = [[21, 31, 33], [15, 33, 63], [2, 3, 5], [31, 32, 33]]


def _agree(reads, ks, limit, clean):
    buf, off = oracle.pack_reads(reads)
    a = arrays(buf, off, ks, limit, clean)
    s = strings([r.upper() for r in reads], ks, limit, clean)
    assert canon_pairs(a[0], a[1], ks[-1]) == canon_pairs(s[0], s[1], ks[-1]), (ks, limit, clean)
    assert a[2] == s[2], (ks, limit, clean)
    return a


@pytest.mark.parametrize("name", unitig_shapes.SHAPES)
def test_restatements_agree_on_shapes(name):
    added = 0
    for ks in LISTS:
        reads = unitig_shapes.shape(name, ks[0])
        for limit, clean in ((0, True), (1, True), (1, False), (2, False)):
            added += sum(st["nodes_added"] for st in _agree(reads, ks, limit, clean)[2])
    if name == "repeats":
        assert added > 0   # the contigs do bring K-mers in


def test_trace_changes_nothing():
    """arrays(trace=...) returns what it returns without, which is what strings returns; the trace is its steps"""
    reads = unitig_shapes.tandem() + unitig_shapes.inverted() + unitig_shapes.repeats()
    buf, off = oracle.pack_reads(reads)
    for ks in ([20, 32, 48], [21, 31, 33]):
        trace = []
        a = arrays(buf, off, ks, 1, trace=trace)
        assert a == arrays(buf, off, ks, 1)
        s = strings([r.upper() for r in reads], ks, 1)
        assert canon_pairs(a[0], a[1], ks[-1]) == canon_pairs(s[0], s[1], ks[-1]) and a[2] == s[2]
        assert [t["K"] for t in trace] == ks and trace[0]["odd_pal"] == 0
        for t, st in zip(trace, a[2]):
            assert len(t["contigs"]) == len(t["weights"]) == st["contigs"]
            assert sum(len(c) for c, _, _ in t["contigs"]) == st["bases"]
        assert [(c, s) for c, _, s in trace[-1]["contigs"]] == list(zip(a[0], a[1]))
        assert any(cyc for t in trace for _, cyc, _ in t["contigs"])   # the bare tandem arrays are cycles


# ---- hand-built cases ---------------------------------------------------------------------------------------------
def _joint_reads():
    """two reads of a 175 bp genome that overlap by 25 bases, twice each: the 21-mers join them, the 31-mers do not"""
    g = _genome(seed=11, n=175)
    return g, [g[:100], g[75:]] * 2


@pytest.mark.parametrize("clean", [True, False])
def test_small_k_contigs_bridge_a_short_overlap(clean):
    g, reads = _joint_reads()
    one, _, _ = strings(reads, [31], 1, clean)
    assert sorted(min(c, twin(c)) for c in one) == sorted(min(c, twin(c)) for c in (g[:100], g[75:]))
    two, sums, steps = strings(reads, [21, 31], 1, clean)
    assert [min(c, twin(c)) for c in two] == [min(g, twin(g))]
    assert steps[1]["nodes_added"] == 5   # the 31-mers across the joint start at 70..74
    buf, off = oracle.pack_reads(reads)
    a = arrays(buf, off, [21, 31], 1, clean)
    assert canon_pairs(a[0], a[1], 31) == canon_pairs(two, sums, 31) and a[2] == steps


def test_contig_shorter_than_next_k_adds_nothing():
    frag = _genome(seed=12, n=27)   # 7 21-mers, fewer than 31 bases
    assert cyclic_windows(frag, 21, 31, False) == [] and cyclic_windows(frag, 21, 27, False) == [frag]
    for ks in ([21, 31], [21, 28]):
        c, _, steps = strings([frag] * 2, ks, 1, clean=False)
        assert steps[0]["contigs"] == 1 and steps[1]["nodes_added"] == 0 and c == []


def test_palindromic_kmer_gets_an_even_count():
    x = _genome(seed=13, n=10)
    pal = x + twin(x)                     # a palindromic 20-mer
    c = "ACGTTGCAAC" + pal + "GGTACCATTG"
    d = raise_counts({}, [(c, 5, False)], 15, 20)
    assert d[pal] == 6 and all(v == 5 for y, v in d.items() if y != pal)
    d = raise_counts({pal: 8}, [(c, 5, False)], 15, 20)
    assert d[pal] == 8


def test_read_count_at_or_below_limit_is_raised():
    g = _genome(seed=14, n=60)
    d = py_build([g], 21, -1)             # every 21-mer once on each strand: count 1
    raised = raise_counts(dict(d), [(g, 7, False)], 15, 21)
    assert set(raised) == set(d) and set(raised.values()) == {7}
    assert raise_counts({g[:21]: 9}, [(g, 7, False)], 15, 21)[g[:21]] == 9   # the maximum, not a sum


def test_cycle_rotation_does_not_matter():
    unit = _genome(seed=15, n=37)
    Kp, K = 21, 31
    L = len(unit)
    expect = None
    for r in range(L):
        s = unit[r:] + unit[:r]
        text = (s * 3)[:L + Kp - 1]      # a cycle of L Kp-mers as the library writes it, entered at rotation r
        for t in (text, twin(text)):
            d = raise_counts({}, [(t, 4, True)], Kp, K)
            assert len(d) == 2 * L
            expect = expect or d
            assert d == expect
    texts = [((unit[r:] + unit[:r]) * 3)[:L + K - 1] for r in (0, 5)]
    assert canon_pairs(texts[:1], [0], K) == canon_pairs([twin(texts[1])], [0], K)   # the comparison is rotation-free


def test_one_step_is_the_clean_up():
    from clean_ref import clean_contigs
    from test_gpu_clean import _error_reads
    reads = [r.upper() for r in _error_reads(21, 3000)]
    c, s, steps = strings(reads, [25], 1)
    exp, esums, est, _ = clean_contigs(reads, 25, 1)
    assert steps[0]["clean"] == est and steps[0]["nodes_added"] == 0
    assert sum(s) == sum(esums) and steps[0]["bases"] == sum(len(x) for x in c)


# ---- command line: refused before the reads are read -------------------------------------------------------------
def test_assembler_cli_k_list_refusals(tmp_path):
    import assembler
    fa = tmp_path / "reads.fa"
    fa.write_text(">r\n%s\n" % ("ACGT" * 40))
    base = ["-i", str(fa), "-o", str(tmp_path / "x.fa")]
    for extra in (["-k", "31", "--k-list", "21,31"], ["--k-list", "21,31", "--mode", "euler"], ["--k-list", "21,x"],
                  ["--k-list", "31,21"], ["--k-list", "21,21"], ["--k-list", "1,21"], ["--k-list", "21,64"],
                  ["--k-list", ",".join(str(k) for k in range(2, 19))]):
        with pytest.raises(SystemExit) as e:
            assembler.main(base + extra)
        assert e.value.code == 2   # argparse's usage error
    assert not (tmp_path / "x.fa").exists()


# ---- the 100 kbp table: synth_reads genome, 30x, 1 % substitutions, limit 1, default clean-up ---------------------
TABLE_MULTIK_100K = {
    # (read length, K list): (contigs, N50, total bases, K-mers off the genome, genome K-mers kept of 199,876)
    (100, (63,)): (166, 788, 106333, 62, 192020),
    (100, (31, 63)): (2, 77537, 100037, 0, 199826),
    (100, (21, 31, 41, 51, 63)): (1, 99983, 99983, 0, 199842),
    (150, (63,)): (11, 24543, 100497, 30, 199600),
    (150, (31, 63)): (1, 99964, 99964, 0, 199804),
}


def synth(G, L, err_ppm=10000, cov=30):
    n = G * cov // L
    return oracle.synth_reads(G, L, err_ppm=err_ppm, first=0, count=n), oracle.fixed_offsets(n, L)


def genome_kmers(G, K):
    genome = bytes(oracle.synth_reads(G, G, err_ppm=0, first=0, count=1)).decode()
    return {s[i:i + K] for s in (genome, twin(genome)) for i in range(G - K + 1)}


@pytest.mark.parametrize("L,ks", sorted(TABLE_MULTIK_100K))
def test_table_rows_100kbp(L, ks):
    buf, off = synth(100_000, L)
    contigs, _, steps = arrays(buf, off, list(ks), 1)
    assert assembly_stats(contigs, ks[-1], genome_kmers(100_000, ks[-1])) == TABLE_MULTIK_100K[(L, ks)]
    assert [s["K"] for s in steps] == list(ks)
