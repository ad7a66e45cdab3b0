"""GPU tests of unitig clean-up (Context.unitigs_clean*, assembler.py --clean) against the string restatement
tests/clean_ref.py, the published clean-up table, and the properties a clean-up must have (it only removes, the
result is deterministic, with every rule off it is the plain unitig set)."""
import random

import numpy as np
import pytest

import oracle
from clean_ref import assembly_stats, clean_contigs
from oracle import py_build, twin
from test_cpu_clean import BASE, G as G300, TABLE_100K, _genome, _sub, _tiling, synth_case
from test_gpu_unitig_wide import _canon_set, _kmer_words

pytestmark = pytest.mark.gpu

ENTRIES = ["reads", "ingested", "kmers"]
OFF = dict(tip_len=0, isolated_len=0, bubble_len=0)


def _dict_keys(A, k):
    v = [int(x.translate(str.maketrans("ACGT", "0123")), 4) for x in A]
    lo = np.array([x & 0xFFFFFFFFFFFFFFFF for x in v], np.uint64)
    hi = np.array([x >> 64 for x in v], np.uint64)
    return lo, hi, np.array(list(A.values()), np.uint32)


def _run(ctx, entry, reads, k, limit, **kw):
    """-> (contigs, kmer_sums, stats) of one entry point"""
    if entry == "reads":
        buf, off = oracle.pack_reads(reads)
        return ctx.unitigs_clean(buf, off, k, limit, **kw)
    if entry == "ingested":
        ctx.ingest("".join(">r%d\n%s\n" % (i, r) for i, r in enumerate(reads)).encode(), 1)
        return ctx.unitigs_clean_ingested(k, limit, **kw)
    lo, hi, cnt = _dict_keys(py_build([r.upper() for r in reads], k, limit), k)
    return ctx.unitigs_clean_from_kmers(lo, cnt, k, keys_hi=hi if k > 32 else None, **kw)


def _check_parity(ctx, reads, k, limit, entries=ENTRIES, **kw):
    exp, _, est, A = clean_contigs([r.upper() for r in reads], k, limit, **kw)
    for entry in entries:
        got, sums, st = _run(ctx, entry, reads, k, limit, **kw)
        assert _canon_set(got, k, A) == _canon_set(exp, k, A), (entry, k, limit)
        assert len(sums) == len(got)
        assert [int(s) for s in sums] == [sum(A[c[i:i + k]] for i in range(len(c) - k + 1)) for c in got], (entry, k, limit)
        assert st == est, (entry, k, limit)
    return est


# ---- 1. the hand-built cases of test_cpu_clean, through every entry point -----------------------------------------
def _hand_cases():
    frag = _genome(seed=9, n=30)
    return {
        "tip": (BASE + [_sub(G300[100:200], 95)] * 2, {}),
        "tip_kept": (BASE + [_sub(G300[100:200], 95)] * 2, {"tip_len": 4}),
        "bubble": (BASE + [_sub(G300[100:200], 50)] * 2, {}),
        "haplotypes": (BASE + _tiling(_sub(G300, 150)), {}),
        "isolated": (BASE + [frag, frag], {}),
        "isolated_kept": (BASE + [frag, frag], {"isolated_len": 0}),
        "all_off": (BASE + [_sub(G300[100:200], 95)] * 2 + [_sub(G300[0:100], 50)] * 2 + [frag] * 2, OFF),
    }


@pytest.mark.parametrize("case", sorted(_hand_cases()))
def test_hand_built_cases(ctx, case):
    reads, kw = _hand_cases()[case]
    st = _check_parity(ctx, reads, 21, 1, **kw)
    expect = {"tip": "tips", "bubble": "bubble_branches", "isolated": "isolated"}
    if case in expect:
        assert st[expect[case]] == 1 and st["rounds"] == 1
    else:
        assert st["rounds"] == 0


def test_palindromic_fragment_even_k(ctx):
    x = _genome(seed=3, n=15)
    pal = x + twin(x)
    base = _genome(seed=4, n=200)
    reads = [pal, pal] + [base] * 3
    for k in (20, 16):
        st = _check_parity(ctx, reads, k, 1)
        assert st["isolated"] >= 1


# ---- 2. random read sets with errors, N's, lower case, both strands ----------------------------------------------------
def _error_reads(seed, genome_len, L=100, cov=30, err=0.01, n_frac=0.05, lower=0.2):
    rng = random.Random(seed)
    g = "".join(rng.choice("ACGT") for _ in range(genome_len))
    comp = {"A": "T", "C": "G", "G": "C", "T": "A"}
    reads = []
    for _ in range(genome_len * cov // L):
        s = rng.randrange(0, genome_len - L)
        r = list(g[s:s + L])
        for i in range(L):
            if rng.random() < err:
                r[i] = rng.choice([b for b in "ACGT" if b != r[i]])
        r = "".join(r)
        if rng.random() < 0.5:
            r = "".join(comp[c] for c in reversed(r))
        if rng.random() < n_frac:
            p = rng.randrange(L)
            r = r[:p] + "N" + r[p + 1:]
        if rng.random() < lower:
            r = r.lower()
        reads.append(r)
    return reads


@pytest.mark.parametrize("K", [15, 21, 31, 32, 33, 48, 63])
def test_random_reads_match_restatement(ctx, K):
    removed = 0
    for seed, glen in ((1, 3000), (2, 5000)):
        reads = _error_reads(seed, glen)
        for limit in (0, 1, 2):
            removed += _check_parity(ctx, reads, K, limit)["kmers_removed"]
    assert removed > 0


def test_max_rounds_and_single_rules(ctx):
    reads = _error_reads(7, 4000)
    for kw in ({"max_rounds": 1}, {"max_rounds": 0}, {"tip_len": 0}, {"bubble_len": 0, "isolated_len": 0},
               {"tip_len": 5, "bubble_len": 7, "isolated_len": 3}):
        _check_parity(ctx, reads, 25, 0, **kw)


# ---- 3. no-op cases -------------------------------------------------------------------------------------------------
def test_all_rules_off_equals_unitigs(ctx):
    reads = _error_reads(3, 4000)
    buf, off = oracle.pack_reads(reads)
    for K in (21, 32, 33, 63):
        d = py_build([r.upper() for r in reads], K, 1)
        plain = _canon_set(ctx.unitigs(buf, off, K, 1), K, d)
        got, _, st = ctx.unitigs_clean(buf, off, K, 1, **OFF)
        assert _canon_set(got, K, d) == plain and st["rounds"] == 0 and st["kmers_removed"] == 0
        lo, hi, cnt = _dict_keys(d, K)
        ref = ctx.unitigs_from_kmers(lo, cnt, K, keys_hi=hi if K > 32 else None)
        got, _, _ = ctx.unitigs_clean_from_kmers(lo, cnt, K, keys_hi=hi if K > 32 else None, **OFF)
        assert _canon_set(got, K, d) == _canon_set(ref, K, d) == plain


def _synth(G, err_ppm, L=150, cov=30):
    n = G * cov // L
    return oracle.synth_reads(G, L, err_ppm=err_ppm, first=0, count=n), oracle.fixed_offsets(n, L)


@pytest.mark.parametrize("K", [31, 63])
def test_error_free_500kbp_is_unchanged(ctx, K):
    reads, off = _synth(500_000, 0)
    plain = ctx.unitigs(reads, off, K, 1)
    got, sums, st = ctx.unitigs_clean(reads, off, K, 1)
    assert sorted(min(c, twin(c)) for c in got) == sorted(min(c, twin(c)) for c in plain)
    assert st["kmers_removed"] == 0 and st["rounds"] == 0


# ---- 4. the published table, exactly; only-removes, better, deterministic -----------------------------------------------
TABLE_500K = {
    31: ((10502, 117, 895976, 161928, 999904), (263, 13582, 510524, 5364, 999904), 2),
    63: ((4178, 387, 805406, 94026, 998714), (62, 15894, 503014, 110, 998230), 1),
}


@pytest.mark.parametrize("G,K", [(100_000, 31), (100_000, 63), (500_000, 31), (500_000, 63)])
def test_table_cells(ctx, G, K):
    today, cleaned, rounds = (TABLE_100K if G == 100_000 else TABLE_500K)[K]
    _, gk = synth_case(G, K)
    reads, off = _synth(G, 10000)
    plain = ctx.unitigs(reads, off, K, 1)
    got, sums, st = ctx.unitigs_clean(reads, off, K, 1)
    again, sums2, st2 = ctx.unitigs_clean(reads, off, K, 1)
    assert sorted(got) == sorted(again) and st == st2 and sorted(sums) == sorted(sums2)   # deterministic
    a, b = assembly_stats(plain, K, gk), assembly_stats(got, K, gk)
    # better: the table's cells imply these; asserted one by one so that a failure says what got worse
    assert b[1] > a[1], "N50"
    assert b[0] < a[0], "contigs"
    assert b[3] < a[3], "K-mers off the genome"
    assert a == today
    assert b == cleaned and st["rounds"] == rounds


@pytest.mark.parametrize("K", [31, 63])
def test_cleaned_500kbp_only_removes(ctx, K):
    reads, off = _synth(500_000, 10000)
    got, sums, _ = ctx.unitigs_clean(reads, off, K, 1)
    klo, khi, kv = ctx.count_mers_wide(reads, off, K, 1)
    lo, hi = _kmer_words(got + [twin(c) for c in got], K)
    key = (hi.astype(object) << 64) | lo.astype(object)
    assert len(set(key.tolist())) == len(key)                                  # each K-mer once over both orientations
    table = dict(zip(((khi.astype(object) << 64) | klo.astype(object)).tolist(), kv.tolist()))
    assert all(x in table for x in key.tolist())                                # a subset of the counted K-mers
    lo, hi = _kmer_words(got, K)
    fkey = ((hi.astype(object) << 64) | lo.astype(object)).tolist()
    pos = 0
    for c, s in zip(got, sums):
        w = len(c) - K + 1
        assert int(s) == sum(table[x] for x in fkey[pos:pos + w])
        pos += w


# ---- 5. command line --------------------------------------------------------------------------------------------------
def _fastq(tmp_path, reads):
    fq = tmp_path / "reads.fq"
    fq.write_text("".join("@r%d\n%s\n+\n%s\n" % (i, r, "I" * len(r)) for i, r in enumerate(reads)))
    return fq


@pytest.mark.parametrize("K", [31, 63])
def test_assembler_cli_clean(ctx, tmp_path, K):
    import assembler
    from referenceassembler import referenceAssembler as ram
    reads = _error_reads(5, 5000, err=0.01, n_frac=0, lower=0)
    reads = reads + reads[::3]   # repeated errors survive limit 1
    fq = _fastq(tmp_path, reads)
    out = tmp_path / "c.fa"
    assert assembler.main(["-i", str(fq), "-o", str(out), "-k", str(K), "--clean"]) == 0
    got = [x for x in out.read_text().split("\n") if x and x[0] != ">"]
    ctx.ingest(fq.read_bytes(), 2)
    exp, sums, st = ctx.unitigs_clean_ingested(K, 1)
    assert got == exp and st["kmers_removed"] > 0
    s_lines = [x.split("\t") for x in (tmp_path / "c.fa.gfa").read_text().splitlines() if x.startswith("S\t")]
    assert [x[2] for x in s_lines] == got
    assert [x[4] for x in s_lines] == ["KC:i:%d" % s for s in sums]
    # without --clean: the files of the plain unitig route, no KC tag
    plain = tmp_path / "p.fa"
    assert assembler.main(["-i", str(fq), "-o", str(plain), "-k", str(K)]) == 0
    ref = tmp_path / "r.fa"
    contigs = ctx.unitigs_ingested(K, 1)
    assembler.write_outputs(str(ref), contigs, ram.link_graph(contigs, K), K)
    assert plain.read_bytes() == ref.read_bytes()
    assert (tmp_path / "p.fa.gfa").read_bytes() == (tmp_path / "r.fa.gfa").read_bytes()
    assert b"KC:i:" not in (tmp_path / "p.fa.gfa").read_bytes()


def test_clean_k64_is_refused(ctx, tmp_path):
    import _native as N
    import assembler
    fq = _fastq(tmp_path, ["ACGT" * 40])
    with pytest.raises(N.EulerError, match="out of range"):
        assembler.main(["-i", str(fq), "-o", str(tmp_path / "x.fa"), "-k", "64", "--clean"])
    buf, off = oracle.pack_reads(["ACGT" * 40])
    for K in (1, 64):
        with pytest.raises(N.EulerError, match="out of range"):
            ctx.unitigs_clean(buf, off, K, 0)
