"""GPU tests of unitig mode and its clean-up on awkward graph shapes and at genome scale.  Small inputs are compared
with the string restatements (py_all_contigs, py_link_graph, clean_ref) at every K; large ones with
tests/unitig_np.py, whose `certify` proves that the contig text is exactly the set of maximal unitigs of the
surviving K-mers, cut at the right K-mers and with the right count sums."""
import resource

import numpy as np
import pytest

import oracle
import unitig_np as U
import unitig_shapes as S
from clean_ref import clean_contigs
from oracle import py_all_contigs, py_build, twin
from test_gpu_clean import ENTRIES, _check_parity, _dict_keys
from test_gpu_unitig_wide import _canon_set
from unitig_ref import py_link_graph

pytestmark = pytest.mark.gpu

CLEAN_KS = [2, 3, 4, 5, 8, 12, 16, 20, 21, 31, 32, 33, 34, 47, 62, 63]


def _certified(got, sums, g, alive, what):
    fails = U.certify(got, sums, g, alive)
    assert not fails, (what, fails)


# ---- 1. the dictionary entry point refuses counts that are not both-strand counts ------------------------------------
@pytest.mark.parametrize("K", [20, 40])
def test_dictionary_counts_must_be_both_strand(ctx, K):
    import _native as N
    d = py_build(S.inverted() + S.pal_once(), K, 0)
    pal = next(x for x in d if x == twin(x))
    pair = next(x for x in d if x != twin(x) and d[x] > 1)
    lo, hi, cnt = _dict_keys(d, K)
    kh = hi if K > 32 else None
    plain = ctx.unitigs_from_kmers(lo, cnt, K, keys_hi=kh)
    got, _, _ = ctx.unitigs_clean_from_kmers(lo, cnt, K, keys_hi=kh)
    exp, _, _, A = clean_contigs(S.inverted() + S.pal_once(), K, 0)
    assert _canon_set(got, K, A) == _canon_set(exp, K, A)
    keys = list(d)
    for bad in ({pal: d[pal] + 1}, {pair: d[pair] + 2}):
        c2 = cnt.copy()
        for x, v in bad.items():
            c2[keys.index(x)] = v
        with pytest.raises(N.EulerError, match="both-strand"):
            ctx.unitigs_clean_from_kmers(lo, c2, K, keys_hi=kh)
        # plain unitigs depend on presence only: any counts are taken, and give the same contigs
        assert ctx.unitigs_from_kmers(lo, c2, K, keys_hi=kh) == plain
    # a key given on one strand only is fine
    one = np.array([x <= twin(x) for x in keys])
    got1, _, _ = ctx.unitigs_clean_from_kmers(lo[one], cnt[one], K, keys_hi=kh[one] if kh is not None else None)
    assert _canon_set(got1, K, A) == _canon_set(exp, K, A)


# ---- 2. a bubble with 65536 * mean count above 2^32 ------------------------------------------------------------------
@pytest.mark.parametrize("K", [31, 63])
def test_high_coverage_bubble(ctx, K):
    reads = S.hot()
    buf, off = oracle.pack_reads(reads)
    g = U.graph(buf, off, K, 1)
    u = U.Unitigs(g, np.ones(g.n, bool))
    branch = u.is_head & (u.L == K)
    assert sorted(u.cov[branch] > 1 << 32) == [False, False, True, True]   # the strong branch only, on both strands
    alive, est = U.clean(g)
    assert est["bubble_branches"] == 1 and est["kmers_removed"] == K
    for entry in ("reads", "kmers"):
        if entry == "reads":
            got, sums, st = ctx.unitigs_clean(buf, off, K, 1)
        else:
            got, sums, st = ctx.unitigs_clean_from_kmers(g.lo, g.cnt.astype(np.uint32), K, keys_hi=g.hi if K > 32 else None)
        assert st == est, entry
        _certified(got, sums, g, alive, entry)


# ---- 3. shape matrix: every shape, plain unitigs and link graph at every K, the clean-up at CLEAN_KS ------------------
@pytest.mark.parametrize("name", S.SHAPES)
def test_shape_clean_up(ctx, name):
    removed = 0
    for K in CLEAN_KS:
        reads = S.shape(name, K)
        for limit in (0, 1, 2):
            removed += _check_parity(ctx, reads, K, limit)["kmers_removed"]
    assert removed > 0


@pytest.mark.parametrize("name", S.SHAPES)
def test_shape_unitigs_and_links(ctx, name):
    from referenceassembler import referenceAssembler as ram
    for K in range(2, 64):
        reads = S.shape(name, K)
        buf, off = oracle.pack_reads(reads)
        for limit in (0, 1, 2):
            d = py_build([r.upper() for r in reads], K, limit)
            got = ctx.unitigs(buf, off, K, limit)
            assert _canon_set(got, K, d) == _canon_set(py_all_contigs(d, K), K, d), (K, limit)
            g = U.from_reads(reads, K, limit)
            _certified(got, None, g, np.ones(g.n, bool), (K, limit))
            if not got:
                continue
            assert ram.link_graph(got, K) == py_link_graph(got, K), (K, limit)
            lst = got + got[:3] + [twin(c) for c in got[1:4]] + ["A" * K, "T" * (K + 1)]   # repeated heads and tails
            assert ram.link_graph(lst, K) == py_link_graph(lst, K), (K, limit)


# ---- 4. genome scale, exact -----------------------------------------------------------------------------------------
def _fasta(buf, off):
    L = int(off[1] - off[0])
    rows = np.empty((off.size - 1, L + 3), np.uint8)
    rows[:, 0], rows[:, 1], rows[:, 2:L + 2], rows[:, L + 2] = ord(">"), ord("\n"), buf.reshape(-1, L), ord("\n")
    return rows.tobytes()


def _scale_check(ctx, buf, off, K, entries):
    """plain unitigs and the clean-up (through `entries`; from reads twice) certified against unitig_np -> (plain
    contigs, cleaned contigs, stats)"""
    g = U.graph(buf, off, K, 1)
    plain = ctx.unitigs(buf, off, K, 1)
    _certified(plain, None, g, np.ones(g.n, bool), "plain")
    alive, est = U.clean(g)
    assert est["kmers_removed"] > 0
    for entry in entries:
        if entry == "reads":
            got, sums, st = ctx.unitigs_clean(buf, off, K, 1)
            # a second call gives the same contigs, sums and stats; the text order follows the count table's slot
            # layout, which concurrent inserts may change from call to call
            again, sums2, st2 = ctx.unitigs_clean(buf, off, K, 1)
            assert st2 == est
            _certified(again, sums2, g, alive, "reads, second call")
        elif entry == "ingested":
            ctx.ingest(_fasta(buf, off), 1)
            got, sums, st = ctx.unitigs_clean_ingested(K, 1)
        else:
            got, sums, st = ctx.unitigs_clean_from_kmers(g.lo, g.cnt.astype(np.uint32), K, keys_hi=g.hi if K > 32 else None)
        assert st == est, entry
        _certified(got, sums, g, alive, entry)
    return plain, got, est


@pytest.mark.parametrize("K", [21, 31, 32, 33, 63])
def test_500kbp_exact(ctx, K):
    G, L = 500_000, 150
    n = G * 30 // L
    buf, off = oracle.synth_reads(G, L, err_ppm=10000, first=0, count=n), oracle.fixed_offsets(n, L)
    _scale_check(ctx, buf, off, K, ENTRIES if K in (31, 63) else ["reads"])


@pytest.mark.parametrize("K", [31, 63])
def test_repeat_rich_1mbp_exact(ctx, K):
    genome = S.repeat_genome(201, 1_000_000, n_families=20, elem_len=(300, 3000), copies=(2, 50))
    buf, off = S.sample_reads_np(202, genome, 150, 30, 0.01)
    _, _, st = _scale_check(ctx, buf, off, K, ["reads"])
    assert st["tips"] and st["bubble_branches"]


# the README's clean-up row: configs[1] shape with 1 % errors, limit 1 -> (contigs, N50) before and after
README_ROW = {
    (100, 31): ((78514, 166), (791, 50102)), (100, 63): ((33198, 381), (8017, 763)),
    (150, 31): ((94094, 122), (2389, 16397)), (150, 63): ((37835, 401), (591, 14893)),
}


@pytest.mark.parametrize("L,K", sorted(README_ROW))
def test_configs1_clean_row(ctx, L, K):
    from clean_ref import n50
    G = 4_600_000
    n = G * 30 // L
    buf, off = oracle.synth_reads(G, L, err_ppm=10000, first=0, count=n), oracle.fixed_offsets(n, L)
    plain, cleaned, st = _scale_check(ctx, buf, off, K, ["ingested"])
    assert st["rounds"] == 2
    # both lists are certified, so these are the restatement's numbers too
    before = (len(plain), n50([len(c) for c in plain]))
    after = (len(cleaned), n50([len(c) for c in cleaned]))
    print("configs[1] L=%d K=%d: %s -> %s, peak host RSS %.1f GB" %
          (L, K, before, after, resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2**20))
    assert (before, after) == README_ROW[(L, K)]
