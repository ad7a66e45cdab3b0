"""String restatement of unitig-mode graph clean-up (tips, isolated fragments, bubble branches; the rules of
euler_unitigs_clean in include/euler_b200.h) -- test infrastructure only.  It works on the oracle's py_build dict
(both strands, both-strand counts) and writes the survivors with py_all_contigs."""
from oracle import _fw, py_all_contigs, py_build, twin


def _fwn(x, A):
    return [y for y in _fw(x) if y in A]


def _bwn(x, A):
    return [twin(y) for y in _fwn(twin(x), A)]


def path_unitigs(A):
    """path unitigs on both strands (lists of K-mers) under the link rule of unitig.cu; cycles are left out"""
    succ = {}
    for x in A:
        f = _fwn(x, A)
        if len(f) == 1 and f[0] != twin(x) and len(_bwn(f[0], A)) == 1:
            succ[x] = f[0]
    pred = set(succ.values())
    out = []
    for x in A:
        if x in pred:
            continue
        c = [x]
        while c[-1] in succ:
            c.append(succ[c[-1]])
        out.append(c)
    return out


def cov(c, A):
    return (65536 * sum(A[x] for x in c)) // len(c)


def clean_round(A, tip_len, isolated_len, bubble_len):
    """one round on the snapshot A -> (survivors, tips, isolated, bubble branches); the counts are once per strand
    pair (a tip's twin never qualifies itself; isolated unitigs and bubble branches qualify on both strands)"""
    chains = path_unitigs(A)
    by_head = {c[0]: c for c in chains}
    tips, iso, groups = [], [], {}
    for c in chains:
        h, t, L = c[0], c[-1], len(c)
        ins, outs = _bwn(h, A), _fwn(t, A)
        if not ins and not outs and L <= isolated_len:
            iso.append(c)
        if not outs and len(ins) == 1 and L <= tip_len:
            rivals = [y for y in _fwn(ins[0], A) if y != h]
            if rivals and cov(c, A) < max(cov(by_head[y], A) for y in rivals):
                tips.append(c)
        if len(ins) == 1 and len(outs) == 1 and L <= bubble_len:
            groups.setdefault((ins[0], outs[0]), []).append(c)
    pops = []
    for g in groups.values():
        m = max(cov(c, A) for c in g)
        pops += [c for c in g if cov(c, A) < m]
    dead = set()
    for c in tips + iso + pops:
        dead.update(c)
        dead.update(twin(x) for x in c)
    pairs = lambda cs: len({min(c[0], twin(c[-1])) for c in cs})   # a unitig and its twin once
    return {x: v for x, v in A.items() if x not in dead}, len(tips), pairs(iso), pairs(pops)


def clean(A, k, tip_len=None, isolated_len=None, bubble_len=None, max_rounds=10):
    """-> (surviving dict, stats dict with the fields of euler_clean_stats)"""
    d = lambda v: 2 * k if v is None else v
    tip_len, isolated_len, bubble_len = d(tip_len), d(isolated_len), d(bubble_len)
    st = {"rounds": 0, "tips": 0, "isolated": 0, "bubble_branches": 0, "kmers_removed": 0}
    for _ in range(max_rounds):
        B, nt, ni, nb = clean_round(A, tip_len, isolated_len, bubble_len)
        if len(B) == len(A):
            break
        st["rounds"] += 1
        st["tips"] += nt
        st["isolated"] += ni
        st["bubble_branches"] += nb
        st["kmers_removed"] += len({min(x, twin(x)) for x in A if x not in B})
        A = B
    return A, st


def clean_contigs(reads, k, limit=1, **kw):
    """-> (contigs, kmer_sums, stats, surviving dict) for reads (upper case; 'N' splits)"""
    A, st = clean(py_build(reads, k, limit), k, **kw)
    contigs = py_all_contigs(A, k)
    sums = [sum(A[c[i:i + k]] for i in range(len(c) - k + 1)) for c in contigs]
    return contigs, sums, st, A


def n50(lengths):
    """the first length, going down the lengths in descending order, at which the running sum reaches half the total"""
    lengths = sorted(lengths, reverse=True)
    tot, acc = sum(lengths), 0
    for x in lengths:
        acc += x
        if 2 * acc >= tot:
            return x
    return 0


def assembly_stats(contigs, k, genome_kmers):
    """(contigs, N50, total bases, K-mers off the genome, genome K-mers kept); K-mers over both orientations"""
    kmers = {s[i:i + k] for c in contigs for s in (c, twin(c)) for i in range(len(c) - k + 1)}
    lens = [len(c) for c in contigs]
    on = len(kmers & genome_kmers)
    return len(contigs), n50(lens), sum(lens), len(kmers) - on, on
