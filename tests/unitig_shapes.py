"""Seeded read sets that give unitig graphs their awkward shapes: tandem arrays (K-mer self-loops, self-twin
cycles), inverted repeats (palindromic K-mers, hairpin stops), repeat families with errors (tips and bubbles next to
repeat branch nodes), palindromes seen once, dense short-K graphs, short and malformed reads, and a bubble whose
coverage exceeds 2^32 / 65536 -- test inputs only."""
import random

from oracle import twin

SUB = {"A": "CGT", "C": "AGT", "G": "ACT", "T": "ACG"}


def _rand(rng, n):
    return "".join(rng.choice("ACGT") for _ in range(n))


def _mutate(rng, s, err):
    return "".join(rng.choice(SUB[c]) if rng.random() < err else c for c in s)


def tandem():
    """tandem arrays of period 1, 2, 3, 4, 6 and 8, bare (cycles: poly-A is its own successor, ACGT^n a self-twin
    4-cycle) and, of other units, between random flanks"""
    rng = random.Random(101)
    reads = []
    for unit in ("A", "AG", "ACG", "ACGT", "AACCGT", "ACGTTGCA"):
        arr = unit * (72 // len(unit))
        reads += [arr, arr]
    for unit in ("C", "CA", "GAT", "AATC", "ACCGTA", "AGGTCCAT"):
        for _ in range(2):
            flanked = _rand(rng, 30) + unit * (48 // len(unit)) + _rand(rng, 30)
            reads += [flanked, twin(flanked)]
    reads.append("T" * 90)
    return reads


def inverted():
    """x + spacer + twin(x): spacer 0 makes palindromic K-mers (even K), 1..3 hairpin stops; bare and flanked"""
    rng = random.Random(102)
    reads = []
    for sp in (0, 1, 2, 3):
        for n in (12, 35):
            x = _rand(rng, n)
            ir = x + _rand(rng, sp) + twin(x)
            reads += [ir, ir, _rand(rng, 25) + ir + _rand(rng, 25)] * 2
    return reads


def repeat_genome(seed, genome_len, n_families, elem_len, copies, tandem_unit=7, tandem_copies=40, tandems=(),
                  inverted=0, inverted_len=(20, 60)):
    """a random genome carrying repeat families: per family an element of elem_len = (lo, hi) bases, inserted
    copies = (lo, hi) times, a third of the copies reverse-complemented and a third with 1..3 substitutions; plus one
    tandem array.  Optional extras, drawn after all of that so that callers without them keep their genome: tandems,
    one array per (unit length, (lo, hi) copies); and `inverted` inverted repeats x + twin(x), |x| in inverted_len
    (palindromic K-mers at even K, hairpins at odd K)"""
    rng = random.Random(seed)
    g = list(_rand(rng, genome_len))
    for _ in range(n_families):
        e = _rand(rng, rng.randint(*elem_len))
        for _ in range(rng.randint(*copies)):
            c = e if rng.random() < 0.66 else twin(e)
            if rng.random() < 0.33:
                c = list(c)
                for _ in range(rng.randint(1, 3)):
                    p = rng.randrange(len(c))
                    c[p] = rng.choice(SUB[c[p]])
                c = "".join(c)
            p = rng.randrange(0, genome_len - len(c))
            g[p:p + len(c)] = c
    unit = _rand(rng, tandem_unit)
    p = rng.randrange(0, genome_len - tandem_unit * tandem_copies)
    g[p:p + tandem_unit * tandem_copies] = unit * tandem_copies
    for n, cp in tandems:
        arr = _rand(rng, n) * rng.randint(*cp)
        p = rng.randrange(0, genome_len - len(arr))
        g[p:p + len(arr)] = arr
    for _ in range(inverted):
        x = _rand(rng, rng.randint(*inverted_len))
        p = rng.randrange(0, genome_len - 2 * len(x))
        g[p:p + 2 * len(x)] = x + twin(x)
    return "".join(g)


def sample_reads(seed, genome, L, cov, err):
    """cov-fold reads of L bases from both strands with err substitutions per base"""
    rng = random.Random(seed)
    reads = []
    for _ in range(len(genome) * cov // L):
        s = rng.randrange(0, len(genome) - L + 1)
        r = _mutate(rng, genome[s:s + L], err)
        reads.append(r if rng.random() < 0.5 else twin(r))
    return reads


def repeats(seed=103, genome_len=2500, n_families=3, elem_len=(60, 300), copies=(2, 6), L=80, cov=12, err=0.01):
    """reads with 1 % errors of a repeat-rich genome (small by default; the GPU suite also runs it at 1 Mbp)"""
    g = repeat_genome(seed, genome_len, n_families, elem_len, copies)
    return sample_reads(seed + 1, g, L, cov, err)


def pal_once():
    """x + twin(x) for |x| = 1..24, each read once: the palindromic K-mers in the middle have both-strand count 2"""
    rng = random.Random(104)
    return [x + twin(x) for x in (_rand(rng, n) for n in range(1, 25))] + [_rand(rng, 60)]


def dense():
    """random short reads: at K = 2..8 almost every K-mer is present"""
    rng = random.Random(105)
    return [_rand(rng, rng.randint(20, 60)) for _ in range(120)]


def awkward(K):
    """reads shorter than K, empty reads, runs of exactly K bases between N's, lower case, poly-T (at K = 32 its
    forward key is the all-ones word)"""
    rng = random.Random(106 + K)
    runs = "N".join(_rand(rng, K) for _ in range(6))
    base = _rand(rng, 3 * K + 20)
    return ["", _rand(rng, K - 1), "", runs, runs, "N" + runs.lower() + "N", base, base.lower(), base[K:].lower(),
            "T" * (K + 3), "T" * (K + 3), "t" * K, "N" * K, base[:K]]


SHAPES = ["tandem", "inverted", "repeats", "pal_once", "dense", "awkward"]


def shape(name, K):
    return awkward(K) if name == "awkward" else globals()[name]()


def hot(copies=(70_000, 65_000), L=200, seed=107):
    """one read and a variant with one substitution in its middle, `copies` times each: a bubble of K-mers with
    count 70,000 against 65,000, so 65536 * mean count exceeds 2^32 on the stronger branch only"""
    rng = random.Random(seed)
    r = _rand(rng, L)
    v = r[:L // 2] + SUB[r[L // 2]][0] + r[L // 2 + 1:]
    return [r] * copies[0] + [v] * copies[1]


def sample_reads_np(seed, genome, L, cov, err):
    """sample_reads for genome-sized inputs, vectorised: (buf, off) as oracle.pack_reads returns them"""
    import numpy as np
    rng = np.random.default_rng(seed)
    code = np.frombuffer(b"ACGT", np.uint8)
    g = np.frombuffer(genome.encode("ascii"), np.uint8)
    idx = np.zeros(256, np.uint8)
    idx[code] = np.arange(4, dtype=np.uint8)
    n = len(genome) * cov // L
    starts = rng.integers(0, len(genome) - L + 1, n)
    r = idx[g[starts[:, None] + np.arange(L)]]
    hit = rng.random(r.shape) < err
    r = np.where(hit, (r + rng.integers(1, 4, r.shape)) % 4, r).astype(np.uint8)
    rc = rng.random(n) < 0.5
    r[rc] = 3 - r[rc, ::-1]
    return code[r].ravel(), np.arange(n + 1, dtype=np.uint64) * np.uint64(L)
