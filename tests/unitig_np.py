"""Vectorised restatement of the unitig link rule and the clean-up rules of include/euler_b200.h (euler_unitigs,
euler_unitigs_clean), plus `certify`, an exact check that a contig list spells the maximal unitigs of a node set --
test infrastructure only.  It uses the oracle's count and numpy, nothing of the library it checks, and is fast
enough for genome-sized inputs.

Nodes are the both-strand K-mers of oracle.count_mers(buf, off, K) with count > limit, in its ascending key order;
a node id is an index into that table.  Absent neighbours are -1."""
import numpy as np

import oracle

M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _rev2(x):
    """reverse the order of the 32 two-bit groups of every u64"""
    x = ((x >> np.uint64(2)) & np.uint64(0x3333333333333333)) | ((x & np.uint64(0x3333333333333333)) << np.uint64(2))
    x = ((x >> np.uint64(4)) & np.uint64(0x0F0F0F0F0F0F0F0F)) | ((x & np.uint64(0x0F0F0F0F0F0F0F0F)) << np.uint64(4))
    return x.byteswap()


class Graph:
    """The node graph of K-mers (lo, hi words) with both-strand counts cnt: nbr[n, 4] (forward extension by
    A, C, G, T), twin[n], cnt[n]"""

    def __init__(self, K, lo, hi, cnt):
        self.K = K
        self.lo = np.ascontiguousarray(lo, np.uint64)
        self.hi = np.ascontiguousarray(hi, np.uint64)
        self.cnt = np.asarray(cnt, np.int64)
        self.n = n = self.lo.size
        self.mlo = M64 if K >= 32 else np.uint64((1 << (2 * K)) - 1)
        self.mhi = np.uint64((1 << max(2 * K - 64, 0)) - 1)
        self.keys = self._pack(self.lo, self.hi)
        if n > 1:
            up = (self.hi[1:] > self.hi[:-1]) | ((self.hi[1:] == self.hi[:-1]) & (self.lo[1:] > self.lo[:-1]))
            assert up.all(), "keys must be ascending and distinct"
        self.twin = self.find(*self.revcomp(self.lo, self.hi))
        assert (self.twin >= 0).all(), "the table must hold both strands"
        self.nbr = np.stack([self.find(*self.extend(self.lo, self.hi, b)) for b in range(4)], axis=1)

    def _pack(self, lo, hi):
        if self.K <= 32:
            return lo
        a = np.empty((lo.size, 2), ">u8")
        a[:, 0], a[:, 1] = hi, lo
        return a.view("V16").ravel()

    def revcomp(self, lo, hi):
        """(lo, hi) of the reverse complements"""
        s = 128 - 2 * self.K
        rhi, rlo = _rev2(~lo), _rev2(~hi)    # the complemented 128-bit value, reversed; then drop the low s bits
        if s >= 64:
            return rhi >> np.uint64(s - 64), np.zeros_like(lo)
        return (rlo >> np.uint64(s)) | (rhi << np.uint64(64 - s)), rhi >> np.uint64(s)

    def extend(self, lo, hi, b):
        """(lo, hi) of km[1:] + 'ACGT'[b]"""
        nhi = ((hi << np.uint64(2)) | (lo >> np.uint64(62))) & self.mhi
        return ((lo << np.uint64(2)) | np.uint64(b)) & self.mlo, nhi

    def find(self, lo, hi):
        """node ids of the K-mers (lo, hi), -1 where absent"""
        q = self._pack(np.asarray(lo, np.uint64), np.asarray(hi, np.uint64))
        if not self.n:
            return np.full(q.size, -1, np.int64)
        i = np.searchsorted(self.keys, q)
        j = np.minimum(i, self.n - 1)
        return np.where((i < self.n) & (self.keys[j] == q), j, -1).astype(np.int64)

    def text(self, i):
        return oracle.decode_key(self.lo[i], self.hi[i], self.K)


def graph(buf, off, K, limit):
    """the node graph of euler_unitigs(buf, off, K, limit)"""
    lo, hi, cnt = oracle.count_mers(buf, off, K)
    keep = cnt > limit
    return Graph(K, lo[keep], hi[keep], cnt[keep])


def from_reads(reads, K, limit):
    return graph(*oracle.pack_reads(reads), K, limit)


# ---- link rule and chains ---------------------------------------------------------------------------------------
def _alive_fw(g, alive):
    """(alive forward degree, the last alive forward extension or -1) of every node"""
    ok = (g.nbr >= 0) & alive[np.maximum(g.nbr, 0)]
    one = np.full(g.n, -1, np.int64)
    for b in range(4):
        one = np.where(ok[:, b], g.nbr[:, b], one)
    return ok.sum(axis=1), one


def links(g, alive):
    """succ[x] = y iff y is x's only alive forward extension, y != twin(x), and x is y's only alive backward
    extension (the alive forward degree of twin(y) is 1); else -1.  Dead nodes have none."""
    deg, one = _alive_fw(g, alive)
    y = np.maximum(one, 0)
    ok = alive & (deg == 1) & (one != g.twin) & (deg[g.twin[y]] == 1)
    return np.where(ok, one, -1)


def chains(succ, alive):
    """(head, dist, cycle): per alive node the head of its path and its distance from it; cycle marks the nodes
    whose chain never reaches a head (their head and dist are meaningless)"""
    n = succ.size
    pred = np.full(n, -1, np.int64)
    src = np.nonzero(succ >= 0)[0]
    pred[succ[src]] = src
    P = np.where(pred >= 0, pred, np.arange(n))
    D = (pred >= 0).astype(np.int64)
    for _ in range(max(int(n).bit_length(), 1) + 1):
        D = D + D[P]
        P = P[P]
    cycle = alive & (pred[P] >= 0)
    return P, D, cycle


class Unitigs:
    """the path unitigs of one alive set: per head h (indexed by node id) L, sum, cov, tail, in and out"""

    def __init__(self, g, alive):
        self.succ = links(g, alive)
        head, dist, cycle = chains(self.succ, alive)
        self.head, self.cycle = head, cycle
        path = alive & ~cycle
        self.is_head = path & (head == np.arange(g.n))
        tails = np.nonzero(path & (self.succ < 0))[0]
        self.tail = np.full(g.n, -1, np.int64)
        self.tail[head[tails]] = tails
        self.L = np.zeros(g.n, np.int64)
        self.L[head[tails]] = dist[tails] + 1
        nodes = np.nonzero(path)[0]
        self.sum = np.zeros(g.n, np.int64)
        np.add.at(self.sum, head[nodes], g.cnt[nodes])
        assert self.sum.max(initial=0) < 1 << 46   # 65536 * sum stays exact in int64
        self.cov = np.where(self.is_head, (self.sum << 16) // np.maximum(self.L, 1), 0)
        deg, one = _alive_fw(g, alive)
        t = np.maximum(self.tail, 0)
        self.din = np.where(self.is_head, deg[g.twin], 0)
        self.P = np.where(self.is_head & (self.din == 1), g.twin[np.maximum(one[g.twin], 0)], -1)
        self.dout = np.where(self.is_head, deg[t], 0)
        self.S = np.where(self.is_head & (self.dout == 1), one[t], -1)
        self.deg, self.one = deg, one


def _rival_max(g, alive, u, heads, rival_ok):
    """per head h of `heads`: (max cov of the alive successors r != h of P(h) with rival_ok[r], whether any)"""
    P = u.P[heads]
    m = np.zeros(heads.size, np.int64)
    anyr = np.zeros(heads.size, bool)
    for b in range(4):
        r = g.nbr[P, b]
        rr = np.maximum(r, 0)
        ok = (r >= 0) & alive[rr] & (r != heads) & rival_ok(rr, heads)
        anyr |= ok
        m = np.where(ok, np.maximum(m, u.cov[rr]), m)
    return m, anyr


def clean_round(g, alive, tip_len, isolated_len, bubble_len):
    """one round on the snapshot `alive` -> (new alive, tips, isolated, bubble branches, canonical K-mers removed);
    counted as euler_clean_stats counts them (a tip once, isolated unitigs and bubble branches once per strand pair)"""
    u = Unitigs(g, alive)
    h = np.nonzero(u.is_head)[0]
    L, din, dout = u.L[h], u.din[h], u.dout[h]
    iso = h[(din == 0) & (dout == 0) & (L <= isolated_len)]
    tc = h[(din == 1) & (dout == 0) & (L <= tip_len)]
    m, anyr = _rival_max(g, alive, u, tc, lambda r, hh: np.ones(r.size, bool))
    tips = tc[anyr & (u.cov[tc] < m)]
    cand = np.zeros(g.n, bool)
    cand[h[(din == 1) & (dout == 1) & (L <= bubble_len)]] = True
    bc = np.nonzero(cand)[0]
    m, anyr = _rival_max(g, alive, u, bc, lambda r, hh: cand[r] & (u.S[r] == u.S[hh]))
    pops = bc[anyr & (u.cov[bc] < m)]
    rm = np.zeros(g.n, bool)
    rm[np.concatenate([tips, iso, pops])] = True
    nodes = np.nonzero(alive & ~u.cycle & rm[u.head])[0]
    dead = np.zeros(g.n, bool)
    dead[nodes] = True
    dead[g.twin[nodes]] = True
    pairs = lambda hs: np.unique(np.minimum(hs, g.twin[u.tail[hs]])).size
    gone = np.nonzero(dead)[0]
    return alive & ~dead, tips.size, pairs(iso), pairs(pops), int((gone <= g.twin[gone]).sum())


def clean(g, tip_len=None, isolated_len=None, bubble_len=None, max_rounds=10):
    """-> (alive mask of the survivors, stats dict with the fields of euler_clean_stats)"""
    d = lambda v: 2 * g.K if v is None else v
    alive = np.ones(g.n, bool)
    st = {"rounds": 0, "tips": 0, "isolated": 0, "bubble_branches": 0, "kmers_removed": 0}
    for _ in range(max_rounds):
        nxt, nt, ni, nb, nk = clean_round(g, alive, d(tip_len), d(isolated_len), d(bubble_len))
        if nk == 0:
            break
        st["rounds"] += 1
        st["tips"] += nt
        st["isolated"] += ni
        st["bubble_branches"] += nb
        st["kmers_removed"] += nk
        alive = nxt
    return alive, st


def path_chains(g, alive):
    """the path unitigs as lists of node ids (both strands), and the cycles as sets of node ids"""
    u = Unitigs(g, alive)
    out = []
    for h in np.nonzero(u.is_head)[0]:
        c = [int(h)]
        while u.succ[c[-1]] >= 0:
            c.append(int(u.succ[c[-1]]))
        out.append(c)
    cyc, seen = [], set()
    for x in np.nonzero(u.cycle)[0]:
        if int(x) in seen:
            continue
        c = [int(x)]
        while int(u.succ[c[-1]]) != c[0]:
            c.append(int(u.succ[c[-1]]))
        seen.update(c)
        cyc.append(c)
    return out, cyc


# ---- certify -----------------------------------------------------------------------------------------------------
_CODE = np.full(256, 255, np.uint8)
_CODE[np.frombuffer(b"ACGT", np.uint8)] = np.arange(4, dtype=np.uint8)


def windows(g, contigs):
    """(node id of every K-window of every contig, -1 where it is not a node; contig index of each window; number
    of windows per contig).  A contig with a non-ACGT character has its windows at -2."""
    K = g.K
    lens = np.array([len(c) for c in contigs], np.int64)
    nw = np.maximum(lens - K + 1, 0)
    owner = np.repeat(np.arange(len(contigs)), nw)
    if not nw.sum():
        return np.zeros(0, np.int64), owner, nw
    text = np.frombuffer("".join(contigs).encode("ascii"), np.uint8)
    code = _CODE[text]
    starts = np.repeat(np.cumsum(lens) - lens, nw) + (np.arange(nw.sum()) - np.repeat(np.cumsum(nw) - nw, nw))
    bad = np.zeros(len(contigs), bool)
    if (code == 255).any():
        bad[np.searchsorted(np.cumsum(lens), np.nonzero(code == 255)[0], side="right")] = True
    c64 = np.minimum(code, 3).astype(np.uint64)
    lo = np.zeros(starts.size, np.uint64)
    hi = np.zeros(starts.size, np.uint64)
    for j in range(K):
        hi = (hi << np.uint64(2)) | (lo >> np.uint64(62))
        lo = (lo << np.uint64(2)) | c64[starts + j]
    ids = g.find(lo, hi)
    ids[bad[owner]] = -2
    return ids, owner, nw


def certify(contigs, sums, g, alive, succ=None, examples=3):
    """[] iff `contigs` (with per-contig count sums `sums`, or None) spell the maximal unitigs of the alive node set
    exactly once up to orientation and cycle rotation; else one line per failed check with a few example contigs:
      a. every window of every contig is an alive node;
      b. every alive node appears once over the windows of the contigs and their twins; a contig that holds x and
         twin(x) (self-twin) holds each of its nodes once, and they appear twice, both times in it;
      c. consecutive windows w, w' have succ[w] == w';
      d. the first window has no predecessor and the last no successor, unless succ[last] == first (a cycle);
      e. sums[i] is the sum of the counts of contig i's windows."""
    if succ is None:
        succ = links(g, alive)
    fails = []

    def fail(what, idx):
        idx = sorted(set(int(i) for i in idx))
        ex = ["#%d %s" % (i, contigs[i] if len(contigs[i]) <= 80 else contigs[i][:77] + "...") for i in idx[:examples]]
        fails.append("%s: %d contigs, e.g. %s" % (what, len(idx), "; ".join(ex)))

    ids, owner, nw = windows(g, contigs)
    if (nw == 0).any():
        fail("shorter than K", np.nonzero(nw == 0)[0])
    ok = ids >= 0
    ok[ok] = alive[ids[ok]]
    if not ok.all():
        fail("a. window is not an alive node", owner[~ok])
        return fails   # the other checks index by node id
    first = np.cumsum(nw) - nw
    last = first + nw - 1
    has = nw > 0
    # b: per contig, whether it holds a node and its twin; occurrences over contigs and twins
    cnt = np.bincount(ids, minlength=g.n) + np.bincount(g.twin[ids], minlength=g.n)
    where = np.full(g.n, -1, np.int64)
    where[ids] = owner
    self_twin = np.zeros(len(contigs), bool)
    self_twin[owner[where[g.twin[ids]] == owner]] = True
    rep = np.bincount(ids, minlength=g.n)[ids] > 1
    if rep.any():
        fail("b. node written more than once", owner[rep])
    expect = np.where(self_twin[owner], 2, 1)
    wrong = cnt[ids] != expect
    if wrong.any():
        fail("b. node count over contigs and twins", owner[wrong])
    missing = alive & (cnt == 0)
    if missing.any():
        fails.append("b. %d alive nodes in no contig, e.g. %s" %
                     (int(missing.sum()), ", ".join(g.text(i) for i in np.nonzero(missing)[0][:examples])))
    # c
    inner = np.ones(ids.size, bool)
    inner[last[has]] = False
    bad = inner & (succ[ids] != np.roll(ids, -1))
    if bad.any():
        fail("c. consecutive windows are not linked", owner[bad])
    # d
    pred = np.full(g.n, -1, np.int64)
    src = np.nonzero(succ >= 0)[0]
    pred[succ[src]] = src
    f, l = ids[first[has]], ids[last[has]]
    cyc = succ[l] == f
    bad = ~cyc & ((pred[f] >= 0) | (succ[l] >= 0))
    if bad.any():
        fail("d. not maximal (the first window has a predecessor or the last a successor)", np.nonzero(has)[0][bad])
    # e
    if sums is not None:
        s = np.zeros(len(contigs), np.int64)
        np.add.at(s, owner, g.cnt[ids])
        got = np.asarray([int(x) for x in sums], np.int64)
        if got.size != len(contigs):
            fails.append("e. %d sums for %d contigs" % (got.size, len(contigs)))
        elif (got != s).any():
            fail("e. wrong count sum", np.nonzero(got != s)[0])
    return fails
