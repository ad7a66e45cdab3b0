"""Two restatements of the multi-k rule of include/euler_b200.h (euler_unitigs_multik) -- test infrastructure only.

`strings` works on the oracle's py_build dict and clean_ref.clean; `arrays` on oracle.count_mers and unitig_np's graph,
fast enough for genome sizes.  Both write a step's contigs as the library does: every maximal unitig of the surviving
node set once, whole (a unitig that is its own reverse complement included, where py_all_contigs stops half-way),
and every cycle once, as the K + L - 1 bases that spell its L K-mers.  A contig is a cycle when the link rule takes
its last K-mer to its first, as unitig_np.certify defines it; the next step reads it as its cyclic sequence, all
rotations.  Each returns (contigs, kmer_sums, steps) like Context.unitigs_multik, steps being dicts with K, contigs,
bases, nodes_added and clean (the euler_clean_stats fields)."""
import numpy as np

import oracle
import unitig_np
from clean_ref import _bwn, _fwn, clean as clean_str, path_unitigs
from oracle import py_build, twin

ZERO = {"rounds": 0, "tips": 0, "isolated": 0, "bubble_branches": 0, "kmers_removed": 0}


def weight(s, L, limit):
    """w_C of a contig with count sum s over L K-mers"""
    return max(limit + 1, s // L)


def cyclic_windows(c, Kp, K, cyc):
    """the K-mers a contig written at Kp spells at K (one orientation): none when it has fewer than K bases; of a
    cycle (L = len(c) - Kp + 1 K-mers at Kp) all L rotations of its cyclic sequence c[:L]"""
    if len(c) < K:
        return []
    if not cyc:
        return [c[i:i + K] for i in range(len(c) - K + 1)]
    L = len(c) - Kp + 1
    s = c[:L] * (K // L + 2)
    return [s[i:i + K] for i in range(L)]


def _params(K, clean, kw):
    if not clean:
        return dict(tip_len=0, isolated_len=0, bubble_len=0, max_rounds=0)
    d = lambda v: 2 * K if v is None else v
    return dict(tip_len=d(kw.get("tip_len")), isolated_len=d(kw.get("isolated_len")), bubble_len=d(kw.get("bubble_len")),
                max_rounds=kw.get("max_rounds", 10))


# ---- on strings ---------------------------------------------------------------------------------------------------
def _succ(A):
    """the link rule of unitig.cu on the node dict A"""
    succ = {}
    for x in A:
        f = _fwn(x, A)
        if len(f) == 1 and f[0] != twin(x) and len(_bwn(f[0], A)) == 1:
            succ[x] = f[0]
    return succ


def str_contigs(A, K):
    """[(contig, is_cycle)]: every maximal unitig and every cycle of A once (one strand of each pair)"""
    out, seen = [], set()
    for c in path_unitigs(A):
        if c[0] in seen:
            continue
        seen.update(c)
        seen.update(twin(x) for x in c)
        out.append((c[0] + "".join(x[-1] for x in c[1:]), False))
    succ = _succ(A)
    for x in sorted(A):
        if x in seen:
            continue
        c = [x]
        while succ[c[-1]] != x:
            c.append(succ[c[-1]])
        seen.update(c)
        seen.update(twin(y) for y in c)
        out.append((c[0] + "".join(y[-1] for y in c[1:]), True))
    return out


def raise_counts(d, prev, Kp, K):
    """steps 2-5 of the rule: d (both-strand K-mer counts, changed in place) raised by prev = [(contig, w_C, is_cycle)]
    written at Kp"""
    for c, w, cyc in prev:
        for x in cyclic_windows(c, Kp, K, cyc):
            for y in (x, twin(x)):
                v = w + (w & 1) if y == twin(y) else w
                if d.get(y, 0) < v:
                    d[y] = v
    return d


def strings(reads, ks, limit=1, clean=True, **kw):
    """the rule on strings: reads upper case, 'N' splits"""
    prev, Kp, steps, sums = [], None, [], []
    for K in ks:
        reads_d = py_build(reads, K, -1)
        d = raise_counts(dict(reads_d), prev, Kp, K)
        A = {x: v for x, v in d.items() if v > limit}
        added = len({min(x, twin(x)) for x in A if reads_d.get(x, 0) <= limit})
        A, st = clean_str(A, K, **_params(K, clean, kw))
        out = str_contigs(A, K)
        sums = [sum(A[c[i:i + K]] for i in range(len(c) - K + 1)) for c, _ in out]
        steps.append({"K": K, "contigs": len(out), "bases": sum(len(c) for c, _ in out), "nodes_added": added, "clean": st})
        prev = [(c, weight(s, len(c) - K + 1, limit), cyc) for (c, cyc), s in zip(out, sums)]
        Kp = K
    return [c for c, _, _ in prev], sums, steps


# ---- on arrays ----------------------------------------------------------------------------------------------------
_CODE = np.full(256, 0, np.uint8)
_CODE[np.frombuffer(b"ACGT", np.uint8)] = np.arange(4, dtype=np.uint8)


def _encode(seqs, K):
    """(lo, hi) of every K-window of every string in seqs, in order; and the number of windows of each"""
    lens = np.array([len(s) for s in seqs], np.int64)
    nw = np.maximum(lens - K + 1, 0)
    if not nw.sum():
        return np.zeros(0, np.uint64), np.zeros(0, np.uint64), nw
    code = _CODE[np.frombuffer("".join(seqs).encode("ascii"), np.uint8)].astype(np.uint64)
    starts = np.repeat(np.cumsum(lens) - lens, nw) + (np.arange(nw.sum()) - np.repeat(np.cumsum(nw) - nw, nw))
    lo = np.zeros(starts.size, np.uint64)
    hi = np.zeros(starts.size, np.uint64)
    mlo = unitig_np.M64 if K >= 32 else np.uint64((1 << (2 * K)) - 1)
    mhi = np.uint64((1 << max(2 * K - 64, 0)) - 1)
    for j in range(K):
        hi = ((hi << np.uint64(2)) | (lo >> np.uint64(62))) & mhi
        lo = ((lo << np.uint64(2)) | code[starts + j]) & mlo
    return lo, hi, nw


def _revcomp(K, lo, hi):
    """(lo, hi) of the reverse complements (unitig_np.Graph.revcomp)"""
    s = 128 - 2 * K
    rhi, rlo = unitig_np._rev2(~lo), unitig_np._rev2(~hi)
    if s >= 64:
        return rhi >> np.uint64(s - 64), np.zeros_like(lo)
    return (rlo >> np.uint64(s)) | (rhi << np.uint64(64 - s)), rhi >> np.uint64(s)


def _find(K, tlo, thi, lo, hi):
    """indices of (lo, hi) in the ascending table (tlo, thi), -1 where absent"""
    if not tlo.size:
        return np.full(lo.size, -1, np.int64)
    t = unitig_np.Graph.__new__(unitig_np.Graph)
    t.K = K
    keys, q = t._pack(tlo, thi), t._pack(lo, hi)
    i = np.searchsorted(keys, q)
    j = np.minimum(i, tlo.size - 1)
    return np.where((i < tlo.size) & (keys[j] == q), j, -1).astype(np.int64)


def _merge_max(K, lo, hi, cnt):
    """sorted distinct (lo, hi) with the largest cnt of each"""
    o = np.lexsort((lo, hi))
    lo, hi, cnt = lo[o], hi[o], cnt[o]
    if not lo.size:
        return lo, hi, cnt
    first = np.ones(lo.size, bool)
    first[1:] = (lo[1:] != lo[:-1]) | (hi[1:] != hi[:-1])
    idx = np.nonzero(first)[0]
    return lo[idx], hi[idx], np.maximum.reduceat(cnt, idx)


def arr_contigs(g, alive):
    """[(contig, is_cycle, sum)] of the alive node set of unitig_np graph g: one strand of each pair"""
    paths, cycles = unitig_np.path_chains(g, alive)
    out = []
    letters = np.frombuffer(b"ACGT", np.uint8)

    def spell(c):
        c = np.asarray(c, np.int64)
        tail = letters[(g.lo[c[1:]] & np.uint64(3)).astype(np.int64)].tobytes().decode()
        return g.text(c[0]) + tail, int(g.cnt[c].sum())

    for c in paths:
        if c[0] <= g.twin[c[-1]]:
            out.append(spell(c) + (False,))
    for c in cycles:
        if min(c) <= int(g.twin[c].min()):
            out.append(spell(c) + (True,))
    return [(s, cyc, sm) for s, sm, cyc in out]


def arrays(buf, off, ks, limit=1, clean=True, last=None, trace=None, **kw):
    """the rule on unitig_np's graph (reads as oracle.pack_reads gives them); last (a dict) receives the last step's
    graph (key "g") and its surviving nodes (key "alive").  trace (a list) receives one dict per step: K, contigs (its
    [(contig, is_cycle, sum)]), weights (the w_C it hands on, one per contig) and odd_pal (the palindromic K-mers whose
    count is the previous contigs' odd weight rounded up to even, above their read count)"""
    prev, Kp, steps, sums = [], None, [], []
    for K in ks:
        odd_pal = 0
        rlo, rhi, rcnt = oracle.count_mers(buf, off, K)
        rcnt = rcnt.astype(np.int64)
        lo, hi, cnt = rlo, rhi, rcnt
        seqs, ws = [], []
        for c, w, cyc in prev:
            if len(c) < K:
                continue
            if cyc:
                L = len(c) - Kp + 1
                c = (c[:L] * (K // L + 2))[:L + K - 1]
            seqs.append(c)
            ws.append(w)
        if seqs:
            wlo, whi, nw = _encode(seqs, K)
            w = np.repeat(np.asarray(ws, np.int64), nw)
            tlo, thi = _revcomp(K, wlo, whi)
            pal = (wlo == tlo) & (whi == thi)
            odd = pal & (w & 1 == 1)
            w = np.where(pal, w + (w & 1), w)
            if trace is not None and odd.any():
                rid = _find(K, rlo, rhi, wlo[odd], whi[odd])
                below = np.where(rid >= 0, rcnt[np.maximum(rid, 0)], 0) < w[odd]
                plo, phi, pw = _merge_max(K, wlo[odd][below], whi[odd][below], w[odd][below])
            wlo, whi, w = np.concatenate([wlo, tlo]), np.concatenate([whi, thi]), np.concatenate([w, w])
            lo, hi, cnt = _merge_max(K, np.concatenate([rlo, wlo]), np.concatenate([rhi, whi]), np.concatenate([rcnt, w]))
            if trace is not None and odd.any():
                odd_pal = int((cnt[_find(K, lo, hi, plo, phi)] == pw).sum())
        keep = cnt > limit
        g = unitig_np.Graph(K, lo[keep], hi[keep], cnt[keep])
        # nodes whose read count is <= limit (absent: 0), counted once per strand pair
        rid = _find(K, rlo, rhi, g.lo, g.hi)
        new = np.where(rid >= 0, rcnt[np.maximum(rid, 0)], 0) <= limit
        ids = np.arange(g.n)
        added = int((new & (ids <= g.twin)).sum())
        p = _params(K, clean, kw)
        if p["max_rounds"]:
            alive, st = unitig_np.clean(g, **p)
        else:
            alive, st = np.ones(g.n, bool), dict(ZERO)
        out = arr_contigs(g, alive)
        if last is not None:
            last.update(g=g, alive=alive)
        sums = [s for _, _, s in out]
        steps.append({"K": K, "contigs": len(out), "bases": sum(len(c) for c, _, _ in out), "nodes_added": added,
                      "clean": st})
        prev = [(c, weight(s, len(c) - K + 1, limit), cyc) for c, cyc, s in out]
        if trace is not None:
            trace.append({"K": K, "contigs": out, "weights": [w for _, w, _ in prev], "odd_pal": odd_pal})
        Kp = K
    return [c for c, _, _ in prev], sums, steps


# ---- comparison ----------------------------------------------------------------------------------------------------
def canon(c, K):
    """orientation- and rotation-free form of a contig written at K: a contig whose text closes on itself (its last
    K-mer extended by its base K - 1 is its first) is read as a cyclic sequence"""
    forms = [c, twin(c)]
    if len(c) >= K and c[len(c) - K + 1:] + c[K - 1] == c[:K]:
        L = len(c) - K + 1
        out = []
        for f in forms:
            s = f[:L]
            out.append(min(s[i:] + s[:i] for i in range(L)))
        return "@" + min(out)
    return min(forms)


def canon_pairs(contigs, sums, K):
    """sorted (canonical contig, sum) pairs"""
    return sorted((canon(c, K), int(s)) for c, s in zip(contigs, sums))
