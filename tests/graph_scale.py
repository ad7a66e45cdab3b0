"""Array-for-array checks of a built de Bruijn graph against the oracle's, vectorised so that they stay cheap at the
sizes the benchmark runs (10^7..10^8 l-mers).  Used by tests/test_gpu_graph_scale.py; tests/test_cpu_graph_scale.py
feeds them the oracle's own graph with one defect at a time to show that each defect is caught.

The helpers read the artefacts through `src.download(which)`, so `src` is a _native.Context after a run or an
`Artifacts` holding arrays.  A mismatch raises AssertionError naming the array and its first differing index."""
import numpy as np

import _native as N

NO_ID = 0xFFFFFFFF
U64 = np.uint64


class Artifacts:
    """The artefacts of an oracle graph in the layout the library downloads them (offsets as u32)."""

    def __init__(self, g):
        self.a = {w: x.copy() for w, x in expected(g).items()}

    def download(self, which):
        return self.a[which]


def expected(g):
    """the oracle graph's arrays by artefact id (views where the dtype already matches)"""
    a = {N.ART_LMER_KEYS: g.lk_lo, N.ART_LMER_KEYS_HI: g.lk_hi, N.ART_LMER_VALUES: g.lvals,
         N.ART_LMER_OFFSETS: g.loffs.astype(np.uint32), N.ART_KMER_KEYS: g.vk_lo, N.ART_KMER_KEYS_HI: g.vk_hi,
         N.ART_LCOUNT: g.lcount, N.ART_ECOUNT: g.ecount, N.ART_LSTART: g.lstart.astype(np.uint32),
         N.ART_ESTART: g.estart.astype(np.uint32), N.ART_EDGE_V1: g.ev1, N.ART_EDGE_V2: g.ev2, N.ART_EV: g.ev}
    if g.expanded:
        a.update({N.ART_EE: g.ee, N.ART_LEV: g.lev, N.ART_ENT: g.ent})
    return a


def relabel(g, seed):
    """The oracle's compressed graph with its l-mers and vertices in a random order, as a slot-order run leaves them:
    offsets, starts and EV recomputed in the new order."""
    rng = np.random.default_rng(seed)
    art = Artifacts(g)
    a = art.a
    po, pv = rng.permutation(g.nl), rng.permutation(g.nv)     # new position -> oracle id
    newid = np.empty(g.nv, np.int64)
    newid[pv] = np.arange(g.nv)
    for w in (N.ART_LMER_KEYS, N.ART_LMER_KEYS_HI, N.ART_LMER_VALUES):
        a[w] = a[w][po]
    a[N.ART_EDGE_V1] = newid[g.ev1[po]].astype(np.uint32)
    a[N.ART_EDGE_V2] = newid[g.ev2[po]].astype(np.uint32)
    a[N.ART_LMER_OFFSETS] = excl_scan(a[N.ART_LMER_VALUES])
    for w in (N.ART_KMER_KEYS, N.ART_KMER_KEYS_HI):
        a[w] = a[w][pv]
    for w in (N.ART_LCOUNT, N.ART_ECOUNT):
        a[w] = a[w].reshape(-1, 4)[pv].ravel()
    a[N.ART_LSTART], a[N.ART_ESTART] = excl_scan(a[N.ART_LCOUNT]), excl_scan(a[N.ART_ECOUNT])
    a[N.ART_EV] = make_ev(a[N.ART_KMER_KEYS], a[N.ART_LCOUNT], a[N.ART_ECOUNT], a[N.ART_LSTART], a[N.ART_ESTART])
    for w in (N.ART_EE, N.ART_LEV, N.ART_ENT):
        a.pop(w, None)
    return art


def excl_scan(x):
    """exclusive scan of u32 counts, modulo 2^32 like the library's offsets"""
    out = np.zeros(x.size, U64)
    if x.size > 1:
        np.cumsum(x[:-1], dtype=U64, out=out[1:])
    return (out & U64(0xFFFFFFFF)).astype(np.uint32)


def make_ev(vk, lc, ec, ls, es):
    ev = np.zeros(vk.size, N.EV_DTYPE)
    ev["vid"] = vk
    ev["lcount"], ev["ecount"] = lc.reshape(-1, 4).sum(1), ec.reshape(-1, 4).sum(1)
    ev["lp"], ev["ep"] = ls[::4], es[::4]
    return ev


def same(name, got, exp):
    """exact equality of two arrays; the message names the array and its first differing index"""
    got, exp = np.asarray(got), np.asarray(exp)
    if got.shape != exp.shape:
        raise AssertionError("%s: shape %s, oracle %s" % (name, got.shape, exp.shape))
    if got.dtype.names:
        for f in got.dtype.names:
            same("%s.%s" % (name, f), got[f], exp[f])
        return
    bad = np.flatnonzero(got != exp)
    if bad.size:
        i = int(bad[0])
        raise AssertionError("%s: %d of %d entries differ, first at %d: %r, oracle %r" % (name, bad.size, got.size, i, got.flat[i],
                                                                                          exp.flat[i]))


def assert_counts(st, g):
    got = (st.distinct_lmers, st.distinct_kmers, st.edge_count)
    assert got == (g.nl, g.nv, g.ne), "stats (U_l, V, E) %s, oracle %s" % (got, (g.nl, g.nv, g.ne))
    assert st.n_lmer_windows * 2 == g.ne


def _hi(src, which, n, wide):
    return src.download(which) if wide else np.zeros(n, U64)


def key_order(lo, hi, wide):
    """positions in ascending key order: (hi, lo) for two-word keys"""
    return np.lexsort((lo, hi)) if wide else np.argsort(lo, kind="stable")


def assert_graph_canonical(src, g, wide):
    """ids = rank in ascending key order: every artefact equals the oracle's, array for array (the expanded edges
    EE / LEV / ENT too when the oracle graph was expanded)"""
    names = ["LMER_KEYS", "LMER_VALUES", "LMER_OFFSETS", "KMER_KEYS", "LCOUNT", "ECOUNT", "LSTART", "ESTART", "EDGE_V1", "EDGE_V2",
             "EV"]
    if wide:
        names += ["LMER_KEYS_HI", "KMER_KEYS_HI"]
    if g.expanded:
        names += ["EE", "LEV", "ENT"]
    exp = expected(g)
    for n in names:
        w = getattr(N, "ART_" + n)
        same(n, src.download(w), exp[w])
        exp.pop(w)


def assert_graph_label_free(src, g, wide):
    """ids in any order (slot order): the same graph up to a bijection of the l-mer and vertex ids.  Sorted keys and
    their multiplicities, the per-slot LCOUNT / ECOUNT rows and the end points of every edge through the bijection
    equal the oracle's; LMER_OFFSETS / LSTART / ESTART are scans of the downloaded arrays and EV is made of its parts."""
    lk, lv = src.download(N.ART_LMER_KEYS), src.download(N.ART_LMER_VALUES)
    lh = _hi(src, N.ART_LMER_KEYS_HI, lk.size, wide)
    o = key_order(lk, lh, wide)
    same("LMER_KEYS (sorted)", lk[o], g.lk_lo)
    if wide:
        same("LMER_KEYS_HI (sorted)", lh[o], g.lk_hi)
    same("LMER_VALUES (key order)", lv[o], g.lvals)
    vk = src.download(N.ART_KMER_KEYS)
    vh = _hi(src, N.ART_KMER_KEYS_HI, vk.size, wide)
    ov = key_order(vk, vh, wide)
    same("KMER_KEYS (sorted)", vk[ov], g.vk_lo)
    if wide:
        same("KMER_KEYS_HI (sorted)", vh[ov], g.vk_hi)
    rank = np.empty(vk.size, np.int64)
    rank[ov] = np.arange(vk.size)           # id of the run -> oracle id
    lc, ec = src.download(N.ART_LCOUNT), src.download(N.ART_ECOUNT)
    same("LCOUNT rows (key order)", lc.reshape(-1, 4)[ov], g.lcount.reshape(-1, 4))
    same("ECOUNT rows (key order)", ec.reshape(-1, 4)[ov], g.ecount.reshape(-1, 4))
    v1, v2 = src.download(N.ART_EDGE_V1), src.download(N.ART_EDGE_V2)
    same("EDGE_V1 (through the bijection)", rank[v1[o]], g.ev1)
    same("EDGE_V2 (through the bijection)", rank[v2[o]], g.ev2)
    ls, es = src.download(N.ART_LSTART), src.download(N.ART_ESTART)
    same("LSTART (scan of LCOUNT)", ls, excl_scan(lc))
    same("ESTART (scan of ECOUNT)", es, excl_scan(ec))
    same("LMER_OFFSETS (scan of LMER_VALUES)", src.download(N.ART_LMER_OFFSETS), excl_scan(lv))
    same("EV (of its parts)", src.download(N.ART_EV), make_ev(vk, lc, ec, ls, es))


def derived_graph(lk, lv, vk, l):
    """the canonical-id artefacts (l <= 32) that follow from the sorted l-mer multiset (lk, lv) and the sorted vertex
    keys vk alone, for checking a graph too large for the oracle's graph build: edge end points are the ranks of the
    prefix and suffix, the leaving slot of v1 is the last base and the entering slot of v2 the first base"""
    k = l - 1
    v1 = np.searchsorted(vk, lk >> U64(2)).astype(np.uint32)
    v2 = np.searchsorted(vk, lk & U64((1 << (2 * k)) - 1)).astype(np.uint32)
    lc = np.zeros(4 * vk.size, np.uint32)
    ec = np.zeros(4 * vk.size, np.uint32)
    lc[4 * v1.astype(np.int64) + (lk & U64(3)).astype(np.int64)] = lv
    ec[4 * v2.astype(np.int64) + (lk >> U64(2 * k)).astype(np.int64)] = lv
    ls, es = excl_scan(lc), excl_scan(ec)
    return {"LMER_OFFSETS": excl_scan(lv), "EDGE_V1": v1, "EDGE_V2": v2, "LCOUNT": lc, "ECOUNT": ec, "LSTART": ls, "ESTART": es,
            "EV": make_ev(vk, lc, ec, ls, es)}


# ---- the k-mer-space partition --------------------------------------------------------------------------------------
def _shr(lo, hi, sh):
    """bits sh.. of two-word keys, low word only"""
    if sh == 0:
        return lo.copy()
    if sh < 64:
        return (lo >> U64(sh)) | (hi << U64(64 - sh))
    return hi >> U64(sh - 64)


def revcomp(w, m):
    """reverse complements of m-mers (m <= 32) held in u64 arrays"""
    r = np.zeros_like(w)
    for _ in range(m):
        r = (r << U64(2)) | (U64(3) - (w & U64(3)))
        w = w >> U64(2)
    return r


def owner(lo, hi, k, world):
    """owning rank of k-mers: the low 16 bits of the least scrambled canonical m-mer score (m = min(12, k)), scaled to
    `world` (the device rule of csrc/dist.cu, restated over arrays)"""
    m = min(12, k)
    mask = U64((1 << (2 * m)) - 1)
    best = np.full(lo.size, 0xFFFFFFFF, U64)
    for j in range(k - m + 1):
        w = _shr(lo, hi, 2 * (k - m - j)) & mask
        c = np.minimum(w, revcomp(w, m))
        s = (c * U64(2654435761)) & U64(0xFFFFFFFF)
        s ^= s >> U64(15)
        np.minimum(best, s, out=best)
    return (((best & U64(0xFFFF)) * U64(world)) >> U64(16)).astype(np.int64)


def prefix_suffix(lo, hi, l):
    """(prefix lo, prefix hi, suffix lo, suffix hi) (k = l - 1) of two-word l-mer keys"""
    k = l - 1
    plo, phi = (lo >> U64(2)) | (hi << U64(62)), hi >> U64(2)
    if 2 * k >= 64:
        slo, shi = lo.copy(), hi & U64((1 << (2 * k - 64)) - 1)
    else:
        slo, shi = lo & U64((1 << (2 * k)) - 1), np.zeros_like(hi)
    return plo, phi, slo, shi


def assert_partitioned(parts, windows, g, world):
    """per-rank graphs of the k-mer-space partition (eulercuda.dist.emulate_partitioned[_bucketed]) against the single
    graph of the oracle: every vertex on exactly one rank, the one it hashes to, with the oracle's LCOUNT / ECOUNT
    rows; every both-strand l-mer exactly once, on the owner of its prefix, with its multiplicity; v1 local, v2 local
    exactly when the suffix has the same owner; per-rank offsets and starts are scans, EV is made of its parts."""
    l = g.l
    k, wide = l - 1, l > 32
    assert sum(w[0] for w in windows) * 2 == g.ne, "l-mer windows over the ranks"
    vlo, vhi, lcs, ecs, llo, lhi, lvs = [], [], [], [], [], [], []
    total_e = 0
    for r, p in enumerate(parts):
        vk = p["KMER_KEYS"]
        vh = p["KMER_KEYS_HI"] if wide else np.zeros(vk.size, U64)
        if vk.size:
            own = owner(vk, vh, k, world)
            assert (own == r).all(), "rank %d holds a vertex of rank %d" % (r, int(own[own != r][0]))
        lc, ec = p["LCOUNT"][:4 * vk.size], p["ECOUNT"][:4 * vk.size]
        if vk.size:
            same("rank %d LSTART" % r, p["LSTART"], excl_scan(lc))
            same("rank %d ESTART" % r, p["ESTART"], excl_scan(ec))
        same("rank %d EV" % r, p["EV"], make_ev(vk, lc, ec, p["LSTART"][:4 * vk.size], p["ESTART"][:4 * vk.size]))
        lk, lv = p["LMER_KEYS"], p["LMER_VALUES"]
        lh = p["LMER_KEYS_HI"] if wide else np.zeros(lk.size, U64)
        total_e += int(lv.sum(dtype=U64))
        assert p["stats"]["edge_count"] == int(lv.sum(dtype=U64)), "rank %d edge_count" % r
        if lk.size:
            same("rank %d LMER_OFFSETS" % r, p["LMER_OFFSETS"], excl_scan(lv))
            plo, phi, slo, shi = prefix_suffix(lk, lh, l)
            v1, v2 = p["EDGE_V1"].astype(np.int64), p["EDGE_V2"]
            assert (v1 < vk.size).all(), "rank %d: v1 not local" % r
            same("rank %d prefix of EDGE_V1" % r, vk[v1], plo)
            same("rank %d prefix hi of EDGE_V1" % r, vh[v1], phi)
            loc = v2 != NO_ID
            vl = v2[loc].astype(np.int64)
            assert (vl < vk.size).all(), "rank %d: v2 out of range" % r
            same("rank %d suffix of EDGE_V2" % r, vk[vl], slo[loc])
            same("rank %d suffix hi of EDGE_V2" % r, vh[vl], shi[loc])
            so = owner(slo, shi, k, world)
            assert (so[loc] == r).all() and (so[~loc] != r).all(), "rank %d: EDGE_V2 locality != suffix owner" % r
        vlo.append(vk); vhi.append(vh); lcs.append(lc.reshape(-1, 4)); ecs.append(ec.reshape(-1, 4))
        llo.append(lk); lhi.append(lh); lvs.append(lv)
    vlo, vhi, llo, lhi = (np.concatenate(x) for x in (vlo, vhi, llo, lhi))
    ov = key_order(vlo, vhi, wide)
    same("vertices over the ranks", vlo[ov], g.vk_lo)
    same("vertex hi words over the ranks", vhi[ov], g.vk_hi if wide else np.zeros(g.nv, U64))
    same("LCOUNT rows over the ranks", np.concatenate(lcs)[ov], g.lcount.reshape(-1, 4))
    same("ECOUNT rows over the ranks", np.concatenate(ecs)[ov], g.ecount.reshape(-1, 4))
    o = key_order(llo, lhi, wide)
    same("l-mers over the ranks", llo[o], g.lk_lo)
    same("l-mer hi words over the ranks", lhi[o], g.lk_hi if wide else np.zeros(g.nl, U64))
    same("LMER_VALUES over the ranks", np.concatenate(lvs)[o], g.lvals)
    assert total_e == g.ne, "edges over the ranks %d, oracle %d" % (total_e, g.ne)


def partition_of(g, world):
    """what a correct partitioned build gives for the oracle graph `g` (local ids in key order): the input the CPU test
    feeds assert_partitioned"""
    l, k, wide = g.l, g.l - 1, g.l > 32
    vown = owner(g.vk_lo, g.vk_hi, k, world)
    plo, phi, slo, shi = prefix_suffix(g.lk_lo, g.lk_hi, l)
    lown = vown[g.ev1]
    parts = []
    for r in range(world):
        vs = np.flatnonzero(vown == r)
        local = np.full(g.nv, NO_ID, np.int64)
        local[vs] = np.arange(vs.size)
        ls = np.flatnonzero(lown == r)
        lc, ec = g.lcount.reshape(-1, 4)[vs].ravel(), g.ecount.reshape(-1, 4)[vs].ravel()
        lv = g.lvals[ls]
        p = {"KMER_KEYS": g.vk_lo[vs], "LCOUNT": lc, "ECOUNT": ec, "LSTART": excl_scan(lc), "ESTART": excl_scan(ec),
             "LMER_KEYS": g.lk_lo[ls], "LMER_VALUES": lv, "LMER_OFFSETS": excl_scan(lv),
             "EDGE_V1": local[g.ev1[ls]].astype(np.uint32), "EDGE_V2": local[g.ev2[ls]].astype(np.uint32),
             "stats": {"edge_count": int(lv.sum(dtype=U64))}}
        if wide:
            p["KMER_KEYS_HI"], p["LMER_KEYS_HI"] = g.vk_hi[vs], g.lk_hi[ls]
        p["EV"] = make_ev(p["KMER_KEYS"], lc, ec, p["LSTART"], p["ESTART"])
        parts.append(p)
    return parts, [(g.ne // 2, 0)] + [(0, 0)] * (world - 1)
