"""ctypes binding of libeuler_b200.so (the C ABI in include/euler_b200.h).

This is the only place Python touches native code.  There is NO CPU fallback: if the shared
library is missing or no CUDA device is present, every entry point raises ``EulerError``.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EULER_B200_LIBPATH") or os.path.join(_HERE, "libeuler_b200.so")

EV_DTYPE = np.dtype([("vid", np.uint64), ("ep", np.uint32), ("ecount", np.uint32),
                     ("lp", np.uint32), ("lcount", np.uint32)])            # pydebruijn.py:607
EE_DTYPE = np.dtype([("eid", np.uint64), ("v1", np.uint32), ("v2", np.uint32),
                     ("s", np.uint32), ("pad", np.uint32)])                # pydebruijn.py:605
SV_DTYPE = np.dtype([("vid", np.uint32), ("n1", np.uint32), ("n2", np.uint32)])   # pyeulertour.py:735
CE_DTYPE = np.dtype([("ceid", np.uint32), ("e1", np.uint32), ("e2", np.uint32),
                     ("c1", np.uint32), ("c2", np.uint32)])                # pyeulertour.py:786

RUN_EXPAND_EDGES = 1
RUN_CANONICAL_IDS = 2

(ART_LMER_KEYS, ART_LMER_VALUES, ART_LMER_OFFSETS, ART_KMER_KEYS, ART_LCOUNT, ART_ECOUNT, ART_LSTART,
 ART_ESTART, ART_EV, ART_EDGE_V1, ART_EDGE_V2, ART_EE, ART_LEV, ART_ENT, ART_LMER_KEYS_HI, ART_KMER_KEYS_HI) = range(16)

_ART_DTYPE = {
    ART_LMER_KEYS: np.uint64, ART_LMER_VALUES: np.uint32, ART_LMER_OFFSETS: np.uint32,
    ART_KMER_KEYS: np.uint64, ART_LCOUNT: np.uint32, ART_ECOUNT: np.uint32, ART_LSTART: np.uint32,
    ART_ESTART: np.uint32, ART_EV: EV_DTYPE, ART_EDGE_V1: np.uint32, ART_EDGE_V2: np.uint32,
    ART_EE: EE_DTYPE, ART_LEV: np.uint32, ART_ENT: np.uint32,
    ART_LMER_KEYS_HI: np.uint64, ART_KMER_KEYS_HI: np.uint64,
}


class EulerError(RuntimeError):
    pass


class Stats(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("n_bases", C.c_uint64), ("n_kmer_windows", C.c_uint64),
                ("n_lmer_windows", C.c_uint64), ("distinct_lmers", C.c_uint64), ("distinct_kmers", C.c_uint64),
                ("edge_count", C.c_uint64), ("lmer_table_capacity", C.c_uint64),
                ("kmer_table_capacity", C.c_uint64), ("retries", C.c_uint32),
                ("ms_count", C.c_float), ("ms_graph", C.c_float), ("ms_total", C.c_float),
                ("ms_count_kernel", C.c_float), ("kernel_launches", C.c_uint32),
                ("ms_build_kernel", C.c_float), ("path", C.c_uint32), ("n_buckets", C.c_uint32), ("redo_buckets", C.c_uint32),
                ("bucket_records", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib = None


def load():
    """Load the shared library (raises EulerError if it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EulerError("libeuler_b200.so not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                         "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    sig = {
        "euler_ctx_create": [i32, C.POINTER(vp)],
        "euler_ctx_set_stream": [vp, vp],
        "euler_ctx_sync": [vp],
        "euler_encode_lmers": [vp, vp, vp, u64, u32, vp, vp, vp],
        "euler_compute_kmers": [vp, vp, u64, u64, vp, vp],
        "euler_count_lmers": [vp, vp, vp, u64, u32, vp, vp, vp, vp, vp, vp],
        "euler_count_mers": [vp, vp, vp, u64, u32, u32, vp, vp, vp],
        "euler_count_mers_wide": [vp, vp, vp, u64, u32, u32, vp, vp, vp, vp],
        "euler_unitigs": [vp, vp, vp, u64, u32, u32, vp, vp, vp],
        "euler_unitigs_from_kmers": [vp, vp, vp, u64, u32, vp, vp, vp],
        "euler_unitigs_from_kmers_wide": [vp, vp, vp, vp, u64, u32, vp, vp, vp],
        "euler_unitig_links": [vp, vp, vp, u64, u32, vp],
        "euler_hash_build": [vp, vp, vp, u64, u64, vp, vp],
        "euler_hash_lookup": [vp, vp, vp, u64, vp, u64, vp],
        "euler_exclusive_scan_u32": [vp, vp, u64, vp],
        "euler_debruijn_count": [vp, vp, vp, u64, vp, vp, u64, u32, u64, vp, vp],
        "euler_setup_vertices": [vp, vp, u64, vp, vp, u64, vp, vp, vp, vp, vp],
        "euler_setup_edges": [vp, vp, vp, vp, u64, vp, vp, u64, u32, vp, vp, u64, vp, vp, vp],
        "euler_assign_successor": [vp, vp, vp, vp, u32, vp, u32],
        "euler_successor_graph": [vp, vp, u32, vp],
        "euler_find_components": [vp, vp, u32, vp],
        "euler_circuit_vertices": [vp, vp, u32, vp, vp, vp, vp],
        "euler_circuit_edges": [vp, vp, vp, u32, vp, vp, u32, vp, vp],
        "euler_spanning_forest": [vp, vp, u64, u32, vp, vp],
        "euler_mark_spanning": [vp, vp, u64, vp, u32, u32, vp],
        "euler_swipe": [vp, vp, vp, u32, vp, vp, u32],
        "euler_contig_starts": [vp, vp, u32, vp],
        "euler_emit_contigs": [vp, vp, u32, vp, u32, u32, vp, vp, vp],
        "euler_pipeline_run_dev": [vp, vp, vp, u64, u64, u32, u32, u64, vp],
        "euler_pipeline_run_host": [vp, vp, vp, u64, u32, u32, u64, vp],
        "euler_pipeline_run_lmers": [vp, vp, vp, u64, u32, u32, vp],
        "euler_pipeline_artifact_bytes": [vp, i32, vp],
        "euler_pipeline_download": [vp, i32, vp, u64],
        "euler_pipeline_device_ptr": [vp, i32, vp],
        "euler_pipeline_contigs": [vp, vp, vp, vp],
        "euler_synth_reads_dev": [vp, u64, u32, u32, u64, u64, vp],
        "euler_ingest": [vp, vp, u64, i32, vp, vp],
        "euler_ingest_download": [vp, vp, vp],
        "euler_pipeline_run_ingested": [vp, u32, u32, u64, vp],
        "euler_unitigs_ingested": [vp, u32, u32, vp, vp, vp],
        "euler_dist_count": [vp, vp, vp, u64, u64, u32, u32, vp],
        "euler_dist_scatter": [vp, vp, vp, u64, u64, u32, u32, vp, vp],
        "euler_dist_scatter_segments": [vp, vp, vp, u64, u64, u32, u32, vp, u64, vp],
        "euler_dist_build": [vp, vp, u64, u32, u32, u32, u64, vp],
        "euler_dist_recv_alloc": [vp, u64, vp, vp],
        "euler_dist_peer_open": [vp, vp, vp],
        "euler_dist_peer_close": [vp, vp],
        "euler_dist_scatter_peers": [vp, vp, vp, u64, u64, u32, u32, vp, u64, vp],
        "euler_dist_build_regions": [vp, vp, u64, vp, u32, u32, u32, u64, vp],
        "euler_bkt_area_bytes": [u32, u32, vp],
        "euler_bkt_area_alloc": [vp, i32, u32, u32, vp, vp],
        "euler_bkt_scatter": [vp, vp, vp, u64, u64, u32, u32, u32, u32, u32, vp, vp, vp],
        "euler_bkt_build": [vp, vp, u32, u32, u32, u32, u32, u64, vp],
        "euler_compat_phase1": [vp, vp, u64, u32, vp, vp],
        "euler_compat_copy_to_bucket": [vp, vp, vp, vp, u64, vp, u32, vp, vp],
        "euler_compat_bucket_sort": [vp, vp, vp, u64, vp, vp, u32, vp, vp],
        "euler_compat_cc_step": [vp, i32, u32, u32, vp, vp, vp, vp, vp, vp, vp, vp, vp],
    }
    for name, args in sig.items():
        fn = getattr(L, name)
        fn.argtypes = args
        fn.restype = i32
    L.euler_ctx_destroy.argtypes = [vp]
    L.euler_ctx_destroy.restype = None
    L.euler_last_error.argtypes = [vp]
    L.euler_last_error.restype = C.c_char_p
    L.euler_hash_capacity.argtypes = [u64]
    L.euler_hash_capacity.restype = u64
    L.euler_version.argtypes = []
    L.euler_version.restype = i32
    _lib = L
    return L


def _p(a):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


def _arr(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


class Context:
    """One euler_ctx: one GPU, one stream (replaces `import pycuda.autoinit`, pyencode.py:3)."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.euler_ctx_create(int(device), C.byref(h))
        if rc != 0:
            raise EulerError("euler_ctx_create(device=%d) failed with %d: %s" %
                             (device, rc, "no CUDA device (there is no CPU fallback)" if rc == -7 else "CUDA error"))
        self.h = h
        self.device = device

    def close(self):
        # peer mappings of the multi-GPU exchanges live on the context (eulercuda/dist.py) and end with it
        for name in ("_bucket_exchange", "_peer_exchange"):
            ex = getattr(self, name, None)
            if ex is not None and hasattr(ex, "close"):
                try:
                    ex.close()
                except Exception:
                    pass
            if hasattr(self, name):
                setattr(self, name, None)
        if getattr(self, "h", None):
            self.lib.euler_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != 0:
            msg = self.lib.euler_last_error(self.h)
            raise EulerError("libeuler_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))

    def set_stream(self, cuda_stream):
        self.check(self.lib.euler_ctx_set_stream(self.h, C.c_void_p(int(cuda_stream))))

    def sync(self):
        self.check(self.lib.euler_ctx_sync(self.h))

    # ------------------------------------------------------------------ encoder
    def encode_lmers(self, buf, off, l, want_rc=True, want_valid=True):
        buf = _arr(buf, np.uint8)
        off = _arr(off, np.uint64)
        B = int(off[-1])
        fwd = np.zeros(B, np.uint64)
        rc = np.zeros(B, np.uint64) if want_rc else None
        valid = np.zeros(B, np.uint8) if want_valid else None
        self.check(self.lib.euler_encode_lmers(self.h, _p(buf), _p(off), len(off) - 1, int(l), _p(fwd), _p(rc), _p(valid)))
        return fwd, rc, valid

    def compute_kmers(self, lmers, mask):
        lmers = _arr(lmers, np.uint64)
        pk = np.zeros_like(lmers)
        sk = np.zeros_like(lmers)
        self.check(self.lib.euler_compute_kmers(self.h, _p(lmers), lmers.size, int(mask), _p(pk), _p(sk)))
        return pk, sk

    def count_mers(self, buf, off, length, limit=0):
        buf = _arr(buf, np.uint8)
        off = _arr(off, np.uint64)
        n = C.c_uint64(0)
        self.check(self.lib.euler_count_mers(self.h, _p(buf), _p(off), len(off) - 1, int(length), int(limit),
                                             C.byref(n), None, None))
        keys = np.zeros(n.value, np.uint64)
        vals = np.zeros(n.value, np.uint32)
        if n.value:
            self.check(self.lib.euler_count_mers(self.h, _p(buf), _p(off), len(off) - 1, int(length), int(limit),
                                                 C.byref(n), _p(keys), _p(vals)))
        return keys, vals

    def count_mers_wide(self, buf, off, length, limit=0):
        """count_mers for length 1..64: (keys_lo, keys_hi, vals), ascending in (hi, lo) order"""
        buf = _arr(buf, np.uint8)
        off = _arr(off, np.uint64)
        n = C.c_uint64(0)
        self.check(self.lib.euler_count_mers_wide(self.h, _p(buf), _p(off), len(off) - 1, int(length), int(limit),
                                                  C.byref(n), None, None, None))
        lo = np.zeros(n.value, np.uint64)
        hi = np.zeros(n.value, np.uint64)
        vals = np.zeros(n.value, np.uint32)
        if n.value:
            self.check(self.lib.euler_count_mers_wide(self.h, _p(buf), _p(off), len(off) - 1, int(length), int(limit),
                                                      C.byref(n), _p(lo), _p(hi), _p(vals)))
        return lo, hi, vals

    def unitigs(self, buf, off, K, limit=1):
        buf = _arr(buf, np.uint8)
        off = _arr(off, np.uint64)
        nb, nc = C.c_uint64(0), C.c_uint64(0)
        self.check(self.lib.euler_unitigs(self.h, _p(buf), _p(off), len(off) - 1, int(K), int(limit), None,
                                          C.byref(nb), C.byref(nc)))
        if not nb.value:
            return []
        out = np.zeros(nb.value, np.uint8)
        cap = C.c_uint64(nb.value)
        self.check(self.lib.euler_unitigs(self.h, _p(buf), _p(off), len(off) - 1, int(K), int(limit), _p(out),
                                          C.byref(cap), C.byref(nc)))
        return out.tobytes().decode("ascii").split("\n")[:-1]

    def unitigs_from_kmers(self, keys, counts, K, keys_hi=None):
        """unitigs of a K-mer dictionary (packed keys, both-strand counts): referenceAssembler.all_contigs(d, k).
        keys_hi: bits 64.. of the keys, needed when K > 32 (without it K > 32 is refused)."""
        keys = _arr(keys, np.uint64)
        counts = _arr(counts, np.uint32)
        if keys_hi is None:
            def call(out, nb, nc):
                return self.lib.euler_unitigs_from_kmers(self.h, _p(keys), _p(counts), len(keys), int(K), out, nb, nc)
        else:
            keys_hi = _arr(keys_hi, np.uint64)
            if keys_hi.size != keys.size:
                raise EulerError("keys_hi has %d entries, keys %d" % (keys_hi.size, keys.size))

            def call(out, nb, nc):
                return self.lib.euler_unitigs_from_kmers_wide(self.h, _p(keys), _p(keys_hi), _p(counts), len(keys), int(K), out,
                                                              nb, nc)
        nb, nc = C.c_uint64(0), C.c_uint64(0)
        self.check(call(None, C.byref(nb), C.byref(nc)))
        if not nb.value:
            return []
        out = np.zeros(nb.value, np.uint8)
        cap = C.c_uint64(nb.value)
        self.check(call(_p(out), C.byref(cap), C.byref(nc)))
        return out.tobytes().decode("ascii").split("\n")[:-1]

    def unitig_links(self, contigs, K):
        """(n, 16) uint32 link table of referenceAssembler.all_contigs' G (see euler_unitig_links)"""
        n = len(contigs)
        links = np.zeros((n, 16), np.uint32)
        if n:
            text = np.frombuffer("".join(contigs).encode("ascii"), dtype=np.uint8)
            off = np.zeros(n + 1, np.uint64)
            off[1:] = np.cumsum([len(c) for c in contigs], dtype=np.uint64)
            self.check(self.lib.euler_unitig_links(self.h, _p(text), _p(off), n, int(K), _p(links)))
        return links

    # ------------------------------------------------------------------ gpuhash
    def hash_capacity(self, n):
        return int(self.lib.euler_hash_capacity(int(n)))

    def hash_build(self, keys, values, capacity=None):
        keys = _arr(keys, np.uint64)
        values = _arr(values, np.uint32)
        cap = int(capacity) if capacity else self.hash_capacity(keys.size)
        TK = np.zeros(cap, np.uint64)
        TV = np.zeros(cap, np.uint32)
        self.check(self.lib.euler_hash_build(self.h, _p(keys), _p(values), keys.size, cap, _p(TK), _p(TV)))
        return TK, TV

    def hash_lookup(self, TK, TV, queries):
        TK = _arr(TK, np.uint64)
        TV = _arr(TV, np.uint32)
        q = _arr(queries, np.uint64)
        out = np.zeros(q.size, np.uint32)
        self.check(self.lib.euler_hash_lookup(self.h, _p(TK), _p(TV), TK.size, _p(q), q.size, _p(out)))
        return out

    def exclusive_scan(self, a):
        a = _arr(a, np.uint32)
        out = np.zeros_like(a)
        self.check(self.lib.euler_exclusive_scan_u32(self.h, _p(a), a.size, _p(out)))
        return out

    # ------------------------------------------------------------------ debruijn
    def debruijn_count(self, lkeys, lvals, TK, TV, l, vertex_count):
        lkeys = _arr(lkeys, np.uint64)
        lvals = _arr(lvals, np.uint32)
        TK = _arr(TK, np.uint64)
        TV = _arr(TV, np.uint32)
        lcount = np.zeros(4 * vertex_count, np.uint32)
        ecount = np.zeros(4 * vertex_count, np.uint32)
        self.check(self.lib.euler_debruijn_count(self.h, _p(lkeys), _p(lvals), lkeys.size, _p(TK), _p(TV), TK.size,
                                                 int(l), int(vertex_count), _p(lcount), _p(ecount)))
        return lcount, ecount

    def setup_vertices(self, kkeys, TK, TV, lcount, lstart, ecount, estart):
        kkeys = _arr(kkeys, np.uint64)
        TK = _arr(TK, np.uint64)
        TV = _arr(TV, np.uint32)
        ev = np.zeros(kkeys.size, EV_DTYPE)
        a = [_arr(x, np.uint32) for x in (lcount, lstart, ecount, estart)]
        self.check(self.lib.euler_setup_vertices(self.h, _p(kkeys), kkeys.size, _p(TK), _p(TV), TK.size,
                                                 _p(a[0]), _p(a[1]), _p(a[2]), _p(a[3]), _p(ev)))
        return ev

    def setup_edges(self, lkeys, lvals, loffs, TK, TV, l, lstart, estart, edge_count):
        lkeys = _arr(lkeys, np.uint64)
        lvals = _arr(lvals, np.uint32)
        loffs = _arr(loffs, np.uint32)
        TK = _arr(TK, np.uint64)
        TV = _arr(TV, np.uint32)
        lstart = _arr(lstart, np.uint32)
        estart = _arr(estart, np.uint32)
        ee = np.zeros(edge_count, EE_DTYPE)
        lev = np.zeros(edge_count, np.uint32)
        ent = np.zeros(edge_count, np.uint32)
        self.check(self.lib.euler_setup_edges(self.h, _p(lkeys), _p(lvals), _p(loffs), lkeys.size, _p(TK), _p(TV),
                                              TK.size, int(l), _p(lstart), _p(estart), int(edge_count),
                                              _p(ee), _p(lev), _p(ent)))
        return ee, lev, ent

    # ------------------------------------------------------------------ eulertour / component
    def assign_successor(self, ev, lev, ent, ee):
        ev = _arr(ev, EV_DTYPE)
        ee = _arr(ee, EE_DTYPE).copy()
        lev = _arr(lev, np.uint32)
        ent = _arr(ent, np.uint32)
        self.check(self.lib.euler_assign_successor(self.h, _p(ev), _p(lev), _p(ent), ev.size, _p(ee), ee.size))
        return ee

    def successor_graph(self, ee):
        ee = _arr(ee, EE_DTYPE)
        v = np.zeros(ee.size, SV_DTYPE)
        self.check(self.lib.euler_successor_graph(self.h, _p(ee), ee.size, _p(v)))
        return v

    def find_components(self, v):
        v = _arr(v, SV_DTYPE)
        D = np.zeros(v.size, np.uint32)
        self.check(self.lib.euler_find_components(self.h, _p(v), v.size, _p(D)))
        return D

    def circuit_vertices(self, D):
        D = _arr(D, np.uint32)
        Cm = np.zeros(D.size, np.uint32)
        off = np.zeros(D.size, np.uint32)
        cv = np.zeros(D.size, np.uint32)
        n = C.c_uint32(0)
        self.check(self.lib.euler_circuit_vertices(self.h, _p(D), D.size, _p(Cm), _p(off), _p(cv), C.byref(n)))
        return Cm, off, cv[:n.value].copy(), n.value

    def circuit_edges(self, ev, ent, D, cmap):
        ev = _arr(ev, EV_DTYPE)
        ent = _arr(ent, np.uint32)
        D = _arr(D, np.uint32)
        cmap = _arr(cmap, np.uint32)
        n = C.c_uint64(0)
        self.check(self.lib.euler_circuit_edges(self.h, _p(ev), _p(ent), ev.size, _p(D), _p(cmap), D.size, None, C.byref(n)))
        out = np.zeros(n.value, CE_DTYPE)
        if n.value:
            self.check(self.lib.euler_circuit_edges(self.h, _p(ev), _p(ent), ev.size, _p(D), _p(cmap), D.size,
                                                    _p(out), C.byref(n)))
        return out

    def spanning_forest(self, cg, cg_vcount):
        cg = _arr(cg, CE_DTYPE)
        tree = np.zeros(max(cg.size, 1), np.uint32)
        n = C.c_uint32(0)
        self.check(self.lib.euler_spanning_forest(self.h, _p(cg), cg.size, int(cg_vcount), _p(tree), C.byref(n)))
        return tree[:n.value].copy()

    def mark_spanning(self, cg, tree, ecount):
        cg = _arr(cg, CE_DTYPE)
        tree = _arr(tree, np.uint32)
        mark = np.zeros(ecount, np.uint32)
        self.check(self.lib.euler_mark_spanning(self.h, _p(cg), cg.size, _p(tree), tree.size, int(ecount), _p(mark)))
        return mark

    def swipe(self, ev, ent, ee, mark):
        ev = _arr(ev, EV_DTYPE)
        ent = _arr(ent, np.uint32)
        ee = _arr(ee, EE_DTYPE).copy()
        mark = _arr(mark, np.uint32)
        self.check(self.lib.euler_swipe(self.h, _p(ev), _p(ent), ev.size, _p(ee), _p(mark), ee.size))
        return ee

    def contig_starts(self, ee):
        ee = _arr(ee, EE_DTYPE)
        st = np.zeros(ee.size, np.uint32)
        self.check(self.lib.euler_contig_starts(self.h, _p(ee), ee.size, _p(st)))
        return st

    def emit_contigs(self, ev, ee, l):
        ev = _arr(ev, EV_DTYPE)
        ee = _arr(ee, EE_DTYPE)
        nb, nc = C.c_uint64(0), C.c_uint64(0)
        self.check(self.lib.euler_emit_contigs(self.h, _p(ev), ev.size, _p(ee), ee.size, int(l), None,
                                               C.byref(nb), C.byref(nc)))
        if not nb.value:
            return []
        out = np.zeros(nb.value, np.uint8)
        cap = C.c_uint64(nb.value)
        self.check(self.lib.euler_emit_contigs(self.h, _p(ev), ev.size, _p(ee), ee.size, int(l), _p(out),
                                               C.byref(cap), C.byref(nc)))
        return out.tobytes().decode("ascii").split("\n")[:-1]

    # ------------------------------------------------------------------ step-level compat wrappers
    def compat_phase1(self, keys, bucket_count, count=None):
        keys = _arr(keys, np.uint64)
        offset = np.zeros(keys.size, np.uint32)
        count = np.zeros(bucket_count, np.uint32) if count is None else _arr(count, np.uint32).copy()
        self.check(self.lib.euler_compat_phase1(self.h, _p(keys), keys.size, int(bucket_count), _p(offset), _p(count)))
        return offset, count

    def compat_copy_to_bucket(self, keys, values, offset, start, bucket_count):
        keys = _arr(keys, np.uint64)
        values = _arr(values, np.uint32)
        offset = _arr(offset, np.uint32)
        start = _arr(start, np.uint32)
        bk = np.zeros(keys.size, np.uint64)
        bv = np.zeros(keys.size, np.uint32)
        self.check(self.lib.euler_compat_copy_to_bucket(self.h, _p(keys), _p(values), _p(offset), keys.size, _p(start),
                                                        int(bucket_count), _p(bk), _p(bv)))
        return bk, bv

    def compat_bucket_sort(self, bufK, bufV, start, bucket_size, bucket_count):
        bufK = _arr(bufK, np.uint64)
        bufV = _arr(bufV, np.uint32)
        start = _arr(start, np.uint32)
        bucket_size = _arr(bucket_size, np.uint32)
        TK = np.zeros(int(bucket_count) * 520, np.uint64)
        TV = np.zeros(int(bucket_count) * 520, np.uint32)
        self.check(self.lib.euler_compat_bucket_sort(self.h, _p(bufK), _p(bufV), bufK.size, _p(start), _p(bucket_size),
                                                     int(bucket_count), _p(TK), _p(TV)))
        return TK, TV

    _CC_STEPS = {"init": 0, "s1p1": 1, "s1p2": 2, "s2p1": 3, "s2p2": 4, "s3p1": 5, "s3p2": 6, "s4p1": 7, "s4p2": 8, "s5": 9}

    def compat_cc_step(self, step, n, v=None, prevD=None, D=None, Q=None, t1=None, val1=None, t2=None, val2=None, s=0):
        """One Shiloach-Vishkin sub-step; returns what the reference wrapper of that step returns."""
        def a32(x):
            return np.zeros(n, np.uint32) if x is None else _arr(x, np.uint32)[:n].copy()
        vv = np.zeros(n, SV_DTYPE) if v is None else _arr(v, SV_DTYPE)[:n]
        prevD, D, Q, t1, val1, t2, val2 = (a32(x) for x in (prevD, D, Q, t1, val1, t2, val2))
        flag = np.zeros(1, np.uint32)
        self.check(self.lib.euler_compat_cc_step(self.h, self._CC_STEPS[step], int(n), int(s), _p(vv), _p(prevD), _p(D),
                                                 _p(Q), _p(t1), _p(val1), _p(t2), _p(val2), _p(flag)))
        return {"init": (D, Q), "s1p1": D, "s1p2": Q, "s2p1": (t1, t2, val1, val2), "s2p2": (D, Q),
                "s3p1": (t1, t2, val1, val2), "s3p2": D, "s4p1": val1, "s4p2": D, "s5": int(flag[0])}[step]

    # ------------------------------------------------------------------ fused pipeline
    def run_host(self, buf, off, l, flags=0, distinct_hint=0):
        buf = _arr(buf, np.uint8)
        off = _arr(off, np.uint64)
        st = Stats()
        self.check(self.lib.euler_pipeline_run_host(self.h, _p(buf), _p(off), len(off) - 1, int(l), int(flags),
                                                    int(distinct_hint), C.byref(st)))
        return st

    def run_lmers(self, keys, counts, l, flags=0):
        """graph stage on an l-mer table (packed keys, both-strand counts) instead of reads"""
        keys = _arr(keys, np.uint64)
        counts = _arr(counts, np.uint32)
        st = Stats()
        self.check(self.lib.euler_pipeline_run_lmers(self.h, _p(keys), _p(counts), len(keys), int(l), int(flags), C.byref(st)))
        return st

    def run_host_ptr(self, buf_ptr, off_ptr, nreads, l, flags=0, distinct_hint=0):
        """run_host on raw host pointers (e.g. pinned torch tensors)."""
        st = Stats()
        self.check(self.lib.euler_pipeline_run_host(self.h, C.c_void_p(int(buf_ptr)), C.c_void_p(int(off_ptr)), int(nreads),
                                                    int(l), int(flags), int(distinct_hint), C.byref(st)))
        return st

    def download_into(self, which, host_ptr, cap_bytes):
        nb = C.c_uint64(0)
        self.check(self.lib.euler_pipeline_artifact_bytes(self.h, which, C.byref(nb)))
        self.check(self.lib.euler_pipeline_download(self.h, which, C.c_void_p(int(host_ptr)), int(cap_bytes)))
        return nb.value

    def run_dev(self, d_buf, d_off, nreads, n_bases, l, flags=0, distinct_hint=0):
        st = Stats()
        self.check(self.lib.euler_pipeline_run_dev(self.h, C.c_void_p(int(d_buf)), C.c_void_p(int(d_off)), int(nreads),
                                                   int(n_bases), int(l), int(flags), int(distinct_hint), C.byref(st)))
        return st

    def download(self, which):
        nb = C.c_uint64(0)
        self.check(self.lib.euler_pipeline_artifact_bytes(self.h, which, C.byref(nb)))
        dt = np.dtype(_ART_DTYPE[which])
        out = np.zeros(nb.value // dt.itemsize, dt)
        if nb.value:
            self.check(self.lib.euler_pipeline_download(self.h, which, _p(out), nb.value))
        return out

    def device_ptr(self, which):
        p = C.c_void_p()
        self.check(self.lib.euler_pipeline_device_ptr(self.h, which, C.byref(p)))
        return p.value

    def pipeline_contigs(self):
        nb, nc = C.c_uint64(0), C.c_uint64(0)
        self.check(self.lib.euler_pipeline_contigs(self.h, None, C.byref(nb), C.byref(nc)))
        if not nb.value:
            return []
        out = np.zeros(nb.value, np.uint8)
        cap = C.c_uint64(nb.value)
        self.check(self.lib.euler_pipeline_contigs(self.h, _p(out), C.byref(cap), C.byref(nc)))
        return out.tobytes().decode("ascii").split("\n")[:-1]

    # ------------------------------------------------------------------ FASTA / FASTQ ingestion on device
    def ingest(self, data, fmt=0):
        """Parse raw FASTA (fmt=1) / FASTQ (fmt=2) bytes on the GPU (0 = auto); returns (nreads, nbases).
        The reads stay resident for run_ingested / unitigs_ingested / ingest_download."""
        arr = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else _arr(data, np.uint8)
        nr, nb = C.c_uint64(0), C.c_uint64(0)
        self.check(self.lib.euler_ingest(self.h, _p(arr) if arr.size else None, arr.size, int(fmt), C.byref(nr), C.byref(nb)))
        self._ingested = (nr.value, nb.value)
        return nr.value, nb.value

    def ingest_download(self):
        nr, nb = self._ingested
        buf = np.zeros(nb, np.uint8)
        off = np.zeros(nr + 1, np.uint64)
        self.check(self.lib.euler_ingest_download(self.h, _p(buf) if nb else None, _p(off)))
        return buf, off

    def run_ingested(self, l, flags=0, distinct_hint=0):
        st = Stats()
        self.check(self.lib.euler_pipeline_run_ingested(self.h, int(l), int(flags), int(distinct_hint), C.byref(st)))
        return st

    def unitigs_ingested(self, K, limit=1):
        nb, nc = C.c_uint64(0), C.c_uint64(0)
        self.check(self.lib.euler_unitigs_ingested(self.h, int(K), int(limit), None, C.byref(nb), C.byref(nc)))
        if not nb.value:
            return []
        out = np.zeros(nb.value, np.uint8)
        cap = C.c_uint64(nb.value)
        self.check(self.lib.euler_unitigs_ingested(self.h, int(K), int(limit), _p(out), C.byref(cap), C.byref(nc)))
        return out.tobytes().decode("ascii").split("\n")[:-1]

    # ------------------------------------------------------------------ k-mer-space partition
    def dist_count(self, d_buf, d_off, nreads, n_bases, l, nranks):
        counts = np.zeros(nranks + 2, np.uint64)
        self.check(self.lib.euler_dist_count(self.h, C.c_void_p(int(d_buf)), C.c_void_p(int(d_off)), int(nreads),
                                             int(n_bases), int(l), int(nranks), _p(counts)))
        return counts

    def dist_scatter(self, d_buf, d_off, nreads, n_bases, l, nranks, d_send, send_off):
        send_off = _arr(send_off, np.uint64)
        self.check(self.lib.euler_dist_scatter(self.h, C.c_void_p(int(d_buf)), C.c_void_p(int(d_off)), int(nreads),
                                               int(n_bases), int(l), int(nranks), C.c_void_p(int(d_send)), _p(send_off)))

    def dist_scatter_segments(self, d_buf, d_off, nreads, n_bases, l, nranks, d_send, seg_cap):
        counts = np.zeros(nranks + 2, np.uint64)
        self.check(self.lib.euler_dist_scatter_segments(self.h, C.c_void_p(int(d_buf)), C.c_void_p(int(d_off)), int(nreads),
                                                        int(n_bases), int(l), int(nranks), C.c_void_p(int(d_send)),
                                                        int(seg_cap), _p(counts)))
        return counts

    def dist_build(self, d_keys, nkeys, l, rank, nranks, distinct_hint=0):
        st = Stats()
        self.check(self.lib.euler_dist_build(self.h, C.c_void_p(int(d_keys)), int(nkeys), int(l), int(rank), int(nranks),
                                             int(distinct_hint), C.byref(st)))
        return st

    def dist_recv_alloc(self, nkeys):
        """(device pointer, 64-byte CUDA IPC handle) of this rank's peer-visible receive buffer"""
        p = C.c_void_p()
        handle = (C.c_ubyte * 64)()
        self.check(self.lib.euler_dist_recv_alloc(self.h, int(nkeys), C.byref(p), handle))
        return p.value, bytes(handle)

    def dist_peer_open(self, handle):
        p = C.c_void_p()
        buf = (C.c_ubyte * 64).from_buffer_copy(handle)
        self.check(self.lib.euler_dist_peer_open(self.h, buf, C.byref(p)))
        return p.value

    def dist_peer_close(self, ptr):
        self.check(self.lib.euler_dist_peer_close(self.h, C.c_void_p(int(ptr))))

    def dist_scatter_peers(self, d_buf, d_off, nreads, n_bases, l, nranks, dst_ptrs, seg_cap):
        counts = np.zeros(nranks + 2, np.uint64)
        arr = (C.c_void_p * nranks)(*[C.c_void_p(int(x)) for x in dst_ptrs])
        self.check(self.lib.euler_dist_scatter_peers(self.h, C.c_void_p(int(d_buf)), C.c_void_p(int(d_off)), int(nreads),
                                                     int(n_bases), int(l), int(nranks), arr, int(seg_cap), _p(counts)))
        return counts

    def dist_build_regions(self, d_keys, region_stride, region_counts, l, rank, nranks, distinct_hint=0):
        st = Stats()
        rc = _arr(region_counts, np.uint64)
        self.check(self.lib.euler_dist_build_regions(self.h, C.c_void_p(int(d_keys)), int(region_stride), _p(rc), int(l),
                                                     int(rank), int(nranks), int(distinct_hint), C.byref(st)))
        return st

    # ------------------------------------------------------------------ multi-GPU form of the bucketed path
    def bkt_area_alloc(self, which, nranks, scap):
        """(device pointer, 64-byte CUDA IPC handle) of receive area `which` (0 / 1) of this rank: nranks streams of scap records"""
        p = C.c_void_p()
        handle = (C.c_ubyte * 64)()
        self.check(self.lib.euler_bkt_area_alloc(self.h, int(which), int(nranks), int(scap), C.byref(p), handle))
        return p.value, bytes(handle)

    def bkt_scatter(self, d_buf, d_off, nreads, n_bases, l, rank, nranks, nb_per_rank, scap, dst_areas, d_out=None):
        """-> uint64[4]: forward l-mer windows, forward k-mer windows, flags (0x10 = a region overflowed), largest region.
        d_out (device pointer to 4 x u64): asynchronous form, the words stay on the device and None is returned."""
        out = np.zeros(4, np.uint64)
        arr = (C.c_void_p * nranks)(*[C.c_void_p(int(x)) for x in dst_areas])
        self.check(self.lib.euler_bkt_scatter(self.h, C.c_void_p(int(d_buf)), C.c_void_p(int(d_off)), int(nreads), int(n_bases),
                                              int(l), int(rank), int(nranks), int(nb_per_rank), int(scap), arr,
                                              None if d_out else _p(out), C.c_void_p(int(d_out)) if d_out else None))
        return None if d_out else out

    def bkt_build(self, d_area, l, rank, nranks, nb_per_rank, scap, distinct_hint=0):
        st = Stats()
        self.check(self.lib.euler_bkt_build(self.h, C.c_void_p(int(d_area)), int(l), int(rank), int(nranks), int(nb_per_rank),
                                            int(scap), int(distinct_hint), C.byref(st)))
        return st

    def synth_reads_dev(self, d_out, G, L, err_ppm, first, nreads):
        self.check(self.lib.euler_synth_reads_dev(self.h, int(G), int(L), int(err_ppm), int(first), int(nreads),
                                                  C.c_void_p(int(d_out))))


_default_ctx = None


def default_context():
    """Process-wide context on device 0 (the reference's implicit pycuda.autoinit context)."""
    global _default_ctx
    if _default_ctx is None:
        dev = int(os.environ.get("EULER_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        _default_ctx = Context(dev)
    return _default_ctx
