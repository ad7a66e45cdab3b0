"""referenceAssembler -- the reference's CPU k-mer assembler (src/referenceassembler/referenceAssembler.py)
with its hot loops on the GPU.

Same names, arguments and return values as the reference:

* ``build(reads, k=31, limit=1)`` (:25-42)  -> ``dict {kmer: count}`` over both strands, reads split at
  ``N``, entries with ``count <= limit`` dropped.  Counting runs in ``euler_count_mers_wide``; k <= 64.
* ``all_contigs(d, k)`` (:79-111)           -> ``(G, contigs)``.  The unitigs come from
  ``euler_unitigs_from_kmers`` / ``_wide`` (each unitig once, in one of its two orientations; the reference's
  order and orientation follow its dict order, so compare as orientation-free sets), the link graph ``G`` from
  ``euler_unitig_links`` -- for a given contig list it is exactly the reference's ``G``.  k <= 63: the
  library's two-word tables mark an empty slot with all ones, the key of the poly-T 64-mer.
* ``get_contig`` / ``get_contig_forward`` (:47-77), string helpers ``twin kmers fw bw contig_to_string``
  (:7-23, :44-45), ``print_GFA`` / ``print_dbg`` (:115-130), ``runAssembler`` (:135-).

Differences: any non-ACGT byte ends a k-mer window (the reference only splits at ``N``), lower case is
folded to upper case, and ``print_GFA`` / ``print_dbg`` print well-formed records (the reference passes
its format arguments to ``print`` instead of applying them).
"""
import sys

import numpy as np

import _native

_COMP = {'A': 'T', 'C': 'G', 'G': 'C', 'T': 'A'}
_CODE = {'A': 0, 'C': 1, 'G': 2, 'T': 3}


def twin(km):
    """reverse complement (:7-10)"""
    return "".join(_COMP.get(base, base) for base in reversed(km))


def kmers(seq, k):
    for i in range(len(seq) - k + 1):
        yield seq[i:i + k]


def fw(km):
    for x in 'ACGT':
        yield km[1:] + x


def bw(km):
    for x in 'ACGT':
        yield x + km[:-1]


def contig_to_string(c):
    return c[0] + ''.join(x[-1] for x in c[1:])


def _pack(reads):
    data = b"".join(r.encode("ascii") if isinstance(r, str) else bytes(r) for r in reads)
    buf = np.frombuffer(data, dtype=np.uint8) if data else np.zeros(0, np.uint8)
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    if len(reads):
        off[1:] = np.cumsum([len(r) for r in reads], dtype=np.uint64)
    return buf, off


_CODE_OF = np.full(256, 255, np.uint8)
_CODE_OF[np.frombuffer(b"ACGT", np.uint8)] = np.arange(4, dtype=np.uint8)


def _decode(keys, k, keys_hi=None):
    """packed 2-bit keys (MSB first; bits 64.. in keys_hi when k > 32) -> list of strings, vectorised"""
    if len(keys) == 0:
        return []
    shifts = (2 * (k - 1 - np.arange(k))).astype(np.uint64)
    low = shifts < 64
    codes = np.empty((len(keys), k), np.uint8)
    codes[:, low] = (keys[:, None] >> shifts[None, low]) & np.uint64(3)
    if not low.all():
        codes[:, ~low] = (keys_hi[:, None] >> (shifts[None, ~low] - np.uint64(64))) & np.uint64(3)
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[codes]
    return [row.tobytes().decode("ascii") for row in text]


def _encode(kms, k):
    """strings of length k -> (lo, hi): the 2-bit packed keys (MSB first), bits 64.. in hi, vectorised"""
    n = len(kms)
    lo = np.zeros(n, np.uint64)
    hi = np.zeros(n, np.uint64)
    if n == 0:
        return lo, hi
    data = "".join(kms).encode("ascii")
    if len(data) != n * k:
        raise ValueError("every k-mer must have length k = %d" % k)
    codes = _CODE_OF[np.frombuffer(data, np.uint8).reshape(n, k)]
    if (codes == 255).any():
        raise ValueError("k-mers must be spelled in A, C, G, T")
    codes = codes.astype(np.uint64)
    for j in range(k):
        s = 2 * (k - 1 - j)
        if s < 64:
            lo |= codes[:, j] << np.uint64(s)
        else:
            hi |= codes[:, j] << np.uint64(s - 64)
    return lo, hi


def build(reads, k=31, limit=1):
    """referenceAssembler.build (:25-42) on the GPU; k <= 64"""
    reads = list(reads)
    buf, off = _pack(reads)
    if buf.size == 0:
        return {}
    lo, hi, vals = _native.default_context().count_mers_wide(buf, off, int(k), int(limit))
    return dict(zip(_decode(lo, int(k), hi), (int(v) for v in vals)))


def _links_to_G(links):
    G = {}
    for i, row in enumerate(links):
        lists = ([], [])
        for side in (0, 1):
            for b in range(4):
                h, t = int(row[8 * side + 2 * b]), int(row[8 * side + 2 * b + 1])
                if h != 0xFFFFFFFF:
                    lists[side].append((h, '+'))
                if t != 0xFFFFFFFF:
                    lists[side].append((t, '-'))
        G[i] = lists
    return G


def link_graph(contigs, k):
    """the G of all_contigs (:90-111) for a given contig list"""
    contigs = list(contigs)
    return _links_to_G(_native.default_context().unitig_links(contigs, int(k)))


def all_contigs(d, k):
    """referenceAssembler.all_contigs (:79-111): (G, contigs) of the k-mer dictionary d"""
    k = int(k)
    if not d:
        return {}, []
    kms = list(d.keys())
    lo, hi = _encode(kms, k)
    counts = np.fromiter((int(d[x]) for x in kms), dtype=np.uint32, count=len(kms))
    r = _native.default_context().unitigs_from_kmers(lo, counts, k, keys_hi=hi if k > 32 else None)
    return link_graph(r, k), r


_LAST = {"key": None, "contigs": None}


def _contig_with(d, km):
    """(s, i): the unitig of d that contains km, oriented so that s[i:i+k] == km"""
    k = len(km)
    key = (id(d), len(d), k)
    if _LAST["key"] != key:
        _LAST["key"], _LAST["contigs"] = key, all_contigs(d, k)[1]
    for c in _LAST["contigs"]:
        for s in (c, twin(c)):
            i = s.find(km)
            if i >= 0:
                return s, i
    return None, -1


def get_contig_forward(d, km):
    """:59-77 -- the k-mers from km along its unitig, in km's orientation.  km must be a key of d."""
    if km not in d:
        raise ValueError("get_contig_forward: %r is not in the k-mer table" % (km,))
    k = len(km)
    s, i = _contig_with(d, km)
    if s is None:
        return [km]
    nodes = list(kmers(s, k))
    path = nodes[i:]
    first, last = nodes[0], nodes[-1]
    if i > 0:
        # an isolated cycle is written from an arbitrary node: the walk goes on around it, up to the node before km
        nxt = [x for x in fw(last) if x in d]
        if len(nxt) == 1 and nxt[0] == first and first != twin(last) and sum(x in d for x in bw(first)) == 1:
            path += nodes[:i]
    tw = twin(km)
    for j in range(1, len(path)):      # "break out of cycles or mobius contigs" (:68-69)
        if path[j] == tw:
            path = path[:j]
            break
    return path


def get_contig(d, km):
    """:47-56"""
    c_fw = get_contig_forward(d, km)
    c_bw = get_contig_forward(d, twin(km))
    if km in fw(c_fw[-1]):
        c = c_fw
    else:
        c = [twin(x) for x in c_bw[-1:0:-1]] + c_fw
    return contig_to_string(c), c


def write_gfa(G, cs, k, out=None, kc=None):
    """GFA 1.0 records of the link graph (the intent of print_GFA :115-125).  kc: per-contig K-mer count sums; when
    given, every S line ends in the KC:i: tag (total K-mer coverage, which graph viewers such as Bandage read)."""
    out = out or sys.stdout
    out.write("H\tVN:Z:1.0\n")
    for i, x in enumerate(cs):
        if kc is None:
            out.write("S\t%d\t%s\t*\n" % (i, x))
        else:
            out.write("S\t%d\t%s\t*\tKC:i:%d\n" % (i, x, int(kc[i])))
    for i in G:
        for j, o in G[i][0]:
            out.write("L\t%d\t+\t%d\t%s\t%dM\n" % (i, j, o, k - 1))
        for j, o in G[i][1]:
            out.write("L\t%d\t-\t%d\t%s\t%dM\n" % (i, j, o, k - 1))


def write_fasta(cs, out=None):
    out = out or sys.stdout
    for i, x in enumerate(cs):
        out.write('>contig%d\n%s\n' % (i, x))


def print_GFA(G, cs, k):
    write_gfa(G, cs, k, sys.stdout)


def print_dbg(cs):
    write_fasta(cs, sys.stdout)


def runAssembler(k, src):
    """:135- -- build + all_contigs; returns (G, contigs) (the reference only prints the table)"""
    kval = int(k)
    d = build(src, k=kval)
    return all_contigs(d, kval)
