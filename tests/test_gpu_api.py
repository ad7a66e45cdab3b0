"""GPU tests of the reference-facing Python surface (same names / argument order as the reference's
modules), against the oracle and the committed golden fixtures."""
import json
import os

import numpy as np
import pytest

import oracle
from util import check_graph_against_pins, random_reads

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    with open(os.path.join(GOLD, name)) as f:
        return json.load(f)


def _min_rotation(s, k):
    """canonical form of an isolated cycle's contig: the reference starts it at a dict-order
    dependent k-mer (SURVEY §8c.5) -> compare by the minimal rotation of the node cycle."""
    nodes = [s[i:i + k] for i in range(len(s) - k + 1)]
    n = len(nodes)
    best = None
    for r in range(n):
        rot = nodes[r:] + nodes[:r]
        t = rot[0] + "".join(x[-1] for x in rot[1:])
        best = t if best is None or t < best else best
    return best


def _canon_set(contigs, k, d):
    out = []
    for c in contigs:
        first, last = c[:k], c[-k:]
        is_cycle = (last[1:] + first[-1]) == first and first in d  # closes on itself
        forms = [c, oracle.twin(c)]
        if is_cycle:
            forms = [_min_rotation(f, k) for f in forms]
        out.append(min(forms))
    return sorted(out)


@pytest.mark.parametrize("fixture", ["g200.json", "synth_small.json"])
def test_unitigs_match_reference_assembler(ctx, fixture):
    fx = _load(fixture)
    buf, off = oracle.pack_reads(fx["reads"])
    for case in fx["cases"]:
        k, limit = case["k"], case["limit"]
        got = ctx.unitigs(buf, off, k, limit)
        d = {km for km, _ in case["kmers"]}
        assert _canon_set(got, k, d) == _canon_set(case["contigs"], k, d), (fixture, k, limit)


@pytest.mark.parametrize("fixture", ["g200.json", "synth_small.json"])
def test_referenceassembler_module(ctx, fixture):
    """The drop-in `referenceassembler` package against outputs of the unmodified reference module:
    build() tables, all_contigs() contig sets, the link graph G on the reference's own contig lists
    (exact), get_contig() strings (exact) and well-formed GFA / FASTA writers."""
    import io
    import referenceassembler as ra
    from referenceassembler import referenceAssembler as ram
    fx = _load(fixture)
    for case in fx["cases"]:
        k, limit = case["k"], case["limit"]
        d = ra.build(fx["reads"], k, limit)
        assert d == {km: c for km, c in case["kmers"]}, (k, limit)
        G, r = ra.all_contigs(d, k)
        assert _canon_set(r, k, d) == _canon_set(case["contigs"], k, d)
        assert sorted(G) == list(range(len(r)))
        # G is a function of the contig list: on the reference's list it must be the reference's G
        got = ram.link_graph(case["contigs"], k)
        exp = {i: ([tuple(x) for x in lk[0]], [tuple(x) for x in lk[1]]) for i, lk in enumerate(case["links"])}
        assert got == exp, (k, limit)
        for km, text in case["get_contig"]:
            s, c = ra.get_contig(d, km)
            assert s == text and ra.contig_to_string(c) == text and km in c
        out = io.StringIO()
        ram.write_gfa(G, r, k, out)
        lines = out.getvalue().splitlines()
        assert lines[0] == "H\tVN:Z:1.0" and sum(x.startswith("S\t") for x in lines) == len(r)
        assert sum(x.startswith("L\t") for x in lines) == sum(len(a) + len(b) for a, b in G.values())
    assert ra.twin("ACGTN") == "NACGT" and list(ra.fw("ACG")) == ["CGA", "CGC", "CGG", "CGT"]
    assert list(ra.bw("ACG")) == ["AAC", "CAC", "GAC", "TAC"] and list(ra.kmers("ACGT", 3)) == ["ACG", "CGT"]
    with pytest.raises(ValueError):
        ra.get_contig_forward({"ACG": 2, "CGT": 2}, "TTT")


@pytest.mark.parametrize("l", [10, 18, 32])
def test_graph_stage_from_an_lmer_table(ctx, g200_reads, l):
    """euler_pipeline_run_lmers: the graph stage fed with a count table (what the multi-GPU driver joins on one
    rank) gives the artefacts and contigs of the run on the reads themselves."""
    import _native as N
    from util import check_graph_against_pins, random_reads
    reads = g200_reads if l <= 18 else random_reads(9, 300, genome_len=3000)
    buf, off = oracle.pack_reads(reads)
    flags = N.RUN_EXPAND_EDGES | N.RUN_CANONICAL_IDS
    st0 = ctx.run_host(buf, off, l, flags)
    names = ("LMER_KEYS", "LMER_VALUES", "LMER_OFFSETS", "KMER_KEYS", "LCOUNT", "ECOUNT", "LSTART", "ESTART", "EV", "EDGE_V1",
             "EDGE_V2", "EE", "LEV", "ENT")
    a0 = {n: ctx.download(getattr(N, "ART_" + n)) for n in names}
    c0 = ctx.pipeline_contigs()
    lk, lv = a0["LMER_KEYS"], a0["LMER_VALUES"]
    perm = np.random.default_rng(l).permutation(lk.size)
    for keys, vals in ((lk[perm], lv[perm]), (lk, lv)):
        st1 = ctx.run_lmers(keys, vals, l, flags)
        assert (st1.distinct_lmers, st1.distinct_kmers, st1.edge_count) == (st0.distinct_lmers, st0.distinct_kmers, st0.edge_count)
        for n in names:
            assert np.array_equal(ctx.download(getattr(N, "ART_" + n)), a0[n]), n
        assert ctx.pipeline_contigs() == c0
    # one strand per l-mer is enough: the table is canonicalised
    canon = np.array([min(int(x), oracle.revcomp(int(x), l)) == int(x) for x in lk])
    ctx.run_lmers(lk[canon], lv[canon], l, flags)
    assert ctx.pipeline_contigs() == c0


def test_partition_driver_on_one_gpu(tmp_path, g200_reads):
    """assembler.py (SURVEY f4) with world = 1: FASTA + GFA from a FASTQ file in unitig mode, the Euler-mode
    contigs of assemble2 in euler mode; the multi-GPU legs are checked by scripts/check_assembler.sh."""
    import assembler
    import eulercuda.eulercuda as ec
    fq = tmp_path / "reads.fq"
    fq.write_text("".join("@r%d\n%s\n+\n%s\n" % (i, r, "I" * len(r)) for i, r in enumerate(g200_reads)))
    out = tmp_path / "contigs.fa"
    assert assembler.main(["-i", str(fq), "-o", str(out), "-k", "9"]) == 0
    got = [x for x in out.read_text().split("\n") if x and x[0] != ">"]
    fx = _load("g200.json")
    gold = {(c["k"], c["limit"]): c for c in fx["cases"]}
    assert oracle.canonical_contigs(got) == oracle.canonical_contigs(gold[(9, 1)]["contigs"])
    gfa = (tmp_path / "contigs.fa.gfa").read_text().splitlines()
    assert gfa[0] == "H\tVN:Z:1.0" and sum(x.startswith("S\t") for x in gfa) == len(got)
    out2 = tmp_path / "euler.fa"
    assert assembler.main(["-i", str(fq), "-o", str(out2), "-k", "10", "--mode", "euler"]) == 0
    got2 = [x for x in out2.read_text().split("\n") if x and x[0] != ">"]
    assert got2 == ec.assemble2(10, buffer=g200_reads, mode="euler")


def test_assemble_entry_points(tmp_path, g200_reads):
    import eulercuda as ec_pkg
    import eulercuda.eulercuda as ec
    fx = _load("g200.json")
    gold = {(c["k"], c["limit"]): c for c in fx["cases"]}
    # k = 9 (tests/runner.py default) and k = 21 (CLI default -> no k-mers: reads are <= 20 bp)
    for k in (9, 21):
        c = ec.assemble2(k, buffer=g200_reads)
        assert oracle.canonical_contigs(c) == oracle.canonical_contigs(gold[(k, 1)]["contigs"])
    assert ec_pkg.assemble is ec.assemble2
    fa = tmp_path / "r.fa"
    fa.write_text("".join(">r%d\n%s\n" % (i, r) for i, r in enumerate(g200_reads)))
    out = tmp_path / "contigs.txt"
    c = ec.assemble(9, infile=str(fa), outfile=str(out))
    assert oracle.canonical_contigs(c) == oracle.canonical_contigs(gold[(9, 1)]["contigs"])
    txt = out.read_text().split("\n")
    assert txt[0] == ">0" and txt[1] == c[0]
    # Euler mode: the GPU-Euler path of the port
    buf, off = oracle.pack_reads(g200_reads)
    ref, _ = oracle.euler_contigs(buf, off, 10)
    assert ec.assemble2(10, buffer=g200_reads, mode="euler") == ref


def test_orchestrator_functions(g200_reads):
    import eulercuda.eulercuda as ec
    reads = [r for r in g200_reads if len(r) == 20]          # the reference layout: fixed-length reads
    readBuffer = "".join(reads).encode("ascii")
    l = 10
    buf, off = oracle.pack_reads(reads)
    g = oracle.graph_build(buf, off, l, expand=True)
    vals = ec.readLmersKmersCuda(readBuffer, 20, len(readBuffer), l, [], [], 0, [], [], 0, len(reads))
    assert vals[0] == g.nl and vals[1] == g.nv
    assert np.array_equal(vals[2], g.lk_lo) and np.array_equal(vals[3], g.lvals)
    assert np.array_equal(vals[4], g.vk_lo) and np.array_equal(vals[5], np.arange(g.nv))
    ee, ev, lev, ent, vcount, ecount = ec.constructDebruijnGraph(readBuffer, len(readBuffer), 20, l, [], [], [], [],
                                                                 len(reads))
    assert (vcount, ecount) == (g.nv, g.ne)
    assert np.array_equal(ee, g.ee) and np.array_equal(ev, g.ev)
    assert np.array_equal(lev, g.lev) and np.array_equal(ent, g.ent)
    contigs = ec.findEulerTour(ev, ee, lev, ent, ecount, vcount, l, "")
    ref, _ = oracle.euler_contigs(buf, off, l)
    assert contigs == ref
    assert ec.getString(4, 27) == "ACGT" and ec.getString(10, 959244) == "TGGGATAATA"


def test_module_level_chain(g200_reads):
    """The reference's own call sequence through the L3 modules (eulercuda.py:237-262)."""
    import eulercuda.pyencode as enc
    import eulercuda.pygpuhash as gh
    import eulercuda.pydebruijn as db
    import eulercuda.pyeulertour as et
    import eulercuda.pycomponent as comp
    reads = [r for r in g200_reads if len(r) == 20]
    flat = np.array("".join(reads).encode("ascii")).astype("S")
    B, l, RL = 20 * len(reads), 12, 20
    buf, off = oracle.pack_reads(reads)
    f0, r0, v0 = oracle.encode_positions(buf, off, l)
    lm = enc.encode_lmer_device(flat, B, np.zeros(B, np.uint64), RL, l)
    assert np.array_equal(lm, f0)
    assert np.array_equal(enc.compute_lmer_complement_device(flat, B, np.zeros(B, np.uint64), RL, l), r0)
    assert np.array_equal(enc.valid_window_mask(flat, RL, l), v0)
    mask = (1 << (2 * (l - 1))) - 1
    pk, sk = enc.compute_kmer_device(lm, None, None, mask, RL, B)
    assert np.array_equal(pk, f0 >> np.uint64(2)) and np.array_equal(sk, f0 & np.uint64(mask))
    assert enc.getOptimalLaunchConfiguration(100000, 512) == ((512, 1, 1), (1, 196, 1))
    assert enc.getOptimalLaunchConfiguration(10, 32) == ((32, 1, 1), (1, 1, 1))

    g = oracle.graph_build(buf, off, l, expand=True)
    tl, bsz, bc, TK, TV = gh.create_hash_table_device(g.vk_lo, np.arange(g.nv, dtype=np.uint32), g.nv, [], [], 0, [], 0)
    assert tl == TK.size
    assert np.array_equal(gh.get_hash_value(g.vk_lo, TK, TV), np.arange(g.nv))
    assert gh.get_hash_value([12345678901234], TK, TV)[0] == 0xFFFFFFFF
    ee, ev, lev, ent, nk, ne = db.construct_debruijn_graph_device(g.lk_lo, g.lvals, g.nl, g.vk_lo, g.nv, l, TK, TV, bsz, bc,
                                                                  [], [], [], [], RL)
    assert (nk, ne) == (g.nv, g.ne)
    assert np.array_equal(ee, g.ee) and np.array_equal(ev, g.ev) and np.array_equal(lev, g.lev) and np.array_equal(ent, g.ent)
    lc, ec_ = db.debruijn_count_device(g.lk_lo, g.lvals, g.nl, TK, TV, bsz, bc, np.zeros(4 * g.nv, np.uint32),
                                       np.zeros(4 * g.nv, np.uint32), mask, RL)
    assert np.array_equal(lc, g.lcount) and np.array_equal(ec_, g.ecount)

    _, ee1 = et.assign_successor_device(ev, lev, ent, nk, ee, ne)
    ee0 = oracle.assign_successor(g.ev, g.lev, g.ent, g.ee)
    assert np.array_equal(ee1, ee0)
    v = et.construct_successor_graphP2_device(ee1, et.construct_successor_graphP1_device(ee1, None, ne), ne)
    assert np.array_equal(v, oracle.successor_graph(ee0))
    D = comp.find_component_device(v, np.zeros(ne, np.uint32), ne)
    assert np.array_equal(D, oracle.components(v))
    cg, ncg, ncirc = et.findEulerDevice(ev, lev, ent, nk, ee, ne, {}, 0, 0)
    C0, off0, cv0, n0 = oracle.circuit_vertices(D)
    assert ncirc == n0
    cg0 = oracle.circuit_edges(g.ev, g.ent, D, off0)
    assert np.array_equal(cg, cg0) and ncg == len(cg0)
    assert np.array_equal(et.identify_contig_start(ee1, None, ne), oracle.contig_starts(ee0))


def test_sv_substeps_reach_the_union_find_labels():
    """The step-level Shiloach-Vishkin wrappers, driven to their fix-point (B8 repaired), give the
    same labels as find_component_device: the minimum node id per component."""
    import eulercuda.pycomponent as comp
    import _native
    rng = np.random.default_rng(5)
    n = 3000
    perm = rng.permutation(n).astype(np.uint32)
    v = np.zeros(n, _native.SV_DTYPE)
    v["vid"] = np.arange(n)
    v["n1"] = n
    v["n2"] = n
    # chains and cycles of random lengths
    i = 0
    while i < n:
        ln = int(rng.integers(1, 60))
        seg = perm[i:i + ln]
        for a, b in zip(seg[:-1], seg[1:]):
            v["n1"][a] = b
            v["n2"][b] = a
        if len(seg) > 2 and rng.random() < 0.3:
            v["n1"][seg[-1]] = seg[0]
            v["n2"][seg[0]] = seg[-1]
        i += ln
    want = comp.find_component_device(v, None, n)
    assert np.array_equal(want, oracle.components(v))
    D, Q = comp.component_step_init(v, None, None, n)
    prevD = np.zeros(n, np.uint32)
    z = np.zeros(n, np.uint32)
    s = 1
    for _ in range(200):
        prevD, D = D, prevD
        D = comp.component_step1_shortcutting_p1(v, prevD, D, Q, n, s)
        Q = comp.component_step1_shortcutting_p2(v, prevD, D, Q, n, s)
        t1, t2, v1, v2 = comp.component_Step2_P1(v, prevD, D, Q, z, z, z, z, n, s)
        D, Q = comp.component_Step2_P2(v, prevD, D, Q, t1, v1, t2, v2, n, s)
        t1, t2, v1, v2 = comp.component_Step3_P1(v, prevD, D, Q, z, z, z, z, n, s)
        D = comp.component_Step3_P2(v, prevD, D, Q, t1, v1, t2, v2, n, s)
        val1 = comp.component_step4_P1(v, D, z, n)
        D = comp.component_step4_P2(v, D, val1, n)
        again = comp.component_step5(Q, n, None, s)
        s += 1
        if not again:
            break
    assert np.array_equal(D, want)


def test_legacy_bucket_phases():
    """pygpuhash phase1 -> scan -> copy_to_bucket -> bucket_sort keeps every (key, value) and sorts
    each bucket ascending (reference layout, 520-slot buckets)."""
    import eulercuda.pygpuhash as gh
    import _native
    rng = np.random.default_rng(3)
    keys = np.unique(rng.integers(0, 1 << 40, 5000, dtype=np.uint64))
    vals = np.arange(keys.size, dtype=np.uint32)
    n = keys.size
    bc = n // 409 + 1                                   # pygpuhash.py:274
    offset, count = gh.phase1_device(keys, None, n, None, bc)
    hb = np.array([gh.hash_h(k, bc) for k in keys])
    assert np.array_equal(count, np.bincount(hb, minlength=bc))
    for b in range(bc):
        assert sorted(offset[hb == b]) == list(range(count[b]))
    start = _native.default_context().exclusive_scan(count)
    bk, bv = gh.copy_to_bucket_device(keys, vals, offset, n, start, bc, None, None)
    assert sorted(zip(bk.tolist(), bv.tolist())) == sorted(zip(keys.tolist(), vals.tolist()))
    TK, TV = gh.bucket_sort_device(bk, bv, start, count, bc, None, None)
    for b in range(bc):
        seg = TK[b * 520:b * 520 + count[b]]
        assert np.array_equal(seg, np.sort(keys[hb == b]))
        assert np.array_equal(keys[TV[b * 520:b * 520 + count[b]]], seg)
    assert gh.hash_h(959244, 409) == 22 and gh.hash_h(0, 409) == 96 and gh.hash_h(27, 409) == 76


def test_medium_scale_properties(ctx):
    """200k reads: size-independent properties (edge conservation, degree balance, scan totals)
    plus full parity with the oracle at this still-cheap size."""
    import _native as N
    G, L, l = 300000, 100, 32
    buf = oracle.synth_reads(G, L, cov=20, err_ppm=5000)
    n = buf.size // L
    off = oracle.fixed_offsets(n, L)
    st = ctx.run_host(buf, off, l, N.RUN_CANONICAL_IDS | N.RUN_EXPAND_EDGES)
    lv = ctx.download(N.ART_LMER_VALUES)
    ev = ctx.download(N.ART_EV)
    assert int(lv.sum()) == st.edge_count == 2 * st.n_lmer_windows == 2 * n * (L - l + 1)
    assert int(ev["lcount"].sum()) == st.edge_count and int(ev["ecount"].sum()) == st.edge_count
    ee = ctx.download(N.ART_EE)
    assert np.array_equal(np.sort(ctx.download(N.ART_LEV)), np.arange(st.edge_count))
    assert np.array_equal(np.bincount(ee["v1"], minlength=len(ev)), ev["lcount"])
    assert np.array_equal(np.bincount(ee["v2"], minlength=len(ev)), ev["ecount"])
    g = oracle.graph_build(buf, off, l, expand=True)
    assert np.array_equal(ev, g.ev) and np.array_equal(ee, g.ee)
    contigs = ctx.pipeline_contigs()
    ref, _ = oracle.euler_contigs(buf, off, l)
    assert contigs == ref
    # reverse-complement closure of the edge multiset
    lk = ctx.download(N.ART_LMER_KEYS)
    d = dict(zip(lk.tolist(), lv.tolist()))
    for x in lk[:2000].tolist():
        assert d[oracle.revcomp(x, l)] == d[x]


def test_errors_are_loud(ctx):
    import _native as N
    buf, off = oracle.pack_reads(["ACGTACGTACGT"])
    with pytest.raises(N.EulerError):
        ctx.run_host(buf, off, 65)          # l > 64 does not fit two key words
    with pytest.raises(N.EulerError):
        ctx.run_host(buf, off, 1)
    with pytest.raises(N.EulerError):
        N.Context(99)
    c2 = N.Context(0)
    with pytest.raises(N.EulerError):
        c2.download(N.ART_EV)               # no run yet
    c2.run_host(buf, off, 4)
    with pytest.raises(N.EulerError):
        c2.download(N.ART_EE)               # edges were not expanded
    c2.close()


def test_full_size_config2_properties_and_parity(ctx):
    """BASELINE.json configs[1] at full size (4.6 Mbp, 100 bp, 30x, k = 31; 96.6 M k-mer windows), reads
    generated on device: size-independent properties of the fast path, then full parity of the l-mer
    and vertex tables with the oracle on the same reads."""
    import torch
    import _native as N
    G, L, cov, l = 4_600_000, 100, 30, 32
    R = G * cov // L
    d = torch.empty(R * L, dtype=torch.uint8, device="cuda")
    ctx.synth_reads_dev(d.data_ptr(), G, L, 0, 0, R)
    offs = torch.arange(R + 1, dtype=torch.int64, device="cuda") * L
    ctx.sync()
    torch.cuda.synchronize()
    st = ctx.run_dev(d.data_ptr(), offs.data_ptr(), R, R * L, l, 0, G)
    assert st.n_kmer_windows == R * (L - l + 2) and st.n_lmer_windows == R * (L - l + 1)
    assert st.edge_count == 2 * st.n_lmer_windows
    lk, lv = ctx.download(N.ART_LMER_KEYS), ctx.download(N.ART_LMER_VALUES)
    ev = ctx.download(N.ART_EV)
    assert int(lv.sum(dtype=np.uint64)) == st.edge_count
    assert int(ev["lcount"].sum(dtype=np.uint64)) == st.edge_count == int(ev["ecount"].sum(dtype=np.uint64))
    lo = ctx.download(N.ART_LMER_OFFSETS)
    assert lo[0] == 0 and int(lo[-1]) + int(lv[-1]) == st.edge_count
    v1, v2 = ctx.download(N.ART_EDGE_V1), ctx.download(N.ART_EDGE_V2)
    kmask = np.uint64((1 << 62) - 1)
    assert np.array_equal(ev["vid"][v1], lk >> np.uint64(2)) and np.array_equal(ev["vid"][v2], lk & kmask)
    # leaving multiplicity per vertex = sum over its edges (checksum of checksums)
    assert np.array_equal(np.bincount(v1, weights=lv, minlength=len(ev)).astype(np.uint64), ev["lcount"].astype(np.uint64))
    assert np.array_equal(np.bincount(v2, weights=lv, minlength=len(ev)).astype(np.uint64), ev["ecount"].astype(np.uint64))
    # parity with the oracle at full size
    buf = d.cpu().numpy()
    g = oracle.graph_build(buf, oracle.fixed_offsets(R, L), l, expand=False)
    assert (st.distinct_lmers, st.distinct_kmers, st.edge_count) == (g.nl, g.nv, g.ne)
    o = np.argsort(lk, kind="stable")
    assert np.array_equal(lk[o], g.lk_lo) and np.array_equal(lv[o], g.lvals)
    ov = np.argsort(ev["vid"], kind="stable")
    assert np.array_equal(ev["vid"][ov], g.vk_lo)
    assert np.array_equal(ev["lcount"][ov], g.ev["lcount"]) and np.array_equal(ev["ecount"][ov], g.ev["ecount"])


def test_device_ingestion_matches_the_reference_readers(ctx, tmp_path, g200_reads):
    """FASTA / FASTQ parsed on the GPU == eulercuda.read_fasta / read_fastq (host restatements of the
    reference readers), including blank lines, CRLF, a missing final newline and multi-line records."""
    import eulercuda.eulercuda as ec
    cases = {
        "g200.fa": "".join(">r%d\n%s\n" % (i, r) for i, r in enumerate(g200_reads)),
        "odd.fa": ">a desc\nACGT\nTTGA\n\n>b\nCC\r\n>c\nGGNNA",          # multi-line, blank line, CRLF, no final newline
        "only_headers.fa": ">x\n>y\n",
        "r.fq": "".join("@q%d\n%s\n+\n%s\n" % (i, r, "I" * len(r)) for i, r in enumerate(g200_reads[:40])),
        "tail.fastq": "@a\nACGTACGT\n+\nIIIIIIII\n@b\nTTTT\n+\nIIII",
    }
    for name, text in cases.items():
        p = tmp_path / name
        p.write_bytes(text.encode("ascii"))
        fq = name.endswith(("fq", "fastq"))
        want = ec.read_fastq(str(p)) if fq else ec.read_fasta(str(p))
        nr, nb = ctx.ingest(text.encode("ascii"), 2 if fq else 1)
        buf, off = ctx.ingest_download()
        got = [buf[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(nr)]
        assert got == want, name
        assert ctx.ingest(text.encode("ascii"), 0)[0] == nr      # auto-detection
    # whole path from a file: ingestion on device -> unitigs / Euler contigs
    fa = tmp_path / "g200.fa"
    fx = _load("g200.json")
    gold = {(c["k"], c["limit"]): c for c in fx["cases"]}
    c = ec.assemble2(11, infile=str(fa))
    assert oracle.canonical_contigs(c) == oracle.canonical_contigs(gold[(11, 1)]["contigs"])
    b, o = oracle.pack_reads(g200_reads)
    ref, _ = oracle.euler_contigs(b, o, 12)
    assert ec.assemble2(12, infile=str(fa), mode="euler") == ref


@pytest.mark.parametrize("name", ["g200", "synth_small"])
def test_graph_equals_the_reference_derived_pins(ctx, name):
    """The GPU path's vertex set, degree arrays, edge multiset and edge end points against pins derived from the
    unmodified reference's build(reads, l, 0) + fw / bw (tests/golden/graph_pins.json) -- independent of the oracle."""
    import _native as N
    reads = _load("g200.json" if name == "g200" else "synth_small.json")["reads"]
    buf, off = oracle.pack_reads(reads)
    for pin in _load("graph_pins.json")[name]:
        ctx.run_host(buf, off, pin["l"], N.RUN_CANONICAL_IDS)
        check_graph_against_pins(pin, ctx.download(N.ART_KMER_KEYS), ctx.download(N.ART_LCOUNT), ctx.download(N.ART_ECOUNT),
                                 ctx.download(N.ART_LMER_KEYS), ctx.download(N.ART_LMER_VALUES), ctx.download(N.ART_EDGE_V1),
                                 ctx.download(N.ART_EDGE_V2), oracle.decode_key)


def test_bench_dump_outputs_equal_the_oracle(tmp_path):
    """bench.py --dump-outputs on the small workload: the files hold the graph of the oracle on the same reads, and a
    second run with the same arguments writes the same files."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for run in ("a", "b"):
        subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "small_smoke", "--steps", "2", "--warmup", "1",
                        "--no-e2e", "--no-cpu", "--no-extra", "--dump-outputs", str(tmp_path / run)], check=True, timeout=600,
                       capture_output=True)
    d = {}
    for n in sorted(os.listdir(tmp_path / "a")):
        a = np.load(tmp_path / "a" / n)
        assert a.dtype == np.float64 and np.array_equal(a, np.load(tmp_path / "b" / n)), n
        d[n[:-4]] = a.astype(np.uint64)
    G, L, cov, l = 200_000, 100, 20, 32             # bench.py WORKLOADS["small_smoke"]
    R = G * cov // L
    g = oracle.graph_build(oracle.synth_reads(G, L, err_ppm=0, first=0, count=R), oracle.fixed_offsets(R, L), l, expand=False)
    assert d["counts"].tolist() == [R * (L - l + 2), R * (L - l + 1), g.nl, g.nv, g.ne]
    lr, vr = d["lmer_rows"], d["kmer_rows"]
    assert lr.size == min(g.nl, 1 << 18) and vr.size == min(g.nv, 1 << 18)
    assert np.array_equal(d["lmer_keys"], np.stack([g.lk_lo >> np.uint64(32), g.lk_lo & np.uint64(0xFFFFFFFF)], axis=1)[lr])
    assert np.array_equal(d["lmer_values"], g.lvals[lr])
    assert np.array_equal(d["edge_v1"], g.ev1[lr]) and np.array_equal(d["edge_v2"], g.ev2[lr])
    assert np.array_equal(d["kmer_keys"], np.stack([g.vk_lo >> np.uint64(32), g.vk_lo & np.uint64(0xFFFFFFFF)], axis=1)[vr])
    assert np.array_equal(d["lcount"], g.lcount.reshape(-1, 4)[vr]) and np.array_equal(d["ecount"], g.ecount.reshape(-1, 4)[vr])
