"""The de Bruijn graph build held to the oracle array for array at the sizes the benchmark runs: BASELINE.json configs[1]
(4.6 Mbp, 100 bp, 30x) with and without read errors, every template instantiation of the bucketed build, the
global-table path and the routing between the two, the second pass, every regrow branch of the bucketed and the wide
build, contexts reused across sizes, l and entry points, 128-bit keys, a ragged input, and the partitioned build.

Cases that need an environment knob (read once per process) run in a child process, which prints its verdict or the
first mismatching array and index.  Every case asserts the branch it exists for (stats.path, redo_buckets, retries,
n_buckets)."""
import gc
import os
import resource
import subprocess
import sys

import numpy as np
import pytest

import oracle
from graph_scale import assert_counts, assert_graph_canonical, assert_graph_label_free, assert_partitioned
from util import random_reads

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G2, L2 = 4_600_000, 100          # BASELINE.json configs[1]
M = 1_000_000                    # the 1 Mbp sets: 100 bp (l <= 32) and 150 bp (128-bit keys), 30x, 1 % errors
ERR = 10000

_ORACLE = {}


def oracle_graph(name, buf, off, l, expand):
    """oracle.graph_build, keeping the last graph only (one full-scale graph with errors takes ~20 GB of host RAM)"""
    key = (name, l, expand)
    if key not in _ORACLE:
        _ORACLE.clear()
        gc.collect()
        _ORACLE[key] = oracle.graph_build(buf, off, l, expand=expand)
    return _ORACLE[key]


def host_reads(G, L, err, cov=30):
    R = G * cov // L
    return oracle.synth_reads(G, L, err_ppm=err, first=0, count=R), oracle.fixed_offsets(R, L), R


def dev_reads(ctx, G, L, err, cov=30, count=None):
    """the same reads as host_reads, generated on the device (test_gpu_core.py::test_synth_reads_match_oracle)"""
    import torch
    R = count or G * cov // L
    d = torch.empty(R * L, dtype=torch.uint8, device="cuda")
    ctx.synth_reads_dev(d.data_ptr(), G, L, err, 0, R)
    offs = torch.arange(R + 1, dtype=torch.int64, device="cuda") * L
    ctx.sync()
    torch.cuda.synchronize()
    return d, offs, R


def run(ctx, dev, L, l, flags, hint=0):
    d, offs, R = dev
    return ctx.run_dev(d.data_ptr(), offs.data_ptr(), R, R * L, l, flags, hint)


def report(tag, st):
    print("%s: path %d, buckets %d, redo %d, retries %d, U_l %d, V %d, host maxrss %.1f GB (children %.1f GB)" % (
        tag, st.path, st.n_buckets, st.redo_buckets, st.retries, st.distinct_lmers, st.distinct_kmers,
        resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6, resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss / 1e6))


_CHILD = r'''
import sys, time, traceback
sys.path.insert(0, %r); sys.path.insert(0, %r); sys.path.insert(0, %r)
import numpy as np, oracle, _native as N
import test_gpu_graph_scale as T
from graph_scale import *
ctx = N.Context(0)
t0 = time.time()
try:
%s
except AssertionError as e:
    print("MISMATCH: %%s" %% e)
    traceback.print_exc()
    sys.exit(1)
print("%%.0f s" %% (time.time() - t0))
print("ok")
'''


def run_child(body, **env):
    _ORACLE.clear()
    gc.collect()
    code = _CHILD % (ROOT, os.path.join(ROOT, "pycuda-euler_b200"), os.path.join(ROOT, "tests"),
                     "\n".join("    " + x for x in body.strip("\n").splitlines()))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=1500)
    print(out.stdout)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout[-3000:] + out.stderr[-3000:]


@pytest.fixture(scope="module")
def gctx():
    """A context of this module's own: the runs here grow its buffers to configs[1] size, and closing it (and emptying
    torch's cache of the read buffers) hands that memory back before the next module runs."""
    import torch
    import _native as N
    c = N.Context(0)
    yield c
    c.close()
    _ORACLE.clear()
    torch.cuda.empty_cache()


C = 2   # N.RUN_CANONICAL_IDS
X = 1   # N.RUN_EXPAND_EDGES


# ---- configs[1] at full size: the bucketed build, its three template instantiations -----------------------------------
@pytest.mark.parametrize("err,l", [(0, 32), (0, 22), (0, 27), (ERR, 22), (ERR, 27), (ERR, 32)])
def test_bucketed_build_full_scale(gctx, err, l):
    dev = dev_reads(gctx, G2, L2, err)
    st = run(gctx, dev, L2, l, C, G2)
    assert st.path == 1
    buf, off, _ = host_reads(G2, L2, err)
    g = oracle_graph(("configs1", err), buf, off, l, False)
    assert_counts(st, g)
    assert_graph_canonical(gctx, g, False)
    report("configs[1] err %d l %d canonical" % (err, l), st)
    if err and l == 32:
        st = run(gctx, dev, L2, l, 0, G2)
        assert st.path == 1
        assert_counts(st, g)
        assert_graph_label_free(gctx, g, False)
        report("configs[1] err %d l %d slot order" % (err, l), st)


def test_routing_on_a_fresh_context():
    """No hint on a fresh context: the distinct count is estimated from the base count (1.38e8 > the bucketed limit), so
    the first run takes the global-table path; the second run of the same reads uses what the first counted and takes
    the bucketed path.  Both are exact."""
    import _native as N
    c = N.Context(0)
    try:
        dev = dev_reads(c, G2, L2, ERR)
        buf, off, _ = host_reads(G2, L2, ERR)
        g = oracle_graph(("configs1", ERR), buf, off, 32, False)
        for want_path in (0, 1):
            st = run(c, dev, L2, 32, C)
            assert st.path == want_path
            assert_counts(st, g)
            assert_graph_canonical(c, g, False)
            report("fresh context, no hint", st)
    finally:
        c.close()


def test_second_pass_full_scale(gctx):
    """The buckets sized from the exact distinct count: with 1 % errors some of them overflow the first pass's tables
    and are rebuilt by the second."""
    buf, off, _ = host_reads(G2, L2, ERR)
    g = oracle_graph(("configs1", ERR), buf, off, 32, False)
    st = run(gctx, dev_reads(gctx, G2, L2, ERR), L2, 32, C, (g.nl + 1) // 2)
    assert st.path == 1 and st.redo_buckets > 0
    assert_counts(st, g)
    assert_graph_canonical(gctx, g, False)
    report("hint = distinct count", st)


def test_global_table_path_full_scale():
    run_child('''
dev = T.dev_reads(ctx, T.G2, T.L2, T.ERR)
st = T.run(ctx, dev, T.L2, 32, N.RUN_CANONICAL_IDS, T.G2)
assert st.path == 0
buf, off, _ = T.host_reads(T.G2, T.L2, T.ERR)
g = oracle.graph_build(buf, off, 32, expand=False)
assert_counts(st, g)
assert_graph_canonical(ctx, g, False)
T.report("EULER_B200_BUCKETED=0", st)
''', EULER_B200_BUCKETED="0")


def test_small_tables_full_scale():
    """256-slot tables at load 0.6 on configs[1] with 1 % errors: more buckets overflow than the second pass takes
    (BKT_REDO_CAP), more buckets do not help the ones that hold a few heavy minimizers, and the build falls back to the
    global-table path -- exact all the same."""
    run_child('''
buf, off, _ = T.host_reads(T.G2, T.L2, T.ERR)
g = oracle.graph_build(buf, off, 32, expand=False)
dev = T.dev_reads(ctx, T.G2, T.L2, T.ERR)
st = T.run(ctx, dev, T.L2, 32, N.RUN_CANONICAL_IDS, (g.nl + 1) // 2)
assert st.path == 0, st.path
assert_counts(st, g)
assert_graph_canonical(ctx, g, False)
T.report("BKT_CAP=256 BKT_LOAD=0.6", st)
''', EULER_B200_BKT_CAP="256", EULER_B200_BKT_LOAD="0.6")


def test_forced_bucketed_build_above_the_limit():
    """EULER_B200_BUCKETED=2 on configs[1] at 3 % errors: more distinct canonical l-mers than the bucketed path takes by
    default (5e7).  The graph of this size is checked against the oracle's count tables (the full oracle graph would
    need ~45 GB of host RAM): the l-mer multiset and the vertex set exactly, and every other artefact exactly as
    derived from them (derived_graph, itself checked against the oracle graph in tests/test_cpu_graph_scale.py)."""
    run_child('''
dev = T.dev_reads(ctx, T.G2, T.L2, 30000)
t = time.time()
st = T.run(ctx, dev, T.L2, 32, N.RUN_CANONICAL_IDS, 0)
print("forced bucketed build: %.1f s including the first-run allocations" % (time.time() - t))
assert st.path == 1
del dev
buf, off, _ = T.host_reads(T.G2, T.L2, 30000)
lk, _, lv = oracle.count_mers(buf, off, 32)
print("distinct both-strand 32-mers: %d" % lk.size)
assert lk.size // 2 > 50_000_000       # canonical distinct = (both-strand + palindromes) / 2
same("LMER_KEYS", ctx.download(N.ART_LMER_KEYS), lk)
same("LMER_VALUES", ctx.download(N.ART_LMER_VALUES), lv)
vk = oracle.count_mers(buf, off, 31)[0]      # no N, every read >= l: the vertices are all the 31-mers
del buf
same("KMER_KEYS", ctx.download(N.ART_KMER_KEYS), vk)
assert (st.distinct_lmers, st.distinct_kmers, st.edge_count) == (lk.size, vk.size, int(lv.sum(dtype=np.uint64)))
exp = derived_graph(lk, lv, vk, 32)
del lk, lv, vk
for name, a in exp.items():
    same(name, ctx.download(getattr(N, "ART_" + name)), a)
T.report("EULER_B200_BUCKETED=2, 3 percent errors", st)
''', EULER_B200_BUCKETED="2")


# ---- regrow branches and context reuse at 1 Mbp ----------------------------------------------------------------------
def test_output_and_region_regrow_on_one_context():
    """OUTPUT: the capacities learned from error-free reads are too small for reads with errors of the same base count.
    REGION: the record regions learned from a varied input overflow on one of the same base count whose records pile
    into few buckets (an error-free 20 kbp genome at 1,500x)."""
    import _native as N
    c = N.Context(0)
    try:
        R = M * 30 // L2
        for tag, G, err, want_retry in (("error-free", M, 0, False), ("1 % errors", M, ERR, True), ("20 kbp at 1500x", 20_000, 0, True)):
            dev = dev_reads(c, G, L2, err, count=R)
            st = run(c, dev, L2, 32, C)
            assert st.path == 1
            if want_retry:
                assert st.retries > 0, tag
            buf = oracle.synth_reads(G, L2, err_ppm=err, first=0, count=R)
            g = oracle_graph(("regrow", G, err), buf, oracle.fixed_offsets(R, L2), 32, False)
            assert_counts(st, g)
            assert_graph_canonical(c, g, False)
            report(tag, st)
    finally:
        c.close()


def test_table_regrow():
    """TABLE: 64 buckets for 6.5e6 distinct canonical l-mers: the shared-memory tables fill up and the input is
    partitioned again into 4x the buckets until it fits."""
    run_child('''
dev = T.dev_reads(ctx, T.M, T.L2, T.ERR)
st = T.run(ctx, dev, T.L2, 32, N.RUN_CANONICAL_IDS, 0)
assert st.path == 1 and st.n_buckets > 64 and st.retries > 0, (st.path, st.n_buckets, st.retries)
buf, off, _ = T.host_reads(T.M, T.L2, T.ERR)
g = oracle.graph_build(buf, off, 32, expand=False)
assert_counts(st, g)
assert_graph_canonical(ctx, g, False)
T.report("BKT_NB=64", st)
''', EULER_B200_BKT_NB="64")


def _fasta(buf, R, L):
    rec = np.empty((R, L + 3), np.uint8)
    rec[:, 0], rec[:, 1] = ord(">"), ord("\n")
    rec[:, 2:L + 2] = buf.reshape(R, L)
    rec[:, L + 2] = ord("\n")
    return rec.tobytes()


def test_one_context_through_sizes_orders_lengths_and_entry_points():
    """One context: big canonical expanded, small in slot order, big in slot order, l = 22 / 64 / 31 / 32, a run from an
    l-mer table in between, and run_host / run_dev / run_ingested on the same reads; Euler contigs after every
    expanded run.  Every result equals the oracle's (hence the fresh-context result)."""
    import _native as N
    c = N.Context(0)
    try:
        buf, off, R = host_reads(M, L2, ERR)
        dev = dev_reads(c, M, L2, ERR)
        g = oracle_graph("1mbp", buf, off, 32, True)
        st = run(c, dev, L2, 32, C | X)
        assert_counts(st, g)
        assert_graph_canonical(c, g, False)
        contigs, _ = oracle.euler_contigs(buf, off, 32)   # the tour kernels at 4.1e7 edges
        assert c.pipeline_contigs() == contigs
        report("big canonical expanded", st)
        sreads = random_reads(7, 2000, genome_len=20000)
        sbuf, soff = oracle.pack_reads(sreads)
        gs = oracle.graph_build(sbuf, soff, 32, expand=False)
        st = c.run_host(sbuf, soff, 32, 0)
        assert_counts(st, gs)
        assert_graph_label_free(c, gs, False)
        st = run(c, dev, L2, 32, 0)
        assert_counts(st, g)
        assert_graph_label_free(c, g, False)
        report("big slot order", st)
        for l in (22, 64, 31, 32):
            gl = g if l == 32 else oracle.graph_build(buf, off, l, expand=False)
            st = run(c, dev, L2, l, C | X if l == 32 else C)
            assert_counts(st, gl)
            assert_graph_canonical(c, gl, l > 32)
            if l == 22:   # the graph stage from the l-mer table, between two runs on reads
                st = c.run_lmers(gl.lk_lo, gl.lvals, 22, C)
                assert_counts(st, gl)
                assert_graph_canonical(c, gl, False)
            if l == 32:
                assert c.pipeline_contigs() == contigs
            report("l %d" % l, st)
            del gl
        for entry in ("host", "dev", "ingested"):
            if entry == "host":
                st = c.run_host(buf, off, 32, C | X)
            elif entry == "dev":
                st = run(c, dev, L2, 32, C | X)
            else:
                assert c.ingest(_fasta(buf, R, L2), 1) == (R, R * L2)
                st = c.run_ingested(32, C | X)
            assert_counts(st, g)
            assert_graph_canonical(c, g, False)
            assert c.pipeline_contigs() == contigs, entry
            report("run_" + entry, st)
    finally:
        c.close()


# ---- 128-bit keys at 1 Mbp --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("l", [64, 48, 33])
def test_wide_build_1mbp(gctx, l):
    buf, off, _ = host_reads(M, 150, ERR)
    dev = dev_reads(gctx, M, 150, ERR)
    g = oracle_graph("1mbp150", buf, off, l, True)
    st = run(gctx, dev, 150, l, C | X)
    assert_counts(st, g)
    assert_graph_canonical(gctx, g, True)
    if l == 64:
        contigs, _ = oracle.euler_contigs(buf, off, 64)
        assert gctx.pipeline_contigs() == contigs
    st = run(gctx, dev, 150, l, 0)
    assert_counts(st, g)
    assert_graph_label_free(gctx, g, True)
    report("wide l %d" % l, st)


def test_wide_regrow_on_one_context():
    """The learned table sizes of the wide path are keyed on the base count only: l = 33 after l = 64 on the same reads
    starts from the size learned at l = 64; a hint of 64 regrows the tables (in one step: the window count bounds the
    distinct count)."""
    import _native as N
    c = N.Context(0)
    try:
        buf, off, _ = host_reads(M, 150, ERR)
        dev = dev_reads(c, M, 150, ERR)
        run(c, dev, 150, 64, C)
        g = oracle_graph("1mbp150", buf, off, 33, False)
        for hint in (0, 64):
            st = run(c, dev, 150, 33, C, hint)
            if hint:
                assert st.retries > 0
            assert_counts(st, g)
            assert_graph_canonical(c, g, True)
            report("wide l 33 after l 64, hint %d" % hint, st)
    finally:
        c.close()


def test_wide_untiled_count_1mbp():
    """EULER_B200_WIDE_TILED=0: the one-thread-per-read count kernel of the wide path"""
    run_child('''
dev = T.dev_reads(ctx, T.M, 150, T.ERR)
st = T.run(ctx, dev, 150, 64, N.RUN_CANONICAL_IDS, 0)
buf, off, _ = T.host_reads(T.M, 150, T.ERR)
g = oracle.graph_build(buf, off, 64, expand=False)
assert_counts(st, g)
assert_graph_canonical(ctx, g, True)
T.report("WIDE_TILED=0", st)
''', EULER_B200_WIDE_TILED="0")


def ragged_reads(seed=3):
    """>= 1e6 bases of reads cut from synthetic ones at seeded points: lengths 0..300, runs of N and lower case"""
    rng = np.random.default_rng(seed)
    base = oracle.synth_reads(400_000, 300, err_ppm=ERR, first=0, count=5000)
    lens = rng.integers(0, 301, 8000)
    lens = lens[:np.searchsorted(np.cumsum(lens), base.size)]
    off = np.zeros(lens.size + 1, np.uint64)
    off[1:] = np.cumsum(lens)
    buf = base[:int(off[-1])].copy()
    n = buf.size
    starts = rng.integers(0, n, n // 400)
    runs = rng.integers(1, 6, starts.size)
    pos = np.repeat(starts, runs) + (np.arange(runs.sum()) - np.repeat(np.cumsum(runs) - runs, runs))
    buf[pos[pos < n]] = ord("N")
    starts = rng.integers(0, n, n // 300)
    runs = rng.integers(1, 80, starts.size)
    pos = np.repeat(starts, runs) + (np.arange(runs.sum()) - np.repeat(np.cumsum(runs) - runs, runs))
    pos = pos[pos < n]
    buf[pos] = np.where(buf[pos] == ord("N"), buf[pos], buf[pos] | 0x20)
    assert n >= 1_000_000 and (lens == 0).any() and (lens == 300).any()
    return buf, off


@pytest.mark.parametrize("l", [32, 64])
def test_ragged_input(gctx, l):
    buf, off = ragged_reads()
    g = oracle_graph("ragged", buf, off, l, True)
    st = gctx.run_host(buf, off, l, C | X)
    if l <= 32:
        assert st.path == 1
    assert_counts(st, g)
    assert_graph_canonical(gctx, g, l > 32)
    report("ragged l %d" % l, st)


# ---- the partitioned build at 1 Mbp ------------------------------------------------------------------------------------
PART_CASES = [("records", 2, 32), ("records", 8, 32), ("keys", 2, 32), ("keys", 8, 32),
              ("records", 2, 22), ("records", 8, 22), ("keys", 2, 22), ("keys", 8, 22), ("keys", 2, 64)]


@pytest.mark.parametrize("impl,world,l", PART_CASES)
def test_partitioned_build_1mbp(gctx, impl, world, l):
    from eulercuda.dist import emulate_partitioned, emulate_partitioned_bucketed
    buf, off, R = host_reads(M, L2, ERR)
    if world == 2:      # uneven: 30 % / 70 % of the reads
        cut = [0, R * 3 // 10, R]
    else:               # seven uneven shards and one idle rank
        cut = [0] + sorted(np.random.default_rng(world).choice(np.arange(1, R), 6, replace=False).tolist()) + [R, R]
    shards = [(buf[cut[r] * L2:cut[r + 1] * L2], oracle.fixed_offsets(cut[r + 1] - cut[r], L2)) for r in range(world)]
    if impl == "records":
        parts, windows = emulate_partitioned_bucketed(gctx, shards, l, world)
    else:
        parts, windows = emulate_partitioned(gctx, shards, l, world)
    g = oracle_graph("1mbp", buf, off, l, False)
    assert_partitioned(parts, windows, g, world)
