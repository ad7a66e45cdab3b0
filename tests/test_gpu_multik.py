"""GPU tests of multi-k unitigs (Context.unitigs_multik*, euler_unitigs_multik*, assembler.py --k-list), exact against
the restatements of tests/multik_ref.py: the contig set up to orientation and cycle rotation with each contig's K-mer
sum, and every field of every step."""
import ctypes as C

import pytest

import oracle
import unitig_np
import unitig_shapes
from clean_ref import assembly_stats
from multik_ref import arrays, canon_pairs, strings
from oracle import twin
from test_cpu_multik import TABLE_MULTIK_100K, _joint_reads, genome_kmers, synth
from test_gpu_clean import _error_reads, _fastq

pytestmark = pytest.mark.gpu

EULER_ERR_ARG = -2   # include/euler_b200.h
LISTS = [[2, 3, 5], [15, 21], [21, 31, 32, 33], [21, 33, 63], [31, 63]]


def _gpu(ctx, entry, reads, ks, limit, clean=True, **kw):
    if entry == "reads":
        buf, off = oracle.pack_reads(reads)
        return ctx.unitigs_multik(buf, off, ks, limit, clean=clean, **kw)
    ctx.ingest("".join(">r%d\n%s\n" % (i, r) for i, r in enumerate(reads)).encode(), 1)
    return ctx.unitigs_multik_ingested(ks, limit, clean=clean, **kw)


def _check(ctx, reads, ks, limit, clean=True, entries=("reads",), **kw):
    buf, off = oracle.pack_reads(reads)
    exp, esums, esteps = arrays(buf, off, ks, limit, clean, **kw)
    for entry in entries:
        got, sums, steps = _gpu(ctx, entry, reads, ks, limit, clean, **kw)
        assert len(sums) == len(got)
        assert canon_pairs(got, sums, ks[-1]) == canon_pairs(exp, esums, ks[-1]), (entry, ks, limit, clean)
        assert steps == esteps, (entry, ks, limit, clean)
    return esteps


@pytest.mark.parametrize("ks", LISTS, ids=lambda ks: ",".join(map(str, ks)))
@pytest.mark.parametrize("name", unitig_shapes.SHAPES)
def test_shapes_match_restatement(ctx, name, ks):
    reads = unitig_shapes.shape(name, ks[0])
    for limit in (0, 1, 2):
        for clean in (True, False):
            _check(ctx, reads, ks, limit, clean)


@pytest.mark.parametrize("ks", LISTS, ids=lambda ks: ",".join(map(str, ks)))
def test_random_reads_match_restatement(ctx, ks):
    added = 0
    for seed, glen in ((1, 3000), (2, 5000)):
        reads = _error_reads(seed, glen)
        for limit in (0, 1, 2):
            for clean in (True, False):
                steps = _check(ctx, reads, ks, limit, clean, entries=("reads", "ingested"))
                added += sum(s["nodes_added"] for s in steps)
    if ks[0] >= 15:   # at K = 2..5 these reads spell every K-mer already
        assert added > 0


def test_string_restatement_and_hand_built_joint(ctx):
    g, reads = _joint_reads()
    for ks in ([31], [21, 31]):
        got, sums, steps = ctx.unitigs_multik(*oracle.pack_reads(reads), ks, 1)
        exp, esums, esteps = strings(reads, ks, 1)
        assert canon_pairs(got, sums, 31) == canon_pairs(exp, esums, 31) and steps == esteps
    assert [min(c, twin(c)) for c in got] == [min(g, twin(g))] and steps[1]["nodes_added"] == 5
    reads = _error_reads(4, 3000)
    got, sums, steps = ctx.unitigs_multik(*oracle.pack_reads(reads), [21, 33, 63], 1)
    exp, esums, esteps = strings([r.upper() for r in reads], [21, 33, 63], 1)
    assert canon_pairs(got, sums, 63) == canon_pairs(exp, esums, 63) and steps == esteps


def test_one_step_is_unitigs_clean(ctx):
    reads = _error_reads(3, 4000)
    buf, off = oracle.pack_reads(reads)
    for K in (2, 21, 32, 33, 63):
        for limit in (0, 1):
            c1, s1, st1 = ctx.unitigs_clean(buf, off, K, limit)
            cm, sm, steps = ctx.unitigs_multik(buf, off, [K], limit)
            assert canon_pairs(cm, sm, K) == canon_pairs(c1, s1, K)
            assert steps == [{"K": K, "contigs": len(c1), "bases": sum(map(len, c1)), "nodes_added": 0, "clean": st1}]
            c1, s1, st1 = ctx.unitigs_clean(buf, off, K, limit, max_rounds=0)
            cm, sm, steps = ctx.unitigs_multik(buf, off, [K], limit, clean=False)
            assert canon_pairs(cm, sm, K) == canon_pairs(c1, s1, K) and steps[0]["clean"] == st1


@pytest.mark.parametrize("L,ks", sorted(TABLE_MULTIK_100K))
def test_table_rows_100kbp(ctx, L, ks):
    buf, off = synth(100_000, L)
    got, sums, steps = ctx.unitigs_multik(buf, off, list(ks), 1)
    assert assembly_stats(got, ks[-1], genome_kmers(100_000, ks[-1])) == TABLE_MULTIK_100K[(L, ks)]
    exp, esums, esteps = arrays(buf, off, list(ks), 1)
    assert canon_pairs(got, sums, ks[-1]) == canon_pairs(exp, esums, ks[-1]) and steps == esteps
    again, sums2, steps2 = ctx.unitigs_multik(buf, off, list(ks), 1)   # deterministic
    assert canon_pairs(again, sums2, ks[-1]) == canon_pairs(got, sums, ks[-1]) and steps2 == steps


def test_500kbp_certified(ctx):
    buf, off = synth(500_000, 100)
    ks = [21, 31, 63]
    got, sums, steps = ctx.unitigs_multik(buf, off, ks, 1)
    last = {}
    exp, esums, esteps = arrays(buf, off, ks, 1, last=last)
    assert unitig_np.certify(got, sums, last["g"], last["alive"]) == []
    assert steps == esteps and sorted(int(s) for s in sums) == sorted(esums)
    assert steps[-1]["nodes_added"] > 0


# ---- command line ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("clean", [True, False])
def test_assembler_cli_k_list(ctx, tmp_path, clean):
    import assembler
    reads = _error_reads(5, 5000, err=0.01, n_frac=0, lower=0)
    fq = _fastq(tmp_path, reads)
    out = tmp_path / "m.fa"
    assert assembler.main(["-i", str(fq), "-o", str(out), "--k-list", "21,41,63"] + (["--clean"] if clean else [])) == 0
    got = [x for x in out.read_text().split("\n") if x and x[0] != ">"]
    ctx.ingest(fq.read_bytes(), 2)
    exp, sums, steps = ctx.unitigs_multik_ingested([21, 41, 63], 1, clean=clean)
    assert got == exp and [s["K"] for s in steps] == [21, 41, 63]
    s_lines = [x.split("\t") for x in (tmp_path / "m.fa.gfa").read_text().splitlines() if x.startswith("S\t")]
    assert [x[2] for x in s_lines] == got
    assert [x[4] for x in s_lines] == ["KC:i:%d" % s for s in sums]


# ---- argument errors ---------------------------------------------------------------------------------------------------
def test_argument_errors(ctx):
    import _native as N
    buf, off = oracle.pack_reads(["ACGT" * 40])
    for ks, msg in (([], "K list of 0 entries"), (list(range(2, 19)), "K list of 17 entries"),
                    ([21, 21], "not strictly increasing"), ([31, 21], "not strictly increasing"),
                    ([1, 21], "out of range"), ([21, 64], "out of range")):
        with pytest.raises(N.EulerError, match=msg):
            ctx.unitigs_multik(buf, off, ks, 1)
        with pytest.raises(N.EulerError, match=msg):
            ctx.unitigs_multik_ingested(ks, 1)
    lib, h = ctx.lib, ctx.h
    ks = (C.c_uint32 * 2)(21, 31)
    P = (N.CleanParams * 2)()
    nb, nc = C.c_uint64(0), C.c_uint64(0)
    b, o = buf.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p)
    calls = [
        lambda: lib.euler_unitigs_multik(h, b, None, 1, ks, 2, 1, P, None, C.byref(nb), C.byref(nc), None, None),
        lambda: lib.euler_unitigs_multik(h, b, o, 1, None, 2, 1, P, None, C.byref(nb), C.byref(nc), None, None),
        lambda: lib.euler_unitigs_multik(h, b, o, 1, ks, 2, 1, None, None, C.byref(nb), C.byref(nc), None, None),
        lambda: lib.euler_unitigs_multik(h, b, o, 1, ks, 2, 1, P, None, None, C.byref(nc), None, None),
        lambda: lib.euler_unitigs_multik(h, b, o, 1, ks, 2, 1, P, None, C.byref(nb), None, None, None),
        lambda: lib.euler_unitigs_multik_ingested(h, None, 2, 1, P, None, C.byref(nb), C.byref(nc), None, None),
        lambda: lib.euler_unitigs_multik_ingested(h, ks, 2, 1, None, None, C.byref(nb), C.byref(nc), None, None),
    ]
    for call in calls:
        assert call() == EULER_ERR_ARG
        assert b"null argument" in lib.euler_last_error(h)
    assert lib.euler_version() == 103
