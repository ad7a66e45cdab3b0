"""GPU tests of multi-k unitigs at the sizes where the README's numbers come from, exact against multik_ref.arrays and
certified by unitig_np.certify: the configs[1] rows (4.6 Mbp, 30x, 1 % errors) from both entry points and twice on one
context; a 1 Mbp repeat-rich genome whose steps hand on cycles, self-twin contigs and palindromic K-mers of odd weight;
and multi-k emissions interleaved with the Euler path and the clean-up on one context, which share its text buffer."""
import random
import resource
import time

import numpy as np
import pytest

import oracle
import unitig_np
import unitig_shapes as S
from clean_ref import n50
from multik_ref import arrays, canon_pairs
from oracle import twin
from test_gpu_clean import _error_reads
from test_gpu_unitig_shapes import _fasta

pytestmark = pytest.mark.gpu

FIVE = (21, 31, 41, 51, 63)
# the README's multi-k row: configs[1] shape with 1 % errors, limit 1, default clean-up -> (contigs, N50) of the last step
README_MULTIK_ROW = {
    (100, (31, 63)): (34, 301843), (100, FIVE): (10, 3372650),
    (150, (31, 63)): (65, 433724), (150, FIVE): (61, 433724),
}


def _same(got, sums, steps, exp, what):
    K = steps[-1]["K"]
    assert len(sums) == len(got), what
    assert canon_pairs(got, sums, K) == exp[0], what
    assert steps == exp[1], what


# ---- 1. the configs[1] rows ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def configs1():
    """(L, ks) -> (canon_pairs, steps) of the restatement; the graphs are not kept (about 9 GB of host memory each)"""
    return {}


def _configs1_reads(L):
    G = 4_600_000
    n = G * 30 // L
    return oracle.synth_reads(G, L, err_ppm=10000, first=0, count=n), oracle.fixed_offsets(n, L)


@pytest.mark.parametrize("L,ks", sorted(README_MULTIK_ROW), ids=lambda v: ",".join(map(str, v)) if isinstance(v, tuple) else str(v))
def test_configs1_row(ctx, configs1, L, ks):
    ks = list(ks)
    buf, off = _configs1_reads(L)
    ctx.ingest(_fasta(buf, off), 1)
    got, sums, steps = ctx.unitigs_multik_ingested(ks, 1)
    t0 = time.perf_counter()
    last = {}
    exp, esums, esteps = arrays(buf, off, ks, 1, last=last)
    secs = time.perf_counter() - t0
    assert unitig_np.certify(got, sums, last["g"], last["alive"]) == []
    del last
    configs1[(L, tuple(ks))] = (canon_pairs(exp, esums, ks[-1]), esteps)
    _same(got, sums, steps, configs1[(L, tuple(ks))], "ingested")
    # the output set depends only on the reads and the parameters; a second call on the same context gives it again
    again, sums2, steps2 = ctx.unitigs_multik_ingested(ks, 1)
    _same(again, sums2, steps2, configs1[(L, tuple(ks))], "ingested, second call")
    assert all(s["nodes_added"] > 0 for s in steps[1:]), steps   # the contigs do raise counts at this size
    row = (len(got), n50([len(c) for c in got]))
    print("configs[1] L=%d ks=%s: %s; restatement %.0f s, peak host RSS %.1f GB" %
          (L, ks, row, secs, resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2**20))
    assert row == README_MULTIK_ROW[(L, tuple(ks))]


@pytest.mark.parametrize("L", [100, 150])
def test_configs1_host_reads(ctx, configs1, L):
    ks = [31, 63]
    buf, off = _configs1_reads(L)
    if (L, tuple(ks)) not in configs1:   # this test run alone
        exp, esums, esteps = arrays(buf, off, ks, 1)
        configs1[(L, tuple(ks))] = (canon_pairs(exp, esums, ks[-1]), esteps)
    got, sums, steps = ctx.unitigs_multik(buf, off, ks, 1)
    _same(got, sums, steps, configs1[(L, tuple(ks))], "reads")


# ---- 2. a repeat-rich genome -------------------------------------------------------------------------------------------
SATELLITES = (7, 12, 40)   # unit lengths


def _repeat_reads():
    """150 bp reads at 30x with 1 % errors of a 1 Mbp genome with repeat families, tandem arrays and inverted repeats;
    plus error-free reads of satellite arrays (a unit repeated, longer than a read, with no flank): they give cycles,
    which a linear genome does not, and which read errors would cut at every period"""
    genome = S.repeat_genome(201, 1_000_000, n_families=20, elem_len=(300, 3000), copies=(2, 50),
                             tandems=((2, (40, 200)), (3, (40, 200)), (7, (40, 200)), (12, (40, 200))), inverted=300)
    parts = [S.sample_reads_np(202, genome, 150, 30, 0.01)]
    rng = random.Random(203)
    for i, n in enumerate(SATELLITES):
        unit = "".join(rng.choice("ACGT") for _ in range(n))
        parts.append(S.sample_reads_np(204 + i, unit * (1200 // n), 150, 30, 0.0))
    buf = np.concatenate([b for b, _ in parts])
    offs = [parts[0][1]]
    for _, o in parts[1:]:
        offs.append(o[1:] + offs[-1][-1])
    return buf, np.concatenate(offs)


@pytest.fixture(scope="module")
def repeat_reads():
    return _repeat_reads()


def _self_twin(c, cyc, K):
    if not cyc:
        return c == twin(c)
    s = c[:len(c) - K + 1]
    return twin(s) in s + s


def clauses(trace, ks, limit):
    """the clauses of the rule a run reached, from multik_ref.arrays' trace"""
    out = set()
    for i, t in enumerate(trace[:-1]):
        K, Kn = t["K"], ks[i + 1]
        for (c, cyc, s), w in zip(t["contigs"], t["weights"]):
            L = len(c) - K + 1
            assert s // L >= limit + 1   # every node has count > limit, so the floor of the mean never falls below
            if cyc:
                out.add("cycle")
                if len(c) < Kn:
                    out.add("cycle shorter than the next K")
            if _self_twin(c, cyc, K) and len(c) >= Kn:
                out.add("self-twin")
            if s % L and len(c) >= Kn:
                out.add("weight rounded down")
            if w == limit + 1 and len(c) >= Kn:
                out.add("weight limit + 1")
    if any(t["odd_pal"] for t in trace[1:]):
        out.add("odd weight on a palindrome")
    return out


COMMON = {"cycle", "weight rounded down", "weight limit + 1"}
SHORT = "cycle shorter than the next K"
REPEAT_CASES = [
    # ks, limit, clean, clauses beyond COMMON that the case must reach
    ((21, 31, 63), 1, True, {SHORT}),
    ((20, 32, 48), 1, True, {SHORT, "self-twin", "odd weight on a palindrome"}),
    ((31, 32, 33), 1, True, {"self-twin"}),   # every cycle spells at K + 1
    ((21, 31, 63), 0, True, {SHORT}),
    ((21, 31, 63), 2, True, {SHORT}),
    ((21, 31, 63), 1, False, {SHORT}),
]


@pytest.mark.parametrize("ks,limit,clean,reach", REPEAT_CASES,
                         ids=["%s-limit%d%s" % (",".join(map(str, c[0])), c[1], "" if c[2] else "-noclean") for c in REPEAT_CASES])
def test_repeat_rich_1mbp(ctx, repeat_reads, ks, limit, clean, reach):
    buf, off = repeat_reads
    ks = list(ks)
    got, sums, steps = ctx.unitigs_multik(buf, off, ks, limit, clean=clean)
    last, trace = {}, []
    exp, esums, esteps = arrays(buf, off, ks, limit, clean, last=last, trace=trace)
    assert unitig_np.certify(got, sums, last["g"], last["alive"]) == []
    del last
    _same(got, sums, steps, (canon_pairs(exp, esums, ks[-1]), esteps), (ks, limit, clean))
    reached = clauses(trace, ks, limit)
    assert COMMON | reach <= reached, reached
    assert all(s["nodes_added"] > 0 for s in steps[1:]), steps


# ---- 3. emissions that share one context --------------------------------------------------------------------------------
def test_emissions_share_one_context(ctx):
    import _native as N
    reads = _error_reads(6, 5000, n_frac=0, lower=0)
    ctx.ingest("".join(">r%d\n%s\n" % (i, r) for i, r in enumerate(reads)).encode(), 1)
    buf, off = ctx.ingest_download()
    ctx.run_ingested(32, N.RUN_EXPAND_EDGES | N.RUN_CANONICAL_IDS)
    tour = ctx.pipeline_contigs()
    assert tour == oracle.euler_contigs(buf, off, 32)[0]
    ks = [21, 33, 63]
    exp, esums, esteps = arrays(buf, off, ks, 1)
    mk = (canon_pairs(exp, esums, 63), esteps)
    _same(*ctx.unitigs_multik_ingested(ks, 1), mk, "multi-k after the tour")
    # multi-k wrote ctx's text buffer: the tour's cached text is stale, so it runs again
    assert ctx.pipeline_contigs() == tour
    got, sums, st = ctx.unitigs_clean_ingested(31, 1)
    fresh = N.Context(0)
    try:
        fresh.ingest("".join(">r%d\n%s\n" % (i, r) for i, r in enumerate(reads)).encode(), 1)
        fgot, fsums, fst = fresh.unitigs_clean_ingested(31, 1)
    finally:
        fresh.close()
    assert canon_pairs(got, sums, 31) == canon_pairs(fgot, fsums, 31) and st == fst
    _same(*ctx.unitigs_multik_ingested(ks, 1), mk, "multi-k after the clean-up")
    assert ctx.pipeline_contigs() == tour


def test_empty_last_step_then_tour(ctx):
    """a multi-k call whose last step has no contigs (reads and earlier contigs shorter than its K) between tours"""
    import _native as N
    reads = _error_reads(7, 4000, n_frac=0, lower=0)
    ctx.ingest("".join(">r%d\n%s\n" % (i, r) for i, r in enumerate(reads)).encode(), 1)
    buf, off = ctx.ingest_download()
    ctx.run_ingested(32, N.RUN_EXPAND_EDGES | N.RUN_CANONICAL_IDS)
    tour = ctx.pipeline_contigs()
    assert tour == oracle.euler_contigs(buf, off, 32)[0]
    rng = random.Random(8)
    g = "".join(rng.choice("ACGT") for _ in range(50))
    short = [g[:40], g[10:], g[5:45]] * 3
    sbuf, soff = oracle.pack_reads(short)
    # without clean-up the first step writes the 50 bp contig; with it, that contig is an isolated fragment of fewer
    # than 2K K-mers and every step is empty
    for clean in (False, True):
        for ks in ([21, 63], [31, 51, 63]):
            got, sums, steps = ctx.unitigs_multik(sbuf, soff, ks, 1, clean=clean)
            exp, esums, esteps = arrays(sbuf, soff, ks, 1, clean)
            assert got == [] and len(sums) == 0 and steps == esteps and steps[-1]["contigs"] == 0
            assert steps[0]["contigs"] == (0 if clean else 1)
            assert ctx.pipeline_contigs() == tour
