"""CPU tests (no GPU): the C-ABI library loads and exports every symbol include/euler_b200.h
declares, the product path fails loudly without a device, and the pure-host pieces of the
drop-in modules behave like the reference's."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "pycuda-euler_b200")


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge.build()
    header = open(os.path.join(ROOT, "include", "euler_b200.h")).read()
    declared = set(re.findall(r"\b(euler_[a-z0-9_]+)\s*\(", header))
    declared -= {"euler_ctx", "euler_stats", "euler_vertex", "euler_edge", "euler_succ_vertex", "euler_circuit_edge"}
    assert len(declared) >= 35
    lib = ctypes.CDLL(ge.LIB)
    missing = [name for name in sorted(declared) if not hasattr(lib, name)]
    assert not missing, missing
    assert lib.euler_version() >= 100


def test_no_cpu_fallback_without_a_device():
    """In a child process that sees no CUDA device (none present, or hidden from it) the product path raises."""
    code = r'''
import sys
sys.path[:0] = [%r, %r]
import pytest, _native
with pytest.raises(_native.EulerError):
    _native.Context(0)
import eulercuda.eulercuda as ec
with pytest.raises(_native.EulerError):
    ec.assemble2(9, buffer=["ACGTACGTACGTACGT"])
print("ok")
''' % (ROOT, PKG)
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                         text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stdout[-1000:] + out.stderr[-2000:]


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "euler_oracle" not in src, f


def test_struct_layouts_match_the_reference_dtypes():
    import _native as N
    assert N.EV_DTYPE.itemsize == 24 and N.EE_DTYPE.itemsize == 24
    assert N.SV_DTYPE.itemsize == 12 and N.CE_DTYPE.itemsize == 20
    assert N.EV_DTYPE.names == ("vid", "ep", "ecount", "lp", "lcount")
    assert N.EE_DTYPE.names == ("eid", "v1", "v2", "s", "pad")
    assert N.CE_DTYPE.names == ("ceid", "e1", "e2", "c1", "c2")


def test_import_layouts():
    """all three import layouts of the reference resolve to the same functions (SURVEY §2.1)."""
    import eulercuda
    import eulercuda.eulercuda as ec
    import eulercuda.pyencode as a
    import encoder.pyencode as b
    import pyencode as c
    assert a.encode_lmer_device is b.encode_lmer_device is c.encode_lmer_device
    import gpuhash.pygpuhash, debruijn.pydebruijn, eulertour.pyeulertour, component.pycomponent  # noqa: E401,F401
    import pygpuhash, pydebruijn, pyeulertour, pycomponent  # noqa: E401,F401
    assert eulercuda.assemble2 is ec.assemble2 and eulercuda.assemble is ec.assemble2
    assert pyeulertour.findEulerDevice is eulertour.pyeulertour.findEulerDevice
    import referenceassembler as ra
    from referenceassembler import referenceAssembler as ram
    assert ra.build is ram.build and ra.all_contigs is ram.all_contigs
    assert ra.twin("AACG") == "CGTT" and ra.contig_to_string(["ACG", "CGT", "GTT"]) == "ACGTT"


def test_host_helpers():
    import eulercuda.eulercuda as ec
    import eulercuda.pyencode as enc
    import eulercuda.pygpuhash as gh
    assert ec.getString(4, 27) == "ACGT" and ec.getString(10, 959244) == "TGGGATAATA"
    assert ec.dna_translate(2) == "G" and ec.dna_translate(7) == "."
    assert ec.doErrorCorrection(None, 17, 0, 0) == 17
    assert enc.getOptimalLaunchConfiguration(100000, 512) == ((512, 1, 1), (1, 196, 1))
    assert enc.getOptimalLaunchConfiguration(70000 * 1024, 1024) == ((1024, 1, 1), (2, 65535, 1))
    assert [gh.hash_h(959244, b) for b in (1, 7, 409, 1000003)] == [0, 6, 22, 209841]
    off = enc._offsets(45, 20)
    assert off.tolist() == [0, 20, 40, 45]
    assert enc._offsets(40, 20).tolist() == [0, 20, 40] and enc._offsets(10, 0).tolist() == [0, 10]
    flat = np.array(b"ACGTACGT").astype("S")
    assert enc._as_bytes(flat).tobytes() == b"ACGTACGT"


def test_readers(tmp_path, g200_reads):
    import eulercuda.eulercuda as ec
    from fastareader.parse_fasta import Fasta
    fa = tmp_path / "g.fa"
    fa.write_text("".join(">r%d\n%s\n" % (i, r) for i, r in enumerate(g200_reads)))
    assert ec.read_fasta(str(fa)) == g200_reads
    with open(fa) as h:
        recs = list(Fasta(h))
    assert [r.sequence for r in recs] == g200_reads        # the reference's tests/test_fasta_reader.py
    assert recs[3].head == "r3" and len(recs[11]) == 3
    multi = tmp_path / "m.fa"
    multi.write_text(">a desc\nACGT\nTTGA\n>b\nCC\n")
    with open(multi) as h:
        recs = list(Fasta(h))
    assert [(r.head, r.sequence) for r in recs] == [("a desc", "ACGTTTGA"), ("b", "CC")]
    fq = tmp_path / "r.fastq"
    fq.write_text("@x\nACGT\n+\nIIII\n@y\nTTGN\n+\nIIII\n")
    assert ec.read_fastq(str(fq)) == ["ACGT", "TTGN"]
    assert ec.parse_fastq(str(fq)) == {"@x": "ACGT", "@y": "TTGN"}


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` prints one JSON line: the UNMODIFIED reference's build() (source in this container,
    the bytecode of oracle/build_ref.py on the GPU box) under multiprocessing.Pool, else the oracle port."""
    import json
    from oracle import ref_loader
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                                   "--warmup", "0", "--workload", "small_smoke", "--ref-genome", "20000"], text=True)
    line = json.loads(out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == ("reference" if ref_loader.kind() else "port")
    assert line["cpu_baseline"]["cores"] >= 1 and line["e2e"]["h2d_bytes_per_step"] == 0


def test_bench_line_guard_prints_once():
    """bench.py's watchdog: a stalled phase after the timed steps costs the extra keys, not the line."""
    code = r'''
import sys, time, importlib.util
spec = importlib.util.spec_from_file_location("bench", %r)
b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)
g = b.LineGuard(0.3, {"metric": "x", "value": 1})
%s
print("main thread went on")
'''
    bench = os.path.join(ROOT, "bench.py")
    stalled = subprocess.run([sys.executable, "-c", code % (bench, "time.sleep(5)")], capture_output=True, text=True, timeout=60)
    assert stalled.returncode == 0 and "main thread went on" not in stalled.stdout
    import json
    line = json.loads(stalled.stdout.strip().splitlines()[-1])
    assert line["value"] == 1 and "incomplete" in line
    fine = subprocess.run([sys.executable, "-c", code % (bench, "g.finish({'metric': 'x', 'value': 2}); time.sleep(0.6)")],
                          capture_output=True, text=True, timeout=60)
    lines = fine.stdout.strip().splitlines()
    assert fine.returncode == 0 and json.loads(lines[0])["value"] == 2 and lines[1] == "main thread went on" and len(lines) == 2


@pytest.mark.parametrize("l", [12, 40])
def test_bench_dump_outputs_do_not_depend_on_slot_order(tmp_path, l):
    """bench.py --dump-outputs: the same graph with its ids in two different slot orders gives the same files, float64,
    in key order (checked against the oracle's graph, whose ids are ranks in key order), sampled beyond max_rows."""
    import importlib.util
    import types
    import _native as N
    import oracle
    from util import random_reads
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    buf, off = oracle.pack_reads(random_reads(3, 200, genome_len=1500, lens=(60, 100), n_frac=0.0))
    g = oracle.graph_build(buf, off, l, expand=False)
    st = types.SimpleNamespace(n_kmer_windows=1, n_lmer_windows=2, distinct_lmers=g.nl, distinct_kmers=g.nv, edge_count=g.ne)

    class SlotOrderContext:
        def __init__(self, seed):
            rng = np.random.default_rng(seed)
            pl, pv = rng.permutation(g.nl), rng.permutation(g.nv)     # slot -> oracle id
            inv = np.empty(g.nv, np.uint32)
            inv[pv] = np.arange(g.nv)
            self.arts = {N.ART_LMER_KEYS: g.lk_lo[pl], N.ART_LMER_KEYS_HI: g.lk_hi[pl], N.ART_LMER_VALUES: g.lvals[pl],
                         N.ART_EDGE_V1: inv[g.ev1[pl]], N.ART_EDGE_V2: inv[g.ev2[pl]], N.ART_KMER_KEYS: g.vk_lo[pv],
                         N.ART_KMER_KEYS_HI: g.vk_hi[pv], N.ART_LCOUNT: g.lcount.reshape(-1, 4)[pv].ravel(),
                         N.ART_ECOUNT: g.ecount.reshape(-1, 4)[pv].ravel()}

        def download(self, which):
            return self.arts[which]

    cap = g.nv // 2
    for seed in (1, 2):
        bench.dump_outputs(SlotOrderContext(seed), st, l, str(tmp_path / str(seed)), max_rows=cap)
    names = sorted(os.listdir(tmp_path / "1"))
    assert names == sorted(os.listdir(tmp_path / "2")) and len(names) == 10
    d = {}
    for n in names:
        a, b = np.load(tmp_path / "1" / n), np.load(tmp_path / "2" / n)
        assert a.dtype == np.float64 and np.array_equal(a, b), n
        d[n[:-4]] = a.astype(np.uint64)
    lr, vr = d["lmer_rows"], d["kmer_rows"]
    assert lr.size == vr.size == cap and (np.diff(lr.astype(np.int64)) > 0).all()
    words = [g.lk_hi >> np.uint64(32), g.lk_hi & np.uint64(0xFFFFFFFF)] if l > 32 else []
    words += [g.lk_lo >> np.uint64(32), g.lk_lo & np.uint64(0xFFFFFFFF)]
    assert np.array_equal(d["lmer_keys"], np.stack(words, axis=1)[lr])
    assert np.array_equal(d["lmer_values"], g.lvals[lr])
    assert np.array_equal(d["edge_v1"], g.ev1[lr]) and np.array_equal(d["edge_v2"], g.ev2[lr])
    assert np.array_equal(d["kmer_keys"][:, -1], g.vk_lo[vr] & np.uint64(0xFFFFFFFF))
    assert np.array_equal(d["lcount"], g.lcount.reshape(-1, 4)[vr]) and np.array_equal(d["ecount"], g.ecount.reshape(-1, 4)[vr])
    assert d["counts"].tolist() == [1, 2, g.nl, g.nv, g.ne]


def _bench_mock(args, world=1, stall=False, timeout=240):
    """bench.main() with the device replaced by stand-ins (tests/bench_flow_mock.py); returns rank 0's stdout"""
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        if stall:
            env["BENCH_MOCK_STALL"] = "1"
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "bench_flow_mock.py")] + args, env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=timeout) for p in procs]
    for p, (out, err) in zip(procs, outs):
        assert p.returncode == 0, err[-2000:]
    assert all(not out.strip() for out, _ in outs[1:])      # only rank 0 prints
    return outs[0][0]


@pytest.mark.parametrize("world", [1, 2])
def test_bench_main_flow_with_stand_ins(world):
    """The control flow of bench.py's GPU arm, without a GPU: one JSON line with the contract's keys, the end-to-end
    and extra phases, the per-rank rows and collectives of the N > 1 path (over gloo) -- and the watchdog: when a phase
    after the timed steps never returns, every rank still exits 0 and rank 0 has printed the line, marked incomplete."""
    import json
    args = ["--gpus", str(world), "--steps", "3", "--warmup", "3", "--no-cpu"]
    line = json.loads(_bench_mock(args, world).strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "roofline", "clocks", "gpu_launches", "e2e", "extra"):
        assert key in line, key
    assert line["n_gpus"] == world and line["steps"] == 3 and "incomplete" not in line
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["value"] > 0
    assert ("per_rank" in line and len(line["per_rank"]["rows"]) == world and line["parity_check"]["ok"]) if world > 1 else "no_hint" in line
    stalled = json.loads(_bench_mock(args + ["--no-extra"], world, stall=True).strip().splitlines()[-1])
    assert "incomplete" in stalled and "e2e" not in stalled and stalled["value"] > 0 and stalled["n_gpus"] == world
