#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (encode -> canonical l-mer table -> de Bruijn
graph build) in forward k-mer windows per second (BASELINE.json `metric`).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

One process per GPU (torchrun for N > 1).  A step is one pass of the hot path over one batch of
synthetic reads.  Rank 0 prints ONE JSON line.

* value      k-mer windows / s, reads already resident in HBM (CUDA events, max over ranks)
* e2e        the same through the host-buffer C-ABI call: pinned host reads -> H2D -> pipeline ->
             D2H of the compressed graph, all inside the timed region
* roofline   the dominant kernel (fused encode+count) against the measured HBM peak
* cpu_baseline / --impl reference   the oracle's C restatement of the reference CPU path
             (kind "port": the reference is pure Python and cannot be compiled or shipped), timed on
             this box's host cores on a bounded sample of the same workload
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "pycuda-euler_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (which may be read-only): no __pycache__

WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on for 1 GPU
    "ecoli_4.6Mbp_100bp_30x_k31": dict(G=4_600_000, L=100, cov=30, err_ppm=0, k=31),
    # configs[2] (per-GPU share when sharded)
    "100Mbp_150bp_40x_1pct_k31": dict(G=100_000_000, L=150, cov=40, err_ppm=10_000, k=31),
    # configs[3]: 1 Gbp, 8 GPUs (strong scaling: the data set is split over the ranks)
    "1Gbp_150bp_30x_k31": dict(G=1_000_000_000, L=150, cov=30, err_ppm=0, k=31),
    "small_smoke": dict(G=200_000, L=100, cov=20, err_ppm=0, k=31),
}
DEFAULT_WORKLOAD = "ecoli_4.6Mbp_100bp_30x_k31"
METRIC = "k-mers/sec (encode+hash+graph build, device-timed)"
UNIT = "k-mers/s"


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {
                getattr(pynvml, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(pynvml, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(pynvml, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(pynvml, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            while not self.stop_flag:
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.002)
        except Exception as e:  # NVML not available: report that instead of inventing numbers
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def algorithmic_bytes(st, w=8):
    """SURVEY §8d: A = B + N_l (w+8) + U_l (w+16) + U_k (2w+84); the count kernel's share is the
    first two terms (every base read once, one table-slot touch per forward l-mer window)."""
    B, Nl, Ul, Uk = st.n_bases, st.n_lmer_windows, st.distinct_lmers, st.distinct_kmers
    kernel = B + Nl * (w + 8)
    return kernel, kernel + Ul * (w + 16) + Uk * (2 * w + 84)


# ---------------------------------------------------------------------------------------------------------------
# CPU baselines.  `reference` = the UNMODIFIED referenceAssembler.build (referenceAssembler.py:25-42) fanned out
# the way the reference does (dask map_partitions(build) / Spark reduceByKey, BASELINE.md §2): multiprocessing.Pool(P)
# over contiguous read shards, dict-sum merge in the parent.  The module is loaded by oracle/ref_loader.py: from
# /root/reference in the authoring container, from the bytecode in oracle/_ref/ on the GPU box.  `port` = the oracle's
# C restatement (OpenMP), used when the reference is not available and reported beside it.
# Sample = a full-coverage data set of a SMALLER genome from the same generator (same read length, coverage and error
# rate), so the distinct-key count scales with the sample like it does in the workload; the rate is the slope between
# two sample sizes (fixed costs such as the pool start-up cancel).
_REF_READS = None   # inherited by the forked pool workers


def _ref_build_shard(args):
    lo, hi, k = args
    from oracle import ref_loader
    ra = ref_loader.load()
    return ra.build(_REF_READS[lo:hi], k, 0)


def _synth_read_strings(wl, G):
    import oracle
    L = wl["L"]
    R = -(-G * wl["cov"] // L)
    buf = oracle.synth_reads(G, L, err_ppm=wl["err_ppm"], first=0, count=R).tobytes()
    return [buf[i * L:(i + 1) * L].decode("ascii") for i in range(R)], R * (L - wl["k"] + 1)


def reference_build_seconds(wl, G, procs):
    """one pass of the reference's build() over a cov-x data set of a G-bp genome: (seconds, k-mer windows, distinct)"""
    global _REF_READS
    import multiprocessing as mp
    _REF_READS, nk = _synth_read_strings(wl, G)
    R = len(_REF_READS)
    bounds = [(R * i // procs, R * (i + 1) // procs, wl["k"]) for i in range(procs)]
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        pool.map(_ref_build_shard, [(0, min(R, 64), wl["k"])] * procs)   # workers started and the module loaded
        t0 = time.perf_counter()
        parts = pool.map(_ref_build_shard, bounds, chunksize=1)
        total = parts[0]
        for d in parts[1:]:   # dict-sum merge (the reduceByKey of src/ref_spark.py:84)
            for km, c in d.items():
                total[km] = total.get(km, 0) + c
        dt = time.perf_counter() - t0
    _REF_READS = None
    return dt, nk, len(total)


def port_build_seconds(wl, G):
    """the oracle's C restatement (encode + both-strand tables + graph build) on the same kind of sample"""
    import oracle
    L, l = wl["L"], wl["k"] + 1
    R = -(-G * wl["cov"] // L)
    buf = oracle.synth_reads(G, L, err_ppm=wl["err_ppm"], first=0, count=R)
    off = oracle.fixed_offsets(R, L)
    t0 = time.perf_counter()
    oracle.graph_build(buf, off, l, expand=False)
    return time.perf_counter() - t0, R * (L - wl["k"] + 1), 0


def cpu_rate(wl, G1, procs, want="auto"):
    """k-mer windows / s of the CPU path from the slope between samples of G1 and 2*G1 bp.  Returns a dict."""
    from oracle import ref_loader
    use_ref = want != "port" and ref_loader.load() is not None and wl["k"] <= 1000
    fn = (lambda G: reference_build_seconds(wl, G, procs)) if use_ref else (lambda G: port_build_seconds(wl, G))
    t1, n1, _ = fn(G1)
    t2, n2, _ = fn(2 * G1)
    # slope between the two sizes; a sample too small to separate them (timer noise) falls back to the larger sample's raw rate
    slope = (n2 - n1) / (t2 - t1) if t2 > 1.25 * t1 else n2 / t2
    return {"value": slope, "unit": UNIT, "cores": procs if use_ref else int(os.environ.get("OMP_NUM_THREADS", os.cpu_count() or 1)),
            "kind": "reference" if use_ref else "port",
            "sample": "%d x data sets of %d bp and %d bp genomes from the workload's generator (%d / %d k-mer windows, %.2f s / %.2f s); "
                      "rate = slope between the two" % (wl["cov"], G1, 2 * G1, n1, n2, t1, t2),
            "rates_raw": [n1 / t1, n2 / t2], "seconds": t1 + t2,
            "code": ("referenceAssembler.build, unmodified (%s), multiprocessing.Pool(%d) over read shards + dict-sum merge" % (ref_loader.kind(), procs))
            if use_ref else "oracle/euler_oracle.c graph_build (C restatement, OpenMP)"}


def run_reference(args, wl, rank, world):
    """--impl reference: the reference's own CPU path on this box's host cores, bounded sample per step."""
    if rank != 0:
        return
    procs = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(procs)   # torchrun pins it to 1: the port's thread count must be explicit
    G1 = args.ref_genome or max(20_000, min(wl["G"] // 2, 12_500 * procs))
    for _ in range(min(args.warmup, 1)):
        cpu_rate(wl, max(G1 // 8, 10_000), procs)
    vals, last = [], None
    for _ in range(args.steps):
        last = cpu_rate(wl, G1, procs)
        vals.append(last["value"])
    value = sorted(vals)[len(vals) // 2]
    nk_step = wl["cov"] * 3 * G1 // wl["L"] * (wl["L"] - wl["k"] + 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals),
        "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * last["seconds"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": {"workload": args.workload, "k": wl["k"], "sample": last["sample"], "code": last["code"],
                   "steps_requested": args.steps,
                   "note": "median over steps of the slope rate; each step runs the two sample sizes once"},
        "cpu_baseline": {k: last[k] for k in ("unit", "cores", "kind", "sample")} | {"value": value},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def roofline_record(st, ms_part, ms_build, ms_step, l, workload, world):
    """The dominant kernel against the measured HBM peak.  Algorithmic bytes (SURVEY §8d, DESIGN.md §3):
    A = B + N_l (w+8) + U_l (w+16) + U_k (2w+84).  The partition kernel reads every base once (B); the per-bucket
    build kernel does the table touches and writes every artefact (the other three terms)."""
    peak, peak_src = measured_peak_gbs()
    w = 16 if l > 32 else 8
    B, Nl, Ul, Uk = st.n_bases, st.n_lmer_windows, st.distinct_lmers, st.distinct_kmers
    a_part, a_build = B, Nl * (w + 8) + Ul * (w + 16) + Uk * (2 * w + 84)
    a_path = a_part + a_build
    if st.path == 1:
        name, a_kernel, t = ("bkt_build_kernel", a_build, ms_build) if ms_build >= ms_part else ("bkt_partition_kernel", a_part, ms_part)
    else:   # round-1 global-table path: the fused encode + count kernel (first two terms)
        name, a_kernel, t = ("count_compact_kernel" if l <= 32 else "wide_count_tiled_kernel"), B + Nl * (w + 8), ms_part
    achieved = a_kernel / (t * 1e-3) / 1e9 if t > 0 else 0.0
    traffic = None
    tfile = os.path.join(ROOT, "profiles", "r02_kernel_traffic.json")
    if os.path.exists(tfile) and world == 1:
        try:
            with open(tfile) as f:
                rec = json.load(f).get(name)
            if rec and rec.get("workload") == workload:   # only for the kernel and workload the capture was taken on
                traffic = rec.get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    return {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": a_kernel,
            "path_algorithmic_bytes": a_path, "path_frac": a_path / (ms_step * 1e-3) / 1e9 / peak,
            "kernels_ms": {"bkt_partition_kernel": ms_part, "bkt_build_kernel": ms_build} if st.path == 1 else {"count_kernel": ms_part}}


def dump_outputs(ctx, st, l, out_dir, max_rows=1 << 18, seed=0):
    """--dump-outputs: the graph the last timed step left in ctx, as float64 .npy files under out_dir, so that two builds can
    be compared output for output.  Ids are in table-slot order, which may differ between runs, so the tables are written in
    key order: l-mers and vertices sorted by key, edge end points as ranks in that vertex order.  A key is stored as its
    32-bit words, most significant first (float64 holds each exactly).  A table of more than max_rows rows is cut to a fixed,
    seeded sample of max_rows rows; lmer_rows / kmer_rows hold their places in the sorted table."""
    import numpy as np
    import _native as N
    wide = l > 32

    def keys(which, which_hi):
        return ctx.download(which), ctx.download(which_hi) if wide else None

    def order(lo, hi):
        return np.lexsort((lo, hi)) if wide else np.argsort(lo, kind="stable")

    def words(lo, hi):
        w = [lo >> np.uint64(32), lo & np.uint64(0xFFFFFFFF)]
        return np.stack(([hi >> np.uint64(32), hi & np.uint64(0xFFFFFFFF)] if wide else []) + w, axis=1)

    def sample(n):
        return np.arange(n) if n <= max_rows else np.sort(np.random.default_rng(seed).choice(n, max_rows, replace=False))

    lk, lk_hi = keys(N.ART_LMER_KEYS, N.ART_LMER_KEYS_HI)
    vk, vk_hi = keys(N.ART_KMER_KEYS, N.ART_KMER_KEYS_HI)
    o, ov = order(lk, lk_hi), order(vk, vk_hi)
    rank = np.empty(vk.size, np.int64)
    rank[ov] = np.arange(vk.size)
    lrows, vrows = sample(lk.size), sample(vk.size)
    li, vi = o[lrows], ov[vrows]
    out = {
        "counts": np.array([st.n_kmer_windows, st.n_lmer_windows, st.distinct_lmers, st.distinct_kmers, st.edge_count]),
        "lmer_rows": lrows, "lmer_keys": words(lk[li], lk_hi[li] if wide else None),
        "lmer_values": ctx.download(N.ART_LMER_VALUES)[li],
        "edge_v1": rank[ctx.download(N.ART_EDGE_V1)[li]], "edge_v2": rank[ctx.download(N.ART_EDGE_V2)[li]],
        "kmer_rows": vrows, "kmer_keys": words(vk[vi], vk_hi[vi] if wide else None),
        "lcount": ctx.download(N.ART_LCOUNT).reshape(-1, 4)[vi], "ecount": ctx.download(N.ART_ECOUNT).reshape(-1, 4)[vi],
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


class Runner:
    """One rank of the benchmark: device buffers of a workload and the step function (single GPU: the resident
    pipeline; N > 1: the partitioned path of eulercuda/dist.py)."""

    def __init__(self, ctx, stream, rank, world, dist):
        self.ctx, self.stream, self.rank, self.world, self.dist = ctx, stream, rank, world, dist

    def barrier(self):
        import torch
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def load(self, wl, strong, hint_mode="genome"):
        import torch
        L = wl["L"]
        world, rank = self.world, self.rank
        self.wl, self.l = wl, wl["k"] + 1
        self.G = wl["G"] if (strong or world == 1) else wl["G"] * world
        R_all = -(-wl["G"] * wl["cov"] // L)
        self.R = -(-R_all // world) if strong else R_all
        first = rank * self.R
        self.d_reads = torch.empty(self.R * L, dtype=torch.uint8, device="cuda")
        self.ctx.synth_reads_dev(self.d_reads.data_ptr(), self.G, L, wl["err_ppm"], first, self.R)
        self.d_off = torch.arange(self.R + 1, dtype=torch.int64, device="cuda") * L
        self.ctx.sync()
        torch.cuda.synchronize()
        # a user knows the genome size: error-free reads have ~G distinct canonical l-mers, of which a rank holds
        # ~1.15 / world (l-mers at bucket borders are held twice).  With sequencing errors nothing is known: 0.
        if wl["err_ppm"] == 0 and hint_mode == "genome":
            self.hint = wl["G"] if world == 1 else int(self.G / world * 1.15)
        else:
            self.hint = 0

    def step(self, hint=None):
        import torch
        hint = self.hint if hint is None else hint
        n_bases = self.R * self.wl["L"]
        if self.world == 1:
            return self.ctx.run_dev(self.d_reads.data_ptr(), self.d_off.data_ptr(), self.R, n_bases, self.l, 0, hint), None
        from eulercuda.dist import build_partitioned
        with torch.cuda.stream(self.stream):
            return build_partitioned(self.ctx, self.d_reads, self.d_off, self.R, n_bases, self.l, self.rank, self.world, hint)

    def measure(self, steps, warmup, hint=None):
        """-> dict: ms per step (CUDA events on the ctx stream around the K steps, max over ranks), stage times, counts"""
        import torch
        st = info = None
        for _ in range(warmup):
            st, info = self.step(hint)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        part_ms = build_ms = graph_ms = 0.0
        launches, per_step = 0, []
        t0 = time.perf_counter()
        e0.record(self.stream)
        for _ in range(steps):
            t_s = time.perf_counter()
            st, info = self.step(hint)
            per_step.append(st.ms_total if self.world == 1 else 1e3 * (time.perf_counter() - t_s))
            part_ms += st.ms_count_kernel if self.world == 1 else st.ms_count
            build_ms += st.ms_build_kernel
            graph_ms += st.ms_graph
            launches += st.kernel_launches + (3 if self.world > 1 else 0)   # + mark_starts, partition, push_counts
        e1.record(self.stream)
        self.barrier()
        wall = 1e3 * (time.perf_counter() - t0) / steps
        ms = e0.elapsed_time(e1) / steps
        if self.world > 1:
            st.n_kmer_windows, st.n_lmer_windows, st.n_bases = info["n_kmer_windows"], info["n_lmer_windows"], self.R * self.wl["L"]
        vals = torch.tensor([ms, part_ms / steps, build_ms / steps, wall, float(st.retries), float(st.redo_buckets)],
                            dtype=torch.float64, device="cuda")
        tot = torch.tensor([float(st.n_kmer_windows), float(launches)], dtype=torch.float64, device="cuda")
        per_rank = None
        if self.dist is not None:   # what every rank saw, before the MAX: ms, partition, build, wall, retries, second-pass buckets
            mine = torch.cat([vals, torch.tensor([graph_ms / steps, float(st.bucket_records), float(st.distinct_lmers)],
                                                 dtype=torch.float64, device="cuda")])
            allr = [torch.empty_like(mine) for _ in range(self.world)]
            self.dist.all_gather(allr, mine)
            per_rank = [[round(float(x), 3) for x in t.tolist()] for t in allr]
        if self.dist is not None:
            self.dist.all_reduce(vals, op=self.dist.ReduceOp.MAX)
            self.dist.all_reduce(tot, op=self.dist.ReduceOp.SUM)
        ms_max, part_max, build_max, wall_max, retries_max, redo_max = (float(x) for x in vals.tolist())
        nk_total, launches_total = (float(x) for x in tot.tolist())
        return {"st": st, "info": info, "ms": ms_max, "part_ms": part_max, "build_ms": build_max, "graph_ms": graph_ms / steps,
                "wall_ms": wall_max, "per_step": per_step, "nk_total": nk_total, "launches": int(launches_total),
                "retries": int(retries_max), "redo_buckets": int(redo_max), "per_rank": per_rank}

    def free(self):
        self.d_reads = self.d_off = None


class LineGuard:
    """Prints the JSON line exactly once.  If the main thread has not called finish() within `seconds`, the guard
    prints the line as it stands (marked incomplete) and ends the process with status 0; with line None it only
    ends the process.  Every rank runs one, so a stalled rank cannot keep the others (or the launcher) waiting."""

    def __init__(self, seconds, line):
        self.seconds, self.line = seconds, line
        self.lock, self.done, self.ev = threading.Lock(), False, threading.Event()
        threading.Thread(target=self._run, daemon=True).start()

    def _run(self):
        if self.ev.wait(self.seconds):
            return
        with self.lock:
            if self.done:
                return
            self.done = True
            if self.line is not None:
                self.line["incomplete"] = "a phase after the timed steps did not finish within %d s; printed by the watchdog" % self.seconds
                try:
                    print(json.dumps(self.line), flush=True)
                except Exception:   # the main thread was adding a key: the headline part is what matters
                    print(json.dumps({k: v for k, v in list(self.line.items()) if k not in ("e2e", "extra", "cpu_baseline")}), flush=True)
        os._exit(0)

    def finish(self, line):
        with self.lock:
            if self.done:
                return
            self.done = True
            if line is not None:
                print(json.dumps(line), flush=True)
        self.ev.set()


def parity_check_partitioned(runner):
    """N > 1: the PRODUCTION partitioned path (peer stores + per-rank build, uneven shards) against the single-GPU
    pipeline on the same reads, before anything is timed: sum of multiplicities, number of distinct both-strand
    l-mers, number of vertices and a checksum sum(key * multiplicity) mod 2^64 over the per-rank edge tables must
    equal the single-GPU values (every both-strand l-mer is homed on exactly one rank)."""
    import numpy as np
    import torch
    import _native as N
    from eulercuda.dist import build_partitioned
    ctx, rank, world, dist = runner.ctx, runner.rank, runner.world, runner.dist
    wl = dict(WORKLOADS["small_smoke"])
    L, l = wl["L"], wl["k"] + 1
    R_all = wl["G"] * wl["cov"] // L
    # uneven shards: rank r takes a slice proportional to r + 1
    cuts = [R_all * (r * (r + 1) // 2) // (world * (world + 1) // 2) for r in range(world + 1)]
    lo, hi = cuts[rank], cuts[rank + 1]
    n = hi - lo
    d_reads = torch.empty(max(n, 1) * L, dtype=torch.uint8, device="cuda")
    if n:
        ctx.synth_reads_dev(d_reads.data_ptr(), wl["G"], L, wl["err_ppm"], lo, n)
    d_off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * L
    ctx.sync()

    def table_sums():
        lk = ctx.download(N.ART_LMER_KEYS)
        lv = ctx.download(N.ART_LMER_VALUES).astype(np.uint64)
        return [int(lv.sum()), int(lk.size), int(ctx.download(N.ART_KMER_KEYS).size), int((lk * lv).sum(dtype=np.uint64))]

    res = {"ok": False}
    try:
        with torch.cuda.stream(runner.stream):
            for _ in range(2):   # twice: the second step runs on the other receive area with learned capacities
                st, info = build_partitioned(ctx, d_reads, d_off, n, n * L, l, rank, world, 0)
        mine = table_sums()
        t = torch.tensor([x & 0x7fffffffffffffff for x in mine[:3]] + [mine[3] & 0xffffffff, mine[3] >> 32], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        got = t.tolist()
        chk = (got[3] + (got[4] << 32)) & 0xffffffffffffffff
        if rank == 0:
            d_all = torch.empty(R_all * L, dtype=torch.uint8, device="cuda")
            ctx.synth_reads_dev(d_all.data_ptr(), wl["G"], L, wl["err_ppm"], 0, R_all)
            d_off_all = torch.arange(R_all + 1, dtype=torch.int64, device="cuda") * L
            ctx.sync()
            ctx.run_dev(d_all.data_ptr(), d_off_all.data_ptr(), R_all, R_all * L, l, 0, 0)
            want = table_sums()
            res = {"ok": got[:3] == want[:3] and chk == want[3], "path": info["transport"], "workload": "small_smoke, shards ~ rank + 1",
                   "edges": got[0], "distinct_lmers": got[1], "vertices": got[2], "checksum": "%016x" % chk,
                   "single_gpu": {"edges": want[0], "distinct_lmers": want[1], "vertices": want[2], "checksum": "%016x" % want[3]}}
    except Exception as e:   # reported, and fatal below
        res = {"ok": False, "error": "%s: %s" % (type(e).__name__, e)}
    flag = torch.tensor([1 if (rank != 0 or res["ok"]) and "error" not in res else 0], dtype=torch.int64, device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    res["ok"] = bool(flag.item())
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = genome and reads grow with N (default); strong = the named data set is split over the ranks")
    ap.add_argument("--k", type=int, default=0,
                    help="override the workload's k (BASELINE configs[4] k sweep: 21 / 31 / 63; k = 63 uses 128-bit keys)")
    ap.add_argument("--ref-genome", type=int, default=0, help="--impl reference: genome size of the smaller of the two samples")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra BASELINE configs (configs[2..4]) reported under `extra`")
    ap.add_argument("--extra-scale", type=float, default=1.0,
                    help="development aid: scale the genome of the extra configs (0.25 on 2 GPUs = the per-rank size of the 8-GPU run)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the graph of the last one as DIR/<name>.npy (float64, key order; see dump_outputs)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or world > 1):
        ap.error("--dump-outputs writes the outputs of the one-GPU path (--impl b200, one process)")
    wl = dict(WORKLOADS[args.workload])
    if args.k:
        wl["k"] = args.k

    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return

    import torch
    import _native as N

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        # a rank that dies must not leave the others waiting for the default 10 minutes
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=90))

    ctx = N.Context(local_rank)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    runner = Runner(ctx, stream, rank, world, dist)

    parity = parity_check_partitioned(runner) if world > 1 else None
    if parity is not None and not parity["ok"]:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "n_gpus": world, "parity_check": parity, "error": "the partitioned path disagrees with the single-GPU pipeline"}))
        dist.barrier()
        dist.destroy_process_group()
        raise SystemExit(3)

    L, k, l = wl["L"], wl["k"], wl["k"] + 1
    strong = args.scaling == "strong" and world > 1
    runner.load(wl, strong)
    R, G, hint = runner.R, runner.G, runner.hint
    sampler = ClockSampler(local_rank)
    sampler.start()
    m = runner.measure(args.steps, args.warmup)
    clocks = sampler.result()
    st, info, ms_max = m["st"], m["info"], m["ms"]
    if args.dump_outputs:
        dump_outputs(ctx, st, l, args.dump_outputs)
    nohint = None
    if world == 1 and hint:   # the same steady state without the genome-size hint (capacities learned from the previous run)
        m0 = runner.measure(max(3, args.steps // 4), 2, hint=0)
        nohint = {"ms_per_step": m0["ms"], "value": m0["nk_total"] / (m0["ms"] * 1e-3)}

    # The headline numbers are in hand: from here on (end-to-end steps, the extra configurations) a stall must not
    # cost the line.  A watchdog on every rank prints what there is (rank 0) and leaves, before the NCCL timeout would
    # abort the processes.
    line = None
    if rank == 0:
        roof = roofline_record(st, m["part_ms"], m["build_ms"], ms_max, l, args.workload, world)
        per_step = m["per_step"]
        line = {
            "metric": METRIC, "value": m["nk_total"] / (ms_max * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max, "higher_is_better": True, "scaling": args.scaling if world > 1 else "weak",
            "vs_baseline": None, "dtype": "u64" if l <= 32 else "u128", "data": "synthetic",
            "config": {
                "workload": args.workload, "genome_bp": wl["G"], "read_len": L, "coverage": wl["cov"], "err_ppm": wl["err_ppm"],
                "k": k, "reads_per_gpu": R, "bases_per_gpu": R * L,
                "parallelism": "1 GPU" if world == 1 else
                "%d GPUs: reads sharded, k-mer space partitioned by the minimizer of each vertex, one exchange (see dist.transport)" % world,
                "genome_bp_total": G,
                "l2": "inputs (%d MB ASCII) and the record regions written / re-read every step exceed the 126 MB L2" % (R * L // 10 ** 6),
                "distinct_hint": hint, "ids": "bucket order (canonical-id sort not in the timed region)",
                "path": "minimizer-bucketed (partition pass + per-bucket shared-memory build)" if st.path == 1 else "global table (round 1)",
                "buckets": int(st.n_buckets),
                "timing": "CUDA events on the library's stream around the K steps, max over ranks",
            },
            "counts": {"n_kmer_windows": int(st.n_kmer_windows), "n_lmer_windows": int(st.n_lmer_windows),
                       "distinct_lmers": int(st.distinct_lmers), "distinct_kmers": int(st.distinct_kmers),
                       "edges": int(st.edge_count), "retries": m["retries"], "second_pass_buckets": m["redo_buckets"]},
            "stage_ms": {"partition_kernel": m["part_ms"], "build_kernel": m["build_ms"], "step_wall": m["wall_ms"],
                         "step_median": sorted(per_step)[len(per_step) // 2], "step_best": min(per_step)},
            "roofline": roof,
            "clocks": clocks,
            "gpu_launches": m["launches"],
        }
        if nohint:
            line["no_hint"] = nohint
        if parity is not None:
            line["parity_check"] = parity
        if m.get("per_rank"):
            line["per_rank"] = {"columns": ["ms_per_step", "partition_kernel_ms", "build_kernel_ms", "step_wall_ms", "retries",
                                            "second_pass_buckets", "graph_ms", "fullest_bucket", "distinct_lmers"], "rows": m["per_rank"]}
        if world > 1 and info:
            line["dist"] = {kk: info[kk] for kk in ("exchange_bytes", "exact_fallback", "transport", "phase_ms", "geometry") if kk in info}
    guard = LineGuard(80.0 if world > 1 else 240.0, line)

    # ---- e2e: host buffers through the reference-facing C-ABI call, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        d_reads, d_off = runner.d_reads, runner.d_off
        h_reads = torch.empty(R * L, dtype=torch.uint8, pin_memory=True)
        h_reads.copy_(d_reads)
        h_off = torch.empty(R + 1, dtype=torch.int64, pin_memory=True)
        h_off.copy_(d_off)
        torch.cuda.synchronize()
        arts = [N.ART_LMER_KEYS, N.ART_LMER_VALUES, N.ART_LMER_OFFSETS, N.ART_EDGE_V1, N.ART_EDGE_V2, N.ART_EV]
        width = {N.ART_LMER_KEYS: 8, N.ART_LMER_VALUES: 4, N.ART_LMER_OFFSETS: 4, N.ART_EDGE_V1: 4, N.ART_EDGE_V2: 4,
                 N.ART_EV: 24}
        cap_items = int(max(st.distinct_lmers, st.distinct_kmers) * (1.05 if world == 1 else 1.15)) + 1024
        h_out = {a: torch.empty(cap_items * width[a], dtype=torch.uint8, pin_memory=True) for a in arts}

        def e2e_step(c=ctx, out=h_out):
            if world > 1:   # this rank's shard in from pinned host memory, the partitioned build, this rank's part of the graph out
                from eulercuda.dist import build_partitioned
                with torch.cuda.stream(stream):
                    d_reads.copy_(h_reads, non_blocking=True)
                    d_off.copy_(h_off, non_blocking=True)
                    s, _ = build_partitioned(c, d_reads, d_off, R, R * L, l, rank, world, hint)
            else:
                s = c.run_host_ptr(h_reads.data_ptr(), h_off.data_ptr(), R, l, 0, hint)
            nb = 0
            for a in arts:
                nb += c.download_into(a, out[a].data_ptr(), out[a].numel())
            return s, nb

        for _ in range(2):
            e2e_step()
        runner.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        d2h = 0
        for _ in range(args.steps):
            s2, d2h = e2e_step()
        e1.record(stream)
        runner.barrier()
        e2e_wall = 1e3 * (time.perf_counter() - t0) / args.steps
        serial_ms = max(e0.elapsed_time(e1) / args.steps, e2e_wall)  # the call returns synchronously: wall is the truth
        piped_ms = serial_ms
        if world == 1:
            # Two contexts (two streams, two host threads) alternate steps, so the PCIe copies of one step
            # overlap the kernels and the opposite-direction copy of the other; every step still moves its own
            # inputs in and its own result out inside the timed region.
            ctx_b = N.Context(local_rank)
            h_out_b = {a: torch.empty(cap_items * width[a], dtype=torch.uint8, pin_memory=True) for a in arts}
            for _ in range(2):
                e2e_step(ctx_b, h_out_b)
            nsteps2 = max(2, args.steps + (args.steps & 1))
            errs = []

            def worker(c, out):
                try:
                    for _ in range(nsteps2 // 2):
                        e2e_step(c, out)
                except Exception as exc:   # surfaced below: a failed step must not look like a fast one
                    errs.append(exc)

            runner.barrier()
            th = [threading.Thread(target=worker, args=(ctx, h_out)), threading.Thread(target=worker, args=(ctx_b, h_out_b))]
            t0 = time.perf_counter()
            for t in th:
                t.start()
            for t in th:
                t.join()
            torch.cuda.synchronize()
            piped_ms = 1e3 * (time.perf_counter() - t0) / nsteps2
            if errs:
                raise errs[0]
            ctx_b.close()
        e2e = {"ms": min(serial_ms, piped_ms), "serial_ms": serial_ms, "piped_ms": piped_ms, "h2d": int(R * L + (R + 1) * 8),
               "d2h": int(d2h)}
        del h_reads, h_off, h_out
    e2e_t = torch.tensor([e2e["ms"] if e2e else 0.0], dtype=torch.float64, device="cuda")
    e2e_b = torch.tensor([e2e["h2d"], e2e["d2h"]] if e2e else [0, 0], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_b, op=dist.ReduceOp.SUM)   # bytes of the whole job: every rank copies its own shard in and its own part out
    e2e_ms_max = float(e2e_t.item())
    e2e_h2d, e2e_d2h = (int(x) for x in e2e_b.tolist())

    # ---- the other BASELINE configs, reported under `extra` (every rank takes part; rank 0 prints)
    extra = []
    if not args.no_extra and args.workload == DEFAULT_WORKLOAD and args.scaling == "weak" and not args.k:
        plan = []
        if world == 1:
            # configs[3] cut to what one GPU's u32 ids hold (E = 2 N_l < 2^32): 1/16 of the 1 Gbp genome at 30x, the single-GPU
            # reference point for the 8-GPU run of configs[3] (16x this data set)
            plan.append(("1Gbp_150bp_30x_k31", dict(WORKLOADS["1Gbp_150bp_30x_k31"], G=62_500_000), False, "1/16 of configs[3] (62.5 Mbp, 150 bp, 30x) on one GPU"))
        sc = args.extra_scale
        if world >= 2:
            w3 = dict(WORKLOADS["100Mbp_150bp_40x_1pct_k31"])
            w3["G"] = int(w3["G"] * sc)
            plan.append(("100Mbp_150bp_40x_1pct_k31", w3, True, "configs[2], strong scaling" + ("" if sc == 1.0 else ", genome x %g" % sc)))
        if world == 8 or sc != 1.0:
            w4 = dict(WORKLOADS["1Gbp_150bp_30x_k31"])
            w4["G"] = int(w4["G"] * sc)
            plan.append(("1Gbp_150bp_30x_k31", w4, True, "configs[3], strong scaling" + ("" if sc == 1.0 else ", genome x %g" % sc)))
        t_extra = time.perf_counter()
        for name, xwl, xstrong, note in plan:
            rec = {"workload": name, "note": note, "n_gpus": world, "scaling": "strong" if xstrong else "single"}
            # every rank must take the same decisions here: elapsed time and failures are reduced over the ranks first
            late = torch.tensor([1 if time.perf_counter() - t_extra > 150 else 0], dtype=torch.int64, device="cuda")
            if dist is not None:
                dist.all_reduce(late, op=dist.ReduceOp.MAX)
            if int(late.item()):
                rec["skipped"] = "time budget of the extra configurations used up"
                extra.append(rec)
                continue
            try:
                runner.free()
                torch.cuda.empty_cache()
                err = None
                try:
                    runner.load(xwl, xstrong)
                except Exception as e:   # e.g. out of memory on one rank: agreed below before any collective step
                    err = e
                bad = torch.tensor([0 if err is None else 1], dtype=torch.int64, device="cuda")
                if dist is not None:
                    dist.all_reduce(bad, op=dist.ReduceOp.MAX)
                if int(bad.item()):
                    raise err if err is not None else RuntimeError("loading the workload failed on another rank")
                xs = ClockSampler(local_rank)
                xs.start()
                xm = runner.measure(2, 1)
                rec.update({"value": xm["nk_total"] / (xm["ms"] * 1e-3), "unit": UNIT, "ms_per_step": xm["ms"], "steps": 2, "warmup": 1,
                            "genome_bp": xwl["G"], "read_len": xwl["L"], "coverage": xwl["cov"], "err_ppm": xwl["err_ppm"], "k": xwl["k"],
                            "counts": {"n_kmer_windows": int(xm["nk_total"]), "distinct_lmers_rank0": int(xm["st"].distinct_lmers),
                                       "distinct_kmers_rank0": int(xm["st"].distinct_kmers), "edges_rank0": int(xm["st"].edge_count)},
                            "roofline": roofline_record(xm["st"], xm["part_ms"], xm["build_ms"], xm["ms"], xwl["k"] + 1, name, world),
                            "clocks": xs.result()})
                if xm["info"]:
                    rec["dist"] = {kk: xm["info"][kk] for kk in ("exchange_bytes", "transport", "phase_ms", "geometry") if kk in xm["info"]}
            except Exception as e:
                rec["error"] = "%s: %s" % (type(e).__name__, e)
            extra.append(rec)

    if rank == 0:
        if e2e:
            line["e2e"] = {"value": m["nk_total"] / (e2e_ms_max * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms_max,
                           "h2d_bytes_per_step": e2e_h2d, "d2h_bytes_per_step": e2e_d2h}
            if world == 1:
                line["e2e"].update({
                    "api": "euler_pipeline_run_host + euler_pipeline_download (compressed graph)",
                    "serial_ms_per_step": e2e["serial_ms"], "pipelined_ms_per_step": e2e["piped_ms"],
                    "pipelining": "2 contexts on 2 host threads alternate steps (copies of one overlap the kernels of the other); "
                                  "serial_ms_per_step is one context, one step at a time"})
            else:
                line["e2e"].update({
                    "api": "per rank: pinned host shard -> device, eulercuda.dist.build_partitioned, euler_pipeline_download of the rank's "
                           "part of the compressed graph; wall clock between barriers, max over ranks; bytes summed over ranks",
                    "pipelining": "none (one step at a time)"})
        if extra:
            line["extra"] = extra
        if world == 1 and not args.no_cpu:
            # the reference arm in a child process (no fork of a process that holds a CUDA context)
            try:
                import subprocess
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0",
                                      "--workload", args.workload] + (["--k", str(args.k)] if args.k else []),
                                     capture_output=True, text=True, timeout=180)
                ref = json.loads(out.stdout.strip().splitlines()[-1])
                line["cpu_baseline"] = dict(ref["cpu_baseline"], code=ref["config"]["code"])
            except Exception as e:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "unavailable",
                                        "sample": "reference arm failed: %s" % e}
    guard.finish(line)
    LineGuard(30.0, None)   # the shutdown (barrier, NCCL teardown) must not keep a finished run alive
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
