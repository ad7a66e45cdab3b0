#!/usr/bin/env python
"""assembler.py -- the partition driver (SURVEY §8 f4): same command line as the reference's
``src/assembler.py`` (``-i -o -k -d``; a stub there) and the job its Spark driver does
(``src/cli_spark_gpu.py:37``: ``mapPartitions(assemble2)`` over read partitions), on the GPUs of one box.

    python assembler.py -i reads.fq -o contigs.fa -k 31                      # one GPU
    python assembler.py -i reads.fq -o contigs.fa -k 63                      # one GPU, k up to 63
    python assembler.py -i reads.fq -o contigs.fa -k 31 --clean              # clip tips, pop bubbles first
    python assembler.py -i reads.fq -o contigs.fa --k-list 21,41,63 --clean  # multi-k: one GPU or replicas
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 \\
           assembler.py -i reads.fq -o contigs.fa -k 31                      # 8 GPUs, one assembly

Modes
  unitig (default)  one assembly of ALL reads: every rank ingests its byte range of the file on its GPU,
                    the k-mer space is partitioned across the ranks (one exchange over NVLink, csrc/dist.cu),
                    every rank counts the k-mers it owns, and the table (count > limit) is joined on rank 0,
                    which compacts it into unitigs and their link graph.  The result equals the single-GPU
                    assembly of the whole file -- unlike the reference's partitions, which never see each
                    other's reads.
  euler             the GPU-Euler path (assemble2 mode='euler': de Bruijn graph with k-mer EDGES, Euler tour,
                    partial contigs).  Across GPUs the per-rank edge tables are joined on rank 0, which runs the
                    graph and tour stages (euler_pipeline_run_lmers): same contigs as on one GPU.
  replicas          the reference's semantics: every rank assembles its own partition of the reads
                    independently and writes <out>.part<rank>.
Outputs: FASTA contigs in -o, the GFA link graph in <out>.gfa (unitig mode).  k: 2..63 on one GPU and in
replicas mode, 2..32 for one assembly across GPUs.

--clean (unitig and replicas modes) removes what sequencing errors leave in the graph before the unitigs are
written: tips (dead-end branches), isolated fragments and the weaker branches of bubbles, each up to a length in
K-mers (--tip-len, --isolated-len, --bubble-len; default 2k, 0 turns a rule off), for up to --clean-rounds rounds
(rules: include/euler_b200.h, euler_unitigs_clean).  The GFA's S lines then carry KC:i:<sum of the contig's K-mer
counts>, and the log gets a line with the rounds and the removals.

--k-list k1,k2,... (strictly increasing, 2..63, at most 16; in place of -k) assembles at each K in turn and adds the
K-mers of each step's contigs to the graph of the next (rule: include/euler_b200.h, euler_unitigs_multik), so a small
K bridges thinly covered places and a large K resolves repeats.  With --clean every step is cleaned up (the lengths
default to 2k at each step).  One GPU and replicas mode only.  The log gets one line per step; the FASTA and the GFA
(link graph at the last K, KC:i: from the last step's sums) are those of the last step.
"""
import argparse
import logging
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)


def detect_format(path, data):
    ext = path.rsplit(".", 1)[-1].lower()
    if ext in ("fa", "fasta", "fsa"):
        return 1
    if ext in ("fq", "fastq"):
        return 2
    return 2 if data[:1] == b"@" else 1


def split_records(data, world, fmt):
    """Byte ranges [(a, b)] * world of `data`, cut at record boundaries: any line start for FASTA (every
    non-header line is a read, eulercuda.py:439-447), every 4th line start for FASTQ (:44-56)."""
    n = len(data)
    if world <= 1 or n == 0:
        return [(0, n)] + [(n, n)] * (max(world, 1) - 1)
    nl = np.flatnonzero(np.frombuffer(data, dtype=np.uint8) == 10)
    starts = np.concatenate([[0], nl + 1])
    starts = starts[starts < n]
    if fmt == 2:
        starts = starts[::4]
    cuts = [0]
    for r in range(1, world):
        target = n * r // world
        j = int(np.searchsorted(starts, target))
        cuts.append(int(starts[j]) if j < len(starts) else n)
    cuts.append(n)
    cuts = [max(c, p) for c, p in zip(cuts, [0] + cuts[:-1])]   # monotone
    for i in range(1, len(cuts)):
        cuts[i] = max(cuts[i], cuts[i - 1])
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def write_outputs(path, contigs, G, k, kc=None):
    from referenceassembler import referenceAssembler as ram
    with open(path, "w") as f:
        ram.write_fasta(contigs, f)
    if G is not None:
        with open(path + ".gfa", "w") as f:
            ram.write_gfa(G, contigs, k, f, kc=kc)


def clean_kwargs(args):
    return dict(tip_len=args.tip_len, isolated_len=args.isolated_len, bubble_len=args.bubble_len, max_rounds=args.clean_rounds)


def log_clean(log, rank, st):
    log.info("rank %d: clean-up: %d rounds, %d tips, %d isolated, %d bubble branches, %d K-mers removed", rank, st["rounds"],
             st["tips"], st["isolated"], st["bubble_branches"], st["kmers_removed"])


def log_step(log, rank, s, clean):
    c = s["clean"]
    log.info("rank %d: K = %d: %d contigs, %d bases, %d K-mers added from the previous contigs%s", rank, s["K"],
             s["contigs"], s["bases"], s["nodes_added"],
             "; clean-up: %d rounds, %d tips, %d isolated, %d bubble branches, %d K-mers removed" %
             (c["rounds"], c["tips"], c["isolated"], c["bubble_branches"], c["kmers_removed"]) if clean else "")


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('-i', dest='input_filename', required=True, help='Input File Name (FASTA / FASTQ)')
    ap.add_argument('-o', dest='output_filename', required=True, help='Output File Name')
    ap.add_argument('-k', dest='k', type=int, default=None, help='kmer size (default 31)')
    ap.add_argument('--k-list', default=None, help='multi-k: strictly increasing K values, e.g. 21,41,63 (not with -k)')
    ap.add_argument('-d', action='store_true', default=False, help='Use DDFS (accepted for compatibility; ignored)')
    ap.add_argument('--limit', type=int, default=1, help='keep k-mers with both-strand count > limit (build() default 1)')
    ap.add_argument('--mode', choices=['unitig', 'euler', 'replicas'], default='unitig')
    ap.add_argument('--clean', action='store_true', help='clip tips, drop isolated fragments and pop bubbles (unitig routes)')
    ap.add_argument('--tip-len', type=int, default=None, help='longest tip removed, in K-mers (default 2k; 0 = off)')
    ap.add_argument('--isolated-len', type=int, default=None, help='longest isolated fragment removed, in K-mers (default 2k)')
    ap.add_argument('--bubble-len', type=int, default=None, help='longest bubble branch removed, in K-mers (default 2k)')
    ap.add_argument('--clean-rounds', type=int, default=10, help='most clean-up rounds')
    args = ap.parse_args(argv)
    ks = None
    if args.k_list is not None:
        if args.k is not None:
            ap.error("give either -k or --k-list, not both")
        try:
            ks = [int(x) for x in args.k_list.split(",")]
        except ValueError:
            ap.error("--k-list takes comma-separated integers, got %r" % args.k_list)
        if args.mode == 'euler':
            ap.error("--k-list is a unitig-mode option; --mode euler takes one -k")
        if not 1 <= len(ks) <= 16:   # EULER_MULTIK_MAX
            ap.error("--k-list takes 1 to 16 values, got %d" % len(ks))
        if any(k < 2 or k > 63 for k in ks):
            ap.error("--k-list values must be in [2, 63], got %s" % args.k_list)
        if any(b <= a for a, b in zip(ks, ks[1:])):
            ap.error("--k-list must be strictly increasing, got %s" % args.k_list)
    if args.k is None:
        args.k = 31 if ks is None else ks[-1]
    logging.basicConfig(level=logging.INFO, format='%(asctime)s %(levelname)s %(message)s')
    log = logging.getLogger("assembler")

    import _native as N
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    K = args.k
    with open(args.input_filename, "rb") as f:
        data = f.read()
    fmt = detect_format(args.input_filename, data)
    a, b = split_records(data, world, fmt)[rank]
    ctx = N.Context(local_rank)
    nreads, nbases = ctx.ingest(data[a:b], fmt)
    log.info("rank %d/%d: bytes [%d, %d): %d reads, %d bases", rank, world, a, b, nreads, nbases)

    if args.mode == 'euler' and world == 1:
        contigs = []
        if nbases:
            ctx.run_ingested(K, N.RUN_CANONICAL_IDS | N.RUN_EXPAND_EDGES)
            contigs = ctx.pipeline_contigs()
        write_outputs(args.output_filename, contigs, None, K)
        log.info("%d contigs -> %s", len(contigs), args.output_filename)
        return 0
    if ks is not None and world > 1 and args.mode != 'replicas':
        raise SystemExit("--k-list runs on one GPU or in replicas mode; one assembly across GPUs takes one -k")
    if world == 1 or args.mode == 'replicas':
        kc = None
        if ks is not None:
            contigs, kc, steps = ctx.unitigs_multik_ingested(ks, args.limit, clean=args.clean, **clean_kwargs(args)) \
                if nbases else ([], None, [])
            for s in steps:
                log_step(log, rank, s, args.clean)
        elif args.clean:
            contigs, kc, st = ctx.unitigs_clean_ingested(K, args.limit, **clean_kwargs(args)) if nbases else ([], None, None)
            if st:
                log_clean(log, rank, st)
        else:
            contigs = ctx.unitigs_ingested(K, args.limit) if nbases else []
        from referenceassembler import referenceAssembler as ram
        G = ram.link_graph(contigs, K) if (contigs and K <= 63) else None
        out = args.output_filename if world == 1 else "%s.part%d" % (args.output_filename, rank)
        write_outputs(out, contigs, G, K, kc)
        log.info("rank %d: %d contigs -> %s", rank, len(contigs), out)
        return 0

    import torch
    import torch.distributed as dist
    from eulercuda.dist import build_partitioned
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if K < 2 or K > 32:
        raise SystemExit("one assembly across GPUs needs 2 <= k <= 32")
    buf, off = ctx.ingest_download()
    d_reads = torch.zeros(max(len(buf), 1) + 16, dtype=torch.uint8, device="cuda")
    d_reads[:len(buf)] = torch.from_numpy(np.ascontiguousarray(buf)).cuda()
    d_off = torch.from_numpy(np.ascontiguousarray(off).astype(np.int64)).cuda()
    # the K-mers are the "l-mers" of the partition: every both-strand K-mer ends up on exactly one rank
    # (the owner of its prefix vertex) with its full multiplicity
    st, info = build_partitioned(ctx, d_reads, d_off, nreads, nbases, K, rank, world, 0)
    keys = ctx.download(N.ART_LMER_KEYS)
    vals = ctx.download(N.ART_LMER_VALUES)
    if args.mode == 'unitig':
        keep = vals > args.limit
        keys, vals = keys[keep], vals[keep]
    log.info("rank %d: %d k-mer windows sent, %d received, %d owned k-mers above the limit", rank, info["sent_keys"],
             info["recv_keys"], len(keys))
    gathered = [None] * world if rank == 0 else None
    dist.gather_object((keys, vals), gathered, dst=0)
    if rank == 0:
        all_k = np.concatenate([g[0] for g in gathered])
        all_v = np.concatenate([g[1] for g in gathered])
        from referenceassembler import referenceAssembler as ram
        kc = None
        if args.mode == 'euler':
            contigs, G = [], None
            if len(all_k):
                ctx.run_lmers(all_k, all_v, K, N.RUN_CANONICAL_IDS | N.RUN_EXPAND_EDGES)
                contigs = ctx.pipeline_contigs()
        else:
            if args.clean and len(all_k):
                contigs, kc, st = ctx.unitigs_clean_from_kmers(all_k, all_v, K, **clean_kwargs(args))
                log_clean(log, rank, st)
            else:
                contigs = ctx.unitigs_from_kmers(all_k, all_v, K) if len(all_k) else []
            G = ram.link_graph(contigs, K) if (contigs and K <= 63) else None
        write_outputs(args.output_filename, contigs, G, K, kc)
        log.info("%d k-mers joined, %d contigs -> %s", len(all_k), len(contigs), args.output_filename)
    dist.barrier()
    dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
