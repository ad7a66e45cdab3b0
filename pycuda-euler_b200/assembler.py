#!/usr/bin/env python
"""assembler.py -- the partition driver (SURVEY §8 f4): same command line as the reference's
``src/assembler.py`` (``-i -o -k -d``; a stub there) and the job its Spark driver does
(``src/cli_spark_gpu.py:37``: ``mapPartitions(assemble2)`` over read partitions), on the GPUs of one box.

    python assembler.py -i reads.fq -o contigs.fa -k 31                      # one GPU
    python assembler.py -i reads.fq -o contigs.fa -k 63                      # one GPU, k up to 63
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


def write_outputs(path, contigs, G, k):
    from referenceassembler import referenceAssembler as ram
    with open(path, "w") as f:
        ram.write_fasta(contigs, f)
    if G is not None:
        with open(path + ".gfa", "w") as f:
            ram.write_gfa(G, contigs, k, f)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('-i', dest='input_filename', required=True, help='Input File Name (FASTA / FASTQ)')
    ap.add_argument('-o', dest='output_filename', required=True, help='Output File Name')
    ap.add_argument('-k', dest='k', type=int, default=31, help='kmer size')
    ap.add_argument('-d', action='store_true', default=False, help='Use DDFS (accepted for compatibility; ignored)')
    ap.add_argument('--limit', type=int, default=1, help='keep k-mers with both-strand count > limit (build() default 1)')
    ap.add_argument('--mode', choices=['unitig', 'euler', 'replicas'], default='unitig')
    args = ap.parse_args(argv)
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
    if world == 1 or args.mode == 'replicas':
        contigs = ctx.unitigs_ingested(K, args.limit) if nbases else []
        from referenceassembler import referenceAssembler as ram
        G = ram.link_graph(contigs, K) if (contigs and K <= 63) else None
        out = args.output_filename if world == 1 else "%s.part%d" % (args.output_filename, rank)
        write_outputs(out, contigs, G, K)
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
        if args.mode == 'euler':
            contigs, G = [], None
            if len(all_k):
                ctx.run_lmers(all_k, all_v, K, N.RUN_CANONICAL_IDS | N.RUN_EXPAND_EDGES)
                contigs = ctx.pipeline_contigs()
        else:
            contigs = ctx.unitigs_from_kmers(all_k, all_v, K) if len(all_k) else []
            G = ram.link_graph(contigs, K) if (contigs and K <= 63) else None
        write_outputs(args.output_filename, contigs, G, K)
        log.info("%d k-mers joined, %d contigs -> %s", len(all_k), len(contigs), args.output_filename)
    dist.barrier()
    dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
