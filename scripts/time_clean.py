#!/usr/bin/env python
"""Time unitig clean-up (Context.unitigs_clean_ingested) against plain unitigs (unitigs_ingested) on one GPU.

Reads: BASELINE configs[1] shape (4.6 Mbp genome, 30x) with 1 % substitutions (err_ppm = 10000) from the library's
seeded generator, at 100 bp and 150 bp; K = 31 and 63, limit 1.  The reads are ingested once per read length; then,
after two warm-up calls of each, `--calls` alternating calls of unitigs_ingested(K, 1) and
unitigs_clean_ingested(K, 1) are timed with a host clock (each call ends in a stream synchronise; the Python wrapper
makes the two-call size / fill protocol, so one call runs the stage twice).  Prints one JSON line with the GPU's name
and power limit, the median times, and rounds, contigs and N50 of both outputs.

    python scripts/time_clean.py [--calls 10]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "pycuda-euler_b200"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.dont_write_bytecode = True

from time_unitigs import COV, G, gpu_info  # noqa: E402

ERR_PPM = 10000


def fasta_bytes(ctx, L):
    import torch
    n = G * COV // L
    d = torch.empty(n * L, dtype=torch.uint8, device="cuda")
    ctx.synth_reads_dev(d.data_ptr(), G, L, ERR_PPM, 0, n)
    ctx.sync()
    reads = d.cpu().numpy().reshape(n, L)
    rows = np.empty((n, L + 3), np.uint8)
    rows[:, 0], rows[:, 1], rows[:, 2:L + 2], rows[:, L + 2] = ord(">"), ord("\n"), reads, ord("\n")
    return rows.tobytes(), n


def n50(contigs):
    lens = sorted((len(c) for c in contigs), reverse=True)
    tot, acc = sum(lens), 0
    for x in lens:
        acc += x
        if 2 * acc >= tot:
            return x
    return 0


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--calls", type=int, default=10)
    args = ap.parse_args()
    import _native as N
    name, power = gpu_info()
    ctx = N.Context(0)
    rows = []
    for L in (100, 150):
        data, n = fasta_bytes(ctx, L)
        assert ctx.ingest(data, 1) == (n, n * L)
        for K in (31, 63):
            for _ in range(2):
                plain = ctx.unitigs_ingested(K, 1)
                cleaned, _, st = ctx.unitigs_clean_ingested(K, 1)
            tp, tc = [], []
            for _ in range(args.calls):
                t0 = time.perf_counter()
                plain = ctx.unitigs_ingested(K, 1)
                tp.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                cleaned, _, st = ctx.unitigs_clean_ingested(K, 1)
                tc.append(time.perf_counter() - t0)
            mp, mc = 1e3 * float(np.median(tp)), 1e3 * float(np.median(tc))
            rows.append({"L": L, "K": K, "reads": n, "ms_unitigs_median": round(mp, 3), "ms_clean_median": round(mc, 3),
                         "clean_over_plain": round(mc / mp, 3), "rounds": st["rounds"], "stats": st,
                         "contigs_plain": len(plain), "n50_plain": n50(plain),
                         "contigs_clean": len(cleaned), "n50_clean": n50(cleaned)})
    ctx.close()
    print(json.dumps({"what": "unitigs_ingested(K, 1) vs unitigs_clean_ingested(K, 1), configs[1] shape (4.6 Mbp, 30x, "
                              "err 1 %)", "calls": args.calls, "gpu": name, "power_limit": power, "results": rows}))


if __name__ == "__main__":
    main()
