#!/usr/bin/env python
"""Time unitig mode (Context.unitigs_ingested) on one GPU at K = 31 (one-word keys) and K = 63 (two-word keys).

Reads: BASELINE configs[1] shape (4.6 Mbp genome, 30x, no errors) from the library's seeded generator, at 100 bp
and 150 bp.  They are written as FASTA bytes in memory and ingested once per read length; then, after two
warm-up calls, `--calls` calls of unitigs_ingested(K, 1) are timed with a host clock (each call ends in a
stream synchronise; the Python wrapper makes the two-call size / fill protocol, so one call runs the stage
twice).  Prints one JSON line with the GPU's name and power limit.

    python scripts/time_unitigs.py [--calls 10]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "pycuda-euler_b200"))
sys.dont_write_bytecode = True

G, COV = 4_600_000, 30


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def fasta_bytes(ctx, L):
    import torch
    n = G * COV // L
    d = torch.empty(n * L, dtype=torch.uint8, device="cuda")
    ctx.synth_reads_dev(d.data_ptr(), G, L, 0, 0, n)
    ctx.sync()
    reads = d.cpu().numpy().reshape(n, L)
    rows = np.empty((n, L + 3), np.uint8)
    rows[:, 0], rows[:, 1], rows[:, 2:L + 2], rows[:, L + 2] = ord(">"), ord("\n"), reads, ord("\n")
    return rows.tobytes(), n


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
                contigs = ctx.unitigs_ingested(K, 1)
            t = []
            for _ in range(args.calls):
                t0 = time.perf_counter()
                contigs = ctx.unitigs_ingested(K, 1)
                t.append(time.perf_counter() - t0)
            ms = 1e3 * float(np.median(t))
            windows = n * (L - K + 1)
            rows.append({"L": L, "K": K, "reads": n, "ms_per_call_median": round(ms, 3), "ms_per_call_min": round(1e3 * min(t), 3),
                         "kmer_windows_per_s": round(windows / (ms / 1e3), 1), "contigs": len(contigs),
                         "text_bytes": sum(len(c) + 1 for c in contigs)})
    ctx.close()
    print(json.dumps({"what": "unitigs_ingested(K, 1), configs[1] shape (4.6 Mbp, 30x, err 0)", "calls": args.calls,
                      "gpu": name, "power_limit": power, "results": rows}))


if __name__ == "__main__":
    main()
