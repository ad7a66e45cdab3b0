#!/usr/bin/env python
"""Time multi-k unitigs (Context.unitigs_multik_ingested) against one K (unitigs_clean_ingested(63, 1)) on one GPU.

Reads: BASELINE configs[1] shape (4.6 Mbp genome, 30x) with 1 % substitutions (err_ppm = 10000) from the library's
seeded generator, at 100 bp and 150 bp; limit 1, default clean-up at every step.  The reads are ingested once per read
length; then, after two warm-up calls of each, `--calls` rounds alternate unitigs_clean_ingested(63, 1),
unitigs_multik_ingested([31, 63]) and unitigs_multik_ingested([21, 31, 41, 51, 63]), each timed with a host clock
(each call ends in a stream synchronise; the Python wrapper makes the two-call size / fill protocol, so one call runs
the whole job twice).  Prints one JSON line with the GPU's name and power limit, the median times, and contigs and N50
of each output.

    python scripts/time_multik.py [--calls 10]
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

from time_clean import fasta_bytes, n50  # noqa: E402
from time_unitigs import gpu_info  # noqa: E402

LISTS = [[63], [31, 63], [21, 31, 41, 51, 63]]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--calls", type=int, default=10)
    args = ap.parse_args()
    import _native as N
    name, power = gpu_info()
    ctx = N.Context(0)

    def run(ks):
        if len(ks) == 1:
            c, _, _ = ctx.unitigs_clean_ingested(ks[0], 1)
            return c
        c, _, _ = ctx.unitigs_multik_ingested(ks, 1)
        return c

    rows = []
    for L in (100, 150):
        data, n = fasta_bytes(ctx, L)
        assert ctx.ingest(data, 1) == (n, n * L)
        out = {}
        for _ in range(2):
            for ks in LISTS:
                out[tuple(ks)] = run(ks)
        times = {tuple(ks): [] for ks in LISTS}
        for _ in range(args.calls):
            for ks in LISTS:
                t0 = time.perf_counter()
                out[tuple(ks)] = run(ks)
                times[tuple(ks)].append(time.perf_counter() - t0)
        for ks in LISTS:
            c = out[tuple(ks)]
            rows.append({"L": L, "ks": ks, "reads": n, "ms_median": round(1e3 * float(np.median(times[tuple(ks)])), 3),
                         "contigs": len(c), "n50": n50(c), "bases": sum(len(x) for x in c)})
    ctx.close()
    print(json.dumps({"what": "unitigs_clean_ingested(63, 1) vs unitigs_multik_ingested(ks, 1), configs[1] shape "
                              "(4.6 Mbp, 30x, err 1 %)", "calls": args.calls, "gpu": name, "power_limit": power,
                      "results": rows}))


if __name__ == "__main__":
    main()
