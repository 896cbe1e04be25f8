#!/usr/bin/env python3
"""Throughput of the off-target counts (csrc/offtarget.cuh) on the benchmark genomes:

    python tools/offtarget_bench.py [workload ...]        (default: arabidopsis maize)

Per workload: commit every chromosome (as many genome handles as the 32-bit limits ask for), scan it, build ONE
index over all handles, then count every candidate of both strands at k = 0, 1, 2, 3.  One JSON line per
(workload, k): sites, queries, comparisons (sum over the 10 part pairs and 65,536 buckets of queries x sites),
ms_sites (site extraction, once per workload), ms_count (device time of all count calls of that k, summed),
comparisons per second, and the device with its power limit and maximum SM clock (nvidia-smi, read only).
arabidopsis (configs[1]) is the size users run most; maize (configs[3]) adds the repeat library -- ~6,500 soft-masked
copies of each of 64 elements -- whose buckets hold 10^4 - 10^5 sites each.
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]
import numpy as np                                     # noqa: E402
import workloads as W                                  # noqa: E402
from cropsr_b200 import engine, pipeline               # noqa: E402


def device_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.splitlines()[0].split(",")]
        return {"device": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                             # the numbers are still device times; say what is missing
        return {"device": None, "nvidia_smi": str(e)}


def run(workload, info):
    t0 = time.time()
    lengths = W.token_lengths(workload)
    parts, index = [], engine.OffTargetIndex()
    for first, cnt in pipeline._groups(lengths):
        g = engine.Genome()
        for k in range(first, first + cnt):
            g.add_token(W.token(workload, k))
        g.commit()
        parts.append((g, g.scan(20)))
        index.add_genome(g)
    ms_sites = index.timing()["ms_sites"]
    queries = sum(r.n_plus + r.n_minus for _, r in parts)
    setup_s = time.time() - t0
    for k in range(4):
        ms, cmp, wall = 0.0, 0, time.time()
        for _, r in parts:
            for strand in "+-":
                index.count_candidates(r, strand, k)
                t = index.timing()
                ms += t["ms_count"]
                cmp += t["comparisons"]
        line = {"workload": workload, "config": W.CONFIG_NAME[workload], "k": k, "sites": index.num_sites(),
                "queries": int(queries), "comparisons": int(cmp), "ms_sites": round(ms_sites, 3), "ms_count": round(ms, 3),
                "comparisons_per_s": cmp / (ms * 1e-3) if ms else None, "count_calls": 2 * len(parts),
                "wall_s": round(time.time() - wall, 3), "setup_s": round(setup_s, 1), **info}
        print(json.dumps(line), flush=True)
    index.free()
    for g, r in parts:
        r.free()
        g.free()


def main(argv):
    engine.init(0)
    info = device_info()
    for workload in argv or ["arabidopsis", "maize"]:
        run(workload, info)


if __name__ == "__main__":
    main(sys.argv[1:])
