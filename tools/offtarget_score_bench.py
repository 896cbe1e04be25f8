#!/usr/bin/env python3
"""Cost of the off-target scores (csrc/offtarget.cuh: k_ot_join<OtScore>) next to the counts (k_ot_join<OtCount>) on
the benchmark genomes:

    python tools/offtarget_score_bench.py [workload ...]     (default: arabidopsis maize)

Per workload: commit every chromosome (as many genome handles as the 32-bit limits ask for), scan it, and build one
index without loci over all handles.  Then, at k = 0, 1, 2, 3, for both strands of every handle, one count call and
one score call with the MIT weights, alternated: ms_count and ms_score are the device times (crp_offtarget_timing,
the same ten counting sorts and the join) summed over all candidates.  One JSON line per (workload, k) with the
score/count ratio, the MIT hit-score sum over all candidates, and the device with its power limit and maximum SM
clock (nvidia-smi, read only, in the same call).
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
    parts = []
    for first, cnt in pipeline._groups(lengths):
        g = engine.Genome()
        for k in range(first, first + cnt):
            g.add_token(W.token(workload, k))
        g.commit()
        parts.append((g, g.scan(20), first, cnt))
    index = engine.OffTargetIndex([g for g, _, _, _ in parts])
    queries = sum(r.n_plus + r.n_minus for _, r, _, _ in parts)
    weights = engine.mit_weights()
    setup_s = time.time() - t0
    for k in range(4):
        ms_count = ms_score = 0.0
        hit_sum = 0.0
        scored = 0
        wall = time.time()
        for _, r, _, _ in parts:
            for strand in "+-":
                index.count_candidates(r, strand, k)
                ms_count += index.timing()["ms_count"]
                sums = index.score_candidates(r, strand, k, weights)
                ms_score += index.timing()["ms_count"]
                ok = sums != np.uint64(index.NO_SCORE)
                scored += int(ok.sum())
                hit_sum += float(sums[ok].astype(np.float64).sum()) / engine.SCORE_ONE   # a summary, in fp64
        line = {"workload": workload, "config": W.CONFIG_NAME[workload], "k": k, "sites": index.num_sites(),
                "queries": int(queries), "scored": scored, "ms_count": round(ms_count, 3),
                "ms_score": round(ms_score, 3), "score_over_count": round(ms_score / ms_count, 3) if ms_count else None,
                "mit_hit_sum_total": hit_sum, "wall_s": round(time.time() - wall, 3),
                "setup_s": round(setup_s, 1), **info}
        print(json.dumps(line), flush=True)
    index.free()
    for g, r, _, _ in parts:
        r.free()
        g.free()


def main(argv):
    engine.init(0)
    info = device_info()
    for workload in argv or ["arabidopsis", "maize"]:
        run(workload, info)


if __name__ == "__main__":
    main(sys.argv[1:])
