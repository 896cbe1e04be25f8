#!/usr/bin/env python3
"""Off-target sites at other PAMs (csrc/offtarget.cuh: k_ot_sites<*, true>, crp_offtarget_new_pam) next to NGG on the
benchmark genomes:

    python tools/offtarget_pam_bench.py [workload ...]     (default: arabidopsis maize)

Per workload: commit every chromosome (as many genome handles as the 32-bit limits ask for) and scan it.  Then one
index without loci per entry of PATTERNS, over all handles: NGG through crp_offtarget_new (the NGG kernel) and again
through crp_offtarget_new_pam("NGG") (the same kernel, chosen by the pattern), then NAG and NGA (the pattern kernel).
Per index: num_sites and ms_sites (device time of every add_genome), and at k = 0, 1, 2, 3 for both strands of every
handle one count call and one score call with the MIT weights: ms_count, comparisons and ms_score summed over all
candidates.  One JSON line per (workload, pattern, k) with the device, its power limit and maximum SM clock
(nvidia-smi, read only, in the same call).
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]
import workloads as W                                  # noqa: E402
from cropsr_b200 import _native as N, engine, pipeline   # noqa: E402

PATTERNS = [("NGG", "crp_offtarget_new"), ("NGG", "crp_offtarget_new_pam"), ("NAG", "crp_offtarget_new_pam"),
            ("NGA", "crp_offtarget_new_pam")]


def device_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.splitlines()[0].split(",")]
        return {"device": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                             # the numbers are still device times; say what is missing
        return {"device": None, "nvidia_smi": str(e)}


def new_index(pam, via, handles):
    """an OffTargetIndex made by the named constructor"""
    import ctypes as C
    if via == "crp_offtarget_new":
        return engine.OffTargetIndex(handles)
    index = engine.OffTargetIndex.__new__(engine.OffTargetIndex)
    index.pam, index.loci, index._h = pam, False, C.c_void_p()
    N.check(N.lib.crp_offtarget_new_pam(C.byref(index._h), pam.encode(), 0))
    for g in handles:
        index.add_genome(g)
    return index


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
    queries = sum(r.n_plus + r.n_minus for _, r, _, _ in parts)
    weights = engine.mit_weights()
    setup_s = round(time.time() - t0, 1)
    for pam, via in PATTERNS:
        index = new_index(pam, via, [g for g, _, _, _ in parts])
        ms_sites = index.timing()["ms_sites"]
        for k in range(4):
            ms_count = ms_score = 0.0
            comparisons = 0
            for _, r, _, _ in parts:
                for strand in "+-":
                    index.count_candidates(r, strand, k)
                    t = index.timing()
                    ms_count += t["ms_count"]
                    comparisons += t["comparisons"]
                    index.score_candidates(r, strand, k, weights)
                    ms_score += index.timing()["ms_count"]
            line = {"workload": workload, "config": W.CONFIG_NAME[workload], "pam": pam, "constructor": via, "k": k,
                    "num_sites": index.num_sites(), "ms_sites": round(ms_sites, 3), "queries": int(queries),
                    "ms_count": round(ms_count, 3), "comparisons": comparisons, "ms_score": round(ms_score, 3),
                    "setup_s": setup_s, **info}
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
